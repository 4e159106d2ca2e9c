"""Host-side orchestration of one contrastive step (engine-agnostic).

Single GPU:   normalise -> forward statistics -> loss      |  backward (two sides) -> normalise-bwd
Row-sharded global batch over a process group (SURVEY.md section 8e; replaces the autograd-blind
``dist.all_gather`` + ``torch.cat`` of old/clip_opt.py:102-112 / run1/full.py:77-84):

    rank p owns rows [p*n, (p+1)*n) of both modalities
    fwd:  gather every rank's B rows (norms fused)  ->  local A rows x all columns  ->  exchange the column
          (shift, sum) partials and the row pairs  ->  sum the scalar loss
    bwd:  side A: local A rows x all B rows -> dA;  side B: local B rows x all (gathered) A rows -> dB.
          Both gradients are complete on their owner: no [N,d] fp32 partial, no reduce-scatter.
    The exchange steps live in exchange.py: kernels over NVLink peer memory on GPUs, collectives under gloo.

The engine (``engine.CudaEngine`` in production) provides the kernels; tests drive the same code
with a CPU stand-in over gloo to cover the sharding/offset/collective logic without a GPU.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Optional

import torch
import torch.distributed as dist

from . import exchange as _exchange

FLAG_FORCE_EXACT = 1
FLAG_UNBOUNDED = 2    # extra columns of arbitrary norm: |S| <= s does not hold (tensor-core kernels with true maxima)


@dataclass
class StepState:
    a: torch.Tensor                 # caller's embeddings (for the normalise backward)
    b: torch.Tensor
    a_c: torch.Tensor               # local rows in the compute dtype
    b_c: torch.Tensor
    y: torch.Tensor                 # all columns: gathered B (+ extra negatives), raw, compute dtype
    y_t: Optional[torch.Tensor]
    xa: Optional[torch.Tensor]      # all rows: gathered A (side B of the backward streams it)
    xa_t: Optional[torch.Tensor]
    rinv_a: torch.Tensor
    rinv_b: torch.Tensor
    rinv_y: torch.Tensor
    rinv_xa: Optional[torch.Tensor]
    row_m: torch.Tensor             # log-sum-exp kept as (shift, sum) pairs: r = row_m + log(row_l); local rows
    row_l: torch.Tensor
    row_m_all: Optional[torch.Tensor]   # the same for every rank's rows (gathered)
    row_l_all: Optional[torch.Tensor]
    col_m: torch.Tensor             # globally combined column statistics
    col_l: torch.Tensor
    diag: torch.Tensor
    scale: float
    scale_dev: Optional[torch.Tensor]   # device scalar s (the kernels read it; `scale` is then only the host's hint)
    symmetric: bool
    n_local: int
    n_global: int
    diag_offset: int
    flags: int
    group: object
    want_t: bool
    compute_dtype: torch.dtype
    xchg: object = None             # the exchange of this step (exchange.py); None on one GPU
    both_sharded: bool = False      # the backward will run the row-sharded two-sided kernel (no gathered A rows needed)
    xchg_generation: int = 0        # lease generation of the exchange buffers (exchange._Pool reclaims abandoned leases)


def contrastive_forward(engine, a, b, scale, *, symmetric=True, extra=None, group=None,
                        compute_dtype=torch.bfloat16, flags=0, need_grad=True, scale_dev=None, rinv_a=None, rinv_b=None):
    """Returns (loss [1] f32 -- the GLOBAL mean loss, identical on every rank --, StepState).

    ``scale`` is s as a float, or a zero-argument callable returning it: the callable is invoked only after the
    scale-independent work (row norms, the gather of the columns) has been enqueued, so that a host read of the
    logit_scale parameter overlaps with it instead of leaving the GPU idle."""
    if a.dim() != 2 or b.dim() != 2 or a.shape != b.shape:
        raise ValueError(f"expected two [N,d] embedding matrices of equal shape, got {tuple(a.shape)} and {tuple(b.shape)}")
    n_local, d = a.shape
    world = dist.get_world_size(group) if group is not None else 1
    rank = dist.get_rank(group) if group is not None else 0
    n_global = n_local * world
    diag_offset = rank * n_local
    n_extra = extra.shape[0] if extra is not None else 0

    xchg = None
    both_sharded = False
    beside = False
    # rinv_a / rinv_b: 1/norms that came with the rows (the fused projection-head tail, heads.py): nothing to recompute
    if rinv_a is None:
        rinv_a, _ = engine.normalize(a)
    a_c, _ = engine.stage(a, compute_dtype)
    if world > 1:
        # the exchange buffers do not depend on the number of extra columns (a hard-negative cache that grows from step
        # to step would otherwise need a new set -- a host-side rendezvous -- for every length)
        xchg = _exchange.open_exchange(engine, group, n_local, d, n_global, compute_dtype, a.device)
        if callable(scale):
            scale = scale()
        # the gather runs BESIDE the forward sweep where the sweep can wait block by block (include/clipnce.h,
        # clipnce_forward_gathered): every rank decides from the same shapes, types and scale hint
        beside = bool(getattr(xchg, "kind", "") == "nvlink-peer" and extra is None
                      and b.dtype == compute_dtype == torch.bfloat16 and n_local % 256 == 0
                      and n_local >= _exchange.GATHER_BESIDE_MIN_ROWS and n_global <= (1 << 22)
                      and hasattr(engine, "forward_gathered") and engine.forward_gathered_ok(compute_dtype, d, scale, flags))
        if beside:
            b_c, rinv_b, y, rinv_y = xchg.gather_cols_beside(b.contiguous(), rinv_b)
        else:
            b_c, rinv_b, y, rinv_y = xchg.gather_cols(b, compute_dtype)
        if need_grad:
            # two-sided backward over peer memory (one sweep emits dA and the reduce-scattered dB): nothing to gather
            both_sharded = bool(symmetric and extra is None and compute_dtype == torch.bfloat16 and
                                getattr(xchg, "kind", "") == "nvlink-peer" and hasattr(engine, "backward_both_sharded_sweep") and
                                engine.backward_both_bytes(n_local, n_global, d, compute_dtype, scale, flags, world) > 0)
            if not both_sharded:   # side B of the backward streams every rank's A rows; they travel behind the forward sweep
                xchg.gather_rows_begin(a, a_c, rinv_a, compute_dtype)
    else:
        if rinv_b is None:
            rinv_b, _ = engine.normalize(b)
        b_c, _ = engine.stage(b, compute_dtype)
        y, rinv_y = b_c, rinv_b
    if callable(scale):
        scale = scale()
    tc = engine.uses_tensor_cores(compute_dtype, d, scale, flags)
    want_t = bool(need_grad and tc and engine.needs_transposed(compute_dtype, d, scale, flags))
    if extra is not None:   # used as stored (old/clip_opt.py:118-121, tong/utils/losses.py:10-11): rinv = 1
        y = torch.cat([y, extra.detach().to(compute_dtype)], dim=0).contiguous()
        rinv_y = torch.cat([rinv_y, torch.ones(n_extra, dtype=rinv_y.dtype, device=rinv_y.device)])
    y_t = None
    if want_t:
        _, y_t = engine.stage(y, compute_dtype, want_t=True)

    kw = {"scale_dev": scale_dev} if scale_dev is not None else {}
    if beside:
        row_m, row_l, col_m, col_l, diag = engine.forward_gathered(a_c, y, rinv_a, rinv_y, scale, xchg.peers, xchg.world,
                                                                   xchg.rank, _exchange.PHASE_BLOCKS, flags, **kw)
    else:
        row_m, row_l, col_m, col_l, diag = engine.forward(a_c, y, rinv_a, rinv_y, diag_offset, scale, flags, **kw)
    xa, rinv_xa, row_m_all, row_l_all = a_c, rinv_a, row_m, row_l
    if world > 1:
        fixed = getattr(engine, "fixed_shift", None)
        fixed = bool(fixed is not None and fixed(compute_dtype, d, scale, flags))
        # only the batch's own columns are exchanged: extra negatives carry no positives, so their column statistics are
        # never used (no column loss, no column soft-max: the sum is set to +inf below)
        gm, gl, row_m_all, row_l_all = xchg.exchange_stats(row_m, row_l, col_m[:n_global], col_l[:n_global], fixed,
                                                           need_grad and not both_sharded)
        if both_sharded:
            row_m_all, row_l_all = row_m, row_l
        col_m = torch.cat([gm, col_m[n_global:]]) if n_extra else gm
        col_l = torch.cat([gl, col_l[n_global:]]) if n_extra else gl
        xa, rinv_xa = xchg.gather_rows_end() if (need_grad and not both_sharded) else ((a_c, rinv_a) if both_sharded else (None, None))
    if n_extra:
        col_l[n_global:] = float("inf")
    loss = engine.loss(row_m, row_l, col_m, col_l, diag, diag_offset, n_global, symmetric)
    if world > 1:
        loss = xchg.sum_scalars(loss, _exchange.PHASE_LOSS)
        if not need_grad:
            xchg.release()
            xchg = None
    st = StepState(a, b, a_c, b_c, y, y_t, xa, None, rinv_a, rinv_b, rinv_y, rinv_xa, row_m, row_l, row_m_all, row_l_all,
                   col_m, col_l, diag, scale, scale_dev, symmetric, n_local, n_global, diag_offset, flags, group, want_t,
                   compute_dtype, xchg, both_sharded, xchg.generation if xchg is not None else 0)
    return loss, st


def contrastive_backward(engine, st: StepState, grad_scale=None, grad_dtype_a=None, grad_dtype_b=None):
    """Returns (dA [n,d], dB [n,d], d_scale_sum [1]) for upstream gradient 1; ``grad_scale`` is an optional
    device scalar multiplied into dA/dB inside the normalise-backward kernel (d_scale_sum is left
    unscaled -- the caller multiplies that single element)."""
    n_glob, n, off = st.n_global, st.n_local, st.diag_offset
    if st.xa is None:
        raise RuntimeError("clip_dplm_b200: this step was run without need_grad")
    if st.xchg is not None and not st.xchg.owned_by(st.xchg_generation):
        raise RuntimeError("clip_dplm_b200: the exchange buffers of this forward were reclaimed by later steps (more than "
                           f"{_exchange._Pool.max_per_key} row-sharded forwards of one shape were live without a backward)")
    coef = 1.0 / ((2.0 if st.symmetric else 1.0) * n_glob)
    if st.row_l_all is st.row_l:
        row_w = row_w_all = engine.softmax_weights(st.row_l, coef)
    else:   # the gathered row statistics hold the local block too
        row_w_all = engine.softmax_weights(st.row_l_all, coef)
        row_w = row_w_all[off:off + n]
    col_m = st.col_m
    col_w = engine.softmax_weights(st.col_l, coef) if st.symmetric else torch.zeros_like(st.col_l)
    diag_w = 1.0 / n_glob
    kw = {"scale_dev": st.scale_dev} if st.scale_dev is not None else {}

    # one GPU, plain symmetric loss: both sides from ONE sweep over the logits tiles where the engine serves the shape
    # (8 N^2 d executed per step instead of 10; csrc/kernels_pair2.cuh)
    both = getattr(engine, "backward_both", None)
    if (both is not None and st.xchg is None and st.symmetric and st.y is st.b_c and st.xa is st.a_c and not st.want_t
            and st.a.dtype == st.b.dtype and (grad_dtype_a or st.a.dtype) == (grad_dtype_b or st.b.dtype)
            and st.compute_dtype == torch.bfloat16 and engine.backward_both_bytes(n, n, st.a_c.shape[1], st.compute_dtype,
                                                                                  st.scale, st.flags) > 0):
        da, db, ds = both(st.a_c, st.b_c, st.rinv_a, st.rinv_b, st.scale, st.row_m, row_w, col_m, col_w, diag_w, st.a, st.b,
                          grad_dtype_a or st.a.dtype, grad_scale, st.flags, want_dscale=True, **kw)
        return da, db, ds

    if st.both_sharded:
        # row-sharded: ONE kernel sweeps local A rows x all columns, emits dA and stores every owner's partial dB straight
        # into its slot over NVLink peer memory (contraction + reduce-scatter); after the barrier the owner finishes dA from
        # the sweep's slabs and dB from its slots
        x = st.xchg
        engine.backward_both_sharded_sweep(st.a_c, st.y, st.rinv_a, st.rinv_y, off, st.scale, st.row_m, row_w, col_m, col_w,
                                           diag_w, x.peers, x.world, x.rank, x.o_slots, st.flags, **kw)
        x.barrier(_exchange.PHASE_GRADS)
        da, db, ds = engine.finish_sharded(st.a_c, st.a, st.rinv_a, st.b_c, st.b, st.rinv_b, x.slots, n_glob, st.scale, x.world,
                                           grad_dtype_a or st.a.dtype, grad_dtype_b or st.b.dtype, grad_scale, st.flags)
        ds = x.sum_scalars(ds, _exchange.PHASE_CLOSE)
        x.release()
        st.xchg = None
        return da, db, ds

    # side A: local rows of A x all columns -> dA (normalise backward fused into the tail) and sum G.S over the local
    # row block
    da, ds = engine.backward_dx(st.a_c, st.y, st.y_t, st.rinv_a, st.rinv_y, off, st.scale, st.row_m, row_w, col_m, col_w,
                                diag_w, st.a, grad_dtype_a or st.a.dtype, grad_scale, st.flags, want_dscale=True, **kw)
    # side B: local rows of B (the positive-carrying columns of this rank) x ALL rows of A -> dB, complete as well:
    # the column statistics of the local block play the row role, the gathered row statistics the column role
    xa_t = None
    if st.want_t:
        _, xa_t = engine.stage(st.xa, st.compute_dtype, want_t=True)
    db, _ = engine.backward_dx(st.b_c, st.xa, xa_t, st.rinv_b, st.rinv_xa, off, st.scale,
                               col_m[off:off + n].contiguous(), col_w[off:off + n].contiguous(),
                               st.row_m_all, row_w_all, diag_w, st.b, grad_dtype_b or st.b.dtype, grad_scale, st.flags,
                               want_dscale=False, **kw)
    if st.xchg is not None:   # sum over the ranks' row blocks; as a barrier it also closes the step (exchange.py)
        ds = st.xchg.sum_scalars(ds, _exchange.PHASE_CLOSE)
        st.xchg.release()
        st.xchg = None
    return da, db, ds
