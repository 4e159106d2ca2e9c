"""`fused_clip_loss`: the one public op of the hot path, as a torch.autograd.Function.

It replaces, in one call, the tail every reference model/loss shares
(F.normalize x2 -> exp(logit_scale) -> matmul * scale -> cross_entropy on S and S^T -> /2, and its
autograd backward; old/clip.py:63-67, current/rna_clip_codes.ipynb:1948-1953, run1/full.py:88-100,
old/clip_opt.py:130-151, tong/utils/losses.py:4-19).  Saved for backward: O(N d) only -- the N x N
logits never exist in HBM.
"""
from __future__ import annotations

import math
import weakref
from typing import Optional

import torch

from . import step as _step
from .engine import default_engine


def _scale_value(logit_scale, scale_is_log: bool, clamp_max: Optional[float]):
    """Host value of s and whether the clamp is active (python-float logit scales, and the first read of a parameter)."""
    t = float(logit_scale.detach()) if torch.is_tensor(logit_scale) else float(logit_scale)
    s = math.exp(t) if scale_is_log else t
    clamped = False
    if clamp_max is not None and s > clamp_max:
        s, clamped = float(clamp_max), True
    return t, s, clamped


class _ScaleHint:
    """Host-side, possibly stale copy of a device-resident s.  The kernels read s on the device (``scale_dev``); the host
    only needs its magnitude to pick the kernel family (tensor-core path while 2 s <= 86).  One blocking read the first
    time a parameter is seen; afterwards every step enqueues a non-blocking copy into pinned memory and picks up
    whichever earlier copy has completed -- no host synchronisation in the step (the reference's loop reads
    ``loss.item()`` every batch; this path does not even need that)."""

    _by_id = {}

    def __init__(self, tensor, s_dev):
        self.ref = weakref.ref(tensor)
        self.pinned = torch.empty(1, dtype=torch.float32).pin_memory()
        self.event = torch.cuda.Event()
        self.value = float(s_dev)          # the one blocking read
        self.pending = False

    @classmethod
    def get(cls, tensor, s_dev):
        h = cls._by_id.get(id(tensor))
        if torch.cuda.is_current_stream_capturing():
            # inside a CUDA-graph capture no event query / host read is legal: use the hint of the warm-up steps
            if h is None or h.ref() is not tensor:
                raise RuntimeError("fused_clip_loss: run at least one eager step with this logit_scale tensor before "
                                   "capturing a CUDA graph (the kernel family is chosen from its value)")
            return h.value
        if h is None or h.ref() is not tensor:
            if len(cls._by_id) > 64:
                cls._by_id = {k: v for k, v in cls._by_id.items() if v.ref() is not None}
            h = cls(tensor, s_dev)
            cls._by_id[id(tensor)] = h
        elif h.pending and h.event.query():
            h.value, h.pending = float(h.pinned[0]), False
        if not h.pending:
            h.pinned.copy_(s_dev, non_blocking=True)
            h.event.record()
            h.pending = True
        return h.value


FAMILY_SWITCH = 40.0      # include/clipnce.h: the fixed shift serves 2 s <= 80


def _agree_near_threshold(hint, group, device):
    """Every rank picks kernels -- and with them the exchange steps it issues -- from ITS copy of s, read at slightly
    different moments.  Far from the family switch all copies select the same kernels; within 12 % of it the ranks agree
    on the largest copy (one small blocking all-reduce per step, only while the scale crosses the switch)."""
    if group is None or abs(hint / FAMILY_SWITCH - 1.0) > 0.12 or torch.cuda.is_current_stream_capturing():
        return hint
    import torch.distributed as dist
    t = torch.tensor([hint], dtype=torch.float32, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def scale_family(logit_scale, scale_is_log, clamp_max, compute_dtype, d, flags, engine):
    """Kernel family (include/clipnce.h: 0 exact, 1 fixed shift, 2 true maxima) the NEXT step with this logit scale would
    select, from the host-side hint -- without a host synchronisation when the tensor has been seen before.  Used by
    `graph.GraphedClipStep` to notice that a captured graph froze a family the scale has since left."""
    if torch.is_tensor(logit_scale) and logit_scale.is_cuda:
        t_dev = logit_scale.detach().to(torch.float32).reshape(1)
        raw = t_dev.exp() if scale_is_log else t_dev.clone()
        s_dev = raw.clamp(max=float(clamp_max)) if clamp_max is not None else raw
        hint = _ScaleHint.get(logit_scale, s_dev) * 1.05
        s = min(hint, float(clamp_max)) if clamp_max is not None else hint
    else:
        s = _scale_value(logit_scale, scale_is_log, clamp_max)[1]
    return engine.lib.clipnce_uses_tensor_cores(_DT_CODE[compute_dtype], d, float(s), flags)


_DT_CODE = {torch.bfloat16: 0, torch.float32: 1}


class _FusedClipLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, logit_scale, extra, symmetric, scale_is_log, clamp_max, group, compute_dtype, flags, engine,
                want_stats=True, grad_mode=True, ddp=False, rinv_a=None, rinv_b=None):
        # grad_mode: autograd's mode at the call (always off inside forward()).  Without a backward to come the step
        # neither gathers the rows side B would stream nor keeps its exchange buffers (step.py)
        need_grad = grad_mode and (a.requires_grad or b.requires_grad or
                                   (torch.is_tensor(logit_scale) and logit_scale.requires_grad))
        info = {}
        s_dev = raw_dev = None
        if torch.is_tensor(logit_scale) and logit_scale.is_cuda:
            # s stays on the device: exp / clamp as two tiny kernels, read by the contraction kernels through scale_dev
            t_dev = logit_scale.detach().to(torch.float32).reshape(1)
            raw_dev = t_dev.exp() if scale_is_log else t_dev.clone()
            s_dev = raw_dev.clamp(max=float(clamp_max)) if clamp_max is not None else raw_dev
            hint = _ScaleHint.get(logit_scale, s_dev) * 1.05   # stale by a step or two at most: keep a margin
            hint = _agree_near_threshold(hint, group, logit_scale.device)
            scale_arg = min(hint, float(clamp_max)) if clamp_max is not None else hint
        else:
            def scale_arg():   # called by the step after the scale-independent kernels and the all-gather are enqueued
                info["v"] = _scale_value(logit_scale, scale_is_log, clamp_max)
                return info["v"][1]

        loss, st = _step.contrastive_forward(engine, a.detach().contiguous(), b.detach().contiguous(), scale_arg,
                                             symmetric=symmetric, extra=extra, group=group,
                                             compute_dtype=compute_dtype, flags=flags, need_grad=need_grad,
                                             scale_dev=s_dev, rinv_a=rinv_a, rinv_b=rinv_b)
        ctx.st, ctx.engine = st, engine
        # DistributedDataParallel AVERAGES parameter gradients over the ranks.  dA / dB are the exact gradient of the GLOBAL
        # mean loss with respect to the LOCAL rows (their sum over ranks is the parameter gradient), d logit_scale is the
        # full sum on every rank (its average is itself): under DDP the row gradients are therefore scaled by the world
        # size, so that every parameter comes out of DDP's mean with the gradient of the global loss.
        ctx.row_grad_mult = float(torch.distributed.get_world_size(group)) if (ddp and group is not None) else 1.0
        if s_dev is None:
            _, s, clamped = info["v"]
            ctx.scale_info = (s, clamped, scale_is_log, None, None, None)
        else:
            ctx.scale_info = (None, None, scale_is_log, s_dev, raw_dev, clamp_max)
        ctx.ls_meta = (logit_scale.dtype, logit_scale.device) if torch.is_tensor(logit_scale) else None
        if want_stats:
            row_lse = engine.combine_lse(st.row_m, st.row_l)
            col_lse = engine.combine_lse(st.col_m, st.col_l)
        else:   # two launches nobody reads
            row_lse = col_lse = st.diag
        ctx.mark_non_differentiable(row_lse, col_lse, st.diag)
        ctx.set_materialize_grads(False)   # no zero-filled "gradients" for the three statistics outputs (three launches)
        return loss.reshape(()), row_lse, col_lse, st.diag

    @staticmethod
    def backward(ctx, g_loss, _g1, _g2, _g3):
        st, engine = ctx.st, ctx.engine
        s, clamped, scale_is_log, s_dev, raw_dev, clamp_max = ctx.scale_info
        if g_loss is None:   # the loss did not take part in the differentiated graph
            if st.xchg is not None and st.xchg.owned_by(st.xchg_generation):   # close the step on every rank, hand the buffers back
                st.xchg.sum_scalars(torch.zeros(1, dtype=torch.float32, device=st.diag.device), _step._exchange.PHASE_CLOSE)
                st.xchg.release()
                st.xchg = None
            ctx.st = None
            return (None,) * 16
        g = g_loss.reshape(1).to(torch.float32).contiguous()
        g_rows = g * ctx.row_grad_mult if ctx.row_grad_mult != 1.0 else g
        da, db, ds = _step.contrastive_backward(engine, st, grad_scale=g_rows)
        d_ls = None
        if ctx.ls_meta is not None and ctx.needs_input_grad[2]:
            # sum G.S = dL/dt for s = exp(t);  dL/ds = sum G.S / s for a raw scale;  0 where the clamp is active
            if s_dev is not None:
                d = ds * g if scale_is_log else ds * g / s_dev
                if clamp_max is not None:
                    d = torch.where(raw_dev > float(clamp_max), torch.zeros_like(d), d)
                d_ls = d.reshape(()).to(dtype=ctx.ls_meta[0])
            elif clamped:
                d_ls = torch.zeros((), dtype=ctx.ls_meta[0], device=ctx.ls_meta[1])
            else:
                coef = 1.0 if scale_is_log else 1.0 / s
                d_ls = (ds * g * coef).reshape(()).to(device=ctx.ls_meta[1], dtype=ctx.ls_meta[0])
        ctx.st = None
        return da, db, d_ls, None, None, None, None, None, None, None, None, None, None, None, None, None


def fused_clip_loss(a, b, logit_scale, *, symmetric: bool = True, scale_is_log: bool = True,
                    clamp_max: Optional[float] = None, extra_cols=None, extra_normalized: bool = True,
                    group=None, compute_dtype: Optional[torch.dtype] = None, return_stats: bool = False,
                    ddp: bool = False, rinv_a=None, rinv_b=None, engine=None):
    """Fused CLIP / InfoNCE loss of two [N,d] embedding batches (un-normalised projection-head outputs).

    logit_scale   0-d tensor (learnable parameter) or float; ``s = exp(logit_scale)`` (scale_is_log) or
                  ``s = logit_scale`` (tong's ``1 / temperature``), optionally clamped (old/clip_opt.py:100).
    symmetric     (CE(S) + CE(S^T)) / 2 (rna_clip_codes.ipynb:1953) or CE(S) only (run1/full.py:133).
    extra_cols    [M,d] additional negative columns (hard-negative cache old/clip_opt.py:118-121, memory
                  queue tong/utils/losses.py:10-11), used as stored, no gradient.  ``extra_normalized=False``
                  (rows of arbitrary norm: logits no longer bounded by s) selects the kernels with true
                  running maxima.
    group         torch.distributed process group: rows are this rank's shard of a global batch; negatives
                  are global, gradients are exact (both sides complete on their owner), the returned loss is the global mean.
    ddp           with ``group``: the model producing ``a``/``b`` is wrapped in DistributedDataParallel (how the reference
                  runs old/clip_opt.py), which AVERAGES parameter gradients over ranks.  The row gradients are then scaled
                  by the world size, so that after DDP's mean every parameter -- encoders, heads and logit_scale alike --
                  holds the gradient of the global mean loss.  Default (False): dA/dB are the plain partial derivatives
                  of the global loss with respect to the local rows (sum them over ranks yourself).
    rinv_a/rinv_b [N] f32 1/max(|row|, 1e-12) of ``a`` / ``b`` when the producer of the rows already has them (the fused
                  projection-head tail, ``heads.fused_linear_layernorm``): the row-norm pass is skipped.
    compute_dtype torch.bfloat16 (tcgen05 tensor-core kernels) or torch.float32 (exact check mode).
                  Default: bf16 for bf16/fp16 inputs or under autocast, else fp32 (the reference's numerics).
    """
    engine = engine or default_engine()
    if a.dtype == torch.float16:
        a = a.to(torch.bfloat16)
    if b.dtype == torch.float16:
        b = b.to(torch.bfloat16)
    if compute_dtype is None:
        low = a.dtype == torch.bfloat16 or b.dtype == torch.bfloat16 or torch.is_autocast_enabled()
        compute_dtype = torch.bfloat16 if low else torch.float32
    flags = 0
    if extra_cols is not None and not extra_normalized:
        flags |= _step.FLAG_UNBOUNDED
    if (symmetric and extra_cols is None and group is None and not return_stats and compute_dtype == torch.bfloat16
            and a.is_cuda and a.shape == b.shape and a.dtype == b.dtype and not _no_group()):
        # small batches on one GPU (the reference trains at 32 ... 4096 rows): a pair's two backward sides are two sweeps of
        # <= 32 row blocks each on a GPU with 74 CTA-pair slots.  The grouped launch (DESIGN.md 5.10) runs them as the two
        # virtual problems of ONE sweep, with one finishing pass -- taken where the two-sided kernel does not serve the shape
        n, d = a.shape
        probe = 14.0 if (torch.is_tensor(logit_scale) and logit_scale.is_cuda) else _scale_value(logit_scale, scale_is_log, clamp_max)[1]
        both_bytes = getattr(engine, "backward_both_bytes", None)
        if n < GROUP_MAX_ROWS and both_bytes is not None and both_bytes(n, n, d, torch.bfloat16, probe, 0) == 0:
            losses = fused_clip_loss_group((a, b), (0,), (1,), logit_scale, scale_is_log=scale_is_log, clamp_max=clamp_max,
                                           engine=engine, autocast_ok=True)
            if losses is not None:
                return losses[0]
    loss, row_lse, col_lse, diag = _FusedClipLoss.apply(a, b, logit_scale, extra_cols, symmetric, scale_is_log,
                                                        clamp_max, group, compute_dtype, flags, engine, bool(return_stats),
                                                        torch.is_grad_enabled(), bool(ddp),
                                                        rinv_a.detach() if rinv_a is not None else None,
                                                        rinv_b.detach() if rinv_b is not None else None)
    if return_stats:
        return loss, {"row_lse": row_lse, "col_lse": col_lse, "diag": diag}
    return loss


# ------------------------------------------------------------------------------------------------------------------------
# several pair problems over shared members in one launch per kernel (the tri-modal model)
# ------------------------------------------------------------------------------------------------------------------------
def _no_group():
    import os
    return os.environ.get("CLIPNCE_NO_GROUP", "0") not in ("", "0")     # test hook: pair steps only


GROUP_MAX_ROWS = 8192     # measured (tools/bench_trimodal.py): 3.4x at N = 1024, 1.43x at 4096, 0.92x at 8192 against three pair steps


class _GroupedClipLoss(torch.autograd.Function):
    """losses[k] = symmetric InfoNCE of (members[x_member[k]], members[y_member[k]]), losses[-1] = their sum, all sharing
    one logit scale (tf_clip_codes (1).ipynb:13146-13165).  One normalise launch over the stacked members, one forward
    sweep, one backward sweep over both sides of every problem, one finishing pass (clipnce_group_*)."""

    @staticmethod
    def forward(ctx, logit_scale, scale_is_log, clamp_max, x_member, y_member, engine, holder, grad_mode, *members):
        n, d = members[0].shape
        n_members, n_prob = len(members), len(x_member)
        n_pad = (n + 255) // 256 * 256
        dev = members[0].device
        if n_pad == n:
            stack_orig = torch.cat([m.detach() for m in members], dim=0)
        else:
            stack_orig = torch.zeros((n_members * n_pad, d), dtype=members[0].dtype, device=dev)
            for i, m in enumerate(members):
                stack_orig[i * n_pad:i * n_pad + n] = m.detach()
        stack = stack_orig if stack_orig.dtype == torch.bfloat16 else stack_orig.to(torch.bfloat16)
        rinv, _ = engine.normalize(stack_orig)
        s_dev = raw_dev = None
        info = None
        if torch.is_tensor(logit_scale) and logit_scale.is_cuda:
            t_dev = logit_scale.detach().to(torch.float32).reshape(1)
            raw_dev = t_dev.exp() if scale_is_log else t_dev.clone()
            s_dev = raw_dev.clamp(max=float(clamp_max)) if clamp_max is not None else raw_dev
            hint = _ScaleHint.get(logit_scale, s_dev) * 1.05
            scale = min(hint, float(clamp_max)) if clamp_max is not None else hint
        else:
            info = _scale_value(logit_scale, scale_is_log, clamp_max)
            scale = info[1]
        kw = {"scale_dev": s_dev} if s_dev is not None else {}
        stat_m, stat_l, _diag, loss = engine.group_forward(stack, rinv, n_members, x_member, y_member, n, scale, **kw)
        need_grad = grad_mode and (any(m.requires_grad for m in members) or
                                   (torch.is_tensor(logit_scale) and logit_scale.requires_grad))
        if need_grad:
            ctx.saved = (stack, stack_orig, rinv, stat_m, stat_l, scale, s_dev, raw_dev, info)
        ctx.meta = (n, n_pad, n_members, tuple(x_member), tuple(y_member), scale_is_log, clamp_max, engine, holder,
                    (logit_scale.dtype, logit_scale.device) if torch.is_tensor(logit_scale) else None,
                    tuple(m.dtype for m in members))
        return loss

    @staticmethod
    def backward(ctx, g):
        n, n_pad, n_members, x_member, y_member, scale_is_log, clamp_max, engine, holder, ls_meta, dtypes = ctx.meta
        stack, stack_orig, rinv, stat_m, stat_l, scale, s_dev, raw_dev, info = ctx.saved
        ctx.saved = None
        n_prob = len(x_member)
        g = g.to(torch.float32)
        gs = (g[:n_prob] + g[n_prob]).contiguous()     # every problem's loss also feeds the sum
        kw = {"scale_dev": s_dev} if s_dev is not None else {}
        d_stack, ds, sq = engine.group_backward(stack, rinv, n_members, x_member, y_member, n, scale, stat_m, stat_l,
                                                stack_orig, stack_orig.dtype, grad_scale=gs, **kw)
        if holder is not None:
            holder["embed_grad_sumsq"] = sq
        d_ls = None
        if ls_meta is not None and ctx.needs_input_grad[0]:
            if s_dev is not None:     # ds already carries the upstream gradients
                dd = ds if scale_is_log else ds / s_dev
                if clamp_max is not None:
                    dd = torch.where(raw_dev > float(clamp_max), torch.zeros_like(dd), dd)
                d_ls = dd.reshape(()).to(dtype=ls_meta[0])
            elif info[2]:
                d_ls = torch.zeros((), dtype=ls_meta[0], device=ls_meta[1])
            else:
                d_ls = (ds * (1.0 if scale_is_log else 1.0 / info[1])).reshape(()).to(device=ls_meta[1], dtype=ls_meta[0])
        grads = tuple(d_stack[i * n_pad:i * n_pad + n] if ctx.needs_input_grad[8 + i] else None for i in range(n_members))
        return (d_ls, None, None, None, None, None, None, None) + grads


def fused_clip_loss_group(members, x_member, y_member, logit_scale, *, scale_is_log: bool = True,
                          clamp_max: Optional[float] = None, holder=None, engine=None, autocast_ok: bool = False):
    """Symmetric InfoNCE losses of several pairs over shared embeddings, one launch per kernel for the whole group.

    members     sequence of [N,d] CUDA embeddings of one dtype (bf16, or fp32/fp16 computed in bf16), un-normalised
    x_member / y_member   problem k pairs members[x_member[k]] (rows) with members[y_member[k]] (columns)
    Returns a [n_prob + 1] tensor (the problems' losses, then their sum), or ``None`` when the grouped launch does not
    serve the shapes (use one `fused_clip_loss` per pair).  ``holder`` (a dict) receives ``embed_grad_sumsq`` -- the
    squared gradient norm of every member, [n_members] f32 -- when the backward runs."""
    members = [m.to(torch.bfloat16) if m.dtype == torch.float16 else m for m in members]
    m0 = members[0]
    if m0.dim() != 2 or not m0.is_cuda:
        return None
    engine = engine or default_engine()
    if not hasattr(engine, "group_forward"):
        return None
    if any((not m.is_cuda) or m.shape != m0.shape or m.dtype != m0.dtype or m.device != m0.device for m in members):
        return None
    if m0.dtype not in (torch.bfloat16, torch.float32) or m0.shape[0] >= GROUP_MAX_ROWS:
        return None
    if _no_group():
        return None
    if m0.dtype == torch.float32 and not (autocast_ok or torch.is_autocast_enabled()):
        return None     # fp32 rows outside autocast are computed exactly (the reference's numerics): no tensor-core group
    n, d = m0.shape
    if torch.is_tensor(logit_scale) and logit_scale.is_cuda:
        probe = 14.0    # family 1 and 2 serve the same shapes: any positive scale answers "is the group served"
    else:
        probe = _scale_value(logit_scale, scale_is_log, clamp_max)[1]
    if engine.group_bytes(len(members), len(x_member), n, d, torch.bfloat16, probe, 0) == 0:
        return None
    return _GroupedClipLoss.apply(logit_scale, scale_is_log, clamp_max, list(x_member), list(y_member), engine, holder,
                                  torch.is_grad_enabled(), *members)
