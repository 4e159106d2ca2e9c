"""The exchange steps of the row-sharded global batch (SURVEY.md section 8e), in two implementations of one interface.

What the reference does with ``dist.all_gather`` x2 + ``torch.cat`` (old/clip_opt.py:102-112, run1/full.py:77-84) is here

    gather_cols       every rank's B rows (+ 1/norm)  -> all columns  [N,d]        before the forward sweep
    gather_rows       every rank's A rows (+ 1/norm)  -> all rows     [N,d]        needed by the backward only: side B is
                      "local B rows x all A rows", complete per rank -- no [N,d] fp32 partial, no reduce-scatter
    exchange_stats    partial column (shift, sum) pairs of the ranks' row blocks -> global; row pairs -> gathered
    sum_scalars       the scalar loss; sum G.S for d logit_scale (also the closing barrier of the step)

`PeerExchange` (the product path on GPUs): kernels of this repository that store straight into the peers' HBM over
NVLink / NVSwitch (csrc/kernels_link.cuh, include/clipnce.h "clipnce_link_*"); torch symmetric memory only provides the
mapping of every rank's buffer into every process.  The normalise is fused into the gather kernel, the A rows travel
on a side stream beside the forward sweep (copy engines: the sweep keeps every SM), statistics and scalars are one-kernel pushes with a device-side barrier;
epochs live on the device, so the step replays inside a CUDA graph.
`CollectiveExchange`: the same steps as torch.distributed collectives -- the gloo CPU tests, and the NCCL baseline the
peer path is measured against (``CLIPNCE_COMM=nccl`` or ``bench.py --comm nccl``).
"""
from __future__ import annotations

import ctypes
import importlib
import os
import warnings

import torch
import torch.distributed as dist

PHASE_COLS, PHASE_STATS, PHASE_LOSS, PHASE_CLOSE, PHASE_GRADS, PHASE_BLOCKS = 0, 1, 2, 3, 4, 5
# The B rows travel BESIDE the forward sweep (copy engines + per-block flags, PeerExchange.gather_cols_beside) where the
# forward kernel can wait block by block and the sweep is long enough to hide the delivery chain (world - 1 blocks, each
# two copy-engine transfers and a flag kernel, ~25 us per block): measured on 8 GPUs, 8192 local rows x 65536 columns x 512
# gain 4.4 % of the step, 4096 local rows x 32768 x 768 (a 190 us sweep) lose 8 %.  Below this the push kernel + barrier
# run in front of the sweep.  CLIPNCE_GATHER_BESIDE_MIN_ROWS: test hook.
GATHER_BESIDE_MIN_ROWS = int(os.environ.get("CLIPNCE_GATHER_BESIDE_MIN_ROWS", "8192"))


def _all_gather(x, group):
    world = dist.get_world_size(group)
    out = torch.empty((world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    if dist.get_backend(group) == "gloo" and x.dtype == torch.bfloat16:
        tmp = torch.empty(out.shape, dtype=torch.float32, device=x.device)
        dist.all_gather_into_tensor(tmp, x.float().contiguous(), group=group)
        return tmp.to(x.dtype)
    dist.all_gather_into_tensor(out, x.contiguous(), group=group)
    return out


class CollectiveExchange:
    """The exchange as torch.distributed collectives (gloo on CPU, NCCL on GPUs)."""

    kind = "collectives"

    def __init__(self, engine, group):
        self.engine, self.group = engine, group
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self._rows = None

    def gather_cols(self, b, compute_dtype):
        rinv_b, _ = self.engine.normalize(b)
        b_c, _ = self.engine.stage(b, compute_dtype)
        y = _all_gather(b_c, self.group)
        if b.dtype == compute_dtype:
            rinv_y, _ = self.engine.normalize(y)   # same kernel on the same rows as on their owner: identical values
        else:   # norms were taken on the caller's (wider) rows before staging: ship them
            rinv_y = _all_gather(rinv_b, self.group)
        return b_c, rinv_b, y, rinv_y

    def gather_rows_begin(self, a, a_c, rinv_a, compute_dtype):
        xa = _all_gather(a_c, self.group)
        self._rows = (xa, _all_gather(rinv_a, self.group))

    def gather_rows_end(self):
        rows, self._rows = self._rows, None
        return rows

    def exchange_stats(self, row_m, row_l, col_m, col_l, fixed_shift, need_rows):
        g = self.group
        # Always the general (shift, sum) combine: `fixed_shift` is derived from a host-side, possibly stale copy of the
        # logit scale (functional._ScaleHint), so ranks may briefly disagree on it while s crosses the kernel-family
        # threshold -- and ranks that disagree must still issue the SAME collectives.
        m_max = col_m.clone()
        dist.all_reduce(m_max, op=dist.ReduceOp.MAX, group=g)
        col_l = col_l * torch.exp(col_m - m_max)
        dist.all_reduce(col_l, op=dist.ReduceOp.SUM, group=g)
        col_m = m_max
        if not need_rows:
            return col_m, col_l, None, None
        return col_m, col_l, _all_gather(row_m, g), _all_gather(row_l, g)

    def sum_scalars(self, vals, phase):
        out = vals.clone()
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=self.group)
        return out

    generation = 0

    def owned_by(self, generation) -> bool:
        return True

    def release(self):
        self._rows = None


class PeerExchange:
    """One set of symmetric buffers for a step of fixed shape; leased from `_Pool` for the life of the step (its gathered
    matrices are what the backward reads) and returned by `release()`.

    Protocol (every rank issues the same sequence; phases are device-side barriers with their own epoch counters):
        push B rows -> barrier 0 -> [forward sweep | A rows by the copy engines on the side stream] -> push statistics
        -> barrier 1
        -> ... -> sum_scalars(loss) = barrier 2 -> [backward] -> sum_scalars(d scale) = barrier 3.
    A rank passes barrier 3 (or 2 in a step without backward) only after every peer finished reading this step's
    buffers, so the next step may overwrite them without any further synchronisation.
    """

    kind = "nvlink-peer"

    def __init__(self, engine, group, n_local, d, n_cols, compute_dtype, device, pool_key):
        import torch.distributed._symmetric_memory as symm_mem
        self.engine, self.group, self.pool_key = engine, group, pool_key
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.n, self.d, self.n_cols, self.dtype = n_local, d, n_cols, compute_dtype
        self.N = n_local * self.world
        esz = 2 if compute_dtype == torch.bfloat16 else 4
        control, self.status_off = engine.link_layout()
        off = control

        def region(nbytes):
            nonlocal off
            o = off
            off = (off + nbytes + 255) // 256 * 256
            return o

        self.o_y = region(self.N * d * esz)
        self.o_xa = region(self.N * d * esz)
        self.o_rinv_y = region(self.N * 4)
        self.o_rinv_xa = region(self.N * 4)
        self.o_colm = region(self.world * n_cols * 4)
        self.o_coll = region(self.world * n_cols * 4)
        self.o_rowm = region(self.N * 4)
        self.o_rowl = region(self.N * 4)
        # partial dB_hat slots of the two-sided backward: rank q stores its contribution to MY columns into slot q
        self.o_slots = region(self.world * n_local * d * 4)
        self.nbytes = off
        self.buf = symm_mem.empty(self.nbytes, dtype=torch.uint8, device=device)
        self.buf.zero_()
        torch.cuda.synchronize(device)
        # every rank has zeroed its control block before any peer holds a mapping of it
        self.handle = symm_mem.rendezvous(self.buf, group.group_name)
        ptrs = [int(p) for p in self.handle.buffer_ptrs]
        if len(ptrs) != self.world or ptrs[self.rank] != self.buf.data_ptr():
            raise RuntimeError("symmetric memory rendezvous returned an unexpected mapping")
        self.peers = (ctypes.c_void_p * self.world)(*ptrs)
        # high priority: the A rows' push shares the GPU with the forward sweep, whose CTAs fill every SM -- its blocks
        # must win the SM slots that free up after the sweep's first wave instead of queueing behind its last one
        self.side = torch.cuda.Stream(device=device, priority=-1)
        self._side_busy = False
        self.generation = 0     # bumped at every lease: a step remembers the generation it was given

        def view(o, count, dt):
            e = 2 if dt == torch.bfloat16 else 4
            return self.buf[o:o + count * e].view(dt)

        self.y = view(self.o_y, self.N * d, compute_dtype).view(self.N, d)
        self.xa = view(self.o_xa, self.N * d, compute_dtype).view(self.N, d)
        self.rinv_y = view(self.o_rinv_y, self.N, torch.float32)
        self.rinv_xa = view(self.o_rinv_xa, self.N, torch.float32)
        self.colm = view(self.o_colm, self.world * n_cols, torch.float32)
        self.coll = view(self.o_coll, self.world * n_cols, torch.float32)
        self.rowm = view(self.o_rowm, self.N, torch.float32)
        self.rowl = view(self.o_rowl, self.N, torch.float32)
        self.slots = view(self.o_slots, self.world * n_local * d, torch.float32)
        self.status = self.buf[self.status_off:self.status_off + 4].view(torch.int32)

    # ---------------------------------------------------------------- the exchange steps
    def gather_cols(self, b, compute_dtype):
        e, lo = self.engine, self.rank * self.n
        e.link_push_rows(b, compute_dtype, self.peers, self.world, self.rank, self.o_y, self.o_rinv_y, lo)
        e.link_barrier(self.peers, self.world, self.rank, PHASE_COLS)
        return self.y[lo:lo + self.n], self.rinv_y[lo:lo + self.n], self.y, self.rinv_y

    def gather_cols_beside(self, b, rinv_b):
        """The gather of the columns for `engine.forward_gathered`: own block copied locally, every peer's copy of it
        delivered by the copy engines on the side stream, flagged block by block.  b [n,d] in the compute type."""
        e, lo = self.engine, self.rank * self.n
        esz = b.element_size()
        if rinv_b is None:
            rinv_b, _ = e.normalize(b)
        self.y[lo:lo + self.n].copy_(b, non_blocking=True)
        self.rinv_y[lo:lo + self.n].copy_(rinv_b, non_blocking=True)
        e.link_epoch_advance(self.peers, self.world, self.rank, PHASE_BLOCKS)
        cur = torch.cuda.current_stream()
        self.side.wait_stream(cur)
        with torch.cuda.stream(self.side):
            e.link_send_blocks(b, rinv_b, self.peers, self.world, self.rank, self.o_y + lo * self.d * esz,
                               self.o_rinv_y + lo * 4, PHASE_BLOCKS)
        self._side_busy = True              # joined before the step's next barrier (exchange_stats)
        return b, rinv_b, self.y, self.rinv_y

    def gather_rows_begin(self, a, a_c, rinv_a, compute_dtype):
        cur = torch.cuda.current_stream()
        self.side.wait_stream(cur)          # behind barrier 0: the columns have the links to themselves
        lo = self.rank * self.n
        # the rows already exist in the compute type (a_c) and their norms too: nothing to compute, so the copy engines
        # move them and the forward sweep keeps every SM (a push kernel beside the sweep takes CTA-pair slots from it and
        # part of an extra wave: a full-grid push 365 -> 435 us on 8 GPUs, 8 blocks of 1024 threads +20 us on 8, +80 us on
        # 2 and 4 GPUs)
        esz = a_c.element_size()
        with torch.cuda.stream(self.side):
            self.engine.link_copy(a_c, self.peers, self.world, self.rank, self.o_xa + lo * self.d * esz)
            self.engine.link_copy(rinv_a, self.peers, self.world, self.rank, self.o_rinv_xa + lo * 4)
        self._side_busy = True

    def gather_rows_end(self):
        return self.xa, self.rinv_xa

    def exchange_stats(self, row_m, row_l, col_m, col_l, fixed_shift, need_rows):
        e, r = self.engine, self.rank
        srcs = [col_m, col_l]
        offs = [self.o_colm + 4 * r * self.n_cols, self.o_coll + 4 * r * self.n_cols]
        if need_rows:
            srcs += [row_m, row_l]
            offs += [self.o_rowm + 4 * r * self.n, self.o_rowl + 4 * r * self.n]
        e.link_push_f32(srcs, offs, self.peers, self.world, r)
        if self._side_busy:                 # the A rows must have left before this rank arrives at the barrier
            torch.cuda.current_stream().wait_stream(self.side)
            self._side_busy = False
        e.link_barrier(self.peers, self.world, r, PHASE_STATS)
        cm, cl = e.combine_partials(self.colm, self.coll, self.world, self.n_cols, self.n_cols)
        return cm, cl, (self.rowm if need_rows else None), (self.rowl if need_rows else None)

    def sum_scalars(self, vals, phase):
        return self.engine.link_sum_scalars(vals, self.peers, self.world, self.rank, phase)

    def barrier(self, phase):
        self.engine.link_barrier(self.peers, self.world, self.rank, phase)

    def owned_by(self, generation) -> bool:
        """False once the buffers were reclaimed for a later step (see _Pool.lease)."""
        return self.generation == generation

    def check(self):
        """Host check of the status word (synchronises): raises if a barrier timed out.  A timeout also traps on the
        device (kernels_link.cuh), so in practice the synchronisation inside this read raises first."""
        code = int(self.status[0])
        if code != 0:
            raise RuntimeError(f"clip_dplm_b200: peer exchange barrier phase {code - 1} timed out (a rank did not arrive)")

    def release(self):
        _Pool.give_back(self)


class _Pool:
    """Leases of `PeerExchange` buffers keyed by (group, shape, dtype).  Allocation is a host-side collective
    (rendezvous), so leases are taken and returned at deterministic points of the step only (never from a finaliser):
    a forward whose autograd graph is dropped without a backward keeps its lease until `reset()`."""

    free = {}
    live = {}          # key -> exchanges out on lease, oldest first
    n_alloc = {}
    max_per_key = 8
    mode = {}          # group name -> "link" | "nccl"

    @classmethod
    def decide(cls, engine, group, device) -> str:
        name = group.group_name
        if name in cls.mode:
            return cls.mode[name]
        want = os.environ.get("CLIPNCE_COMM", "").lower()
        ok = 1
        if want in ("nccl", "collectives") or device.type != "cuda" or dist.get_backend(group) == "gloo":
            ok = 0
        elif dist.get_world_size(group) > 16 or not hasattr(engine, "link_push_rows"):
            ok = 0
        else:
            try:
                importlib.import_module("torch.distributed._symmetric_memory")
            except Exception:
                ok = 0
        if device.type == "cuda" and dist.get_backend(group) != "gloo":
            flag = torch.tensor([ok], dtype=torch.int32, device=device)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
            ok = int(flag.item())
        cls.mode[name] = "link" if ok else "nccl"
        return cls.mode[name]

    @classmethod
    def lease(cls, engine, group, n_local, d, n_cols, compute_dtype, device):
        key = (group.group_name, n_local, d, n_cols, compute_dtype, device)
        fl = cls.free.setdefault(key, [])
        lv = cls.live.setdefault(key, [])
        if not fl and cls.n_alloc.get(key, 0) >= cls.max_per_key and lv:
            # Every buffer is out on lease: forwards whose backward never ran (an evaluation loop under enable_grad).
            # Reclaim the OLDEST lease -- the same one on every rank, since all ranks run the same sequence of steps; a
            # backward that still turns up for it finds a newer generation and raises (PeerExchange.owned_by).
            x = lv.pop(0)
            x.generation += 1
            fl.append(x)
        if fl:
            x = fl.pop()
            x.generation += 1
            lv.append(x)
            return x
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("clip_dplm_b200: run one eager step of this shape before capturing a CUDA graph (the peer "
                               "exchange buffers are allocated by a host-side rendezvous)")
        if cls.n_alloc.get(key, 0) >= cls.max_per_key:
            raise RuntimeError("clip_dplm_b200: too many live row-sharded steps of one shape (forward passes whose backward "
                               "never ran keep their exchange buffers); call clip_dplm_b200.exchange.reset()")
        ok, x, err = 1, None, None
        try:
            x = PeerExchange(engine, group, n_local, d, n_cols, compute_dtype, device, key)
        except Exception as ex:   # no multi-GPU fabric mapping on this box: fall back TOGETHER to the NCCL collectives
            ok, err = 0, ex
        flag = torch.tensor([ok], dtype=torch.int32, device=device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag.item()) == 0:
            if os.environ.get("CLIPNCE_COMM", "").lower() == "link":
                raise RuntimeError(f"clip_dplm_b200: CLIPNCE_COMM=link but the peer exchange could not be set up: {err}")
            warnings.warn(f"clip_dplm_b200: peer-memory exchange unavailable ({err}); using NCCL collectives")
            cls.mode[group.group_name] = "nccl"
            return None
        cls.n_alloc[key] = cls.n_alloc.get(key, 0) + 1
        x.generation += 1
        lv.append(x)
        return x

    @classmethod
    def give_back(cls, x):
        lv = cls.live.get(x.pool_key, [])
        if x in lv:
            lv.remove(x)
            cls.free.setdefault(x.pool_key, []).append(x)


def reset():
    """Forget every cached exchange buffer (call on all ranks; before destroying the process group)."""
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    _Pool.free.clear()
    _Pool.live.clear()
    _Pool.n_alloc.clear()
    _Pool.mode.clear()


def open_exchange(engine, group, n_local, d, n_cols, compute_dtype, device):
    """The exchange object of one step: a leased `PeerExchange` on NVLink-connected GPUs, else `CollectiveExchange`."""
    if _Pool.decide(engine, group, device) == "link":
        x = _Pool.lease(engine, group, n_local, d, n_cols, compute_dtype, device)
        if x is not None:
            return x
    return CollectiveExchange(engine, group)


def comm_kind(group) -> str:
    return _Pool.mode.get(group.group_name, "undecided")
