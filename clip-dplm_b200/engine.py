"""CudaEngine: the C-ABI calls of include/clipnce.h on torch CUDA tensors.

torch is plumbing only (device memory, current stream).  Every method enqueues on the current CUDA
stream and returns freshly allocated (or cached-workspace) tensors; nothing synchronises the host.
"""
from __future__ import annotations

import ctypes

import torch

from . import _lib

_DT = {torch.bfloat16: _lib.BF16, torch.float32: _lib.F32}


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _guard(fn):
    """Run an engine method on the device of its tensor arguments: the C library launches on the CURRENT device and on
    the stream handed to it, so tensors on cuda:1 while cuda:0 is current would otherwise be worked on from the wrong
    device.  All tensor arguments must share one device."""
    import functools

    @functools.wraps(fn)
    def inner(self, *args, **kw):
        dev = None
        for t in list(args) + list(kw.values()):
            if torch.is_tensor(t) and t.is_cuda:
                if dev is None:
                    dev = t.device
                elif t.device != dev:
                    raise RuntimeError(f"clip_dplm_b200: tensors on different devices ({dev} and {t.device}) in one call")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(self, *args, **kw)
        with torch.cuda.device(dev):
            return fn(self, *args, **kw)
    return inner


def padded_ld(n: int) -> int:
    """Leading dimension of a transposed operand [d, ld]: rows stay 128-byte aligned for TMA."""
    return (n + 63) // 64 * 64


class CudaEngine:
    """One instance per process; caches the scratch workspace per shape and stream."""

    name = "cuda"

    def __init__(self):
        self.lib = _lib.load()
        self._ws = {}

    # ------------------------------------------------------------------ helpers
    @staticmethod
    def _chk(t, dtypes, what):
        if not t.is_cuda:
            raise RuntimeError(f"clip_dplm_b200: {what} must be a CUDA tensor (there is no CPU path)")
        if t.dtype not in dtypes:
            raise RuntimeError(f"clip_dplm_b200: {what} has unsupported dtype {t.dtype}")
        if not t.is_contiguous():
            raise RuntimeError(f"clip_dplm_b200: {what} must be contiguous")

    def uses_tensor_cores(self, dtype, d, scale, flags=0):
        return bool(self.lib.clipnce_uses_tensor_cores(_DT[dtype], d, float(scale), flags))

    def fixed_shift(self, dtype, d, scale, flags=0):
        """True when forward() returns col_m == row_m == scale (kernel family 1, the fixed shift): partial sums of
        different ranks then add up directly, no max exchange needed."""
        return self.lib.clipnce_uses_tensor_cores(_DT[dtype], d, float(scale), flags) == 1

    def needs_transposed(self, dtype, d, scale, flags=0):
        return bool(self.lib.clipnce_needs_transposed(_DT[dtype], d, float(scale), flags))

    def workspace(self, n_rows, n_cols, d, dtype, flags, device):
        key = (n_rows, n_cols, d, dtype, flags, device, torch.cuda.current_stream(device).cuda_stream)
        ws = self._ws.get(key)
        if ws is None:
            nbytes = ctypes.c_size_t(0)
            _lib.check(self.lib.clipnce_workspace_bytes(n_rows, n_cols, d, _DT[dtype], flags, ctypes.byref(nbytes)),
                       "workspace_bytes")
            ws = torch.empty(nbytes.value, dtype=torch.uint8, device=device)
            if len(self._ws) > 16:
                self._ws.clear()
            self._ws[key] = ws
        return ws

    # ------------------------------------------------------------------ stages
    @_guard
    def normalize(self, x, want_hat=None):
        """-> (rinv [n] f32, x_hat [n,d] in dtype `want_hat` or None)   (F.normalize, old/clip.py:63-64)"""
        self._chk(x, (torch.bfloat16, torch.float32), "embedding")
        n, d = x.shape
        rinv = torch.empty((n,), dtype=torch.float32, device=x.device)
        xh = torch.empty((n, d), dtype=want_hat, device=x.device) if want_hat is not None else None
        _lib.check(self.lib.clipnce_normalize(_p(x), _DT[x.dtype], n, d, _p(rinv), _p(xh),
                                              _DT[want_hat] if want_hat is not None else 0, _stream()), "normalize")
        return rinv, xh

    @_guard
    def stage(self, x, c_dtype, want_t=False):
        """-> (x_c [n,d] raw rows in the compute dtype (x itself when it already has it),
               x_c_t [d,ld] transposed copy or None)"""
        self._chk(x, (torch.bfloat16, torch.float32), "embedding")
        n, d = x.shape
        xc = x if x.dtype == c_dtype else torch.empty((n, d), dtype=c_dtype, device=x.device)
        xt, ld = None, 0
        if want_t:
            ld = padded_ld(n)
            xt = torch.empty((d, ld), dtype=c_dtype, device=x.device)
        if xc is not x or xt is not None:
            _lib.check(self.lib.clipnce_stage_operand(_p(x), _DT[x.dtype], n, d, _p(xc) if xc is not x else None, _p(xt),
                                                      ld, _DT[c_dtype], _stream()), "stage_operand")
        return xc, xt

    @_guard
    def forward(self, x, y, rinv_x, rinv_y, diag_offset, scale, flags=0, scale_dev=None):
        """-> row_m, row_l [n_rows], col_m, col_l [n_cols], diag [n_rows]   (LSE = m + log l, kept as pairs).
        ``scale_dev``: optional 1-element f32 CUDA tensor holding s; the kernels then read s on the device and the float
        ``scale`` only selects the kernel family."""
        self._chk(x, (torch.bfloat16, torch.float32), "x")
        self._chk(y, (x.dtype,), "y")
        n_rows, d = x.shape
        n_cols = y.shape[0]
        dev = x.device
        ws = self.workspace(n_rows, n_cols, d, x.dtype, flags, dev)
        row_m = torch.empty(n_rows, dtype=torch.float32, device=dev)
        row_l = torch.empty(n_rows, dtype=torch.float32, device=dev)
        col_m = torch.empty(n_cols, dtype=torch.float32, device=dev)
        col_l = torch.empty(n_cols, dtype=torch.float32, device=dev)
        diag = torch.empty(n_rows, dtype=torch.float32, device=dev)   # every row's positive column exists: all written
        _lib.check(self.lib.clipnce_forward(_p(x), _p(y), _p(rinv_x), _p(rinv_y), n_rows, n_cols, d, int(diag_offset),
                                            float(scale), _p(scale_dev), _DT[x.dtype], flags, _p(row_m), _p(row_l), _p(col_m),
                                            _p(col_l), _p(diag), _p(ws), ws.numel(), _stream()), "forward")
        return row_m, row_l, col_m, col_l, diag

    @_guard
    def backward(self, x, y, y_t, rinv_x, rinv_y, diag_offset, scale, row_m, row_w, col_m, col_w, diag_w, grad_out,
                 flags=0, want_dscale=True, scale_dev=None):
        """-> dx_hat [n_rows,d] f32, d_scale_sum [1] f32 (or None)"""
        n_rows, d = x.shape
        n_cols = y.shape[0]
        dev = x.device
        ws = self.workspace(n_rows, n_cols, d, x.dtype, flags, dev)
        dx = torch.empty((n_rows, d), dtype=torch.float32, device=dev)
        ds = torch.zeros(1, dtype=torch.float32, device=dev) if want_dscale else None
        ld_t = y_t.shape[1] if y_t is not None else 0
        _lib.check(self.lib.clipnce_backward(_p(x), _p(y), _p(y_t), ld_t, _p(rinv_x), _p(rinv_y), n_rows, n_cols, d,
                                             int(diag_offset), float(scale), _p(scale_dev), _p(row_m), _p(row_w), _p(col_m), _p(col_w),
                                             float(diag_w), float(grad_out), _DT[x.dtype], flags, _p(dx), _p(ds),
                                             _p(ws), ws.numel(), _stream()), "backward")
        return dx, ds

    @_guard
    def backward_dx(self, x, y, y_t, rinv_x, rinv_y, diag_offset, scale, row_m, row_w, col_m, col_w, diag_w, x_orig,
                    out_dtype, grad_scale=None, flags=0, want_dscale=True, scale_dev=None):
        """One backward side including the normalise backward -> dx [n_rows,d] in ``out_dtype`` (gradient of the caller's
        rows ``x_orig``), d_scale_sum [1] f32 (or None).  The fp32 gradient of the normalised rows stays in the workspace."""
        n_rows, d = x.shape
        n_cols = y.shape[0]
        dev = x.device
        self._chk(x_orig, (torch.bfloat16, torch.float32), "x_orig")
        ws = self.workspace(n_rows, n_cols, d, x.dtype, flags, dev)
        dx = torch.empty((n_rows, d), dtype=out_dtype, device=dev)
        ds = torch.zeros(1, dtype=torch.float32, device=dev) if want_dscale else None
        ld_t = y_t.shape[1] if y_t is not None else 0
        xo = x if x_orig.dtype == x.dtype else x_orig
        _lib.check(self.lib.clipnce_backward_dx(_p(x), _p(y), _p(y_t), ld_t, _p(rinv_x), _p(rinv_y), n_rows, n_cols, d,
                                                int(diag_offset), float(scale), _p(scale_dev), _p(row_m), _p(row_w),
                                                _p(col_m), _p(col_w), float(diag_w), _DT[x.dtype], flags, _p(xo),
                                                _DT[xo.dtype], _p(grad_scale), _p(dx), _DT[out_dtype], _p(ds), _p(ws),
                                                ws.numel(), _stream()), "backward_dx")
        return dx, ds

    def backward_both_bytes(self, n_rows, n_cols, d, dtype, scale, flags=0, world=0):
        """Workspace of the two-sided backward (one sweep over the logits tiles emits dA and dB) for [n_rows,d] x [n_cols,d];
        world = 0: one GPU, world >= 2: the row-sharded step.  0 = the shape is not served."""
        nbytes = ctypes.c_size_t(0)
        _lib.check(self.lib.clipnce_backward_both_workspace_bytes(n_rows, n_cols, d, _DT[dtype], float(scale), flags, world,
                                                                  ctypes.byref(nbytes)), "backward_both_workspace_bytes")
        return nbytes.value

    def _both_ws(self, n_rows, n_cols, d, dtype, scale, flags, world, dev):
        nbytes = self.backward_both_bytes(n_rows, n_cols, d, dtype, scale, flags, world)   # host-only; depends on the producer split
        if nbytes == 0:
            raise RuntimeError("clip_dplm_b200: the two-sided backward does not serve this shape")
        key = ("both", n_rows, n_cols, d, dtype, flags, world, dev, torch.cuda.current_stream(dev).cuda_stream)
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws[key] = ws
        return ws

    @_guard
    def backward_both(self, x, y, rinv_x, rinv_y, scale, row_m, row_w, col_m, col_w, diag_w, x_orig, y_orig, out_dtype,
                      grad_scale=None, flags=0, want_dscale=True, scale_dev=None):
        """Both backward sides of the single-GPU symmetric step in one sweep over the logits tiles (clipnce_backward_both_dx)
        -> dx, dy [n,d] in ``out_dtype`` (gradients of the caller's rows), d_scale_sum [1] f32 (or None)."""
        n, d = x.shape
        dev = x.device
        self._chk(x_orig, (torch.bfloat16, torch.float32), "x_orig")
        self._chk(y_orig, (x_orig.dtype,), "y_orig")
        ws = self._both_ws(n, n, d, x.dtype, scale, flags, 0, dev)
        dx = torch.empty((n, d), dtype=out_dtype, device=dev)
        dy = torch.empty((n, d), dtype=out_dtype, device=dev)
        ds = torch.zeros(1, dtype=torch.float32, device=dev) if want_dscale else None
        xo = x if x_orig.dtype == x.dtype else x_orig
        yo = y if y_orig.dtype == y.dtype else y_orig
        _lib.check(self.lib.clipnce_backward_both_dx(_p(x), _p(y), _p(rinv_x), _p(rinv_y), n, d, float(scale), _p(scale_dev),
                                                     _p(row_m), _p(row_w), _p(col_m), _p(col_w), float(diag_w), _DT[x.dtype],
                                                     flags, _p(xo), _p(yo), _DT[xo.dtype], _p(grad_scale), _p(dx), _p(dy),
                                                     _DT[out_dtype], _p(ds), _p(ws), ws.numel(), _stream()), "backward_both_dx")
        return dx, dy, ds

    @_guard
    def backward_both_sharded_sweep(self, x, y, rinv_x, rinv_y, diag_offset, scale, row_m, row_w, col_m, col_w, diag_w, peers,
                                    world, rank, slots_off, flags=0, scale_dev=None):
        """Row-sharded two-sided backward sweep (clipnce_backward_both_sharded): dA_hat stays in the workspace as segment
        slabs, the partial dB_hat of every owner rank is stored into its slot over NVLink peer memory; publish with a
        barrier, then finish both sides with `finish_sharded`."""
        n, d = x.shape
        n_cols = y.shape[0]
        ws = self._both_ws(n, n_cols, d, x.dtype, scale, flags, world, x.device)
        _lib.check(self.lib.clipnce_backward_both_sharded(_p(x), _p(y), _p(rinv_x), _p(rinv_y), n, n_cols, d, int(diag_offset),
                                                          float(scale), _p(scale_dev), _p(row_m), _p(row_w), _p(col_m), _p(col_w),
                                                          float(diag_w), _DT[x.dtype], flags, peers, world, rank, int(slots_off),
                                                          _p(ws), ws.numel(), _stream()), "backward_both_sharded")

    @_guard
    def finish_sharded(self, x, x_orig, rinv_x, y_local, y_orig, rinv_y_local, slots, n_cols, scale, world, out_dtype_x,
                       out_dtype_y, grad_scale=None, flags=0, want_dscale=True):
        """Both tails of the row-sharded two-sided backward -> dx [n,d] in ``out_dtype_x``, dy [n,d] in ``out_dtype_y``
        (gradients of the caller's rows x_orig / y_orig), d_scale_sum [1] f32 (or None).  One launch when both sides have
        the same types."""
        n, d = x.shape
        dev = x.device
        self._chk(x_orig, (torch.bfloat16, torch.float32), "x_orig")
        self._chk(y_orig, (torch.bfloat16, torch.float32), "y_orig")
        ws = self._both_ws(n, n_cols, d, x.dtype, scale, flags, world, dev)
        dx = torch.empty((n, d), dtype=out_dtype_x, device=dev)
        dy = torch.empty((n, d), dtype=out_dtype_y, device=dev)
        ds = torch.zeros(1, dtype=torch.float32, device=dev) if want_dscale else None
        xo = x if x_orig.dtype == x.dtype else x_orig
        yo = y_local if y_orig.dtype == y_local.dtype else y_orig
        _lib.check(self.lib.clipnce_finish_sharded(_p(x), _p(xo), _p(rinv_x), _p(dx), _p(y_local), _p(yo), _p(rinv_y_local), _p(dy),
                                                   _p(slots), n, n_cols, d, _DT[x.dtype], float(scale), flags, world, _DT[xo.dtype],
                                                   _DT[out_dtype_x], _DT[yo.dtype], _DT[out_dtype_y], _p(grad_scale), _p(ds),
                                                   _p(ws), ws.numel(), _stream()), "finish_sharded")
        return dx, dy, ds

    # ------------------------------------------------------------------ several pair problems in one launch
    def group_bytes(self, n_members, n_prob, n, d, dtype, scale, flags=0):
        """Workspace of `group_forward` / `group_backward`; 0 = the group is not served (issue the problems one by one)."""
        nbytes = ctypes.c_size_t(0)
        _lib.check(self.lib.clipnce_group_workspace_bytes(n_members, n_prob, n, d, _DT[dtype], float(scale), flags,
                                                          ctypes.byref(nbytes)), "group_workspace_bytes")
        return nbytes.value

    def _group_ws(self, n_members, n_prob, n, d, dtype, scale, flags, dev):
        nbytes = self.group_bytes(n_members, n_prob, n, d, dtype, scale, flags)
        if nbytes == 0:
            raise RuntimeError("clip_dplm_b200: the grouped launch does not serve this shape")
        key = ("group", n_members, n_prob, n, d, dtype, flags, dev, torch.cuda.current_stream(dev).cuda_stream)
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            self._ws[key] = ws
        return ws

    @staticmethod
    def _members(x_member, y_member):
        k = len(x_member)
        return (ctypes.c_int * k)(*x_member), (ctypes.c_int * k)(*y_member)

    @_guard
    def group_forward(self, stack, rinv, n_members, x_member, y_member, n, scale, flags=0, scale_dev=None):
        """Forward statistics and losses of len(x_member) pair problems over the members of ``stack`` [n_members*n_pad, d]
        (clipnce_group_forward) -> stat_m, stat_l [2, n_prob*n_pad], diag [n_prob*n_pad], loss [n_prob + 1]."""
        self._chk(stack, (torch.bfloat16,), "stack")
        d = stack.shape[1]
        n_prob = len(x_member)
        n_pad = stack.shape[0] // n_members
        dev = stack.device
        ws = self._group_ws(n_members, n_prob, n, d, stack.dtype, scale, flags, dev)
        stat_m = torch.empty((2, n_prob * n_pad), dtype=torch.float32, device=dev)
        stat_l = torch.empty((2, n_prob * n_pad), dtype=torch.float32, device=dev)
        diag = torch.empty(n_prob * n_pad, dtype=torch.float32, device=dev)
        loss = torch.empty(n_prob + 1, dtype=torch.float32, device=dev)
        xm, ym = self._members(x_member, y_member)
        _lib.check(self.lib.clipnce_group_forward(_p(stack), _p(rinv), n_members, n_prob, xm, ym, n, d, float(scale),
                                                  _p(scale_dev), _DT[stack.dtype], flags, _p(stat_m), _p(stat_l), _p(diag),
                                                  _p(loss), _p(ws), ws.numel(), _stream()), "group_forward")
        return stat_m, stat_l, diag, loss

    @_guard
    def group_backward(self, stack, rinv, n_members, x_member, y_member, n, scale, stat_m, stat_l, stack_orig, out_dtype,
                       grad_scale=None, flags=0, scale_dev=None, want_dscale=True, want_sumsq=True):
        """Both backward sides of every problem in one sweep launch + one finishing pass (clipnce_group_backward)
        -> d_stack [n_members*n_pad, d] in ``out_dtype``, d_scale_sum [1] or None, grad_sumsq [n_members] or None."""
        d = stack.shape[1]
        n_prob = len(x_member)
        dev = stack.device
        ws = self._group_ws(n_members, n_prob, n, d, stack.dtype, scale, flags, dev)
        d_stack = torch.zeros(stack.shape, dtype=out_dtype, device=dev) if n % 256 else \
            torch.empty(stack.shape, dtype=out_dtype, device=dev)
        ds = torch.zeros(1, dtype=torch.float32, device=dev) if want_dscale else None
        sq = torch.empty(n_members, dtype=torch.float32, device=dev) if want_sumsq else None
        so = stack if stack_orig.dtype == stack.dtype else stack_orig
        xm, ym = self._members(x_member, y_member)
        _lib.check(self.lib.clipnce_group_backward(_p(stack), _p(rinv), n_members, n_prob, xm, ym, n, d, float(scale),
                                                   _p(scale_dev), _p(stat_m), _p(stat_l), _DT[stack.dtype], flags, _p(so),
                                                   _DT[so.dtype], _p(grad_scale), _p(d_stack), _DT[out_dtype], _p(ds), _p(sq),
                                                   _p(ws), ws.numel(), _stream()), "group_backward")
        return d_stack, ds, sq

    @_guard
    def softmax_weights(self, l, coef):
        out = torch.empty_like(l)
        _lib.check(self.lib.clipnce_softmax_weights(_p(l), l.numel(), float(coef), _p(out), _stream()), "softmax_weights")
        return out

    @_guard
    def combine_lse(self, m, l):
        out = torch.empty_like(m)
        _lib.check(self.lib.clipnce_combine_lse(_p(m), _p(l), m.numel(), _p(out), _stream()), "combine_lse")
        return out

    @_guard
    def normalize_backward(self, x, rinv, dx_hat, out_dtype, grad_scale=None):
        n, d = x.shape
        dx = torch.empty((n, d), dtype=out_dtype, device=x.device)
        _lib.check(self.lib.clipnce_normalize_backward(_p(x), _DT[x.dtype], _p(rinv), _p(dx_hat), _p(grad_scale), n, d,
                                                       _p(dx), _DT[out_dtype], _stream()), "normalize_backward")
        return dx

    @_guard
    def topk(self, q, lib, rinv_q, rinv_lib, k, col_offset=0):
        """-> scores [n_q,k] f32 (descending), indices [n_q,k] i64 of the k most similar library rows per query
        (cosine similarity; run1/full.py:152,157).  bf16, d in {128,...,512}, k <= 16; raises otherwise."""
        self._chk(q, (torch.bfloat16,), "queries")
        self._chk(lib, (torch.bfloat16,), "library")
        n_q, d = q.shape
        n_lib = lib.shape[0]
        nbytes = ctypes.c_size_t(0)
        _lib.check(self.lib.clipnce_topk_workspace_bytes(n_q, n_lib, d, int(k), _DT[q.dtype], ctypes.byref(nbytes)),
                   "topk_workspace_bytes")
        ws = torch.empty(nbytes.value, dtype=torch.uint8, device=q.device)
        scores = torch.empty((n_q, k), dtype=torch.float32, device=q.device)
        idx = torch.empty((n_q, k), dtype=torch.int64, device=q.device)
        _lib.check(self.lib.clipnce_topk(_p(q), _p(lib), _p(rinv_q), _p(rinv_lib), n_q, n_lib, d, int(col_offset), int(k),
                                         _DT[q.dtype], _p(scores), _p(idx), _p(ws), ws.numel(), _stream()), "topk")
        return scores, idx

    # ------------------------------------------------------------------ exchange over NVLink peer memory
    def link_layout(self):
        """-> (control_bytes, status_offset) of the control block at the start of every symmetric buffer."""
        cb, so = ctypes.c_int64(0), ctypes.c_int64(0)
        _lib.check(self.lib.clipnce_link_control_bytes(ctypes.byref(cb), ctypes.byref(so)), "link_control_bytes")
        return cb.value, so.value

    def link_barrier(self, peers, world, rank, phase):
        _lib.check(self.lib.clipnce_link_barrier(peers, world, rank, phase, _stream()), "link_barrier")

    @_guard
    def link_push_rows(self, x, c_dtype, peers, world, rank, rows_off, rinv_off, row0):
        self._chk(x, (torch.bfloat16, torch.float32), "embedding")
        n, d = x.shape
        _lib.check(self.lib.clipnce_link_push_rows(_p(x), _DT[x.dtype], n, d, _DT[c_dtype], peers, world, rank, rows_off,
                                                   rinv_off, row0, _stream()), "link_push_rows")

    @_guard
    def link_copy(self, src, peers, world, rank, dst_off):
        """Copy-engine broadcast of a contiguous local tensor to byte offset ``dst_off`` of every rank's buffer."""
        self._chk(src, (torch.bfloat16, torch.float32), "rows")
        _lib.check(self.lib.clipnce_link_copy(_p(src), src.numel() * src.element_size(), peers, world, rank, dst_off,
                                              _stream()), "link_copy")

    def forward_gathered_ok(self, dtype, d, scale, flags=0):
        return bool(self.lib.clipnce_forward_gathered_ok(_DT[dtype], d, float(scale), flags))

    def link_epoch_advance(self, peers, world, rank, phase):
        _lib.check(self.lib.clipnce_link_epoch_advance(peers, world, rank, phase, _stream()), "link_epoch_advance")

    @_guard
    def link_send_blocks(self, rows, rinv, peers, world, rank, rows_off, rinv_off, phase):
        """Copy-engine delivery of this rank's rows / 1-norms to every peer, each followed by a flag (enqueue on a side
        stream behind `link_epoch_advance`)."""
        self._chk(rows, (torch.bfloat16, torch.float32), "rows")
        self._chk(rinv, (torch.float32,), "rinv")
        _lib.check(self.lib.clipnce_link_send_blocks(_p(rows), rows.numel() * rows.element_size(), _p(rinv), rinv.numel() * 4,
                                                     peers, world, rank, int(rows_off), int(rinv_off), phase, _stream()),
                   "link_send_blocks")

    @_guard
    def forward_gathered(self, x, y, rinv_x, rinv_y, scale, peers, world, rank, phase, flags=0, scale_dev=None):
        """`forward` over the gathered columns while their blocks are still arriving (clipnce_forward_gathered)."""
        self._chk(x, (torch.bfloat16,), "x")
        self._chk(y, (x.dtype,), "y")
        n_rows, d = x.shape
        n_cols = y.shape[0]
        dev = x.device
        ws = self.workspace(n_rows, n_cols, d, x.dtype, flags, dev)
        row_m = torch.empty(n_rows, dtype=torch.float32, device=dev)
        row_l = torch.empty(n_rows, dtype=torch.float32, device=dev)
        col_m = torch.empty(n_cols, dtype=torch.float32, device=dev)
        col_l = torch.empty(n_cols, dtype=torch.float32, device=dev)
        diag = torch.empty(n_rows, dtype=torch.float32, device=dev)
        _lib.check(self.lib.clipnce_forward_gathered(_p(x), _p(y), _p(rinv_x), _p(rinv_y), n_rows, n_cols, d, float(scale),
                                                     _p(scale_dev), _DT[x.dtype], flags, _p(row_m), _p(row_l), _p(col_m),
                                                     _p(col_l), _p(diag), peers, world, rank, phase, _p(ws), ws.numel(),
                                                     _stream()), "forward_gathered")
        return row_m, row_l, col_m, col_l, diag

    def link_push_f32(self, srcs, dst_offs, peers, world, rank):
        k = len(srcs)
        for t in srcs:
            self._chk(t, (torch.float32,), "statistics vector")
        src = (ctypes.c_void_p * k)(*[t.data_ptr() for t in srcs])
        n = (ctypes.c_int64 * k)(*[t.numel() for t in srcs])
        off = (ctypes.c_int64 * k)(*dst_offs)
        _lib.check(self.lib.clipnce_link_push_f32(src, n, off, k, peers, world, rank, _stream()), "link_push_f32")

    @_guard
    def link_sum_scalars(self, vals, peers, world, rank, phase):
        self._chk(vals, (torch.float32,), "scalars")
        out = torch.empty_like(vals)
        _lib.check(self.lib.clipnce_link_sum_scalars(_p(vals), vals.numel(), peers, world, rank, phase, _p(out), _stream()),
                   "link_sum_scalars")
        return out

    @_guard
    def combine_partials(self, part_m, part_l, n_part, ld, n):
        out_m = torch.empty(n, dtype=torch.float32, device=part_m.device)
        out_l = torch.empty(n, dtype=torch.float32, device=part_m.device)
        _lib.check(self.lib.clipnce_combine_partials(_p(part_m), _p(part_l), n_part, ld, n, _p(out_m), _p(out_l), _stream()),
                   "combine_partials")
        return out_m, out_l

    @_guard
    def loss(self, row_m, row_l, col_m, col_l, diag, diag_offset, n_global, symmetric):
        out = torch.empty(1, dtype=torch.float32, device=row_m.device)
        _lib.check(self.lib.clipnce_loss(_p(row_m), _p(row_l), _p(col_m), _p(col_l), _p(diag), row_m.numel(),
                                         int(diag_offset), int(n_global), int(bool(symmetric)), _p(out), _stream()),
                   "loss")
        return out


_engine = None


def default_engine() -> CudaEngine:
    global _engine
    if _engine is None:
        _engine = CudaEngine()
    return _engine
