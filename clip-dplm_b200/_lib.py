"""ctypes binding of the C-ABI library (include/clipnce.h).

The library is built in-tree (``clip-dplm_b200/csrc/libclipnce.so``) by ``build()`` /
``make -C clip-dplm_b200/csrc``.  There is NO fallback: if the library is missing or a call fails the
product path raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libclipnce.so")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "clipnce.h")

BF16, F32 = 0, 1
FLAG_FORCE_EXACT = 1
FLAG_UNBOUNDED = 2

_lock = threading.Lock()
_lib = None

_vp, _i64, _f32, _int, _sz = ctypes.c_void_p, ctypes.c_int64, ctypes.c_float, ctypes.c_int, ctypes.c_size_t

# name -> argtypes (restype is int unless listed in _RESTYPES); mirrors include/clipnce.h one to one
SIGNATURES = {
    "clipnce_version": [],
    "clipnce_last_error": [],
    "clipnce_uses_tensor_cores": [_int, _i64, _f32, _int],
    "clipnce_needs_transposed": [_int, _i64, _f32, _int],
    "clipnce_workspace_bytes": [_i64, _i64, _i64, _int, _int, ctypes.POINTER(_sz)],
    "clipnce_normalize": [_vp, _int, _i64, _i64, _vp, _vp, _int, _vp],
    "clipnce_stage_operand": [_vp, _int, _i64, _i64, _vp, _vp, _i64, _int, _vp],
    "clipnce_forward": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _f32, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp, _vp,
                        _sz, _vp],
    "clipnce_backward": [_vp, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _f32, _f32,
                         _int, _int, _vp, _vp, _vp, _sz, _vp],
    "clipnce_backward_dx": [_vp, _vp, _vp, _i64, _vp, _vp, _i64, _i64, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _f32,
                            _int, _int, _vp, _int, _vp, _vp, _int, _vp, _vp, _sz, _vp],
    "clipnce_backward_both_workspace_bytes": [_i64, _i64, _i64, _int, _f32, _int, _int, ctypes.POINTER(_sz)],
    "clipnce_backward_both_sharded": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _f32, _int, _int,
                                      ctypes.POINTER(_vp), _int, _int, _i64, _vp, _sz, _vp],
    "clipnce_finish_sharded": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _f32, _int, _int, _int, _int,
                               _int, _int, _vp, _vp, _vp, _sz, _vp],
    "clipnce_backward_both_dx": [_vp, _vp, _vp, _vp, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp, _f32, _int, _int, _vp, _vp,
                                 _int, _vp, _vp, _vp, _int, _vp, _vp, _sz, _vp],
    "clipnce_group_workspace_bytes": [_int, _int, _i64, _i64, _int, _f32, _int, ctypes.POINTER(_sz)],
    "clipnce_group_forward": [_vp, _vp, _int, _int, ctypes.POINTER(_int), ctypes.POINTER(_int), _i64, _i64, _f32, _vp, _int,
                              _int, _vp, _vp, _vp, _vp, _vp, _sz, _vp],
    "clipnce_group_backward": [_vp, _vp, _int, _int, ctypes.POINTER(_int), ctypes.POINTER(_int), _i64, _i64, _f32, _vp, _vp,
                               _vp, _int, _int, _vp, _int, _vp, _vp, _int, _vp, _vp, _vp, _sz, _vp],
    "clipnce_head_tail": [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _f32, _vp, _vp, _vp, _vp, _vp],
    "clipnce_head_tail_backward": [_vp, _int, _vp, _vp, _vp, _i64, _i64, _vp, _vp],
    "clipnce_softmax_weights": [_vp, _i64, _f32, _vp, _vp],
    "clipnce_combine_lse": [_vp, _vp, _i64, _vp, _vp],
    "clipnce_normalize_backward": [_vp, _int, _vp, _vp, _vp, _i64, _i64, _vp, _int, _vp],
    "clipnce_topk_workspace_bytes": [_i64, _i64, _i64, _int, _int, ctypes.POINTER(_sz)],
    "clipnce_topk": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _int, _int, _vp, _vp, _vp, _sz, _vp],
    "clipnce_loss": [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _vp, _vp],
    "clipnce_link_control_bytes": [ctypes.POINTER(_i64), ctypes.POINTER(_i64)],
    "clipnce_link_barrier": [ctypes.POINTER(_vp), _int, _int, _int, _vp],
    "clipnce_link_push_rows": [_vp, _int, _i64, _i64, _int, ctypes.POINTER(_vp), _int, _int, _i64, _i64, _i64, _vp],
    "clipnce_link_copy": [_vp, _sz, ctypes.POINTER(_vp), _int, _int, _i64, _vp],
    "clipnce_link_epoch_advance": [ctypes.POINTER(_vp), _int, _int, _int, _vp],
    "clipnce_link_send_blocks": [_vp, _sz, _vp, _sz, ctypes.POINTER(_vp), _int, _int, _i64, _i64, _int, _vp],
    "clipnce_forward_gathered_ok": [_int, _i64, _f32, _int],
    "clipnce_forward_gathered": [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _f32, _vp, _int, _int, _vp, _vp, _vp, _vp, _vp,
                                 ctypes.POINTER(_vp), _int, _int, _int, _vp, _sz, _vp],
    "clipnce_link_push_f32": [ctypes.POINTER(_vp), ctypes.POINTER(_i64), ctypes.POINTER(_i64), _int, ctypes.POINTER(_vp),
                              _int, _int, _vp],
    "clipnce_link_sum_scalars": [_vp, _int, ctypes.POINTER(_vp), _int, _int, _int, _vp, _vp],
    "clipnce_combine_partials": [_vp, _vp, _int, _i64, _i64, _vp, _vp, _vp],
}
_RESTYPES = {"clipnce_last_error": ctypes.c_char_p}


def _source_hash(files) -> str:
    import hashlib
    h = hashlib.sha256()
    for f in sorted(files):
        h.update(os.path.basename(f).encode())
        with open(f, "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile the CUDA library for sm_100a with nvcc (cross-compiles without a GPU).  The library is reused only when
    the hash of its sources, recorded next to it at build time, still matches (file times do not survive a checkout or
    the copy onto a GPU box); where nvcc is missing (a box that received a prebuilt library) the existing file is kept."""
    import shutil
    src_files = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))] + [HEADER]
    want = _source_hash(src_files)
    stamp = LIB_PATH + ".srchash"
    if not force and os.path.exists(LIB_PATH):
        have = open(stamp).read().strip() if os.path.exists(stamp) else None
        if have == want or (have is None and os.path.getmtime(LIB_PATH) >= max(os.path.getmtime(f) for f in src_files)):
            return LIB_PATH
        if shutil.which("nvcc") is None:
            raise RuntimeError("clip_dplm_b200: libclipnce.so was built from different sources and nvcc is not available")
    cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo", "-Xcompiler",
           "-fPIC", "-shared", "-diag-suppress", "177", "-o", LIB_PATH, os.path.join(CSRC, "clipnce_api.cu")]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(" ".join(cmd))
        print(res.stdout, res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building libclipnce.so:\n" + res.stderr)
    with open(stamp, "w") as fh:
        fh.write(want + "\n")
    return LIB_PATH


def load():
    """Load libclipnce.so (once) and attach the prototypes.  Raises if it is not built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"clip_dplm_b200: CUDA library not built ({LIB_PATH} missing). Run `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C clip-dplm_b200/csrc`. There is no CPU fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, argtypes in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError here == header/library mismatch
            fn.argtypes = argtypes
            fn.restype = _RESTYPES.get(name, ctypes.c_int)
        if lib.clipnce_version() != 110:
            raise RuntimeError("clip_dplm_b200: libclipnce.so version mismatch; rebuild")
        _lib = lib
        return lib


def check(rc: int, what: str):
    if rc != 0:
        msg = load().clipnce_last_error()
        raise RuntimeError(f"clipnce {what} failed (code {rc}): {msg.decode() if msg else ''}")
