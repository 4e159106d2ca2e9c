"""CPU suite (`pytest -m "not gpu"`): oracle vs golden fixtures, closed-form identities, host logic
through a CPU stand-in engine (incl. world_size-2 gloo), and the C-ABI surface (load + exports only --
no compute call is made without a GPU)."""
import ctypes
import glob
import json
import math
import os
import re

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ref_step as O
from tests.cpu_engine import TorchCpuEngine

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLDEN = sorted(glob.glob(os.path.join(HERE, "golden", "*.npz")))


def rel(x, ref):
    x, ref = torch.as_tensor(x).double(), torch.as_tensor(ref).double()
    return float((x - ref).norm() / ref.norm().clamp_min(1e-300))


def from_bits(bits):
    return torch.from_numpy(bits.astype(np.int16)).view(torch.bfloat16)


# ------------------------------------------------------------------------------------------------ oracle
def test_oracle_is_pinned_to_reference():
    pinned = json.load(open(os.path.join(HERE, "golden", "PINNED.json")))
    checks = pinned["checks"]
    for key in ("old/clip.py forward tail", "rna_clip_codes.ipynb RNARBPCLIPModel loss", "old/clip_opt.py optimized_clip_loss"):
        assert checks[key] == "exact"
    assert checks["param count 71,646,299"] == "reproduced"
    assert len(GOLDEN) >= 8


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_oracle_reproduces_golden(path):
    z = np.load(path)
    a, b = from_bits(z["a_bits"]).float(), from_bits(z["b_bits"]).float()
    kw = json.loads(str(z["meta"]))
    if "extra_bits" in z:
        kw["extra_cols"] = from_bits(z["extra_bits"]).float()
    ls = float(z["logit_scale"])
    r64 = O.ref_step(a.double(), b.double(), ls, **{k: (v.double() if torch.is_tensor(v) else v) for k, v in kw.items()})
    assert abs(float(r64["loss"]) - float(z["loss64"])) <= 1e-12 * max(1.0, abs(float(z["loss64"])))
    rows = z["grad_rows"] if "grad_rows" in z else slice(None)     # larger fixtures store a sample of gradient rows
    assert rel(r64["d_a"].float()[rows], z["d_a64"]) < 1e-6 and rel(r64["d_b"].float()[rows], z["d_b64"]) < 1e-6
    r32 = O.ref_step(a, b, ls, **kw)
    assert abs(float(r32["loss"]) - float(z["loss32"])) <= 2e-6 * max(1.0, abs(float(z["loss32"])))


@pytest.mark.parametrize("symmetric", [True, False])
def test_closed_form_matches_autograd(symmetric):
    a, b = O.make_inputs(96, 40, seed=5)
    s = 1 / 0.07
    cf = O.closed_form(a.numpy(), b.numpy(), s, symmetric=symmetric)
    ref = O.ref_step(a.double(), b.double(), math.log(s), symmetric=symmetric)
    assert abs(cf["loss"] - float(ref["loss"])) < 1e-12
    assert rel(cf["d_a"], ref["d_a"]) < 1e-12 and rel(cf["d_b"], ref["d_b"]) < 1e-12
    assert abs(cf["d_scale_sum"] - float(ref["d_logit_scale"])) < 1e-12


def test_known_answers():
    # untrained model, batch 32: loss ~ ln 32 (rna_clip_codes.ipynb:2333 records 3.5013 at s = 14.3 on real data)
    a, b = O.make_inputs(32, 512, seed=7, correlated=False)
    assert abs(float(O.ref_loss(a, b, torch.tensor(0.0))) - math.log(32)) < 0.05
    # perfectly aligned pairs: loss -> log(1 + (N-1) exp(-s (1 - cos)))  with cos ~ 0 off the diagonal
    n, s = 64, 5.0
    a = torch.eye(n, 128)
    l = float(O.ref_loss(a, a.clone(), torch.tensor(math.log(s))))
    assert abs(l - math.log(1 + (n - 1) * math.exp(-s))) < 1e-6


# ------------------------------------------------------------------------------------------------ C-ABI surface
def test_library_exports_every_declared_symbol():
    from clip_dplm_b200 import _lib
    header = open(os.path.join(ROOT, "include", "clipnce.h")).read()
    declared = set(re.findall(r"\b(clipnce_[a-z0-9_]+)\s*\(", header))
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.clipnce_version() == 110


def test_host_only_entry_points():
    from clip_dplm_b200 import _lib
    lib = _lib.load()
    nbytes = ctypes.c_size_t(0)
    assert lib.clipnce_workspace_bytes(65536, 65536, 512, _lib.BF16, 0, ctypes.byref(nbytes)) == 0
    assert nbytes.value >= 2 * 1024 * 65536 * 4          # [2 x 1024 row blocks][65536] fp32 column partials
    assert lib.clipnce_workspace_bytes(0, 10, 512, _lib.BF16, 0, ctypes.byref(nbytes)) == -1
    assert b"bad shape" in lib.clipnce_last_error()
    assert lib.clipnce_uses_tensor_cores(_lib.BF16, 512, 14.3, 0) == 1
    assert lib.clipnce_uses_tensor_cores(_lib.BF16, 512, 100.0, 0) == 2      # exp(S - s) would leave fp32: true running maxima
    assert lib.clipnce_uses_tensor_cores(_lib.BF16, 512, 14.3, _lib.FLAG_UNBOUNDED) == 2
    assert lib.clipnce_uses_tensor_cores(_lib.BF16, 192, 100.0, 0) == 0      # family 2 lives in the CTA-pair kernels (d % 128)
    assert lib.clipnce_uses_tensor_cores(_lib.F32, 512, 14.3, 0) == 0        # check mode
    assert lib.clipnce_uses_tensor_cores(_lib.BF16, 516, 14.3, 0) == 0       # d % 8
    assert lib.clipnce_uses_tensor_cores(_lib.BF16, 512, 14.3, _lib.FLAG_FORCE_EXACT) == 0


def test_group_and_gathered_host_entry_points():
    """Host-side answers of the entry points added for the grouped launch (tri-modal model, small batches) and for the
    gather beside the forward sweep: which shapes are served, argument validation -- no GPU involved."""
    from clip_dplm_b200 import _lib
    lib = _lib.load()
    nb = ctypes.c_size_t(7)
    # three pairs over three members, N = 4096, d = 512: served by both tensor-core families
    for s in (14.3, 100.0):
        assert lib.clipnce_group_workspace_bytes(3, 3, 4096, 512, _lib.BF16, s, 0, ctypes.byref(nb)) == 0
        assert nb.value >= 6 * 4096 * 512 * 4              # one split's gradient slabs of the six backward sides
    # not served: fp32 (check mode), d % 128 != 0, un-normalised columns -> 0 bytes, the caller issues the pairs one by one
    for dt, d, fl in ((_lib.F32, 512, 0), (_lib.BF16, 192, 0), (_lib.BF16, 512, _lib.FLAG_UNBOUNDED)):
        assert lib.clipnce_group_workspace_bytes(3, 3, 4096, d, dt, 14.3, fl, ctypes.byref(nb)) == 0 and nb.value == 0
    assert lib.clipnce_group_workspace_bytes(5, 3, 4096, 512, _lib.BF16, 14.3, 0, ctypes.byref(nb)) == -1   # > 4 members
    assert lib.clipnce_group_workspace_bytes(3, 5, 4096, 512, _lib.BF16, 14.3, 0, ctypes.byref(nb)) == -1   # > 4 problems
    # the gathered forward is a function of type, d and flags only (every rank of a step must answer alike)
    assert lib.clipnce_forward_gathered_ok(_lib.BF16, 512, 14.3, 0) == 1
    assert lib.clipnce_forward_gathered_ok(_lib.BF16, 512, 100.0, 0) == 1
    assert lib.clipnce_forward_gathered_ok(_lib.BF16, 512, 500.0, 0) == 1
    assert lib.clipnce_forward_gathered_ok(_lib.BF16, 512, 14.3, _lib.FLAG_UNBOUNDED) == 0
    assert lib.clipnce_forward_gathered_ok(_lib.BF16, 192, 14.3, 0) == 0
    assert lib.clipnce_forward_gathered_ok(_lib.F32, 512, 14.3, 0) == 0
    # the two-sided backward answers 0 bytes below 12288 rows (host-only part of the plan; the device check comes after)
    assert lib.clipnce_backward_both_workspace_bytes(8192, 8192, 512, _lib.BF16, 14.3, 0, 0, ctypes.byref(nb)) == 0 and nb.value == 0


def test_grouped_loss_declines_what_it_does_not_serve():
    """functional.fused_clip_loss_group returns None (the caller then issues pair steps) for CPU tensors, mixed shapes,
    and when CLIPNCE_NO_GROUP is set -- it never falls back to a CPU computation."""
    from clip_dplm_b200.functional import fused_clip_loss_group
    a, b = O.make_inputs(16, 64)
    assert fused_clip_loss_group((a, b), (0,), (1,), 2.0) is None
    assert fused_clip_loss_group((a, b[:8]), (0,), (1,), 2.0) is None


def test_source_hash_of_the_build_changes_with_the_sources(tmp_path):
    from clip_dplm_b200 import _lib
    f1, f2 = tmp_path / "a.cu", tmp_path / "b.cuh"
    f1.write_text("int x;")
    f2.write_text("int y;")
    h0 = _lib._source_hash([str(f1), str(f2)])
    assert h0 == _lib._source_hash([str(f2), str(f1)])      # order of discovery does not matter
    f2.write_text("int y; ")
    assert _lib._source_hash([str(f1), str(f2)]) != h0
    assert os.path.exists(_lib.LIB_PATH + ".srchash") or os.path.exists(_lib.LIB_PATH)


def test_product_path_refuses_cpu_tensors():
    from clip_dplm_b200 import fused_clip_loss
    a, b = O.make_inputs(16, 64)
    with pytest.raises(RuntimeError, match="CUDA"):
        fused_clip_loss(a, b, 2.0)


# ------------------------------------------------------------------------------------------------ host logic
CASES = [({}, 0), ({"symmetric": False}, 0), ({"clamp_max": 100.0, "ls": 5.0, "mix": 0.12}, 0),
         ({"scale_is_log": False, "ls": 10.0, "symmetric": False}, 0), ({}, 40), ({"symmetric": False}, 24)]


@pytest.mark.parametrize("kw,n_extra", CASES)
def test_step_logic_matches_oracle(kw, n_extra):
    from clip_dplm_b200 import fused_clip_loss
    kw = dict(kw)
    ls = kw.pop("ls", O.LOGIT_SCALE_INIT)
    a, b = O.make_inputs(100, 48, n_cols=100 + n_extra, mix=kw.pop("mix", 0.5))
    extra = None
    if n_extra:
        extra = torch.nn.functional.normalize(b[100:].double(), dim=-1)
        b = b[:100]
    okw = dict(kw, **({"extra_cols": extra} if extra is not None else {}))
    ref = O.ref_step(a.double(), b.double(), ls, **okw)
    ac, bc = a.double().requires_grad_(True), b.double().requires_grad_(True)
    t = torch.tensor(ls, dtype=torch.float64, requires_grad=True)
    loss = fused_clip_loss(ac, bc, t, engine=TorchCpuEngine(), compute_dtype=torch.float64, extra_cols=extra, **kw)
    (2.5 * loss).backward()                     # a non-trivial upstream gradient
    assert abs(float(loss.detach()) - float(ref["loss"])) < 1e-12
    assert rel(ac.grad / 2.5, ref["d_a"]) < 1e-9 and rel(bc.grad / 2.5, ref["d_b"]) < 1e-9
    assert abs(float(t.grad) / 2.5 - float(ref["d_logit_scale"])) < 1e-9


def _gloo_worker(rank, world, port, n, d, symmetric, n_extra, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from clip_dplm_b200 import fused_clip_loss
        torch.set_num_threads(1)
        a, b = O.make_inputs(n, d, n_cols=n + n_extra, seed=21)
        extra = torch.nn.functional.normalize(b[n:].double(), dim=-1) if n_extra else None
        nl = n // world
        ac = a[rank * nl:(rank + 1) * nl].double().requires_grad_(True)
        bc = b[rank * nl:(rank + 1) * nl].double().requires_grad_(True)
        t = torch.tensor(O.LOGIT_SCALE_INIT, dtype=torch.float64, requires_grad=True)
        loss = fused_clip_loss(ac, bc, t, engine=TorchCpuEngine(), compute_dtype=torch.float64, group=dist.group.WORLD,
                               symmetric=symmetric, extra_cols=extra)
        loss.backward()
        from clip_dplm_b200 import exchange
        assert exchange.comm_kind(dist.group.WORLD) == "nccl"      # CPU tensors over gloo: the collectives implementation
        with torch.no_grad():                                       # evaluation: no rows gathered for a backward
            le = fused_clip_loss(ac, bc, t, engine=TorchCpuEngine(), compute_dtype=torch.float64, group=dist.group.WORLD,
                                 symmetric=symmetric, extra_cols=extra)
        assert abs(float(le) - float(loss.detach())) < 1e-12
        q.put((rank, float(loss.detach()), ac.grad.numpy(), bc.grad.numpy(), float(t.grad)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("symmetric,n_extra", [(True, 0), (False, 0), (True, 24)])
def test_row_sharded_global_batch_gloo(symmetric, n_extra):
    """world_size 2 over gloo: global negatives (plus shared hard-negative cache columns), exact gradients -- side B of the
    backward runs on the gathered rows -- compared with the single-process reference on the concatenated batch
    (SURVEY.md section 8e)."""
    world, n, d = 2, 96, 32
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, world, port, n, d, symmetric, n_extra, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = sorted([q.get(timeout=120) for _ in range(world)], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    a, b = O.make_inputs(n, d, n_cols=n + n_extra, seed=21)
    okw = {"extra_cols": torch.nn.functional.normalize(b[n:].double(), dim=-1)} if n_extra else {}
    ref = O.ref_step(a.double(), b[:n].double(), O.LOGIT_SCALE_INIT, symmetric=symmetric, **okw)
    nl = n // world
    for rank, loss, da, db, dt in out:
        assert abs(loss - float(ref["loss"])) < 1e-12
        assert rel(da, ref["d_a"][rank * nl:(rank + 1) * nl]) < 1e-9
        assert rel(db, ref["d_b"][rank * nl:(rank + 1) * nl]) < 1e-9
        assert abs(dt - float(ref["d_logit_scale"])) < 1e-9


# ------------------------------------------------------------------------------------------------ retrieval (top-k)
def test_ref_topk_is_the_reference_evaluation_tail():
    """oracle.ref_topk == the reference's own forms: F.cosine_similarity(a.unsqueeze(1), b.unsqueeze(0), dim=2)
    (run1/full.py:157) ranked by topk, and logits.argmax(dim=1) (run1/full.py:152) for k = 1."""
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(3)
    q, lib = torch.randn(37, 24, generator=g, dtype=torch.float64), torch.randn(91, 24, generator=g, dtype=torch.float64)
    s, i, sim = O.ref_topk(q, lib, 5)
    sim_ref = F.cosine_similarity(q.unsqueeze(1), lib.unsqueeze(0), dim=2)
    assert torch.allclose(sim, sim_ref, atol=1e-12)
    s2, i2 = torch.topk(sim_ref, 5, dim=1)
    assert torch.equal(i, i2) and torch.allclose(s, s2, atol=1e-12)
    logits = 14.3 * (F.normalize(q, dim=-1) @ F.normalize(lib, dim=-1).t())
    assert torch.equal(O.ref_topk(q, lib, 1)[1][:, 0], logits.argmax(dim=1))


def _gloo_topk_worker(rank, world, port, n_q, n_lib, d, k, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from clip_dplm_b200.retrieval import topk_similarity
        torch.set_num_threads(1)
        g = torch.Generator().manual_seed(5)
        qs, lib = torch.randn(n_q, d, generator=g, dtype=torch.float64), torch.randn(n_lib, d, generator=g, dtype=torch.float64)
        nl = n_lib // world
        s, i = topk_similarity(qs, lib[rank * nl:(rank + 1) * nl], k, group=dist.group.WORLD, engine=TorchCpuEngine())
        q.put((rank, s.numpy(), i.numpy()))
    finally:
        dist.destroy_process_group()


def test_sharded_retrieval_gloo():
    """Library row-sharded over 2 ranks (BASELINE config 5 layout): per-shard top-k with global indices, candidates
    all-gathered and merged -- must equal the single-process oracle on the whole library."""
    world, n_q, n_lib, d, k = 2, 19, 64, 16, 5
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_topk_worker, args=(r, world, port, n_q, n_lib, d, k, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = sorted([q.get(timeout=120) for _ in range(world)], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    g = torch.Generator().manual_seed(5)
    qs, lib = torch.randn(n_q, d, generator=g, dtype=torch.float64), torch.randn(n_lib, d, generator=g, dtype=torch.float64)
    s_ref, i_ref, _ = O.ref_topk(qs, lib, k)
    for rank, s, i in out:
        assert np.array_equal(i, i_ref.numpy()) and np.allclose(s, s_ref.numpy(), atol=1e-6)


# ------------------------------------------------------------------------------------------------ drop-in surface
REFERENCE = os.environ.get("CLIP_DPLM_REFERENCE")
REFERENCE_CLIP = os.path.join(REFERENCE, "old", "clip.py") if REFERENCE else ""


@pytest.mark.skipif(not os.path.isfile(REFERENCE_CLIP),
                    reason="needs a checkout of the reference project named by CLIP_DPLM_REFERENCE")
def test_module_parameter_names_match_reference():
    """state_dicts of the reference modules must load into the drop-in modules (same names and shapes)."""
    import importlib.util
    import sys
    import types
    stub = types.ModuleType("configuration_hybrid_clip")
    stub.HybridCLIPConfig = object
    sys.modules.setdefault("configuration_hybrid_clip", stub)
    spec = importlib.util.spec_from_file_location("ref_old_clip_t", REFERENCE_CLIP)
    ref = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref)
    from clip_dplm_b200 import modules as M
    sub = lambda h: types.SimpleNamespace(hidden_size=h, num_hidden_layers=2, layer_norm_eps=1e-5)
    cfg = types.SimpleNamespace(rna_config=sub(24), protein_config=sub(32), diffmap_config=sub(24), projection_dim=16,
                                logit_scale_init_value=2.6592, cache_size=8)
    for name in ("RNAProteinCLIPModule", "DiffMapProteinCLIPModule"):
        a = {k: tuple(v.shape) for k, v in getattr(ref, name)(cfg).state_dict().items()}
        b = {k: tuple(v.shape) for k, v in getattr(M, name)(cfg).state_dict().items()}
        assert a == b, name


@pytest.mark.parametrize("symmetric", [True, False])
def test_sampled_oracle_matches_closed_form(symmetric):
    """oracle/sampled.py (blockwise statistics + float64 gradient rows of a sample; what bench.py's `parity` key and the
    large-shape GPU tests compare with) against the dense closed form on a size where both fit."""
    from oracle import sampled as SO
    n, d, s = 300, 64, 14.2857
    a, b = O.make_inputs(n, d, seed=5)
    cf = O.closed_form(a.numpy(), b.numpy(), s, symmetric=symmetric)
    rows_a, rows_b = np.array([0, 7, 150, 299]), np.array([3, 299, 42])
    ref = SO.sampled_reference(a, b, s, rows_a, rows_b, chunk=128, symmetric=symmetric)
    assert abs(ref["loss"] - cf["loss"]) <= 1e-6 * abs(cf["loss"])
    assert np.allclose(ref["row_lse"], cf["row_lse"], atol=2e-5)
    assert np.allclose(ref["col_lse"], cf["col_lse"], atol=2e-5)
    assert np.allclose(ref["diag"], cf["diag"], atol=1e-9)
    assert abs(ref["d_scale_sum"] - cf["d_scale_sum"]) <= 1e-4 * abs(cf["d_scale_sum"])
    assert rel(ref["d_a"], cf["d_a"][rows_a]) <= 1e-4   # the blockwise LSEs come from an fp32 GEMM
    assert rel(ref["d_b"], cf["d_b"][rows_b]) <= 1e-4
    cmp = SO.compare(ref, cf["loss"], cf["d_a"][rows_a], cf["d_b"][rows_b], cf["d_scale_sum"])
    assert cmp["ok"] and cmp["rows"] == 4


# ------------------------------------------------------------------------------------------------ DDP convention
class _TinyTwoTower(torch.nn.Module):
    def __init__(self, d_in, d):
        super().__init__()
        g = torch.Generator().manual_seed(4)
        self.wa = torch.nn.Parameter(torch.randn(d_in, d, generator=g, dtype=torch.float64) * 0.3)
        self.wb = torch.nn.Parameter(torch.randn(d_in, d, generator=g, dtype=torch.float64) * 0.3)
        self.logit_scale = torch.nn.Parameter(torch.tensor(O.LOGIT_SCALE_INIT, dtype=torch.float64))

    def forward(self, xa, xb, group=None, ddp=False):
        from clip_dplm_b200 import fused_clip_loss
        return fused_clip_loss(xa @ self.wa, xb @ self.wb, self.logit_scale, engine=TorchCpuEngine(),
                               compute_dtype=torch.float64, group=group, ddp=ddp)


def _ddp_worker(rank, world, port, n, d_in, d, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from torch.nn.parallel import DistributedDataParallel as DDP
        torch.set_num_threads(1)
        g = torch.Generator().manual_seed(8)
        xa, xb = torch.randn(n, d_in, generator=g, dtype=torch.float64), torch.randn(n, d_in, generator=g, dtype=torch.float64)
        nl = n // world
        model = DDP(_TinyTwoTower(d_in, d))
        loss = model(xa[rank * nl:(rank + 1) * nl], xb[rank * nl:(rank + 1) * nl], group=dist.group.WORLD, ddp=True)
        loss.backward()                                   # DDP averages every parameter gradient over the ranks
        m = model.module
        q.put((rank, float(loss.detach()), m.wa.grad.numpy(), m.wb.grad.numpy(), float(m.logit_scale.grad)))
    finally:
        dist.destroy_process_group()


def test_ddp_parameter_gradients_match_single_process():
    """Under DistributedDataParallel (how the reference runs old/clip_opt.py:154, run1/full.py:172) EVERY parameter --
    tower weights and logit_scale alike -- must come out of DDP's gradient averaging with the gradient of the global
    mean loss of a single-process run on the whole batch (`fused_clip_loss(..., ddp=True)`)."""
    world, n, d_in, d = 2, 64, 12, 16
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 25500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_ddp_worker, args=(r, world, port, n, d_in, d, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = sorted([q.get(timeout=120) for _ in range(world)], key=lambda x: x[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    g = torch.Generator().manual_seed(8)
    xa, xb = torch.randn(n, d_in, generator=g, dtype=torch.float64), torch.randn(n, d_in, generator=g, dtype=torch.float64)
    ref = _TinyTwoTower(d_in, d)
    loss = O.ref_loss(xa @ ref.wa, xb @ ref.wb, ref.logit_scale)
    loss.backward()
    for rank, l, gwa, gwb, gt in out:
        assert abs(l - float(loss.detach())) < 1e-12
        assert rel(gwa, ref.wa.grad) < 1e-9 and rel(gwb, ref.wb.grad) < 1e-9
        assert abs(gt - float(ref.logit_scale.grad)) < 1e-9 * max(1.0, abs(float(ref.logit_scale.grad)))
