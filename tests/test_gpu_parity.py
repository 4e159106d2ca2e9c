"""GPU parity tests (run with `pytest -m gpu` on a B200).

Everything goes through the C-ABI (clip_dplm_b200.engine.CudaEngine -> libclipnce.so) and is compared
with the CPU oracle (oracle/ref_step.py) and the committed golden fixtures (tests/golden/*.npz, which
were generated from the reference's own code by oracle/gen_golden.py).

Tolerances (BASELINE.json north_star): bf16 tensor-core path -- loss 1e-3 relative, embedding
gradients 2e-2 Frobenius-relative; fp32 check mode -- 1e-5, widened only to 3x the fp32 PyTorch
reference's own distance from the fp64 truth when that is larger (the reference is not exact either).
"""
import glob
import json
import math
import os

import numpy as np
import pytest
import torch

from oracle import ref_step as O

pytestmark = pytest.mark.gpu

GOLDEN = sorted(glob.glob(os.path.join(os.path.dirname(__file__), "golden", "*.npz")))
LOSS_RTOL_BF16, GRAD_RTOL_BF16, RTOL_F32 = 1e-3, 2e-2, 1e-5


def rel(x, ref):
    x = torch.as_tensor(x).double().cpu()
    ref = torch.as_tensor(ref).double().cpu()
    return float((x - ref).norm() / ref.norm().clamp_min(1e-300))


def from_bits(bits):
    return torch.from_numpy(bits.astype(np.int16)).view(torch.bfloat16)


@pytest.fixture(scope="module")
def eng():
    from clip_dplm_b200.engine import CudaEngine
    return CudaEngine()


def run_fused(a, b, ls, compute_dtype, **kw):
    from clip_dplm_b200 import fused_clip_loss
    in_dt = torch.bfloat16 if compute_dtype == torch.bfloat16 else torch.float32
    ac = a.cuda().to(in_dt).requires_grad_(True)
    bc = b.cuda().to(in_dt).requires_grad_(True)
    t = torch.tensor(float(ls), device="cuda", dtype=torch.float32, requires_grad=True)
    if "extra_cols" in kw:
        kw = dict(kw, extra_cols=kw["extra_cols"].cuda().to(in_dt))
    loss = fused_clip_loss(ac, bc, t, compute_dtype=compute_dtype, **kw)
    loss.backward()
    torch.cuda.synchronize()
    return float(loss.detach()), ac.grad.float().cpu(), bc.grad.float().cpu(), float(t.grad)


# ------------------------------------------------------------------------------------------------
# golden fixtures generated from the reference itself
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
@pytest.mark.parametrize("mode", ["bf16", "fp32"])
def test_golden(path, mode):
    z = np.load(path)
    a, b = from_bits(z["a_bits"]).float(), from_bits(z["b_bits"]).float()
    kw = json.loads(str(z["meta"]))
    if "extra_bits" in z:
        kw["extra_cols"] = from_bits(z["extra_bits"]).float()
    ls = float(z["logit_scale"])
    cd = torch.bfloat16 if mode == "bf16" else torch.float32
    loss, da, db, dt = run_fused(a, b, ls, cd, **kw)
    l64, da64, db64, dt64 = float(z["loss64"]), z["d_a64"], z["d_b64"], float(z["d_ls64"])
    if "grad_rows" in z:
        # the fixture stores a sample of the gradient rows: the whole matrices come from the float64 oracle, which must
        # reproduce the stored rows first
        r64 = O.ref_step(a.double(), b.double(), ls, **{k: (v.double() if torch.is_tensor(v) else v) for k, v in kw.items()})
        rows = z["grad_rows"]
        assert rel(r64["d_a"][rows], da64) < 1e-6 and rel(r64["d_b"][rows], db64) < 1e-6
        da64, db64 = r64["d_a"].float().numpy(), r64["d_b"].float().numpy()
    if mode == "bf16":
        assert abs(loss - l64) <= LOSS_RTOL_BF16 * abs(l64) + 1e-7
        assert rel(da, da64) <= GRAD_RTOL_BF16 and rel(db, db64) <= GRAD_RTOL_BF16
        assert abs(dt - dt64) <= 2e-2 * abs(dt64) + 1e-6
    else:
        # fp32 reference's own distance from fp64 on this fixture
        ref32 = O.ref_step(a, b, ls, **kw)
        own = max(rel(ref32["d_a"], da64), rel(ref32["d_b"], db64))
        tol = max(RTOL_F32, 3 * own)
        assert abs(loss - l64) <= RTOL_F32 * abs(l64) + 1e-7
        assert rel(da, da64) <= tol and rel(db, db64) <= tol, (rel(da, da64), rel(db, db64), own)
        assert abs(dt - dt64) <= 1e-4 * abs(dt64) + 1e-6


# ------------------------------------------------------------------------------------------------
# stage-level checks through the C-ABI against the float64 closed form
# ------------------------------------------------------------------------------------------------
SHAPES = [(128, 128, 64), (64, 64, 128), (256, 256, 512), (333, 333, 192), (1000, 1000, 512), (192, 192, 768),
          (200, 333, 128), (130, 70, 256), (1, 1, 64), (65, 129, 8)]


@pytest.mark.parametrize("n,m,d", SHAPES)
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_forward_stats(eng, n, m, d, dtype):
    scale = 1 / 0.07
    a, b = O.make_inputs(max(n, m), d, seed=7)
    a, b = a[:n], b[:m]
    if n > m:   # every row needs its positive column inside the matrix for the diagonal read
        a = a[:m]
        n = m
    cf = O.closed_form(a.numpy(), b.numpy(), scale)
    x, _ = eng.stage(a.cuda(), dtype)
    y, _ = eng.stage(b.cuda(), dtype)
    rx, _ = eng.normalize(x)
    ry, _ = eng.normalize(y)
    row_m, row_l, col_m, col_l, diag = eng.forward(x, y, rx, ry, 0, scale)
    torch.cuda.synchronize()
    row_lse = (row_m.double() + row_l.double().log()).cpu()
    col_lse = (col_m.double() + col_l.double().log()).cpu()
    assert eng.uses_tensor_cores(dtype, d, scale) == (dtype == torch.bfloat16)
    tol = 5e-6
    assert torch.allclose(row_lse, torch.from_numpy(cf["row_lse"]), rtol=0, atol=tol * 15)
    assert torch.allclose(col_lse, torch.from_numpy(cf["col_lse"]), rtol=0, atol=tol * 15)
    assert torch.allclose(diag.double().cpu(), torch.from_numpy(cf["diag"]), rtol=0, atol=tol * 15)
    assert rel(rx, cf["rinv_a"]) < 1e-6


@pytest.mark.parametrize("n,d,scale,corr", [(256, 128, 14.2857, True), (333, 192, 10.0, True), (512, 256, 10.0, False),
                                            (1000, 512, 14.2857, True), (192, 768, 30.0, True), (200, 64, 100.0, False)])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32])
def test_backward_sides(eng, n, d, scale, corr, dtype):
    a, b = O.make_inputs(n, d, seed=11, correlated=corr, mix=0.3)
    cf = O.closed_form(a.numpy(), b.numpy(), scale)
    tc = eng.uses_tensor_cores(dtype, d, scale)
    x, xt = eng.stage(a.cuda(), dtype, want_t=tc)
    y, yt = eng.stage(b.cuda(), dtype, want_t=tc)
    rx, _ = eng.normalize(x)
    ry, _ = eng.normalize(y)
    row_m, row_l, col_m, col_l, diag = eng.forward(x, y, rx, ry, 0, scale)
    coef = 1.0 / (2 * n)
    rw, cw = eng.softmax_weights(row_l, coef), eng.softmax_weights(col_l, coef)
    da, ds = eng.backward(x, y, yt, rx, ry, 0, scale, row_m, rw, col_m, cw, 1.0 / n, 1.0)
    db, _ = eng.backward(y, x, xt, ry, rx, 0, scale, col_m, cw, row_m, rw, 1.0 / n, 1.0, want_dscale=False)
    torch.cuda.synchronize()
    # fp32: 1 - p_ii is formed from fp32 logits (abs. rounding ~ s * 6e-8); at s = 30 that alone is ~2e-5 relative
    tol = GRAD_RTOL_BF16 if dtype == torch.bfloat16 else 5e-5
    assert rel(da, cf["d_a_hat"]) <= tol, rel(da, cf["d_a_hat"])
    assert rel(db, cf["d_b_hat"]) <= tol, rel(db, cf["d_b_hat"])
    assert abs(float(ds) - cf["d_scale_sum"]) <= (2e-2 if dtype == torch.bfloat16 else 1e-4) * abs(cf["d_scale_sum"]) + 1e-6


def test_row_shard_offsets(eng):
    """Row-sharded layout on one device: rank r's rows against all columns with diag_offset = r * n_local
    must reproduce the single-process statistics and gradients (SURVEY.md section 8e)."""
    n, d, world, scale = 384, 128, 3, 1 / 0.07
    a, b = O.make_inputs(n, d, seed=3)
    cf = O.closed_form(a.numpy(), b.numpy(), scale)
    y, yt = eng.stage(b.cuda().bfloat16(), torch.bfloat16, want_t=True)
    ry, _ = eng.normalize(y)
    nl = n // world
    col_parts, rows = [], []
    for r in range(world):
        x, _ = eng.stage(a[r * nl:(r + 1) * nl].cuda().bfloat16(), torch.bfloat16)
        rx, _ = eng.normalize(x)
        row_m, row_l, col_m, col_l, diag = eng.forward(x, y, rx, ry, r * nl, scale)
        rows.append((x, rx, row_m, row_l, diag))
        col_parts.append((col_m, col_l))
    M = torch.stack([c[0] for c in col_parts]).max(0).values
    L = sum(c[1] * torch.exp(c[0] - M) for c in col_parts)
    col_lse = (M.double() + L.double().log()).cpu()
    assert torch.allclose(col_lse, torch.from_numpy(cf["col_lse"]), atol=1e-4, rtol=0)
    cw = eng.softmax_weights(L, 1.0 / (2 * n))
    for r, (x, rx, row_m, row_l, diag) in enumerate(rows):
        sl = slice(r * nl, (r + 1) * nl)
        assert torch.allclose(diag.double().cpu(), torch.from_numpy(cf["diag"][sl]), atol=1e-4, rtol=0)
        rw = eng.softmax_weights(row_l, 1.0 / (2 * n))
        da, _ = eng.backward(x, y, yt, rx, ry, r * nl, scale, row_m, rw, M, cw, 1.0 / n, 1.0)
        torch.cuda.synchronize()
        assert rel(da, cf["d_a_hat"][sl]) <= GRAD_RTOL_BF16


def test_large_properties(eng):
    """Size-independent properties at a many-tile size the dense oracle does not reach cheaply:
    sum_j softmax_row = 1 via the gradient identity sum_ij G_ij = 0, symmetry under swapping the two
    sides, and agreement between the tensor-core and the exact kernels on a row sample."""
    n, d, scale = 8192, 512, 1 / 0.07
    g = torch.Generator(device="cuda").manual_seed(5)
    a = torch.randn(n, d, device="cuda", generator=g).bfloat16()
    b = (0.4 * a.float() + 0.6 * torch.randn(n, d, device="cuda", generator=g)).bfloat16()
    ra, _ = eng.normalize(a)
    rb, _ = eng.normalize(b)
    _, bt = eng.stage(b, torch.bfloat16, want_t=True)
    row_m, row_l, col_m, col_l, diag = eng.forward(a, b, ra, rb, 0, scale)
    # swapping the operands swaps row and column statistics
    row_m2, row_l2, col_m2, col_l2, diag2 = eng.forward(b, a, rb, ra, 0, scale)
    r1 = row_m + row_l.log()
    c2 = col_m2 + col_l2.log()
    assert torch.allclose(r1, c2, atol=2e-5, rtol=0)
    assert torch.allclose(diag, diag2, atol=2e-5, rtol=0)
    # exact kernels on the first 256 rows agree with the tensor-core statistics
    rm_e, rl_e, _, _, dg_e = eng.forward(a[:256].contiguous(), b, ra[:256].contiguous(), rb, 0, scale, flags=1)
    assert torch.allclose(rm_e + rl_e.log(), r1[:256], atol=2e-5, rtol=0)
    assert torch.allclose(dg_e, diag[:256], atol=2e-5, rtol=0)
    # gradient identity: rows of G sum to (p_row - 1)/2N + sum_j p_col/2N  ->  total sum is 0  =>  sum_i dA_hat_i . 0 ...
    coef = 1.0 / (2 * n)
    rw, cw = eng.softmax_weights(row_l, coef), eng.softmax_weights(col_l, coef)
    da, ds = eng.backward(a, b, bt, ra, rb, 0, scale, row_m, rw, col_m, cw, 1.0 / n, 1.0)
    da_e, _ = eng.backward(a[:128].contiguous(), b, None, ra[:128].contiguous(), rb, 0, scale, row_m[:128].contiguous(),
                           rw[:128].contiguous(), col_m, cw, 1.0 / n, 1.0, flags=1, want_dscale=False)
    torch.cuda.synchronize()
    assert rel(da[:128], da_e) <= GRAD_RTOL_BF16
    assert torch.isfinite(da).all() and math.isfinite(float(ds))


def test_errors_are_loud(eng):
    x = torch.zeros(8, 64, device="cuda", dtype=torch.bfloat16)
    r = torch.ones(8, device="cuda")
    with pytest.raises(RuntimeError):
        eng.forward(x, x, r, r, 0, float("nan"))
    with pytest.raises(RuntimeError):
        eng.normalize(torch.zeros(8, 64))          # CPU tensor: no CPU path
    with pytest.raises(RuntimeError):
        eng.backward(x, x, None, r, r, 0, 10.0, r, r, r, r, 0.1, 1.0)   # tensor-core path without y_t


def test_zero_row_is_clamped_like_F_normalize():
    a, b = O.make_inputs(64, 64, seed=2)
    a[5] = 0
    ref = O.ref_step(a.double(), b.double(), O.LOGIT_SCALE_INIT)
    loss, da, db, dt = run_fused(a, b, O.LOGIT_SCALE_INIT, torch.float32)
    assert abs(loss - float(ref["loss"])) <= 1e-5 * abs(float(ref["loss"]))
    assert rel(db, ref["d_b"]) <= 5e-5
    assert torch.isfinite(da).all()


# ------------------------------------------------------------------------------------------------
# CTA-pair kernels (d % 128 == 0): no transposed operand, column-sweep splits, ragged edges
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m,d,split", [(3000, 3000, 512, 0), (3000, 3000, 512, 3), (1111, 2500, 256, 2),
                                         (2100, 2100, 768, 4), (2049, 2304, 128, 1)])
def test_pair_kernels_split_and_ragged(eng, monkeypatch, n, m, d, split):
    """Forward statistics and both backward sides of the pair kernels against the float64 closed form with the
    column sweep cut into work items (CLIPNCE_SPLIT_STEPS test hook), y_t = None, rows/columns that are not
    multiples of the 128-row / 256-column tiles, and n_cols > n_rows (extra negative columns)."""
    if split:
        monkeypatch.setenv("CLIPNCE_SPLIT_STEPS", str(split))
    else:
        monkeypatch.delenv("CLIPNCE_SPLIT_STEPS", raising=False)
    scale = 1 / 0.07
    assert eng.uses_tensor_cores(torch.bfloat16, d, scale) and not eng.needs_transposed(torch.bfloat16, d, scale)
    a, b = O.make_inputs(max(n, m), d, seed=21, mix=0.4)
    a, b = a[:n], b[:m]
    cf = O.closed_form(a.numpy(), b.numpy(), scale)
    x, y = a.cuda().bfloat16(), b.cuda().bfloat16()
    rx, _ = eng.normalize(x)
    ry, _ = eng.normalize(y)
    row_m, row_l, col_m, col_l, diag = eng.forward(x, y, rx, ry, 0, scale)
    torch.cuda.synchronize()
    row_lse = (row_m.double() + row_l.double().log()).cpu()
    col_lse = (col_m.double() + col_l.double().log()).cpu()
    assert torch.allclose(row_lse, torch.from_numpy(cf["row_lse"]), rtol=0, atol=1e-4)
    assert torch.allclose(col_lse, torch.from_numpy(cf["col_lse"]), rtol=0, atol=1e-4)
    assert torch.allclose(diag.double().cpu(), torch.from_numpy(cf["diag"]), rtol=0, atol=1e-4)
    if n != m:
        return   # rectangular: the closed form's gradients assume positives for every column
    coef = 1.0 / (2 * n)
    rw, cw = eng.softmax_weights(row_l, coef), eng.softmax_weights(col_l, coef)
    da, ds = eng.backward(x, y, None, rx, ry, 0, scale, row_m, rw, col_m, cw, 1.0 / n, 1.0)
    db, _ = eng.backward(y, x, None, ry, rx, 0, scale, col_m, cw, row_m, rw, 1.0 / n, 1.0, want_dscale=False)
    torch.cuda.synchronize()
    assert rel(da, cf["d_a_hat"]) <= GRAD_RTOL_BF16, rel(da, cf["d_a_hat"])
    assert rel(db, cf["d_b_hat"]) <= GRAD_RTOL_BF16, rel(db, cf["d_b_hat"])
    assert abs(float(ds) - cf["d_scale_sum"]) <= 2e-2 * abs(cf["d_scale_sum"]) + 1e-6


def test_device_scale_and_graphed_step():
    """The kernels read s from a device scalar (scale_dev); the host only passes a stale hint.  A CUDA-graph replay of
    the whole step must follow the logit scale written into its static input, without re-capture."""
    from clip_dplm_b200 import fused_clip_loss
    from clip_dplm_b200.graph import GraphedClipStep
    n, d = 1024, 256
    a, b = O.make_inputs(n, d, seed=31, mix=0.4)
    ac, bc = a.cuda().bfloat16(), b.cuda().bfloat16()
    step = GraphedClipStep(n, d)
    for ls in (math.log(1 / 0.07), 2.0, 3.2):
        ref = O.ref_step(a.double(), b.double(), ls)
        loss, da, db, dt = step(ac, bc, ls)
        torch.cuda.synchronize()
        assert abs(float(loss) - float(ref["loss"])) <= LOSS_RTOL_BF16 * abs(float(ref["loss"]))
        assert rel(da.float(), ref["d_a"]) <= GRAD_RTOL_BF16 and rel(db.float(), ref["d_b"]) <= GRAD_RTOL_BF16
        assert abs(float(dt) - float(ref["d_logit_scale"])) <= 2e-2 * abs(float(ref["d_logit_scale"])) + 1e-6
        # and the eager call agrees bit for bit with the replay (same kernels, same order)
        t = torch.tensor(ls, device="cuda", requires_grad=True)
        ar, br = ac.clone().requires_grad_(True), bc.clone().requires_grad_(True)
        l2 = fused_clip_loss(ar, br, t)
        l2.backward()
        assert torch.equal(l2.detach(), loss) and torch.equal(ar.grad, da) and torch.equal(br.grad, db)


@pytest.mark.parametrize("split", [False, True])
def test_host_fed_step_pipelines_batches(split):
    """HostFedClipStep: batches from pinned host memory, H2D of batch k+1 overlapped with step k; every step must
    return the results of ITS batch.  split: forward and backward captured as two graphs, the H2D ordered behind the forward."""
    from clip_dplm_b200.graph import GraphedClipStep, HostFedClipStep
    n, d = 512, 128
    batches = []
    for seed in (41, 42, 43):
        a, b = O.make_inputs(n, d, seed=seed, mix=0.4)
        batches.append((a.bfloat16().pin_memory(), b.bfloat16().pin_memory()))
    ref_step = GraphedClipStep(n, d)
    feeder = HostFedClipStep(n, d, split=split)
    feeder.prefetch(*batches[0])
    for k, (ah, bh) in enumerate(batches):
        loss, da, db, dt = feeder.step()
        if k + 1 < len(batches):
            feeder.prefetch(*batches[k + 1])
        got = (loss.clone(), da.clone(), db.clone())
        want = ref_step(ah.cuda(), bh.cuda(), feeder.logit_scale.detach())
        torch.cuda.synchronize()
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]) and torch.equal(got[2], want[2])


# ------------------------------------------------------------------------------------------------
# retrieval: top-k on the similarity sweep (SURVEY.md section 8f rank 1, BASELINE config 5)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_q,n_lib,d,k,split", [(300, 5000, 512, 10, 0), (1000, 777, 128, 1, 0), (257, 20000, 256, 16, 9),
                                                 (64, 9, 128, 10, 0), (513, 4096, 384, 5, 4)])
def test_topk_matches_oracle(eng, monkeypatch, n_q, n_lib, d, k, split):
    if split:
        monkeypatch.setenv("CLIPNCE_SPLIT_STEPS", str(split))
    else:
        monkeypatch.delenv("CLIPNCE_SPLIT_STEPS", raising=False)
    from clip_dplm_b200.retrieval import topk_similarity
    g = torch.Generator().manual_seed(17)
    q = torch.randn(n_q, d, generator=g).bfloat16()
    lib = (torch.randn(n_lib, d, generator=g) * torch.rand(n_lib, 1, generator=g).add(0.5)).bfloat16()   # rows of varied norm
    lib[: min(n_q, n_lib)] += 0.7 * q[: min(n_q, n_lib)]                                                 # planted neighbours
    s_ref, i_ref, sim = O.ref_topk(q.double(), lib.double(), k)
    s, i = topk_similarity(q.cuda(), lib.cuda(), k, library_offset=0)
    torch.cuda.synchronize()
    s, i = s.cpu().double(), i.cpu()
    kk = min(k, n_lib)
    assert (i[:, kk:] == -1).all() and torch.isinf(s[:, kk:]).all()
    s, i = s[:, :kk], i[:, :kk]
    assert torch.allclose(s, s_ref, atol=2e-5, rtol=0)
    # same columns up to exact ties: the oracle's similarity AT the returned indices is the oracle's k-th best or better
    assert torch.allclose(torch.gather(sim, 1, i), s_ref, atol=2e-5, rtol=0)
    assert (i == i_ref).double().mean() > 0.999
    assert all(len(set(r.tolist())) == kk for r in i)


def test_top1_accuracy_matches_argmax(eng):
    from clip_dplm_b200.retrieval import top1_accuracy
    a, b = O.make_inputs(1500, 256, seed=23, mix=0.25)
    _, i_ref, _ = O.ref_topk(a.double(), b.double(), 1)
    want = (i_ref[:, 0] == torch.arange(1500)).double().mean()
    got = top1_accuracy(a.cuda().bfloat16(), b.cuda().bfloat16())
    assert abs(float(got) - float(want)) < 2e-3
    with pytest.raises(RuntimeError):
        eng.topk(torch.zeros(8, 64, device="cuda", dtype=torch.bfloat16), torch.zeros(8, 64, device="cuda", dtype=torch.bfloat16),
                 torch.ones(8, device="cuda"), torch.ones(8, device="cuda"), 3)      # d = 64: not served -> loud


def test_topk_negative_scores_and_shared_threshold(eng, monkeypatch):
    """Queries anti-correlated with most of the library: the k best similarities are negative, so the threshold that
    work items share through atomicMax (an order-preserving int key) and its safety margin are exercised below zero;
    many short work items (forced split) make later items start from earlier items' bounds."""
    monkeypatch.setenv("CLIPNCE_SPLIT_STEPS", "8")
    from clip_dplm_b200.retrieval import topk_similarity
    g = torch.Generator().manual_seed(29)
    n_q, n_lib, d, k = 256, 30000, 128, 10
    base = torch.randn(1, d, generator=g)
    q = (base + 0.3 * torch.randn(n_q, d, generator=g)).bfloat16()
    lib = (-base + 0.6 * torch.randn(n_lib, d, generator=g)).bfloat16()
    s_ref, i_ref, sim = O.ref_topk(q.double(), lib.double(), k)
    assert float(s_ref.max()) < 0
    s, i = topk_similarity(q.cuda(), lib.cuda(), k)
    torch.cuda.synchronize()
    assert torch.allclose(s.cpu().double(), s_ref, atol=2e-5, rtol=0)
    assert torch.allclose(torch.gather(sim, 1, i.cpu()), s_ref, atol=2e-5, rtol=0)


# ------------------------------------------------------------------------------------------------
# clipnce_backward_dx: backward side + split-partial sum + row dots + normalise backward in one call
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,split,in_dt,c_dt,out_dt", [
    (3000, 512, 0, torch.bfloat16, torch.bfloat16, torch.bfloat16),     # 16-byte path, no split
    (3000, 512, 3, torch.bfloat16, torch.bfloat16, torch.bfloat16),     # 16-byte path over split partials
    (2100, 256, 2, torch.float32, torch.bfloat16, torch.float32),       # fp32 rows of a bf16 step (x_orig != x)
    (1111, 128, 4, torch.bfloat16, torch.bfloat16, torch.float32),
    (300, 50, 0, torch.float32, torch.float32, torch.float32),          # exact path, d % 4 != 0: scalar finish
    (260, 192, 0, torch.bfloat16, torch.bfloat16, torch.bfloat16),      # single-CTA tensor-core kernels (transposed operand)
])
def test_backward_dx_matches_unfused(eng, monkeypatch, n, d, split, in_dt, c_dt, out_dt):
    """The fused call against the two calls it replaces (clipnce_backward -> clipnce_normalize_backward), on the same
    statistics, with an upstream gradient on the device and one all-zero row (the clamp_min sub-gradient branch)."""
    if split:
        monkeypatch.setenv("CLIPNCE_SPLIT_STEPS", str(split))
    else:
        monkeypatch.delenv("CLIPNCE_SPLIT_STEPS", raising=False)
    scale = 1 / 0.07
    a, b = O.make_inputs(n, d, seed=5, mix=0.4)
    a[7] = 0
    xo, yo = a.cuda().to(in_dt), b.cuda().to(in_dt)
    x, _ = eng.stage(xo, c_dt)
    y, _ = eng.stage(yo, c_dt)
    want_t = eng.uses_tensor_cores(c_dt, d, scale) and eng.needs_transposed(c_dt, d, scale)
    y_t = eng.stage(y, c_dt, want_t=True)[1] if want_t else None
    rx, _ = eng.normalize(xo)
    ry, _ = eng.normalize(yo)
    row_m, row_l, col_m, col_l, diag = eng.forward(x, y, rx, ry, 0, scale)
    coef = 1.0 / (2 * n)
    rw, cw = eng.softmax_weights(row_l, coef), eng.softmax_weights(col_l, coef)
    gs = torch.tensor([2.5], device="cuda")
    dx_hat, ds_ref = eng.backward(x, y, y_t, rx, ry, 0, scale, row_m, rw, col_m, cw, 1.0 / n, 1.0)
    want = eng.normalize_backward(xo, rx, dx_hat, out_dt, gs)
    got, ds = eng.backward_dx(x, y, y_t, rx, ry, 0, scale, row_m, rw, col_m, cw, 1.0 / n, xo, out_dt, gs)
    torch.cuda.synchronize()
    tol = 1e-2 if out_dt == torch.bfloat16 else 2e-5     # one bf16 ulp / fp32 rounding of a reordered dot product
    err = (got.float() - want.float()).abs().max()
    assert float(err) <= tol * float(want.float().abs().max()), float(err)
    assert torch.isfinite(got.float()).all()
    assert abs(float(ds) - float(ds_ref)) <= 1e-4 * abs(float(ds_ref)) + 1e-7


# ------------------------------------------------------------------------------------------------
# the benchmarked shapes (BASELINE.json configs 2, 3, 4) against the sampled-row CPU oracle
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,ls,mix", [(4096, 512, O.LOGIT_SCALE_INIT, 0.5), (32768, 768, O.LOGIT_SCALE_INIT, 0.5),
                                        (65536, 512, O.LOGIT_SCALE_INIT, 0.5), (8192, 128, 3.0, 0.5),
                                        (16384, 256, math.log(100.0), 0.12)])
def test_benchmarked_shapes_against_sampled_oracle(n, d, ls, mix):
    """Loss and d logit_scale against a blockwise host pass over all N^2 logits; gradient rows of 128 random indices per
    modality against all N columns / rows in float64 (oracle/sampled.py).  Covers the split counts / wave shapes these
    sizes select (pick_split_steps), d = 768's one-buffer variant, and s = 100 (the clamp(max=100) regime of
    old/clip_opt.py:100; weakly correlated pairs there, so that the loss does not underflow to 0)."""
    from oracle import sampled as SO
    torch.set_num_threads(os.cpu_count() or 1)
    a, b = O.make_inputs(n, d, seed=77, mix=mix)
    loss, da, db, dt = run_fused(a, b, ls, torch.bfloat16)
    rng = np.random.default_rng(n + d)
    rows_a, rows_b = np.sort(rng.choice(n, 128, replace=False)), np.sort(rng.choice(n, 128, replace=False))
    ref = SO.sampled_reference(a, b, math.exp(ls), rows_a, rows_b)
    cmp = SO.compare(ref, loss, da[rows_a].numpy(), db[rows_b].numpy(), dt, loss_tol=LOSS_RTOL_BF16, grad_tol=GRAD_RTOL_BF16)
    assert cmp["ok"], cmp


# ------------------------------------------------------------------------------------------------
# two-sided backward (csrc/kernels_pair2.cuh): one sweep over the logits tiles emits dA and dB
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d,forced_p,seg", [(4096, 512, 0, 0), (4096, 512, 5, 1), (2048, 256, 3, 1), (2048, 128, 0, 0),
                                                (3072, 384, 7, 1), (4096, 512, 5, 2), (4096, 256, 0, 2), (2048, 512, 70, 8), (2048, 768, 0, 0), (2560, 640, 9, 1)])
def test_two_sided_backward(monkeypatch, n, d, forced_p, seg):
    """clipnce_backward_both_dx against the dense float64 closed form AND against the two-sweep path on the same inputs.
    `forced_p` producer pairs force several rounds of work items (the last one partly filled), ring wrap-around and the
    read-modify-write of dB across rounds at a size the dense oracle still reaches; `seg` column segments force rounds
    that straddle segment boundaries (several consumer tasks per step) and per-segment dA slabs."""
    from clip_dplm_b200.engine import CudaEngine
    monkeypatch.setenv("CLIPNCE_BWD2_MIN_N", "256")
    if forced_p:
        monkeypatch.setenv("CLIPNCE_BWD2_P", str(forced_p))
    if seg:
        monkeypatch.setenv("CLIPNCE_BWD2_SEG", str(seg))
    assert CudaEngine().backward_both_bytes(n, n, d, torch.bfloat16, 1 / 0.07) > 0, "two-sided backward not served on this device"
    a, b = O.make_inputs(n, d, seed=91)
    loss2, da2, db2, dt2 = run_fused(a, b, O.LOGIT_SCALE_INIT, torch.bfloat16)
    monkeypatch.setenv("CLIPNCE_NO_BWD2", "1")
    loss1, da1, db1, dt1 = run_fused(a, b, O.LOGIT_SCALE_INIT, torch.bfloat16)
    monkeypatch.delenv("CLIPNCE_NO_BWD2")
    cf = O.closed_form(a.numpy(), b.numpy(), math.exp(O.LOGIT_SCALE_INIT))
    assert loss1 == loss2
    assert rel(da2, cf["d_a"]) <= GRAD_RTOL_BF16 and rel(db2, cf["d_b"]) <= GRAD_RTOL_BF16
    assert abs(dt2 - cf["d_scale_sum"]) <= GRAD_RTOL_BF16 * abs(cf["d_scale_sum"])
    # the two paths round G the same way; only the 1/norm factors move between G and the bf16 operands
    assert rel(da2, da1) <= 5e-3 and rel(db2, db1) <= 5e-3
    # rerun: bit-identical (fixed-order accumulation, no atomics on data)
    _, da3, db3, _ = run_fused(a, b, O.LOGIT_SCALE_INIT, torch.bfloat16)
    assert torch.equal(da2, da3) and torch.equal(db2, db3)


@pytest.mark.parametrize("n,d,s,forced_p,seg", [(4096, 512, 100.0, 0, 0), (2048, 256, 60.0, 5, 1), (2048, 768, 100.0, 0, 0),
                                                  (3072, 384, 100.0, 7, 2)])
def test_two_sided_backward_large_scale(monkeypatch, n, d, s, forced_p, seg):
    """The two-sided backward in kernel family 2 (bwd2_kernel<true>: exp(S - m_i) w_i + exp(S - m_j) w_j from the true
    maxima of the online soft-max forward) -- the clamp(max=100) regime of old/clip_opt.py:100, run1/full.py:76 -- against
    the float64 oracle and against the two-sweep family-2 path."""
    from clip_dplm_b200.engine import CudaEngine
    monkeypatch.setenv("CLIPNCE_BWD2_MIN_N", "256")
    if forced_p:
        monkeypatch.setenv("CLIPNCE_BWD2_P", str(forced_p))
    if seg:
        monkeypatch.setenv("CLIPNCE_BWD2_SEG", str(seg))
    assert CudaEngine().backward_both_bytes(n, n, d, torch.bfloat16, s) > 0, "two-sided backward (family 2) not served"
    a, b = O.make_inputs(n, d, seed=17, mix=0.12)
    kw = dict(scale_is_log=False)
    loss2, da2, db2, dt2 = run_fused(a, b, s, torch.bfloat16, **kw)
    monkeypatch.setenv("CLIPNCE_NO_BWD2", "1")
    loss1, da1, db1, dt1 = run_fused(a, b, s, torch.bfloat16, **kw)
    monkeypatch.delenv("CLIPNCE_NO_BWD2")
    ref = O.ref_step(a.double(), b.double(), s, **kw)
    assert loss1 == loss2 and abs(loss2 - float(ref["loss"])) <= LOSS_RTOL_BF16 * abs(float(ref["loss"]))
    assert rel(da2, ref["d_a"]) <= GRAD_RTOL_BF16 and rel(db2, ref["d_b"]) <= GRAD_RTOL_BF16
    assert abs(dt2 - float(ref["d_logit_scale"])) <= GRAD_RTOL_BF16 * abs(float(ref["d_logit_scale"])) + 1e-7
    assert rel(da2, da1) <= 5e-3 and rel(db2, db1) <= 5e-3
    _, da3, db3, _ = run_fused(a, b, s, torch.bfloat16, **kw)
    assert torch.equal(da2, da3) and torch.equal(db2, db3)


# ------------------------------------------------------------------------------------------------
# kernel family 2: tensor cores with true running maxima (s up to the clamp at 100, unbounded logits)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,m_extra,d,s,symmetric,normalized", [(1500, 0, 256, 100.0, True, True), (1024, 0, 768, 60.0, True, True),
                                                                (777, 300, 128, 100.0, True, True), (900, 500, 512, 10.0, False, False),
                                                                (2048, 0, 512, 100.0, False, True)])
def test_large_scale_and_unbounded_logits_on_tensor_cores(eng, n, m_extra, d, s, symmetric, normalized):
    """old/clip_opt.py:100 / run1/full.py:76 clamp the logit scale at 100, tong/utils/losses.py:10-14 appends queue rows of
    arbitrary norm: both leave the fixed shift's range and must still run on the tcgen05 kernels (family 2: online
    soft-max forward -- two launches, rows and columns -- and the two-exponential backward), against the float64 oracle."""
    from clip_dplm_b200 import _lib
    flags = 0 if normalized else _lib.FLAG_UNBOUNDED
    assert eng.lib.clipnce_uses_tensor_cores(_lib.BF16, d, float(s), flags) == 2
    a, b = O.make_inputs(n, d, seed=13, n_cols=n + m_extra, mix=0.12 if s > 50 else 0.5)
    extra = None
    if m_extra:
        extra = b[n:].double()
        extra = torch.nn.functional.normalize(extra, dim=-1) if normalized else extra * 0.2   # norms ~4.5: logits up to ~45
        extra = extra.to(torch.bfloat16).double()
        b = b[:n]
    kw = dict(symmetric=symmetric, scale_is_log=False)
    okw = dict(kw, **({"extra_cols": extra} if extra is not None else {}))
    ref = O.ref_step(a.double(), b.double(), s, **okw)
    fkw = dict(kw, **({"extra_cols": extra.float(), "extra_normalized": normalized} if extra is not None else {}))
    loss, da, db, dt = run_fused(a, b, s, torch.bfloat16, **fkw)
    assert abs(loss - float(ref["loss"])) <= LOSS_RTOL_BF16 * abs(float(ref["loss"]))
    assert rel(da, ref["d_a"]) <= GRAD_RTOL_BF16 and rel(db, ref["d_b"]) <= GRAD_RTOL_BF16
    assert abs(dt - float(ref["d_logit_scale"])) <= GRAD_RTOL_BF16 * abs(float(ref["d_logit_scale"])) + 1e-7


@pytest.mark.parametrize("flip", ["none", "rows", "cols"])
@pytest.mark.parametrize("n,d", [(1024, 256), (1500, 512)])
def test_speculative_large_scale_forward_and_its_exact_fallback(monkeypatch, n, d, flip):
    """s = 100 (clamp regime, old/clip_opt.py:100): clipnce_forward runs ONE fixed-shift sweep with the shift lowered to
    s - 72 and falls back to the exact online sweeps, on the device, when a row or column has every logit below s - 134.
    `flip` builds such rows / columns (embeddings pointing away from everything, positive pair included); all three
    cases must match the float64 oracle and the always-exact path (CLIPNCE_NO_SPECULATE=1)."""
    g = torch.Generator().manual_seed(n + d)
    v = torch.nn.functional.normalize(torch.randn(1, d, generator=g), dim=-1)
    a = (v * 8.0 + 0.25 * torch.randn(n, d, generator=g)).bfloat16().float()
    b = (v * 8.0 + 0.25 * torch.randn(n, d, generator=g)).bfloat16().float()
    idx = [5, 77, n - 3]
    if flip == "rows":
        a[idx] = -a[idx]
    elif flip == "cols":
        b[idx] = -b[idx]
    s = 100.0
    kw = dict(scale_is_log=False)
    ref = O.ref_step(a.double(), b.double(), s, **kw)
    loss, da, db, dt = run_fused(a, b, s, torch.bfloat16, **kw)
    monkeypatch.setenv("CLIPNCE_NO_SPECULATE", "1")
    loss_x, da_x, db_x, dt_x = run_fused(a, b, s, torch.bfloat16, **kw)
    monkeypatch.delenv("CLIPNCE_NO_SPECULATE")
    assert abs(loss - float(ref["loss"])) <= LOSS_RTOL_BF16 * abs(float(ref["loss"]))
    assert abs(loss - loss_x) <= 2e-5 * abs(loss_x)
    assert rel(da, ref["d_a"]) <= GRAD_RTOL_BF16 and rel(db, ref["d_b"]) <= GRAD_RTOL_BF16
    assert rel(da, da_x) <= 2e-3 and rel(db, db_x) <= 2e-3
    assert abs(dt - float(ref["d_logit_scale"])) <= GRAD_RTOL_BF16 * abs(float(ref["d_logit_scale"])) + 1e-7
    if flip != "none":    # the flipped entries decide the loss: it is ~ 2 s cos / n per entry, far from the unflipped value
        assert float(ref["loss"]) > 0.05


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_second_device_in_one_process():
    """The kernels' shared-memory limit is raised per device: one process that runs the loss on cuda:0 and then on cuda:1
    (16384 x 512: the pair forward and the two-sided backward) gets the same loss and gradients, bit for bit, on both."""
    from clip_dplm_b200 import fused_clip_loss
    a, b = O.make_inputs(16384, 512, seed=41)
    outs = []
    for dev in ("cuda:0", "cuda:1"):
        ac = a.to(dev).bfloat16().requires_grad_(True)
        bc = b.to(dev).bfloat16().requires_grad_(True)
        t = torch.tensor(O.LOGIT_SCALE_INIT, device=dev, requires_grad=True)
        loss = fused_clip_loss(ac, bc, t)
        loss.backward()
        torch.cuda.synchronize(dev)
        outs.append([x.detach().cpu() for x in (loss, ac.grad, bc.grad, t.grad)])
    for x0, x1 in zip(*outs):
        assert torch.equal(x0, x1)
