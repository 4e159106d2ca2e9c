"""Every kernel route of `fused_clip_loss`, pinned and checked entry by entry against the float64 reference of
``oracle/rowwise.py``: the loss, every row of dA and dB, d logit_scale and, where the route returns them, every entry of
the row / column log-sum-exp and the diagonal -- each against its own error budget, not a whole-matrix tolerance.

The first part checks the checker and needs no GPU: the reference against the closed form the golden fixtures pin, a
rounding-only emulation of the kernels (the gradient tile rounded to bf16) that must pass with a margin, and planted
corruptions of the kind a tiled kernel gets wrong (one row, one column, one 128-row block, one loss term) that must be
rejected with a margin.  The second part runs every route on the GPU; a spy on the engine records which route served
each case, and a case fails if another route served it."""
import inspect
import math
import os

import numpy as np
import pytest
import torch

from oracle import ref_step as O
from oracle import rowwise as R

G_UP = 0.37      # upstream gradient of the loss in every GPU case except the g = 1 control


# ------------------------------------------------------------------------------------------------------------------------
# the checker itself (CPU)
# ------------------------------------------------------------------------------------------------------------------------
def test_reference_matches_closed_form():
    a, b = O.make_inputs(256, 128, seed=3, mix=0.4)
    s = 1 / 0.07
    for symmetric in (True, False):
        cf = O.closed_form(a.numpy(), b.numpy(), s, symmetric=symmetric)
        ref = R.reference(a, b, s, symmetric=symmetric, compute_dtype=torch.float32, g=1.0, block=100)
        for k in ("row_lse", "col_lse", "diag", "d_a", "d_b"):
            assert np.abs(ref[k].numpy() - cf[k]).max() <= 1e-12 * max(1.0, np.abs(cf[k]).max()), k
        assert abs(float(ref["loss"]) - cf["loss"]) <= 1e-12
        assert abs(float(ref["d_scale_sum"]) - cf["d_scale_sum"]) <= 1e-12
    # staging: fp32 rows of a bf16 step are rounded for the contraction only
    a32 = a + 1e-3 * torch.randn(a.shape, generator=torch.Generator().manual_seed(1))
    ref = R.reference(a32, b, s, compute_dtype=torch.bfloat16)
    ra = 1.0 / a32.double().norm(dim=1)
    want = s * (a32.bfloat16().double() * ra[:, None] * b.double() / b.double().norm(dim=1)[:, None]).sum(1)
    assert torch.allclose(ref["diag"], want, rtol=0, atol=1e-12)


def _emulate(a, b, s, ref, *, symmetric=True, tamper=None):
    """The kernels' arithmetic with only the rounding that matters: the reference G rounded to bf16 entry by entry,
    contracted and finished in float64; statistics and loss rounded to fp32.  ``tamper(G)`` edits the rounded G."""
    n = a.shape[0]
    a64, ra, ac = R.staged(a, torch.bfloat16)
    b64, rb, bc = R.staged(b, torch.bfloat16)
    S = s * ac @ bc.T
    w = 1.0 / (2 * n) if symmetric else 1.0 / n
    G = (S - ref["row_lse"][:, None]).exp() * w
    if symmetric:
        G += (S - ref["col_lse"][None, :]).exp() * w
    G -= torch.eye(n, dtype=torch.float64) / n
    Gq = G.to(torch.bfloat16).double()
    if tamper is not None:
        tamper(Gq)
    d_ah, d_bh = s * Gq @ bc, s * Gq.T @ ac
    out = {"d_ah": d_ah, "d_bh": d_bh, "d_a": R.normalize_backward(a64, ra, d_ah, ref["g"]),
           "d_b": R.normalize_backward(b64, rb, d_bh, ref["g"]), "d_scale_sum": float((Gq * S).sum()),
           "loss": float(ref["loss"].float())}
    for k in ("row_lse", "col_lse", "diag"):
        out[k] = ref[k].float().double()
    out["ac"], out["bc"], out["Gq"], out["a64"], out["ra"], out["b64"], out["rb"] = ac, bc, Gq, a64, ra, b64, rb
    return out


def _ratios(ref, em):
    return R.check(ref, loss=em["loss"], d_a=em["d_a"], d_b=em["d_b"], d_scale_sum=em["d_scale_sum"],
                   row_lse=em["row_lse"], col_lse=em["col_lse"], diag=em["diag"])


@pytest.mark.parametrize("s", [14.3, 100.0])
@pytest.mark.parametrize("mix", [0.3, 0.95])
@pytest.mark.parametrize("n", [300, 1000])
def test_rounding_only_emulation_passes_with_margin(n, mix, s):
    a, b = O.make_inputs(n, 256, seed=n, mix=mix)
    ref = R.reference(a, b, s, g=G_UP)
    rep = _ratios(ref, _emulate(a, b, s, ref))
    assert max(r["max"] for r in rep.values()) <= 0.5, R.describe(rep, "bf16-tile emulation")


def _corruptions(n, s, ref=None):
    """name -> function(a, b, ref) -> emulated result with one planted fault.  A fault can only show where the gradient
    is above what fp32 statistics resolve; at s = 100 most positives are so well separated that only a few percent of
    the rows are, so the faults go to the row with the largest reference gradient, and to its 128-row block."""
    k = int(ref["d_a"].norm(dim=1).argmax()) if ref is not None else 0
    blk = slice(k // 128 * 128, min(n, k // 128 * 128 + 128))

    def refinish(em, d_ah=None, d_bh=None):
        if d_ah is not None:
            em["d_a"] = R.normalize_backward(em["a64"], em["ra"], d_ah, G_UP)
        if d_bh is not None:
            em["d_b"] = R.normalize_backward(em["b64"], em["rb"], d_bh, G_UP)
        return em

    def row_zeroed(a, b, ref):
        em = _emulate(a, b, s, ref)
        em["d_a"][k] = 0
        return em

    def row_scaled(a, b, ref):
        em = _emulate(a, b, s, ref)
        em["d_a"][k] *= 1.1
        return em

    def column_dropped(a, b, ref):
        em = _emulate(a, b, s, ref)
        return refinish(em, d_ah=em["d_ah"] - s * em["Gq"][:, k:k + 1] * em["bc"][k][None, :])

    def block_missing_late_rows(a, b, ref):   # a producer round that never reached this block of dB
        em = _emulate(a, b, s, ref)
        h = n // 2
        d_bh = em["d_bh"].clone()
        d_bh[blk] = s * em["Gq"][:h, blk].T @ em["ac"][:h]
        return refinish(em, d_bh=d_bh)

    def diag_w_high(a, b, ref):
        def tamper(Gq):
            i = torch.arange(blk.start, blk.stop)
            Gq[i, i] -= 0.1 / n
        return _emulate(a, b, s, ref, tamper=tamper)

    def loss_term_missing(a, b, ref):
        em = _emulate(a, b, s, ref)
        em["loss"] -= float(ref["row_lse"][k] - ref["diag"][k]) / (2 * n)
        return em

    def d_scale_off(a, b, ref):
        em = _emulate(a, b, s, ref)
        em["d_scale_sum"] *= 1.01
        return em

    return {f.__name__: f for f in (row_zeroed, row_scaled, column_dropped, block_missing_late_rows, diag_w_high,
                                    loss_term_missing, d_scale_off)}


FAULTS = list(_corruptions(1000, 1.0))
# s = 100, mix 0.3: the positives sit so far apart that the loss and sum G.S are themselves within a few fp32 budgets of
# zero, and the best-resolved row's gradient is about 90 of its budgets -- a 1 % change of the scalars or a 10 % change
# of a row cannot reach a ratio of 10 there.  The faults that remove or add whole contributions are planted there too;
# all seven are planted at s = 100 in the weakly correlated pairs the suite uses at that scale (mix 0.12).
RESOLVED_AT_MIX_03_S100 = ("row_zeroed", "column_dropped", "block_missing_late_rows", "diag_w_high")
FAULT_CASES = ([(f, 14.3, 0.3) for f in FAULTS] + [(f, 100.0, 0.12) for f in FAULTS] +
               [(f, 100.0, 0.3) for f in RESOLVED_AT_MIX_03_S100])


@pytest.mark.parametrize("fault,s,mix", FAULT_CASES)
def test_planted_corruption_is_rejected(fault, s, mix):
    n = 1000
    a, b = O.make_inputs(n, 256, seed=n, mix=mix)
    ref = R.reference(a, b, s, g=G_UP)
    rep = _ratios(ref, _corruptions(n, s, ref)[fault](a, b, ref))
    worst = max(r["max"] for r in rep.values())
    assert worst >= 10, R.describe(rep, fault)


# ------------------------------------------------------------------------------------------------------------------------
# every route on the GPU
# ------------------------------------------------------------------------------------------------------------------------
F32, BF16 = torch.float32, torch.bfloat16
SPIED = ("group_forward", "group_backward", "forward", "backward_both", "backward_dx", "backward_both_sharded_sweep")


def _spy_engine(eng, setattr_):
    """Wrap the engine's route entry points; every call appends what served it (the kernel family the library selects
    for its arguments, whether the operand is transposed, whether a family-2 forward speculates).

    "speculate" is the library's own answer for the call's arguments (clipnce_forward_gathered_ok), which reads the same
    CLIPNCE_NO_SPECULATE switch as the forward: it shows that the switch reached the library and that the forward ran in
    family 2, not that the speculative sweep itself ran -- no hook exposes that."""
    calls = []
    lib = eng.lib

    def wrap(name):
        fn = getattr(eng, name)
        sig = inspect.signature(fn)

        def spy(*args, **kw):
            p = sig.bind(*args, **kw)
            p.apply_defaults()
            p = p.arguments
            x = p["x"] if "x" in p else p["stack"]
            dt, d, scale, flags = (0 if x.dtype == BF16 else 1), x.shape[1], float(p["scale"]), int(p["flags"])
            calls.append({"call": name, "family": lib.clipnce_uses_tensor_cores(dt, d, scale, flags),
                          "transposed": bool(lib.clipnce_needs_transposed(dt, d, scale, flags)),
                          "speculate": bool(lib.clipnce_forward_gathered_ok(dt, d, scale, flags))})
            return fn(*args, **kw)
        setattr_(eng, name, spy)

    for name in SPIED:
        wrap(name)
    return calls


def _route(calls):
    """-> (backward route, its kernel family, whether the forward speculated) of the recorded calls."""
    names, fams = set(), set()
    for c in calls:
        if c["call"] == "group_backward":
            names.add("group")
        elif c["call"] == "backward_both":
            names.add("both")
        elif c["call"] == "backward_both_sharded_sweep":
            names.add("sharded")
        elif c["call"] == "backward_dx":
            names.add("exact" if c["family"] == 0 else ("tc" if c["transposed"] else "pair"))
        else:
            continue
        fams.add(c["family"])
    spec = any(c["speculate"] for c in calls if c["call"] in ("forward", "group_forward") and c["family"] == 2)
    return "+".join(sorted(names)), (fams.pop() if len(fams) == 1 else tuple(sorted(fams))), spec


@pytest.fixture
def route_spy(monkeypatch):
    from clip_dplm_b200.engine import default_engine
    return _spy_engine(default_engine(), monkeypatch.setattr)


def _inputs(n, d, *, seed, mix, n_extra=0, extra_normalized=True, flip=False, fp32_rows=False):
    """Caller's rows (fp32 rows are NOT pre-rounded to bf16, so that a bf16 step's staging is exercised) and the extra
    columns as the kernels store them (bf16)."""
    if flip:    # test_speculative_large_scale_forward_and_its_exact_fallback's rows: one direction, three rows reversed
        g = torch.Generator().manual_seed(n + d)
        v = torch.nn.functional.normalize(torch.randn(1, d, generator=g), dim=-1)
        a = (v * 8.0 + 0.25 * torch.randn(n, d, generator=g)).bfloat16().float()
        b = (v * 8.0 + 0.25 * torch.randn(n, d, generator=g)).bfloat16().float()
        a[[5, 77, n - 3]] *= -1
        return a, b, None
    a, b = O.make_inputs(n, d, seed=seed, mix=mix, n_cols=n + n_extra, round_bf16=not fp32_rows)
    extra = None
    if n_extra:
        e = b[n:]
        extra = (torch.nn.functional.normalize(e, dim=-1) if extra_normalized else e * 0.2).bfloat16()
        b = b[:n].contiguous()
    return a, b, extra


def _check_report(rep, route, case_id):
    worst = max(r["max"] for r in rep.values())
    print(f"\nRATIOS {case_id} route={route} " + " ".join(f"{k}={v['max']:.3g}" for k, v in rep.items()))
    assert worst <= 1.0, R.describe(rep, route)


# id, n, d, options, expected (route, family)
CASES = [
    # one grouped launch for both sides of a pair (n < 8192, where the two-sided kernel does not serve the shape)
    ("group-255x128", 255, 128, {}, ("group", 1)),
    ("group-257x256", 257, 256, {}, ("group", 1)),
    ("group-4095x768", 4095, 768, {}, ("group", 1)),
    ("group-8191x512", 8191, 512, {}, ("group", 1)),
    ("group-1000x384-s100", 1000, 384, dict(s=100.0, mix=0.12), ("group", 2)),
    ("group-2048x512-fp32-autocast", 2048, 512, dict(a_dtype=F32, b_dtype=F32, autocast=True), ("group", 1)),
    ("group-3000x256-mix095", 3000, 256, dict(mix=0.95), ("group", 1)),
    ("group-1024x256-g1-control", 1024, 256, dict(g=1.0), ("group", 1)),
    # two-sided backward (clipnce_backward_both_dx)
    ("both-12288x512-default", 12288, 512, {}, ("both", 1)),
    ("both-16384x768", 16384, 768, {}, ("both", 1)),
    ("both-12288x256-s100", 12288, 256, dict(s=100.0, mix=0.12), ("both", 2)),
    ("both-4096x512-P5-SEG2", 4096, 512, dict(env={"CLIPNCE_BWD2_MIN_N": "256", "CLIPNCE_BWD2_P": "5",
                                                   "CLIPNCE_BWD2_SEG": "2"}), ("both", 1)),
    ("both-65536x512", 65536, 512, {}, ("both", 1)),
    # two sweeps of the CTA-pair kernels
    ("pair-8192x512", 8192, 512, dict(stats=False), ("pair", 1)),    # the first size the grouped launch leaves
    ("pair-12300x256", 12300, 256, {}, ("pair", 1)),
    ("pair-20000x512", 20000, 512, {}, ("pair", 1)),
    ("pair-3000x512-fp32A-bf16B", 3000, 512, dict(a_dtype=F32), ("pair", 1)),
    ("pair-2048x256-stats", 2048, 256, dict(stats=True), ("pair", 1)),
    ("pair-2000x384-onedir", 2000, 384, dict(symmetric=False), ("pair", 1)),
    ("pair-1500x256-cache700", 1500, 256, dict(n_extra=700), ("pair", 1)),
    ("pair-900x512-queue300", 900, 512, dict(n_extra=300, extra_normalized=False, symmetric=False, s=10.0), ("pair", 2)),
    ("pair-3000x512-split3", 3000, 512, dict(env={"CLIPNCE_SPLIT_STEPS": "3"}), ("pair", 1)),
    ("pair-16384x512-nobwd2", 16384, 512, dict(env={"CLIPNCE_NO_BWD2": "1"}), ("pair", 1)),
    ("pair-4096x512-nogroup", 4096, 512, dict(env={"CLIPNCE_NO_GROUP": "1"}, stats=False), ("pair", 1)),
    # single-CTA tensor-core kernels (d % 128 != 0: transposed operand)
    ("tc-3000x192", 3000, 192, {}, ("tc", 1)),
    ("tc-1111x320", 1111, 320, {}, ("tc", 1)),
    ("tc-777x64", 777, 64, {}, ("tc", 1)),
    # exact kernels
    ("exact-500x512-fp32", 500, 512, dict(a_dtype=F32, b_dtype=F32), ("exact", 0)),
    ("exact-600x1024-bf16", 600, 1024, {}, ("exact", 0)),
    ("exact-333x1280-bf16", 333, 1280, {}, ("exact", 0)),
    ("exact-700x100-bf16", 700, 100, {}, ("exact", 0)),
    # family-2 forward: one speculative fixed-shift sweep with its exact fallback, and the exact sweeps alone
    ("spec-1500x512-s100-flip", 1500, 512, dict(s=100.0, flip=True, speculate=True), ("pair", 2)),
    ("nospec-1500x512-s100-flip", 1500, 512, dict(s=100.0, flip=True, speculate=False,
                                                  env={"CLIPNCE_NO_SPECULATE": "1"}), ("pair", 2)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case_id,n,d,opt,expect", CASES, ids=[c[0] for c in CASES])
def test_route_rowwise(route_spy, monkeypatch, case_id, n, d, opt, expect):
    from clip_dplm_b200 import fused_clip_loss
    for k in ("CLIPNCE_BWD2_MIN_N", "CLIPNCE_BWD2_P", "CLIPNCE_BWD2_SEG", "CLIPNCE_SPLIT_STEPS", "CLIPNCE_NO_BWD2",
              "CLIPNCE_NO_GROUP", "CLIPNCE_NO_SPECULATE"):
        monkeypatch.delenv(k, raising=False)
    for k, v in opt.get("env", {}).items():
        monkeypatch.setenv(k, v)
    s, g = opt.get("s", 1 / 0.07), opt.get("g", G_UP)
    a_dt, b_dt = opt.get("a_dtype", BF16), opt.get("b_dtype", BF16)
    symmetric, extra_normalized = opt.get("symmetric", True), opt.get("extra_normalized", True)
    # every route but the grouped one can return the statistics; asking for them keeps a shape below 8192 rows off it
    stats = opt.get("stats", expect[0] != "group")
    a, b, extra = _inputs(n, d, seed=n + d, mix=opt.get("mix", 0.5), n_extra=opt.get("n_extra", 0),
                          extra_normalized=extra_normalized, flip=opt.get("flip", False),
                          fp32_rows=F32 in (a_dt, b_dt))
    ac = a.cuda().to(a_dt).requires_grad_(True)
    bc = b.cuda().to(b_dt).requires_grad_(True)
    ex = extra.cuda() if extra is not None else None
    t = torch.tensor(math.log(s), device="cuda", dtype=torch.float32, requires_grad=True)
    kw = dict(symmetric=symmetric, return_stats=stats)
    if ex is not None:
        kw.update(extra_cols=ex, extra_normalized=extra_normalized)
    with torch.autocast("cuda", dtype=BF16, enabled=opt.get("autocast", False)):
        out = fused_clip_loss(ac, bc, t, **kw)
    loss, st = out if stats else (out, None)
    (g * loss).backward()
    torch.cuda.synchronize()
    route = _route(route_spy)
    assert route[:2] == expect, f"{case_id}: served by {route}, expected {expect}"
    if "speculate" in opt:
        assert route[2] == opt["speculate"], f"{case_id}: speculative forward {route[2]}"

    compute = F32 if (a_dt == F32 and b_dt == F32 and not opt.get("autocast", False)) else BF16
    s_dev = float(t.detach().exp())        # the scale the kernels read
    ref = R.reference(ac.detach(), bc.detach(), s_dev, symmetric=symmetric, extra=ex, extra_normalized=extra_normalized,
                      g=g, compute_dtype=compute, u=R.U_TILE_F32 if expect[0] == "exact" else R.U_TILE_BF16)
    st = st or {}
    rep = R.check(ref, loss=loss.detach(), d_a=ac.grad, d_b=bc.grad, d_scale_sum=float(t.grad) / g,
                  row_lse=st.get("row_lse"), col_lse=st.get("col_lse"), diag=st.get("diag"))
    _check_report(rep, route, case_id)


# ------------------------------------------------------------------------------------------------------------------------
# row-sharded over two GPUs: every rank's rows against one global reference
# ------------------------------------------------------------------------------------------------------------------------
def _sharded_worker(rank, world, port, n, d, both, n_extra, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["CLIPNCE_COMM"] = "link"
    os.environ.setdefault("CLIPNCE_LINK_TIMEOUT_MS", "30000")
    if both:
        os.environ["CLIPNCE_BWD2_MIN_N"] = "256"
    else:
        os.environ["CLIPNCE_NO_BWD2"] = "1"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from clip_dplm_b200 import exchange, fused_clip_loss
        from clip_dplm_b200.engine import default_engine
        calls = _spy_engine(default_engine(), setattr)
        a, b, extra = _inputs(n, d, seed=n + d, mix=0.5, n_extra=n_extra)
        nl = n // world
        ac = a[rank * nl:(rank + 1) * nl].cuda().bfloat16().requires_grad_(True)
        bc = b[rank * nl:(rank + 1) * nl].cuda().bfloat16().requires_grad_(True)
        t = torch.tensor(math.log(1 / 0.07), device="cuda", requires_grad=True)
        loss, st = fused_clip_loss(ac, bc, t, group=dist.group.WORLD, return_stats=True,
                                   extra_cols=extra.cuda() if extra is not None else None)
        (G_UP * loss).backward()
        torch.cuda.synchronize()
        q.put((rank, float(loss.detach()), ac.grad.cpu(), bc.grad.cpu(), float(t.grad), float(t.detach().exp()),
               {k: v.cpu() for k, v in st.items()}, _route(calls)))
        exchange.reset()
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("n,d,both,n_extra,expect", [(8192, 512, True, 0, ("sharded", 1)),
                                                     (4096, 256, False, 700, ("pair", 1))],
                         ids=["two-sided-sharded", "peer-two-sweep-cache700"])
def test_row_sharded_rowwise(n, d, both, n_extra, expect):
    from tests.test_gpu_dist import _run
    world = 2
    out = _run(_sharded_worker, (24700 + (os.getpid() % 2000), n, d, both, n_extra), world)
    a, b, extra = _inputs(n, d, seed=n + d, mix=0.5, n_extra=n_extra)
    ref = R.reference(a.cuda().bfloat16(), b.cuda().bfloat16(), out[0][5], extra=extra.cuda() if extra is not None else None,
                      g=G_UP)
    nl = n // world
    for rank, loss, da, db, dt, _, st, route in out:
        assert route[:2] == expect, f"rank {rank}: served by {route}, expected {expect}"
        rep = R.check(ref, loss=loss, d_a=da.cuda(), d_b=db.cuda(), d_scale_sum=dt / G_UP, row_lse=st["row_lse"].cuda(),
                      col_lse=st["col_lse"].cuda(), diag=st["diag"].cuda(), row0=rank * nl)
        _check_report(rep, route, f"sharded-{n}x{d}-rank{rank}")
