"""The grouped launch of several pair problems and the projection-head tail, checked entry by entry against the float64
references of ``oracle/rowwise_modules.py`` -- each output against its own error budget, not a whole-matrix tolerance.

As in ``tests/test_rowwise.py``, the first part checks the checker without a GPU: a rounding emulation of each kernel
must pass with a margin, and planted faults of the kind these kernels can get wrong must be rejected with a margin.  The
second part runs the kernels on the GPU, and every case asserts which route served it."""
import math

import pytest
import torch

from oracle import rowwise as R
from oracle import rowwise_modules as M
from tests.test_gpu_modules import _tri_inputs
from tests.test_rowwise import _emulate, _route, _spy_engine

BF16, F32 = torch.bfloat16, torch.float32
TRI = ((0, 0, 1), (1, 2, 2))          # (cell, pert), (cell, protein), (pert, protein)
W_TRI = (0.7, 1.3, -0.4, 0.9)         # upstream weights of the three losses and of their sum


# ------------------------------------------------------------------------------------------------------------------------
# the group checker (CPU)
# ------------------------------------------------------------------------------------------------------------------------
def _emulate_group(members, xm, ym, s, gref, *, side_w=None, drop=None, col_pad=None, ds_coef=0.5, diag_from=None):
    """The grouped launch's arithmetic with only the rounding that matters: each problem's bf16 gradient tile
    (`test_rowwise._emulate`), the X and Y sides weighted by gscale and summed per member before the normalise backward
    (the finishing pass), the result rounded to the members' dtype; statistics and losses in fp32.

    Planted faults: side_w[(k, side)] replaces a side's weight; drop = (k, side, rows) removes one contribution from some
    rows; col_pad = k adds a zero column (S = 0) to problem k's column soft-max; ds_coef replaces the halving of the row
    dots; diag_from = (k, j): problem k's loss reads problem j's diagonal."""
    n_prob = len(xm)
    ems = []
    for k, (x, y) in enumerate(zip(xm, ym)):
        ref = gref["refs"][k]
        if col_pad == k:
            ref = dict(ref, col_lse=torch.logaddexp(ref["col_lse"], torch.zeros_like(ref["col_lse"])))
            ref["loss"] = ref["loss"] + (ref["col_lse"] - gref["refs"][k]["col_lse"]).sum() / (2 * ref["n"])
        ems.append(_emulate(members[x], members[y], s, ref))
    dhat = [torch.zeros(members[0].shape, dtype=torch.float64) for _ in members]
    ds = 0.0
    for k, (x, y) in enumerate(zip(xm, ym)):
        for side, m, part in ((0, x, ems[k]["d_ah"]), (1, y, ems[k]["d_bh"])):
            w = (side_w or {}).get((k, side), gref["g"][k])
            part = part * w
            ds += ds_coef * w * ems[k]["d_scale_sum"]
            if drop is not None and drop[:2] == (k, side):
                # the finishing pass takes sum G.S from the row dots of the summed parts: the dropped rows leave it too
                xc = R.staged(members[m], BF16)[2]
                ds -= ds_coef * float((xc[drop[2]] * part[drop[2]]).sum())
                part = part.clone()
                part[drop[2]] = 0
            dhat[m] += part
    grads, sq = [], []
    for m, mem in enumerate(members):
        x64, rinv, _ = R.staged(mem, BF16)
        d = R.normalize_backward(x64, rinv, dhat[m])
        sq.append(float(d.pow(2).sum()))
        grads.append(d.to(mem.dtype))
    losses = [float(e["loss"]) for e in ems]
    if diag_from is not None:
        k, j = diag_from
        losses[k] = float(torch.tensor(losses[k] + float((gref["refs"][k]["diag"] - gref["refs"][j]["diag"]).sum())
                                       / gref["n"], dtype=F32))
    losses.append(float(torch.tensor(sum(losses), dtype=F32)))
    return {"losses": torch.tensor(losses, dtype=torch.float64), "grads": grads, "d_scale": ds, "sumsq": sq,
            "stats": [(e["row_lse"], e["col_lse"], e["diag"]) for e in ems]}


def _group_report(gref, em):
    rep = M.group_check(gref, losses=em["losses"], grads=em["grads"], d_scale=em["d_scale"], sumsq=em["sumsq"])
    for k, (r, c, dg) in enumerate(em["stats"]):
        ref = gref["refs"][k]
        rep[f"row_lse{k}"] = {"max": float(((r - ref["row_lse"]).abs() / R.stat_budget(ref["row_lse"], ref["s_err"])).max()),
                              "worst": []}
        rep[f"col_lse{k}"] = {"max": float(((c - ref["col_lse"]).abs() / R.stat_budget(ref["col_lse"], ref["s_err"])).max()),
                              "worst": []}
    return rep


def _cpu_tri(n=300, d=128, mixes=(1.0, 0.5, 0.3)):
    return [x.bfloat16() for x in _tri_inputs(n, d, 11 + n, mixes=mixes)]


@pytest.mark.parametrize("s,mixes", [(14.3, (1.0, 0.5, 0.3)), (100.0, (1.0, 0.1, 0.05))], ids=["s14", "s100"])
def test_group_emulation_passes_with_margin(s, mixes):
    members = _cpu_tri(mixes=mixes)
    gref = M.group_reference(members, *TRI, s, W_TRI)
    rep = _group_report(gref, _emulate_group(members, *TRI, s, gref))
    assert M.worst_ratio(rep) <= 0.5, M.describe(rep, "group emulation")


def _group_faults(gref, n):
    k2 = int(gref["d"][2].norm(dim=1).argmax())
    blk = slice(k2 // 128 * 128, min(n, k2 // 128 * 128 + 128))
    return {
        "gscale_index": dict(side_w={(2, 1): gref["g"][0]}),    # problem 2's Y side weighted with problem 0's g
        "second_contribution_missing": dict(drop=(2, 1, blk)),    # protein's second contribution, one 128-row block
        "ds_not_halved": dict(ds_coef=1.0),
        "padding_column_leaks": dict(col_pad=1),                  # n % 256 != 0: a zero row's S = 0 in the soft-max
        "sumsq_wrong_member": "swap",
        "loss_reads_wrong_diag": dict(diag_from=(1, 0)),
    }


GROUP_FAULTS = list(_group_faults({"d": [torch.zeros(1, 1)] * 3, "g": [0.0] * 3}, 1))


@pytest.mark.parametrize("fault", GROUP_FAULTS)
def test_group_planted_fault_is_rejected(fault):
    s, n = 14.3, 300
    members = _cpu_tri(n)
    gref = M.group_reference(members, *TRI, s, W_TRI)
    kw = _group_faults(gref, n)[fault]
    em = _emulate_group(members, *TRI, s, gref, **(kw if isinstance(kw, dict) else {}))
    if kw == "swap":
        em["sumsq"][0], em["sumsq"][1] = em["sumsq"][1], em["sumsq"][0]
    rep = _group_report(gref, em)
    assert M.worst_ratio(rep) >= 10, M.describe(rep, fault)


API_CASES = [
    ("four-members-member3-idle", 4, (0, 1, 0), (1, 2, 2)),
    ("both-orders", 2, (0, 1), (1, 0)),
    ("self-pairs-6-of-8", 2, (0, 0, 1, 0), (0, 1, 0, 0)),
    ("self-pair-x4-8-contributions", 1, (0, 0, 0, 0), (0, 0, 0, 0)),
]
API_N, API_D = 1000, 256


def _api_members(n_members, n=API_N, d=API_D):
    """Members whose rows share one direction (besides a base common to the members' row i): a self-pair problem's
    off-diagonal cosines are then about 0.66, so its soft-max is not saturated and its gradient is resolved.  With
    independent rows the diagonal logit s stands alone, p_ii is about 1 and a self-pair's gradient lies below its budget,
    where no fault in its contributions could show."""
    g = torch.Generator().manual_seed(17)
    v = torch.randn(1, d, generator=g)
    base = torch.randn(n, d, generator=g)
    return [(v + 0.6 * base + 0.4 * torch.randn(n, d, generator=g)).bfloat16() for _ in range(n_members)]


def _api_weights(n_prob):
    return (0.7, 1.3, -0.4, 1.1)[:n_prob] + (0.9,)


@pytest.mark.parametrize("case_id,n_members,xm,ym", API_CASES, ids=[c[0] for c in API_CASES])
def test_group_problem_list_emulation_and_faults(case_id, n_members, xm, ym):
    """The problem lists of `test_group_problem_lists_rowwise`, on its inputs: the emulation passes with a margin, and the
    last problem's Y side -- in the self-pair lists a self-pair contribution of member 0, the 8th in the last list --
    missing from one 128-row block (the block of member 0's best-resolved row), or weighted with problem 0's g, is
    rejected.  In the self-pair lists the gradient alone resolves the missing block at 8.6 (8 contributions) and 10.5;
    d logit_scale, which the finishing pass takes from the row dots of the same summed parts, at 27.  A self pair's X and
    Y sides are equal, so a wrong weight on one of them moves the gradient by about 2 budgets and d logit_scale by 43."""
    s = 1 / 0.07
    members = _api_members(n_members)
    gref = M.group_reference(members, xm, ym, s, _api_weights(len(xm)))
    rep = _group_report(gref, _emulate_group(members, xm, ym, s, gref))
    assert M.worst_ratio(rep) <= 0.5, M.describe(rep, f"{case_id} emulation")
    k0 = int((gref["d"][0].norm(dim=1) / gref["budget"][0]).argmax())
    blk = slice(k0 // 128 * 128, min(API_N, k0 // 128 * 128 + 128))
    last = len(xm) - 1
    for fault, kw in (("block missing", dict(drop=(last, 1, blk))), ("gscale index", dict(side_w={(last, 1): gref["g"][0]}))):
        rep = _group_report(gref, _emulate_group(members, xm, ym, s, gref, **kw))
        assert M.worst_ratio(rep) >= 10, M.describe(rep, f"{case_id} {fault}")


# ------------------------------------------------------------------------------------------------------------------------
# the head-tail checker (CPU)
# ------------------------------------------------------------------------------------------------------------------------
def _head_inputs(n, k, p, *, seed=0, bias=True, offset=0.0, bias_spread=0.02, zero_row=None, dtype=BF16):
    g = torch.Generator().manual_seed(seed)
    h = torch.randn(n, k, generator=g)
    if zero_row is not None:
        h[zero_row] = 0
    w = (torch.rand(p, k, generator=g) * 2 - 1) / math.sqrt(k)
    b = offset + bias_spread * torch.randn(p, generator=g) if bias else None
    gamma = 0.5 + torch.rand(p, generator=g)
    beta = 0.6 * torch.rand(p, generator=g) - 0.3
    return h.to(dtype), w.to(dtype), b, gamma, beta


def _emulate_head(h, w, bias, gamma, beta, eps, *, fault=None):
    """fp32 torch in the kernel's order (acc + bias, mean, two-pass variance, rsqrt, (z - mean) rstd, z_hat gamma + beta)
    with round-to-nearest bf16 outputs."""
    hb, wb = h.bfloat16().float(), w.bfloat16().float()
    n, p = h.shape[0], w.shape[0]
    z = hb @ wb.T
    if bias is not None:
        z = z + bias.float()
    mean = z.sum(dim=1, keepdim=True) / p
    dev = z - mean
    var = (dev * dev).sum(dim=1, keepdim=True)
    rstd = torch.rsqrt(var / (p - 1 if fault == "variance_over_p_minus_1" else p)
                       + (0.0 if fault == "eps_ignored" else eps))
    if fault == "ragged_last_row_neighbour_rstd":
        rstd[n - 1] = rstd[n - 2]
    zh = dev * rstd
    be = beta.float().clone()
    if fault == "beta_missing_256_383":
        be[256:384] = 0
    e32 = zh * gamma.float() + be
    if fault == "e_round_toward_zero":
        e = (e32.view(torch.int32) & -65536).view(torch.float32).bfloat16()
    else:
        e = e32.bfloat16()
    rinv = 1.0 / e.float().norm(dim=1).clamp_min(1e-12)
    return {"e": e, "zhat": zh.bfloat16(), "rstd": rstd[:, 0], "rinv": rinv}


def _emulate_head_backward(em, de, w, h, gamma, *, fault=None):
    g = de.float() * gamma.float()
    zh = em["zhat"].float()
    m1 = g.mean(dim=1, keepdim=True)
    m2 = (g * zh).mean(dim=1, keepdim=True)
    dz32 = em["rstd"][:, None] * (g - m1 - (0 if fault == "dz_without_zhat_term" else zh * m2))
    dz = dz32.bfloat16()
    hb, wb = h.bfloat16().float(), w.bfloat16().float()
    d_gamma = (de.float() * (em["e"].float() if fault == "d_gamma_from_e" else zh)).sum(dim=0)
    return {"dz": dz, "d_h": (dz.float() @ wb).bfloat16(), "d_w": (dz.float().T @ hb).bfloat16(),
            "d_gamma": d_gamma, "d_beta": de.float().sum(dim=0), "d_bias": dz.float().sum(dim=0)}


def _head_report(h, w, bias, gamma, beta, eps, de, *, fault=None):
    ref = M.head_reference(h, w, bias, gamma, beta, eps)
    em = _emulate_head(h, w, bias, gamma, beta, eps, fault=fault)
    rep = M.head_check(ref, e=em["e"], zhat=em["zhat"], rstd=em["rstd"], rinv=em["rinv"])
    bw = _emulate_head_backward(em, de, w, h, gamma, fault=fault)
    dz_ref, eta = M.ln_backward_reference(de, em["zhat"], em["rstd"], gamma.float())
    rep.update(M.ln_backward_check(bw["dz"], dz_ref, eta))
    gref = M.head_grads_reference(ref, de, bias is not None)
    rep.update(M.head_grads_check(gref, d_h=bw["d_h"], d_w=bw["d_w"], d_gamma=bw["d_gamma"], d_beta=bw["d_beta"],
                                  d_bias=bw["d_bias"] if bias is not None else None))
    return rep


HEAD_CPU = dict(n=300, k=128, p=384)     # three CTAs, the last one ragged (44 rows); the 256 + 128 column chunks


@pytest.mark.parametrize("de_dtype", [BF16, F32])
@pytest.mark.parametrize("variant", ["bias", "nobias", "offset30"])
def test_head_emulation_passes_with_margin(variant, de_dtype):
    n, k, p = HEAD_CPU.values()
    h, w, b, gamma, beta = _head_inputs(n, k, p, bias=variant != "nobias", offset=30.0 if variant == "offset30" else 0.0,
                                        zero_row=3)
    de = torch.randn(n, p, generator=torch.Generator().manual_seed(1)).to(de_dtype)
    rep = _head_report(h, w, b, gamma, beta, 1e-5, de)
    assert M.worst_ratio(rep) <= 0.5, M.describe(rep, "head emulation")


HEAD_FAULTS = ["e_round_toward_zero", "beta_missing_256_383", "variance_over_p_minus_1", "eps_ignored",
               "ragged_last_row_neighbour_rstd", "dz_without_zhat_term", "d_gamma_from_e"]


@pytest.mark.parametrize("fault", HEAD_FAULTS)
def test_head_planted_fault_is_rejected(fault):
    n, k, p = HEAD_CPU.values()
    # row 3 is h = 0: its z is the bias (spread 0.02, variance 4e-4), a low-variance row where eps = 1e-5 matters
    h, w, b, gamma, beta = _head_inputs(n, k, p, zero_row=3)
    de = torch.randn(n, p, generator=torch.Generator().manual_seed(1)).bfloat16()
    rep = _head_report(h, w, b, gamma, beta, 1e-5, de, fault=fault)
    assert M.worst_ratio(rep) >= 10, M.describe(rep, fault)


# ------------------------------------------------------------------------------------------------------------------------
# the grouped launch on the GPU
# ------------------------------------------------------------------------------------------------------------------------
ENV_HOOKS = ("CLIPNCE_NO_SPECULATE", "CLIPNCE_NO_GROUP", "CLIPNCE_SPLIT_STEPS")


@pytest.fixture
def group_spy(monkeypatch):
    """Route spy of `test_rowwise` plus a record of every `group_forward` call (arguments and returned statistics)."""
    from clip_dplm_b200.engine import default_engine
    for k in ENV_HOOKS:
        monkeypatch.delenv(k, raising=False)
    eng = default_engine()
    calls = _spy_engine(eng, monkeypatch.setattr)
    fwd = []
    spied = eng.group_forward
    raw = type(eng).group_forward.__get__(eng)

    def record(*args, **kw):
        out = spied(*args, **kw)
        fwd.append((args, kw, out))
        return out
    monkeypatch.setattr(eng, "group_forward", record)
    return {"calls": calls, "fwd": fwd, "raw_forward": raw}


def _assert_group_route(spy, n_prob, family, case_id):
    route = _route(spy["calls"])
    assert route[:2] == ("group", family), f"{case_id}: served by {route}"
    assert len(spy["fwd"]) == 1, f"{case_id}: {len(spy['fwd'])} group_forward calls"
    x_member = spy["fwd"][0][0][3]
    assert len(x_member) == n_prob, f"{case_id}: group_forward with {len(x_member)} problems"
    assert any(c["call"] == "group_backward" for c in spy["calls"]), f"{case_id}: no group_backward"
    return route


def _stats_of(spy):
    args, _, (stat_m, stat_l, diag, _loss) = spy["fwd"][0]
    stack, n_members = args[0], args[2]
    return stat_m, stat_l, diag, stack.shape[0] // n_members


def _report_and_assert(rep, case_id, route):
    print(f"\nRATIOS {case_id} route={route} " + " ".join(f"{k}={v['max']:.3g}" for k, v in rep.items()))
    assert M.worst_ratio(rep) <= 1.0, M.describe(rep, f"{case_id} {route}")


def _flip_members(n, d):
    """One direction for every row, so every logit is near +-s; rows 5, 77, n - 3 of the cell member reversed: at s = 100
    their row sums underflow the speculative sweep's lowered shift and force the exact fallback."""
    g = torch.Generator().manual_seed(n + d)
    v = torch.nn.functional.normalize(torch.randn(1, d, generator=g), dim=-1)
    out = [(v * 8.0 + 0.25 * torch.randn(n, d, generator=g)).bfloat16().float() for _ in range(3)]
    out[0][[5, 77, n - 3]] *= -1
    return out


TRI_CASES = [
    ("tri-255x128", 255, 128, {}, 1),
    ("tri-257x256", 257, 256, {}, 1),
    ("tri-1000x512", 1000, 512, {}, 1),
    ("tri-4095x768", 4095, 768, {}, 1),
    ("tri-8191x512", 8191, 512, {}, 1),
    ("tri-2048x384-s100", 2048, 384, dict(s=100.0, mixes=(1.0, 0.1, 0.05), fallback=False), 2),
    ("tri-1500x512-s100-flip", 1500, 512, dict(s=100.0, flip=True, fallback=True), 2),
    ("tri-1500x512-s100-nospec", 1500, 512, dict(s=100.0, flip=True, env={"CLIPNCE_NO_SPECULATE": "1"}), 2),
    ("tri-2048x512-fp32-autocast", 2048, 512, dict(dtype=F32), 1),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case_id,n,d,opt,family", TRI_CASES, ids=[c[0] for c in TRI_CASES])
def test_trimodal_group_rowwise(group_spy, monkeypatch, case_id, n, d, opt, family):
    from clip_dplm_b200 import modules as Mod
    for k, v in opt.get("env", {}).items():
        monkeypatch.setenv(k, v)
    s, dtype = opt.get("s", 1 / 0.07), opt.get("dtype", BF16)
    rows = _flip_members(n, d) if opt.get("flip") else _tri_inputs(n, d, 11 + n, mixes=opt.get("mixes", (1.0, 0.5, 0.3)))
    embs = [x.cuda().to(dtype).requires_grad_(True) for x in rows]
    t = torch.tensor(math.log(s), device="cuda", requires_grad=True)
    with torch.autocast("cuda", dtype=BF16, enabled=dtype == F32):
        out = Mod.trimodal_contrastive_losses(*embs, t)
    losses = [out["cell_pert_loss"], out["cell_protein_loss"], out["pert_protein_loss"], out["loss"]]
    sum(w * l for w, l in zip(W_TRI, losses)).backward()
    torch.cuda.synchronize()
    route = _assert_group_route(group_spy, 3, family, case_id)
    if family == 2:
        assert route[2] == ("env" not in opt), f"{case_id}: speculative forward {route[2]}"

    s_dev = float(t.detach().exp())
    gref = M.group_reference([e.detach() for e in embs], *TRI, s_dev, W_TRI)
    rep = M.group_check(gref, losses=torch.stack([l.detach() for l in losses]), grads=[e.grad for e in embs],
                        d_scale=float(t.grad), sumsq=out.grad_info["embed_grad_sumsq"], stats=_stats_of(group_spy))
    for e in embs:
        assert e.grad.dtype == dtype
    _report_and_assert(rep, case_id, route)

    if "fallback" in opt:
        # when the gated exact sweeps run they write every statistic, exactly as with speculation off
        # (valid rows only: nothing reads the statistics of the padding rows)
        args, kw, (stat_m, stat_l, _, _) = group_spy["fwd"][0]
        monkeypatch.setenv("CLIPNCE_NO_SPECULATE", "1")
        m2, l2, _, _ = group_spy["raw_forward"](*args, **kw)
        torch.cuda.synchronize()
        n_pad = args[0].shape[0] // args[2]
        valid = torch.cat([torch.arange(k * n_pad, k * n_pad + n) for k in range(3)]).cuda()
        same = torch.equal(stat_m[:, valid], m2[:, valid]) and torch.equal(stat_l[:, valid], l2[:, valid])
        assert same == opt["fallback"], f"{case_id}: statistics bit-identical to the exact sweeps: {same}"


@pytest.mark.gpu
@pytest.mark.parametrize("weights,zero", [((0.0, 1.0, 0.0, 0.0), 1), ((0.0, 0.0, 1.0, 0.0), 0)],
                         ids=["only-cell-protein", "only-pert-protein"])
def test_group_weight_isolation(group_spy, weights, zero):
    """With one problem weighted, the member outside it gets exactly zero: a wrong gscale index or cshift shows here."""
    from clip_dplm_b200 import modules as Mod
    n, d = 1000, 256
    embs = [x.cuda().bfloat16().requires_grad_(True) for x in _tri_inputs(n, d, 5)]
    t = torch.tensor(math.log(1 / 0.07), device="cuda", requires_grad=True)
    out = Mod.trimodal_contrastive_losses(*embs, t)
    losses = [out["cell_pert_loss"], out["cell_protein_loss"], out["pert_protein_loss"], out["loss"]]
    sum(w * l for w, l in zip(weights, losses)).backward()
    torch.cuda.synchronize()
    route = _assert_group_route(group_spy, 3, 1, "isolation")
    assert torch.count_nonzero(embs[zero].grad) == 0
    assert float(out.grad_info["embed_grad_sumsq"][zero]) == 0.0
    gref = M.group_reference([e.detach() for e in embs], *TRI, float(t.detach().exp()), weights)
    rep = M.group_check(gref, losses=torch.stack([l.detach() for l in losses]), grads=[e.grad for e in embs],
                        d_scale=float(t.grad), sumsq=out.grad_info["embed_grad_sumsq"])
    _report_and_assert(rep, f"isolation-{zero}", route)




@pytest.mark.gpu
@pytest.mark.parametrize("case_id,n_members,xm,ym", API_CASES, ids=[c[0] for c in API_CASES])
def test_group_problem_lists_rowwise(group_spy, case_id, n_members, xm, ym):
    """Problem lists `fused_clip_loss_group` accepts that the models do not use: a member in no problem (the finishing
    pass's n_slabs == 0 side), both orders of one pair, and self-pairs up to FINISH_CONTRIB = 8 contributions."""
    from clip_dplm_b200.functional import fused_clip_loss_group
    embs = [x.cuda().requires_grad_(True) for x in _api_members(n_members)]
    t = torch.tensor(math.log(1 / 0.07), device="cuda", requires_grad=True)
    weights = _api_weights(len(xm))
    holder = {}
    losses = fused_clip_loss_group(embs, xm, ym, t, holder=holder)
    assert losses is not None, f"{case_id}: the grouped launch did not serve the problem list"
    (losses * torch.tensor(weights, device="cuda")).sum().backward()
    torch.cuda.synchronize()
    route = _assert_group_route(group_spy, len(xm), 1, case_id)
    if n_members == 4:
        assert embs[3].grad is not None and torch.count_nonzero(embs[3].grad) == 0
        assert float(holder["embed_grad_sumsq"][3]) == 0.0
    gref = M.group_reference([e.detach() for e in embs], xm, ym, float(t.detach().exp()), weights)
    rep = M.group_check(gref, losses=losses.detach(), grads=[e.grad for e in embs], d_scale=float(t.grad),
                        sumsq=holder["embed_grad_sumsq"], stats=_stats_of(group_spy))
    _report_and_assert(rep, case_id, route)


@pytest.mark.gpu
def test_group_returns_none_past_its_member_and_problem_limits():
    """More than 4 members or 4 problems: the library has no finishing side / virtual problem slot for them, and the API
    says so by returning None (one `fused_clip_loss` per pair) instead of raising."""
    from clip_dplm_b200.functional import fused_clip_loss_group
    embs = [torch.randn(256, 128, device="cuda").bfloat16() for _ in range(5)]
    t = torch.tensor(2.6592, device="cuda")
    assert fused_clip_loss_group(embs, (0, 1, 2, 3), (1, 2, 3, 4), t) is None
    assert fused_clip_loss_group(embs[:2], (0, 0, 0, 1, 1), (1, 1, 1, 0, 0), t) is None
    assert fused_clip_loss_group(embs[:4], (0, 1, 2, 3), (1, 2, 3, 0), t) is not None


# ------------------------------------------------------------------------------------------------------------------------
# the projection-head tail on the GPU
# ------------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def head_calls(monkeypatch):
    from clip_dplm_b200.engine import default_engine
    lib = default_engine().lib
    count = {"clipnce_head_tail": 0, "clipnce_head_tail_backward": 0}
    for name in count:
        fn = getattr(lib, name)

        def wrap(*a, _fn=fn, _name=name):
            count[_name] += 1
            return _fn(*a)
        monkeypatch.setattr(lib, name, wrap)
    return count


def _direct_ln_backward(de, zhat, rstd, gamma):
    import ctypes
    from clip_dplm_b200 import _lib
    from clip_dplm_b200.engine import default_engine
    n, p = zhat.shape
    dz = torch.empty((n, p), dtype=BF16, device=de.device)
    ptr = lambda x: ctypes.c_void_p(x.data_ptr())
    _lib.check(default_engine().lib.clipnce_head_tail_backward(
        ptr(de), _lib.BF16 if de.dtype == BF16 else _lib.F32, ptr(zhat), ptr(rstd), ptr(gamma), n, p, ptr(dz),
        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "head_tail_backward")
    return dz


def _head_modules(k, p, *, bias, eps, dtype, offset=0.0, beta_zero=False, seed=7):
    torch.manual_seed(seed)
    lin = torch.nn.Linear(k, p, bias=bias).cuda()
    ln = torch.nn.LayerNorm(p, eps=eps).cuda()
    with torch.no_grad():
        ln.weight.uniform_(0.5, 1.5)
        if beta_zero:
            ln.bias.zero_()
        else:
            ln.bias.uniform_(-0.3, 0.3)
        if bias:
            lin.bias.add_(offset)
        if dtype == BF16:
            lin.to(BF16)
            ln.to(BF16)
    return lin, ln


def _check_head(lin, ln, h, de, case_id):
    """The tail through `heads.fused_linear_layernorm` and its autograd backward with upstream ``de``, then the LayerNorm
    backward kernel called directly with fp32 and bf16 de."""
    from clip_dplm_b200.heads import fused_linear_layernorm
    e, rinv = fused_linear_layernorm(h, lin, ln)
    _hb, _wb, zhat, rstd, g32 = e.grad_fn.saved_tensors
    ref = M.head_reference(h.detach(), lin.weight, lin.bias, ln.weight, ln.bias, ln.eps)
    rep = M.head_check(ref, e=e.detach(), zhat=zhat, rstd=rstd, rinv=rinv)
    e.backward(de)
    torch.cuda.synchronize()
    gref = M.head_grads_reference(ref, de, lin.bias is not None)
    rep.update(M.head_grads_check(gref, d_h=h.grad, d_w=lin.weight.grad, d_gamma=ln.weight.grad, d_beta=ln.bias.grad,
                                  d_bias=lin.bias.grad if lin.bias is not None else None))
    for dt in (F32, BF16):
        de_t = de.float() * (1 + 1e-3 * torch.randn_like(de.float())) if dt == F32 else de   # fp32 de off the bf16 grid
        dz = _direct_ln_backward(de_t.contiguous(), zhat, rstd, g32)
        dz_ref, eta = M.ln_backward_reference(de_t, zhat, rstd, g32)
        rep.update({f"{k}-{'f32' if dt == F32 else 'bf16'}de": v for k, v in M.ln_backward_check(dz, dz_ref, eta).items()})
    _report_and_assert(rep, case_id, "head")
    return e, rinv, zhat, rstd


HEAD_CASES = [
    ("head-1x64x128", 1, 64, 128, {}),
    ("head-127x320x256-nobias", 127, 320, 256, dict(bias=False)),
    ("head-129x1280x384", 129, 1280, 384, {}),
    ("head-8192x1280x512", 8192, 1280, 512, {}),
    ("head-4097x2560x512", 4097, 2560, 512, {}),
    ("head-1000x640x128-eps1e-12-zero-row", 1000, 640, 128, dict(eps=1e-12, bias=False, beta_zero=True, zero_row=True)),
    ("head-1000x640x128-offset30", 1000, 640, 128, dict(offset=30.0)),
    ("head-513x640x384-fp32", 513, 640, 384, dict(dtype=F32)),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case_id,n,k,p,opt", HEAD_CASES, ids=[c[0] for c in HEAD_CASES])
def test_head_tail_rowwise(head_calls, case_id, n, k, p, opt):
    dtype = opt.get("dtype", BF16)
    lin, ln = _head_modules(k, p, bias=opt.get("bias", True), eps=opt.get("eps", 1e-5), dtype=dtype,
                            offset=opt.get("offset", 0.0), beta_zero=opt.get("beta_zero", False))
    g = torch.Generator(device="cuda").manual_seed(n + k)
    h = torch.randn(n, k, device="cuda", generator=g)
    if dtype == F32:   # fp32 operands the kernel reads rounded to bf16
        assert not torch.equal(h, h.bfloat16().float()) and not torch.equal(lin.weight, lin.weight.bfloat16().float())
    if opt.get("zero_row"):
        h[n // 2] = 0
    h = h.to(dtype).requires_grad_(True)
    de = torch.randn(n, p, device="cuda", generator=g).bfloat16()
    e, rinv, _, _ = _check_head(lin, ln, h, de, case_id)
    assert head_calls == {"clipnce_head_tail": 1, "clipnce_head_tail_backward": 3}, head_calls
    if opt.get("zero_row"):
        assert torch.count_nonzero(e[n // 2]) == 0 and float(rinv[n // 2]) == pytest.approx(1e12, rel=1e-6)


@pytest.mark.gpu
def test_projection_head_pair_into_fused_loss_rowwise(head_calls, route_spy, monkeypatch):
    """The product chain at 8192 rows: two bf16 ProjectionHeads with the fused tail hand their rows and 1/norm to
    `fused_clip_loss`.  Checked in two steps so that the budgets do not compound: the loss and dE against
    `rowwise.reference` on the heads' own e, then each head's backward against the head reference with de = dE."""
    from clip_dplm_b200 import heads, modules as Mod
    from clip_dplm_b200 import fused_clip_loss
    n, k, p = 8192, 1280, 512
    tails = []
    orig = heads.fused_linear_layernorm

    def record(h, lin, ln):
        h.retain_grad()
        e, rinv = orig(h, lin, ln)
        tails.append((h, lin, ln, e))
        return e, rinv
    monkeypatch.setattr(heads, "fused_linear_layernorm", record)
    torch.manual_seed(11)
    ph = [Mod.ProjectionHead(k, p, k).cuda().bfloat16().eval() for _ in range(2)]
    x = [torch.randn(n, k, device="cuda").bfloat16() for _ in range(2)]
    ea, eb = ph[0](x[0]), ph[1](x[1])
    assert len(tails) == 2 and head_calls["clipnce_head_tail"] == 2
    ea.retain_grad()
    eb.retain_grad()
    t = torch.tensor(math.log(1 / 0.07), device="cuda", requires_grad=True)
    loss = fused_clip_loss(ea, eb, t, rinv_a=ea._clipnce_rinv, rinv_b=eb._clipnce_rinv)
    g = 0.37
    (g * loss).backward()
    torch.cuda.synchronize()
    route = _route(route_spy)
    assert route[:2] == ("pair", 1), f"served by {route}"
    assert head_calls["clipnce_head_tail_backward"] == 2
    ref = R.reference(ea.detach(), eb.detach(), float(t.detach().exp()), g=g)
    rep = R.check(ref, loss=loss.detach(), d_a=ea.grad, d_b=eb.grad, d_scale_sum=float(t.grad) / g)
    for side, (h, lin, ln, e) in zip("ab", tails):
        hr = M.head_reference(h.detach(), lin.weight, lin.bias, ln.weight, ln.bias, ln.eps)
        rep.update({f"{kk}-{side}": v for kk, v in M.head_check(hr, e=e.detach()).items()})
        gref = M.head_grads_reference(hr, e.grad, True)
        rep.update({f"{kk}-{side}": v for kk, v in M.head_grads_check(
            gref, d_h=h.grad, d_w=lin.weight.grad, d_gamma=ln.weight.grad, d_beta=ln.bias.grad, d_bias=lin.bias.grad).items()})
    _report_and_assert(rep, "product-chain-8192x1280x512", route)


@pytest.fixture
def route_spy(monkeypatch):
    from clip_dplm_b200.engine import default_engine
    return _spy_engine(default_engine(), monkeypatch.setattr)
