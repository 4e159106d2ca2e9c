"""Float64 references with per-entry error budgets for the two kernel paths the models run besides `fused_clip_loss`: the
grouped launch of several pair problems (``clipnce_group_*``, `functional.fused_clip_loss_group`) and the projection-head
tail (``head::linear_ln_kernel`` + ``head::ln_backward_rows``, `heads.fused_linear_layernorm`).  TEST INFRASTRUCTURE ONLY
(same rule as ``oracle/rowwise.py``, whose budgets the group reuses).

Every check returns {name: {"max": largest error / budget, "worst": [(index, ratio), ...]}}; it passes when every max is
<= 1.  An entry whose error is exactly zero has ratio 0 even when its budget is zero (a member in no problem, a zero row),
and any other error against a zero budget is infinite.

Group.  Problem k is one symmetric pair whose loss reaches the caller with upstream weight g_k = w_k + w_sum (every loss
also feeds the sum).  Its reference is `rowwise.reference` with g = g_k.  A member's gradient is the sum of the d_a of the
problems where it is the row operand and the d_b of those where it is the column operand, and its budget is the sum of
their budgets.  d logit_scale = sum_k g_k sum(G.S)_k with budget sum_k |g_k| budget_k.  Each loss gets
`rowwise.stat_budget`; their sum gets the sum of those budgets.

Head tail.  e = LayerNorm(h W^T + b) gamma + beta on the bf16-rounded h and W (what the kernel reads), in float64.  The
kernel's fp32 arithmetic is bounded to first order, per row (one line per term):

    dz_c   = (K/16 + 1) 2^-23 sum_k |h_k W_ck|     the tensor cores' accumulator: at most K/16 + 1 additions, one-signed
             + 2^-24 |z_c|                          the bias add
    dmu    = mean_c dz_c + 2^-24 sum_c |z_c|        mean of the computed z: a p-term fp32 sum, each partial <= sum |z|
    dss    = sum_c 2 |z_c - mu| (dz_c + dmu + 2^-23 (|z_c| + |z_c - mu|))     squares of the computed deviations
             + p 2^-24 sum_c (z_c - mu)^2 + p dmu^2                           the p-term fmaf chain; second order
    drstd  = dss / (2 (ss + p eps)) + 2^-24 + 2 2^-23    relative: var / p + eps, and rsqrtf (<= 2 ulp)
    eta_zh = rstd (dz_c + dmu) + |zh_c| (drstd + 2 2^-24)                     (z - mu) rstd: two roundings
    eta_e  = |gamma_c| eta_zh + 2^-24 (|zh_c gamma_c| + |e_c|)                 fmaf, or a product and a sum

e and z_hat are stored in bf16: an entry is allowed a bf16 ulp of the reference plus eta (a factor 2 over the half ulp
that round-to-nearest can take, as rowwise.u_out), and wherever the reference lies more than eta from a bf16 rounding
boundary the kernel's entry must equal bf16(reference) exactly (the "exact" outputs: ratio |got - bf16(ref)| / (margin -
eta), which is >= 2 for any other bf16 value).  The exact rule is what sees a wrong rounding mode: a value rounded the
wrong way is still within one ulp.  rstd gets drstd
relative.  rinv = 1 / max(|e|, 1e-12) of the kernel's OWN bf16 row (what the loss kernels see), to (p + 4) 2^-24
relative.

LayerNorm backward dz = rstd (g - mean(g) - z_hat mean(g z_hat)), g = de gamma, is checked on the kernel's own de, z_hat,
rstd and gamma with the same exact-where-decidable rule, eta_dz from the fp32 products, the two lane-strided sums
((p/32 + 5) additions each) and the final expression.

The parameter and input gradients of `heads._LinearLayerNorm.backward` are checked against float64 autograd of the exact
math.  Their budgets carry, per entry of dz, an independent part (half a bf16 ulp of dz; the bf16 rounding of z_hat through
rstd mean(g z_hat)) that adds in quadrature (C_RAND_HEAD) and a one-signed part (eta_dz, eta_zh through the
same term, z_hat's share of mean(g z_hat), drstd |dz|) that adds linearly; then the fp32 accumulators of the two bf16
GEMMs ((K/16 + 1) 2^-23 of the absolute products), their bf16 output (2^-8 of the row, as rowwise.u_out) and the rounding
to the parameter dtype.  The column sums (d_gamma, d_beta, d_bias) get C_RAND_HEAD sqrt(n) 2^-24 of the summed magnitudes for
their fp32 sum.
"""
from __future__ import annotations

import torch

from . import rowwise as R

U32 = 2.0 ** -24
F64 = torch.float64
# quadrature constant of the head gradients' independent roundings.  A uniform rounding error has an RMS of half its bound
# over sqrt(3), so C sqrt(sum bound^2) is C sqrt(3) standard deviations: rowwise.C_RAND = 4 (6.9 sigma) left the rounding
# emulation at 0.51 of one d_gamma entry among 2304 (a 3.6 sigma column); 6 is 10.4 sigma
C_RAND_HEAD = 6.0


def _ratio(err, budget):
    r = err / budget
    r = torch.where(err == 0, torch.zeros_like(r), r)
    return torch.where(torch.isnan(r), torch.full_like(r, float("inf")), r)


def _put(out, name, ratio, index_of=None):
    r = ratio.flatten()
    if r.numel() == 0:
        out[name] = {"max": 0.0, "worst": []}
        return
    top = torch.topk(r, min(5, r.numel()))
    worst = [(int(i), float(v)) for v, i in zip(top.values.cpu(), top.indices.cpu())]
    if index_of is not None:
        worst = [(index_of(i), v) for i, v in worst]
    out[name] = {"max": float(r.max()), "worst": worst}


def worst_ratio(report):
    return max(r["max"] for r in report.values())


def describe(report, title=""):
    lines = [title] if title else []
    for name, r in report.items():
        lines.append(f"{name}: max ratio {r['max']:.3g}; worst " + ", ".join(f"{i} {v:.3g}" for i, v in r["worst"]))
    return "\n".join(lines)


# ------------------------------------------------------------------------------------------------------------------------
# the grouped launch
# ------------------------------------------------------------------------------------------------------------------------
def group_reference(members, x_member, y_member, s, weights, *, block=4096):
    """members: [N,d] rows (any float type); problem k pairs members[x_member[k]] (rows) with members[y_member[k]]
    (columns); weights: the n_prob + 1 upstream gradients of the losses and of their sum.

    -> dict: refs (one `rowwise.reference` per problem), g [n_prob], loss [n_prob + 1], loss_budget [n_prob + 1],
    d [member] and budget [member] (per row), d_scale (sum_k g_k sum G.S_k, what d logit_scale is), budget_d_scale."""
    n_prob = len(x_member)
    g = [float(weights[k]) + float(weights[n_prob]) for k in range(n_prob)]
    refs = [R.reference(members[x], members[y], s, g=g[k], block=block)
            for k, (x, y) in enumerate(zip(x_member, y_member))]
    n, d = members[0].shape
    dev = members[0].device
    grads = [torch.zeros(n, d, dtype=F64, device=dev) for _ in members]
    budgets = [torch.zeros(n, dtype=F64, device=dev) for _ in members]
    for k, (x, y) in enumerate(zip(x_member, y_member)):
        grads[x] += refs[k]["d_a"]
        budgets[x] += refs[k]["budget_a"]
        grads[y] += refs[k]["d_b"]
        budgets[y] += refs[k]["budget_b"]
    losses = torch.stack([r["loss"] for r in refs])
    loss_budget = torch.stack([R.stat_budget(r["loss"], r["s_err"]) for r in refs])
    return {"refs": refs, "g": g, "loss": torch.cat([losses, losses.sum().reshape(1)]),
            "loss_budget": torch.cat([loss_budget, loss_budget.sum().reshape(1)]), "d": grads, "budget": budgets,
            "d_scale": sum(gk * r["d_scale_sum"] for gk, r in zip(g, refs)),
            "budget_d_scale": sum(abs(gk) * r["budget_d_scale"] for gk, r in zip(g, refs)), "n": n}


def sumsq_own_tolerance(sq_own, out_dtype, d):
    """|embed_grad_sumsq - |dx|^2 of the returned rows|: the output rounding (bf16 rounds each entry by at most 2^-8 of
    itself, so |round(o)|^2 - |o|^2 <= 2^-7 |o|^2 to first order) and the fp32 sum of squares (a d/32-term fmaf chain per
    lane, then trees)."""
    u = 2.0 ** -7 * 1.01 if out_dtype == torch.bfloat16 else 0.0
    return (u + (d / 32 + 8) * U32) * sq_own


def group_check(ref, *, losses=None, grads=None, d_scale=None, sumsq=None, stats=None):
    """losses [n_prob + 1]; grads: per member [N,d]; d_scale: d logit_scale; sumsq: embed_grad_sumsq [members];
    stats: (stat_m, stat_l, diag, n_pad) of `engine.group_forward` (row / column statistics of problem k at
    [k n_pad, k n_pad + n))."""
    out = {}
    n = ref["n"]
    if losses is not None:
        got = torch.as_tensor(losses).to(device=ref["loss"].device, dtype=F64).reshape(-1)
        _put(out, "loss", _ratio((got - ref["loss"]).abs(), ref["loss_budget"]))
    if grads is not None:
        for m, (gm, want, bud) in enumerate(zip(grads, ref["d"], ref["budget"])):
            err = (gm.to(device=want.device, dtype=F64) - want).norm(dim=1)
            _put(out, f"d{m}", _ratio(err, bud), lambda i: f"row {i} (block {i // 128})")
    if d_scale is not None:
        err = torch.as_tensor(abs(float(d_scale) - float(ref["d_scale"])), dtype=F64)
        _put(out, "d_scale", _ratio(err, torch.as_tensor(float(ref["budget_d_scale"]), dtype=F64)))
    if sumsq is not None:
        sq = torch.as_tensor(sumsq).to(dtype=F64).cpu()
        own, tol_own, vs_ref, tol_ref = [], [], [], []
        for m, (gm, want, bud) in enumerate(zip(grads, ref["d"], ref["budget"])):
            o = float(gm.double().pow(2).sum())
            t = float(sumsq_own_tolerance(o, gm.dtype, gm.shape[1]))
            b2, w = float(bud.pow(2).sum().sqrt()), float(want.norm())
            own.append(abs(float(sq[m]) - o))
            tol_own.append(t)
            vs_ref.append(abs(float(sq[m]) - w * w))
            tol_ref.append(2 * w * b2 + b2 * b2 + t)
        _put(out, "sumsq_own", _ratio(torch.tensor(own, dtype=F64), torch.tensor(tol_own, dtype=F64)))
        _put(out, "sumsq_ref", _ratio(torch.tensor(vs_ref, dtype=F64), torch.tensor(tol_ref, dtype=F64)))
    if stats is not None:
        stat_m, stat_l, diag, n_pad = stats
        lse = stat_m.double() + stat_l.double().log()
        for k, r in enumerate(ref["refs"]):
            rows = slice(k * n_pad, k * n_pad + n)
            dev = r["row_lse"].device
            for name, got, want in (("row_lse", lse[0, rows], r["row_lse"]), ("col_lse", lse[1, rows], r["col_lse"]),
                                    ("diag", diag[rows].double(), r["diag"])):
                got = got.to(dev)
                _put(out, f"{name}{k}", _ratio((got - want).abs(), R.stat_budget(want, r["s_err"])))
    return out


# ------------------------------------------------------------------------------------------------------------------------
# bf16 rounding geometry
# ------------------------------------------------------------------------------------------------------------------------
def bf16_half_ulp(v):
    """Half the bf16 spacing at |v| (float64 in, float64 out)."""
    a = v.abs().clamp_min(2.0 ** -126)
    return torch.exp2(torch.floor(torch.log2(a)) - 8)


def bf16_round_margin(v):
    """-> (bf16(v) as float64, distance of v to the nearer bf16 rounding boundary)."""
    r16 = v.to(torch.float32).to(torch.bfloat16)   # the f32 step moves v by <= 2^-24 |v| <= every eta below
    r = r16.double()
    bits = r16.view(torch.int16).to(torch.int32)
    out = (bits + 1).to(torch.int16).view(torch.bfloat16).double()        # next value of larger magnitude
    inn = torch.where(r == 0, -out, (bits - 1).to(torch.int16).view(torch.bfloat16).double())
    margin = torch.minimum((v - 0.5 * (r + out)).abs(), (v - 0.5 * (r + inn)).abs())
    return r, margin


def _rounded_check(out, name, got, want, eta, index_of=None):
    """The plain budget (a bf16 ulp + eta) as ``name`` and the exact-where-decidable rule as ``name``_exact."""
    got = got.to(device=want.device, dtype=F64)
    _put(out, name, _ratio((got - want).abs(), 2 * bf16_half_ulp(want.abs() + eta) + eta), index_of)
    r, margin = bf16_round_margin(want)
    decidable = margin > eta
    ratio = torch.where(decidable, _ratio((got - r).abs(), (margin - eta).clamp_min(1e-300)), torch.zeros_like(want))
    _put(out, name + "_exact", ratio, index_of)


def _entry(p):
    return lambda i: f"({i // p}, {i % p})"


# ------------------------------------------------------------------------------------------------------------------------
# the projection-head tail
# ------------------------------------------------------------------------------------------------------------------------
def head_reference(h, weight, bias, gamma, beta, eps):
    """Forward of the tail on what the kernel reads (h, W rounded to bf16; bias, gamma, beta in fp32), float64, with the
    first-order fp32 bounds of the module docstring.  -> dict of float64 tensors."""
    hb = h.detach().to(torch.bfloat16).double()
    wb = weight.detach().to(torch.bfloat16).double()
    n, k = hb.shape
    p = wb.shape[0]
    z = hb @ wb.T
    if bias is not None:
        z = z + bias.detach().float().double()
    ga = gamma.detach().float().double()
    be = beta.detach().float().double()
    mu = z.mean(dim=1, keepdim=True)
    dev = z - mu
    ss = dev.square().sum(dim=1, keepdim=True)
    eps32 = float(torch.tensor(eps, dtype=torch.float32))
    rstd = 1.0 / (ss / p + eps32).sqrt()
    zh = dev * rstd
    e = zh * ga + be
    acc = (hb.abs() @ wb.abs().T)
    dz = (k / 16 + 1) * 2.0 ** -23 * acc + U32 * z.abs()
    dmu = dz.mean(dim=1, keepdim=True) + U32 * z.abs().sum(dim=1, keepdim=True)
    dss = ((2 * dev.abs() * (dz + dmu + 2.0 ** -23 * (z.abs() + dev.abs()))).sum(dim=1, keepdim=True)
           + p * U32 * ss + p * dmu.square())
    drstd = dss / (2 * (ss + p * eps32)) + U32 + 2 * 2.0 ** -23
    eta_zh = rstd * (dz + dmu) + zh.abs() * (drstd + 2 * U32)
    eta_e = ga.abs() * eta_zh + U32 * ((zh * ga).abs() + e.abs())
    return {"hb": hb, "wb": wb, "z": z, "mu": mu[:, 0], "rstd": rstd[:, 0], "zhat": zh, "e": e, "gamma": ga,
            "eta_zhat": eta_zh, "eta_e": eta_e, "drstd": drstd[:, 0], "n": n, "k": k, "p": p}


def head_check(ref, *, e=None, zhat=None, rstd=None, rinv=None):
    out = {}
    p = ref["p"]
    if e is not None:
        _rounded_check(out, "e", e, ref["e"], ref["eta_e"], _entry(p))
    if zhat is not None:
        _rounded_check(out, "zhat", zhat, ref["zhat"], ref["eta_zhat"], _entry(p))
    if rstd is not None:
        want = ref["rstd"]
        _put(out, "rstd", _ratio((rstd.to(want.device).double() - want).abs(), ref["drstd"] * want))
    if rinv is not None and e is not None:
        want = 1.0 / e.double().norm(dim=1).clamp_min(R.EPS)
        _put(out, "rinv", _ratio((rinv.double() - want).abs(), (p + 4) * U32 * want))
    return out


def ln_backward_reference(de, zhat, rstd, gamma):
    """dz of `head::ln_backward_rows` in float64 on ITS inputs (de bf16 or fp32, z_hat bf16, rstd and gamma fp32), and
    eta_dz: the fp32 products, the two (p/32 + 5)-addition sums, the means and the final expression."""
    g = de.double() * gamma.double()
    zh = zhat.double()
    rs = rstd.double()[:, None]
    p = g.shape[1]
    m1 = g.mean(dim=1, keepdim=True)
    m2 = (g * zh).mean(dim=1, keepdim=True)
    dz = rs * (g - m1 - zh * m2)
    c = (p / 32 + 5) * U32
    dg = U32 * g.abs()
    dm1 = c * g.abs().mean(dim=1, keepdim=True) + dg.mean(dim=1, keepdim=True) + U32 * m1.abs()
    dm2 = 2 * c * (g * zh).abs().mean(dim=1, keepdim=True) + (dg * zh.abs()).mean(dim=1, keepdim=True) + U32 * m2.abs()
    eta = rs * (dg + dm1 + zh.abs() * dm2 + 2 * U32 * (g.abs() + m1.abs() + 2 * (zh * m2).abs())) + U32 * dz.abs()
    return dz, eta


def ln_backward_check(dz_got, dz_ref, eta):
    out = {}
    _rounded_check(out, "dz", dz_got, dz_ref, eta, _entry(dz_ref.shape[1]))
    return out


def _dtype_ulp(dtype):
    """Relative bound for the rounding to a parameter dtype: one ulp (a factor 2 over round-to-nearest's half ulp)."""
    return {torch.bfloat16: 2.0 ** -7, torch.float16: 2.0 ** -10}.get(dtype, 2.0 ** -23)


def head_grads_reference(ref, de, bias_present):
    """Float64 autograd of e = LayerNorm(hb W^T + b) gamma + beta against ``de`` (the upstream gradient the kernel got),
    and the budgets of the module docstring.  -> dict with d_h [n,k], d_w [p,k], d_gamma, d_beta, d_bias [p] and their
    budgets (per row of d_h and d_w, per entry of the others), before the rounding to the parameter dtypes."""
    hb, wb = ref["hb"], ref["wb"]
    n, k, p = ref["n"], ref["k"], ref["p"]
    de64 = de.double()
    ga = ref["gamma"]
    # exact backward (the LayerNorm formula, equal to autograd of the forward above)
    gg = de64 * ga
    zh, rs = ref["zhat"], ref["rstd"][:, None]
    m2 = (gg * zh).mean(dim=1, keepdim=True)
    dz = rs * (gg - gg.mean(dim=1, keepdim=True) - zh * m2)
    d_h, d_w = dz @ wb, dz.T @ hb
    d_gamma, d_beta, d_bias = (de64 * zh).sum(dim=0), de64.sum(dim=0), dz.sum(dim=0)
    # per-entry error of the kernel's dz: independent and one-signed parts
    hz = bf16_half_ulp(zh.abs() + ref["eta_zhat"])
    _, eta_dz = ln_backward_reference(de, zh, ref["rstd"], ga)
    dzh = hz + ref["eta_zhat"]
    dm2 = (gg.abs() * dzh).mean(dim=1, keepdim=True)
    rand = bf16_half_ulp(dz.abs()) + rs * m2.abs() * hz
    coh = eta_dz + rs * m2.abs() * ref["eta_zhat"] + rs * zh.abs() * dm2 + ref["drstd"][:, None] * dz.abs()
    wa, ha = wb.abs(), hb.abs()
    b_dh = (C_RAND_HEAD * (rand.square() @ wb.square()).sum(dim=1).sqrt() + (coh @ wa).norm(dim=1)
            + (p / 16 + 1) * 2.0 ** -23 * (dz.abs() @ wa).norm(dim=1) + 2.0 ** -8 * d_h.norm(dim=1))
    b_dw = (C_RAND_HEAD * (rand.square().T @ hb.square()).sum(dim=1).sqrt() + (coh.T @ ha).norm(dim=1)
            + (n / 16 + 1) * 2.0 ** -23 * (dz.abs().T @ ha).norm(dim=1) + 2.0 ** -8 * d_w.norm(dim=1))
    sq_n = C_RAND_HEAD * n ** 0.5 * U32
    b_dbias = C_RAND_HEAD * rand.square().sum(dim=0).sqrt() + coh.sum(dim=0) + sq_n * dz.abs().sum(dim=0)
    b_dgamma = (C_RAND_HEAD * (de64 * hz).square().sum(dim=0).sqrt() + (de64.abs() * ref["eta_zhat"]).sum(dim=0)
                + (sq_n + U32) * (de64 * zh).abs().sum(dim=0))
    b_dbeta = sq_n * de64.abs().sum(dim=0)
    out = {"d_h": d_h, "d_w": d_w, "d_gamma": d_gamma, "d_beta": d_beta, "budget_h": b_dh, "budget_w": b_dw,
           "budget_gamma": b_dgamma, "budget_beta": b_dbeta}
    if bias_present:
        out.update(d_bias=d_bias, budget_bias=b_dbias)
    return out


def head_grads_check(gref, *, d_h, d_w, d_gamma, d_beta, d_bias=None):
    """Gradients as the module returns them (in the parameters' dtypes): the rounding to that dtype joins the budget."""
    out = {}
    for name, got, key, rows in (("d_h", d_h, "h", True), ("d_w", d_w, "w", True), ("d_gamma", d_gamma, "gamma", False),
                                 ("d_beta", d_beta, "beta", False), ("d_bias", d_bias, "bias", False)):
        if got is None:
            continue
        want, bud = gref[name], gref["budget_" + key]
        g = got.to(device=want.device, dtype=F64)
        if rows:    # the bf16 output of the GEMMs is in the budget; the cast to the parameter dtype adds nothing
            _put(out, name, _ratio((g - want).norm(dim=1), bud))
        else:
            _put(out, name, _ratio((g - want).abs(), bud + _dtype_ulp(got.dtype) * want.abs()))
    return out
