"""Float64 reference of the fused loss with a per-row error budget.  TEST INFRASTRUCTURE ONLY (same rule as
``oracle/ref_step.py``: imported by ``tests/`` and tools only).

`reference` computes the loss, its statistics and both gradients the way the C ABI defines the operation, on the device
of its inputs, one [block, N] slab of the logits at a time (so that 65536 x 512 fits a GPU).  Staging follows
`step.contrastive_forward` and `aux::finish_rows`: the contraction sees the rows rounded to the compute type, scaled by
1/|row| of the UNROUNDED rows, and the normalise backward uses the unrounded rows; extra columns are used as stored
(rinv = 1).

Every output comes with a budget, so that a check can be made entry by entry instead of over the whole matrix.  With
G the gradient of the loss with respect to the logits S, and C_ij the magnitude of G's components
(exp(S - r_i) w_r + exp(S - c_j) w_c + delta_ij / N), a gradient row i is allowed

    budget_i = ( C_RAND s sqrt( sum_j (u |G_ij| + 2^-20 s C_ij)^2 )     independent rounding of the tile's entries
               + 2^-18 s sum_j C_ij )                                     the row's share of the forward statistics' error
               rinv_i |g|  +  u_out |dA_ref_i|                            normalise backward; output rounding

u is the unit roundoff of the route's gradient tile (bf16 on the tensor-core routes, fp32 on the exact kernels).  The
C_ij term is there because a separated positive makes G_ii a cancellation whose fp32 error is relative to 1/N, not to
|G_ii|; the square root is there because rounding errors of different entries add in quadrature -- a sum of absolute
values would grow like N and stop seeing a missing block of columns.  The statistics and the loss are allowed
C_STAT s 2^-21 + 2^-20 |value| each.

sum G.S (the logit-scale gradient) gets the same two terms with |G_ij S_ij|, except that the statistics' share adds in
quadrature over rows and columns (each row's and column's statistics are separate sums), plus a bias common to all rows
and, on the tensor-core routes, the one-signed error of the fp32 accumulators over a row's contraction.
"""
from __future__ import annotations

import torch

U_TILE_BF16 = 2.0 ** -9    # tensor-core routes: the gradient tile is rounded to bf16
U_TILE_F32 = 2.0 ** -22    # exact kernels: the gradient tile stays fp32
C_RAND = 4.0
C_STAT = 8.0
EPS = 1e-12                # F.normalize's clamp (old/clip.py:63-64)


def u_out(dtype) -> float:
    """Relative rounding of a gradient row stored in ``dtype`` (norm-wise, with a factor 2 over half an ulp)."""
    return 2.0 ** -8 if dtype == torch.bfloat16 else 0.0


def staged(x, compute_dtype):
    """-> (x in float64, rinv of the unrounded rows, the rows the contraction sees: round(x) * rinv)."""
    x64 = x.detach().to(torch.float64)
    rinv = 1.0 / x64.norm(dim=1).clamp_min(EPS)
    xc = x.detach().to(compute_dtype).to(torch.float64) * rinv[:, None]
    return x64, rinv, xc


def normalize_backward(x64, rinv, d_hat, g=1.0):
    """Gradient of the caller's rows from the gradient of the normalised rows (aux::finish_rows; clamped rows: d_hat rinv)."""
    xh = x64 * rinv[:, None]
    dot = (xh * d_hat).sum(dim=1, keepdim=True)
    dot = torch.where(rinv[:, None] >= 0.5 / EPS, torch.zeros_like(dot), dot)
    return (d_hat - xh * dot) * rinv[:, None] * g


def stat_budget(value, s_err):
    return C_STAT * s_err * 2.0 ** -21 + 2.0 ** -20 * torch.as_tensor(value, dtype=torch.float64).abs()


def reference(a, b, s, *, symmetric=True, extra=None, extra_normalized=True, g=1.0, block=4096,
              compute_dtype=torch.bfloat16, u=U_TILE_BF16):
    """a, b: [N,d] the caller's rows (any float type, on any device); s: the scale; extra: [M,d] extra negative columns;
    extra_normalized: their rows have norm <= 1 (|S| <= s), else the error terms are scaled by the largest norm;
    g: upstream gradient of the loss; compute_dtype: the type the contraction reads; u: the gradient tile's roundoff.

    -> dict of float64 tensors: loss, row_lse [N], col_lse [N] (batch columns), diag [N], d_a, d_b [N,d] (times g),
    d_scale_sum (sum G.S, NOT times g), budget_a, budget_b [N], budget_d_scale, and s_err (the logit magnitude the
    statistics' budgets use)."""
    s = float(s)
    n, d = a.shape
    a64, ra, ac = staged(a, compute_dtype)
    b64, rb, bc = staged(b, compute_dtype)
    y, nu, s_err = bc, None, s
    if extra is not None:
        e = extra.detach().to(compute_dtype).to(torch.float64)
        y = torch.cat([bc, e])
        nu = torch.cat([torch.ones(n, dtype=torch.float64, device=a.device), e.norm(dim=1)])
        if not extra_normalized:
            s_err = s * max(1.0, float(nu.max()))
    dev = a.device
    f64 = dict(dtype=torch.float64, device=dev)

    row_lse, diag = torch.empty(n, **f64), torch.empty(n, **f64)
    col_lse = torch.full((n,), -float("inf"), **f64)
    for i0 in range(0, n, block):
        i1 = min(n, i0 + block)
        S = (ac[i0:i1] @ y.T).mul_(s)
        row_lse[i0:i1] = torch.logsumexp(S, dim=1)
        col_lse = torch.logaddexp(col_lse, torch.logsumexp(S[:, :n], dim=0))
        k = torch.arange(i1 - i0, device=dev)
        diag[i0:i1] = S[k, i0 + k]
        del S
    if symmetric:
        loss = ((row_lse - diag).sum() + (col_lse - diag).sum()) / (2 * n)
    else:
        loss = (row_lse - diag).sum() / n

    w_r = 1.0 / (2 * n) if symmetric else 1.0 / n
    w_c = 1.0 / (2 * n) if symmetric else 0.0
    d_ah, d_bh = torch.empty(n, d, **f64), torch.zeros(n, d, **f64)
    rand_a, coh_a = torch.empty(n, **f64), torch.empty(n, **f64)
    rand_b, coh_b = torch.zeros(n, **f64), torch.zeros(n, **f64)
    ds = torch.zeros((), **f64)
    rand_ds = torch.zeros((), **f64)
    coh_ds_rows = torch.zeros((), **f64)
    coh_ds_cols = torch.zeros(y.shape[0], **f64)
    for i0 in range(0, n, block):
        i1 = min(n, i0 + block)
        k = torch.arange(i1 - i0, device=dev)
        S = (ac[i0:i1] @ y.T).mul_(s)
        G = (S - row_lse[i0:i1, None]).exp_().mul_(w_r)
        if symmetric:
            G[:, :n] += (S[:, :n] - col_lse[None, :]).exp_().mul_(w_c)
        C = G.clone()
        G[k, i0 + k] -= 1.0 / n
        C[k, i0 + k] += 1.0 / n
        d_ah[i0:i1] = (G @ y).mul_(s)
        d_bh += (G[:, :n].T @ ac[i0:i1]).mul_(s)
        ds += (G * S).sum()
        T = G.abs().mul_(u).add_(C, alpha=2.0 ** -20 * s_err)     # per-entry error of the tile
        Tc = T * nu if nu is not None else T
        rand_a[i0:i1] = Tc.square().sum(dim=1)
        coh_a[i0:i1] = (C * nu).sum(dim=1) if nu is not None else C.sum(dim=1)
        rand_b += T[:, :n].square().sum(dim=0)
        coh_b += C[:, :n].sum(dim=0)
        del T, Tc
        # sum G.S: the tile's rounding times |S|, and the logits' own error times |G|
        CS = C.mul_(S.abs())
        rand_ds += (G * S).abs_().mul_(u).add_(CS, alpha=2.0 ** -20 * s_err).add_(G.abs(), alpha=2.0 ** -20 * s_err).square_().sum()
        coh_ds_rows += CS.sum(dim=1).square().sum()
        coh_ds_cols += CS.sum(dim=0)
        del S, G, C, CS

    d_a = normalize_backward(a64, ra, d_ah, g)
    d_b = normalize_backward(b64, rb, d_bh, g)
    budget_a = ((C_RAND * s) * rand_a.sqrt() + 2.0 ** -18 * s_err * coh_a) * ra * abs(g) + u_out(a.dtype) * d_a.norm(dim=1)
    budget_b = ((C_RAND * s) * rand_b.sqrt() + 2.0 ** -18 * s_err * coh_b) * rb * abs(g) + u_out(b.dtype) * d_b.norm(dim=1)
    # the statistics' error is shared along one row (r_i) or one column (c_j), and different rows' statistics are separate
    # sums: over the whole matrix these shares add in quadrature, plus a bias common to all of them (approximate exp / log)
    coh_ds = coh_ds_rows.sqrt() + coh_ds_cols.square().sum().sqrt()
    budget_ds = C_RAND * rand_ds.sqrt() + 2.0 ** -18 * s_err * coh_ds + 2.0 ** -22 * s_err * coh_ds_cols.sum()
    if u == U_TILE_BF16:
        # the tensor cores' fp32 accumulators do not round to nearest: over the additions of a row's contraction their
        # error has one sign, about 2^-24 of the row per addition -- at most N / 16 of them (K = 16 per MMA; a column sweep
        # cut into work items or segments adds fewer in each fp32 slab).  In dA this is a shrink of the row by about
        # (N / 16) 2^-24, far inside its budget (the component along a_hat_i is also projected out by the normalise
        # backward); sum G.S = sum_i <a_hat_i, dA_hat_i> adds it up over all rows with one sign
        budget_ds = budget_ds + 2.0 ** -24 * (y.shape[0] / 16) * d_ah.norm(dim=1).sum()
    return {"loss": loss, "row_lse": row_lse, "col_lse": col_lse, "diag": diag, "d_a": d_a, "d_b": d_b,
            "d_scale_sum": ds, "budget_a": budget_a, "budget_b": budget_b, "budget_d_scale": budget_ds, "s_err": s_err,
            "n": n, "g": float(g)}


def _worst(ratio, k=5):
    r = ratio.flatten()
    top = torch.topk(r, min(k, r.numel()))
    return [(int(i), float(v)) for v, i in zip(top.values.cpu(), top.indices.cpu())]


def check(ref, *, loss=None, d_a=None, d_b=None, d_scale_sum=None, row_lse=None, col_lse=None, diag=None, row0=0):
    """Ratios error / budget of every output given, against ``ref`` (from `reference`).  d_a, d_b, row_lse, diag are the
    rows [row0, row0 + len) of the global batch (a rank's shard); col_lse covers every batch column.

    -> {name: {"max": largest ratio, "worst": [(global row, ratio), ...]}}; a check passes when every max is <= 1."""
    out = {}

    def put(name, got, want, budget, offset=0):
        got = torch.as_tensor(got).to(device=want.device, dtype=torch.float64)
        if got.dim() == 2:
            err = (got - want).norm(dim=1)
        else:
            err = (got.reshape(want.shape) - want).abs()
        ratio = err / budget
        ratio = torch.where(torch.isnan(ratio), torch.full_like(ratio, float("inf")), ratio)
        out[name] = {"max": float(ratio.max()) if ratio.numel() else 0.0,
                     "worst": [(i + offset, v) for i, v in _worst(ratio)]}

    def rows(x, m):
        return x[row0:row0 + m]

    s_err = ref["s_err"]
    if loss is not None:
        put("loss", torch.as_tensor(float(loss), dtype=torch.float64), ref["loss"], stat_budget(ref["loss"], s_err))
    if d_a is not None:
        m = d_a.shape[0]
        put("dA", d_a, rows(ref["d_a"], m), rows(ref["budget_a"], m), row0)
    if d_b is not None:
        m = d_b.shape[0]
        put("dB", d_b, rows(ref["d_b"], m), rows(ref["budget_b"], m), row0)
    if d_scale_sum is not None:
        put("d_scale", torch.as_tensor(float(d_scale_sum), dtype=torch.float64), ref["d_scale_sum"], ref["budget_d_scale"])
    for name, got in (("row_lse", row_lse), ("diag", diag)):
        if got is not None:
            want = rows(ref[name], got.shape[0])
            put(name, got, want, stat_budget(want, s_err), row0)
    if col_lse is not None:
        want = ref["col_lse"]
        put("col_lse", torch.as_tensor(col_lse)[:want.shape[0]], want, stat_budget(want, s_err))
    return out


def describe(report, route=""):
    """One line per output: the largest ratio and the worst rows with their 128-row block."""
    lines = [f"route {route}"] if route else []
    for name, r in report.items():
        worst = ", ".join(f"row {i} (block {i // 128}) {v:.3g}" for i, v in r["worst"])
        lines.append(f"{name}: max ratio {r['max']:.3g}; worst {worst}")
    return "\n".join(lines)
