"""Pin the oracle against the reference itself and write tests/golden/*.npz.

Needs a checkout of the reference project (SrikarK-code/clip-dplm), named by CLIP_DPLM_REFERENCE:

    CLIP_DPLM_REFERENCE=<checkout> python oracle/gen_golden.py

What it does
  1. imports the reference's own modules from that checkout
       - old/clip.py           RNAProteinCLIPModule / DiffMapProteinCLIPModule   (forward tail :63-67, :100-104)
       - old/clip_opt.py       optimized_clip_loss                               (:130-151)
       - tong/utils/losses.py  contrastive_loss                                  (:4-19)
       - current/rna_clip_codes.ipynb cells 24+28  RNARBPCLIPModel               (raw :1925-1954)
     (current/tf_clip_codes (1).ipynb cell 41, raw :13146-13165, repeats the notebook lines above for three pairs with one
      shared logit scale; it is NOT loaded -- its loss is three calls of the pinned pair form)
  2. asserts oracle/ref_step.py reproduces each of them EXACTLY (torch.equal) on seeded inputs,
  3. stores inputs (bf16-rounded, as uint16 bit patterns) + reference outputs as small fixtures; fixtures with more
     than GRAD_FULL_MAX gradient entries per side keep a seeded sample of GRAD_SAMPLE_ROWS gradient rows (`grad_rows`),
     so that every file stays under 1 MB.

Nothing here is imported by the product path.
"""
from __future__ import annotations

import importlib.util
import json
import math
import os
import sys
import types

import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("CLIP_DPLM_REFERENCE", "")
sys.path.insert(0, ROOT)
from oracle import ref_step as O  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
GRAD_FULL_MAX, GRAD_SAMPLE_ROWS = 1 << 16, 64


def grad_rows(n, d):
    """Rows of d_a64 / d_b64 a fixture stores: all of them, or a fixed seeded sample for the larger fixtures."""
    if n * d <= GRAD_FULL_MAX:
        return None
    return np.sort(np.random.default_rng(0).choice(n, size=GRAD_SAMPLE_ROWS, replace=False))


def _load(path, name):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def load_reference():
    if not os.path.isdir(REF):
        sys.exit("gen_golden: set CLIP_DPLM_REFERENCE to a checkout of the reference project")
    ref = {}
    # old/clip.py imports `configuration_hybrid_clip` (needs transformers; its ctor is broken on
    # transformers 5.5 -> duck-typed config below) -- stub the module so the import succeeds.
    stub = types.ModuleType("configuration_hybrid_clip")
    stub.HybridCLIPConfig = object
    sys.modules["configuration_hybrid_clip"] = stub
    ref["clip"] = _load(os.path.join(REF, "old", "clip.py"), "ref_old_clip")
    ref["losses"] = _load(os.path.join(REF, "tong", "utils", "losses.py"), "ref_tong_losses")
    ref["clip_opt"] = _load(os.path.join(REF, "old", "clip_opt.py"), "ref_old_clip_opt")
    nb = json.load(open(os.path.join(REF, "current", "rna_clip_codes.ipynb")))
    cells = ["".join(c["source"]) for c in nb["cells"] if c["cell_type"] == "code"]
    ns = {"torch": torch, "nn": nn, "F": F, "np": np}
    for src in cells:
        if "def create_padding_mask" in src or "class RNARBPCLIPModel" in src:
            exec(src, ns)
    ref["rnarbp"] = ns
    return ref


def bf16_bits(x: torch.Tensor) -> np.ndarray:
    return x.to(torch.bfloat16).view(torch.int16).numpy().astype(np.uint16)


def cfg(hidden_a, hidden_b, proj):
    sub = lambda h: types.SimpleNamespace(hidden_size=h, num_hidden_layers=2, layer_norm_eps=1e-5)
    return types.SimpleNamespace(rna_config=sub(hidden_a), protein_config=sub(hidden_b), diffmap_config=sub(hidden_a),
                                 projection_dim=proj, logit_scale_init_value=2.6592, cache_size=64)


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = load_reference()
    torch.manual_seed(0)
    report = {}

    # ---- (1) old/clip.py forward tail == oracle.ref_logits -------------------------------------
    m = ref["clip"].RNAProteinCLIPModule(cfg(48, 64, 128)).eval()
    x, y = torch.randn(40, 48), torch.randn(40, 64)
    with torch.no_grad():
        out = m(x, y)
        ea = m.rna_projection(m.rna_model(x))
        eb = m.protein_projection(m.protein_model(y))
        logits, ah, bh = O.ref_logits(ea, eb, m.logit_scale)
    assert torch.equal(out["logits_per_rna_protein"], logits)
    assert torch.equal(out["rna_embeds"], ah) and torch.equal(out["protein_embeds"], bh)
    m2 = ref["clip"].DiffMapProteinCLIPModule(cfg(48, 64, 128)).eval()
    with torch.no_grad():
        out2 = m2(x, y)
        logits2, _, _ = O.ref_logits(m2.diffmap_projection(m2.diffmap_model(x)),
                                     m2.protein_projection(m2.protein_model(y)), m2.logit_scale)
    assert torch.equal(out2["logits_per_diffmap_protein"], logits2)
    report["old/clip.py forward tail"] = "exact"

    # ---- (2) notebook RNARBPCLIPModel loss == oracle.ref_loss (symmetric) ------------------------
    ns = ref["rnarbp"]
    model = ns["RNARBPCLIPModel"](rna_dim=16, rbp_dim=24, projection_dim=32).eval()
    n_params_small = sum(p.numel() for p in model.parameters())
    rna, rbp = torch.randn(12, 5, 16), torch.randn(12, 7, 24)   # [batch, seq, dim] as the notebook feeds it
    with torch.no_grad():
        ra, rb, loss = model(rna, rbp)
        rna_enc = model.rna_encoder(rna, src_key_padding_mask=~ns["create_padding_mask"](rna).transpose(0, 1))
        rbp_enc = model.rbp_encoder(rbp, src_key_padding_mask=~ns["create_padding_mask"](rbp).transpose(0, 1))
        pa, pb = model.rna_projection(rna_enc[:, 0]), model.rbp_projection(rbp_enc[:, 0])
        loss_o = O.ref_loss(pa, pb, model.logit_scale)
    assert torch.equal(loss, loss_o), (loss, loss_o)
    report["rna_clip_codes.ipynb RNARBPCLIPModel loss"] = "exact"
    # recorded known answer: 71,646,299 parameters at (120, 1280, 512)  (rna_clip_codes.ipynb:2312)
    full = ns["RNARBPCLIPModel"]()
    n_params = sum(p.numel() for p in full.parameters())
    assert n_params == 71_646_299, n_params
    report["param count 71,646,299"] = "reproduced"
    del full

    # ---- (3) tong contrastive_loss == oracle one-directional (+queue) ---------------------------
    xa, yb, q = torch.randn(33, 40), torch.randn(33, 40), torch.randn(17, 40)
    l_ref = ref["losses"].contrastive_loss(xa, yb, temperature=0.1)
    l_o = O.ref_loss(xa, yb, torch.tensor(1 / 0.1), symmetric=False, scale_is_log=False)
    assert torch.allclose(l_ref, l_o, rtol=0, atol=2e-6), (l_ref, l_o)   # `/ temperature` vs `* (1/temperature)`
    l_ref_q = ref["losses"].contrastive_loss(xa, yb, temperature=0.1, queue=q)
    l_o_q = O.ref_loss(xa, yb, torch.tensor(1 / 0.1), symmetric=False, scale_is_log=False, extra_cols=q)
    assert torch.allclose(l_ref_q, l_o_q, rtol=0, atol=2e-6), (l_ref_q, l_o_q)
    report["tong/utils/losses.py contrastive_loss"] = "within 2e-6 (divide vs multiply by temperature)"

    # ---- (4) old/clip_opt.py optimized_clip_loss == oracle cache variant --------------------------
    ea, eb = torch.randn(24, 32), torch.randn(24, 32)
    cache = F.normalize(torch.randn(10, 32), dim=-1)
    t = torch.tensor(math.log(1 / 0.07))
    sim, ah, bh = O.ref_logits(ea, eb, t, clamp_max=100)
    outputs = {"logits_per_diffmap_protein": sim, "logits_per_diffmap_cache": (ah @ cache.t()) * t.exp().clamp(max=100)}
    l_ref = ref["clip_opt"].optimized_clip_loss(outputs)
    l_o = O.ref_loss(ea, eb, t, clamp_max=100, extra_cols=cache)
    assert torch.equal(l_ref, l_o), (l_ref, l_o)
    report["old/clip_opt.py optimized_clip_loss"] = "exact"

    # ---- golden vectors for the CUDA parity tests -----------------------------------------------
    cases = [
        # name, n, d, n_cols, correlated, logit_scale, kwargs
        ("c1_n256_d512", 256, 512, None, True, O.LOGIT_SCALE_INIT, {}),                     # BASELINE config 1
        ("rand_n256_d128", 256, 128, None, False, O.LOGIT_SCALE_INIT, {}),
        ("n32_d128", 32, 128, None, True, O.LOGIT_SCALE_INIT, {}),                          # notebook batch 32
        ("ragged_n333_d192", 333, 192, None, True, O.LOGIT_SCALE_INIT, {}),
        ("d768_n192", 192, 768, None, True, O.LOGIT_SCALE_INIT, {}),                        # config 3 width
        ("clamp100_n256_d128", 256, 128, None, True, 5.0, {"clamp_max": 100, "mix": 0.12}),  # e^5 > 100 -> clamped
        ("tong_t0p1_n256_d128", 256, 128, None, True, 10.0, {"symmetric": False, "scale_is_log": False}),
        ("onedir_n256_d128", 256, 128, None, True, O.LOGIT_SCALE_INIT, {"symmetric": False}),
        ("cache_n256_d128", 256, 128, 256 + 96, True, O.LOGIT_SCALE_INIT, {"clamp_max": 100, "cache": 96}),
    ]
    for name, n, d, n_cols, corr, ls, kw in cases:
        kw = dict(kw)
        n_cache = kw.pop("cache", 0)
        a, b = O.make_inputs(n, d, seed=1234, correlated=corr, n_cols=n_cols, mix=kw.pop("mix", 0.5))
        extra = None
        if n_cache:
            extra = F.normalize(b[n:], dim=-1).to(torch.bfloat16).to(torch.float32)  # cache rows are stored normalised
            b = b[:n]
            kw["extra_cols"] = extra
        r32 = O.ref_step(a, b, ls, **kw)
        r64 = O.ref_step(a.double(), b.double(), ls,
                         **{k: (v.double() if torch.is_tensor(v) else v) for k, v in kw.items()})
        arrs = dict(a_bits=bf16_bits(a), b_bits=bf16_bits(b), logit_scale=np.float64(ls),
                    loss32=r32["loss"].numpy(), loss64=r64["loss"].numpy(),
                    d_a64=r64["d_a"].numpy().astype(np.float32), d_b64=r64["d_b"].numpy().astype(np.float32),
                    d_ls32=r32["d_logit_scale"].numpy(), d_ls64=r64["d_logit_scale"].numpy(),
                    meta=np.array(json.dumps({k: v for k, v in kw.items() if not torch.is_tensor(v)})))
        if extra is not None:
            arrs["extra_bits"] = bf16_bits(extra)
        rows = grad_rows(n, d)
        if rows is not None:
            arrs.update(grad_rows=rows, d_a64=arrs["d_a64"][rows], d_b64=arrs["d_b64"][rows])
        np.savez_compressed(os.path.join(OUT, name + ".npz"), **arrs)
        report["golden/" + name] = f"loss={float(r64['loss']):.6f}"

    # recorded anchor: untrained model, B=32 -> loss ~ ln 32 (rna_clip_codes.ipynb:2333 prints 3.5013)
    a, b = O.make_inputs(32, 512, seed=7, correlated=False)
    l = float(O.ref_loss(a, b, torch.tensor(0.0)))    # s = 1: nearly uniform soft-max
    assert abs(l - math.log(32)) < 0.05, l
    report["ln(32) anchor"] = f"{l:.4f} vs {math.log(32):.4f}"

    with open(os.path.join(OUT, "PINNED.json"), "w") as f:
        json.dump({"torch": torch.__version__, "small_model_params": n_params_small, "checks": report}, f, indent=1)
    for k, v in report.items():
        print(f"{k:55s} {v}")


if __name__ == "__main__":
    main()
