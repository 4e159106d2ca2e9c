"""Small-shape pass over every hand-written kernel family, meant to run under compute-sanitizer
(`compute-sanitizer --tool memcheck|synccheck|racecheck python tools/sanitize.py`); results are checked against the oracle."""
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.environ.setdefault("CLIPNCE_BWD2_MIN_N", "256")
import torch  # noqa: E402

from clip_dplm_b200 import fused_clip_loss  # noqa: E402
from clip_dplm_b200.retrieval import topk_similarity  # noqa: E402
from oracle import ref_step as O  # noqa: E402


def one(n, d, s, tag, **env):
    for k, v in env.items():
        os.environ[k] = v
    a, b = O.make_inputs(n, d, seed=3, mix=0.12 if s > 50 else 0.5)
    ref = O.ref_step(a.double(), b.double(), s, scale_is_log=False)
    ac, bc = a.cuda().bfloat16().requires_grad_(True), b.cuda().bfloat16().requires_grad_(True)
    loss = fused_clip_loss(ac, bc, s, scale_is_log=False)
    loss.backward()
    torch.cuda.synchronize()
    rel = lambda x, r: float((x.float().cpu().double() - r).norm() / r.norm())
    e = (abs(float(loss) - float(ref["loss"])) / abs(float(ref["loss"])), rel(ac.grad, ref["d_a"]), rel(bc.grad, ref["d_b"]))
    print(f"{tag:28s} n={n} d={d} s={s:g}: loss rel {e[0]:.1e} dA {e[1]:.1e} dB {e[2]:.1e}", flush=True)
    assert e[0] <= 1e-3 and e[1] <= 2e-2 and e[2] <= 2e-2
    for k in env:
        os.environ.pop(k)


one(1024, 128, 1 / 0.07, "two-sided backward")
one(1024, 512, 1 / 0.07, "two-sided, 3 producers, 2 seg", CLIPNCE_BWD2_P="3", CLIPNCE_BWD2_SEG="2")
one(512, 512, 1 / 0.07, "two-sweep backward", CLIPNCE_NO_BWD2="1")
one(512, 256, 1 / 0.07, "two-sweep, split sweep", CLIPNCE_NO_BWD2="1", CLIPNCE_SPLIT_STEPS="1")
one(512, 256, 100.0, "family 2, speculative forward")
one(512, 256, 100.0, "family 2, exact online sweeps", CLIPNCE_NO_SPECULATE="1")
one(1024, 256, 100.0, "family 2, two-sided backward", CLIPNCE_BWD2_P="5")
one(300, 192, 10.0, "single-CTA tcgen05 kernels")
one(200, 100, 10.0, "exact CUDA-core kernels")
# grouped launch: three pairs over three embeddings (tri-modal model), ragged rows
from clip_dplm_b200 import modules as M  # noqa: E402
gg = torch.Generator().manual_seed(4)
base = torch.randn(700, 256, generator=gg)
embs = [(m * base + (1 - m) * torch.randn(700, 256, generator=gg)).bfloat16() for m in (1.0, 0.5, 0.3)]
refs = [e.double().requires_grad_(True) for e in embs]
rt = torch.tensor(2.6592, dtype=torch.float64)
rl = O.ref_loss(refs[0], refs[1], rt) + O.ref_loss(refs[0], refs[2], rt) + O.ref_loss(refs[1], refs[2], rt)
rl.backward()
ce = [e.cuda().requires_grad_(True) for e in embs]
out = M.trimodal_contrastive_losses(*ce, torch.tensor(2.6592, device="cuda"))
out["loss"].backward()
torch.cuda.synchronize()
assert "embed_grad_sumsq" in out.grad_info, "grouped launch not taken"
relg = lambda x, r: float((x.float().cpu().double() - r).norm() / r.norm())
eg = [relg(c.grad, r.grad) for c, r in zip(ce, refs)]
print(f"grouped tri-modal launch      n=700 d=256: loss rel {abs(float(out['loss']) - float(rl)) / float(rl):.1e} grads {eg[0]:.1e} {eg[1]:.1e} {eg[2]:.1e}", flush=True)
assert abs(float(out["loss"]) - float(rl)) <= 1e-3 * float(rl) and max(eg) <= 2e-2
g = torch.Generator().manual_seed(1)
q, lib = torch.randn(300, 256, generator=g).bfloat16().cuda(), torch.randn(2000, 256, generator=g).bfloat16().cuda()
s, i = topk_similarity(q, lib, 10)
rs, ri, _ = O.ref_topk(q.float().cpu(), lib.float().cpu(), 10)
torch.cuda.synchronize()
assert (i.cpu() == ri).float().mean() > 0.99
print("retrieval top-10 ok", flush=True)
print("SANITIZE PASS OK")
