"""Row-sharded global batch (needs >= 2 GPUs; skipped on a single-GPU box): every rank's loss and gradients must equal
the single-process reference on the concatenated batch (SURVEY.md section 8e) -- through the NVLink peer-memory exchange
kernels (the product path, "link") and through the NCCL collectives (the baseline it is measured against, "nccl").
The exchange kernels themselves also run on ONE GPU (a one-rank group): test_peer_exchange_kernels_single_rank."""
import math
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import ref_step as O

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, n, d, comm, q, both=False, ls=O.LOGIT_SCALE_INIT, mix=0.5, a_dtype=torch.bfloat16):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    if both:
        os.environ["CLIPNCE_BWD2_MIN_N"] = "256"    # serve the small test shape with the two-sided kernel
        # ... and gather the columns BESIDE the forward sweep (copy engines + per-block flags, clipnce_forward_gathered),
        # which by default starts at 8192 local rows; the other tests keep the push kernel + barrier in front of the sweep
        os.environ["CLIPNCE_GATHER_BESIDE_MIN_ROWS"] = "256"
    else:
        os.environ["CLIPNCE_NO_BWD2"] = "1"
    os.environ.setdefault("CLIPNCE_LINK_TIMEOUT_MS", "30000")   # a lost rank fails the test in 30 s, not in 10 min
    os.environ["CLIPNCE_COMM"] = comm
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from clip_dplm_b200 import fused_clip_loss
        a, b = O.make_inputs(n, d, seed=33, mix=mix)
        nl = n // world
        ac = a[rank * nl:(rank + 1) * nl].cuda().to(a_dtype).requires_grad_(True)
        bc = b[rank * nl:(rank + 1) * nl].cuda().bfloat16().requires_grad_(True)
        t = torch.tensor(ls, device="cuda", requires_grad=True)
        loss = fused_clip_loss(ac, bc, t, group=dist.group.WORLD)
        loss.backward()
        torch.cuda.synchronize()
        from clip_dplm_b200 import exchange
        assert exchange.comm_kind(dist.group.WORLD) == comm
        if both:
            from clip_dplm_b200.engine import default_engine
            assert default_engine().backward_both_bytes(nl, n, d, torch.bfloat16, math.exp(ls), 0, world) > 0, "two-sided path not served"
        q.put((rank, float(loss.detach()), ac.grad.float().cpu().numpy(), bc.grad.float().cpu().numpy(), float(t.grad)))
        exchange.reset()
    finally:
        dist.destroy_process_group()


def _run(target, args, world, timeout=300, extra=()):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=target, args=(r, world) + tuple(args) + (q,) + tuple(extra)) for r in range(world)]
    for p in procs:
        p.start()
    import queue as _queue
    import time
    try:
        out, t0 = [], time.time()
        while len(out) < world:       # fail fast when a rank dies instead of waiting out the timeout
            try:
                out.append(q.get(timeout=1.0))
            except _queue.Empty:
                dead = [p.exitcode for p in procs if p.exitcode not in (None, 0)]
                assert not dead, f"worker exited with {dead}"
                assert time.time() - t0 < timeout, "workers timed out"
        out.sort(key=lambda x: x[0])
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    return out


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("comm", ["link", "nccl"])
def test_row_sharded_matches_single_process(comm):
    world, n, d = 2, 1024, 256
    port = 29700 + (os.getpid() % 2000) + (7 if comm == "link" else 0)
    out = _run(_worker, (port, n, d, comm), world)
    a, b = O.make_inputs(n, d, seed=33)
    ref = O.ref_step(a.double(), b.double(), O.LOGIT_SCALE_INIT)
    nl = n // world
    rel = lambda x, r: float((torch.as_tensor(x).double() - r.double()).norm() / r.double().norm())
    for rank, loss, da, db, dt in out:
        assert abs(loss - float(ref["loss"])) <= 1e-3 * abs(float(ref["loss"]))
        assert rel(da, ref["d_a"][rank * nl:(rank + 1) * nl]) <= 2e-2
        assert rel(db, ref["d_b"][rank * nl:(rank + 1) * nl]) <= 2e-2
        assert abs(dt - float(ref["d_logit_scale"])) <= 2e-2 * abs(float(ref["d_logit_scale"]))


def _worker_topk_and_graph(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ.setdefault("CLIPNCE_LINK_TIMEOUT_MS", "30000")   # a lost rank fails the test in 30 s, not in 10 min
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from clip_dplm_b200.graph import GraphedClipStep
        from clip_dplm_b200.retrieval import topk_similarity
        # (1) library row-sharded retrieval, candidates merged over NCCL
        g = torch.Generator().manual_seed(9)
        qs, lib = torch.randn(200, 128, generator=g).bfloat16(), torch.randn(3000, 128, generator=g).bfloat16()
        nl = lib.shape[0] // world
        s, i = topk_similarity(qs.cuda(), lib[rank * nl:(rank + 1) * nl].cuda(), 10, group=dist.group.WORLD)
        # (2) the row-sharded training step replayed as one CUDA graph (collectives captured)
        n, d = 1024, 256
        a, b = O.make_inputs(n, d, seed=33)
        ml = n // world
        step = GraphedClipStep(ml, d, group=dist.group.WORLD)
        out = None
        for ls in (O.LOGIT_SCALE_INIT, 2.2):
            loss, da, db, dt = step(a[rank * ml:(rank + 1) * ml].cuda().bfloat16(), b[rank * ml:(rank + 1) * ml].cuda().bfloat16(), ls)
            torch.cuda.synchronize()
            out = (float(loss), da.float().cpu().numpy(), db.float().cpu().numpy(), float(dt))
        q.put((rank, s.cpu().numpy(), i.cpu().numpy(), out))
        step.close()                # a live graph holding captured NCCL kernels would stall the communicator teardown
        from clip_dplm_b200 import exchange
        exchange.reset()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("n,d,ls,mix,a_dtype", [(1024, 256, O.LOGIT_SCALE_INIT, 0.5, "bfloat16"),
                                                (8192, 512, O.LOGIT_SCALE_INIT, 0.5, "bfloat16"),
                                                (4096, 512, math.log(100.0), 0.12, "bfloat16"),
                                                (1024, 256, O.LOGIT_SCALE_INIT, 0.5, "float32")])
def test_row_sharded_two_sided_backward(n, d, ls, mix, a_dtype):
    """The row-sharded step through the two-sided kernel: local A rows x all columns in one sweep, dA finished from the
    sweep's slabs, every owner's partial dB stored into its slot over NVLink peer memory (contraction + reduce-scatter),
    summed in fixed order -- against the sampled-row CPU oracle on the concatenated batch."""
    import numpy as np
    from oracle import sampled as SO
    world = 2
    # the third case runs kernel family 2 (true maxima; the clamp(max=100) regime of old/clip_opt.py:100) row-sharded;
    # the last one fp32 A rows with bf16 B rows: the two sides are finished with different types
    out = _run(_worker, (21700 + (os.getpid() % 2000), n, d, "link"), world,
               extra=(True, ls, mix, getattr(torch, a_dtype)))
    a, b = O.make_inputs(n, d, seed=33, mix=mix)
    rng = np.random.default_rng(n)
    rows = np.sort(rng.choice(n, 128, replace=False))
    ref = SO.sampled_reference(a, b, math.exp(ls), rows, rows)
    da = np.concatenate([o[2] for o in out])
    db = np.concatenate([o[3] for o in out])
    for rank, loss, _, _, dt in out:
        cmp = SO.compare(ref, loss, da[rows], db[rows], dt)
        assert cmp["ok"], cmp


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_nccl_sharded_retrieval_and_graphed_step():
    world = 2
    out = _run(_worker_topk_and_graph, (27700 + (os.getpid() % 2000),), world, timeout=120)
    g = torch.Generator().manual_seed(9)
    qs, lib = torch.randn(200, 128, generator=g).bfloat16(), torch.randn(3000, 128, generator=g).bfloat16()
    s_ref, i_ref, sim = O.ref_topk(qs.double(), lib.double(), 10)
    a, b = O.make_inputs(1024, 256, seed=33)
    ref = O.ref_step(a.double(), b.double(), 2.2)
    rel = lambda x, r: float((torch.as_tensor(x).double() - r.double()).norm() / r.double().norm())
    for rank, s, i, (loss, da, db, dt) in out:
        assert torch.allclose(torch.from_numpy(s).double(), s_ref, atol=2e-5, rtol=0)
        assert torch.allclose(torch.gather(sim, 1, torch.from_numpy(i)), s_ref, atol=2e-5, rtol=0)
        assert abs(loss - float(ref["loss"])) <= 1e-3 * abs(float(ref["loss"]))
        assert rel(da, ref["d_a"][rank * 512:(rank + 1) * 512]) <= 2e-2 and rel(db, ref["d_b"][rank * 512:(rank + 1) * 512]) <= 2e-2
        assert abs(dt - float(ref["d_logit_scale"])) <= 2e-2 * abs(float(ref["d_logit_scale"]))


def _worker_sequence(rank, world, port, q):
    """A sequence of steps through ONE set of peer buffers: train, evaluate (no backward), train with other inputs and
    scale, two forwards before their backwards (two leases), fp32 check mode (exact kernels: true (max, sum) pairs
    exchanged), hard-negative cache columns.  Every result is checked on the parent against the oracle."""
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ.setdefault("CLIPNCE_LINK_TIMEOUT_MS", "30000")   # a lost rank fails the test in 30 s, not in 10 min
    os.environ["CLIPNCE_COMM"] = "link"
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from clip_dplm_b200 import exchange, fused_clip_loss
        G = dist.group.WORLD
        res = []

        def shard(x, n):
            nl = n // world
            return x[rank * nl:(rank + 1) * nl]

        def train(n, d, seed, ls, dtype=torch.bfloat16, n_extra=0, **kw):
            a, b = O.make_inputs(n, d, n_cols=n + n_extra, seed=seed)
            extra = torch.nn.functional.normalize(b[n:], dim=-1).cuda().to(dtype) if n_extra else None
            ac = shard(a, n).cuda().to(dtype).requires_grad_(True)
            bc = shard(b[:n], n).cuda().to(dtype).requires_grad_(True)
            t = torch.tensor(ls, device="cuda", requires_grad=True)
            loss = fused_clip_loss(ac, bc, t, group=G, extra_cols=extra, **kw)
            return loss, ac, bc, t

        def finish(loss, ac, bc, t):
            loss.backward()
            torch.cuda.synchronize()
            res.append((float(loss.detach()), ac.grad.float().cpu().numpy(), bc.grad.float().cpu().numpy(), float(t.grad)))

        finish(*train(1024, 256, 33, O.LOGIT_SCALE_INIT))                 # 0
        with torch.no_grad():                                             # 1: evaluation, no backward
            a, b = O.make_inputs(1024, 256, seed=34)
            le = fused_clip_loss(shard(a, 1024).cuda().bfloat16(), shard(b, 1024).cuda().bfloat16(), 2.0, group=G)
            res.append((float(le),))
        finish(*train(1024, 256, 35, 2.2))                                # 2: same buffers, other inputs and scale
        s1 = train(1024, 256, 36, 2.4)                                    # 3, 4: two live steps -> two leases
        s2 = train(1024, 256, 37, 2.5)
        finish(*s1)
        finish(*s2)
        finish(*train(512, 128, 38, 1.0, dtype=torch.float32))            # 5: fp32 check mode
        finish(*train(1024, 256, 39, O.LOGIT_SCALE_INIT, n_extra=256))    # 6: cache columns
        finish(*train(1024, 256, 40, 2.3, symmetric=False))               # 7: one-directional
        assert exchange.comm_kind(G) == "link"
        for fl in exchange._Pool.free.values():
            for x in fl:
                x.check()
        n_alloc = dict((k[1:4], v) for k, v in exchange._Pool.n_alloc.items())
        q.put((rank, res, n_alloc))
        exchange.reset()
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_peer_exchange_step_sequence():
    world = 2
    out = _run(_worker_sequence, (25700 + (os.getpid() % 2000),), world)
    rel = lambda x, r: float((torch.as_tensor(x).double() - r.double()).norm() / r.double().norm())

    def check(got, n, d, seed, ls, rank, tol_l=1e-3, tol_g=2e-2, n_extra=0, **kw):
        a, b = O.make_inputs(n, d, n_cols=n + n_extra, seed=seed)
        okw = dict(kw)
        if n_extra:
            okw["extra_cols"] = torch.nn.functional.normalize(b[n:], dim=-1).bfloat16().double()
        if tol_g > 1e-3:   # the bf16 path sees bf16-rounded inputs
            a, b = a.bfloat16(), b.bfloat16()
        ref = O.ref_step(a.double(), b[:n].double(), ls, **okw)
        nl = n // world
        loss, da, db, dt = got
        assert abs(loss - float(ref["loss"])) <= tol_l * abs(float(ref["loss"]))
        assert rel(da, ref["d_a"][rank * nl:(rank + 1) * nl]) <= tol_g
        assert rel(db, ref["d_b"][rank * nl:(rank + 1) * nl]) <= tol_g
        assert abs(dt - float(ref["d_logit_scale"])) <= max(tol_g, 1e-4) * abs(float(ref["d_logit_scale"]))

    for rank, res, n_alloc in out:
        check(res[0], 1024, 256, 33, O.LOGIT_SCALE_INIT, rank)
        a, b = O.make_inputs(1024, 256, seed=34)
        ref = O.ref_step(a.bfloat16().double(), b.bfloat16().double(), 2.0)
        assert abs(res[1][0] - float(ref["loss"])) <= 1e-3 * abs(float(ref["loss"]))
        check(res[2], 1024, 256, 35, 2.2, rank)
        check(res[3], 1024, 256, 36, 2.4, rank)
        check(res[4], 1024, 256, 37, 2.5, rank)
        check(res[5], 512, 128, 38, 1.0, rank, tol_l=1e-5, tol_g=5e-5)
        check(res[6], 1024, 256, 39, O.LOGIT_SCALE_INIT, rank, n_extra=256)
        check(res[7], 1024, 256, 40, 2.3, rank, symmetric=False)
        assert n_alloc[(512, 256, 1024)] == 2          # steps 0-4 and 7 shared two sets of buffers


def _worker_single(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ.setdefault("CLIPNCE_LINK_TIMEOUT_MS", "30000")   # a lost rank fails the test in 30 s, not in 10 min
    torch.cuda.set_device(0)
    dist.init_process_group("nccl", rank=0, world_size=1, device_id=torch.device("cuda", 0))
    try:
        from clip_dplm_b200 import exchange
        from clip_dplm_b200.engine import default_engine
        eng = default_engine()
        n, d = 300, 256
        x = exchange.PeerExchange(eng, dist.group.WORLD, n, d, n + 7, torch.bfloat16, torch.device("cuda", 0), "k")
        g = torch.Generator().manual_seed(5)
        ok = True
        for it in range(3):      # repeated use: epochs advance on the device
            b = torch.randn(n, d, generator=g).cuda().bfloat16()
            a = torch.randn(n, d, generator=g).cuda()
            b_c, rinv_b, y, rinv_y = x.gather_cols(b, torch.bfloat16)
            ra, _ = eng.normalize(a)
            x.gather_rows_begin(a, a.bfloat16(), ra, torch.bfloat16)
            stats = [torch.rand(n, generator=g).cuda() + 0.5 for _ in range(2)] + \
                    [torch.rand(n + 7, generator=g).cuda() + 0.5 for _ in range(2)]
            cm, cl, rm, rl = x.exchange_stats(stats[0], stats[1], stats[2], stats[3], False, True)
            xa, rinv_xa = x.gather_rows_end()
            v = torch.tensor([1.5, -2.0, float(it)], device="cuda")
            s = x.sum_scalars(v, exchange.PHASE_LOSS)
            s2 = x.sum_scalars(v * 2, exchange.PHASE_CLOSE)
            torch.cuda.synchronize()
            x.check()
            rb, _ = eng.normalize(b)
            ok &= torch.equal(y, b) and torch.equal(b_c, b) and torch.equal(rinv_y, rb) and torch.equal(rinv_b, rb)
            ok &= torch.equal(xa, a.bfloat16()) and torch.equal(rinv_xa, ra)
            ok &= torch.equal(cm, stats[2]) and torch.equal(cl, stats[3]) and torch.equal(rm, stats[0]) and torch.equal(rl, stats[1])
            ok &= torch.equal(s, v) and torch.equal(s2, v * 2)
        q.put((0, bool(ok), int(x.status[0])))
    finally:
        dist.destroy_process_group()


def test_peer_exchange_kernels_single_rank():
    """The exchange kernels on a one-rank group (runs on a single-GPU box): symmetric-memory mapping, fused
    normalise + push, statistics push + combine, one-kernel scalar sums, device-side epochs over repeated use."""
    out = _run(_worker_single, (23700 + (os.getpid() % 2000),), 1, timeout=180)
    assert out[0][1] is True and out[0][2] == 0
