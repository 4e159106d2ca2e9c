"""Benchmark of the hot path: contrastive fwd+bwd pairs/sec @ global batch 65536, d=512, bf16.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--n 65536] [--d 512] [--dump-outputs DIR]

One JSON line on rank 0: `value` = pairs/s with inputs resident in HBM,
`e2e` = the same through the public API from pinned HOST buffers (H2D of the embeddings + D2H of the
loss inside the timed region), `roofline` for the dominant kernel (tcgen05 backward side), and a
`cpu_baseline` (the reference's op sequence on the box's host cores, bounded sample).

N > 1 (torchrun, one rank per GPU, NCCL): the global batch is row-sharded -- strong scaling at the
named global batch (BASELINE.json: "65536 ... at 1/2/4/8 GPU").
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "contrastive_fwd_bwd_pairs_per_sec"
UNIT = "pairs/s"


def load_peaks():
    try:
        p = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return {"burst": float(p["bf16_tflops"]), "sustained": float(p["bf16_tflops_sustained"]), "hbm": float(p["hbm_gbs"]),
                "src": "measured"}
    except Exception:
        return {"burst": 1590.0, "sustained": 1400.0, "hbm": 6650.0, "src": "fallback"}


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of this rank's GPU through NVML while the timed region runs (NVML is initialised
    before the region starts, one sample every 5 ms: the timed region of the default run is ~150 ms)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
        self._nv = self._h = None
        try:
            import pynvml as nv
            nv.nvmlInit()
            self._nv, self._h = nv, nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(self._h, nv.NVML_CLOCK_SM)
        except Exception as e:  # NVML missing: report that instead of inventing clocks
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")

    def run(self):
        nv, h = self._nv, self._h
        if nv is None:
            return
        names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                 "hw_power_brake": 0x80, "sync_boost": 0x10, "applications_clocks": 0x2}
        try:
            while not self._stop_evt.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
                time.sleep(0.005)
        except Exception as e:
            self.reasons.add(f"nvml_error:{type(e).__name__}")

    def finish(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def measured_traffic(n_global, d, world, two_sided):
    """DRAM bytes per launch of the dominant kernel from the committed `ncu --set full` capture (dram__bytes_read.sum +
    dram__bytes_write.sum), valid for the configuration it was captured on (N = 65536, d = 512, one GPU); None otherwise.
    Round 2: pair2::bwd2_kernel (profiles/r2_ncu_full_two_sided_n65536.csv, column 3); round-1 kernel: pair::bwd_kernel."""
    if (n_global, d, world) != (65536, 512, 1):
        return None
    name, unit = ("r2_ncu_full_two_sided_n65536.csv", "Gbyte") if two_sided else ("r1_ncu_full_pair_kernels_n65536.csv", "Mbyte")
    try:
        import csv
        rd = wr = None
        for row in csv.reader(open(os.path.join(ROOT, "profiles", name))):
            if row and row[0].startswith("dram__bytes_read.sum") and row[1] == unit:
                rd = float(row[3])
            if row and row[0].startswith("dram__bytes_write.sum") and row[1] == unit:
                wr = float(row[3])
        mult = 1e9 if unit == "Gbyte" else 1e6
        return (rd + wr) * mult if rd is not None and wr is not None else None
    except Exception:
        return None


def visible_gpu_index(local_rank):
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        try:
            return int(vis.split(",")[local_rank])
        except Exception:
            return local_rank
    return local_rank


# ------------------------------------------------------------------------------------------------ reference arm
def reference_step_sample(n_global, d, rows, steps, warmup, threads, scale=1 / 0.07, mix=0.5):
    """The reference's own op sequence (oracle/ref_step.py == old/clip.py:63-67 + rna_clip_codes.ipynb:
    1952-1953 + loss.backward()) on the host cores, on a bounded sample of the workload: a block of
    `rows` rows of the global batch against ALL n_global columns, so every sampled pair costs what it costs
    in the full problem (the full 65536^2 fp32 logits + autograd buffers need ~86 GB and do not fit)."""
    import torch
    import torch.nn.functional as F
    from oracle import ref_step as O
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(1234)
    a = torch.randn(rows, d, generator=g).to(torch.bfloat16).float()
    b = torch.randn(n_global, d, generator=g).to(torch.bfloat16).float()
    b[:rows] = (mix * a + (1.0 - mix) * b[:rows]).to(torch.bfloat16).float()
    t = torch.tensor(math.log(scale))
    times = []
    for it in range(warmup + steps):
        ar, br, tr = a.clone().requires_grad_(True), b.clone().requires_grad_(True), t.clone().requires_grad_(True)
        t0 = time.perf_counter()
        sim, _, _ = O.ref_logits(ar, br, tr)                      # [rows, n_global]
        labels = torch.arange(rows)
        loss = (F.cross_entropy(sim, labels) + F.cross_entropy(sim[:, :rows].t(), labels)) / 2
        loss.backward()
        dt = time.perf_counter() - t0
        if it >= warmup:
            times.append(dt)
    t_med = sorted(times)[len(times) // 2]
    return rows / t_med, t_med


def workload_desc(n, d):
    """The same description on both arms (ours computes in bf16, the reference arm in fp32 on the same rounded values)."""
    return (f"symmetric InfoNCE fwd+bwd, global batch {n}, d={d}, bf16 embeddings (b = 0.5a + 0.5 noise), "
            f"logit_scale = ln(1/0.07)")


def config_dict(n, d, scale=1 / 0.07, mix=0.5):
    """`config` of the JSON line -- byte-identical on both arms (what differs between them lives under `run`)."""
    wl = workload_desc(n, d)
    if abs(scale - 1 / 0.07) > 1e-9:
        wl = wl.replace("logit_scale = ln(1/0.07)", f"logit_scale = ln({scale:g})")
    if mix != 0.5:
        wl = wl.replace("b = 0.5a + 0.5 noise", f"b = {mix:g}a + {1 - mix:g} noise")
    return {"workload": wl, "global_batch": n, "d": d,
            "l2": f"no flush: operands + outputs + partials of one step (>= {max(1, 8 * n * d // 1000000)} MB at this size; "
                  "450 MB at N=65536) exceed the 126 MB L2"}


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    rows = args.ref_rows
    value, t_med = reference_step_sample(args.n, args.d, rows, args.steps, max(args.warmup, 1), threads, args.scale, args.mix)
    sample = (f"{rows} rows of the global batch x all {args.n} columns per step (per-pair cost identical to the full "
              f"problem; full N^2 fp32 logits do not fit in host RAM), fp32, torch CPU {threads} threads")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_med, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.n, args.d, args.scale, args.mix),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def gathered(x, group, world):
    """The row shards of every rank, concatenated in rank order (NCCL, untimed); `x` itself on one GPU."""
    if world == 1:
        return x
    import torch
    import torch.distributed as dist
    out = torch.empty((world * x.shape[0],) + tuple(x.shape[1:]), dtype=x.dtype, device=x.device)
    dist.all_gather_into_tensor(out, x.contiguous(), group=group)
    return out


# ------------------------------------------------------------------------------------------------ outputs
DUMP_GRAD_BYTES = 32 << 20     # --dump-outputs: the two gradient arrays together, as float32


def dump_outputs(out_dir, outs, group, rank, world):
    """--dump-outputs: what the timed step returns to its caller -- loss, d_a, d_b, d_logit_scale -- as float32 .npy files
    in `out_dir`, so that two builds can be compared output for output (the inputs are seeded).  Gradients of every
    rank are gathered to rank 0; above DUMP_GRAD_BYTES a fixed, seeded sample of global rows is written (`rows.npy`,
    float64, holds their indices)."""
    import numpy as np
    import torch
    loss, da, db, dls = outs
    da, db = gathered(da, group, world), gathered(db, group, world)
    if rank != 0:
        return
    n, d = da.shape
    k = min(n, DUMP_GRAD_BYTES // (2 * 4 * d))
    rows = np.arange(n) if k == n else np.sort(np.random.default_rng(20261020).choice(n, size=k, replace=False))
    idx = torch.as_tensor(rows, device=da.device)
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": loss, "d_a": da[idx], "d_b": db[idx], "d_logit_scale": dls}
    for name, x in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), x.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "rows.npy"), rows.astype(np.float64))


# ------------------------------------------------------------------------------------------------ parity
def parity_check(step_fn, a, b, logit_scale, group, rank, world, n_rows_sample):
    """One extra step OUTSIDE the timed region, compared with the sampled-row CPU oracle (oracle/sampled.py) at the
    benchmarked shape: the loss against a blockwise pass over all N x N logits on the host, d logit_scale, and the
    gradient rows dA[i], dB[j] of `n_rows_sample` random GLOBAL indices against all N columns / rows in float64.
    N > 1: inputs and gradients of every rank are gathered to rank 0 first (NCCL, untimed) -- the sample covers all ranks'
    shards.  -> the `parity` dict on rank 0, None elsewhere."""
    import numpy as np
    import torch
    loss, da, db, dls = step_fn()
    torch.cuda.synchronize()
    a_all, b_all, da_all, db_all = (gathered(x, group, world) for x in (a, b, da, db))
    if rank != 0:
        return None
    from oracle import sampled as SO
    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    n = a_all.shape[0]
    rng = np.random.default_rng(20261018)
    k = min(n_rows_sample, n)
    rows_a = np.sort(rng.choice(n, size=k, replace=False))
    rows_b = np.sort(rng.choice(n, size=k, replace=False))
    s = math.exp(float(logit_scale.detach()))
    ref = SO.sampled_reference(a_all.float().cpu(), b_all.float().cpu(), s, rows_a, rows_b)
    out = SO.compare(ref, float(loss), da_all[torch.as_tensor(rows_a, device=da_all.device)].float().cpu().numpy(),
                     db_all[torch.as_tensor(rows_b, device=db_all.device)].float().cpu().numpy(), float(dls))
    out.update({"against": "oracle/sampled.py: blockwise host pass over all N^2 logits (loss, d logit_scale) + float64 "
                           "gradient rows of the sampled global indices", "n": int(n), "host_seconds": round(time.perf_counter() - t0, 1)})
    return out


# ------------------------------------------------------------------------------------------------ our arm
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from clip_dplm_b200 import fused_clip_loss
    from clip_dplm_b200.engine import CudaEngine

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    group = dist.group.WORLD if world > 1 else None
    n_global, d = args.n, args.d
    assert n_global % world == 0
    n_local = n_global // world
    peaks = load_peaks()

    class TimedEngine(CudaEngine):
        """Records CUDA events around the two contraction entry points and counts kernel launches."""

        def __init__(self):
            super().__init__()
            self.ev, self.launches, self.on = {"fwd": [], "bwd": [], "bwd2": []}, 0, False

        def _timed(self, key, fn, *a, **k):
            if not self.on:
                return fn(*a, **k)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            self.ev[key].append((e0, e1))
            return out

        def forward(self, *a, **k):
            self.launches += 2          # contraction kernel + column-partial reduction
            return self._timed("fwd", super().forward, *a, **k)

        def backward(self, *a, **k):
            self.launches += 2 if k.get("want_dscale", True) else 1
            return self._timed("bwd", super().backward, *a, **k)

        def backward_dx(self, *a, **k):
            # contraction kernel + finish_rows (split sum, row dots, normalise backward) [+ the scalar reduction]
            self.launches += 3 if k.get("want_dscale", True) else 2
            return self._timed("bwd", super().backward_dx, *a, **k)

        def backward_both(self, *a, **k):
            # the two-sided contraction kernel, 2 x finish_rows, the scalar reduction
            self.launches += 4
            return self._timed("bwd2", super().backward_both, *a, **k)

        def backward_both_sharded(self, *a, **k):
            # the two-sided contraction + reduce-scatter kernel, finish_rows of side A, the scalar reduction
            self.launches += 3
            return self._timed("bwd2", super().backward_both_sharded, *a, **k)

        def finish_slots(self, *a, **k):
            self.launches += 1
            return super().finish_slots(*a, **k)

        def group_forward(self, *a, **k):
            # small batches: grouped launch (DESIGN.md 5.10) -- sweep, two partial reductions, per-problem losses
            self.launches += 4
            return self._timed("fwd", super().group_forward, *a, **k)

        def group_backward(self, *a, **k):
            # soft-max weights, ONE sweep over both backward sides, finishing pass, scalar reduction
            self.launches += 4
            self.grouped = True
            return self._timed("bwd2", super().group_backward, *a, **k)

        def backward_both_sharded_sweep(self, *a, **k):
            self.launches += 1          # the two-sided contraction + reduce-scatter kernel
            return self._timed("bwd2", super().backward_both_sharded_sweep, *a, **k)

        def finish_sharded(self, *a, **k):
            self.launches += 2          # both tails in one launch + the scalar reduction
            return super().finish_sharded(*a, **k)

        def normalize(self, *a, **k):
            self.launches += 1
            return super().normalize(*a, **k)

        def stage(self, x, c_dtype, want_t=False):
            self.launches += 1 if (want_t or x.dtype != c_dtype) else 0
            return super().stage(x, c_dtype, want_t)

        def softmax_weights(self, *a, **k):
            self.launches += 1
            return super().softmax_weights(*a, **k)

        def combine_lse(self, *a, **k):
            self.launches += 1
            return super().combine_lse(*a, **k)

        def normalize_backward(self, *a, **k):
            self.launches += 1
            return super().normalize_backward(*a, **k)

        def loss(self, *a, **k):
            self.launches += 1
            return super().loss(*a, **k)

        # the exchange kernels over NVLink peer memory (one launch each)
        def link_push_rows(self, *a, **k):
            self.launches += 1
            return super().link_push_rows(*a, **k)

        def link_barrier(self, *a, **k):
            self.launches += 1
            return super().link_barrier(*a, **k)

        def forward_gathered(self, *a, **k):
            self.launches += 3          # contraction kernel + the two partial reductions (the gather runs beside it)
            return self._timed("fwd", super().forward_gathered, *a, **k)

        def link_epoch_advance(self, *a, **k):
            self.launches += 1
            return super().link_epoch_advance(*a, **k)

        def link_send_blocks(self, rows, rinv, peers, world, *a, **k):
            self.launches += world - 1  # copy-engine transfers + one flag kernel per peer
            return super().link_send_blocks(rows, rinv, peers, world, *a, **k)

        def link_copy(self, *a, **k):      # copy engines: no kernel launch
            return super().link_copy(*a, **k)

        def link_push_f32(self, *a, **k):
            self.launches += 1
            return super().link_push_f32(*a, **k)

        def link_sum_scalars(self, *a, **k):
            self.launches += 1
            return super().link_sum_scalars(*a, **k)

        def combine_partials(self, *a, **k):
            self.launches += 1
            return super().combine_partials(*a, **k)

    eng = TimedEngine()
    trace = {}
    if args.trace:
        # per-phase device timeline of one step: CUDA events around every engine call and every collective
        from clip_dplm_b200 import exchange as _xchg_mod

        def wrap(name, fn):
            def inner(*a, **k):
                if not eng.on:
                    return fn(*a, **k)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = fn(*a, **k)
                if isinstance(out, tuple) and len(out) == 2 and hasattr(out[1], "wait"):   # async collective: time to completion
                    work = out[1]

                    class _W:
                        def wait(self_inner):
                            work.wait()
                            e1.record()
                    trace.setdefault(name, []).append((e0, e1))
                    return out[0], _W()
                e1.record()
                trace.setdefault(name, []).append((e0, e1))
                return out
            return inner

        for nm in ("normalize", "stage", "softmax_weights", "combine_lse", "normalize_backward", "loss", "link_push_rows",
                   "link_barrier", "link_copy", "link_push_f32", "link_sum_scalars", "combine_partials"):
            setattr(eng, nm, wrap(nm, getattr(eng, nm)))
        _xchg_mod._all_gather = wrap("all_gather", _xchg_mod._all_gather)
        _orig_ar = dist.all_reduce
        dist.all_reduce = wrap("all_reduce", _orig_ar)
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    a = torch.randn(n_local, d, device=dev, generator=g)
    b = (args.mix * a + (1.0 - args.mix) * torch.randn(n_local, d, device=dev, generator=g)).to(torch.bfloat16)
    a = a.to(torch.bfloat16)
    logit_scale = torch.tensor(math.log(args.scale), device=dev, requires_grad=True)
    a_host = a.cpu().pin_memory()
    b_host = b.cpu().pin_memory()
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()

    def step_resident():
        # logit_scale.grad accumulates over the steps of a run (nothing clears it), as in a loop without zero_grad
        ar, br = a.detach().requires_grad_(True), b.detach().requires_grad_(True)
        loss = fused_clip_loss(ar, br, logit_scale, group=group, engine=eng)
        loss.backward()
        return loss.detach(), ar.grad, br.grad, logit_scale.grad

    def step_e2e():
        ar = a_host.to(dev, non_blocking=True).requires_grad_(True)
        br = b_host.to(dev, non_blocking=True).requires_grad_(True)
        loss = fused_clip_loss(ar, br, logit_scale, group=group, engine=eng)
        loss.backward()
        loss_host.copy_(loss.detach(), non_blocking=True)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """-> (ms for `steps` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t)
        return ms, out

    for _ in range(max(args.warmup, 3)):
        step_resident()
    if args.timeline:
        # kernel-level timeline of three steps (CUPTI through torch.profiler), rank 0 writes it as text
        from torch.profiler import profile, ProfilerActivity
        barrier()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(3):
                step_resident()
            barrier()
        if rank == 0:
            evs = [e for e in prof.events() if e.device_type is not None and "cuda" in str(e.device_type).lower()]
            evs.sort(key=lambda e: e.time_range.start)
            t0 = evs[0].time_range.start if evs else 0
            with open(args.timeline, "w") as f:
                for e in evs:
                    f.write(f"{(e.time_range.start - t0) / 1e3:10.3f} ms  {e.time_range.elapsed_us():9.1f} us  {e.name[:110]}\n")
    # eager pass: per-kernel CUDA events (roofline) and the launch count
    eng.on, eng.launches = True, 0
    ms_eager, _ = timed(step_resident, args.steps)
    launches = eng.launches
    eng.on = False
    t_fwd = sum(e0.elapsed_time(e1) for e0, e1 in eng.ev["fwd"]) / max(1, len(eng.ev["fwd"]))
    t_bwd = sum(e0.elapsed_time(e1) for e0, e1 in eng.ev["bwd"]) / max(1, len(eng.ev["bwd"]))
    two_sided = len(eng.ev["bwd2"]) > 0
    if two_sided:
        t_bwd = sum(e0.elapsed_time(e1) for e0, e1 in eng.ev["bwd2"]) / len(eng.ev["bwd2"])

    # the step as the library runs it in production: forward + backward (collectives included) replayed as ONE CUDA
    # graph (clip_dplm_b200.graph.GraphedClipStep); the logit scale is read on the device, nothing needs the host
    gstep, graph_note = None, "eager launches (--no-graph)"
    if not args.no_graph:
        try:
            from clip_dplm_b200.graph import GraphedClipStep
            gstep = GraphedClipStep(n_local, d, group=group, engine=eng)
            with torch.no_grad():
                gstep.a.copy_(a)
                gstep.b.copy_(b)
                gstep.logit_scale.copy_(logit_scale.detach())
            gstep.recapture()
            for _ in range(2):
                gstep.replay()
            torch.cuda.synchronize()
            graph_note = "one CUDA graph per step (GraphedClipStep)"
        except Exception as e:   # never lose the number to a capture problem: report eager instead and say so
            gstep, graph_note = None, f"eager launches (graph capture failed: {type(e).__name__}: {e})"[:200]
    ok = torch.tensor([1 if gstep is not None else 0], device=dev)
    if world > 1:
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    if int(ok) == 0:
        gstep = None

    sampler = ClockSampler(visible_gpu_index(local_rank))
    sampler.start()
    ms_total, outs = timed(gstep.replay if gstep is not None else step_resident, args.steps)
    clocks = sampler.finish()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outs, group, rank, world)

    feeder = None
    if gstep is not None:
        from clip_dplm_b200.graph import HostFedClipStep
        feeder = None
        e2e_split = os.environ.get("CLIPNCE_E2E_SPLIT", "auto")
        if (world >= 4 and e2e_split != "0") or (world > 1 and e2e_split == "1"):
            # row-sharded: a step captured as forward graph + backward graph, so that the next batch's H2D starts behind
            # the forward (graph.GraphedClipStep.split) instead of beside the push / barrier phase of the step.  Measured:
            # pays from 4 GPUs on (e2e gap 4.5 % -> 2.5 %); on 2 GPUs the 64 MB transfer beside the backward sweep costs
            # more than the stretched barriers did (gap -2 % -> 5 %)
            try:
                g2 = GraphedClipStep(n_local, d, group=group, engine=eng, split=True)
                with torch.no_grad():
                    g2.a.copy_(a)
                    g2.b.copy_(b)
                    g2.logit_scale.copy_(logit_scale.detach())
                g2.recapture()
                feeder = HostFedClipStep(inner=g2)
            except Exception as e:
                print(f"bench: split capture failed ({type(e).__name__}: {e}); e2e shares the one-graph step", file=sys.stderr)
                feeder = None
            okf = torch.tensor([1 if feeder is not None else 0], device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if int(okf) == 0:
                feeder = None
        if feeder is None:
            feeder = HostFedClipStep(inner=gstep)      # shares the already captured graph

    def step_e2e_graph():
        # every step: this batch's embeddings come from pinned host memory (the transfer of the NEXT batch is started
        # right away so that it overlaps this step's graph), the loss goes back to pinned host memory
        loss = feeder.step(a_host, b_host)[0]
        feeder.prefetch(a_host, b_host)
        loss_host.copy_(loss, non_blocking=True)

    e2e_fn = step_e2e_graph if gstep is not None else step_e2e
    for _ in range(2):
        e2e_fn()
    ms_e2e, _ = timed(e2e_fn, args.steps)
    if args.timeline_e2e:
        # kernel / copy timeline of four host-fed steps (CUPTI through torch.profiler), rank 0 writes it as text
        from torch.profiler import profile, ProfilerActivity
        barrier()
        with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
            for _ in range(4):
                e2e_fn()
            barrier()
        if rank == 0:
            evs = [e for e in prof.events() if e.device_type is not None and "cuda" in str(e.device_type).lower()]
            evs.sort(key=lambda e: e.time_range.start)
            t0 = evs[0].time_range.start if evs else 0
            with open(args.timeline_e2e, "w") as f:
                for e in evs:
                    f.write(f"{(e.time_range.start - t0) / 1e3:10.3f} ms  {e.time_range.elapsed_us():9.1f} us  {e.name[:110]}\n")

    comm = "none"
    if world > 1:
        from clip_dplm_b200 import exchange as _xchg
        comm = _xchg.comm_kind(group)
        torch.cuda.synchronize()
        for fl in _xchg._Pool.free.values():     # a barrier that timed out would have left its mark here
            for x in fl:
                x.check()
    final_loss = float((gstep.out[0] if gstep is not None else step_resident()[0]).detach())
    if not math.isfinite(final_loss):
        raise RuntimeError(f"bench: loss is not finite ({final_loss})")
    parity = None
    if not args.no_parity:
        def step_for_parity():   # the step that was timed (the graph when there is one), its outputs read back
            if gstep is not None:
                gstep.replay()
                return gstep.out[0], gstep.out[1], gstep.out[2], gstep.out[3]
            ar, br = a.detach().requires_grad_(True), b.detach().requires_grad_(True)
            ls = logit_scale.detach().clone().requires_grad_(True)
            loss = fused_clip_loss(ar, br, ls, group=group, engine=eng)
            loss.backward()
            return loss.detach(), ar.grad, br.grad, ls.grad
        parity = parity_check(step_for_parity, a, b, logit_scale, group, rank, world, args.parity_rows)
    if gstep is not None:
        gstep.close()     # before the process group goes away
    if world > 1:
        _xchg.reset()
    if rank != 0:
        return
    if args.trace:
        rows = [("forward (contraction + reductions)", eng.ev["fwd"]), ("backward side (avg of both)", eng.ev["bwd"])] + list(trace.items())
        print(f"--- device time per step, rank 0, N={n_global} world={world} ---", file=sys.stderr)
        for nm, evs in rows:
            tot = sum(e0.elapsed_time(e1) for e0, e1 in evs) / args.steps
            print(f"{nm:40s} {len(evs) / args.steps:5.1f} calls/step {tot:8.3f} ms/step", file=sys.stderr)
    ms_step = ms_total / args.steps
    value = n_global / (ms_step * 1e-3)
    e2e_value = n_global / (ms_e2e / args.steps * 1e-3)
    flops_step = 6.0 * n_global * n_global * d
    # dominant kernel: one backward side = recompute S tile + gradient GEMM; algorithmic work of the launch is
    # its gradient GEMM, 2 * rows * cols * d (the three launches of a step add up to 6 N^2 d)
    flops_bwd_launch = (4.0 if two_sided else 2.0) * n_local * n_global * d
    achieved = flops_bwd_launch / (t_bwd * 1e-3) / 1e12
    peak = peaks["sustained"]           # the kernel is timed inside a long, power-capped step
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        v, t_med = reference_step_sample(n_global, d, args.ref_rows, 3, 1, threads, args.scale, args.mix)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": f"{args.ref_rows} rows x all {n_global} columns per step, fp32 torch CPU, median of 3 ({t_med:.2f} s/step)"}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic",
        "config": config_dict(n_global, d, args.scale, args.mix),
        "run": {"rows_per_gpu": n_local, "parallelism": f"row-sharded x{world}" if world > 1 else "single GPU",
                "comm": {"link": "own kernels over NVLink peer memory (fused normalise+gather, pushes, device barriers)",
                         "nccl": "NCCL collectives", "none": "none"}.get(comm, comm),
                "loss": final_loss},
        "parity": parity,
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": 2 * n_local * d * 2, "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches, "launch_mode": graph_note, "eager_ms_per_step": ms_eager / args.steps,
        "roofline": {"bound": "tensor",
                     "kernel": ("pair::bwd_kernel, grouped launch (both backward sides of the pair as the two virtual problems of "
                                "one sweep + finishing pass: small batches, algorithmic 4 N^2 d of 8 N^2 d executed)"
                                if getattr(eng, "grouped", False) else
                                "pair2::bwd2_kernel (both backward sides in one sweep: logits recompute + dA and dB gradient GEMMs, "
                                "algorithmic 4 N^2 d of 6 N^2 d executed, cta_group::2)" if two_sided else
                                "pair::bwd_kernel (one backward side: logits recompute + gradient GEMM, cta_group::2)"),
                     "achieved": achieved,
                     "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak, "traffic": measured_traffic(n_global, d, world, two_sided),
                     "peak_kind": f"{peaks['src']} sustained bf16 cuBLAS", "frac_of_burst": achieved / peaks["burst"],
                     "ms_per_launch": t_bwd, "fwd_ms_per_launch": t_fwd,
                     "fwd_achieved": 2.0 * n_local * n_global * d / (t_fwd * 1e-3) / 1e12,
                     "step_tflops": flops_step / world / (ms_step * 1e-3) / 1e12,
                     "step_frac_of_burst": flops_step / world / (ms_step * 1e-3) / 1e12 / peaks["burst"]},
    }
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    if parity is not None and not parity["ok"]:
        print(f"bench: PARITY FAILED against the oracle: {parity}", file=sys.stderr, flush=True)
        sys.exit(3)


def main():
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # stdout carries exactly one JSON line
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    # (--global-batch / --embed-dim: torchrun's own parser rejects "--n" as an ambiguous abbreviation of its options)
    ap.add_argument("--n", "--global-batch", dest="n", type=int, default=65536, help="global batch")
    ap.add_argument("--d", "--embed-dim", dest="d", type=int, default=512)
    ap.add_argument("--scale", type=float, default=1 / 0.07, help="s = exp(logit_scale); beyond 40 the kernels with true "
                    "running maxima serve the step (the clamp(max=100) regime of old/clip_opt.py:100)")
    ap.add_argument("--mix", type=float, default=0.5, help="b = mix a + (1 - mix) noise (use ~0.1 with --scale 100: at 0.5 the "
                    "loss underflows to 0)")
    ap.add_argument("--ref-rows", type=int, default=1024, help="row block of the CPU reference sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the sampled-row oracle check of the benchmarked step")
    ap.add_argument("--parity-rows", type=int, default=256)
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the CUDA-graph step")
    ap.add_argument("--timeline", default=None, help="write a kernel timeline of three steps (torch.profiler) to this file")
    ap.add_argument("--timeline-e2e", dest="timeline_e2e", default=None,
                    help="write a kernel / copy timeline of four host-fed (e2e) steps to this file")
    ap.add_argument("--trace", action="store_true", help="print a per-phase device-time breakdown of the step to stderr")
    ap.add_argument("--dump-outputs", dest="dump_outputs", default=None, metavar="DIR",
                    help="write what the last timed step returned (loss, d_a, d_b, d_logit_scale; a seeded row sample of "
                         "large gradients) to DIR/<name>.npy as float32")
    ap.add_argument("--comm", default="auto", choices=["auto", "link", "nccl"],
                    help="multi-GPU exchange: this repository's kernels over NVLink peer memory (link; the default where "
                         "available) or the NCCL collectives it is measured against")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    if args.comm != "auto":
        os.environ["CLIPNCE_COMM"] = args.comm
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
