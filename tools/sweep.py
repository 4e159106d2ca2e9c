"""Several bench.py configurations in ONE launch (one process group, one CUDA context per rank).

A torchrun start costs ~20 s per process before the first kernel (imports, NCCL init, symmetric-memory rendezvous), and GPU
time on a multi-GPU box is charged per GPU: comparing two exchange implementations on 8 GPUs as two bench.py runs pays that
start-up sixteen times.  This tool pays it once:

    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 tools/sweep.py \
        --configs 65536x512:link 65536x512:nccl 262144x512:link 32768x768:link --steps 20

Every configuration is `bench.run_ours` unchanged: same timing rules, the same JSON line on rank 0's stdout, in the order
of --configs (stderr carries a "# sweep: <config>" marker before each).  A measurement convenience, not part of the product path.
Format of a configuration:  <global batch>x<d>[:<comm>[:s<scale>][:parity]]   with comm in {auto, link, nccl}; s<scale> sets
exp(logit_scale) (s100: the clamp regime, weakly correlated pairs), `parity` runs the sampled-row oracle check on that line.
"""
import argparse
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--configs", nargs="+", required=True)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-graph", action="store_true")
    args = ap.parse_args()

    import torch
    import torch.distributed as dist
    import bench
    from clip_dplm_b200 import exchange

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        for cfg in args.configs:
            parts = cfg.split(":")
            shape, opts = parts[0], parts[1:]
            n, d = (int(v) for v in shape.lower().split("x"))
            comm, scale, parity = "auto", 1 / 0.07, False
            os.environ.pop("CLIPNCE_E2E_SPLIT", None)
            for o in opts:
                if o in ("auto", "link", "nccl"):
                    comm = o
                elif o == "parity":
                    parity = True
                elif o in ("split", "nosplit"):     # host-fed (e2e) step as forward graph + backward graph, or as one graph
                    os.environ["CLIPNCE_E2E_SPLIT"] = "1" if o == "split" else "0"
                elif o.startswith("s"):
                    scale = float(o[1:])
                elif o:
                    raise SystemExit(f"sweep: unknown option '{o}' in '{cfg}'")
            if comm not in ("auto", "link", "nccl"):
                raise SystemExit(f"sweep: unknown comm '{comm}' in '{cfg}'")
            if comm == "auto":
                os.environ.pop("CLIPNCE_COMM", None)
            else:
                os.environ["CLIPNCE_COMM"] = comm
            exchange.reset()     # forget the previous configuration's buffers and its link/nccl decision
            ns = argparse.Namespace(gpus=world, steps=args.steps, warmup=args.warmup, impl="ours", n=n, d=d, ref_rows=1024,
                                    no_cpu_baseline=True, no_graph=args.no_graph, timeline=None, timeline_e2e=None, trace=False,
                                    comm=comm, scale=scale, mix=0.1 if scale > 50 else 0.5, no_parity=not parity,
                                    parity_rows=256)
            if rank == 0:
                print(f"# sweep: {cfg}", file=sys.stderr, flush=True)
            bench.run_ours(ns, rank, local_rank, world)
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
