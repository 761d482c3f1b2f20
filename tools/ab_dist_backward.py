"""Forward and backward steps of the peer-memory multi-GPU GCN aggregation, alternated in one job (gnnagg_dist_gcn_run /
_gcn_layer against gnnagg_dist_gcn_backward).  Launched as bench.py is launched at N > 1:

    python -m torch.distributed.run --nproc-per-node N tools/ab_dist_backward.py [--workloads ...] [--rounds 3]
                                    [--steps 10] [--out FILE]

For every workload the graph, the partition and the X shard are built by bench.Workload exactly as bench.py builds them
(`reddit_gcn_layer_128`: the weak-scaling C2 layer; `rmat26_gcn_agg_64`: the c5 strong-scaling aggregation); the rank's
peer halo is then rebuilt with backward enabled.  Forward step and backward step (dY of the aggregation's width, dX of
the shard) alternate round by round, with bench.py's 256 MiB L2 flush before every timed step.  At N = 1 the tool builds
a one-rank group over the whole graph (no halo), frees it and then times the one-GPU gnnagg_gcn_backward of the same
graph, the reference the multi-GPU rows are compared with.  Reported: median / min / max ms per step over the rounds (the max over
ranks of each round), launches per step, and the bytes every owner pulls per backward step (rows peers reference x F x 4).
Rank 0 prints one JSON line per workload, with the card's name, power limit and maximum SM clock read in the same job."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gnn-computing_b200"))

import bench  # noqa: E402

DEFAULT = "reddit_gcn_layer_128,rmat26_gcn_agg_64"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch
    import torch.distributed as tdist

    import gnnagg
    from gnnagg.partition import PeerHalo

    N = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda:%d" % local)
    torch.cuda.set_device(dev)
    dist = None
    if N > 1:
        tdist.init_process_group("nccl", device_id=dev)
        dist = tdist
    info = gnnagg.device_info()
    q = subprocess.run(["nvidia-smi", "-i", str(local), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    card = {"name": info["name"], "sm_count": info["sm_count"],
            "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "power limit not readable: %s" % q.stderr.strip()}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    timed, barrier = bench.make_timer(dev, dist, None, flush)
    wargs = argparse.Namespace(scheduled=0, sources="rmat", halo="peer", stages=-1, locality_slices=-1)
    lines = []
    for wname in args.workloads.split(","):
        t0 = time.time()
        wl = bench.Workload(wargs, wname, N, rank, dev, dist)
        stages = wl.stages if N > 1 else 0
        if wl.ph is not None:
            wl.ph.close()
        bounds = [r * wl.n for r in range(N + 1)]
        ph = PeerHalo(wl.ptr, wl.idx, wl.val, bounds, rank, N, wl.fin, remote_stages=stages, backward=True)
        wl.ph = ph
        F = wl.fin
        ph.x(0, F).copy_(wl.Xs)
        dY = torch.randn((wl.n, F), device=dev, generator=torch.Generator(device=dev).manual_seed(11 + rank))
        dX = torch.empty((wl.n, F), device=dev)
        torch.cuda.synchronize()

        def forward():
            if wl.agg_only:
                ph.gcn_run(wl.H, 0, F)
            else:
                ph.gcn_layer(wl.W, wl.H, 0)

        arms = {"forward": forward, "backward": lambda: ph.gcn_backward(dY, dX)}
        res = {a: {"ms": [], "launches": []} for a in arms}
        order = list(arms)
        for r in range(args.rounds):
            for arm in (order if r % 2 == 0 else order[::-1]):
                l0 = ph.launches
                res[arm]["ms"].append(timed(arms[arm], args.steps, args.warmup))
                res[arm]["launches"].append((ph.launches - l0) / float(args.steps + args.warmup))
                ph.check()
        num_send = ph.num_send
        if N == 1:
            # the plain single-GPU backward of the same graph, timed after the group is freed (RMAT-26 does not hold both)
            wl.ph = None
            ph.close()
            agg = gnnagg.Aggregator(wl.ptr, wl.idx, wl.val)
            agg.transpose_build(wl.src_n)
            dX1 = torch.empty((wl.src_n, F), device=dev)
            res["one_gpu_gcn_backward"] = {"ms": [], "launches": []}
            for r in range(args.rounds):
                l0 = agg.launches
                res["one_gpu_gcn_backward"]["ms"].append(timed(lambda: agg.gcn_backward(dY, dX1), args.steps, args.warmup))
                res["one_gpu_gcn_backward"]["launches"].append((agg.launches - l0) / float(args.steps + args.warmup))
            agg.close()
            del agg, dX1
        d = {"workload": wname, "n_gpus": N, "gpu": card, "F": F, "rows_per_rank": wl.n, "edges_per_rank": wl.m,
             "scaling": "strong" if wl.strong else "weak", "remote_stages": stages,
             "halo": "peer memory" if N > 1 else "none (one-rank group)", "rounds": args.rounds, "steps": args.steps,
             "backward_bytes_pulled_rank0": num_send * F * 4, "setup_s": round(time.time() - t0, 1)}
        for arm, v in res.items():
            d[arm] = {"ms_median": round(statistics.median(v["ms"]), 4), "ms_min": round(min(v["ms"]), 4),
                      "ms_max": round(max(v["ms"]), 4), "launches_per_step": v["launches"][-1],
                      "per_round_ms": [round(x, 4) for x in v["ms"]]}
        d["backward_over_forward"] = round(d["backward"]["ms_median"] / d["forward"]["ms_median"], 3)
        if rank == 0:
            print(json.dumps(d), flush=True)
            lines.append(d)
        barrier()
        wl.close()
        arms.clear()
        del wl, ph, dY, dX
        torch.cuda.empty_cache()
    if args.out and rank == 0:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")
    if dist is not None:
        tdist.barrier()
        tdist.destroy_process_group()


if __name__ == "__main__":
    main()
