"""A/B of bf16 against fp32 X shards on the peer-memory multi-GPU step (gnnagg_dist_gcn_run_bf16 / _gcn_layer_bf16 /
_gcn_layer_host_bf16 against their fp32 twins).  Launched as bench.py is launched at N > 1:

    python -m torch.distributed.run --nproc-per-node N tools/ab_dist_bf16.py [--workloads ...] [--rounds 3] [--steps 10]
                                    [--out FILE]

For every workload the graph, the partition and the fp32 X shard are built by bench.Workload exactly as bench.py builds
them (`rmat26_gcn_agg_64`: the c5 strong-scaling aggregation, 4 row chunks; `reddit_gcn_layer_128`: the weak-scaling
layer).  The shard is written in fp32 into shard buffer 0 and, rounded once to bf16, into shard buffer 1; the two arms
alternate round by round in the same job, with bench.py's 256 MiB L2 flush before every timed step.  At N = 1 (no
multi-GPU workload in bench.py) the tool builds a one-rank group over the whole graph: the same stage kernels, no halo.
Reported per arm (medians over the rounds, the max over ranks of each round):
  * ms per step; kernels only (exchange=False: the receive slots of the previous step are re-used);
  * halo ms of gnnagg_dist_profile_read (first push issued .. last push complete) and the GB/s it gives for the bytes
    pushed per rank = rows pushed (send_counts) x F x element size, which is exactly half for bf16;
  * the host-buffer step (pinned X shard -> H2D -> step -> D2H, synchronised), for fp32 shards up to 8 GiB;
  * speedup (c5) or weak-scaling efficiency (reddit) against BOTH single-GPU references: the fp32 and the bf16 runs of
    the same workload on one GPU (profiles/c5_base_1gpu.json / BASELINE §6.2 and profiles/r4_ab_bf16.jsonl).
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

DEFAULT = "rmat26_gcn_agg_64,reddit_gcn_layer_128"
# the host-buffer step pins the X shard (in both dtypes), H and W in host memory: skipped above this shard size (the
# whole RMAT-26 X of a one-rank group is 17 GB)
E2E_MAX_SHARD_BYTES = 8 << 30
# one-GPU ms per step of the same workloads (B200, 1000 W): fp32 from the base of bench.py's strong-scaling series and the
# reddit headline, bf16 from tools/ab_bf16.py (profiles/r4_ab_bf16.jsonl)
REF_1GPU = {"rmat26_gcn_agg_64": {"fp32": 35.7, "bf16": 30.07}, "reddit_gcn_layer_128": {"fp32": 2.022, "bf16": 1.479}}


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
        if N == 1:
            wl.ph = PeerHalo(wl.ptr, wl.idx, wl.val, [0, wl.n], 0, 1, wl.fin, remote_stages=0)
        ph, F = wl.ph, wl.fin
        ph.x(0, F).copy_(wl.Xs)
        ph.x(1, F, torch.bfloat16).copy_(wl.Xs)
        torch.cuda.synchronize()
        arms = {"fp32": (0, torch.float32, 4), "bf16": (1, torch.bfloat16, 2)}

        def step(arm, exchange=True):
            buf, dt, _ = arms[arm]
            if wl.agg_only:
                ph.gcn_run(wl.H, buf, F, exchange=exchange, dtype=dt)
            else:
                ph.gcn_layer(wl.W, wl.H, buf, exchange=exchange, dtype=dt)

        e2e = 4 * wl.n * F <= E2E_MAX_SHARD_BYTES
        hX = hW = hH = None
        if e2e:
            hX = {"fp32": torch.empty((wl.n, F), pin_memory=True).copy_(wl.Xs),
                  "bf16": torch.empty((wl.n, F), dtype=torch.bfloat16, pin_memory=True).copy_(wl.Xs)}
            hW = None if wl.agg_only else torch.empty(tuple(wl.W.shape), pin_memory=True).copy_(wl.W)
            hH = torch.empty(tuple(wl.H.shape), pin_memory=True)
        res = {a: {"ms": [], "kernels_ms": [], "halo_ms": [], "e2e_ms": [], "launches": []} for a in arms}
        order = list(arms)
        for r in range(args.rounds):
            for arm in (order if r % 2 == 0 else order[::-1]):
                prof = []
                ph.profile(True)
                l0 = ph.launches
                res[arm]["ms"].append(timed(lambda: step(arm), args.steps, args.warmup, after_step=lambda: prof.append(ph.profile_read())))
                res[arm]["launches"].append((ph.launches - l0) / float(args.steps + args.warmup))
                ph.profile(False)
                res[arm]["halo_ms"].append(bench.max_over_ranks(statistics.mean(p["exchange"] for p in prof), dev, dist))
                res[arm]["kernels_ms"].append(timed(lambda: step(arm, exchange=False), args.steps, args.warmup))
                if e2e:
                    res[arm]["e2e_ms"].append(timed(lambda: ph.gcn_layer_host(hX[arm], hW, hH), max(3, args.steps // 2), 2))
                ph.check()
        d = {"workload": wname, "n_gpus": N, "gpu": card, "F": F, "rows_per_rank": wl.n, "edges_per_rank": wl.m,
             "scaling": "strong" if wl.strong else "weak", "remote_stages": wl.stages if N > 1 else 0,
             "halo": "peer memory" if N > 1 else "none (one-rank group)", "rounds": args.rounds, "steps": args.steps,
             "setup_s": round(time.time() - t0, 1)}
        ref = REF_1GPU.get(wname, {})
        for arm, (_, _, eb) in arms.items():
            v = res[arm]
            med = lambda k: round(statistics.median(v[k]), 4)
            pushed = ph.num_send * F * eb
            a = {"ms_median": med("ms"), "ms_min": round(min(v["ms"]), 4), "ms_max": round(max(v["ms"]), 4),
                 "kernels_only_ms": med("kernels_ms"), "halo_ms": med("halo_ms"), "bytes_pushed_rank0": pushed,
                 "halo_GBps_rank0": round(pushed / (med("halo_ms") * 1e-3) / 1e9, 1) if N > 1 and med("halo_ms") > 0 else None,
                 "e2e_host_ms": med("e2e_ms") if e2e else None, "launches_per_step": v["launches"][-1], "per_round_ms": [round(x, 4) for x in v["ms"]]}
            for rname, rms in ref.items():
                key = "speedup_vs_1gpu_%s" % rname if wl.strong else "efficiency_vs_1gpu_%s" % rname
                a[key] = round(rms / a["ms_median"], 3)
            d[arm] = a
        d["one_gpu_references_ms"] = ref
        d["speedup_bf16_over_fp32"] = round(d["fp32"]["ms_median"] / d["bf16"]["ms_median"], 4)
        if rank == 0:
            print(json.dumps(d), flush=True)
            lines.append(d)
        barrier()
        wl.close()
        del wl, ph, hX, hW, hH
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
