"""A/B of the merged view of duplicate edges (gnnagg_set_merge_duplicates) on bench.py's workloads, one GPU.

For every workload: the graph is built by bench.Workload exactly as bench.py builds it; then the layer (or, for the
R-MAT workloads, the aggregation) is timed with merging forced off and forced on, alternating arm by arm, `--rounds`
rounds of `--steps` steps each, with bench.py's 256 MiB L2 flush before every timed step.  Reported per arm: median /
min / max of the per-round ms per step and the mean aggregation-kernel time of the library's events; per workload:
m, m', the longest run, the time to build the view and to re-sum its values (the mirror after gnnagg_set_val).
One JSON line per workload, and the automatic rule's decision for it; every line carries the card's name, power
limit and maximum SM clock as nvidia-smi reports them in the same job.

    python tools/ab_merge.py [--workloads reddit_gcn_layer_128,...] [--rounds 3] [--steps 20] [--out FILE]
"""
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

OFF, ON = 1, 2
DEFAULT = "reddit_gcn_layer_128,proteins_gcn_layer_64,arxiv_gcn_layer_32,products_gcn_layer_256,rmat26_gcn_agg_64"


def run_stats(ptr, idx):
    """(m', longest run) of the CSR on the GPU: runs of equal adjacent sources inside a row"""
    import torch

    m = idx.numel()
    head = torch.ones(m, dtype=torch.bool, device=idx.device)
    head[1:] = idx[1:] != idx[:-1]
    starts = ptr[:-1][ptr[:-1] < ptr[1:]].long()
    head[starts] = True
    pos = torch.nonzero(head).squeeze(1)
    lens = torch.diff(torch.cat([pos, torch.tensor([m], device=idx.device)]))
    return int(pos.numel()), int(lens.max().item())


def event_ms(fn, reps):
    import torch

    out = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        out.append(a.elapsed_time(b))
    return statistics.median(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default=DEFAULT)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch

    import gnnagg

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    info = gnnagg.device_info()
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    card = {"name": info["name"], "sm_count": info["sm_count"],
            "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "power limit not readable: %s" % q.stderr.strip()}
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    timed, _ = bench.make_timer(dev, None, None, flush)
    wargs = argparse.Namespace(scheduled=0, sources="rmat", halo="auto", stages=-1, locality_slices=-1)
    lines = []
    for wname in args.workloads.split(","):
        t0 = time.time()
        wl = bench.Workload(wargs, wname, 1, 0, dev, None)
        agg = wl.agg
        m = wl.m
        mm, longest = run_stats(wl.ptr, wl.idx)
        # view build (host-synchronised) and the value mirror (one extra kernel ahead of a run after set_val)
        agg.set_merge_duplicates(ON)
        torch.cuda.synchronize()
        tb = time.perf_counter()
        assert agg.merged_edges == mm, (agg.merged_edges, mm)
        build_ms = (time.perf_counter() - tb) * 1e3
        wl.step()

        def resum_step():
            agg.set_val(wl.val)
            wl.step()

        mirror_ms = event_ms(resum_step, 5) - event_ms(wl.step, 5)
        agg.set_merge_duplicates(0)
        auto_m = agg.merged_edges
        per = {OFF: [], ON: []}
        kern = {OFF: [], ON: []}
        for r in range(args.rounds):
            for arm in ((OFF, ON) if r % 2 == 0 else (ON, OFF)):
                agg.set_merge_duplicates(arm)
                prof = []
                agg.profile(True)
                per[arm].append(timed(wl.step, args.steps, args.warmup, after_step=lambda: prof.append(agg.profile_read()["agg"])))
                agg.profile(False)
                kern[arm].append(statistics.mean(prof))
        d = {"workload": wname, "gpu": card, "n": wl.n, "m": m, "merged_edges": mm, "merged_fraction": round(1 - mm / m, 4),
             "longest_run": longest, "view_build_ms": round(build_ms, 2),
             "value_mirror_ms": round(mirror_ms, 3), "automatic_rule_merges": auto_m != m,
             "rounds": args.rounds, "steps": args.steps, "setup_s": round(time.time() - t0, 1)}
        for arm, key in ((OFF, "off"), (ON, "on")):
            v = per[arm]
            d[key] = {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4),
                      "agg_kernel_ms": round(statistics.mean(kern[arm]), 4), "per_round": [round(x, 4) for x in v]}
        d["speedup_median"] = round(d["off"]["ms_median"] / d["on"]["ms_median"], 4)
        print(json.dumps(d), flush=True)
        lines.append(d)
        wl.close()
        del wl, agg
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
