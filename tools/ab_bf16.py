"""A/B of bf16 against fp32 storage of X (gnnagg_gcn_run_bf16 / gnnagg_gcn_layer_bf16) on bench.py's workloads, one GPU.

For every workload: the graph and the fp32 X are built by bench.Workload exactly as bench.py builds them, and X_b is X
rounded once to bf16.  The layer (or, for the R-MAT workload, the aggregation) is timed with X and with X_b at the same
F, the automatic rules (merged view, locality slices) in force, alternating arm by arm, `--rounds` rounds of `--steps`
steps each, with bench.py's 256 MiB L2 flush before every timed step.  Reported per arm: median / min / max of the
per-round ms per step and the mean aggregation-kernel time of the library's events.

Accuracy, on a fixed sample of rows (numpy default_rng(0)) of the aggregation A X:
  * bf16_gate_fraction: max |y_b - y64| / (1e-5 * sum|val * x|) with y64 the fp64 oracle of the bf16-rounded X
    (<= 1 passes the project's fp32 parity gate);
  * rounding_cost: max |y_b - y_fp32| of the bf16 output against the fp32-input output, absolute and as a fraction of
    sum|val * x| -- what rounding X costs a user; not a gate.
One JSON line per workload; every line carries the card's name, power limit and maximum SM clock as nvidia-smi reports
them in the same job.

    python tools/ab_bf16.py [--workloads reddit_gcn_layer_128,...] [--rounds 3] [--steps 20] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gnn-computing_b200"))

import bench  # noqa: E402

# C2 (reddit layer), the GCN layer on the C3 (proteins) shape, C4 (products), C5 (RMAT-26 aggregation)
DEFAULT = "reddit_gcn_layer_128,proteins_gcn_layer_64,products_gcn_layer_256,rmat26_gcn_agg_64"
SAMPLE_ROWS = 4096


def sampled_oracle(orc, wl, rows, X):
    """(y64, scale) of the fp64 oracle for `rows` of A X: the rows' edges, re-indexed onto the sources they touch, so
    only those rows of X leave the device"""
    import torch

    ptr = wl.ptr.cpu().numpy().astype(np.int64)
    lo, hi = ptr[rows], ptr[rows + 1]
    sel = np.concatenate([np.arange(a, b) for a, b in zip(lo, hi)]) if len(rows) else np.zeros(0, np.int64)
    sub_ptr = np.zeros(len(rows) + 1, np.int32)
    sub_ptr[1:] = np.cumsum(hi - lo)
    sel_d = torch.from_numpy(sel).to(wl.dev)
    src = wl.idx[sel_d].long()
    uniq, inv = torch.unique(src, return_inverse=True)
    Xs = X[uniq].float().cpu().numpy()
    val = wl.val[sel_d].cpu().numpy()
    return orc.spmm_f64(sub_ptr, inv.int().cpu().numpy(), val, np.ascontiguousarray(Xs))


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
    import oracle as orc

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
        X32 = wl.Xs
        Xb = X32.to(torch.bfloat16)
        arms = {"fp32": X32, "bf16": Xb}

        # accuracy of the aggregation A X on a row sample
        rows = np.sort(np.random.default_rng(0).choice(wl.n, min(SAMPLE_ROWS, wl.n), replace=False))
        rows_d = torch.from_numpy(rows).to(dev)
        Yf = agg.gcn_run(X32, torch.empty((wl.n, wl.fin), device=dev))[rows_d].cpu().numpy().astype(np.float64)
        Yb = agg.gcn_run(Xb, torch.empty((wl.n, wl.fin), device=dev))[rows_d].cpu().numpy().astype(np.float64)
        y64, scale = sampled_oracle(orc, wl, rows, Xb)
        scale = scale.astype(np.float64)
        bound = 1e-5 * scale + 1e-30
        gate_fraction = float((np.abs(Yb - y64) / bound).max())
        diff = np.abs(Yb - Yf)
        rounding = {"max_abs": float(diff.max()), "max_frac_of_terms": float((diff / (scale + 1e-30)).max()),
                    "max_abs_y_fp32": float(np.abs(Yf).max())}
        del Yf, Yb

        per = {k: [] for k in arms}
        kern = {k: [] for k in arms}
        order = list(arms)
        for r in range(args.rounds):
            for arm in (order if r % 2 == 0 else order[::-1]):
                wl.Xs = arms[arm]
                prof = []
                agg.profile(True)
                per[arm].append(timed(wl.step, args.steps, args.warmup, after_step=lambda: prof.append(agg.profile_read()["agg"])))
                agg.profile(False)
                kern[arm].append(statistics.mean(prof))
        wl.Xs = X32
        d = {"workload": wname, "gpu": card, "n": wl.n, "m": wl.m, "F": wl.fin,
             "x_bytes": {"fp32": 4 * wl.n * wl.fin, "bf16": 2 * wl.n * wl.fin},
             "rounds": args.rounds, "steps": args.steps, "sample_rows": len(rows),
             "bf16_gate_fraction": round(gate_fraction, 4), "rounding_cost": rounding,
             "setup_s": round(time.time() - t0, 1)}
        for arm in arms:
            v = per[arm]
            d[arm] = {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4),
                      "agg_kernel_ms": round(statistics.mean(kern[arm]), 4), "per_round": [round(x, 4) for x in v]}
        d["speedup_median"] = round(d["fp32"]["ms_median"] / d["bf16"]["ms_median"], 4)
        print(json.dumps(d), flush=True)
        lines.append(d)
        wl.close()
        del wl, agg, X32, Xb, arms
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
