"""A/B of bf16 against fp32 storage of X for the fused GAT aggregation (gnnagg_gat_run_bf16) and its backward
(gnnagg_gat_backward_bf16), one GPU.

Graphs: synth.rmat_csr(*synth.shape_of(shape), seed=123) on the device, as test_backward_timing_full_size builds them;
X, dY ~ N(0, 1) and att ~ U(0.05, 0.95) from a seeded torch generator; X_b is X rounded once to bf16.  For every case
the forward (gat_run) and the full backward (gat_backward, both passes and the row kernels) are timed in three arms:
  fp32   the fp32 entry point on X;
  bf16   the bf16 entry point on X_b;
  widen  what a bf16 user does without it: X_b.float() and then the fp32 entry point (the widening is timed too; in
         the backward this is the cost of widening again -- a user who kept the fp32 copy alive instead pays arm fp32).
The arms alternate round by round (order reversed every other round), `--rounds` rounds of `--steps` calls each, with a
256 MiB L2 flush before every timed call.  Reported per arm: median / min / max of the per-round ms per call and, for
the forward, the mean aggregation-kernel time of the library's events (gnnagg_profile_read).  One more line times
plugin.gat_aggregate forward + backward() on reddit F=128 with a bf16 leaf against an fp32 leaf.

Accuracy:
  forward, on a fixed sample of rows (numpy default_rng(0)): bf16_gate_fraction = max |y_b - y64| / (1.2e-5 * sum|alpha x|)
    with y64 the fp64 oracle (oracle.gat_f64) of the widened X on the sampled rows' edges (<= 1 passes the GAT parity
    gate); rounding_cost = max |y_b - y_fp32| against the output from the unrounded X, absolute and as a fraction of
    sum|alpha x| -- what rounding X costs, not a gate;
  backward, whole graph: whether dX and datt of the bf16 entry point equal the fp32 entry point on the widened X bit for
    bit (same Y), and the rounding cost of dX and datt (bf16 X and its Y against fp32 X and its Y), absolute and as a
    fraction of the largest |value|.  dX = sum alpha dY does not depend on X, so its rounding cost is expected to be 0.
Every line carries the card's name, power limit and maximum SM clock as nvidia-smi reports them in the same job.

    python tools/ab_gat_bf16.py [--cases arxiv:32,reddit:128,...] [--rounds 5] [--steps 10] [--out FILE]
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

DEFAULT = "arxiv:32,reddit:32,reddit:128,proteins:64,products:256"
SAMPLE_ROWS = 4096
TOL_GAT = 1.2e-5  # __expf / __fdividef against exp() in fp64 (tests/test_gpu_gat.py)


def card_info():
    import torch

    import gnnagg

    info = gnnagg.device_info()
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"name": info["name"], "sm_count": info["sm_count"],
            "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "power limit not readable: %s" % q.stderr.strip()}


def sampled_gat_oracle(orc, ptr, idx_d, att, rows, X):
    """(y64, scale) of oracle.gat_f64 for `rows` of the GAT aggregation: the rows' edges re-indexed onto the sources
    they touch (att keeps the destination half of the rows and the source half of the sources), so only those rows of
    X leave the device"""
    import torch

    lo, hi = ptr[rows], ptr[rows + 1]
    sel = np.concatenate([np.arange(a, b) for a, b in zip(lo, hi)])
    sub_ptr = np.zeros(len(rows) + 1, np.int32)
    sub_ptr[1:] = np.cumsum(hi - lo)
    src = idx_d[torch.from_numpy(sel).to(idx_d.device)].long()
    uniq, inv = torch.unique(src, return_inverse=True)
    uq = uniq.cpu().numpy()
    sub_att = np.zeros((max(len(rows), len(uq)), 2), np.float32)
    sub_att[: len(rows), 0] = att[rows, 0]
    sub_att[: len(uq), 1] = att[uq, 1]
    Xs = np.ascontiguousarray(X[uniq].float().cpu().numpy())
    y64, _, scale = orc.gat_f64(sub_ptr, inv.int().cpu().numpy(), sub_att, Xs)
    return y64, scale


def stats(v):
    return {"ms_median": round(statistics.median(v), 4), "ms_min": round(min(v), 4), "ms_max": round(max(v), 4),
            "per_round": [round(x, 4) for x in v]}


def rounding(a, b):
    d = (a - b).abs().max().item()
    ref = b.abs().max().item()
    return {"max_abs": d, "max_frac_of_max_value": d / ref if ref else 0.0}


def same_bits(a, b):
    import torch

    return bool(torch.equal(a.view(torch.int32), b.view(torch.int32)))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cases", default=DEFAULT)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import torch

    import gnnagg
    import gnnagg.plugin as gnc
    import oracle as orc
    from gnnagg import synth

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    card = card_info()
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)

    def timed(fn, steps, warmup, after=None):
        """mean ms per call, L2 flushed before each call outside the events"""
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in evs:
            flush.fill_(1)
            a.record()
            fn()
            b.record()
            if after is not None:
                after()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in evs) / steps

    def alternate(arms, after=None):
        """{arm: [ms per round]} and {arm: [mean kernel ms per round]} (when `after` returns one value per call)"""
        per, kern, order = {k: [] for k in arms}, {k: [] for k in arms}, list(arms)
        for r in range(args.rounds):
            for arm in (order if r % 2 == 0 else order[::-1]):
                got = []
                per[arm].append(timed(arms[arm], args.steps, args.warmup, (lambda: got.append(after())) if after else None))
                if got:
                    kern[arm].append(statistics.mean(got[-args.steps:]))
        return per, kern

    lines = []
    graphs = {}
    for case in args.cases.split(","):
        shape, F = case.split(":")
        F = int(F)
        t0 = time.time()
        n, m = synth.shape_of(shape)
        if shape not in graphs:
            graphs.clear()
            torch.cuda.empty_cache()
            ptr_d, idx_d = synth.rmat_csr(n, m, seed=123, device=dev)
            agg = gnnagg.Aggregator(ptr_d, idx_d)
            agg.transpose_build()
            graphs[shape] = (ptr_d, idx_d, agg, ptr_d.cpu().numpy().astype(np.int64))
        ptr_d, idx_d, agg, ptr = graphs[shape]
        g = torch.Generator(device=dev).manual_seed(123)
        X = torch.randn((n, F), device=dev, generator=g)
        dY = torch.randn((n, F), device=dev, generator=g)
        att_d = torch.rand((n, 2), device=dev, generator=g) * 0.9 + 0.05
        Xb = X.to(torch.bfloat16)
        Xw = Xb.float()
        Y, Y2, dX, dA = (torch.empty((n, F), device=dev), torch.empty((n, F), device=dev), torch.empty((n, F), device=dev),
                         torch.empty((n, 2), device=dev))

        # ---- accuracy
        rows = np.sort(np.random.default_rng(0).choice(n, min(SAMPLE_ROWS, n), replace=False))
        rows_d = torch.from_numpy(rows).to(dev)
        Y32 = agg.gat_run(X, att_d, torch.empty((n, F), device=dev))
        Yb = agg.gat_run_bf16(Xb, att_d, torch.empty((n, F), device=dev))
        fwd_bits = same_bits(Yb, agg.gat_run(Xw, att_d, Y))
        y64, scale = sampled_gat_oracle(orc, ptr, idx_d, att_d.cpu().numpy(), rows, Xw)
        scale = scale.astype(np.float64)
        yb_s, y32_s = Yb[rows_d].cpu().numpy().astype(np.float64), Y32[rows_d].cpu().numpy().astype(np.float64)
        gate_fraction = float((np.abs(yb_s - y64) / (TOL_GAT * scale + 1e-30)).max())
        diff = np.abs(yb_s - y32_s)
        fwd_rounding = {"max_abs": float(diff.max()), "max_frac_of_terms": float((diff / (scale + 1e-30)).max()),
                        "max_abs_y_fp32": float(np.abs(y32_s).max())}
        dXb, dAb = agg.gat_backward_bf16(Xb, att_d, Yb, dY, torch.empty_like(dX), torch.empty_like(dA))
        dXw, dAw = agg.gat_backward(Xw, att_d, Yb, dY, torch.empty_like(dX), torch.empty_like(dA))
        bwd_bits = {"dX": same_bits(dXb, dXw), "datt": same_bits(dAb, dAw)}
        dX32, dA32 = agg.gat_backward(X, att_d, Y32, dY, torch.empty_like(dX), torch.empty_like(dA))
        bwd_rounding = {"dX": rounding(dXb, dX32), "datt": rounding(dAb, dA32)}
        del Y32, dXb, dAb, dXw, dAw, dX32, dA32

        # ---- forward
        agg.profile(True)
        fwd, fwd_kern = alternate({
            "fp32": lambda: agg.gat_run(X, att_d, Y),
            "bf16": lambda: agg.gat_run_bf16(Xb, att_d, Y),
            "widen": lambda: agg.gat_run(Xb.float(), att_d, Y),
        }, after=lambda: agg.profile_read()["agg"])
        agg.profile(False)
        # ---- backward (Y of the arm's own forward)
        agg.gat_run(X, att_d, Y)
        agg.gat_run_bf16(Xb, att_d, Y2)
        bwd, _ = alternate({
            "fp32": lambda: agg.gat_backward(X, att_d, Y, dY, dX, dA),
            "bf16": lambda: agg.gat_backward_bf16(Xb, att_d, Y2, dY, dX, dA),
            "widen": lambda: agg.gat_backward(Xb.float(), att_d, Y2, dY, dX, dA),
        })
        d = {"case": "%s_gat_%d" % (shape, F), "gpu": card, "n": n, "m": m, "F": F,
             "x_bytes": {"fp32": 4 * n * F, "bf16": 2 * n * F}, "rounds": args.rounds, "steps": args.steps,
             "sample_rows": len(rows), "forward_bits_equal_widened_fp32": fwd_bits, "bf16_gate_fraction": round(gate_fraction, 4),
             "forward_rounding_cost": fwd_rounding, "backward_bits_equal_widened_fp32": bwd_bits,
             "backward_rounding_cost": bwd_rounding}
        for name, per, kern in (("forward", fwd, fwd_kern), ("backward", bwd, None)):
            d[name] = {arm: dict(stats(per[arm]), **({"agg_kernel_ms": round(statistics.mean(kern[arm]), 4)} if kern else {}))
                       for arm in per}
            d[name]["speedup_median_bf16_vs_fp32"] = round(d[name]["fp32"]["ms_median"] / d[name]["bf16"]["ms_median"], 4)
            d[name]["speedup_median_bf16_vs_widen"] = round(d[name]["widen"]["ms_median"] / d[name]["bf16"]["ms_median"], 4)
        d["setup_s"] = round(time.time() - t0, 1)
        print(json.dumps(d), flush=True)
        lines.append(d)

        # ---- plugin.gat_aggregate, forward + backward(), bf16 leaf against fp32 leaf
        if (shape, F) == ("reddit", 128):
            at = gnc.gat_init(ptr_d, idx_d)

            def step(X0):
                Xl = X0.detach().requires_grad_(True)
                gnc.gat_aggregate(at, Xl, att_d).backward(dY)

            per, _ = alternate({"fp32_leaf": lambda: step(X), "bf16_leaf": lambda: step(Xb)})
            gnc.destroy(at)
            p = {"case": "reddit_gat_aggregate_fwd_bwd_128", "gpu": card, "n": n, "m": m, "F": F, "rounds": args.rounds,
                 "steps": args.steps, **{arm: stats(per[arm]) for arm in per}}
            p["speedup_median"] = round(p["fp32_leaf"]["ms_median"] / p["bf16_leaf"]["ms_median"], 4)
            print(json.dumps(p), flush=True)
            lines.append(p)
        del X, dY, att_d, Xb, Xw, Y, Y2, dX, dA, Yb
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
