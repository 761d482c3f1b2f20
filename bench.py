#!/usr/bin/env python
"""bench.py -- headline benchmark of the neighbour-aggregation hot path (BASELINE.json).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload NAME] [--dump-outputs DIR] ...

N = 1 (default): BASELINE.json configs[1] -- the fused GCN layer H = (A X) W, feat 128 -> 128, on the
synthetic reddit-shaped power-law graph (232,965 vertices / 114,615,891 edges), one B200.
N > 1 (launched by torch.distributed.run, one rank per GPU): the same layer on a graph that is
1-D row-partitioned by destination: every rank owns a reddit-shaped row block (232,965 rows,
114,615,891 edges whose sources span all N*232,965 vertices) and the matching X shard (weak scaling).
A step = the source-feature halo, pulled from the owners' shards over NVLink peer memory by the library's
own kernels and overlapped stage by stage with the aggregation (gnnagg_dist_*, csrc/dist.cu), + the local layer.

Besides the headline, every run also measures BASELINE.json configs[4] -- GCN aggregation feat 64 on the
R-MAT scale-26 graph (2^26 vertices / 2^30 edges), the whole graph partitioned over the N ranks (strong
scaling; N = 1 gives the single-GPU base) -- and prints it as the `c5` key; at N > 1 a row sample of both
results is checked on rank 0 against the fp64 CPU oracle (`parity` keys).

A "step" = one pass of the layer over the whole graph.  Reported metric: algorithmic GB/s of the layer
(gather model of SURVEY.md 8(d): 4(n+1) + 8m + 4mF_in + 4nF_out + 4F_inF_out bytes per rank).
`value`: inputs resident in HBM; `e2e`: the same step with pinned HOST X/W/H and the copies inside the timed
region (gnnagg_gcn_layer_host at N = 1).  `--impl reference`: the reference has no CPU implementation of this
path (SURVEY 8(c)); the arm times the scalar CPU port (oracle/) on all host threads on a bounded sample.

`--dump-outputs DIR` writes the layer output H of the last timed step as DIR/H.npy (float32).  The inputs are a pure
function of the arguments (seeded graph and features), so two builds run with the same arguments can be compared
output for output; an output larger than DUMP_BYTES is written as a fixed, seeded row sample.  At N > 1 every rank
writes its own row block as DIR/H_rank<r>.npy.  The option belongs to the GPU path: `--impl reference` refuses it.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gnn-computing_b200"))

WORKLOADS = {
    # name: (shape name, feat_in, feat_out)
    "reddit_gcn_layer_128": ("reddit", 128, 128),
    "arxiv_gcn_layer_32": ("arxiv", 32, 32),
    "proteins_gcn_layer_64": ("proteins", 64, 64),
    "products_gcn_layer_256": ("products", 256, 256),
    # BASELINE.json configs[4]: GCN aggregation only on the RMAT scale-26 graph (2^26 vertices / 2^30 edges), the
    # whole graph 1-D row-partitioned over the N ranks (strong scaling); a step = halo exchange + aggregation
    "rmat26_gcn_agg_64": ("rmat26", 64, None),
    "rmat22_gcn_agg_64": ("rmat22", 64, None),   # down-scaled variant of the same workload
}
RMAT_SCALES = {"rmat26": (1 << 26, 1 << 30), "rmat22": (1 << 22, 1 << 26)}
C5_WORKLOAD = "rmat26_gcn_agg_64"
NVLINK_PEAK_GBS = 770.0  # measured peer-copy bandwidth per direction per GPU (B200_PROFILING.md); nominal 900
DUMP_BYTES = 48 << 20    # --dump-outputs: at most this many bytes of output in all (split over the ranks)


def layer_bytes(n, m, fin, fout):
    """algorithmic bytes of one fused layer (or, fout=None, of the aggregation alone) on one rank
    (SURVEY.md 8(d), gather model)"""
    if fout is None:
        return spmm_bytes(n, m, fin)
    return 4 * (n + 1) + 4 * m + 4 * m + 4 * m * fin + 4 * n * fout + 4 * fin * fout


def spmm_bytes(n, m, F):
    return 4 * (n + 1) + 8 * m + 4 * m * F + 4 * n * F


def compulsory_bytes(n, m, F, n_src=None):
    """every array once, perfect reuse (SURVEY 8(d) model A)"""
    return 4 * (n + 1) + 8 * m + 4 * (n if n_src is None else n_src) * F + 4 * n * F


class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons of one GPU through NVML while the timed region runs"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
        self.active = False

    def run(self):
        try:
            import pynvml as nv

            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {"hw_slowdown": 0x8, "sw_power_cap": 0x4, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20,
                     "hw_power_brake": 0x80, "sync_boost": 0x10, "app_clocks": 0x2}
            while not self._stop_evt.is_set():
                if self.active:
                    self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    self.reasons.update(k for k, bit in names.items() if r & bit)
                time.sleep(0.02)
        except Exception as e:  # NVML missing: report it rather than fake numbers
            self.reasons.add("nvml_unavailable:%s" % type(e).__name__)

    def result(self):
        self._stop_evt.set()
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "samples": len(s),
                "reasons": sorted(self.reasons)}


def cpu_port_time(orc, hp, hi, hv, hX, hW, rows, fin, fout):
    """seconds of the scalar CPU port (oracle.c, all OpenMP threads) on rows [0, rows)"""
    import numpy as np

    AX = np.zeros((rows, fin), np.float32)
    H = np.zeros((rows, fout), np.float32) if fout is not None else None
    t0 = time.perf_counter()
    orc.spmm_f32(hp, hi, hv, hX, 0, rows, out=AX)
    if fout is not None:
        orc.dense_f32(AX, hW, 0, rows, out=H)
    return time.perf_counter() - t0


def cpu_sample(orc, ptr, idx, val, X, W, fin, fout, budget_s):
    """times the CPU port on a leading row block sized for ~budget_s seconds; returns
    (GB/s of the sample, seconds, rows, edges)"""
    import numpy as np

    n = ptr.numel() - 1
    hp_full = ptr.cpu().numpy()
    hX, hW = X.cpu().numpy(), W.cpu().numpy()

    def block(rows):
        e = int(hp_full[rows])
        return np.ascontiguousarray(hp_full[: rows + 1]), idx[:e].cpu().numpy(), val[:e].cpu().numpy(), e

    probe_rows = int(np.searchsorted(hp_full, min(int(hp_full[-1]), 2_000_000), side="left"))
    probe_rows = max(1, min(n, probe_rows))
    hp, hi, hv, e = block(probe_rows)
    cpu_port_time(orc, hp, hi, hv, hX, hW, probe_rows, fin, fout)  # warm-up (page faults, OpenMP pool)
    t = cpu_port_time(orc, hp, hi, hv, hX, hW, probe_rows, fin, fout)
    rate = max(e, 1) / max(t, 1e-6)  # edges/s
    want_edges = int(min(int(hp_full[-1]), rate * budget_s))
    rows = max(probe_rows, min(n, int(np.searchsorted(hp_full, want_edges, side="left"))))
    hp, hi, hv, e = block(rows)
    t = min(cpu_port_time(orc, hp, hi, hv, hX, hW, rows, fin, fout) for _ in range(2))
    return layer_bytes(rows, e, fin, fout) / t / 1e9, t, rows, e


def auto_stages(shape, N):
    """groups of owners the remote part of the halo is pulled and accumulated in (gnnagg_dist_set_graph).  More groups
    = finer overlap of the pulls with the aggregation but one more read-modify-write pass over the output per group;
    chosen from the sweeps in profiles/r2_sweep_*.jsonl."""
    if N <= 1:
        return 0
    if shape in RMAT_SCALES:            # 16 edges per output row: an extra pass over Y per owner group costs more than it
        return -4                       # hides (8 GPUs: 9.2 vs 8.65 ms) -> row pipelining, 4 row chunks of the one CSR (8.05 ms; 8 chunks: 8.5-8.8)
    return min(N - 1, 3)                # 490 edges per output row: Y passes are cheap, overlap by owner groups pays


class Workload:
    """one named workload on this rank: graph block, inputs, the step functions"""

    def __init__(self, args, name, N, rank, dev, dist, stages=None, halo=None):
        import torch

        import gnnagg
        from gnnagg import synth

        self.args, self.name, self.N, self.rank, self.dev, self.dist = args, name, N, rank, dev, dist
        shape, fin, fout = WORKLOADS[name]
        self.shape, self.fin, self.fout = shape, fin, fout
        self.strong = shape in RMAT_SCALES
        self.agg_only = fout is None
        if self.strong:  # one fixed graph, partitioned: per-rank block = total / N
            n_tot, m_tot = RMAT_SCALES[shape]
            n, m = n_tot // N, m_tot // N
            what = "GCN aggregation (CSR SpMM) feat %d on the R-MAT %s graph (%d vertices / %d edges in total), %d rows / %d " \
                   "edges per GPU" % (fin, shape, n_tot, m_tot, n, m)
        else:
            n, m = synth.shape_of(shape)
            what = "fused GCN layer (CSR SpMM aggregation + dense combination) feat %d->%d on synthetic %s-shaped R-MAT graph, " \
                   "%d vertices / %d edges per GPU" % (fin, fout, shape, n, m)
        self.n, self.m, self.src_n = n, m, n * N
        self.config = {"workload": "%s: %s" % (name, what),
                       "graph": "rmat(a=.57,b=.19,c=.19,d=.05) seed=123, val=1/sqrt((deg_u+1)(deg_v+1)), X~N(0,1), W~N(0,1)/sqrt(F)",
                       "partition": "1d-row-by-destination" if N > 1 else "single-gpu",
                       "scheduled": bool(args.scheduled), "sources": args.sources,
                       "l2": "flushed between timed steps (256 MiB write) and inputs (idx+val %.0f MB, X %.0f MB) exceed the 126 MB L2"
                             % (8 * m / 1e6, 4 * n * fin / 1e6)}
        t0 = time.time()
        # graph: rank r owns rows [r*n, (r+1)*n) of an (N*n)-vertex R-MAT graph, sources are global ids
        ptr, idx = synth.rmat_csr(n, m, seed=123, device=dev, src_num_v=self.src_n if N > 1 else None,
                                  dst_prefix=rank if N > 1 else None)
        if args.sources == "uniform":
            idx = torch.randint(0, self.src_n, (m,), device=dev, dtype=torch.int32,
                                generator=torch.Generator(device=dev).manual_seed(99 + rank))
        deg = (ptr[1:] - ptr[:-1]).to(torch.float32)
        if N > 1:
            deg_all = torch.empty(self.src_n, device=dev)
            dist.all_gather_into_tensor(deg_all, deg)
            val = synth.gcn_norm_val(ptr, idx, src_deg=deg_all)
            del deg_all
        else:
            val = synth.gcn_norm_val(ptr, idx)
        self.ptr, self.idx, self.val = ptr, idx, val
        g = torch.Generator(device=dev).manual_seed(123 + rank)
        self.Xs = torch.randn((n, fin), device=dev, generator=g)          # this rank's X shard
        self.W = torch.randn((fin, fout or fin), device=dev, generator=torch.Generator(device=dev).manual_seed(7)) / fin ** 0.5
        self.H = torch.empty((n, fout or fin), device=dev)
        self.ph = self.agg = self.nccl = self.Xfull = None
        self.halo = "none"
        if N > 1:
            self._setup_multi(stages, halo or args.halo)
        else:
            self.agg = gnnagg.Aggregator(ptr, idx, val)
            if args.scheduled:
                self.agg.schedule(gnnagg.SCHED_NEIGHBOR_GROUPING, [32])
            if getattr(args, "locality_slices", -1) >= 0:
                self.agg.set_locality_slices(args.locality_slices)
                self.config["locality_slices"] = args.locality_slices
        torch.cuda.synchronize()
        self.setup_s = time.time() - t0
        self.hX = self.hW = self.hH = None

    # -------------------------------------------------------------- multi-GPU set-up
    def _setup_multi(self, stages, halo):
        import torch

        import gnnagg
        from gnnagg.partition import PeerHalo, PrunedHalo

        N, rank, dev, dist = self.N, self.rank, self.dev, self.dist
        n, fin = self.n, self.fin
        self.stages = stages if stages is not None else (self.args.stages if self.args.stages >= 0 else auto_stages(self.shape, N))
        err = ""
        if halo in ("auto", "peer"):
            try:
                self.ph = PeerHalo(self.ptr, self.idx, self.val, [r * n for r in range(N + 1)], rank, N, fin, remote_stages=self.stages)
                ok = 1
            except Exception as e:  # e.g. cudaIpcOpenMemHandle not permitted in this container
                ok, err = 0, "%s: %s" % (type(e).__name__, e)
            t = torch.tensor([ok], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            if int(t.item()) == 1:
                self.halo = "peer"
                self.ph.x(0, fin).copy_(self.Xs)
                self.config["halo"] = (
                    "peer memory: every owner pushes the rows its peers' blocks reference (rank 0 receives %d distinct remote rows = "
                    "%.1f%% of X) straight into their receive slots with 128-bit stores over NVLink (cudaIpc mappings, no NCCL in "
                    "the step); %s" % (self.ph.num_recv, 100.0 * (self.ph.num_recv + 0.0) / self.src_n,
                                       ("row pipelining: %d edge-balanced row chunks of the one CSR, chunk c starts when round c "
                                        "of the pushes (the rows it needs first) has landed" % min(-self.stages, 16)) if self.stages < 0 else
                                       "one aggregation pass after all arrivals" if self.ph.num_stages == 1 else
                                       "stage 0 = local sources, %d remote stage(s) accumulated as their owners land" % (self.ph.num_stages - 1)))
                return
            if self.ph is not None:
                self.ph = None
            if halo == "peer":
                raise RuntimeError("peer-memory halo unavailable on some rank (%s)" % (err or "another rank failed"))
        # NCCL paths (round-1 code, kept as the fallback when peer mappings are not available)
        if halo == "auto":
            frac = torch.tensor([torch.unique(self.idx).numel() / float(self.src_n)], device=dev)
            dist.broadcast(frac, src=0)
            halo = "pruned" if float(frac.item()) < 0.7 else "allgather"
        if halo == "pruned":
            self.nccl = PrunedHalo(self.ptr, self.idx, self.val, n, N, rank, fin)
            self.agg = self.nccl.agg
            self.halo = "nccl-pruned"
            self.config["halo"] = "NCCL fallback%s: pack kernel + all_to_all_single of the referenced rows (%.1f%% of X on rank 0)" % (
                (" (%s)" % err) if err else "", 100 * self.nccl.referenced_fraction)
        else:
            self.agg = gnnagg.Aggregator(self.ptr, self.idx, self.val)
            self.Xfull = torch.empty((self.src_n, fin), device=dev)
            self.halo = "nccl-allgather"
            self.config["halo"] = "NCCL fallback%s: one all-gather of X, then the layer" % ((" (%s)" % err) if err else "")

    # -------------------------------------------------------------- steps
    def step(self, exchange=True):
        sched = bool(self.args.scheduled)
        if self.ph is not None:
            if self.agg_only:
                self.ph.gcn_run(self.H, 0, self.fin, exchange=exchange)
            else:
                self.ph.gcn_layer(self.W, self.H, 0, exchange=exchange)
            return
        x = self.Xs
        if self.nccl is not None:
            x = self.nccl.exchange(self.Xs) if exchange else self.nccl.recv_buf
        elif self.Xfull is not None:
            if exchange:
                self.dist.all_gather_into_tensor(self.Xfull, self.Xs)
            x = self.Xfull
        if self.agg_only:
            self.agg.gcn_run(x, self.H, scheduled=sched)
        else:
            self.agg.gcn_layer(x, self.W, self.H, None, scheduled=sched)

    def host_buffers(self):
        import torch

        if self.hX is None:
            self.hX = torch.empty((self.n, self.fin), pin_memory=True).copy_(self.Xs)
            self.hW = torch.empty((self.fin, self.fout or self.fin), pin_memory=True).copy_(self.W)
            self.hH = torch.empty((self.n, self.fout or self.fin), pin_memory=True)

    def step_e2e(self):
        import torch

        sched = bool(self.args.scheduled)
        if self.N == 1 and self.agg_only:
            self.agg.gcn_run_host(self.hX, self.hH, scheduled=sched)
        elif self.N == 1:
            self.agg.gcn_layer_host(self.hX, self.hW, self.hH, scheduled=sched)  # H2D + layer + D2H + sync inside
        elif self.ph is not None:
            # H2D of the shard into the peer-visible buffer, the step, row-chunked copy back overlapping the last stage
            self.ph.gcn_layer_host(self.hX, None if self.agg_only else self.hW, self.hH)
        else:
            self.Xs.copy_(self.hX, non_blocking=True)
            self.step()
            self.hH.copy_(self.H, non_blocking=True)
            torch.cuda.current_stream().synchronize()

    def copies_only(self):
        """the two host copies of step_e2e alone (what PCIe / the host memory system allows on this box at this N)"""
        import torch

        dst = self.ph.x(0, self.fin) if self.ph is not None else self.Xs
        dst.copy_(self.hX, non_blocking=True)
        self.hH.copy_(self.H, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    def launch_count(self):
        if self.ph is not None:
            return self.ph.launches
        return self.agg.launches

    def close(self):
        if self.ph is not None:
            self.ph.close()
        self.ph = self.agg = self.nccl = self.Xfull = None


def make_timer(dev, dist, sampler, flush):
    import torch

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, after_step=None):
        for _ in range(warmup):
            fn()
        barrier()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        if sampler is not None:
            sampler.active = True
        for a, b in evs:
            flush.fill_(1)  # L2 flush, outside the timed events
            a.record()
            fn()
            b.record()
            if after_step is not None:
                after_step()
        barrier()
        if sampler is not None:
            sampler.active = False
        total_ms = sum(a.elapsed_time(b) for a, b in evs)
        if dist is not None:
            t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t.item())
        return total_ms / steps

    return timed, barrier


def max_over_ranks(x, dev, dist):
    import torch

    if dist is None:
        return float(x)
    t = torch.tensor([float(x)], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def output_sample(Y, budget_bytes, seed=0):
    """what a caller of the timed path receives, copied to the host: the whole output when it fits in budget_bytes,
    else a fixed row sample (rows drawn by numpy default_rng(seed) without replacement, in ascending order) -- the same
    rows on every run with the same arguments.  Returns (array, description)."""
    import numpy as np

    n, F = Y.shape
    k = min(n, max(1, budget_bytes // (Y.element_size() * F)))
    if k == n:
        return Y.cpu().numpy(), "all %d rows" % n
    rows = np.sort(np.random.default_rng(seed).choice(n, k, replace=False))
    return Y[rows].cpu().numpy(), "%d of %d rows, drawn by numpy default_rng(%d).choice(n, k, replace=False), sorted" % (k, n, seed)


def measure(wl, timed, steps, warmup, e2e=True, dump_bytes=0):
    """times one workload: step, kernels-only step, exchange span, (optionally) end-to-end.  Collective: every rank
    calls it.  dump_bytes > 0: out["output"] = output_sample() of what the last timed step computed."""
    import numpy as np

    out = {}
    prof = []
    l0 = wl.launch_count()
    if wl.ph is not None:
        wl.ph.profile(True)
        ms = timed(wl.step, steps, warmup, after_step=lambda: prof.append(wl.ph.profile_read()))
        wl.ph.profile(False)
    elif wl.N == 1:
        wl.agg.profile(True)
        ms = timed(wl.step, steps, warmup, after_step=lambda: prof.append(wl.agg.profile_read()))
        wl.agg.profile(False)
    else:
        ms = timed(wl.step, steps, warmup)
    out["launches_per_step"] = (wl.launch_count() - l0) / float(steps + warmup)
    out["ms"] = ms
    if dump_bytes > 0:  # taken before the passes below run the layer again
        out["output"] = output_sample(wl.H, dump_bytes)
    out["prof"] = {k: float(np.mean([p[k] for p in prof])) for k in prof[0]} if prof else {}
    if wl.N > 1:
        out["compute_ms"] = timed(lambda: wl.step(exchange=False), max(3, steps // 2), 2)
        if wl.ph is not None:
            out["exchange_ms"] = max_over_ranks(out["prof"]["exchange"], wl.dev, wl.dist)
            wl.ph.check()
    if e2e:
        wl.host_buffers()
        out["ms_e2e"] = timed(wl.step_e2e, max(3, steps // 2), 3)
        if wl.N > 1:
            out["ms_copies"] = timed(wl.copies_only, 3, 1)
    return out


def parity_check(wl, max_rows=1024, max_edges=3_000_000):
    """rank 0 checks a sample of its output rows against the fp64 CPU oracle.  The source rows the sample needs are
    fetched from their owners with plain NCCL send/recv (independent of the library's halo path).  Collective."""
    import numpy as np
    import torch

    dev, dist, N, rank, n, fin = wl.dev, wl.dist, wl.N, wl.rank, wl.n, wl.fin
    wl.step()  # a fresh result from the path under test
    torch.cuda.synchronize()
    count = torch.zeros(1, dtype=torch.int64, device=dev)
    if rank == 0:
        ptr, idx, val = wl.ptr, wl.idx, wl.val
        deg_all = (ptr[1:] - ptr[:-1]).long()
        hub = int(torch.argmax(deg_all).item())
        k = min(max_rows, n)
        spread = (torch.arange(k, device=dev, dtype=torch.int64) * (n - 1)) // max(k - 1, 1)   # integer arithmetic: n ~ 2^25
        rows = torch.unique(torch.cat([spread, torch.tensor([hub], device=dev)]))
        deg = deg_all[rows]
        keep = torch.cumsum(deg, 0) <= max_edges
        keep[0] = True
        rows, deg = rows[keep], deg[keep]
        sub_ptr = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=dev)
        sub_ptr[1:] = torch.cumsum(deg, 0)
        e_tot = int(sub_ptr[-1].item())
        eid = torch.arange(e_tot, device=dev) - torch.repeat_interleave(sub_ptr[:-1], deg) + torch.repeat_interleave(ptr[rows].long(), deg)
        g_src = idx[eid].long()
        U = torch.unique(g_src)
        sub_idx = torch.searchsorted(U, g_src).to(torch.int32)
        sub_val = val[eid]
        count[0] = U.numel()
    if dist is not None:
        dist.broadcast(count, src=0)
        Ub = U if rank == 0 else torch.empty(int(count.item()), dtype=torch.int64, device=dev)
        dist.broadcast(Ub, src=0)
        owner = torch.div(Ub, n, rounding_mode="floor")
        mine = Ub[owner == rank] - rank * n
        send = wl.Xs[mine].contiguous()
        if rank == 0:
            Xsub = torch.empty((Ub.numel(), fin), device=dev)
            counts = torch.bincount(owner, minlength=N).tolist()
            off = 0
            for r in range(N):
                if r == 0:
                    Xsub[off:off + counts[0]] = send
                elif counts[r]:
                    dist.recv(Xsub[off:off + counts[r]], src=r)
                off += counts[r]
        elif send.numel():
            dist.send(send, dst=0)
    else:
        Xsub = wl.Xs[U]
    res = None
    if rank == 0:
        import oracle as orc

        orc.use_all_cores()
        hp, hi, hv = sub_ptr.to(torch.int32).cpu().numpy(), sub_idx.cpu().numpy(), sub_val.cpu().numpy()
        got = wl.H[rows].cpu().numpy().astype(np.float64)
        if wl.agg_only:
            y64, scale = orc.spmm_f64(hp, hi, hv, Xsub.cpu().numpy())
        else:
            _, y64, scale = orc.gcn_layer_f64(hp, hi, hv, Xsub.cpu().numpy(), wl.W.cpu().numpy())
        err = np.abs(got - y64.astype(np.float64)) / (1e-5 * scale.astype(np.float64) + 1e-30)
        res = {"rows": int(rows.numel()), "edges": e_tot, "includes_max_degree_row": True,
               "worst_err_over_bound": round(float(err.max()), 4), "tolerance": "|y - y_fp64| <= 1e-5 * sum|terms|",
               "ok": bool(err.max() <= 1.0),
               "checked": "rank 0's output rows against oracle/oracle.c (fp64) with source rows fetched from their owners by NCCL send/recv"}
    if dist is not None:
        dist.barrier()
    return res


def c5_block(args, N, rank, dev, dist, timed, steps, warmup):
    """BASELINE.json configs[4] on the same ranks, after the headline.  Collective."""
    import torch

    stage_list = [int(s) for s in args.c5_sweep.split(",")] if args.c5_sweep else [None]
    best = None
    for st in stage_list:
        wl = Workload(args, C5_WORKLOAD, N, rank, dev, dist, stages=st)
        r = measure(wl, timed, steps, warmup, e2e=False)
        par = parity_check(wl) if N > 1 else None
        nbytes = N * spmm_bytes(wl.n, wl.m, wl.fin)
        d = {"workload": wl.config["workload"], "scaling": "strong", "ms_per_step": round(r["ms"], 4),
             "value": round(nbytes / (r["ms"] * 1e-3) / 1e9, 1), "unit": "GB/s", "steps": steps, "warmup": warmup,
             "edges_feat_per_s": round(N * wl.m * wl.fin / (r["ms"] * 1e-3), 1), "setup_s": round(wl.setup_s, 2),
             "gpu_launches_per_step": round(r["launches_per_step"], 1)}
        if N > 1:
            d["halo"] = wl.config.get("halo")
            d["compute_only_ms"] = round(r["compute_ms"], 4)
            d["exposed_exchange_ms"] = round(r["ms"] - r["compute_ms"], 4)
            if wl.ph is not None:
                ex_bytes = wl.ph.num_send * wl.fin * 4
                d["remote_stages"] = wl.stages if wl.stages < 0 else wl.ph.num_stages - 1
                d["bytes_exchanged_per_rank"] = ex_bytes
                d["exchange_ms"] = round(r["exchange_ms"], 4)
                d["nvlink_GBps_per_rank"] = round(ex_bytes / (r["exchange_ms"] * 1e-3) / 1e9, 1) if r["exchange_ms"] > 0 else None
                d["nvlink_frac_of_770"] = round(d["nvlink_GBps_per_rank"] / NVLINK_PEAK_GBS, 3) if d["nvlink_GBps_per_rank"] else None
            d["parity"] = par
            base = None
            try:
                base = json.load(open(os.path.join(ROOT, "profiles", "c5_base_1gpu.json")))["ms_per_step"]
            except Exception:
                pass
            d["base_1gpu_ms"] = base
            d["speedup_vs_1gpu"] = round(base / r["ms"], 3) if base else None
            d["base_source"] = "profiles/c5_base_1gpu.json (the N=1 `c5` value of this bench on the same pool)" if base else None
        else:
            d["kernel_ms"] = round(r["prof"].get("agg", 0.0), 4)
            d["note"] = "single-GPU base of the strong-scaling series"
            try:  # HBM fraction of the kernel from the committed ncu capture of this workload (profiles/ncu_summary.json)
                sm = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json"))).get(C5_WORKLOAD, {})
                peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0))
                if sm.get("dram_bytes_per_launch") and d["kernel_ms"] > 0:
                    d["roofline"] = {"bound": "hbm", "traffic": sm["dram_bytes_per_launch"], "peak": peak, "unit": "GB/s",
                                     "frac_dram": round(sm["dram_bytes_per_launch"] / (d["kernel_ms"] * 1e-3) / 1e9 / peak, 4),
                                     "l2_hit_pct": sm.get("l2_hit_pct"), "source": sm.get("source"),
                                     "compulsory_bytes": compulsory_bytes(wl.n, wl.m, wl.fin)}
            except Exception:
                pass
        if len(stage_list) > 1 and rank == 0:
            print(json.dumps({"c5_sweep": d}), flush=True)
        if best is None or d["ms_per_step"] < best["ms_per_step"]:
            best = d
        wl.close()
        del wl
        torch.cuda.empty_cache()
    return best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="reddit_gcn_layer_128", choices=sorted(WORKLOADS))
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="CPU work budget of the cpu_baseline sample")
    ap.add_argument("--scheduled", type=int, default=0, help="1: run the neighbour-grouped (NG=32) path")
    ap.add_argument("--sources", default="rmat", choices=["rmat", "uniform"],
                    help="rmat: the R-MAT source distribution of the workload definition (default, headline); uniform: same "
                         "degree sequence but uniformly random sources -- the cache-hostile extreme, reported as context")
    ap.add_argument("--halo", default="auto", choices=["auto", "peer", "pruned", "allgather"],
                    help="N>1: peer = the library's own NVLink peer-memory exchange (default); pruned / allgather = the NCCL "
                         "paths of round 1 (also the automatic fallback when peer mappings cannot be opened)")
    ap.add_argument("--stages", type=int, default=-1, help="N>1, peer halo: remote stages (-1 = automatic, 0 = one pass after all arrivals)")
    ap.add_argument("--sweep", default="", help="N>1: comma-separated remote-stage counts to time on the headline workload")
    ap.add_argument("--locality-slices", type=int, default=-1,
                    help="N=1: gnnagg_set_locality_slices (-1 = library default: automatic; 1 = off; 2..16 forced)")
    ap.add_argument("--c5", type=int, default=-1, help="1/0: also measure the RMAT-26 strong-scaling config (default: only "
                                                        "with the default workload)")
    ap.add_argument("--c5-sweep", default="", help="comma-separated remote-stage counts for the c5 block")
    ap.add_argument("--ref-kernels", type=int, default=1, help="N=1: time the reference's own kernels (oracle/_ref) after the headline")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the headline output of the last timed step as DIR/H.npy (float32; a fixed row sample when "
                         "it exceeds %d MiB; one file per rank, H_rank<r>.npy, at N > 1)" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's output: not with --impl reference")
    args.warmup = max(args.warmup, 3)

    import numpy as np
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        args.gpus = world
    shape, fin, fout = WORKLOADS[args.workload]
    do_c5 = (args.workload == "reddit_gcn_layer_128" and not args.scheduled and args.sources == "rmat") if args.c5 < 0 else bool(args.c5)

    from gnnagg import synth

    strong = shape in RMAT_SCALES

    # ------------------------------------------------------------------ reference arm (CPU port)
    if args.impl == "reference":
        if rank != 0:
            return 0
        import oracle as orc

        orc.use_all_cores()  # rank 0 alone runs this arm: every host core, also under torchrun (OMP_NUM_THREADS=1 there)
        if strong:
            n_tot, m_tot = RMAT_SCALES[shape]
            n, m = n_tot // args.gpus, m_tot // args.gpus
        else:
            n, m = synth.shape_of(shape)
        config = {"workload": "%s (rank 0's block of the same synthetic graph)" % args.workload, "partition":
                  "1d-row-by-destination" if args.gpus > 1 else "single-gpu", "scheduled": bool(args.scheduled), "sources": args.sources}
        dev = torch.device("cuda:%d" % local_rank) if torch.cuda.is_available() else torch.device("cpu")
        # the same graph; a leading row block is what gets timed, so only that block is built when no GPU is around
        gen_rows, gen_edges = (n, m) if dev.type == "cuda" else (n, min(m, 4_000_000))
        src_total = n * args.gpus
        ptr, idx = synth.rmat_csr(gen_rows, gen_edges, seed=123, device=dev, src_num_v=src_total if args.gpus > 1 else None,
                                  dst_prefix=0 if args.gpus > 1 else None)
        val = synth.gcn_norm_val(ptr, idx) if src_total == n else torch.rand(idx.numel(), device=dev) + 0.5
        g = torch.Generator(device=dev).manual_seed(123)
        X = torch.randn((src_total, fin), device=dev, generator=g)
        W = torch.randn((fin, fout or fin), device=dev, generator=g) / fin ** 0.5
        per_step = []
        info = None
        for it in range(args.warmup + args.steps):
            budget = max(1.0, min(args.cpu_seconds, 120.0 / (args.warmup + args.steps)))
            gbs, t, rows, e = cpu_sample(orc, ptr, idx, val, X, W, fin, fout, budget) if it == 0 else info
            if it == 0:
                info = (gbs, t, rows, e)
                hp = ptr[: rows + 1].cpu().numpy()
                hi, hv = idx[:e].cpu().numpy(), val[:e].cpu().numpy()
                hX, hW = X.cpu().numpy(), W.cpu().numpy()
            t = cpu_port_time(orc, hp, hi, hv, hX, hW, rows, fin, fout)
            if it >= args.warmup:
                per_step.append(t)
        t_mean = float(np.mean(per_step))
        gbs = layer_bytes(rows, e, fin, fout) / t_mean / 1e9
        sample = "rows [0,%d) of the workload graph = %d edges (%.2f%% of m), scalar fp32 CSR port + fp32 GEMM, OpenMP" % (
            rows, e, 100.0 * e / m)
        line = {"impl": "reference", "metric": "gcn_aggregation_algorithmic_GBps" if fout is None else "gcn_layer_algorithmic_GBps",
                "value": round(gbs, 3), "unit": "GB/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t_mean * 1e3, 3),
                "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "config": config,
                "cpu_baseline": {"value": round(gbs, 3), "unit": "GB/s", "cores": orc.num_threads(), "kind": "port",
                                 "sample": sample},
                "e2e": {"value": round(gbs, 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "the reference has no CPU implementation of the float path (SURVEY 8(c)); this is the CPU port "
                        "in oracle/oracle.c; each step processes the bounded sample, GB/s is per sample bytes"}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ our arm
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback); use --impl reference for the CPU port"
    import gnnagg  # noqa: F401  (fails loudly when libgnnagg.so is missing)

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda:%d" % local_rank)
    dist = None
    if args.gpus > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    N = args.gpus
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
    sampler = ClockSampler(local_rank)
    sampler.start()
    timed, barrier = make_timer(dev, dist, sampler, flush)

    wl = Workload(args, args.workload, N, rank, dev, dist)
    n, m = wl.n, wl.m
    agg_only = wl.agg_only

    # optional: remote-stage sweep on the headline workload (builder's tuning runs; one JSON line per setting)
    if args.sweep and N > 1 and wl.ph is not None:
        for st in [int(s) for s in args.sweep.split(",")]:
            w2 = wl if st == wl.stages else Workload(args, args.workload, N, rank, dev, dist, stages=st)
            if w2.ph is None:
                continue
            r = measure(w2, timed, max(5, args.steps // 2), 3, e2e=False)
            if rank == 0:
                print(json.dumps({"sweep": {"workload": args.workload, "n_gpus": N, "remote_stages": st, "ms_per_step": round(r["ms"], 4),
                                            "compute_only_ms": round(r["compute_ms"], 4), "exchange_ms": round(r["exchange_ms"], 4),
                                            "nvlink_GBps_per_rank": round(w2.ph.num_send * fin * 4 / (r["exchange_ms"] * 1e-3) / 1e9, 1),
                                            "stage_edges": w2.ph.stage_edges}}), flush=True)
            if w2 is not wl:
                w2.close()
                del w2
                torch.cuda.empty_cache()

    r = measure(wl, timed, args.steps, args.warmup, e2e=True, dump_bytes=DUMP_BYTES // N if args.dump_outputs else 0)
    clocks = sampler.result()
    dumped = None
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)
        name = "H" if N == 1 else "H_rank%d" % rank
        H, how = r["output"]
        np.save(os.path.join(args.dump_outputs, name + ".npy"), H)
        # printed by rank 0: every rank's file is listed, the details are those of rank 0's (the others have the same
        # dtype and width, and their rows are sampled the same way from their own row blocks)
        dumped = {"dir": args.dump_outputs, "files": ["H.npy"] if N == 1 else ["H_rank%d.npy" % q for q in range(N)],
                  name: {"dtype": str(H.dtype), "shape": list(H.shape), "rows": how}}
    timed, barrier = make_timer(dev, dist, None, flush)  # the clock sampler covers the headline region only
    ms, ms_e2e = r["ms"], r["ms_e2e"]
    parity = parity_check(wl) if N > 1 else None

    bytes_rank = layer_bytes(n, m, fin, fout)
    value = N * bytes_rank / (ms * 1e-3) / 1e9
    e2e_value = N * bytes_rank / (ms_e2e * 1e-3) / 1e9

    line = None
    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)" if "hbm_gbs" in peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        prof = r["prof"]
        lpr, nv = (8, 1) if fin <= 32 else (16, 1) if fin <= 64 else (32, 1) if fin <= 128 else (32, 2)
        if N == 1:
            agg_ms, total_ms, dense_ms = prof["agg"], prof["total"], prof["dense"]
            breakdown = {k: round(prof[k], 4) for k in ("agg", "agg_rest", "dense", "total")}
        else:
            total_ms = r["compute_ms"]
            dense_ms = prof.get("dense", 0.0)
            agg_ms = max(total_ms - dense_ms, 1e-6)  # all stages' aggregation kernels + their fix-ups
            breakdown = {"aggregation_all_stages": round(agg_ms, 4), "dense": round(dense_ms, 4), "compute_total": round(total_ms, 4),
                         "stage0_local_sources": round(prof.get("stage0", 0.0), 4)}
        achieved = spmm_bytes(n, m, fin) / (agg_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": "agg_kernel<%d,%d,GCN,%s,%d> (CSR SpMM aggregation)%s" % (
                        lpr, nv, "sched" if args.scheduled else "csr", 128 if m < 4000000 else 512,
                        "" if N == 1 else ", %d stage launches per step" % (wl.ph.num_stages if wl.ph is not None else 1)),
                    "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                    "traffic": None, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": spmm_bytes(n, m, fin), "kernel_ms": round(agg_ms, 4),
                    "step_breakdown_ms": breakdown,
                    "note": "gather model (SURVEY 8(d)): one F-float source row per edge, so L1/L2 hits count as bytes: `frac` is an "
                            "effective-bandwidth figure and exceeds 1 where X (%.0f MB) is cache resident; `frac_dram` is the HBM "
                            "fraction proper" % (4 * n * fin / 1e6)}
        if N == 1:
            try:  # counters of the dominant kernel from the committed `ncu --set full` capture of this very command
                summ = json.load(open(os.path.join(ROOT, "profiles", "ncu_summary.json")))
                key = args.workload + ("_sched" if args.scheduled else "") + ("_uniform" if args.sources == "uniform" else "")
                s = summ.get(key, {})
                if s.get("dram_bytes_per_launch"):
                    roofline["traffic"] = s["dram_bytes_per_launch"]
                    comp = compulsory_bytes(n, m, fin)
                    roofline["compulsory_bytes"] = comp
                    roofline["traffic_over_compulsory"] = round(s["dram_bytes_per_launch"] / comp, 3)
                    roofline["frac_dram"] = round(s["dram_bytes_per_launch"] / (agg_ms * 1e-3) / 1e9 / peak, 4)
                units = {k: s[k] for k in ("l1tex_throughput_pct", "lts_throughput_pct", "dram_throughput_pct") if s.get(k) is not None}
                if units:
                    top = max(units, key=units.get)
                    roofline["binding_unit"] = {"unit": top.split("_")[0], "pct_of_peak": units[top]}
                roofline["ncu"] = {k: s[k] for k in ("l1tex_throughput_pct", "lts_throughput_pct", "dram_GBps", "l2_hit_pct",
                                                     "l1_hit_pct", "duration_ms", "source") if k in s}
            except Exception:
                pass
        else:
            roofline["note"] += "; ncu counters are captured at N = 1 only and are not repeated here"

        import oracle as orc

        orc.use_all_cores()
        # the CPU port on a leading block of rank 0's rows; at N > 1 the sample's sources are re-indexed onto their
        # own X rows, regenerated from the per-rank seeds (same generator, same device type)
        if N > 1:
            hp_full = wl.ptr.cpu()
            rows_c = int(torch.searchsorted(hp_full, min(int(hp_full[-1]), 40_000_000)).item())
            e_c = int(hp_full[rows_c])
            U = torch.unique(wl.idx[:e_c].long())
            idx_c = torch.searchsorted(U, wl.idx[:e_c].long()).to(torch.int32)
            Xc = torch.empty((U.numel(), fin), device=dev)
            for rr in range(N):
                sel = (U >= rr * n) & (U < (rr + 1) * n)
                if bool(sel.any()):
                    shard = torch.randn((n, fin), device=dev, generator=torch.Generator(device=dev).manual_seed(123 + rr))
                    Xc[sel] = shard[U[sel] - rr * n]
                    del shard
            gbs, t_cpu, rows, e = cpu_sample(orc, wl.ptr[: rows_c + 1].contiguous(), idx_c, wl.val[:e_c], Xc, wl.W, fin, fout,
                                             args.cpu_seconds)
        else:
            gbs, t_cpu, rows, e = cpu_sample(orc, wl.ptr, wl.idx, wl.val, wl.Xs, wl.W, fin, fout, args.cpu_seconds)
        cpu_baseline = {"value": round(gbs, 3), "unit": "GB/s", "cores": orc.num_threads(), "kind": "port",
                        "sample": "rows [0,%d) = %d edges (%.2f%% of m) of rank 0's graph, %.1f s; scalar fp32 CSR port + fp32 GEMM "
                                  "(oracle/oracle.c, OpenMP dynamic,64)" % (rows, e, 100.0 * e / m, t_cpu)}

        line = {"metric": "gcn_aggregation_algorithmic_GBps" if agg_only else "gcn_layer_algorithmic_GBps", "value": round(value, 1),
                "unit": "GB/s", "n_gpus": N,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 4), "higher_is_better": True,
                "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": wl.config,
                "edges_feat_per_s": round(N * m * fin / (ms * 1e-3), 1),
                "clocks": clocks,
                "e2e": {"value": round(e2e_value, 1), "unit": "GB/s", "ms_per_step": round(ms_e2e, 4),
                        # whole job: every rank copies its X shard (and W) in and its H shard out
                        "h2d_bytes_per_step": N * (4 * n * fin + (4 * fin * fout if not agg_only else 0)),
                        "d2h_bytes_per_step": N * 4 * n * (fout or fin),
                        "api": ("gnnagg_gcn_run_host (pinned host X -> Y)" if agg_only else "gnnagg_gcn_layer_host (pinned host X, W -> H)") if N == 1 else
                               "gnnagg_dist_gcn_layer_host: pinned H2D of the X shard into the peer-visible buffer + the step (halo pushes + "
                               "staged aggregation + combination) with the copy back of the H shard overlapping the last stage"},
                "gpu_launches": int(round(r["launches_per_step"] * args.steps)),
                "compute_only": {"ms_per_step": round(total_ms, 4),
                                 "value": round(N * bytes_rank / (total_ms * 1e-3) / 1e9, 1), "unit": "GB/s",
                                 "note": "kernels only (X already resident, no halo exchange)" + (
                                     ", the library's own CUDA events" if N == 1 else ", timed like the step with the exchange switched off, max over ranks")},
                "roofline": roofline, "cpu_baseline": cpu_baseline,
                "setup_s": round(wl.setup_s, 2)}
        if dumped is not None:
            line["outputs_dumped"] = dumped
        if N > 1:
            line["e2e"]["copies_only_ms"] = round(r["ms_copies"], 4)
            line["e2e"]["note"] = "copies_only_ms = the H2D + D2H of the same buffers alone, all ranks at once: what the host side of this box allows at this N"
            hal = {"kind": wl.halo, "exposed_ms": round(ms - r["compute_ms"], 4)}
            if wl.ph is not None:
                ex_bytes = wl.ph.num_send * fin * 4
                hal.update({"remote_stages": wl.stages if wl.stages < 0 else wl.ph.num_stages - 1, "stage_edges": wl.ph.stage_edges,
                            "bytes_per_rank": ex_bytes, "exchange_ms": round(r["exchange_ms"], 4),
                            "nvlink_GBps_per_rank": round(ex_bytes / (r["exchange_ms"] * 1e-3) / 1e9, 1),
                            "nvlink_frac_of_770": round(ex_bytes / (r["exchange_ms"] * 1e-3) / 1e9 / NVLINK_PEAK_GBS, 3),
                            "note": "bytes_per_rank = what rank 0 pushes per step; exchange_ms = its first push issued .. last push "
                                    "complete on the comm stream (max over ranks), running concurrently with the aggregation; "
                                    "exposed_ms = step - kernels-only step"})
            line["halo"] = hal
            line["parity"] = parity

    # ---- the kernel to beat: the reference's own kernels recompiled for sm_100 (oracle/_ref), after the headline
    if rank == 0 and N == 1 and args.ref_kernels and not args.scheduled:
        try:
            line["ref_kernels_sm100"] = ref_kernels(wl, flush)
        except Exception as e:
            line["ref_kernels_sm100"] = {"unavailable": "%s: %s" % (type(e).__name__, e)}

    wl.close()
    del wl
    torch.cuda.empty_cache()

    if do_c5:
        try:
            c5 = c5_block(args, N, rank, dev, dist, timed, 5, 3)
        except Exception as e:  # never lose the headline line to the extra block
            c5 = {"error": "%s: %s" % (type(e).__name__, e)}
        if rank == 0:
            line["c5"] = c5
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()
    return 0


def ref_kernels(wl, flush):
    """ours vs the reference's aggr_gcn (un-scheduled) and aggr_gcn_target (NG 32) on the headline graph, same inputs.
    oracle/_ref/libref.so = the reference's sources compiled for sm_100 by oracle/Makefile; used as the measured
    'kernel to beat' beside the headline, never on the product path."""
    import ctypes as C

    import numpy as np
    import torch

    import oracle as orc

    if not orc.ref_available():
        return {"unavailable": "oracle/_ref/libref.so not built (needs /root/reference at build time)"}
    ref = orc.ref()
    n, m, F = wl.n, wl.m, wl.fin
    P = lambda t: C.c_void_p(t.data_ptr())
    Y, Yr = torch.empty((n, F), device=wl.dev), torch.zeros((n, F), device=wl.dev)

    def timeit(fn, reps):
        fn()
        torch.cuda.synchronize()
        ts = []
        for _ in range(reps):
            flush.fill_(1)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        return float(np.median(ts))

    ref.ref_set_globals(n, m)
    h = C.c_void_p(ref.ref_gcn_create(P(wl.ptr), P(wl.idx), P(wl.val), n, m, F, F))
    out = {"graph": wl.name, "F": F}
    out["ours_gcn_ms"] = round(timeit(lambda: wl.agg.gcn_run(wl.Xs, Y), 5), 4)
    out["ref_aggr_gcn_ms"] = round(timeit(lambda: ref.ref_gcn_run(h, P(wl.Xs), P(Yr), max(128, F), 0, F), 3), 4)
    wl.agg.schedule(1, [32])
    ref.ref_gcn_schedule(h, 1, 32, 0)
    out["ours_gcn_ng32_ms"] = round(timeit(lambda: wl.agg.gcn_run(wl.Xs, Y, scheduled=True), 5), 4)
    out["ref_aggr_gcn_target_ng32_ms"] = round(timeit(lambda: ref.ref_gcn_run(h, P(wl.Xs), P(Yr), max(128, F), 1, F), 3), 4)
    out["speedup_vs_aggr_gcn"] = round(out["ref_aggr_gcn_ms"] / out["ours_gcn_ms"], 2)
    out["speedup_vs_aggr_gcn_target"] = round(out["ref_aggr_gcn_target_ng32_ms"] / min(out["ours_gcn_ms"], out["ours_gcn_ng32_ms"]), 2)
    diff = (Y - Yr).abs().max().item() / max(1e-30, Yr.abs().max().item())
    out["max_abs_diff_over_max_abs"] = float("%.3g" % diff)
    out["source"] = "include/aggr_gcn.h:5-36 (aggr_gcn), :78-114 (aggr_gcn_target) compiled from /root/reference for sm_100 (-O2 --use_fast_math)"
    return out


if __name__ == "__main__":
    sys.exit(main())
