"""GPU tier: the peer-memory multi-GPU step with the X shards stored in bf16 (gnnagg_dist_gcn_run_bf16 / _gcn_layer_bf16 /
_gcn_layer_host_bf16) and the bf16 stage entry points it is built on (gnnagg_gcn_run_acc_bf16 / _rows_bf16).

The bf16 step widens every gathered value exactly to fp32 and runs the fp32 step's plan, kernels and summation order, so
its result must EQUAL the fp32 step run on the widened X, bit for bit, and lie within the project's 1e-5 * sum|terms|
gate of the fp64 oracle of the widened X.  As in test_gpu_dist.py, all ranks live on device 0 on a one-GPU box (the flag
protocol, the push kernels and the staged accumulation run exactly as across GPUs); the torchrun test at the end needs
>= 2 GPUs."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT
from gnnagg import partition, synth
from gpu_util import make_graph

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


def _bf16_x(rng, n, F):
    """N(0,1) features rounded once to bf16 (CPU tensor)"""
    return torch.from_numpy(rng.standard_normal((n, F)).astype(np.float32)).to(BF16)


def _connect(cuda, ptr, idx, val, bounds, stages, cap):
    world = len(bounds) - 1
    ld = partition.LocalDist(bounds, cap, devices=[0] * world)
    for r in range(world):
        lp, li, lv = partition.local_block(ptr, idx, val, bounds, r)
        ld.set_graph(r, *(torch.from_numpy(a).to(cuda) for a in (lp, li, lv)), stages)
    ld.connect()
    ld.streams = [torch.cuda.Stream(device=cuda) for _ in range(world)]
    return ld


def _step(ld, cuda, X, buf, W=None, exchange=True):
    """writes X (a CPU tensor, float32 or bfloat16) into shard buffer `buf` of every rank in X's dtype, runs one step of
    every rank on its own stream and returns the concatenated fp32 output"""
    b, F = ld.bounds, X.shape[1]
    for r in range(ld.world):
        ld.ranks[r].x(buf, F, X.dtype).copy_(X[b[r]:b[r + 1]].to(cuda))
    torch.cuda.synchronize()
    fo = F if W is None else W.shape[1]
    Y = [torch.full((b[r + 1] - b[r], fo), float("nan"), device=cuda) for r in range(ld.world)]
    for r in range(ld.world):
        with torch.cuda.stream(ld.streams[r]):
            if W is None:
                ld.ranks[r].gcn_run(Y[r], buf, F, exchange=exchange, dtype=X.dtype)
            else:
                ld.ranks[r].gcn_layer(W, Y[r], buf, exchange=exchange, dtype=X.dtype)
    torch.cuda.synchronize()
    for r in range(ld.world):
        ld.ranks[r].check()
    return torch.cat(Y).cpu().numpy()


def _gate(got, want, scale):
    err = np.abs(got.astype(np.float64) - want)
    bound = 1e-5 * scale + 1e-30
    assert np.all(err <= bound), float((err / bound).max())


@pytest.mark.parametrize("world,stages", [(1, 1), (2, 0), (2, 1), (3, 1), (3, 2), (4, 0), (4, 3), (2, -4), (3, -16), (4, -3)])
@pytest.mark.parametrize("F", [32, 64, 128, 100])
def test_bf16_step_equals_fp32_step_on_widened_x(gn, orc, cuda, world, stages, F):
    """owner stages, one pass, row pipelining (stages < 0) and, at F = 100, the 8-byte push of bf16 rows; two steps through
    both shard buffers, each bf16 step after the fp32 step of the same epoch pair on the same handles"""
    rng = np.random.default_rng(world * 100 + stages * 10 + F + 7)
    sizes = rng.integers(300, 900, world)
    bounds = [0] + [int(s) for s in np.cumsum(sizes)]
    n = bounds[-1]
    ptr, idx = synth.small_random_csr(n, 20.0, 5 + world, hub=9000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    Xb = _bf16_x(rng, n, F)
    want, scale = orc.spmm_f64(ptr, idx, val, Xb.float().numpy())
    ld = _connect(cuda, ptr, idx, val, bounds, stages, F)
    try:
        for step in range(2):
            Xs = Xb * (1.0 + step)  # exact in bf16
            y32 = _step(ld, cuda, Xs.float(), step & 1)
            yb = _step(ld, cuda, Xs, step & 1)
            assert np.array_equal(yb, y32), (step, float(np.abs(yb - y32).max()))
            _gate(yb, want * (1.0 + step), scale * (1.0 + step))
    finally:
        ld.close()


def test_bf16_layer_with_an_empty_rank(gn, orc, cuda):
    rng = np.random.default_rng(3)
    bounds = [0, 700, 700, 1900, 2500]          # rank 1 owns nothing
    n, F = bounds[-1], 64
    ptr, idx = synth.small_random_csr(n, 30.0, 9, hub=20000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    Xb = _bf16_x(rng, n, F)
    W = (rng.standard_normal((F, 32)) / 8).astype(np.float32)
    _, h64, hs = orc.gcn_layer_f64(ptr, idx, val, Xb.float().numpy(), W)
    ld = _connect(cuda, ptr, idx, val, bounds, 2, F)
    try:
        dW = torch.from_numpy(W).to(cuda)
        h32 = _step(ld, cuda, Xb.float(), 0, W=dW)
        hb = _step(ld, cuda, Xb, 1, W=dW)
    finally:
        ld.close()
    assert np.array_equal(hb, h32)
    _gate(hb, h64, hs)


def test_bf16_narrower_width_wide_rows_and_dtype_switches(gn, orc, cuda):
    """feat < feat_cap and F = 256 on one set of handles (every rank prepared for a new width first), then fp32 -> bf16 ->
    fp32 steps on the same handles: the epochs continue across dtypes and both stay correct"""
    rng = np.random.default_rng(41)
    bounds = [0, 500, 1300, 2000]
    n, cap = bounds[-1], 256
    ptr, idx = synth.small_random_csr(n, 15.0, 17, hub=7000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    ld = _connect(cuda, ptr, idx, val, bounds, 2, cap)
    try:
        for F in (256, 64):
            for r in range(3):
                gn.check(gn.lib().gnnagg_dist_prepare(ld.ranks[r].h, F, None))
            Xb = _bf16_x(rng, n, F)
            want, scale = orc.spmm_f64(ptr, idx, val, Xb.float().numpy())
            got = {}
            for k, X in enumerate((Xb.float(), Xb, Xb.float(), Xb)):
                got[k] = _step(ld, cuda, X, k & 1)
                _gate(got[k], want, scale)
            assert np.array_equal(got[0], got[1]) and np.array_equal(got[1], got[2]) and np.array_equal(got[2], got[3])
    finally:
        ld.close()


def test_first_step_after_connect_is_bf16(gn, orc, cuda):
    """fresh handles, three ranks driven by one process, the first step a bf16 one at F = 100: its push instance (8-byte
    units) must have been loaded when the rank was created -- a lazy load in the middle of the step would wait for the
    device while a peer's kernel spins on this rank's flag"""
    rng = np.random.default_rng(5)
    bounds = [0, 400, 1100, 1600]
    n, F = bounds[-1], 100
    ptr, idx = synth.small_random_csr(n, 12.0, 31, hub=5000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    Xb = _bf16_x(rng, n, F)
    want, scale = orc.spmm_f64(ptr, idx, val, Xb.float().numpy())
    ld = _connect(cuda, ptr, idx, val, bounds, -3, F)
    try:
        got = _step(ld, cuda, Xb, 0)          # checks every rank's error word
    finally:
        ld.close()
    _gate(got, want, scale)


@pytest.mark.parametrize("layer", [False, True])
def test_bf16_host_buffer_entry_point_single_rank(gn, orc, cuda, layer):
    """gnnagg_dist_gcn_layer_host_bf16: half-size H2D copy of a pinned bf16 shard, row-chunked last stage, copy back"""
    rng = np.random.default_rng(11)
    n, F = 9000, 64
    ptr, idx = synth.small_random_csr(n, 25.0, 21, hub=30000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    Xb = _bf16_x(rng, n, F)
    W = (rng.standard_normal((F, 96)) / 8).astype(np.float32)
    ld = partition.LocalDist([0, n], F, devices=[0])
    try:
        ph = ld.set_graph(0, *(torch.from_numpy(a).to(cuda) for a in (ptr, idx, val)), 0)
        ld.connect()
        hW = torch.from_numpy(W).pin_memory() if layer else None
        fo = 96 if layer else F
        hb, h32 = torch.empty((n, fo)).pin_memory(), torch.empty((n, fo)).pin_memory()
        ph.gcn_layer_host(Xb.pin_memory(), hW, hb)
        ph.gcn_layer_host(Xb.float().pin_memory(), hW, h32)
        ph.check()
    finally:
        ld.close()
    if layer:
        _, want, scale = orc.gcn_layer_f64(ptr, idx, val, Xb.float().numpy(), W)
    else:
        want, scale = orc.spmm_f64(ptr, idx, val, Xb.float().numpy())
    assert np.array_equal(hb.numpy(), h32.numpy())
    _gate(hb.numpy(), want, scale)


def test_bf16_launches_and_profile_match_fp32(gn, cuda):
    rng = np.random.default_rng(13)
    bounds = [0, 600, 1500, 2100]
    n, F = bounds[-1], 64
    ptr, idx = synth.small_random_csr(n, 18.0, 3, hub=6000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    Xb = _bf16_x(rng, n, F)
    ld = _connect(cuda, ptr, idx, val, bounds, 2, F)
    try:
        for r in ld.ranks:
            r.profile(True)
        counts, profs = {}, {}
        for X in (Xb.float(), Xb, Xb.float(), Xb):   # the second pair: steady state
            l0 = [r.launches for r in ld.ranks]
            _step(ld, cuda, X, 0)
            counts[X.dtype] = [r.launches - a for r, a in zip(ld.ranks, l0)]
            profs[X.dtype] = [r.profile_read() for r in ld.ranks]
    finally:
        ld.close()
    assert counts[BF16] == counts[torch.float32]
    for p in profs[BF16] + profs[torch.float32]:
        assert all(np.isfinite(v) and v >= 0.0 for v in p.values()), p
        assert p["step"] >= p["stage0"] and p["step"] > 0.0, p


def test_bf16_argument_errors_are_reported_not_crashed(gn, cuda):
    L = gn.lib()
    bounds = (C.c_int64 * 3)(0, 8, 16)
    h = C.c_void_p()
    assert L.gnnagg_dist_create_rank(0, 2, bounds, 32, C.byref(h)) == 0
    Y = torch.empty((8, 32), device=cuda)
    assert L.gnnagg_dist_gcn_run_bf16(h, 0, C.c_void_p(Y.data_ptr()), 32, 0, None) == -4          # no graph
    ptr = torch.zeros(9, dtype=torch.int32, device=cuda)
    assert L.gnnagg_dist_set_graph(h, C.c_void_p(ptr.data_ptr()), None, None, 0, 1, None) == 0
    assert L.gnnagg_dist_gcn_run_bf16(h, 0, C.c_void_p(Y.data_ptr()), 32, 0, None) == -4          # peers not connected
    assert b"connect" in L.gnnagg_last_error()
    assert L.gnnagg_dist_destroy(h) == 0

    rng = np.random.default_rng(1)
    n = 64
    hp, hi = synth.small_random_csr(n, 4.0, 2)
    hv = rng.standard_normal(len(hi)).astype(np.float32)
    ld = partition.LocalDist([0, n], 32, devices=[0])
    try:
        ph = ld.set_graph(0, *(torch.from_numpy(a).to(cuda) for a in (hp, hi, hv)), 0)
        ld.connect()
        Yd = torch.empty((n, 48), device=cuda)
        for feat in (30, 48):                                                                      # not a multiple of 4 / > feat_cap
            assert L.gnnagg_dist_gcn_run_bf16(ph.h, 0, C.c_void_p(Yd.data_ptr()), feat, 0, None) == -1
        W = torch.zeros((32, 32), device=cuda)
        assert L.gnnagg_dist_gcn_layer_bf16(ph.h, 0, C.c_void_p(W.data_ptr()), C.c_void_p(Yd.data_ptr()), 36, 32, 0, None) == -1
        assert L.gnnagg_dist_gcn_layer_bf16(ph.h, 0, None, C.c_void_p(Yd.data_ptr()), 32, 32, 0, None) == -1   # NULL W
        hout = torch.empty((n, 32))
        assert L.gnnagg_dist_gcn_layer_host_bf16(ph.h, 0, None, None, C.c_void_p(hout.data_ptr()), 32, 32, None) == -1  # NULL h_X
        with pytest.raises(gn.GnnaggError):
            ph.gcn_run(torch.empty((n, 32), device=cuda), 0, 34, dtype=BF16)
        with pytest.raises(ValueError):
            ph.x(0, 32, torch.float16)
        with pytest.raises(gn.GnnaggError):                   # a host bf16 shard must be a CPU tensor
            ph.gcn_layer_host(torch.zeros((n, 32), dtype=BF16, device=cuda), None, hout)
        ph.check()
    finally:
        ld.close()


def test_shard_views_share_the_buffer(gn, cuda):
    """x(buf, F, bfloat16) is a view of the same peer-visible memory as the fp32 view: the bf16 rows take the first half"""
    n, F = 50, 32
    hp, hi = synth.small_random_csr(n, 3.0, 4)
    hv = np.ones(len(hi), np.float32)
    ld = partition.LocalDist([0, n], F, devices=[0])
    try:
        ph = ld.set_graph(0, *(torch.from_numpy(a).to(cuda) for a in (hp, hi, hv)), 0)
        xb, xf = ph.x(0, F, BF16), ph.x(0, F)
        assert xb.dtype == BF16 and xb.shape == (n, F) and xb.data_ptr() == xf.data_ptr()
        xf.zero_()
        xb.fill_(1.5)
        torch.cuda.synchronize()
        raw = xf.view(torch.int32).flatten().cpu()
        half = n * F // 2
        assert bool((raw[:half] == 0x3FC03FC0).all()) and bool((raw[half:] == 0).all())
    finally:
        ld.close()


def test_two_bf16_layers_through_the_two_shard_buffers(gn, cuda):
    """a two-layer bf16 model across ranks: layer 1 reads bf16 buffer 0 and writes H1 in fp32, one torch copy rounds H1
    into bf16 buffer 1, layer 2 reads it.  Each layer equals the fp32 layer on its widened input."""
    rng = np.random.default_rng(23)
    bounds = [0, 900, 2100, 3000]
    n, F = bounds[-1], 64
    ptr, idx = synth.small_random_csr(n, 18.0, 29, hub=8000)
    val = ((rng.random(len(idx)) + 0.1) / 20).astype(np.float32)
    Xb = _bf16_x(rng, n, F)
    W1 = torch.from_numpy((rng.standard_normal((F, F)) / 8).astype(np.float32)).to(cuda)
    W2 = torch.from_numpy((rng.standard_normal((F, F)) / 8).astype(np.float32)).to(cuda)
    ld = _connect(cuda, ptr, idx, val, bounds, 2, F)
    b = bounds
    try:
        for r in range(3):
            ld.ranks[r].x(0, F, BF16).copy_(Xb[b[r]:b[r + 1]].to(cuda))
        torch.cuda.synchronize()
        H1 = [torch.zeros((b[r + 1] - b[r], F), device=cuda) for r in range(3)]
        H2 = [torch.empty((b[r + 1] - b[r], F), device=cuda) for r in range(3)]
        # the conversion kernel runs between two steps of ranks driven by one process, so it must be loaded before the
        # first step: a first (lazy) load waits for the device, where rank 0's step already spins on its peers' flags
        for r in range(3):
            ld.ranks[r].x(1, F, BF16).copy_(H1[r])
        torch.cuda.synchronize()
        for r in range(3):
            with torch.cuda.stream(ld.streams[r]):
                ld.ranks[r].gcn_layer(W1, H1[r], buf=0, dtype=BF16)
                ld.ranks[r].x(1, F, BF16).copy_(H1[r])                  # the one conversion between the layers
                ld.ranks[r].gcn_layer(W2, H2[r], buf=1, dtype=BF16)
        torch.cuda.synchronize()
        for r in range(3):
            ld.ranks[r].check()
        h1 = torch.cat(H1).cpu()
        h2 = torch.cat(H2).cpu().numpy()
        ref1 = _step(ld, cuda, Xb.float(), 0, W=W1)
        ref2 = _step(ld, cuda, h1.to(BF16).float(), 1, W=W2)
    finally:
        ld.close()
    assert np.array_equal(h1.numpy(), ref1)
    assert np.array_equal(h2, ref2)


@pytest.mark.parametrize("name", ["medium", "hub", "short_rows"])
def test_aggregator_acc_and_rows_take_bf16(gn, cuda, name):
    """Aggregator.gcn_run_acc / gcn_run_rows dispatch on X's dtype: bf16 X equals fp32 on the widened X, bit for bit"""
    import gnnagg

    ptr, idx = make_graph(name, 3)
    n, F = len(ptr) - 1, 36
    rng = np.random.default_rng(9)
    val = torch.from_numpy(rng.standard_normal(len(idx)).astype(np.float32)).to(cuda)
    agg = gnnagg.Aggregator(torch.from_numpy(ptr).to(cuda), torch.from_numpy(idx).to(cuda), val)
    Xb = _bf16_x(rng, n, F).to(cuda)
    X2 = _bf16_x(rng, n, F).to(cuda)
    out = {}
    for dt in (BF16, torch.float32):
        a, b = Xb.to(dt), X2.to(dt)
        Y = torch.full((n, F), float("nan"), device=cuda)
        agg.gcn_run_acc(a, Y, accumulate=False)
        agg.gcn_run_acc(b, Y, accumulate=True)
        R = torch.full((n, F), float("nan"), device=cuda)
        cuts = [0, n // 3, n // 3, (2 * n) // 3, n]
        for lo, hi in zip(cuts[:-1], cuts[1:]):
            agg.gcn_run_rows(a, R, lo, hi)
            agg.gcn_run_rows(b, R, lo, hi, accumulate=True)
        torch.cuda.synchronize()
        out[dt] = (Y.cpu().numpy(), R.cpu().numpy())
    assert np.array_equal(out[BF16][0], out[torch.float32][0])
    assert np.array_equal(out[BF16][1], out[torch.float32][1])
    assert not np.isnan(out[BF16][0]).any() and not np.isnan(out[BF16][1]).any()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_multi_process_bf16_equals_fp32(tmp_path):
    """one process per GPU (torchrun, cudaIpc peer mappings, NVLink): on a down-scaled R-MAT the bf16 step equals the fp32
    step on the widened X in the same job and lies within the gate of the fp64 oracle; the job's log goes to tmp_path"""
    nproc = min(8, torch.cuda.device_count())
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", "29633", os.path.join(ROOT, "tests", "multirank_bf16_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    (tmp_path / ("multirank_bf16_n%d.log" % nproc)).write_text(r.stdout + "\n--- stderr ---\n" + r.stderr[-4000:])
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert lines and all(l["ok"] for l in lines)
