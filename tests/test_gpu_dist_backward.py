"""GPU tier: the multi-GPU GCN backward (gnnagg_dist_enable_backward / gnnagg_dist_gcn_backward, csrc/dist.cu) and the
autograd op over it (partition.dist_gcn_aggregate).

On a one-GPU box every rank lives on device 0 (LocalDist, one stream per rank): the flag protocol, the G buffers, the
return tables and the pull kernel run exactly as across GPUs, but the numbers say nothing about NVLink rates.  With
>= 2 GPUs the torchrun test at the end runs one process per GPU (tests/multirank_bwd_worker.py)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT, rel_gate
from gnnagg import partition, plugin, synth

pytestmark = pytest.mark.gpu


def _blocks(ptr, idx, val, bounds, cuda):
    for r in range(len(bounds) - 1):
        lp, li, lv = partition.local_block(ptr, idx, val, bounds, r)
        yield r, torch.from_numpy(lp).to(cuda), torch.from_numpy(li).to(cuda), torch.from_numpy(lv).to(cuda)


def _shards(A, bounds, cuda):
    return [torch.from_numpy(np.ascontiguousarray(A[bounds[r]:bounds[r + 1]])).to(cuda) for r in range(len(bounds) - 1)]


def _run(cuda, ptr, idx, val, bounds, stages, X, dYs, feat_cap=None, prepare=False):
    """per step s: forward on buffer 0, backward with dYs[s], forward on buffer 1 (X * (1 + s)); every rank on its own
    stream.  Returns (dX per step, Y per forward, launches added by every rank's backward calls)"""
    world, F = len(bounds) - 1, X.shape[1]
    ld = partition.LocalDist(bounds, feat_cap or F, devices=[0] * world)
    streams = [torch.cuda.Stream(device=cuda) for _ in range(world)]
    dxs, ys, launches = [], [], []
    try:
        for r, lp, li, lv in _blocks(ptr, idx, val, bounds, cuda):
            ld.set_graph(r, lp, li, lv, stages, backward=True)
        ld.connect()
        ranks = ld.ranks
        if prepare:   # a width below feat_cap: every rank is readied before its first step (one process, several ranks)
            from gnnagg import check, lib

            for ph in ranks:
                check(lib().gnnagg_dist_prepare(ph.h, F, None))
        for s, dY in enumerate(dYs):
            dYd = _shards(dY, bounds, cuda)
            Xs = [_shards((X * (1.0 + s + b)).astype(np.float32), bounds, cuda) for b in range(2)]
            Y = [[torch.full((ph.rows, F), float("nan"), device=cuda) for ph in ranks] for _ in range(2)]
            dX = [torch.full((ph.rows, F), float("nan"), device=cuda) for ph in ranks]
            step_launches = []
            for r, ph in enumerate(ranks):
                with torch.cuda.stream(streams[r]):
                    ph.x(0, F).copy_(Xs[0][r])
                    ph.gcn_run(Y[0][r], 0, F)
                    before = ph.launches
                    ph.gcn_backward(dYd[r], dX[r])
                    step_launches.append(ph.launches - before)
                    ph.x(1, F).copy_(Xs[1][r])
                    ph.gcn_run(Y[1][r], 1, F)
            torch.cuda.synchronize()
            for ph in ranks:
                ph.check()
            dxs.append(torch.cat(dX).cpu().numpy())
            ys += [torch.cat(Y[b]).cpu().numpy() for b in range(2)]
            launches.append(step_launches)
    finally:
        ld.close()
    return dxs, ys, launches


def _inputs(world, stages, F, seed_extra=0):
    rng = np.random.default_rng(world * 100 + stages * 10 + F + 7 + seed_extra)
    sizes = rng.integers(300, 900, world)
    bounds = [0] + [int(b) for b in np.cumsum(sizes)]
    n = bounds[-1]
    ptr, idx = synth.small_random_csr(n, 20.0, 5 + world, hub=9000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    X = rng.standard_normal((n, F)).astype(np.float32)
    dYs = [rng.standard_normal((n, F)).astype(np.float32) for _ in range(2)]
    return bounds, ptr, idx, val, X, dYs


def _check_against_oracle(orc, ptr, idx, val, X, dYs, dxs, ys):
    n = len(ptr) - 1
    for s, dY in enumerate(dYs):
        want, scale = orc.spmm_t_f64(ptr, idx, val, dY, n)
        assert not np.isnan(dxs[s]).any(), s
        bad, worst = rel_gate(dxs[s], want, scale, 1e-5)
        assert bad == 0, (s, worst)
    y64, ys64 = orc.spmm_f64(ptr, idx, val, X)
    for k, Y in enumerate(ys):          # the forward steps around the backward are unchanged
        mult = 1.0 + k // 2 + k % 2
        bad, worst = rel_gate(Y, y64 * mult, ys64 * mult, 1e-5)
        assert bad == 0, (k, worst)


@pytest.mark.parametrize("world,stages", [(1, 1), (2, 0), (2, 1), (3, 1), (3, 2), (4, 0), (4, 3), (2, -4), (3, -16), (4, -3)])
@pytest.mark.parametrize("F", [32, 64, 128, 100])
def test_local_ranks_backward_match_oracle(gn, orc, cuda, world, stages, F):
    """two backward steps with different dY, interleaved with forward steps on both shard buffers (separate epochs,
    write-after-read protection of G); concatenated dX within 1e-5 * sum|terms| of the fp64 A^T dY; every rank's backward
    adds the same number of launches at every step, 5 of them the protocol's when world > 1"""
    bounds, ptr, idx, val, X, dYs = _inputs(world, stages, F)
    dxs, ys, launches = _run(cuda, ptr, idx, val, bounds, stages, X, dYs)
    _check_against_oracle(orc, ptr, idx, val, X, dYs, dxs, ys)
    assert launches[0] == launches[1]
    if world > 1:
        assert all(k >= 5 + 1 for k in launches[0])


@pytest.mark.parametrize("world,stages", [(4, 3), (3, -16), (2, 0)])
def test_backward_is_bit_reproducible(gn, cuda, world, stages):
    bounds, ptr, idx, val, X, dYs = _inputs(world, stages, 64, seed_extra=1)
    a = _run(cuda, ptr, idx, val, bounds, stages, X, dYs)[0]
    b = _run(cuda, ptr, idx, val, bounds, stages, X, dYs)[0]
    for s in range(2):
        assert not np.isnan(a[s]).any()
        assert np.array_equal(a[s], b[s])


def _edge_graph(kind, rng):
    if kind == "empty_and_local":
        # rank 1 owns nothing; rank 3 references only its own rows
        bounds = [0, 600, 600, 1500, 2300]
        n = bounds[-1]
        ptr, idx = synth.small_random_csr(n, 12.0, 31, hub=4000)
        e0, e1 = int(ptr[bounds[3]]), int(ptr[bounds[4]])
        idx[e0:e1] = bounds[3] + idx[e0:e1] % (bounds[4] - bounds[3])
    else:
        # source 10 (rank 0) is referenced by every other rank, from many rows
        bounds = [0, 500, 1100, 1800, 2400]
        n = bounds[-1]
        ptr, idx = synth.small_random_csr(n, 12.0, 37, hub=4000)
        first = ptr[:-1][np.diff(ptr) > 0]
        idx[first[first >= ptr[500]][::3]] = 10
    val = rng.standard_normal(len(idx)).astype(np.float32)
    return bounds, ptr, idx, val


@pytest.mark.parametrize("kind", ["empty_and_local", "hub"])
@pytest.mark.parametrize("stages", [1, 0, -4])
def test_edge_cases_at_a_narrower_width(gn, orc, cuda, kind, stages):
    """an empty rank, a rank without remote sources, a source wanted by every peer; F = 64 under feat_cap = 128,
    prepared with gnnagg_dist_prepare on every rank before the first step"""
    rng = np.random.default_rng(5)
    bounds, ptr, idx, val = _edge_graph(kind, rng)
    n, F = bounds[-1], 64
    X = rng.standard_normal((n, F)).astype(np.float32)
    dYs = [rng.standard_normal((n, F)).astype(np.float32) for _ in range(2)]
    dxs, ys, _ = _run(cuda, ptr, idx, val, bounds, stages, X, dYs, feat_cap=128, prepare=True)
    _check_against_oracle(orc, ptr, idx, val, X, dYs, dxs, ys)
    if kind == "hub":
        ld = partition.LocalDist(bounds, 128, devices=[0] * 4)
        try:
            for r, lp, li, lv in _blocks(ptr, idx, val, bounds, cuda):
                ld.set_graph(r, lp, li, lv, stages, backward=True)
            ld.connect()
            assert all(ld.ranks[q].recv_counts[0] > 0 for q in range(1, 4))
        finally:
            ld.close()


def test_adjoint_at_scale(gn, cuda):
    """sum_r <A_r X, dY_r> == <X, dX> on a 4 M-edge R-MAT graph split over 4 local ranks"""
    n, m, F, world = 200000, 4200000, 64, 4
    ptr, idx = synth.rmat_csr(n, m, seed=123, device=cuda)
    val = synth.gcn_norm_val(ptr, idx)
    g = torch.Generator(device=cuda).manual_seed(5)
    X = torch.rand((n, F), device=cuda, generator=g)
    dY = torch.rand((n, F), device=cuda, generator=g)
    hp = ptr.cpu().numpy()
    bounds = [int(b) for b in partition.split_rows(hp, world, "edges")]
    ld = partition.LocalDist(bounds, F, devices=[0] * world)
    streams = [torch.cuda.Stream(device=cuda) for _ in range(world)]
    try:
        for r in range(world):
            r0, r1 = bounds[r], bounds[r + 1]
            e0, e1 = int(hp[r0]), int(hp[r1])
            ld.set_graph(r, (ptr[r0:r1 + 1] - e0).contiguous(), idx[e0:e1].contiguous(), val[e0:e1].contiguous(), 1, backward=True)
        ld.connect()
        Y = [torch.empty((bounds[r + 1] - bounds[r], F), device=cuda) for r in range(world)]
        dX = [torch.empty_like(y) for y in Y]
        torch.cuda.synchronize()
        for r, ph in enumerate(ld.ranks):
            with torch.cuda.stream(streams[r]):
                ph.x(0, F).copy_(X[bounds[r]:bounds[r + 1]])
                ph.gcn_run(Y[r], 0, F)
                ph.gcn_backward(dY[bounds[r]:bounds[r + 1]].contiguous(), dX[r])
        torch.cuda.synchronize()
        for ph in ld.ranks:
            ph.check()
    finally:
        ld.close()
    lhs = float((torch.cat(Y).double() * dY.double()).sum())
    rhs = float((X.double() * torch.cat(dX).double()).sum())
    assert abs(lhs - rhs) <= 1e-6 * abs(lhs)


def _rel(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm())


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_autograd_two_layers_match_one_gpu(gn, cuda, dtype):
    """relu(agg(X) @ W1) then agg(H1) @ W2 through shard buffers 0 and 1, one stream per rank, loss summed over ranks:
    X.grad, W1.grad and W2.grad equal the same model on one GPU through plugin.gcn_aggregate within 1e-5 relative (X in
    fp32 or bf16, H1 in fp32; a bf16 X.grad within one bf16 step of the one-GPU value)"""
    rng = np.random.default_rng(17)
    bounds = [0, 900, 2100, 3000]
    n, F, world = bounds[-1], 64, 3
    ptr, idx = synth.small_random_csr(n, 18.0, 29, hub=8000)
    val = ((rng.random(len(idx)) + 0.1) / 20).astype(np.float32)
    X0 = torch.from_numpy(rng.standard_normal((n, F)).astype(np.float32)).to(cuda).to(dtype)
    W1_0 = torch.from_numpy((rng.standard_normal((F, F)) / 8).astype(np.float32)).to(cuda)
    W2_0 = torch.from_numpy((rng.standard_normal((F, F)) / 8).astype(np.float32)).to(cuda)
    R = torch.from_numpy(rng.standard_normal((n, F)).astype(np.float32)).to(cuda)

    # one GPU
    at = plugin.gcn_init(*(torch.from_numpy(a).to(cuda) for a in (ptr, idx, val)))
    try:
        Xs = X0.clone().requires_grad_(True)
        W1, W2 = W1_0.clone().requires_grad_(True), W2_0.clone().requires_grad_(True)
        H1 = torch.relu(plugin.gcn_aggregate(at, Xs) @ W1)
        loss = ((plugin.gcn_aggregate(at, H1) @ W2) * R).sum()
        loss.backward()
        ref = (Xs.grad.float(), W1.grad.clone(), W2.grad.clone())
    finally:
        plugin.destroy(at)

    # three ranks on this device
    ld = partition.LocalDist(bounds, F, devices=[0] * world)
    streams = [torch.cuda.Stream(device=cuda) for _ in range(world)]
    try:
        for r, lp, li, lv in _blocks(ptr, idx, val, bounds, cuda):
            ld.set_graph(r, lp, li, lv, 1, backward=True)
        ld.connect()
        torch.cuda.synchronize()
        W1, W2 = W1_0.clone().requires_grad_(True), W2_0.clone().requires_grad_(True)
        Xr = [X0[bounds[r]:bounds[r + 1]].clone().requires_grad_(True) for r in range(world)]
        H1 = [None] * world
        for r in range(world):   # layer 1 on every rank, then layer 2 on every rank
            with torch.cuda.stream(streams[r]):
                H1[r] = torch.relu(partition.dist_gcn_aggregate(ld.ranks[r], Xr[r], 0) @ W1)
        losses = []
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                out = partition.dist_gcn_aggregate(ld.ranks[r], H1[r], 1) @ W2
                losses.append((out * R[bounds[r]:bounds[r + 1]]).sum())
        torch.cuda.synchronize()
        sum(losses).backward()
        torch.cuda.synchronize()
        for ph in ld.ranks:
            ph.check()
        got = (torch.cat([x.grad.float() for x in Xr]), W1.grad, W2.grad)
    finally:
        ld.close()
    for name, g, w in zip(("X", "W1", "W2"), got, ref):
        assert not torch.isnan(g).any(), name
        if name == "X" and dtype == torch.bfloat16:
            # dX is rounded to bf16 once on either path, from fp32 sums grouped differently: a value next to a rounding
            # boundary lands one bf16 step apart, so almost every element is equal and the rest are close
            same, rel = float((g == w).double().mean()), _rel(g, w)
            assert same >= 0.99 and rel <= 1e-3, (same, rel)
        else:
            assert _rel(g, w) <= 1e-5, (name, _rel(g, w))


def test_errors_are_reported_before_any_launch(gn, cuda):
    L = gn.lib()
    bounds = [0, 40, 80]
    rng = np.random.default_rng(3)
    ptr, idx = synth.small_random_csr(80, 6.0, 3, hub=200)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    dY = torch.zeros((40, 32), device=cuda)
    dX = torch.zeros((40, 32), device=cuda)

    def bwd(h, a, b, feat):
        return L.gnnagg_dist_gcn_backward(h, None if a is None else C.c_void_p(a.data_ptr()),
                                          None if b is None else C.c_void_p(b.data_ptr()), feat, None)

    # backward not enabled
    ld = partition.LocalDist(bounds, 32, devices=[0, 0])
    try:
        blocks = list(_blocks(ptr, idx, val, bounds, cuda))
        for r, lp, li, lv in blocks:
            ld.set_graph(r, lp, li, lv, 1)
        ld.connect()
        h = ld.handles[0]
        before = L.gnnagg_dist_launch_count(h)
        assert bwd(h, dY, dX, 32) == -4
        assert b"enable" in L.gnnagg_last_error()
        assert L.gnnagg_dist_enable_backward(h) == -4           # after set_graph
        assert L.gnnagg_dist_launch_count(h) == before
    finally:
        ld.close()
    assert L.gnnagg_dist_enable_backward(None) == -1
    # enabled, not connected; then bad feat and NULLs once connected
    ld = partition.LocalDist(bounds, 32, devices=[0, 0])
    try:
        for r, lp, li, lv in blocks:
            ld.set_graph(r, lp, li, lv, 1, backward=True)
        h = ld.handles[0]
        assert bwd(h, dY, dX, 32) == -4
        assert b"connect" in L.gnnagg_last_error()
        ld.connect()
        before = L.gnnagg_dist_launch_count(h)
        for feat in (0, 6, 36, 64):
            assert bwd(h, dY, dX, feat) == -1, feat
        assert bwd(h, None, dX, 32) == -1
        assert bwd(h, dY, None, 32) == -1
        odd = torch.zeros(40 * 32 + 1, device=cuda)[1:].view(40, 32)
        assert bwd(h, odd, dX, 32) == -1                          # misaligned
        assert L.gnnagg_dist_launch_count(h) == before
        assert L.gnnagg_dist_gcn_backward(None, None, None, 32, None) == -1
    finally:
        ld.close()
    # no graph yet
    hs = (C.c_void_p * 2)()
    assert L.gnnagg_dist_create(2, (C.c_int * 2)(0, 0), partition._bounds_array(bounds), 32, hs) == 0
    try:
        assert L.gnnagg_dist_enable_backward(hs[0]) == 0
        assert bwd(hs[0], dY, dX, 32) == -4
    finally:
        for h in hs:
            L.gnnagg_dist_destroy(h)
    # a group whose ranks disagree on backward is refused at connect
    ld = partition.LocalDist(bounds, 32, devices=[0, 0])
    try:
        for r, lp, li, lv in blocks:
            ld.set_graph(r, lp, li, lv, 1, backward=(r == 0))
        assert L.gnnagg_dist_connect_local(ld._hs, 2) == -1
        assert b"enable_backward" in L.gnnagg_last_error()
    finally:
        ld.close()


def test_forward_only_group_allocates_as_before(gn, cuda):
    """without gnnagg_dist_enable_backward the peer-visible allocation, the blob and the forward launches are those of a
    group that never heard of the backward; with it, the allocation grows by exactly one X buffer"""
    rng = np.random.default_rng(9)
    bounds = [0, 700, 1500]
    ptr, idx = synth.small_random_csr(1500, 10.0, 11, hub=3000)
    val = rng.standard_normal(len(idx)).astype(np.float32)
    sizes, fwd = [], []
    for backward in (False, True):
        ld = partition.LocalDist(bounds, 64, devices=[0, 0])
        try:
            for r, lp, li, lv in _blocks(ptr, idx, val, bounds, cuda):
                ld.set_graph(r, lp, li, lv, 1, backward=backward)
            ld.connect()
            blob = C.create_string_buffer(256)
            gn.check(gn.lib().gnnagg_dist_export(ld.handles[0], blob))
            sizes.append(int.from_bytes(blob.raw[40:48], "little"))   # DistBlob.bytes
            x0 = gn.lib().gnnagg_dist_x(ld.handles[0], 0)
            x1 = gn.lib().gnnagg_dist_x(ld.handles[0], 1)
            xbuf = x1 - x0
            ph = ld.ranks[0]
            before = ph.launches
            streams = [torch.cuda.Stream(device=cuda) for _ in range(2)]
            Y = [torch.empty((ld.ranks[r].rows, 64), device=cuda) for r in range(2)]
            for r in range(2):
                with torch.cuda.stream(streams[r]):
                    ld.ranks[r].gcn_run(Y[r], 0, 64)
            torch.cuda.synchronize()
            fwd.append(ph.launches - before)
        finally:
            ld.close()
    assert sizes[1] == sizes[0] + xbuf
    assert fwd[0] == fwd[1]


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
def test_multi_process_backward(tmp_path):
    """one process per GPU (torchrun, cudaIpc peer mappings, NVLink): on a down-scaled R-MAT the backward matches the
    single-GPU gnnagg_gcn_backward within the gate, repeats bit for bit, and the autograd gradients of a two-layer model
    match one GPU; the job's log goes to tmp_path"""
    nproc = min(8, torch.cuda.device_count())
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(nproc), "--master-addr", "127.0.0.1",
           "--master-port", "29635", os.path.join(ROOT, "tests", "multirank_bwd_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    (tmp_path / ("multirank_bwd_n%d.log" % nproc)).write_text(r.stdout + "\n--- stderr ---\n" + r.stderr[-4000:])
    print(r.stdout[-3000:], r.stderr[-2000:])
    assert r.returncode == 0
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert lines and all(l["ok"] for l in lines)
