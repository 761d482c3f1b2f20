"""GPU tier: the merged view of duplicate edges (gnnagg_set_merge_duplicates).  Runs of adjacent equal sources inside
a row become one entry whose value is the run's fp64 sum rounded once; every un-scheduled, un-sliced GCN entry point
of one aggregator runs on it, and the results stay within the 1e-5 * sum|terms| gate of the fp64 oracle."""
import numpy as np
import pytest
import torch

from conftest import rel_gate
from gpu_util import dev, rand_inputs

pytestmark = pytest.mark.gpu
TOL = 1e-5
OFF, ON = 1, 2


def dup_csr(n=5000, seed=11):
    """rows sorted by source with heavy adjacent duplicates: Zipf sources (runs of thousands of edges in the hub row,
    longer than an item and a warp's edges), 20 % empty rows (the first and last row among them), a row that is one
    single run of 1500 edges, and equal sources on both sides of row boundaries -- rows 20 / 21 directly, rows 30 / 33
    with only empty rows between them -- which must stay separate entries"""
    rng = np.random.default_rng(seed)
    deg = rng.poisson(24, n).astype(np.int64)
    deg[rng.random(n) < 0.2] = 0
    deg[0] = deg[n - 1] = 0
    deg[7] = 6000   # hub
    deg[11] = 1500  # one run
    deg[[20, 21, 30, 33]] = 40
    deg[[31, 32]] = 0
    ptr = np.zeros(n + 1, np.int64)
    ptr[1:] = np.cumsum(deg)
    idx = ((rng.zipf(1.3, int(ptr[-1])) - 1) % n).astype(np.int32)
    idx[ptr[11]:ptr[12]] = 42
    for r in range(n):
        idx[ptr[r]:ptr[r + 1]].sort()
    for a, b in ((20, 21), (30, 33)):  # row b starts with row a's last source (and stays sorted)
        idx[ptr[b]:ptr[b + 1]] = np.maximum(idx[ptr[b]:ptr[b + 1]], idx[ptr[a + 1] - 1])
        idx[ptr[b]] = idx[ptr[a + 1] - 1]
    return ptr.astype(np.int32), idx


def merged_np(ptr, idx, val=None):
    """restatement of the device build: heads, merged row pointers, run sources, fp64 run sums rounded once (None
    without val)"""
    n, m = len(ptr) - 1, len(idx)
    row = np.repeat(np.arange(n), np.diff(ptr))
    head = np.ones(m, bool)
    head[1:] = (idx[1:] != idx[:-1]) | (row[1:] != row[:-1])
    pos = np.concatenate([np.cumsum(head) - head, [head.sum()]])
    start = np.flatnonzero(head)
    end = np.append(start[1:], m)
    if val is None:
        return pos[ptr].astype(np.int32), idx[start], None
    v64 = val.astype(np.float64)
    mval = np.empty(len(start), np.float32)
    for k, (s, e) in enumerate(zip(start.tolist(), end.tolist())):
        acc = 0.0
        for x in v64[s:e].tolist():
            acc += x
        mval[k] = np.float32(acc)
    return pos[ptr].astype(np.int32), idx[start], mval


@pytest.fixture(scope="module")
def graph():
    ptr, idx = dup_csr()
    assert len(idx) - len(np.unique(np.repeat(np.arange(len(ptr) - 1), np.diff(ptr)) * len(ptr) + idx)) > len(idx) // 4
    return ptr, idx


def test_merged_view_bit_exact(gn, cuda, graph):
    ptr, idx = graph
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, 32, seed=1)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.set_merge_duplicates(ON)
    agg.gcn_run(dev(X), torch.empty((n, 32), device=cuda))
    mp, mi, mv = agg.merged_arrays()
    ep, ei, ev = merged_np(ptr, idx, val)
    assert agg.merged_edges == len(ei) < m
    assert np.array_equal(mp, ep)
    assert np.array_equal(mi, ei)
    assert np.array_equal(mv.view(np.int32), ev.view(np.int32))


@pytest.mark.parametrize("F", [32, 64, 100, 128, 256])
@pytest.mark.parametrize("we", [128, 512])
def test_merged_parity(gn, orc, cuda, graph, F, we):
    ptr, idx = graph
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.set_warp_edges(we)
    y64, scale = orc.spmm_f64(ptr, idx, val, X)
    agg.set_merge_duplicates(ON)
    Y = agg.gcn_run(dev(X), torch.full((n, F), float("nan"), device=cuda))
    assert rel_gate(Y.cpu().numpy(), y64, scale, TOL)[0] == 0
    assert torch.equal(Y, agg.gcn_run(dev(X), torch.empty_like(Y)))  # run to run
    agg.set_merge_duplicates(OFF)
    Yoff = agg.gcn_run(dev(X), torch.empty_like(Y))
    assert agg.merged_edges == m
    assert rel_gate(Yoff.cpu().numpy(), y64, scale, TOL)[0] == 0
    assert rel_gate(Y.cpu().numpy(), Yoff.cpu().numpy().astype(np.float64), scale, 2 * TOL)[0] == 0  # on vs off


@pytest.mark.parametrize("F", [32, 128])
def test_merged_entry_points(gn, orc, cuda, graph, F):
    """gcn_run_acc, gcn_layer, gcn_run_rows and the row-chunk host pipeline all run on the merged view; the host
    pipeline is bit-identical to gcn_run"""
    ptr, idx = graph
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=5)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.set_merge_duplicates(ON)
    gn.check(gn.lib().gnnagg_prepare(agg.h, F, None))  # builds the view and its long-row records ahead of the runs
    y64, scale = orc.spmm_f64(ptr, idx, val, X)
    Xd = dev(X)
    Y = agg.gcn_run(Xd, torch.empty((n, F), device=cuda))
    assert rel_gate(Y.cpu().numpy(), y64, scale, TOL)[0] == 0
    # accumulate onto a base: Y + A X
    base = torch.randn((n, F), device=cuda)
    acc = agg.gcn_run_acc(Xd, base.clone())
    assert rel_gate(acc.cpu().numpy(), y64 + base.cpu().numpy().astype(np.float64), scale + np.abs(base.cpu().numpy()), TOL)[0] == 0
    assert torch.equal(agg.gcn_run_acc(Xd, torch.empty_like(Y), accumulate=False), Y)
    # row ranges, one of them inside the hub / single-run rows, together cover every row
    Yr = torch.full((n, F), float("nan"), device=cuda)
    for lo, hi in [(0, 7), (7, 8), (8, 12), (12, n // 2), (n // 2, n)]:
        agg.gcn_run_rows(Xd, Yr, lo, hi)
    assert rel_gate(Yr.cpu().numpy(), y64, scale, TOL)[0] == 0
    # layer
    W = (np.random.default_rng(4).standard_normal((F, 64)) / np.sqrt(F)).astype(np.float32)
    H = torch.empty((n, 64), device=cuda)
    AX = torch.empty((n, F), device=cuda)
    agg.gcn_layer(Xd, dev(W), H, AX)
    assert torch.equal(AX, Y)
    _, h64, hs = orc.gcn_layer_f64(ptr, idx, val, X, W)
    assert rel_gate(H.cpu().numpy(), h64, hs, TOL)[0] == 0
    # row-chunk host pipeline (n >= 4096, below 4M edges: no source slices)
    hX = torch.from_numpy(X).pin_memory()
    hY = torch.full((n, F), float("nan")).pin_memory()
    agg.gcn_run_host(hX, hY)
    assert np.array_equal(hY.numpy(), Y.cpu().numpy())


def test_merged_values_follow_set_val(gn, orc, cuda, graph):
    ptr, idx = graph
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, 64, seed=6)
    dval = dev(val)
    agg = gn.Aggregator(dev(ptr), dev(idx), dval)
    agg.set_merge_duplicates(ON)
    Xd = dev(X)
    Y = torch.empty((n, 64), device=cuda)
    agg.gcn_run(Xd, Y)
    # new values in a new buffer, then new contents in the same buffer: both re-summed on the next run
    for step in range(2):
        val2 = (val * (0.5 + step) - 0.25).astype(np.float32)
        if step == 0:
            dval = dev(val2)
        else:
            dval.copy_(torch.from_numpy(val2))
        agg.set_val(dval)
        agg.gcn_run(Xd, Y)
        y64, scale = orc.spmm_f64(ptr, idx, val2, X)
        assert rel_gate(Y.cpu().numpy(), y64, scale, TOL)[0] == 0
        assert np.array_equal(agg.merged_arrays()[2].view(np.int32), merged_np(ptr, idx, val2)[2].view(np.int32))


def test_merge_automatic_rule(gn, cuda, graph):
    """automatic: small graphs and graphs without adjacent duplicates keep the CSR"""
    ptr, idx = graph
    X, val = rand_inputs(len(ptr) - 1, len(idx), 32, seed=7)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    assert agg.merged_edges == len(idx)  # below the automatic edge floor
    agg.set_merge_duplicates(ON)
    assert agg.merged_edges < len(idx)
    # 4.2M edges, sources distinct within each row
    n, d = 70000, 60
    rng = np.random.default_rng(3)
    ptr2 = (np.arange(n + 1, dtype=np.int64) * d).astype(np.int32)
    idx2 = ((np.arange(n)[:, None] * 7919 + np.arange(d)[None, :] * 1009 + rng.integers(0, 50, (n, 1))) % n).astype(np.int32).ravel()
    agg2 = gn.Aggregator(dev(ptr2), dev(idx2), torch.ones(len(idx2), device=cuda))
    assert agg2.merged_edges == len(idx2)
    with pytest.raises(gn.GnnaggError):
        agg2.merged_arrays()
    # the same rows with every source doubled (and row r ending with the source row r+1 starts with): merged, and the
    # count the automatic rule decides on is the m' of the view it then builds
    idx3 = np.repeat(idx2.reshape(n, d)[:, : d // 2], 2, axis=1)
    idx3[:-1, -1] = idx3[1:, 0]
    idx3 = idx3.ravel()
    assert len(idx3) == len(idx2) >= 4_000_000
    agg3 = gn.Aggregator(dev(ptr2), dev(idx3), torch.ones(len(idx3), device=cuda))
    want = merged_np(ptr2, idx3)
    assert agg3.merged_edges == len(want[1])
    assert np.array_equal(agg3.merged_arrays()[0], want[0])
