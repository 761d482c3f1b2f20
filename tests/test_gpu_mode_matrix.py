"""GAT, GAT backward, MLP and SDDMM through every instance of the shared walk agg_kernel<LPR, NV, MODE, SCHED, WE>.

The feature width F picks the virtual-warp width LPR and the float4 per lane NV, and with them the column chunk
CHUNK = LPR * 4 * NV that one pass covers.  Three kinds of branch in the walk depend on F: partial chunks (lanes with
no columns), several column passes (F > CHUNK: per-row scalars are written on the first pass only, per-edge dot
products are added across passes) and the item size WE (128 or 512 edges per warp; a graph below 4M edges gets 512
only through set_warp_edges).  Every case prefills its outputs with NaN, so an element nobody writes fails, and
compares with the fp64 oracle; un-scheduled runs are repeated and must come out bit-identical.
test_mode_matrix_reaches_every_instance (CPU tier) restates the kernel choice and fails when the parametrization
stops reaching an instance, a partial chunk or a multi-pass width."""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from conftest import rel_gate
from gnnagg import synth
from gpu_util import dev, make_graph, rand_inputs

gpu = pytest.mark.gpu
TOL = 1e-5        # MLP, SDDMM, GCN
TOL_GAT = 1.2e-5  # __expf / __fdividef against exp() in fp64 (test_gpu_gat.py)
TOL_X = 1.2e-5    # GAT backward (test_gpu_backward.py)
TOL_A = 2.5e-5

EDGE_GRAPHS = ["bighub", "exact_items", "leading_trailing_empty", "short_rows", "hub"]
ITEM_SIZES = [128, 512]
SCHEDULES = [(1, [16]), (0, [4]), (2, [4, 32])]  # neighbour grouping, locality, locality + neighbour grouping


# ---------------------------------------------------------------- the kernel choice, restated
def lanes_for(F):
    """LPR, lanes per virtual warp (lanes_for, csrc/capi.cu:346)"""
    return 8 if F <= 32 else (16 if F <= 64 else 32)


def vectors_for(F):
    """NV, float4 per lane (agg_kernel_for, csrc/capi.cu:366-377)"""
    return 1 if F <= 128 else 2


def chunk_for(F):
    """columns covered by one pass (CHUNK, csrc/agg_kernels.cuh:115)"""
    return lanes_for(F) * 4 * vectors_for(F)


INSTANCES = {(lpr, nv, we) for lpr, nv in ((8, 1), (16, 1), (32, 1), (32, 2)) for we in ITEM_SIZES}


def _cases(names, lists, skip=()):
    """parametrize over the cross product of `lists`, without the combinations in `skip` (run by an existing test)"""
    out = [()]
    for values in lists:
        out = [c + (v,) for c in out for v in values]
    return pytest.mark.parametrize(names, [c for c in out if c not in skip])


# ---------------------------------------------------------------- helpers
def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda:0")


def _att(n, seed):
    return np.random.default_rng(seed).standard_normal((n, 2)).astype(np.float32)


def _sched_order(orc, ptr, idx, kind, params):
    """CSR edge id of every edge in scheduled order: the locality schedules permute the edges (the ids travel through
    them as fp32 values, exact below 2^24 edges), neighbour grouping keeps the CSR order"""
    m = len(idx)
    if kind == 1:
        return np.arange(m)
    assert m < (1 << 24)
    _, _, _, ids = orc.locality(ptr, idx, params[0], len(ptr) - 1, np.arange(m, dtype=np.float32),
                                neighbor_num=params[1] if kind == 2 else 0)
    assert len(ids) == m
    return ids.astype(np.int64)


def _to_csr_order(gn, agg, in_sched, out_csr):
    """gnnagg_sched_to_csr_order; in_sched is a tensor or a raw device pointer"""
    src = C.c_void_p(in_sched if isinstance(in_sched, int) else in_sched.data_ptr())
    gn.check(gn.lib().gnnagg_sched_to_csr_order(agg.h, src, C.c_void_p(out_csr.data_ptr()), gn._stream()))
    return out_csr


def _edge_weights(gn, agg, m):
    """the un-normalised edge weights the last scheduled GAT run left (scheduled order)"""
    w = np.empty(m, np.float32)
    gn.check(gn.lib().gnnagg_memcpy_d2h(w.ctypes.data, agg.gat_edge_weights_ptr(), m * 4))
    return w


# ---------------------------------------------------------------- GAT forward
GAT_WIDTHS = [4, 20, 36, 100, 132, 160, 260, 512, 1000, 1024]  # 256: test_gpu_gat.test_gat_fused_unscheduled
GAT_SCHED_WIDTHS = [20, 36, 100, 160, 256, 260, 512]


@gpu
@_cases("gname,F,we", [EDGE_GRAPHS, GAT_WIDTHS, ITEM_SIZES])
def test_gat_unscheduled(gn, orc, cuda, gname, F, we):
    ptr, idx = make_graph(gname, seed=F + we)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 1)
    att = _att(n, F + 2)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    Y = agg.gat_run(dev(X), dev(att), _nan(n, F))
    y64, _, scale = orc.gat_f64(ptr, idx, att, X)
    bad, worst = rel_gate(Y.cpu().numpy(), y64, scale, TOL_GAT)
    assert bad == 0, (gname, F, we, worst)
    assert torch.equal(Y, agg.gat_run(dev(X), dev(att), _nan(n, F)))


@gpu
@_cases("sched,F,we", [SCHEDULES, GAT_SCHED_WIDTHS, ITEM_SIZES])
def test_gat_scheduled(gn, orc, cuda, sched, F, we):
    """Y and the un-normalised edge weights in scheduled order.  Under the locality schedules the groups of one target
    lie in several slices: the denominator is added with atomics (on the first column pass only), the rows with RED,
    and gat_scale_kernel divides at the end."""
    kind, params = sched
    ptr, idx = make_graph("hub", seed=F + kind)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 3)
    att = _att(n, F + 4)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    agg.schedule(kind, params)
    Y = agg.gat_run(dev(X), dev(att), _nan(n, F), scheduled=True)
    y64, _, scale = orc.gat_f64(ptr, idx, att, X)
    bad, worst = rel_gate(Y.cpu().numpy(), y64, scale, TOL_GAT)
    assert bad == 0, (sched, F, we, worst)
    w64 = orc.edge_weight_f64(ptr, idx, att)
    np.testing.assert_allclose(_edge_weights(gn, agg, m), w64[_sched_order(orc, ptr, idx, kind, params)], rtol=3e-6)


@gpu
@pytest.mark.parametrize("scheduled", [False, True])
@pytest.mark.parametrize("F", [64, 160])
def test_gat_run_host(gn, orc, cuda, F, scheduled):
    """gnnagg_gat_run_host (square graph): the oracle, and bit-equality with the device call when un-scheduled"""
    ptr, idx = make_graph("hub", seed=F)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 9)
    att = _att(n, F + 10)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    if scheduled:
        agg.schedule(0, [4])
    hY = torch.full((n, F), float("nan")).pin_memory()
    agg.gat_run_host(torch.from_numpy(X).pin_memory(), torch.from_numpy(att).pin_memory(), hY, scheduled=scheduled)
    y64, _, scale = orc.gat_f64(ptr, idx, att, X)
    bad, worst = rel_gate(hY.numpy(), y64, scale, TOL_GAT)
    assert bad == 0, (F, scheduled, worst)
    if not scheduled:
        assert np.array_equal(hY.numpy(), agg.gat_run(dev(X), dev(att), _nan(n, F)).cpu().numpy())


# ---------------------------------------------------------------- gnnagg_sched_to_csr_order
@gpu
@pytest.mark.parametrize("sched", SCHEDULES)
@pytest.mark.parametrize("F", [20, 160, 260])
def test_sched_to_csr_order_feeds_gat_backward(gn, orc, cuda, sched, F):
    """the weights a scheduled GAT run leaves, brought back to CSR order, are what gnnagg_gat_backward(w = ...) takes"""
    kind, params = sched
    ptr, idx = make_graph("hub", seed=F + 10 * kind)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 5)
    dY, _ = rand_inputs(n, m, F, seed=F + 6)
    att = _att(n, F + 7)
    Xd, dYd = dev(X), dev(dY)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.transpose_build()
    agg.schedule(kind, params)
    Y = agg.gat_run(Xd, dev(att), _nan(n, F), scheduled=True)
    w = _to_csr_order(gn, agg, agg.gat_edge_weights_ptr(), _nan(m))
    np.testing.assert_allclose(w.cpu().numpy(), orc.edge_weight_f64(ptr, idx, att), rtol=3e-6)
    x64, a64, sx, sa = orc.gat_backward_f64(ptr, idx, att, X, dY)
    for den in (agg.add_to_center(w, _nan(n)), None):
        dX, dA = agg.gat_backward(Xd, None, Y, dYd, _nan(n, F), _nan(n, 2), w=w, den=den)
        bad, worst = rel_gate(dX.cpu().numpy(), x64, sx, TOL_X)
        assert bad == 0, ("dX", sched, F, den is None, worst)
        bad, worst = rel_gate(dA.cpu().numpy(), a64, sa, TOL_A)
        assert bad == 0, ("datt", sched, F, den is None, worst)


@gpu
def test_sched_to_csr_order_copies_and_errors(gn, orc, cuda):
    """a plain copy without a schedule and under neighbour grouping (in place too), the inverse permutation after a
    locality schedule; rejected on the host in place after a locality schedule and after one that dropped edges"""
    ptr, idx = make_graph("hub", seed=3)
    n, m = len(ptr) - 1, len(idx)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    src = torch.randn(m, device=cuda)
    assert torch.equal(_to_csr_order(gn, agg, src, _nan(m)), src)
    agg.schedule(1, [16])
    assert torch.equal(_to_csr_order(gn, agg, src, _nan(m)), src)
    same = src.clone()
    assert torch.equal(_to_csr_order(gn, agg, same, same), src)
    agg.schedule(0, [4])
    expect = torch.empty_like(src)
    expect[dev(_sched_order(orc, ptr, idx, 0, [4]))] = src  # scheduled edge k is CSR edge order[k]
    assert torch.equal(_to_csr_order(gn, agg, src, _nan(m)), expect)
    before = agg.launches
    with pytest.raises(gn.GnnaggError, match="in place"):
        _to_csr_order(gn, agg, same, same)
    assert agg.launches == before and torch.equal(same, src)
    agg.schedule(0, [4], total_num_v=n // 2)  # sources >= n/2 lie outside every slice
    assert int(agg.scheduled_arrays()[0][-1]) < m
    before, out = agg.launches, _nan(m)
    with pytest.raises(gn.GnnaggError, match="dropped"):
        _to_csr_order(gn, agg, src, out)
    assert agg.launches == before and bool(torch.isnan(out).all())


# ---------------------------------------------------------------- GAT backward
BWD_WIDTHS = [4, 20, 36, 100, 160, 260, 512, 1024]
BWD_LARGE = (160, 512)  # (F, WE) of test_gat_backward_large_graph_wide_rows: 4.2M edges pick 512 automatically


@gpu
@_cases("gname,F,we", [EDGE_GRAPHS, BWD_WIDTHS, ITEM_SIZES])
def test_gat_backward(gn, orc, cuda, gname, F, we):
    """both traversals: pass 1 over the CSR (dot products added across column passes, row sums on the last pass) and
    pass 2 over the transposed CSR (dX and the source half of d att, a row scalar written on the first pass)"""
    ptr, idx = make_graph(gname, seed=F + we + 1)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 11)
    dY, _ = rand_inputs(n, m, F, seed=F + 12)
    att = _att(n, F + 13)
    Xd, dYd, attd = dev(X), dev(dY), dev(att)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    agg.transpose_build()
    Y = agg.gat_run(Xd, attd, _nan(n, F))
    dX, dA = agg.gat_backward(Xd, attd, Y, dYd, _nan(n, F), _nan(n, 2))
    x64, a64, sx, sa = orc.gat_backward_f64(ptr, idx, att, X, dY)
    bad, worst = rel_gate(dX.cpu().numpy(), x64, sx, TOL_X)
    assert bad == 0, ("dX", gname, F, we, worst)
    for half, name in ((0, "destination"), (1, "source")):
        bad, worst = rel_gate(dA.cpu().numpy()[:, half], a64[:, half], sa[:, half], TOL_A)
        assert bad == 0, ("datt " + name, gname, F, we, worst)
    dX2, dA2 = agg.gat_backward(Xd, attd, Y, dYd, _nan(n, F), _nan(n, 2))
    assert torch.equal(dX, dX2) and torch.equal(dA, dA2)


@gpu
def test_gat_backward_large_graph_wide_rows(gn, orc, cuda):
    """4.2M edges at F = 160 (two float4 per lane, partial second vector): the 512-edge kernels and the large-graph
    pass 2 (permute, row sum, plain aggregation), against the oracle on the whole graph"""
    F = BWD_LARGE[0]
    n, m = 150000, 4200000
    ptr_d, idx_d = synth.rmat_csr(n, m, seed=322, device=cuda)
    ptr, idx = ptr_d.cpu().numpy(), idx_d.cpu().numpy()
    X, _ = rand_inputs(n, 1, F, seed=98)
    dY, _ = rand_inputs(n, 1, F, seed=99)
    att = _att(n, 100)
    Xd, dYd, attd = dev(X), dev(dY), dev(att)
    agg = gn.Aggregator(ptr_d, idx_d)
    agg.transpose_build()
    Y = agg.gat_run(Xd, attd, _nan(n, F))
    dX, dA = agg.gat_backward(Xd, attd, Y, dYd, _nan(n, F), _nan(n, 2))
    x64, a64, sx, sa = orc.gat_backward_f64(ptr, idx, att, X, dY)
    bad, worst = rel_gate(dX.cpu().numpy(), x64, sx, TOL_X)
    assert bad == 0, ("dX", worst)
    bad, worst = rel_gate(dA.cpu().numpy(), a64, sa, TOL_A)
    assert bad == 0, ("datt", worst)
    dX2, dA2 = agg.gat_backward(Xd, attd, Y, dYd, _nan(n, F), _nan(n, 2))
    assert torch.equal(dX, dX2) and torch.equal(dA, dA2)


# ---------------------------------------------------------------- MLP
MLP_WIDTHS = [4, 20, 32, 36, 96, 100, 160, 256, 260, 512]
MLP_SCHED_WIDTHS = [20, 36, 100, 160, 260]
# run by test_gpu_mlp.test_mlp_parity (F = 32 with the automatic 128-edge items)
MLP_SKIP = {(g, 32, 128) for g in ("short_rows", "hub", "leading_trailing_empty", "exact_items")}


def _mlp_inputs(n, F, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal((n, F)).astype(np.float32), (rng.standard_normal((F, F)) / np.sqrt(F)).astype(np.float32)


@functools.lru_cache(maxsize=None)
def _mlp_case(gname, F):
    """graph, inputs and fp64 oracle of an MLP case, shared by both item sizes and the scheduled runs (the oracle
    runs a mat-vec per edge, seconds on the hub rows at the widest F)"""
    import oracle

    ptr, idx = make_graph(gname, seed=F + 7)
    X, W = _mlp_inputs(len(ptr) - 1, F, F + 8)
    return ptr, idx, X, W, oracle.mlp_f64(ptr, idx, X, W)


@gpu
@_cases("gname,F,we", [EDGE_GRAPHS, MLP_WIDTHS, ITEM_SIZES], skip=MLP_SKIP)
def test_mlp_unscheduled(gn, cuda, gname, F, we):
    ptr, idx, X, W, (y64, scale) = _mlp_case(gname, F)
    n = len(ptr) - 1
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    Y = agg.mlp_run(dev(X), dev(W), _nan(n, F))
    bad, worst = rel_gate(Y.cpu().numpy(), y64, scale, TOL)
    assert bad == 0, (gname, F, we, worst)
    assert torch.equal(Y, agg.mlp_run(dev(X), dev(W), _nan(n, F)))


@gpu
@_cases("sched,F,we", [SCHEDULES, MLP_SCHED_WIDTHS, ITEM_SIZES])
def test_mlp_scheduled(gn, cuda, sched, F, we):
    ptr, idx, X, W, (y64, scale) = _mlp_case("hub", F)
    n = len(ptr) - 1
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    agg.schedule(*sched)
    Y = agg.mlp_run(dev(X), dev(W), _nan(n, F), scheduled=True)
    bad, worst = rel_gate(Y.cpu().numpy(), y64, scale, TOL)
    assert bad == 0, (sched, F, we, worst)


@gpu
@pytest.mark.parametrize("F", [30, 1028])
def test_mlp_rejects_bad_width(gn, cuda, F):
    """F must be a multiple of 4 in [4, 1024]: rejected on the host, before the projection or the walk launches"""
    ptr, idx = make_graph("short_rows", seed=1)
    n = len(ptr) - 1
    agg = gn.Aggregator(dev(ptr), dev(idx))
    X, W = _mlp_inputs(n, F, 1)
    Y = _nan(n, F)
    before = agg.launches
    with pytest.raises(gn.GnnaggError, match="multiple of 4"):
        agg.mlp_run(dev(X), dev(W), Y)
    assert agg.launches == before and bool(torch.isnan(Y).all())
    empty = gn.Aggregator(torch.zeros(1, dtype=torch.int32, device=cuda), torch.zeros(0, dtype=torch.int32, device=cuda))
    with pytest.raises(gn.GnnaggError, match="multiple of 4"):  # also on a graph with nothing to aggregate
        empty.mlp_run(torch.zeros((0, F), device=cuda), torch.zeros((F, F), device=cuda), torch.zeros((0, F), device=cuda))


@gpu
def test_mlp_rejects_non_square_w(gn, cuda):
    ptr, idx = make_graph("short_rows", seed=1)
    n = len(ptr) - 1
    agg = gn.Aggregator(dev(ptr), dev(idx))
    with pytest.raises(gn.GnnaggError, match="W must be"):
        agg.mlp_run(torch.zeros((n, 32), device=cuda), torch.zeros((32, 64), device=cuda), _nan(n, 32))


# ---------------------------------------------------------------- SDDMM
SDDMM_WIDTHS = [4, 20, 36, 100, 160, 260, 512, 1024]
# run by test_gpu_gat.test_sddmm (F = 20 with the automatic 128-edge items)
SDDMM_SKIP = {(g, 20, 128) for g in ("short_rows", "hub", "leading_trailing_empty")}


@gpu
@_cases("gname,F,we", [EDGE_GRAPHS, SDDMM_WIDTHS, ITEM_SIZES], skip=SDDMM_SKIP)
def test_sddmm(gn, orc, cuda, gname, F, we):
    """un-scheduled and under neighbour grouping (the one schedule SDDMM takes; it keeps the CSR edge order)"""
    ptr, idx = make_graph(gname, seed=F + we + 2)
    n, m = len(ptr) - 1, len(idx)
    rng = np.random.default_rng(F + 14)
    X1 = rng.standard_normal((n, F)).astype(np.float32)
    X2 = rng.standard_normal((n, F)).astype(np.float32)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    v64, scale = orc.sddmm_f64(ptr, idx, X1, X2)
    out = agg.sddmm(dev(X1), dev(X2), _nan(m))
    bad, worst = rel_gate(out.cpu().numpy(), v64, scale, TOL)
    assert bad == 0, (gname, F, we, worst)
    assert torch.equal(out, agg.sddmm(dev(X1), dev(X2), _nan(m)))
    agg.schedule(1, [16])
    out_s = agg.sddmm(dev(X1), dev(X2), _nan(m), scheduled=True)
    bad, worst = rel_gate(out_s.cpu().numpy(), v64, scale, TOL)
    assert bad == 0, ("scheduled", gname, F, we, worst)


# ---------------------------------------------------------------- edge-wise GCN (its own kernel, RED per edge)
@gpu
@pytest.mark.parametrize("gname", ["hub", "bighub"])
@pytest.mark.parametrize("F", [4, 20, 36, 100, 160, 260, 1024])
def test_gcn_edgewise_widths(gn, orc, cuda, gname, F):
    ptr, idx = make_graph(gname, seed=F + 15)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + 16)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    Y = agg.gcn_run_edgewise(dev(X), _nan(n, F))
    y64, scale = orc.spmm_f64(ptr, idx, val, X)
    bad, worst = rel_gate(Y.cpu().numpy(), y64, scale, TOL)
    assert bad == 0, (gname, F, worst)


# ---------------------------------------------------------------- the matrix reaches every instance (CPU tier)
def _params(test):
    """every parameter set of a test function, as dicts"""
    sets = [{}]
    for mark in getattr(test, "pytestmark", []):
        if mark.name != "parametrize":
            continue
        names = [s.strip() for s in mark.args[0].split(",")]
        rows = [dict(zip(names, v if len(names) > 1 else (v,))) for v in mark.args[1]]
        sets = [dict(s, **r) for s in sets for r in rows]
    return sets


def _reached(mode):
    """(F, WE, scheduled) of every case that runs `mode` through agg_kernel"""
    out = []
    if mode == "GAT":
        out += [(p["F"], p["we"], False) for p in _params(test_gat_unscheduled)]
        out += [(p["F"], p["we"], True) for p in _params(test_gat_scheduled)]
    elif mode in ("GATBWD", "GATBWD2"):  # the two traversals of one backward call
        out += [(p["F"], p["we"], False) for p in _params(test_gat_backward)]
        if mode == "GATBWD":  # pass 2 of a graph this large is permute + row sum + the GCN aggregation
            out += [BWD_LARGE + (False,)]
    elif mode == "MLP":
        out += [(p["F"], p["we"], False) for p in _params(test_mlp_unscheduled)]
        out += [(p["F"], p["we"], True) for p in _params(test_mlp_scheduled)]
    elif mode == "SDDMM":
        out += [(p["F"], p["we"], s) for p in _params(test_sddmm) for s in (False, True)]
    return out


@pytest.mark.parametrize("mode", ["GAT", "GATBWD", "GATBWD2", "MLP", "SDDMM"])
def test_mode_matrix_reaches_every_instance(mode):
    cases = _reached(mode)
    for sched in sorted({s for _, _, s in cases}):
        widths = {(F, we) for F, we, s in cases if s == sched}
        assert {(lanes_for(F), vectors_for(F), we) for F, we in widths} == INSTANCES, (mode, sched)
        for lpr, nv in {(lanes_for(F), vectors_for(F)) for F, _ in widths}:
            assert any(F % chunk_for(F) and (lanes_for(F), vectors_for(F)) == (lpr, nv) for F, _ in widths), \
                (mode, sched, "no partial chunk for", (lpr, nv))
        assert any(F > chunk_for(F) for F, _ in widths), (mode, sched, "no multi-pass width")
    scheduled = {s for _, _, s in cases}
    assert scheduled == ({False} if mode.startswith("GATBWD") else {False, True}), mode
    if mode in ("GAT", "MLP"):
        assert {p["sched"][0] for p in _params(test_gat_scheduled if mode == "GAT" else test_mlp_scheduled)} == {0, 1, 2}


def test_kernel_choice_restatement():
    """the width classes of the restatement, at their borders"""
    assert [(lanes_for(F), vectors_for(F), chunk_for(F)) for F in (4, 32, 36, 64, 68, 128, 132, 256, 260, 1024)] == [
        (8, 1, 32), (8, 1, 32), (16, 1, 64), (16, 1, 64), (32, 1, 128), (32, 1, 128), (32, 2, 256), (32, 2, 256),
        (32, 2, 256), (32, 2, 256)]
