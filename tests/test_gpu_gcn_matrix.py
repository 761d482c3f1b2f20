"""GCN aggregation through every instance of the shared walk agg_kernel<LPR, NV, kModeGCN, SCHED, WE, XBF16>: the
counterpart of test_gpu_mode_matrix.py for gcn_run, gcn_run_acc, gcn_run_rows, the locality slices, the merged view,
the scheduled runs, gcn_backward (the transposed view) and gcn_layer.

Every width class of the walk is run with a partial chunk (lanes without columns) and, for two float4 per lane, with
several column passes (F > CHUNK), at both item sizes, on graphs whose rows cross items: one item (fix-up phase 1) and
more than kFixChunk = 32 carry items (phase 2, which also runs the out_row remapping of a compacted slice and the
clipping of a row range).  Every output starts as NaN, so an element nobody writes fails; results are compared with the
fp64 oracle at 1e-5 * sum|terms|; un-scheduled runs are repeated and must come out bit-identical.  A bf16 X (or dY) must
give, bit for bit, the fp32 run on the widened operand.  test_gcn_matrix_reaches_every_instance (CPU tier) restates the
kernel choice and the fix-up phases and fails when the parametrization stops reaching one of them."""
import functools

import numpy as np
import pytest
import torch

from conftest import rel_gate
from gnnagg import synth
from gpu_util import dev, make_graph, rand_inputs
from test_gpu_merge import dup_csr
from test_gpu_mode_matrix import (EDGE_GRAPHS, INSTANCES, ITEM_SIZES, SCHEDULES, _cases, _params, chunk_for, lanes_for,
                                  vectors_for)

gpu = pytest.mark.gpu
TOL = 1e-5
FIX_CHUNK = 32  # kFixChunk, csrc/agg_kernels.cuh: carry items one phase-1 fix-up thread sums
XDTS = ["fp32", "bf16"]

# 32 / 64 / 128 / 256: test_gpu_gcn.test_gcn_unscheduled_parity and test_gpu_bf16.test_bf16_bit_identical_to_widened_fp32
WIDTHS = [4, 20, 36, 100, 132, 160, 260, 512, 1000, 1024]
# 32 / 128 / 256: test_gpu_gcn.test_gcn_scheduled_parity_and_schedule_upload
SCHED_WIDTHS = [20, 36, 100, 160, 260, 512, 1024]
BWD_WIDTHS = [4, 20, 36, 100, 160, 260, 512, 1024]
MERGE_WIDTHS = [20, 36, 100, 160, 260, 1024]
SLICES = [2, 3, 5]
BWD_GRAPHS = EDGE_GRAPHS + ["hub_source"]
LAYERS = [(20, 12), (160, 64), (260, 32), (1024, 32)]  # (160, 64) combines on the tensor cores, the others in fp32
NUM_SRC_EXTRA = 37


# ---------------------------------------------------------------- graphs (numpy only: the CPU tier restates them)
@functools.lru_cache(maxsize=None)
def _graph(name):
    """the test graphs of gpu_util (hub and bighub with the hub row away from both ends and empty rows on both sides of
    it), and hub_source: bighub with 90 % of its edges pointing at source 3, so that row 3 of the transposed CSR spans
    more than 32 carry items at every item size"""
    if name == "hub_source":
        ptr, idx = make_graph("bighub", seed=2)
        idx = idx.copy()
        idx[np.random.default_rng(5).random(len(idx)) < 0.9] = 3
        return ptr, idx
    return make_graph(name, seed=2)


def _slice_bounds(n, S):
    """first source of every slice block (the width of gnnagg_set_locality_slices: ceil(n / S)), and n"""
    width = -(-n // S)
    return [min(c * width, n) for c in range(S)] + [n]


@functools.lru_cache(maxsize=None)
def _slice_graph(S):
    """a hub row whose sources all lie in the LAST source block (a long row in a compacted slice c > 0, summed by fix-up
    phase 2 through out_row), and one source block without edges: block 1, or block 0 for S = 2 (then slice 0, the one
    that writes every row, has nothing to walk)"""
    n = 4000
    ptr, idx = synth.small_random_csr(n, 9.0, 70 + S, empty_frac=0.3, hub=30000)
    idx = idx.copy()
    b = _slice_bounds(n, S)
    lo, width = b[S - 1], n - b[S - 1]
    rng = np.random.default_rng(S)
    empty = 1 if S > 2 else 0
    moved = (idx >= b[empty]) & (idx < b[empty + 1])
    idx[moved] = lo + rng.integers(0, width, int(moved.sum()))
    h = int(np.argmax(np.diff(ptr)))
    idx[ptr[h]:ptr[h + 1]] = lo + rng.integers(0, width, int(ptr[h + 1] - ptr[h]))
    return ptr, idx.astype(np.int32)


def _slice_ptrs(ptr, idx, S):
    """row pointers of the sub-CSRs a sliced run walks: slice 0 over all rows, the others compacted to their rows with
    edges"""
    n = len(ptr) - 1
    b = _slice_bounds(n, S)
    row = np.repeat(np.arange(n), np.diff(ptr))
    out = []
    for c in range(S):
        deg = np.bincount(row[(idx >= b[c]) & (idx < b[c + 1])], minlength=n)
        if c > 0:
            deg = deg[deg > 0]
        out.append(np.concatenate([[0], np.cumsum(deg)]))
    return out


def _transposed_ptr(idx, num_src):
    return np.concatenate([[0], np.cumsum(np.bincount(idx, minlength=num_src))])


@functools.lru_cache(maxsize=None)
def _dup_graph():
    return dup_csr()


def _row_partitions(gname, ptr):
    """two sets of row ranges that each cover every row once.  hub / bighub: the ranges of the second end just before the
    hub row, hold the hub row alone, and hold only empty rows; the first starts at the hub row.  leading_trailing_empty:
    ranges of empty rows only, single long rows, and a range that ends in the trailing empty rows.  exact_items: ranges
    whose first edge lies on an item boundary (row 3, edge 1024) and inside an item of 256 and 512 edges (row 5, edge
    2176)"""
    n = len(ptr) - 1
    if gname == "leading_trailing_empty":
        return [[0, 8, n], [0, 3, 5, 6, 8, 9, n]]
    if gname == "exact_items":
        return [[0, 4, n], [0, 3, 5, n]]
    deg = np.diff(ptr)
    h = int(np.argmax(deg))
    e0 = next(r for r in range(n - 1) if deg[r] == 0 and deg[r + 1] == 0 and r not in (h - 1, h + 1))
    return [[0, h, n], sorted({0, h // 2, h, h + 1, e0, e0 + 2, n})]


# ---------------------------------------------------------------- helpers
def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda:0")


def _written(Y):
    """no element still holds the NaN prefill (rel_gate counts err > bound, which is False for NaN)"""
    return not bool(torch.isnan(Y).any())


def same_bits(a, b):
    """equal bit patterns, and written: two outputs left at their NaN prefill have equal bits too"""
    return (a.dtype == b.dtype == torch.float32 and _written(a) and _written(b)
            and torch.equal(a.view(torch.int32), b.view(torch.int32)))


def _operand(X, xdt):
    """(what the case hands in, the fp32 X it stands for): X itself, or X rounded to bf16 and that widened exactly"""
    Xd = dev(X)
    if xdt == "fp32":
        return Xd, Xd
    Xb = Xd.to(torch.bfloat16)
    return Xb, Xb.float()


def _agg(gn, ptr, idx, val, we):
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.set_warp_edges(we)
    return agg


def _gate(Y, y64, scale, what):
    assert _written(Y), what + ("unwritten elements",)
    bad, worst = rel_gate(Y.cpu().numpy(), y64, scale, TOL)
    assert bad == 0, what + (worst,)


# ---------------------------------------------------------------- 1. un-scheduled forward
@gpu
@_cases("gname,F,we,xdt", [EDGE_GRAPHS, WIDTHS, ITEM_SIZES, XDTS])
def test_gcn_unscheduled(gn, orc, cuda, gname, F, we, xdt):
    ptr, idx = _graph(gname)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + we)
    agg = _agg(gn, ptr, idx, val, we)
    Xin, Xw = _operand(X, xdt)
    Y = agg.gcn_run(Xin, _nan(n, F))
    y64, scale = orc.spmm_f64(ptr, idx, val, Xw.cpu().numpy())
    _gate(Y, y64, scale, (gname, F, we, xdt))
    assert same_bits(Y, agg.gcn_run(Xin, _nan(n, F)))
    if xdt == "bf16":
        assert same_bits(Y, agg.gcn_run(Xw, _nan(n, F)))


# ---------------------------------------------------------------- 2. accumulate
@gpu
@_cases("gname,F,we,xdt", [["hub", "bighub"], WIDTHS, ITEM_SIZES, XDTS])
def test_gcn_accumulate(gn, orc, cuda, gname, F, we, xdt):
    """Y += A X onto a random base (rows of the base whose partial sum is exactly zero are skipped, row by row and
    column pass by column pass); accumulate=False is gcn_run"""
    ptr, idx = _graph(gname)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + we + 1)
    base, _ = rand_inputs(n, 1, F, seed=F + 2)
    agg = _agg(gn, ptr, idx, val, we)
    Xin, Xw = _operand(X, xdt)
    Y = agg.gcn_run_acc(Xin, dev(base))
    y64, scale = orc.spmm_f64(ptr, idx, val, Xw.cpu().numpy())
    _gate(Y, y64 + base.astype(np.float64), scale + np.abs(base), (gname, F, we, xdt))
    assert same_bits(Y, agg.gcn_run_acc(Xin, dev(base)))
    if xdt == "bf16":
        assert same_bits(Y, agg.gcn_run_acc(Xw, dev(base)))
    assert same_bits(agg.gcn_run_acc(Xin, _nan(n, F), accumulate=False), agg.gcn_run(Xin, _nan(n, F)))


# ---------------------------------------------------------------- 3. row ranges
ROW_GRAPHS = ["hub", "bighub", "leading_trailing_empty", "exact_items"]


@gpu
@_cases("gname,F,we,xdt", [ROW_GRAPHS, WIDTHS, ITEM_SIZES, XDTS])
def test_gcn_rows(gn, orc, cuda, gname, F, we, xdt):
    """gcn_run_rows over two partitions of the rows: the union is the oracle, bit for bit gcn_run (items keep their
    global numbering, a range only clips them); accumulating ranges add onto a base; a single range leaves every row
    outside it untouched"""
    ptr, idx = _graph(gname)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + we + 3)
    base, _ = rand_inputs(n, 1, F, seed=F + 4)
    agg = _agg(gn, ptr, idx, val, we)
    Xin, Xw = _operand(X, xdt)
    y64, scale = orc.spmm_f64(ptr, idx, val, Xw.cpu().numpy())
    full = agg.gcn_run(Xin, _nan(n, F))
    for cuts in _row_partitions(gname, ptr):
        ranges = list(zip(cuts[:-1], cuts[1:]))
        Y, Yacc = _nan(n, F), dev(base)
        for lo, hi in ranges:
            agg.gcn_run_rows(Xin, Y, lo, hi)
            agg.gcn_run_rows(Xin, Yacc, lo, hi, accumulate=True)
        _gate(Y, y64, scale, (gname, F, we, xdt, cuts))
        assert same_bits(Y, full), cuts
        _gate(Yacc, y64 + base.astype(np.float64), scale + np.abs(base), (gname, F, we, xdt, cuts, "accumulate"))
        if xdt == "bf16":
            Yw = _nan(n, F)
            for lo, hi in ranges:
                agg.gcn_run_rows(Xw, Yw, lo, hi)
            assert same_bits(Y, Yw), cuts
    full = full.cpu().numpy()
    for lo, hi in ranges:  # each range of the finer partition on its own
        Y = agg.gcn_run_rows(Xin, _nan(n, F), lo, hi).cpu().numpy()
        assert np.isnan(Y[:lo]).all() and np.isnan(Y[hi:]).all(), (lo, hi)
        assert np.array_equal(Y[lo:hi], full[lo:hi]), (lo, hi)


# ---------------------------------------------------------------- 4. locality slices
@gpu
@_cases("S,F,we,xdt", [SLICES, WIDTHS, ITEM_SIZES, XDTS])
def test_gcn_slices(gn, orc, cuda, S, F, we, xdt):
    """forced source slices: slice 0 writes every row, the compacted slices behind it add to theirs (out_row) -- here
    with a hub row in the last slice and a source block without edges; plain and accumulating runs"""
    ptr, idx = _slice_graph(S)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + we + 5)
    base, _ = rand_inputs(n, 1, F, seed=F + 6)
    agg = _agg(gn, ptr, idx, val, we)
    agg.set_locality_slices(S)
    Xin, Xw = _operand(X, xdt)
    y64, scale = orc.spmm_f64(ptr, idx, val, Xw.cpu().numpy())
    Y = agg.gcn_run(Xin, _nan(n, F))
    _gate(Y, y64, scale, (S, F, we, xdt))
    assert same_bits(Y, agg.gcn_run(Xin, _nan(n, F)))
    Yacc = agg.gcn_run_acc(Xin, dev(base))
    _gate(Yacc, y64 + base.astype(np.float64), scale + np.abs(base), (S, F, we, xdt, "accumulate"))
    if xdt == "bf16":
        assert same_bits(Y, agg.gcn_run(Xw, _nan(n, F)))
        assert same_bits(Yacc, agg.gcn_run_acc(Xw, dev(base)))


# ---------------------------------------------------------------- 5. merged view
@gpu
@_cases("F,we", [MERGE_WIDTHS, ITEM_SIZES])
def test_gcn_merged(gn, orc, cuda, F, we):
    """gcn_run, gcn_run_acc and gcn_run_rows on the merged view of a graph with long runs of duplicate edges"""
    ptr, idx = _dup_graph()
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + we + 7)
    base, _ = rand_inputs(n, 1, F, seed=F + 8)
    agg = _agg(gn, ptr, idx, val, we)
    agg.set_merge_duplicates(2)
    Xd = dev(X)
    y64, scale = orc.spmm_f64(ptr, idx, val, X)
    Y = agg.gcn_run(Xd, _nan(n, F))
    assert agg.merged_edges < m
    _gate(Y, y64, scale, (F, we))
    assert same_bits(Y, agg.gcn_run(Xd, _nan(n, F)))
    Yacc = agg.gcn_run_acc(Xd, dev(base))
    _gate(Yacc, y64 + base.astype(np.float64), scale + np.abs(base), (F, we, "accumulate"))
    assert same_bits(agg.gcn_run_acc(Xd, _nan(n, F), accumulate=False), Y)
    Yr = _nan(n, F)
    for lo, hi in [(0, 7), (7, 8), (8, 11), (11, 12), (12, n // 2), (n // 2, n)]:  # the hub row and the single-run row alone
        agg.gcn_run_rows(Xd, Yr, lo, hi)
    assert same_bits(Yr, Y)


# ---------------------------------------------------------------- 6. scheduled
@gpu
@_cases("sched,F,we,xdt", [SCHEDULES, SCHED_WIDTHS, ITEM_SIZES, XDTS])
def test_gcn_scheduled(gn, orc, cuda, sched, F, we, xdt):
    """groups of one target meet in registers, in Y through RED (every column pass); against the oracle of the uploaded
    schedule and of the CSR"""
    kind, params = sched
    ptr, idx = _graph("hub")
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=F + we + 9)
    agg = _agg(gn, ptr, idx, val, we)
    agg.schedule(kind, params)
    sp, si, stt, sv = agg.scheduled_arrays()
    Xin, Xw = _operand(X, xdt)
    Xw = Xw.cpu().numpy()
    Y = agg.gcn_run(Xin, _nan(n, F), scheduled=True)
    y64, scale = orc.spmm_grouped_f64(n, sp, si, val if sv is None else sv, stt, Xw)
    _gate(Y, y64, scale, (sched, F, we, xdt, "schedule"))
    y64, scale = orc.spmm_f64(ptr, idx, val, Xw)
    _gate(Y, y64, scale, (sched, F, we, xdt, "CSR"))


# ---------------------------------------------------------------- 7. backward
@gpu
@_cases("gname,F,we,xdt", [BWD_GRAPHS, BWD_WIDTHS, ITEM_SIZES, XDTS])
def test_gcn_backward(gn, orc, cuda, gname, F, we, xdt):
    """dX = A^T dY over the transposed CSR, with as many sources as rows and with 37 sources more (empty rows at the end
    of the transposed CSR: dX is 0 there)"""
    ptr, idx = _graph(gname)
    n, m = len(ptr) - 1, len(idx)
    dY, val = rand_inputs(n, m, F, seed=F + we + 10)
    agg = _agg(gn, ptr, idx, val, we)
    dYin, dYw = _operand(dY, xdt)
    for num_src in (n, n + NUM_SRC_EXTRA):
        agg.transpose_build(num_src)
        dX = agg.gcn_backward(dYin, _nan(num_src, F))
        d64, scale = orc.spmm_t_f64(ptr, idx, val, dYw.cpu().numpy(), num_src)
        _gate(dX, d64, scale, (gname, F, we, xdt, num_src))
        assert bool((dX[n:] == 0).all())
        assert same_bits(dX, agg.gcn_backward(dYin, _nan(num_src, F)))
        if xdt == "bf16":
            assert same_bits(dX, agg.gcn_backward(dYw, _nan(num_src, F)))


# ---------------------------------------------------------------- 8. layer
@gpu
@pytest.mark.parametrize("we", ITEM_SIZES)
@pytest.mark.parametrize("fin,fout", LAYERS)
def test_gcn_layer(gn, orc, cuda, fin, fout, we):
    ptr, idx = _graph("bighub")
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, fin, seed=fin + fout)
    W = (np.random.default_rng(fin).standard_normal((fin, fout)) / np.sqrt(fin)).astype(np.float32)
    agg = _agg(gn, ptr, idx, val, we)
    AX = _nan(n, fin)
    H = agg.gcn_layer(dev(X), dev(W), _nan(n, fout), AX)
    ax64, h64, hs = orc.gcn_layer_f64(ptr, idx, val, X, W)
    _gate(AX, ax64, orc.spmm_f64(ptr, idx, val, X)[1], (fin, fout, we, "AX"))
    _gate(H, h64, hs, (fin, fout, we, "H"))
    AX2 = _nan(n, fin)
    assert same_bits(H, agg.gcn_layer(dev(X), dev(W), _nan(n, fout), AX2)) and same_bits(AX, AX2)


# ---------------------------------------------------------------- 9. the item size follows the setting
@functools.lru_cache(maxsize=None)
def _follow_graph():
    """5000 rows (the host pipeline chunks above 4096), a hub row, and a third of the edges on source 17 (a long row of
    the transposed CSR)"""
    ptr, idx = synth.small_random_csr(5000, 9.0, 13, empty_frac=0.3, hub=30000)
    idx = idx.copy()
    idx[::3] = 17
    return ptr, idx


def _follow_run(gn, view, settings, X, val):
    """sets the item size before the view is built, runs, and runs again after each further setting"""
    ptr, idx = _dup_graph() if view == "merged" else _follow_graph()
    n, F = len(ptr) - 1, X.shape[1]
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.set_warp_edges(settings[0])
    if view == "merged":
        agg.set_merge_duplicates(2)
    elif view == "sliced":
        agg.set_locality_slices(3)
    elif view == "host":
        agg.set_host_pipeline(3)
    elif view == "transposed":
        agg.transpose_build()

    def run():
        if view == "host":
            hY = torch.full((n, F), float("nan")).pin_memory()
            return agg.gcn_run_host(torch.from_numpy(X).pin_memory(), hY).cuda()
        if view == "transposed":
            return agg.gcn_backward(dev(X), _nan(n, F))
        return agg.gcn_run(dev(X), _nan(n, F))

    out = [run()]
    for we in settings[1:]:
        agg.set_warp_edges(we)
        out.append(run())
    return out


@gpu
@pytest.mark.parametrize("before,after", [(0, 512), (512, 128), (512, 0)])
@pytest.mark.parametrize("view", ["transposed", "merged", "sliced", "host"])
def test_item_size_follows_setting(gn, cuda, view, before, after):
    """set_warp_edges after a derived view exists: the next run is bit for bit that of an aggregator that had the
    setting before its first run (the two item sizes sum long rows in different orders, which the last check confirms)"""
    ptr, idx = _dup_graph() if view == "merged" else _follow_graph()
    X, val = rand_inputs(len(ptr) - 1, len(idx), 100, seed=21)
    first, late = _follow_run(gn, view, (before, after), X, val)
    (fresh,) = _follow_run(gn, view, (after,), X, val)
    assert same_bits(late, fresh), (view, before, after)
    assert _written(first) and not same_bits(first, fresh)


# ---------------------------------------------------------------- 10. equal-valued duplicates
def _dup_run_graph():
    """300 rows; row 5 holds a run of 1300 edges from source 9 between other edges (the transposed row 9 then holds the
    run too).  1300 > 2 * 512 - 1: at least one whole 512-edge item lies inside the run"""
    ptr, idx = synth.small_random_csr(300, 8.0, 17, empty_frac=0.2)
    deg = np.diff(ptr).astype(np.int64)
    rng = np.random.default_rng(17)
    rows = [idx[ptr[r]:ptr[r + 1]] for r in range(300)]
    rows[5] = np.concatenate([rng.integers(0, 300, 40), np.full(1300, 9), rng.integers(0, 300, 20)]).astype(np.int32)
    deg[5] = len(rows[5])
    ptr = np.concatenate([[0], np.cumsum(deg)]).astype(np.int32)
    return ptr, np.concatenate(rows).astype(np.int32)


@gpu
@pytest.mark.parametrize("F", [100, 260])
def test_gcn_equal_valued_duplicates(gn, orc, cuda, F):
    """GCN normalisation gives every duplicate (row, source) pair one value, so a run of duplicates adds identical terms
    along one fp32 chain of up to 512 FMA per item, whose rounding errors do not cancel; forward and backward, merge off"""
    ptr, idx = _dup_run_graph()
    n, m = len(ptr) - 1, len(idx)
    val = synth.gcn_norm_val(torch.from_numpy(ptr), torch.from_numpy(idx)).numpy()
    X, _ = rand_inputs(n, m, F, seed=F + 11)
    agg = _agg(gn, ptr, idx, val, 512)
    agg.set_merge_duplicates(1)
    y64, scale = orc.spmm_f64(ptr, idx, val, X)
    _gate(agg.gcn_run(dev(X), _nan(n, F)), y64, scale, (F, "forward"))
    agg.transpose_build()
    d64, scale = orc.spmm_t_f64(ptr, idx, val, X, n)
    _gate(agg.gcn_backward(dev(X), _nan(n, F)), d64, scale, (F, "backward"))


# ---------------------------------------------------------------- 11. the matrix reaches every instance (CPU tier)
def _spans(ptr, EB):
    """(rows that span more than one item: fix-up phase 1, rows with more than FIX_CHUNK carry items: phase 2)"""
    ptr = np.asarray(ptr, np.int64)
    rs, re = ptr[:-1], ptr[1:]
    nz = re > rs
    first, last = rs[nz] // EB + 1, (re[nz] - 1) // EB
    return bool((last >= first).any()), bool((last - first >= FIX_CHUNK).any())


def _reached(group):
    """(F, WE, xdt, row pointers of every CSR the case walks un-scheduled) of every case of a group"""
    if group == "unscheduled":
        return [(p["F"], p["we"], p["xdt"], [_graph(p["gname"])[0]]) for p in _params(test_gcn_unscheduled)]
    if group == "accumulate":
        return [(p["F"], p["we"], p["xdt"], [_graph(p["gname"])[0]]) for p in _params(test_gcn_accumulate)]
    if group == "rows":
        return [(p["F"], p["we"], p["xdt"], [_graph(p["gname"])[0]]) for p in _params(test_gcn_rows)]
    if group == "sliced":
        return [(p["F"], p["we"], p["xdt"], _slice_ptrs(*_slice_graph(p["S"]), p["S"])) for p in _params(test_gcn_slices)]
    if group == "backward":
        out = []
        for p in _params(test_gcn_backward):
            ptr, idx = _graph(p["gname"])
            out.append((p["F"], p["we"], p["xdt"], [_transposed_ptr(idx, len(ptr) - 1)]))
        return out
    assert group == "scheduled"  # no carries: groups meet in Y through RED
    return [(p["F"], p["we"], p["xdt"], []) for p in _params(test_gcn_scheduled)]


@pytest.mark.parametrize("group", ["unscheduled", "scheduled", "accumulate", "rows", "sliced", "backward"])
def test_gcn_matrix_reaches_every_instance(group):
    cases = _reached(group)
    for xdt in XDTS:
        mine = [c for c in cases if c[2] == xdt]
        assert {(lanes_for(F), vectors_for(F), we) for F, we, _, _ in mine} == INSTANCES, (group, xdt)
        for lpr, nv, we in INSTANCES:
            inst = [(F, ptrs) for F, w, _, ptrs in mine if (lanes_for(F), vectors_for(F), w) == (lpr, nv, we)]
            assert any(F % chunk_for(F) for F, _ in inst), (group, xdt, "no partial chunk for", (lpr, nv, we))
            if nv == 2:
                assert any(F > chunk_for(F) for F, _ in inst), (group, xdt, "no multi-pass width for", (lpr, nv, we))
            if group == "scheduled":
                continue
            EB = we // (32 // lpr)
            spans = [_spans(p, EB) for _, ptrs in inst for p in ptrs]
            assert any(s[0] for s in spans), (group, xdt, "no fix-up phase 1 for", (lpr, nv, we))
            assert any(s[1] for s in spans), (group, xdt, "no fix-up phase 2 for", (lpr, nv, we))
    if group == "scheduled":
        assert {p["sched"][0] for p in _params(test_gcn_scheduled)} == {0, 1, 2}


def test_gcn_matrix_graphs():
    """what the graph builders promise: the hub row away from both ends with two empty rows elsewhere, the hub row of a
    slice graph in the last source block with a block without edges, a transposed hub row beyond 32 carry items of 512
    edges, and a duplicate run covering a whole 512-edge item"""
    for gname in ("hub", "bighub"):
        ptr, _ = _graph(gname)
        cuts = _row_partitions(gname, ptr)[1]
        h = int(np.argmax(np.diff(ptr)))
        assert cuts[0] < h and h in cuts and h + 1 in cuts and cuts[-1] > h + 1 and all(np.diff(cuts) > 0)
    for S in SLICES:
        ptr, idx = _slice_graph(S)
        b = _slice_bounds(len(ptr) - 1, S)
        h = int(np.argmax(np.diff(ptr)))
        assert (idx[ptr[h]:ptr[h + 1]] >= b[S - 1]).all()
        assert not ((idx >= b[1 if S > 2 else 0]) & (idx < b[2 if S > 2 else 1])).any()
        assert _spans(_slice_ptrs(ptr, idx, S)[S - 1], 512)[1]
    ptr, idx = _graph("hub_source")
    assert _spans(_transposed_ptr(idx, len(ptr) - 1), 512)[1]
    ptr, idx = _dup_run_graph()
    run = ptr[5] + 40
    assert (idx[run:run + 1300] == 9).all() and -(-run // 512) * 512 + 512 <= run + 1300


def test_gcn_matrix_checks_reject_the_nan_prefill():
    """an output the kernel never wrote (still NaN) fails the gate and the bit-equality checks"""
    y64, scale = np.ones((2, 4), np.float32), np.ones((2, 4), np.float32)
    Y = torch.ones((2, 4))
    _gate(Y, y64, scale, ())
    Y[1, 3] = float("nan")
    assert rel_gate(Y.numpy(), y64, scale, TOL)[0] == 0  # what the gate alone would let through
    with pytest.raises(AssertionError, match="unwritten"):
        _gate(Y, y64, scale, ())
    assert not same_bits(Y, Y.clone())
    assert not same_bits(torch.full((2, 4), float("nan")), torch.full((2, 4), float("nan")))
