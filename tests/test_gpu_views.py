"""GPU tier: the graphs an aggregator derives from its CSR (source slices of the host pipeline, locality slices, the
transposed CSR, the merged view of duplicate edges, the schedules).  Launch counts per entry point, edge values that
follow gnnagg_set_val into every derived copy, profiling brackets that reach the aggregator's own events, and
derived structures rebuilt on one aggregator."""
import numpy as np
import pytest
import torch

from conftest import rel_gate
from gnnagg import synth
from gpu_util import dev, rand_inputs
from test_gpu_merge import dup_csr

pytestmark = pytest.mark.gpu
TOL = 1e-5
F = 64

# launches counted by gnnagg_launch_count for each step of launch_script, recorded on a B200 by running launch_script on
# the commit before the aggregator's derived graphs became owned views; every count must stay as it was there
EXPECTED_LAUNCHES = {
    "gcn_we128": 5, "gcn_we512": 4,
    "merge_first": 11, "merge_second": 2, "merge_set_val": 3,
    "loc_first": 31, "loc_second": 7, "loc_set_val": 10,
    "host_slices2": 38, "host_chunks": 12, "layer_host": 20,
    "prepare": 0, "run_rows": 3,
    "transpose_build": 5, "gcn_backward": 6, "gat_run": 3, "gat_backward": 6,
    "schedule_ng": 1, "schedule_loc": 2, "sched_set_val": 1, "sched_gcn": 1, "sched_gat": 2,
    "sddmm": 1, "edge_softmax": 5,
    "large_auto_merge": 14, "large_second": 3, "large_transpose_build": 5, "large_gat_run": 5, "large_gat_backward": 12,
    "large_gcn_backward": 4,
}


@pytest.fixture(scope="module")
def small():
    ptr, idx = dup_csr()  # 5000 rows (host pipeline chunks rows), hub rows (second fix-up pass), 1/3 duplicates
    return ptr, idx


@pytest.fixture(scope="module")
def large(cuda):
    """R-MAT, 4.2M edges of which 15 % repeat their row's previous source: above the automatic merge rule's floor and
    the large-graph path of the GAT backward"""
    ptr_d, idx_d = synth.rmat_csr(100000, 4200000, seed=321, device=cuda)
    return ptr_d, idx_d, ptr_d.cpu().numpy(), idx_d.cpu().numpy()


def _att(n, seed):
    return (np.random.default_rng(seed).standard_normal((n, 2)) * 0.5).astype(np.float32)


def launch_script(gn, cuda, small, large):
    """the launches of each step of a fixed sequence of calls, {step: delta}"""
    out = {}
    ptr, idx = small
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=1)
    Xd, Y = dev(X), torch.empty((n, F), device=cuda)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))

    def step(name, fn):
        before = agg.launches
        fn()
        out[name] = agg.launches - before

    step("gcn_we128", lambda: (agg.set_warp_edges(128), agg.gcn_run(Xd, Y)))
    step("gcn_we512", lambda: (agg.set_warp_edges(512), agg.gcn_run(Xd, Y)))
    agg.set_warp_edges(0)
    agg.set_merge_duplicates(2)
    step("merge_first", lambda: agg.gcn_run(Xd, Y))
    step("merge_second", lambda: agg.gcn_run(Xd, Y))
    step("merge_set_val", lambda: (agg.set_val(dev(val * 2)), agg.gcn_run(Xd, Y)))
    agg.set_merge_duplicates(1)
    agg.set_locality_slices(3)
    step("loc_first", lambda: agg.gcn_run(Xd, Y))
    step("loc_second", lambda: agg.gcn_run(Xd, Y))
    step("loc_set_val", lambda: (agg.set_val(dev(val)), agg.gcn_run(Xd, Y)))
    agg.set_locality_slices(1)
    hX, hY = torch.from_numpy(X).pin_memory(), torch.empty((n, F)).pin_memory()
    W = (np.random.default_rng(2).standard_normal((F, 32)) / 8).astype(np.float32)
    step("host_slices2", lambda: (agg.set_host_pipeline(2), agg.gcn_run_host(hX, hY)))
    step("host_chunks", lambda: (agg.set_host_pipeline(-1), agg.gcn_run_host(hX, hY)))
    step("layer_host", lambda: agg.gcn_layer_host(hX, torch.from_numpy(W), torch.empty((n, 32)).pin_memory()))
    step("prepare", lambda: gn.check(gn.lib().gnnagg_prepare(agg.h, F, None)))
    step("run_rows", lambda: agg.gcn_run_rows(Xd, Y, 0, n // 2))
    att = dev(_att(n, 3))
    step("transpose_build", lambda: agg.transpose_build())
    step("gcn_backward", lambda: agg.gcn_backward(Xd, torch.empty_like(Y)))
    step("gat_run", lambda: agg.gat_run(Xd, att, Y))
    step("gat_backward", lambda: agg.gat_backward(Xd, att, Y, Xd, torch.empty_like(Y), torch.empty((n, 2), device=cuda)))
    step("schedule_ng", lambda: agg.schedule(1, [16]))
    step("schedule_loc", lambda: agg.schedule(0, [4]))
    step("sched_set_val", lambda: agg.set_val(dev(val)))
    step("sched_gcn", lambda: agg.gcn_run(Xd, Y, scheduled=True))
    step("sched_gat", lambda: agg.gat_run(Xd, att, Y, scheduled=True))
    step("sddmm", lambda: agg.sddmm(Xd, Xd, torch.empty(m, device=cuda)))
    step("edge_softmax", lambda: agg.edge_softmax(att, torch.empty(m, device=cuda)))
    agg.close()

    ptr_d, idx_d, _, _ = large
    nl, ml = ptr_d.numel() - 1, idx_d.numel()
    XL = torch.randn((nl, 32), device=cuda)
    YL = torch.empty_like(XL)
    attl = torch.randn((nl, 2), device=cuda) * 0.5
    agg = gn.Aggregator(ptr_d, idx_d, synth.gcn_norm_val(ptr_d, idx_d))
    step("large_auto_merge", lambda: agg.gcn_run(XL, YL))
    step("large_second", lambda: agg.gcn_run(XL, YL))
    step("large_transpose_build", lambda: agg.transpose_build())
    step("large_gat_run", lambda: agg.gat_run(XL, attl, YL))
    step("large_gat_backward", lambda: agg.gat_backward(XL, attl, YL, XL, torch.empty_like(XL),
                                                        torch.empty((nl, 2), device=cuda)))
    step("large_gcn_backward", lambda: agg.gcn_backward(XL, torch.empty_like(XL)))
    agg.close()
    torch.cuda.synchronize()
    assert ml >= 4_000_000
    return out


def test_launch_counts(gn, cuda, small, large):
    got = launch_script(gn, cuda, small, large)
    assert got == EXPECTED_LAUNCHES


def test_locality_slices_follow_set_val_in_place(gn, orc, cuda, small):
    ptr, idx = small
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=2)
    dval, Xd = dev(val), dev(X)
    agg = gn.Aggregator(dev(ptr), dev(idx), dval)
    agg.set_locality_slices(3)
    agg.gcn_run(Xd, torch.empty((n, F), device=cuda))
    val2 = (val * 1.5 - 0.25).astype(np.float32)
    dval.copy_(torch.from_numpy(val2))  # same pointer, new contents
    agg.set_val(dval)
    Y = agg.gcn_run(Xd, torch.empty((n, F), device=cuda))
    y64, scale = orc.spmm_f64(ptr, idx, val2, X)
    assert rel_gate(Y.cpu().numpy(), y64, scale, TOL)[0] == 0
    fresh = gn.Aggregator(dev(ptr), dev(idx), dev(val2))
    fresh.set_locality_slices(3)
    assert torch.equal(Y, fresh.gcn_run(Xd, torch.empty_like(Y)))


def test_host_slices_follow_set_val_in_place(gn, orc, cuda, small):
    ptr, idx = small
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=3)
    dval = dev(val)
    agg = gn.Aggregator(dev(ptr), dev(idx), dval)
    agg.set_host_pipeline(2)
    hX = torch.from_numpy(X).pin_memory()
    agg.gcn_run_host(hX, torch.empty((n, F)).pin_memory())
    val2 = (val * 0.5 + 0.75).astype(np.float32)
    dval.copy_(torch.from_numpy(val2))
    agg.set_val(dval)
    hY = agg.gcn_run_host(hX, torch.empty((n, F)).pin_memory())
    y64, scale = orc.spmm_f64(ptr, idx, val2, X)
    assert rel_gate(hY.numpy(), y64, scale, TOL)[0] == 0
    fresh = gn.Aggregator(dev(ptr), dev(idx), dev(val2))
    fresh.set_host_pipeline(2)
    assert np.array_equal(hY.numpy(), fresh.gcn_run_host(hX, torch.empty((n, F)).pin_memory()).numpy())


def test_gcn_backward_after_large_gat_backward(gn, orc, cuda, large):
    """the large-graph GAT backward borrows the transposed edge values; the GCN backward that follows re-mirrors them
    without a gnnagg_set_val in between"""
    ptr_d, idx_d, ptr, idx = large
    n = ptr_d.numel() - 1
    val = synth.gcn_norm_val(ptr_d, idx_d)
    dY = torch.randn((n, 32), device=cuda)
    att = torch.randn((n, 2), device=cuda) * 0.5
    agg = gn.Aggregator(ptr_d, idx_d, val)
    agg.transpose_build()
    agg.gcn_backward(dY, torch.empty_like(dY))
    Y = agg.gat_run(dY, att, torch.empty_like(dY))
    agg.gat_backward(dY, att, Y, dY, torch.empty_like(dY), torch.empty((n, 2), device=cuda))
    dX = agg.gcn_backward(dY, torch.empty_like(dY))
    d64, scale = orc.spmm_t_f64(ptr, idx, val.cpu().numpy(), dY.cpu().numpy(), n)
    assert rel_gate(dX.cpu().numpy(), d64, scale, TOL)[0] == 0
    fresh = gn.Aggregator(ptr_d, idx_d, val)
    fresh.transpose_build()
    assert torch.equal(dX, fresh.gcn_backward(dY, torch.empty_like(dY)))


@pytest.mark.parametrize("mode", ["merge", "loc"])
def test_profile_brackets_reach_the_aggregator(gn, cuda, large, mode):
    """the aggregation kernel of the merged view and the loop over the locality slices are bracketed by the events
    gnnagg_profile_read reads; without the brackets `agg` would read about 0"""
    ptr_d, idx_d, _, _ = large
    n = ptr_d.numel() - 1
    agg = gn.Aggregator(ptr_d, idx_d, synth.gcn_norm_val(ptr_d, idx_d))
    if mode == "merge":
        agg.set_merge_duplicates(2)
    else:
        agg.set_locality_slices(3)
    agg.profile(True)
    X, Y = torch.randn((n, F), device=cuda), torch.empty((n, F), device=cuda)
    agg.gcn_run(X, Y)
    agg.gcn_run(X, Y)
    ms = agg.profile_read()
    assert ms["agg"] >= 0.5 * (ms["agg"] + ms["agg_rest"]), ms


def test_rebuild_derived_structures(gn, orc, cuda, small):
    ptr, idx = small
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=4)
    Xd = dev(X)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    y64, scale = orc.spmm_f64(ptr, idx, val, X)
    t64, tscale = orc.spmm_t_f64(ptr, idx, val, X, n)

    def check(Y, want=y64, s=scale):
        assert rel_gate(Y.cpu().numpy(), want, s, TOL)[0] == 0

    for _ in range(2):
        agg.transpose_build()
        check(agg.gcn_backward(Xd, torch.empty((n, F), device=cuda)), t64, tscale)
    for slices in (3, 2):
        agg.set_locality_slices(slices)
        check(agg.gcn_run(Xd, torch.empty((n, F), device=cuda)))
    agg.set_locality_slices(1)
    for kind, params in ((1, [16]), (0, [4])):
        agg.schedule(kind, params)
        check(agg.gcn_run(Xd, torch.empty((n, F), device=cuda), scheduled=True))
    for mode in (2, 1, 2):
        agg.set_merge_duplicates(mode)
        check(agg.gcn_run(Xd, torch.empty((n, F), device=cuda)))
    torch.cuda.synchronize()
    assert gn.lib().gnnagg_destroy(agg.h) == 0
    agg.h = None
