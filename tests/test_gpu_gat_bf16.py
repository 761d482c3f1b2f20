"""GPU tier: GAT aggregation from bf16 features (gnnagg_gat_run_bf16, gnnagg_gat_backward_bf16) and plugin.gat_aggregate
on bf16 leaves.  X is stored in bf16; att, w, den, Y, dY and every output stay fp32.  Each bf16 value widens exactly to
fp32 and the walk keeps the lane mapping, items and carries of the fp32 run of the same width, so:
  * the un-scheduled forward and both routes of the backward equal the fp32 entry point on the widened X bit for bit;
  * the scheduled forward stays within the oracle gate (RED.ADD order), and its edge weights, which do not depend on X,
    equal the fp32 run's bit for bit.
Every output is prefilled with NaN and checked finite.  The forward and backward matrices run every bf16 instance of
agg_kernel (GAT: 2 SCHED x 2 WE x 4 (LPR, NV); pass 1 of the backward: 2 WE x 4) with partial column chunks and
multi-pass widths; test_gat_bf16_matrix_reaches_every_instance (CPU tier) fails when the parametrization stops doing so."""
import numpy as np
import pytest
import torch

import gnnagg.plugin as gnc
from conftest import rel_gate
from gnnagg import synth
from gpu_util import dev, make_graph, rand_inputs
from test_gpu_mode_matrix import (EDGE_GRAPHS, INSTANCES, ITEM_SIZES, SCHEDULES, TOL_A, TOL_GAT, TOL_X, _cases, _edge_weights,
                                  _params, chunk_for, lanes_for, vectors_for)

gpu = pytest.mark.gpu

FWD_WIDTHS = [4, 20, 36, 100, 160, 260, 512, 1024]
SCHED_WIDTHS = [20, 36, 100, 160, 260, 512]
BWD_WIDTHS = [4, 20, 36, 100, 160, 260, 512, 1024]
BWD_LARGE_WIDTHS = [32, 160]  # 4.2M edges: 512-edge items chosen automatically, pass 2 as permute + row sum + GCN


# ---------------------------------------------------------------- helpers
def _nan(*shape):
    return torch.full(shape, float("nan"), device="cuda:0")


def _att(n, seed):
    return np.random.default_rng(seed).standard_normal((n, 2)).astype(np.float32)


def bf16_pair(X):
    """(X_b, X_w): X rounded to bf16 on the device, and X_b widened back to fp32"""
    Xb = dev(X).to(torch.bfloat16)
    return Xb, Xb.float()


def same_bits(a, b):
    return a.dtype == b.dtype == torch.float32 and torch.equal(a.view(torch.int32), b.view(torch.int32))


def finite(*ts):
    return all(bool(torch.isfinite(t).all()) for t in ts)


def check_backward(agg, orc, ptr, idx, att, Xb, Xw, Y, dY, slope=0.2, w=None, den=None, label=()):
    """gat_backward_bf16 against gat_backward on X_w (bits), the fp64 oracle of X_w (gate) and itself (run to run)"""
    num_src, F = Xb.shape
    rows = att.shape[0]
    attd = None if w is not None else dev(att)
    dYd = dev(dY)

    def run(fn, X):
        return fn(X, attd, Y, dYd, _nan(num_src, F), _nan(rows, 2), slope=slope, w=w, den=den)

    dXb, dAb = run(agg.gat_backward_bf16, Xb)
    dXw, dAw = run(agg.gat_backward, Xw)
    assert finite(dXb, dAb), label
    assert same_bits(dXb, dXw) and same_bits(dAb, dAw), label
    x64, a64, sx, sa = orc.gat_backward_f64(ptr, idx, att, Xw.cpu().numpy(), dY, slope)
    bad, worst = rel_gate(dXb.cpu().numpy(), x64, sx, TOL_X)
    assert bad == 0, ("dX",) + label + (worst,)
    bad, worst = rel_gate(dAb.cpu().numpy(), a64, sa, TOL_A)
    assert bad == 0, ("datt",) + label + (worst,)
    dXb2, dAb2 = run(agg.gat_backward_bf16, Xb)
    assert same_bits(dXb, dXb2) and same_bits(dAb, dAb2), label


# ---------------------------------------------------------------- forward
@gpu
@_cases("gname,F,we", [EDGE_GRAPHS, FWD_WIDTHS, ITEM_SIZES])
def test_gat_bf16_unscheduled(gn, orc, cuda, gname, F, we):
    ptr, idx = make_graph(gname, seed=F + we)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 21)
    att = _att(n, F + 22)
    attd = dev(att)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    Yb = agg.gat_run_bf16(Xb, attd, _nan(n, F))
    assert finite(Yb)
    assert same_bits(Yb, agg.gat_run(Xw, attd, _nan(n, F)))
    y64, _, scale = orc.gat_f64(ptr, idx, att, Xw.cpu().numpy())
    bad, worst = rel_gate(Yb.cpu().numpy(), y64, scale, TOL_GAT)
    assert bad == 0, (gname, F, we, worst)
    assert same_bits(Yb, agg.gat_run_bf16(Xb, attd, _nan(n, F)))


@gpu
@_cases("sched,F,we", [SCHEDULES, SCHED_WIDTHS, ITEM_SIZES])
def test_gat_bf16_scheduled(gn, orc, cuda, sched, F, we):
    kind, params = sched
    ptr, idx = make_graph("hub", seed=F + kind)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 23)
    att = _att(n, F + 24)
    attd = dev(att)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    agg.schedule(kind, params)
    Yb = agg.gat_run_bf16(Xb, attd, _nan(n, F), scheduled=True)
    wb = _edge_weights(gn, agg, m)
    assert finite(Yb)
    y64, _, scale = orc.gat_f64(ptr, idx, att, Xw.cpu().numpy())
    bad, worst = rel_gate(Yb.cpu().numpy(), y64, scale, TOL_GAT)
    assert bad == 0, (sched, F, we, worst)
    agg.gat_run(Xw, attd, _nan(n, F), scheduled=True)
    assert np.array_equal(wb.view(np.int32), _edge_weights(gn, agg, m).view(np.int32))


# ---------------------------------------------------------------- backward
@gpu
@_cases("gname,F,we", [EDGE_GRAPHS, BWD_WIDTHS, ITEM_SIZES])
def test_gat_bf16_backward(gn, orc, cuda, gname, F, we):
    ptr, idx = make_graph(gname, seed=F + we + 1)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, F, seed=F + 25)
    dY, _ = rand_inputs(n, m, F, seed=F + 26)
    att = _att(n, F + 27)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.set_warp_edges(we)
    agg.transpose_build()
    Y = agg.gat_run(Xw, dev(att), _nan(n, F))
    check_backward(agg, orc, ptr, idx, att, Xb, Xw, Y, dY, label=(gname, F, we))


@gpu
@pytest.mark.parametrize("F", BWD_LARGE_WIDTHS)
def test_gat_bf16_backward_large_graph(gn, orc, cuda, F):
    """4.2M edges: the 512-edge kernels, and pass 2 as permute + row sum + the plain aggregation of dY (fp32)"""
    n, m = 150000, 4200000
    ptr_d, idx_d = synth.rmat_csr(n, m, seed=323, device=cuda)
    ptr, idx = ptr_d.cpu().numpy(), idx_d.cpu().numpy()
    X, _ = rand_inputs(n, 1, F, seed=F + 28)
    dY, _ = rand_inputs(n, 1, F, seed=F + 29)
    att = _att(n, F + 30)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(ptr_d, idx_d)
    agg.transpose_build()
    Yb = agg.gat_run_bf16(Xb, dev(att), _nan(n, F))
    Y = agg.gat_run(Xw, dev(att), _nan(n, F))
    assert finite(Yb) and same_bits(Yb, Y)
    check_backward(agg, orc, ptr, idx, att, Xb, Xw, Y, dY, label=(F,))


@gpu
@pytest.mark.parametrize("slope", [0.2, 0.0, 1.0])
def test_gat_bf16_backward_from_weights_and_rectangular(gn, orc, cuda, slope):
    """a rectangular block (num_src != num_v), the att convention and the (w, den) / (w, den=None) conventions"""
    n, num_src, F = 400, 1000, 64
    ptr, idx = synth.small_random_csr(n, 9.0, 4, empty_frac=0.1, hub=3000, num_src=num_src)
    ptr, idx = ptr.astype(np.int32), idx.astype(np.int32)
    rng = np.random.default_rng(16)
    X = rng.standard_normal((num_src, F)).astype(np.float32)
    dY = rng.standard_normal((n, F)).astype(np.float32)
    att = _att(num_src, 17)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.transpose_build(num_src)
    Yb = agg.gat_run_bf16(Xb, dev(att), _nan(n, F), slope=slope)
    Y = agg.gat_run(Xw, dev(att), _nan(n, F), slope=slope)
    assert finite(Yb) and same_bits(Yb, Y)
    check_backward(agg, orc, ptr, idx, att, Xb, Xw, Y, dY, slope=slope, label=("att", slope))
    w = dev(orc.edge_weight_f64(ptr, idx, att, slope))
    den = agg.add_to_center(w, torch.empty(n, device=cuda))
    check_backward(agg, orc, ptr, idx, att, Xb, Xw, Y, dY, slope=slope, w=w, den=den, label=("w, den", slope))
    check_backward(agg, orc, ptr, idx, att, Xb, Xw, Y, dY, slope=slope, w=w, label=("w", slope))


# ---------------------------------------------------------------- autograd
def _grads(at, X, att, dY):
    """(Y, X.grad, att.grad) of gat_aggregate on fresh leaves made from X and att"""
    X = X.detach().clone().requires_grad_(True)
    att = att.detach().clone().requires_grad_(True)
    Y = gnc.gat_aggregate(at, X, att)
    Y.backward(dY)
    return Y.detach(), X.grad, att.grad


@gpu
def test_gat_bf16_autograd(gn, cuda):
    """a bf16 leaf X: fp32 Y equal to the fp32 path on the widened X, X.grad in bf16 = the fp32 dX rounded once, att.grad
    equal to the fp32 path's; a bf16 att: att.grad in bf16 = the fp32 path's rounded once; an fp32 leaf as before"""
    ptr, idx = make_graph("hub", seed=2)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, 64, seed=31)
    att = dev(_att(n, 32))
    dY = torch.randn((n, 64), device=cuda)
    at = gnc.gat_init(dev(ptr), dev(idx))
    try:
        Xb, Xw = bf16_pair(X)
        Y32, gX32, gA32 = _grads(at, Xw, att, dY)
        Yb, gXb, gAb = _grads(at, Xb, att, dY)
        assert Yb.dtype == torch.float32 and same_bits(Yb, Y32)
        assert gXb.dtype == torch.bfloat16 and torch.equal(gXb.view(torch.int16), gX32.to(torch.bfloat16).view(torch.int16))
        assert same_bits(gAb, gA32)
        # bf16 att: widened once in the forward, its gradient rounded once
        attb = att.to(torch.bfloat16)
        Y32a, gX32a, gA32a = _grads(at, Xw, attb.float(), dY)
        Yba, gXba, gAba = _grads(at, Xb, attb, dY)
        assert same_bits(Yba, Y32a)
        assert torch.equal(gXba.view(torch.int16), gX32a.to(torch.bfloat16).view(torch.int16))
        assert gAba.dtype == torch.bfloat16 and torch.equal(gAba.view(torch.int16), gA32a.to(torch.bfloat16).view(torch.int16))
        # an fp32 leaf: the library's fp32 calls, unchanged
        agg = gnc._get(at)
        Yd = agg.gat_run(Xw, att, _nan(n, 64))
        dX, dA = agg.gat_backward(Xw, att, Yd, dY, _nan(n, 64), _nan(n, 2))
        assert same_bits(Y32, Yd) and same_bits(gX32, dX) and same_bits(gA32, dA)
    finally:
        gnc.destroy(at)


@gpu
def test_gat_bf16_autocast(gn, cuda):
    """under torch.autocast(bf16), Linear layers produce a bf16 X and a bf16 att that feed gat_aggregate: Y equals the
    fp32 aggregation of their widened values bit for bit, and both Linear weights receive finite gradients"""
    ptr, idx = make_graph("hub", seed=5)
    n, F = len(ptr) - 1, 64
    torch.manual_seed(0)
    lin_x, lin_a = torch.nn.Linear(32, F).to(cuda), torch.nn.Linear(32, 2).to(cuda)
    H = torch.randn((n, 32), device=cuda)
    at = gnc.gat_init(dev(ptr), dev(idx))
    try:
        with torch.autocast("cuda", dtype=torch.bfloat16):
            X, att = lin_x(H), lin_a(H)
            assert X.dtype == att.dtype == torch.bfloat16
            Y = gnc.gat_aggregate(at, X, att)
        assert Y.dtype == torch.float32
        assert same_bits(Y.detach(), gnc.gat_aggregate(at, X.detach().float(), att.detach().float()))
        (Y * torch.randn_like(Y)).sum().backward()
        for lin in (lin_x, lin_a):
            assert lin.weight.grad is not None and finite(lin.weight.grad) and bool(lin.weight.grad.abs().sum() > 0)
    finally:
        gnc.destroy(at)


# ---------------------------------------------------------------- launches, profiling, CUDA graphs, errors
@gpu
def test_gat_bf16_launches_profile_and_graph_capture(gn, cuda):
    """each bf16 call launches as many kernels as its fp32 twin; gat_run_bf16 reaches gnnagg_profile_read; after a
    first call both bf16 entry points can be captured in a CUDA graph and replay bit-identically"""
    ptr, idx = make_graph("bighub", seed=1)
    n, m = len(ptr) - 1, len(idx)
    F = 128
    X, _ = rand_inputs(n, m, F, seed=33)
    att = dev(_att(n, 34))
    dY = torch.randn((n, F), device=cuda)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    agg.transpose_build()
    agg.profile(True)
    Y, dX, dA = torch.empty((n, F), device=cuda), torch.empty((n, F), device=cuda), torch.empty((n, 2), device=cuda)
    calls = {
        "run": (lambda x: agg.gat_run(x, att, Y), lambda x: agg.gat_run_bf16(x, att, Y)),
        "scheduled": (lambda x: agg.gat_run(x, att, Y, scheduled=True), lambda x: agg.gat_run_bf16(x, att, Y, scheduled=True)),
        "backward": (lambda x: agg.gat_backward(x, att, Y, dY, dX, dA), lambda x: agg.gat_backward_bf16(x, att, Y, dY, dX, dA)),
    }
    for name, (fp32, bf16) in calls.items():
        if name == "scheduled":
            agg.schedule(1, [16])
        fp32(Xw)  # one-time tables of this width
        counts = []
        for call, x in ((fp32, Xw), (bf16, Xb)):
            before = agg.launches
            call(x)
            counts.append(agg.launches - before)
            if name != "backward":
                assert agg.profile_read()["agg"] > 0, name
        assert counts[0] == counts[1] > 0, (name, counts)

    agg2 = gn.Aggregator(dev(ptr), dev(idx))
    agg2.transpose_build()
    Y2, dX2, dA2 = _nan(n, F), _nan(n, F), _nan(n, 2)
    agg2.gat_run_bf16(Xb, att, Y2)
    agg2.gat_backward_bf16(Xb, att, Y2, dY, dX2, dA2)
    torch.cuda.synchronize()
    ref = [t.clone() for t in (Y2, dX2, dA2)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            agg2.gat_run_bf16(Xb, att, Y2)
            agg2.gat_backward_bf16(Xb, att, Y2, dY, dX2, dA2)
    for t in (Y2, dX2, dA2):
        t.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert all(same_bits(a, b) for a, b in zip((Y2, dX2, dA2), ref))


@gpu
def test_gat_bf16_errors(gn, cuda):
    """rejected before anything is launched: the launch count stays put and the outputs stay NaN"""
    ptr, idx = make_graph("medium", seed=1)
    n, m = len(ptr) - 1, len(idx)
    X, _ = rand_inputs(n, m, 32, seed=35)
    att = dev(_att(n, 36))
    dY = torch.randn((n, 32), device=cuda)
    Xb, Xw = bf16_pair(X)
    agg = gn.Aggregator(dev(ptr), dev(idx))
    Y = agg.gat_run_bf16(Xb, att, torch.empty((n, 32), device=cuda))
    torch.cuda.synchronize()
    before = agg.launches
    Yo, dX, dA = _nan(n, 32), _nan(n, 32), _nan(n, 2)
    with pytest.raises(gn.GnnaggError, match="transpose_build"):
        agg.gat_backward_bf16(Xb, att, Y, dY, dX, dA)
    assert agg.launches == before
    agg.transpose_build()
    agg.gat_backward_bf16(Xb, att, Y, dY, torch.empty((n, 32), device=cuda), torch.empty((n, 2), device=cuda))
    torch.cuda.synchronize()
    before = agg.launches
    X30 = torch.ones((n, 30), device=cuda, dtype=torch.bfloat16)
    with pytest.raises(gn.GnnaggError, match="multiple of 4"):
        agg.gat_run_bf16(X30, att, _nan(n, 30))
    with pytest.raises(gn.GnnaggError, match="multiple of 4"):
        agg.gat_backward_bf16(X30, att, _nan(n, 30), _nan(n, 30), _nan(n, 30), _nan(n, 2))
    buf = torch.zeros(n * 32 + 1, device=cuda, dtype=torch.bfloat16)
    off = buf[1:].view(n, 32)  # 2 bytes off
    with pytest.raises(gn.GnnaggError, match="8-byte aligned"):
        agg.gat_run_bf16(off, att, Yo)
    with pytest.raises(gn.GnnaggError, match="8-byte aligned"):
        agg.gat_backward_bf16(off, att, Y, dY, dX, dA)
    with pytest.raises(gn.GnnaggError, match="schedule"):
        agg.gat_run_bf16(Xb, att, Yo, scheduled=True)
    for dt in (torch.float16, torch.float64):
        with pytest.raises(gn.GnnaggError):
            agg.gat_run_bf16(Xb.to(dt), att, Yo)
        with pytest.raises(gn.GnnaggError):
            agg.gat_backward_bf16(Xb.to(dt), att, Y, dY, dX, dA)
    bf = lambda t: t.to(torch.bfloat16)  # noqa: E731
    with pytest.raises(gn.GnnaggError):
        agg.gat_run_bf16(Xb, att, bf(Yo))
    with pytest.raises(gn.GnnaggError):
        agg.gat_run_bf16(Xb, bf(att), Yo)
    for args in ((bf(att), Y, dY, dX, dA), (att, bf(Y), dY, dX, dA), (att, Y, bf(dY), dX, dA), (att, Y, dY, bf(dX), dA),
                 (att, Y, dY, dX, bf(dA))):
        with pytest.raises(gn.GnnaggError):
            agg.gat_backward_bf16(Xb, *args)
    with pytest.raises(gn.GnnaggError, match="att or w"):
        agg.gat_backward_bf16(Xb, None, Y, dY, dX, dA)
    torch.cuda.synchronize()
    assert agg.launches == before
    assert bool(torch.isnan(Yo).all() and torch.isnan(dX).all() and torch.isnan(dA).all())


# ---------------------------------------------------------------- the matrix reaches every bf16 instance (CPU tier)
def _reached(mode):
    """(F, WE, scheduled) of every case that runs the bf16 instances of `mode`"""
    if mode == "GAT":
        return ([(p["F"], p["we"], False) for p in _params(test_gat_bf16_unscheduled)] +
                [(p["F"], p["we"], True) for p in _params(test_gat_bf16_scheduled)])
    # pass 1 of the backward; graphs of 4.2M edges take 512-edge items
    return ([(p["F"], p["we"], False) for p in _params(test_gat_bf16_backward)] +
            [(F, 512, False) for F in BWD_LARGE_WIDTHS])


@pytest.mark.parametrize("mode", ["GAT", "GATBWD"])
def test_gat_bf16_matrix_reaches_every_instance(mode):
    cases = _reached(mode)
    for sched in sorted({s for _, _, s in cases}):
        widths = {(F, we) for F, we, s in cases if s == sched}
        assert {(lanes_for(F), vectors_for(F), we) for F, we in widths} == INSTANCES, (mode, sched)
        for lpr, nv in {(lanes_for(F), vectors_for(F)) for F, _ in widths}:
            assert any(F % chunk_for(F) and (lanes_for(F), vectors_for(F)) == (lpr, nv) for F, _ in widths), \
                (mode, sched, "no partial chunk for", (lpr, nv))
        assert any(F > chunk_for(F) for F, _ in widths), (mode, sched, "no multi-pass width")
    assert {s for _, _, s in cases} == ({False, True} if mode == "GAT" else {False}), mode
    if mode == "GAT":
        assert {p["sched"][0] for p in _params(test_gat_bf16_scheduled)} == {0, 1, 2}
    # 16 GAT + 8 GATBWD instances
    assert len({(lanes_for(F), vectors_for(F), we, s) for F, we, s in cases}) == (16 if mode == "GAT" else 8)
