"""GPU tier: GCN aggregation from bf16 features (gnnagg_gcn_run_bf16, gnnagg_gcn_layer_bf16, gnnagg_gcn_backward_bf16).
X / dY are stored in bf16, edge values, sums and outputs stay fp32.  Every bf16 value widens exactly to fp32, so a bf16
run equals the fp32 entry point run on the widened X bit for bit (un-scheduled: CSR, merged view, locality slices), and
everything stays within the 1e-5 * sum|terms| gate of the fp64 oracle of the widened X."""
import numpy as np
import pytest
import torch

import gnnagg.plugin as gnc
from conftest import rel_gate
from gnnagg import synth
from gpu_util import GRAPHS, dev, make_graph, rand_inputs
from test_gpu_merge import dup_csr

pytestmark = pytest.mark.gpu
TOL = 1e-5


def bf16_pair(X):
    """(X_b, X_w): X rounded to bf16 on the device, and X_b widened back to fp32"""
    Xb = dev(X).to(torch.bfloat16)
    return Xb, Xb.float()


def same_bits(a, b):
    return a.dtype == b.dtype == torch.float32 and torch.equal(a.view(torch.int32), b.view(torch.int32))


def nan_like(n, F, cuda):
    return torch.full((n, F), float("nan"), device=cuda)


def check_run(agg, orc, ptr, idx, val, Xb, Xw, cuda, scheduled=False):
    """bf16 run against the fp32 run on X_w (bits) and the fp64 oracle of X_w (gate); returns the bf16 output"""
    n, F = len(ptr) - 1, Xb.shape[1]
    Yb = agg.gcn_run(Xb, nan_like(n, F, cuda), scheduled)
    Yw = agg.gcn_run(Xw, nan_like(n, F, cuda), scheduled)
    y64, scale = orc.spmm_f64(ptr, idx, val, Xw.cpu().numpy())
    bad, worst = rel_gate(Yb.cpu().numpy(), y64, scale, TOL)
    assert bad == 0, worst
    if not scheduled:
        assert same_bits(Yb, Yw)
    return Yb


@pytest.mark.parametrize("gname", list(GRAPHS))
@pytest.mark.parametrize("F", [32, 64, 128, 256])
@pytest.mark.parametrize("we", [128, 512])
def test_bf16_bit_identical_to_widened_fp32(gn, orc, cuda, gname, F, we):
    ptr, idx = make_graph(gname, seed=F)
    X, val = rand_inputs(len(ptr) - 1, len(idx), F, seed=1)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.set_warp_edges(we)
    Xb, Xw = bf16_pair(X)
    Yb = check_run(agg, orc, ptr, idx, val, Xb, Xw, cuda)
    assert same_bits(Yb, agg.gcn_run(Xb, torch.empty_like(Yb)))  # run to run


@pytest.mark.parametrize("F", [4, 20, 96, 160, 512, 1024])
def test_bf16_odd_feature_widths(gn, orc, cuda, F):
    ptr, idx = make_graph("medium", seed=3)
    X, val = rand_inputs(len(ptr) - 1, len(idx), F, seed=2)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    check_run(agg, orc, ptr, idx, val, *bf16_pair(X), cuda)


@pytest.mark.parametrize("route", ["merged", "slices"])
def test_bf16_routing_follows_settings_and_set_val(gn, orc, cuda, route):
    """the merged view (forced on, a graph with adjacent duplicate runs) and locality slices (forced to 4) run the bf16
    operand too, bit-identical to the fp32 run under the same setting; edge values rewritten in place reach both (the
    merged re-sum, the slice values)"""
    if route == "merged":
        ptr, idx = dup_csr()
    else:
        ptr, idx = synth.small_random_csr(4000, 9.0, 77, empty_frac=0.3, hub=30000)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, 64, seed=8)
    dval = dev(val)
    agg = gn.Aggregator(dev(ptr), dev(idx), dval)
    if route == "merged":
        agg.set_merge_duplicates(2)
        assert agg.merged_edges < m
    else:
        agg.set_locality_slices(4)
    Xb, Xw = bf16_pair(X)
    check_run(agg, orc, ptr, idx, val, Xb, Xw, cuda)
    val2 = (val * 1.5 - 0.25).astype(np.float32)
    dval.copy_(torch.from_numpy(val2))
    agg.set_val(dval)
    Yb = agg.gcn_run(Xb, nan_like(n, 64, cuda))  # the bf16 run is the first after the rewrite
    y64, scale = orc.spmm_f64(ptr, idx, val2, Xw.cpu().numpy())
    assert rel_gate(Yb.cpu().numpy(), y64, scale, TOL)[0] == 0
    assert same_bits(Yb, agg.gcn_run(Xw, nan_like(n, 64, cuda)))
    if route == "merged":
        agg.set_merge_duplicates(1)  # and back on the CSR
        assert same_bits(agg.gcn_run(Xb, nan_like(n, 64, cuda)), agg.gcn_run(Xw, nan_like(n, 64, cuda)))


@pytest.mark.parametrize("kind,params", [(1, [16]), (0, [4]), (2, [4, 32])])
@pytest.mark.parametrize("F", [32, 256])
def test_bf16_scheduled(gn, orc, cuda, kind, params, F):
    """scheduled runs combine with RED.ADD in arbitrary order: within the oracle gate"""
    ptr, idx = make_graph("hub", seed=kind * 10 + F)
    X, val = rand_inputs(len(ptr) - 1, len(idx), F, seed=5)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.schedule(kind, params)
    check_run(agg, orc, ptr, idx, val, *bf16_pair(X), cuda, scheduled=True)


@pytest.mark.parametrize("F,Fo", [(32, 64), (64, 32), (128, 128), (256, 64), (20, 12)])
def test_bf16_layer(gn, orc, cuda, F, Fo):
    """H and AX bit-identical to gcn_layer on X_w: tensor-core widths and a width that takes the fp32 fallback"""
    ptr, idx = make_graph("hub", seed=F)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, F, seed=3)
    W = (np.random.default_rng(F).standard_normal((F, Fo)) / np.sqrt(F)).astype(np.float32)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    Xb, Xw = bf16_pair(X)
    Hb, AXb = nan_like(n, Fo, cuda), nan_like(n, F, cuda)
    agg.gcn_layer(Xb, dev(W), Hb, AXb)
    Hw, AXw = nan_like(n, Fo, cuda), nan_like(n, F, cuda)
    agg.gcn_layer(Xw, dev(W), Hw, AXw)
    assert same_bits(AXb, AXw) and same_bits(Hb, Hw)
    assert same_bits(agg.gcn_layer(Xb, dev(W), nan_like(n, Fo, cuda)), Hw)  # AX in the library's scratch
    _, h64, hs = orc.gcn_layer_f64(ptr, idx, val, Xw.cpu().numpy(), W)
    assert rel_gate(Hb.cpu().numpy(), h64, hs, TOL)[0] == 0


@pytest.mark.parametrize("gname", ["hub", "bighub", "short_rows"])
@pytest.mark.parametrize("F", [32, 128])
def test_bf16_backward(gn, orc, cuda, gname, F):
    ptr, idx = make_graph(gname, seed=4)
    n, m = len(ptr) - 1, len(idx)
    dY, val = rand_inputs(n, m, F, seed=6)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.transpose_build()
    dYb, dYw = bf16_pair(dY)
    dXb = agg.gcn_backward(dYb, nan_like(n, F, cuda))
    assert same_bits(dXb, agg.gcn_backward(dYw, nan_like(n, F, cuda)))
    d64, scale = orc.spmm_t_f64(ptr, idx, val, dYw.cpu().numpy(), n)
    assert rel_gate(dXb.cpu().numpy(), d64, scale, TOL)[0] == 0


def test_bf16_autograd(gn, cuda):
    """plugin.gcn_aggregate on a bf16 leaf: fp32 Y equal to the fp32 path, bf16 X.grad = (A^T dY) rounded once"""
    ptr, idx = make_graph("hub", seed=2)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, 64, seed=9)
    at = gnc.gcn_init(dev(ptr), dev(idx), dev(val))
    try:
        Xb, Xw = bf16_pair(X)
        Xb.requires_grad_(True)
        Y = gnc.gcn_aggregate(at, Xb)
        assert Y.dtype == torch.float32
        assert same_bits(Y.detach(), gnc.gcn_aggregate(at, Xw))
        dY = torch.randn((n, 64), device=cuda)
        Y.backward(dY)
        assert Xb.grad.dtype == torch.bfloat16
        agg = gnc._get(at)
        want = agg.gcn_backward(dY, torch.empty((n, 64), device=cuda)).to(torch.bfloat16)
        assert torch.equal(Xb.grad.view(torch.int16), want.view(torch.int16))
        # an fp32 leaf keeps the fp32 gradient
        Xf = Xw.clone().requires_grad_(True)
        gnc.gcn_aggregate(at, Xf).backward(dY)
        assert same_bits(Xf.grad, agg.gcn_backward(dY, torch.empty((n, 64), device=cuda)))
    finally:
        gnc.destroy(at)


def test_bf16_launches_profile_and_graph_capture(gn, cuda):
    """each bf16 call launches as many kernels as its fp32 twin and reaches gnnagg_profile_read; after
    gnnagg_prepare a bf16 run can be captured in a CUDA graph"""
    ptr, idx = make_graph("bighub", seed=1)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, 128, seed=4)
    W = (np.random.default_rng(0).standard_normal((128, 64)) / 12).astype(np.float32)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    agg.transpose_build()
    agg.profile(True)
    Xb, Xw = bf16_pair(X)
    Y, H, dX = torch.empty((n, 128), device=cuda), torch.empty((n, 64), device=cuda), torch.empty((n, 128), device=cuda)
    calls = {
        "run": lambda x: agg.gcn_run(x, Y),
        "layer": lambda x: agg.gcn_layer(x, dev(W), H),
        "backward": lambda x: agg.gcn_backward(x, dX),
    }
    for name, call in calls.items():
        call(Xw)  # one-time tables of this width
        counts = []
        for x in (Xw, Xb):
            before = agg.launches
            call(x)
            counts.append(agg.launches - before)
            if name != "backward":
                assert agg.profile_read()["agg"] > 0, name
        assert counts[0] == counts[1] > 0, (name, counts)
    ref = Y.clone()
    # a fresh aggregator: gnnagg_prepare builds this width's tables, so the captured run never waits on the host
    agg2 = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    gn.check(gn.lib().gnnagg_prepare(agg2.h, 128, None))
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            agg2.gcn_run(Xb, Y)
    Y.fill_(float("nan"))
    graph.replay()
    torch.cuda.synchronize()
    assert same_bits(Y, ref)


def test_bf16_errors(gn, cuda):
    """rejected before anything is launched"""
    ptr, idx = make_graph("medium", seed=1)
    n, m = len(ptr) - 1, len(idx)
    X, val = rand_inputs(n, m, 32, seed=1)
    agg = gn.Aggregator(dev(ptr), dev(idx), dev(val))
    Xb, _ = bf16_pair(X)
    agg.gcn_run(Xb, torch.empty((n, 32), device=cuda))
    torch.cuda.synchronize()
    before = agg.launches
    with pytest.raises(gn.GnnaggError, match="multiple of 4"):
        agg.gcn_run(torch.ones((n, 30), device=cuda, dtype=torch.bfloat16), torch.empty((n, 30), device=cuda))
    buf = torch.zeros(n * 32 + 1, device=cuda, dtype=torch.bfloat16)
    with pytest.raises(gn.GnnaggError, match="8-byte aligned"):
        agg.gcn_run(buf[1:].view(n, 32), torch.empty((n, 32), device=cuda))  # 2 bytes off
    with pytest.raises(gn.GnnaggError, match="schedule"):
        agg.gcn_run(Xb, torch.empty((n, 32), device=cuda), scheduled=True)
    with pytest.raises(gn.GnnaggError, match="transpose_build"):
        agg.gcn_backward(Xb, torch.empty((n, 32), device=cuda))
    for dt in (torch.float16, torch.float64):
        with pytest.raises(gn.GnnaggError):
            agg.gcn_run(Xb.to(dt), torch.empty((n, 32), device=cuda))
        with pytest.raises(gn.GnnaggError):
            agg.gcn_layer(Xb.to(dt), torch.ones((32, 32), device=cuda), torch.empty((n, 32), device=cuda))
    with pytest.raises(gn.GnnaggError):
        agg.gcn_run(Xb, torch.empty((n, 32), device=cuda, dtype=torch.bfloat16))  # outputs stay fp32
    with pytest.raises(gn.GnnaggError):
        agg.gat_run(Xb, torch.zeros((n, 2), device=cuda), torch.empty((n, 32), device=cuda))  # GAT keeps fp32
    assert agg.launches == before
