"""plugin.py -- the reference's PyTorch extension surface (Figure7/kernel.cpp:37-179, module
`gnncompile` in Figure7/our.py:15-22) on top of the C ABI.

Same function names, argument order and meaning; handles are plain ints like the reference's
`int64_t` (there: a heap `Aggregator*`, never destroyed; here: a key into a registry, `destroy(at)` is
an addition).  `blocksize` is accepted and ignored.  Launches go to torch's CURRENT stream (the
reference uses the legacy default stream, which is torch's default current stream).

    import gnnagg.plugin as gnc
    ptrs, idxs = gnc.new_load(dset, "_thres_0.2", 0)
    at = gnc.gcn_init(ptrs, idxs, vals); gnc.gcn_schedule(at, 32)
    gnc.gcn_run(at, feat2, output_feat, 128, 1)
"""
import itertools

import torch

from . import Aggregator, GnnaggError, SCHED_NEIGHBOR_GROUPING, load_graph

_registry = {}
_ids = itertools.count(1)
n = -1  # the reference publishes the loaded sizes as globals (kernel.cpp:52-53)
m = -1
datadir = "../data/"  # load_graph hard-codes this relative path (src/data.cu:34)


def _get(at):
    try:
        return _registry[int(at)]
    except KeyError:
        raise GnnaggError("unknown aggregator handle %r" % (at,))


def _check(*tensors):
    for t in tensors:  # CHECK_INPUT of kernel.cpp:71-75
        if not t.is_cuda:
            raise GnnaggError("tensor must be a CUDA tensor")
        if not t.is_contiguous():
            raise GnnaggError("tensor must be contiguous")


def new_load(dset, reorder="", devid=0):
    """kernel.cpp:37-67: load_graph on the host (with optional .reorder<suffix>), two int32 CUDA tensors"""
    global n, m
    ptr, idx, _, _ = load_graph(dset, datadir, reorder)
    n, m = len(ptr) - 1, len(idx)
    dev = torch.device("cuda", devid)
    return [torch.from_numpy(ptr).to(dev), torch.from_numpy(idx).to(dev)]


def gcn_init(ptrs, idxs, val):
    _check(ptrs, idxs, val)
    at = next(_ids)
    _registry[at] = Aggregator(ptrs, idxs, val)
    return at


def gcn_update_val(at, val):
    _check(val)
    _get(at).set_val(val)


def gcn_run(at, feat, outfeat, blocksize, scheduled):
    _check(feat, outfeat)
    _get(at).gcn_run(feat, outfeat, bool(scheduled))  # feature width = feat.size(1), kernel.cpp:100


def gcn_schedule(at, neighbor_num):
    _get(at).schedule(SCHED_NEIGHBOR_GROUPING, [int(neighbor_num)])


def gat_init(ptrs, idxs):
    _check(ptrs, idxs)
    at = next(_ids)
    _registry[at] = Aggregator(ptrs, idxs)
    return at


def gat_run(at, feat, att, outfeat, blocksize, scheduled):
    _check(feat, att, outfeat)
    _get(at).gat_run(feat, att, outfeat, 0.2, bool(scheduled))


def gat_run_u_add_v(at, att, outval, blocksize):
    _check(att, outval)
    _get(at).u_add_v(att, outval)


def gat_run_add_to_center(at, inval, outatt, blocksize):
    _check(inval, outatt)
    _get(at).add_to_center(inval, outatt)


def gat_run_div_each(at, inatt, inoutval, blocksize):
    _check(inatt, inoutval)
    _get(at).each_div(inatt, inoutval)


def gat_schedule(at, neighbor_num):
    _get(at).schedule(SCHED_NEIGHBOR_GROUPING, [int(neighbor_num)])


def destroy(at):
    _registry.pop(int(at)).close()


# ------------------------------------------------------------------------------------------------
# autograd: the aggregations as differentiable torch ops (the reference's our.py trains nothing -- it times forward
# passes, Figure7/our.py:247-290 -- but its kernel set includes an experimental backward, aggr_gat_fine_bwd,
# include/aggr_gat.h:222-294; these tie the forward entry points to gnnagg_gcn_backward / gnnagg_gat_backward).
# ------------------------------------------------------------------------------------------------
def _transposed(agg, num_src):
    if getattr(agg, "num_src", None) != num_src:
        agg.transpose_build(num_src)
    return agg


class GCNAggregate(torch.autograd.Function):
    """Y = A X for the aggregator `at` (edge values are constants of the graph).  backward: dX = A^T dY through the
    GPU-built transposed CSR (deterministic gather, no atomics).  X may be float32 or bfloat16; Y is float32.  dX is
    computed in float32 and rounded once to X's dtype."""

    @staticmethod
    def forward(ctx, at, X, scheduled=False):
        agg = _get(at)
        X = X.contiguous()
        _check(X)
        Y = torch.empty((agg.n, X.shape[1]), device=X.device, dtype=torch.float32)
        agg.gcn_run(X, Y, bool(scheduled))
        ctx.at, ctx.num_src, ctx.x_dtype = at, X.shape[0], X.dtype
        return Y

    @staticmethod
    def backward(ctx, dY):
        agg = _transposed(_get(ctx.at), ctx.num_src)
        dX = torch.empty((ctx.num_src, dY.shape[1]), device=dY.device, dtype=torch.float32)
        agg.gcn_backward(dY.contiguous(), dX)
        return None, dX.to(ctx.x_dtype), None


class GATAggregate(torch.autograd.Function):
    """Y = fused GAT aggregation of X with the attention table att [n, 2] (destination term, source term), slope 0.2
    as in the reference (aggr_gat.h:339).  backward: full gradient w.r.t. X and att.  X may be float32 or bfloat16: a
    bf16 X is gathered as stored (gnnagg_gat_run_bf16 / gnnagg_gat_backward_bf16) and kept for the backward at half
    the memory.  att may be float32 or bfloat16; it is widened to float32 once per forward.  Y is float32.  dX and
    datt are computed in float32 and rounded once to the dtypes of X and att."""

    @staticmethod
    def forward(ctx, at, X, att, slope=0.2):
        agg = _get(at)
        X, att = X.contiguous(), att.contiguous()
        _check(X, att)
        att32 = att.float() if att.dtype == torch.bfloat16 else att
        Y = torch.empty((agg.n, X.shape[1]), device=X.device, dtype=torch.float32)
        run = agg.gat_run_bf16 if X.dtype == torch.bfloat16 else agg.gat_run
        run(X, att32, Y, slope, False)
        ctx.at, ctx.slope, ctx.att_dtype = at, slope, att.dtype
        ctx.save_for_backward(X, att32, Y)
        return Y

    @staticmethod
    def backward(ctx, dY):
        X, att, Y = ctx.saved_tensors
        agg = _transposed(_get(ctx.at), X.shape[0])
        dX = torch.empty(X.shape, device=X.device, dtype=torch.float32)
        datt = torch.empty((max(agg.n, X.shape[0]), 2), device=X.device, dtype=torch.float32)
        backward = agg.gat_backward_bf16 if X.dtype == torch.bfloat16 else agg.gat_backward
        backward(X, att, Y, dY.contiguous(), dX, datt, ctx.slope)
        return None, dX.to(X.dtype), datt[: att.shape[0]].to(ctx.att_dtype), None


def gcn_aggregate(at, X, scheduled=False):
    return GCNAggregate.apply(at, X, scheduled)


def gat_aggregate(at, X, att, slope=0.2):
    return GATAggregate.apply(at, X, att, slope)
