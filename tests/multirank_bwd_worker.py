"""torchrun worker of tests/test_gpu_dist_backward.py::test_multi_process_backward (also runnable by hand:
`torchrun --nproc-per-node N tests/multirank_bwd_worker.py`).  Every rank builds the SAME down-scaled R-MAT graph (scale
20 by default, F = 64), keeps its row block and runs the multi-GPU backward for several remote-stage settings.  Checked:
  * dX equals the single-GPU gnnagg_gcn_backward within 2e-5 * sum|terms| (both lie within 1e-5 of the exact sum);
  * a second backward step with the same dY repeats the first bit for bit;
  * a two-layer model relu(agg(X) @ W1) -> agg(H1) @ W2 through partition.dist_gcn_aggregate gives X.grad, W1.grad and
    W2.grad within 1e-5 (relative, in norm) of the same model on one GPU through plugin.gcn_aggregate.
Prints one JSON line per setting on rank 0."""
import json
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gnn-computing_b200"))


def _model(agg, X, W1, W2, R):
    """loss of the two-layer model; agg(T, buf) is the aggregation"""
    H1 = torch.relu(agg(X, 0) @ W1)
    return ((agg(H1, 1) @ W2) * R).sum()


def main():
    from gnnagg import Aggregator, partition, plugin, synth
    from gnnagg.partition import PeerHalo

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda:%d" % local)
    dist.init_process_group("nccl", device_id=dev)
    scale = int(os.environ.get("GNNAGG_MR_SCALE", "20"))
    n, m, F = 1 << scale, 1 << (scale + 4), 64
    ptr, idx = synth.rmat_csr(n, m, seed=123, device=dev)          # identical on every rank
    val = synth.gcn_norm_val(ptr, idx)
    g = torch.Generator(device=dev).manual_seed(7)
    X = torch.randn((n, F), device=dev, generator=g)
    dY = torch.randn((n, F), device=dev, generator=g)
    R = torch.randn((n, F), device=dev, generator=g)
    W1 = torch.randn((F, F), device=dev, generator=g) / 8
    W2 = torch.randn((F, F), device=dev, generator=g) / 8
    hp = ptr.cpu().numpy()
    bounds = [int(b) for b in partition.split_rows(hp, world, "edges")]
    r0, r1 = bounds[rank], bounds[rank + 1]
    e0, e1 = int(hp[r0]), int(hp[r1])
    lptr = (ptr[r0:r1 + 1] - e0).contiguous()
    lidx, lval = idx[e0:e1].contiguous(), val[e0:e1].contiguous()

    # one GPU: dX, the gate's sum|terms| and the autograd gradients of the whole graph (every rank computes them)
    agg = Aggregator(ptr, idx, val)
    agg.transpose_build()
    dX1 = agg.gcn_backward(dY, torch.empty((n, F), device=dev))
    agg_abs = Aggregator(ptr, idx, val.abs())
    agg_abs.transpose_build()
    S = agg_abs.gcn_backward(dY.abs(), torch.empty((n, F), device=dev))
    at = plugin.gcn_init(ptr, idx, val)
    ref = [t.clone().requires_grad_(True) for t in (X, W1, W2)]
    _model(lambda T, buf: plugin.gcn_aggregate(at, T), ref[0], ref[1], ref[2], R).backward()
    ref = [t.grad for t in ref]
    plugin.destroy(at)

    for stages in sorted({-4, 0, 1, world - 1}):
        ph = PeerHalo(lptr, lidx, lval, bounds, rank, world, F, remote_stages=stages, backward=True)
        dXa = torch.empty((r1 - r0, F), device=dev)
        dXb = torch.empty_like(dXa)
        ph.gcn_backward(dY[r0:r1].contiguous(), dXa)
        ph.gcn_backward(dY[r0:r1].contiguous(), dXb)
        torch.cuda.synchronize()
        ph.check()
        same = int(torch.equal(dXa, dXb))
        worst = float(((dXa - dX1[r0:r1]).abs() / (2e-5 * S[r0:r1] + 1e-30)).max()) if r1 > r0 else 0.0
        # the same model across ranks: X is this rank's shard, W1 / W2 replicated, their gradients summed over ranks
        mine = [X[r0:r1].clone().requires_grad_(True), W1.clone().requires_grad_(True), W2.clone().requires_grad_(True)]
        _model(lambda T, buf: partition.dist_gcn_aggregate(ph, T, buf), mine[0], mine[1], mine[2], R[r0:r1]).backward()
        torch.cuda.synchronize()
        ph.check()
        dW = torch.stack([mine[1].grad, mine[2].grad])
        dist.all_reduce(dW)
        # squared norms of the differences and of the references: X.grad shard by shard, summed over ranks
        sums = torch.stack([((mine[0].grad - ref[0][r0:r1]).double() ** 2).sum(), (ref[0][r0:r1].double() ** 2).sum()])
        dist.all_reduce(sums)
        rel = [float((sums[0] / sums[1]).sqrt())] + [float((dW[k] - ref[1 + k]).norm() / ref[1 + k].norm()) for k in range(2)]
        stats = torch.tensor([worst, max(rel), float(1 - same)], device=dev, dtype=torch.float64)
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        if rank == 0:
            line = {"test": "multirank_backward", "world": world, "remote_stages": stages, "graph": "rmat%d" % scale, "n": n,
                    "m": m, "F": F, "worst_err_over_gate_vs_one_gpu": round(float(stats[0]), 4),
                    "bit_reproducible": bool(stats[2] == 0), "autograd_worst_rel": float(stats[1])}
            line["ok"] = bool(stats[0] <= 1.0 and stats[2] == 0 and stats[1] <= 1e-5)
            print(json.dumps(line), flush=True)
        ph.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
