"""torchrun worker of tests/test_gpu_dist_bf16.py::test_multi_process_bf16_equals_fp32 (also runnable by hand:
`torchrun --nproc-per-node N tests/multirank_bf16_worker.py`).  Every rank builds the SAME down-scaled R-MAT graph (scale
20 by default, F = 64), keeps its row block, writes its shard rounded to bf16 into shard buffer 0 and the widened fp32
shard into buffer 1, and runs the peer-memory step on both, for several remote-stage settings.  Checked:
  * the bf16 step equals the fp32 step on the widened X, bit for bit, on every rank (and so does the host-buffer form);
  * rank 0's first rows lie within the 1e-5 * sum|terms| gate of the fp64 oracle of the widened X.
Prints one JSON line per setting on rank 0."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "gnn-computing_b200"))


def main():
    from gnnagg import partition, synth
    from gnnagg.partition import PeerHalo

    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dev = torch.device("cuda:%d" % local)
    dist.init_process_group("nccl", device_id=dev)
    scale = int(os.environ.get("GNNAGG_MR_SCALE", "20"))
    n, m, F = 1 << scale, 1 << (scale + 4), 64
    ptr, idx = synth.rmat_csr(n, m, seed=123, device=dev)          # identical on every rank
    val = synth.gcn_norm_val(ptr, idx)
    Xb = torch.randn((n, F), device=dev, generator=torch.Generator(device=dev).manual_seed(5)).to(torch.bfloat16)
    hp = ptr.cpu().numpy()
    bounds = [int(b) for b in partition.split_rows(hp, world, "edges")]
    r0, r1 = bounds[rank], bounds[rank + 1]
    e0, e1 = int(hp[r0]), int(hp[r1])
    lptr = (ptr[r0:r1 + 1] - e0).contiguous()
    lidx, lval = idx[e0:e1].contiguous(), val[e0:e1].contiguous()
    for stages in sorted({-4, 0, 1, world - 1}):
        ph = PeerHalo(lptr, lidx, lval, bounds, rank, world, F, remote_stages=stages)
        ph.x(0, F, torch.bfloat16).copy_(Xb[r0:r1])
        ph.x(1, F).copy_(Xb[r0:r1].float())
        Yb = torch.empty((r1 - r0, F), device=dev)
        Y32 = torch.empty_like(Yb)
        ph.gcn_run(Yb, 0, F, dtype=torch.bfloat16)
        ph.gcn_run(Y32, 1, F)
        torch.cuda.synchronize()
        ph.check()
        same = bool(torch.equal(Yb, Y32))
        hX = torch.empty((r1 - r0, F), dtype=torch.bfloat16).pin_memory().copy_(Xb[r0:r1])
        hY = torch.empty((r1 - r0, F)).pin_memory()
        ph.gcn_layer_host(hX, None, hY)
        ph.check()
        same = same and bool(torch.equal(hY.to(dev), Yb))
        flags = torch.tensor([int(same)], device=dev)
        dist.all_reduce(flags, op=dist.ReduceOp.MIN)
        if rank == 0:
            import oracle as orc

            orc.use_all_cores()
            rows = min(r1 - r0, 3000)
            e = int(hp[rows])
            y64, sc = orc.spmm_f64(np.ascontiguousarray(hp[:rows + 1]), idx[:e].cpu().numpy(), val[:e].cpu().numpy(),
                                   Xb.float().cpu().numpy())
            err = np.abs(Yb[:rows].cpu().numpy().astype(np.float64) - y64) / (1e-5 * sc.astype(np.float64) + 1e-30)
            worst = float(err.max()) if rows else 0.0
            line = {"test": "multirank_bf16_equals_fp32", "world": world, "remote_stages": stages, "graph": "rmat%d" % scale,
                    "n": n, "m": m, "F": F, "bf16_equals_fp32_on_widened_x": bool(flags.item()),
                    "worst_err_over_bound_vs_fp64_oracle": round(worst, 4), "rows_checked": rows}
            line["ok"] = bool(flags.item() == 1 and worst <= 1.0)
            print(json.dumps(line), flush=True)
        ph.close()
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
