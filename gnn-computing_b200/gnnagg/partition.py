"""partition.py -- 1-D row partitioning by destination for multi-GPU aggregation (SURVEY.md 8(e)).

The reference is single-GPU (every driver asserts GPUNUM == 1, Figure9/main.cu:19; the prepare*Multi
prototypes of include/data.h:48-58 have no definitions), so this is new functionality built around the
same aggregator: rank p owns a contiguous block of destination rows and the matching X / Y shard; its
local CSR keeps GLOBAL source ids and gathers from a replicated X_full that an all-gather of the X
shards fills (NCCL over NVLink on GPUs, gloo in the CPU tests).  No partial sums cross ranks.
"""
import numpy as np


def split_rows(ptr, parts, balance="edges"):
    """row boundaries [parts+1] of contiguous blocks; balance='edges' puts ~m/parts edges in each block
    (power-law graphs make equal-row blocks unbalanced), 'rows' gives equal row counts"""
    ptr = np.asarray(ptr)
    n = len(ptr) - 1
    if balance == "rows":
        return np.array([(n * p) // parts for p in range(parts + 1)], np.int64)
    m = int(ptr[-1])
    cuts = [0]
    for p in range(1, parts):
        target = (m * p) // parts
        r = int(np.searchsorted(ptr, target, side="left"))
        cuts.append(min(max(r, cuts[-1]), n))
    cuts.append(n)
    return np.array(cuts, np.int64)


def local_block(ptr, idx, val, bounds, rank):
    """(ptr_local, idx_local, val_local) of rank's row block; source ids stay global"""
    r0, r1 = int(bounds[rank]), int(bounds[rank + 1])
    e0, e1 = int(ptr[r0]), int(ptr[r1])
    lp = (np.asarray(ptr[r0:r1 + 1]) - e0).astype(np.int32)
    return lp, np.ascontiguousarray(idx[e0:e1]), (None if val is None else np.ascontiguousarray(val[e0:e1]))


def gather_sizes(bounds):
    """rows owned by every rank (the all-gather of X is ragged when blocks are edge-balanced)"""
    return [int(bounds[p + 1] - bounds[p]) for p in range(len(bounds) - 1)]


def all_gather_rows(x_shard, bounds, group=None):
    """X_full [n, F] from per-rank shards [rows_p, F]; works for equal and ragged blocks and for any
    torch.distributed backend (nccl on GPUs, gloo on CPU)"""
    import torch
    import torch.distributed as dist

    sizes = gather_sizes(bounds)
    F = x_shard.shape[1]
    full = torch.empty((int(bounds[-1]), F), dtype=x_shard.dtype, device=x_shard.device)
    if len(set(sizes)) == 1:
        dist.all_gather_into_tensor(full, x_shard.contiguous(), group=group)
    else:
        # ragged blocks: one broadcast per owner into its slice of X_full (all_gather needs equal shapes)
        rank = dist.get_rank(group)
        full[int(bounds[rank]):int(bounds[rank + 1])].copy_(x_shard)
        for p in range(len(sizes)):
            if sizes[p]:
                dist.broadcast(full[int(bounds[p]):int(bounds[p + 1])], src=dist.get_global_rank(group, p) if group else p,
                               group=group)
    return full


# ------------------------------------------------------------------------------------------------
# pipelined halo exchange: the all-gather of X is cut into `chunks` row chunks and the rank's row block
# is split by the chunk its SOURCE falls into (the same idea as the slices of the reference's
# locality_schedule, graph_schedule.h:24-29, applied to the communication order).  Chunk c of every
# shard is gathered into its own buffer Xc[c] = [world, rows_c, F]; the sub-CSR of chunk c indexes that
# buffer directly and is accumulated (gnnagg_gcn_run_acc) as soon as all-gather c has completed, while
# all-gather c+1 is in flight.  Edges whose source lives on this rank need no communication: their
# sub-CSR runs first, hiding the first all-gather.
# ------------------------------------------------------------------------------------------------
def chunk_rows(n_per, chunks):
    """[chunks+1] row boundaries of the chunks inside one shard of n_per rows"""
    step = -(-n_per // chunks)
    return [min(n_per, c * step) for c in range(chunks + 1)]


def split_by_source_chunk(ptr, idx, val, n_per, world, rank, chunks):
    """torch tensors (any device).  Returns a list of (ptr_c, idx_c, val_c); entry 0 = edges whose source
    is owned by `rank` (idx_c = local row in this rank's X shard), entry 1+c = remote edges whose source
    falls in chunk c (idx_c = owner * rows_c + offset inside the chunk, an index into Xc[c])."""
    import torch

    n = ptr.numel() - 1
    deg = (ptr[1:] - ptr[:-1]).long()
    row = torch.repeat_interleave(torch.arange(n, device=ptr.device), deg)
    g = idx.long()
    owner, local = g // n_per, g % n_per
    cb = chunk_rows(n_per, chunks)
    bounds = torch.tensor(cb, device=ptr.device)
    chunk = torch.bucketize(local, bounds[1:], right=True)  # chunk c: cb[c] <= local < cb[c+1]
    own = owner == rank
    out = []

    def sub(mask, new_idx):
        cnt = torch.bincount(row[mask], minlength=n)
        p = torch.zeros(n + 1, dtype=torch.int64, device=ptr.device)
        p[1:] = torch.cumsum(cnt, 0)
        return p.to(torch.int32), new_idx.to(torch.int32).contiguous(), val[mask].contiguous()

    out.append(sub(own, local[own]))
    for c in range(chunks):
        mask = (~own) & (chunk == c)
        rows_c = cb[c + 1] - cb[c]
        out.append(sub(mask, owner[mask] * rows_c + (local[mask] - cb[c])))
    return out


class HaloPipeline:
    """per-rank driver of the pipelined exchange + aggregation (device side; one process per GPU)"""

    def __init__(self, ptr, idx, val, n_per, world, rank, feat, chunks=4, group=None):
        import torch

        from . import Aggregator

        self.n, self.n_per, self.world, self.rank, self.F, self.group = ptr.numel() - 1, n_per, world, rank, feat, group
        self.cb = chunk_rows(n_per, chunks)
        self.chunks = chunks
        parts = split_by_source_chunk(ptr, idx, val, n_per, world, rank, chunks)
        self.aggs = [Aggregator(p, i, v) for p, i, v in parts]
        for agg in self.aggs:  # multi-GPU blocks keep their CSR as given (as the gnnagg_dist_* stages do)
            agg.set_merge_duplicates(1)
        self.edges = [int(i.numel()) for _, i, _ in parts]
        self.Xc = [torch.empty((world * (self.cb[c + 1] - self.cb[c]), feat), device=ptr.device) for c in range(chunks)]

    def aggregate(self, Xs, Y):
        """Y = A_block * X_full with X_full never materialised contiguously"""
        import torch.distributed as dist

        works = [dist.all_gather_into_tensor(self.Xc[c], Xs[self.cb[c]:self.cb[c + 1]], group=self.group, async_op=True)
                 for c in range(self.chunks)]
        self.aggs[0].gcn_run_acc(Xs, Y, accumulate=False)  # local sources: overlaps the first all-gather
        for c in range(self.chunks):
            works[c].wait()  # stream-level dependency, the host does not block
            self.aggs[1 + c].gcn_run_acc(self.Xc[c], Y, accumulate=True)
        return Y

    @property
    def launches(self):
        return sum(a.launches for a in self.aggs)


# ------------------------------------------------------------------------------------------------
# pruned halo exchange: a rank only receives the source rows its row block actually references.
# On power-law graphs that is a small fraction of X (R-MAT scale 26 on 8 ranks: ~19 % of the rows), and
# the local CSR is re-indexed into the compact receive buffer, which also shrinks the gather footprint.
# ------------------------------------------------------------------------------------------------
def pruned_plan(idx, n_per, world, rank, group=None):
    """index bookkeeping of the pruned exchange (any device / backend).  Returns a dict with
    idx_compact (int32, idx re-indexed into the sorted unique list U of referenced sources), recv_counts /
    send_counts (rows per peer), send_rows (int64 rows of MY shard to pack, ordered by destination rank)
    and num_recv = |U|."""
    import torch
    import torch.distributed as dist

    U = torch.unique(idx.long())                                         # sorted global ids this block references
    idx_compact = torch.searchsorted(U, idx.long()).to(torch.int32)
    owner = torch.div(U, n_per, rounding_mode="floor")
    recv_counts = torch.bincount(owner, minlength=world).tolist()
    rc = torch.tensor(recv_counts, device=idx.device, dtype=torch.int64)
    sc = torch.empty_like(rc)
    dist.all_to_all_single(sc, rc, group=group)                           # how many of my rows every rank wants
    send_counts = sc.tolist()
    req = torch.empty(int(sum(send_counts)), device=idx.device, dtype=torch.int64)
    dist.all_to_all_single(req, U, output_split_sizes=send_counts, input_split_sizes=recv_counts, group=group)
    return {"idx_compact": idx_compact, "recv_counts": recv_counts, "send_counts": send_counts,
            "send_rows": (req - rank * n_per).contiguous(), "num_recv": int(U.numel())}


class PrunedHalo:
    """setup: pruned_plan; step: pack (gnnagg_gather_rows) -> all_to_all_single with uneven splits ->
    aggregate on the compact receive buffer"""

    def __init__(self, ptr, idx, val, n_per, world, rank, feat, group=None):
        import torch

        from . import Aggregator

        dev = ptr.device
        self.world, self.rank, self.group, self.F = world, rank, group, feat
        plan = pruned_plan(idx, n_per, world, rank, group)
        self.idx_compact, self.recv_counts, self.send_counts = plan["idx_compact"], plan["recv_counts"], plan["send_counts"]
        self.send_rows, self.num_recv = plan["send_rows"], plan["num_recv"]
        self.send_buf = torch.empty((self.send_rows.numel(), feat), device=dev)
        self.recv_buf = torch.empty((self.num_recv, feat), device=dev)
        self.agg = Aggregator(ptr, self.idx_compact, val)
        self.agg.set_merge_duplicates(1)  # multi-GPU blocks keep their CSR as given (as the gnnagg_dist_* stages do)
        self.referenced_fraction = self.num_recv / float(n_per * world)

    def exchange(self, Xs):
        import torch.distributed as dist

        from . import gather_rows

        gather_rows(Xs, self.send_rows, self.send_buf)
        dist.all_to_all_single(self.recv_buf, self.send_buf, output_split_sizes=self.recv_counts,
                               input_split_sizes=self.send_counts, group=self.group)
        return self.recv_buf

    def aggregate(self, Xs, Y):
        self.agg.gcn_run(self.exchange(Xs), Y)
        return Y


# ------------------------------------------------------------------------------------------------
# pipelined pruned halo exchange: the row block is cut into edge-balanced ROW chunks; chunk c only needs
# the source rows it references that no earlier chunk already fetched (the hubs arrive with chunk 0, later
# chunks fetch their tails).  Exchange c+1 is in flight while chunk c is aggregated.  Every row is computed
# exactly once by the ordinary kernel on a rebased slice of the CSR: no accumulation passes, no duplicated
# walk, no extra traffic on Y.
# ------------------------------------------------------------------------------------------------
def incremental_plan(ptr, idx, n_per, world, rank, chunks, group=None):
    """bookkeeping of the pipelined pruned exchange (any device / backend).  Returns a dict:
    row_bounds [chunks+1], idx_compact (int32 positions in the receive buffer), per stage c: recv_counts[c],
    send_counts[c] (rows per peer), send_rows[c] (int64 rows of MY shard, ordered by destination), recv_offset[c]
    (first receive-buffer row of stage c) and num_recv (receive-buffer rows in total)."""
    import torch
    import torch.distributed as dist

    dev = idx.device
    hp = ptr.cpu().numpy()
    rb = split_rows(hp, chunks, "edges")
    total_src = n_per * world
    seen = torch.zeros(total_src, dtype=torch.bool, device=dev)
    pos = torch.zeros(total_src, dtype=torch.int32, device=dev)
    plan = {"row_bounds": rb, "recv_counts": [], "send_counts": [], "send_rows": [], "recv_offset": []}
    offset = 0
    for c in range(chunks):
        e0, e1 = int(hp[rb[c]]), int(hp[rb[c + 1]])
        Uc = torch.unique(idx[e0:e1].long())
        new = Uc[~seen[Uc]]                                   # sorted: grouped by owner, ascending
        seen[new] = True
        pos[new] = torch.arange(offset, offset + new.numel(), device=dev, dtype=torch.int32)
        owner = torch.div(new, n_per, rounding_mode="floor")
        rc_list = torch.bincount(owner, minlength=world).tolist()
        rc = torch.tensor(rc_list, device=dev, dtype=torch.int64)
        sc = torch.empty_like(rc)
        dist.all_to_all_single(sc, rc, group=group)
        sc_list = sc.tolist()
        req = torch.empty(int(sum(sc_list)), device=dev, dtype=torch.int64)
        dist.all_to_all_single(req, new, output_split_sizes=sc_list, input_split_sizes=rc_list, group=group)
        plan["recv_counts"].append(rc_list)
        plan["send_counts"].append(sc_list)
        plan["send_rows"].append((req - rank * n_per).contiguous())
        plan["recv_offset"].append(offset)
        offset += int(new.numel())
    plan["num_recv"] = offset
    plan["idx_compact"] = pos[idx.long()]
    return plan


class PipelinedPrunedHalo:
    """device-side driver of incremental_plan (one process per GPU, NCCL)"""

    def __init__(self, ptr, idx, val, n_per, world, rank, feat, chunks=4, group=None):
        import torch

        from . import Aggregator

        dev = ptr.device
        self.group, self.chunks, self.F = group, chunks, feat
        plan = incremental_plan(ptr, idx, n_per, world, rank, chunks, group)
        self.plan = plan
        rb = plan["row_bounds"]
        hp = ptr.cpu()
        self.aggs, self.rows = [], []
        for c in range(chunks):
            r0, r1 = int(rb[c]), int(rb[c + 1])
            e0, e1 = int(hp[r0]), int(hp[r1])
            sub_ptr = (ptr[r0:r1 + 1] - e0).contiguous()
            self.aggs.append(Aggregator(sub_ptr, plan["idx_compact"][e0:e1].contiguous(), val[e0:e1].contiguous()))
            self.aggs[-1].set_merge_duplicates(1)  # as above: multi-GPU blocks keep their CSR as given
            self.rows.append((r0, r1))
        self.send_rows = torch.cat(plan["send_rows"]) if chunks else torch.empty(0, dtype=torch.int64, device=dev)
        self.send_off = np.concatenate([[0], np.cumsum([t.numel() for t in plan["send_rows"]])]).astype(np.int64)
        self.send_buf = torch.empty((int(self.send_off[-1]), feat), device=dev)
        self.recv_buf = torch.empty((plan["num_recv"], feat), device=dev)
        self.referenced_fraction = plan["num_recv"] / float(n_per * world)
        self.stage_fraction = [sum(rc) / max(1, plan["num_recv"]) for rc in plan["recv_counts"]]

    def aggregate(self, Xs, Y):
        import torch.distributed as dist

        from . import gather_rows

        p = self.plan
        gather_rows(Xs, self.send_rows, self.send_buf)       # pack every stage's rows once
        works = []
        for c in range(self.chunks):
            o = p["recv_offset"][c]
            cnt = sum(p["recv_counts"][c])
            works.append(dist.all_to_all_single(self.recv_buf[o:o + cnt], self.send_buf[int(self.send_off[c]):int(self.send_off[c + 1])],
                                                output_split_sizes=p["recv_counts"][c], input_split_sizes=p["send_counts"][c],
                                                group=self.group, async_op=True))
        for c in range(self.chunks):
            works[c].wait()                                   # stream dependency only
            r0, r1 = self.rows[c]
            if r1 > r0:
                self.aggs[c].gcn_run(self.recv_buf, Y[r0:r1])
        return Y

    @property
    def launches(self):
        return sum(a.launches for a in self.aggs)


# ------------------------------------------------------------------------------------------------
# peer-memory halo: binding over gnnagg_dist_* (csrc/dist.cu).  The exchange is not a collective: every owner
# pushes the rows each peer wants from its shard straight into that peer's receive slots with 128-bit stores
# over NVLink, receiver by receiver, while the receivers aggregate the edges whose sources have already
# landed.  torch.distributed is only used once, to all-gather the 256-byte connection blobs (cudaIpc
# handles) at set-up, and for the barriers of the teardown.
# ------------------------------------------------------------------------------------------------
class _DeviceMemory:
    """a library-owned device buffer exposed through __cuda_array_interface__ (zero-copy torch view).  The interface
    has no bf16 typestr: a bf16 view is taken as "<i2" and reinterpreted with .view(torch.bfloat16)."""

    def __init__(self, ptr, shape, owner, typestr="<f4"):
        self.owner = owner
        self.__cuda_array_interface__ = {"shape": tuple(int(s) for s in shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 3, "strides": None}


def _bounds_array(bounds):
    import ctypes as C

    return (C.c_int64 * len(bounds))(*[int(b) for b in bounds])


class PeerHalo:
    """one rank of the peer-memory multi-GPU aggregation.  `handle` is passed in by LocalDist (single process
    driving several ranks, which connects them itself); otherwise the rank is created on the current device and
    connected to its peers through torch.distributed (any backend: the blobs are plain bytes).
    remote_stages = 0: one pass after all rows have arrived; R >= 1: stage 0 = local sources, then R groups of
    owners accumulated as they land.  backward=True (on every rank alike) also readies gcn_backward: the transposed
    block, a G buffer the size of one X buffer and the return tables."""

    def __init__(self, ptr, idx, val, bounds, rank, world, feat_cap, remote_stages=1, group=None, handle=None, backward=False):
        import ctypes as C

        import torch

        from . import DIST_BLOB_BYTES, _dp, _stream, check, lib

        L = lib()
        self.rank, self.world, self.feat_cap, self.group = rank, world, feat_cap, group
        self.bounds = [int(b) for b in bounds]
        self.rows = self.bounds[rank + 1] - self.bounds[rank]
        self.device = ptr.device
        self._owns = handle is None
        assert ptr.dtype == torch.int32 and idx.dtype == torch.int32 and val.dtype == torch.float32
        assert ptr.numel() - 1 == self.rows, "the row block must match the rank's shard of X"
        if handle is None:
            h = C.c_void_p()
            check(L.gnnagg_dist_create_rank(rank, world, _bounds_array(self.bounds), feat_cap, C.byref(h)))
            self.h = h
        else:
            self.h = handle
        self.backward = bool(backward)
        if self.backward:
            check(L.gnnagg_dist_enable_backward(self.h))
        check(L.gnnagg_dist_set_graph(self.h, _dp(ptr.contiguous()), _dp(idx.contiguous()), _dp(val.contiguous()), idx.numel(),
                                      int(remote_stages), _stream()))
        if handle is None and world > 1:
            import torch.distributed as dist

            blob = C.create_string_buffer(DIST_BLOB_BYTES)
            check(L.gnnagg_dist_export(self.h, blob))
            on_gpu = dist.get_backend(group) == "nccl"
            mine = torch.frombuffer(bytearray(blob.raw), dtype=torch.uint8)
            mine = mine.to(self.device) if on_gpu else mine
            every = torch.empty(world * DIST_BLOB_BYTES, dtype=torch.uint8, device=mine.device)
            dist.all_gather_into_tensor(every, mine, group=group)
            check(L.gnnagg_dist_connect(self.h, every.cpu().numpy().tobytes()))
        self.refresh_info()

    def refresh_info(self):
        import ctypes as C

        from . import check, lib

        world = self.world
        nrecv, counts, nst = C.c_int64(), (C.c_int64 * world)(), C.c_int()
        edges, sends = (C.c_int64 * 16)(), (C.c_int64 * world)()
        check(lib().gnnagg_dist_info(self.h, C.byref(nrecv), counts, C.byref(nst), edges, sends))
        self.num_recv, self.recv_counts, self.num_stages = int(nrecv.value), [int(c) for c in counts], int(nst.value)
        self.stage_edges = [int(edges[s]) for s in range(self.num_stages)]
        self.send_counts = [int(c) for c in sends]
        self.num_send = sum(self.send_counts)
        self.referenced_fraction = (self.num_recv + 0.0) / max(1, self.bounds[-1])

    def x(self, buf=0, feat=None, dtype=None):
        """torch view [rows, feat] of peer-visible shard buffer `buf` (write X here, or let a layer write H here).
        dtype torch.float32 (default) or torch.bfloat16: a bf16 shard of the same width takes half of the buffer; steps
        on it pass dtype=torch.bfloat16 too"""
        import torch

        from . import lib

        dtype = torch.float32 if dtype is None else dtype
        if dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("PeerHalo.x: dtype must be torch.float32 or torch.bfloat16, got %s" % dtype)
        feat = self.feat_cap if feat is None else feat
        p = lib().gnnagg_dist_x(self.h, int(buf))
        if self.rows == 0:
            return torch.empty((0, feat), device=self.device, dtype=dtype)
        if dtype == torch.bfloat16:
            return torch.as_tensor(_DeviceMemory(p, (self.rows, feat), self, "<i2"), device=self.device).view(torch.bfloat16)
        return torch.as_tensor(_DeviceMemory(p, (self.rows, feat), self), device=self.device)

    @staticmethod
    def _is_bf16(dtype):
        import torch

        if dtype is None or dtype == torch.float32:
            return False
        if dtype == torch.bfloat16:
            return True
        raise ValueError("the shard dtype must be torch.float32 or torch.bfloat16, got %s" % dtype)

    def gcn_run(self, Y, buf=0, feat=None, exchange=True, dtype=None):
        """Y = A_block X with X = shard buffer `buf` of every rank, stored as `dtype` (float32 or bfloat16; Y is float32)"""
        from . import DIST_NO_EXCHANGE, _f32, _stream, check, lib

        feat = Y.shape[1] if feat is None else feat
        run = lib().gnnagg_dist_gcn_run_bf16 if self._is_bf16(dtype) else lib().gnnagg_dist_gcn_run
        check(run(self.h, int(buf), _f32(Y, "Y"), int(feat), 0 if exchange else DIST_NO_EXCHANGE, _stream()))
        return Y

    def gcn_layer(self, W, H, buf=0, exchange=True, dtype=None):
        """H = (A_block X) W with X = shard buffer `buf` stored as `dtype` (float32 or bfloat16; W, H are float32)"""
        from . import DIST_NO_EXCHANGE, _f32, _stream, check, lib

        run = lib().gnnagg_dist_gcn_layer_bf16 if self._is_bf16(dtype) else lib().gnnagg_dist_gcn_layer
        check(run(self.h, int(buf), _f32(W, "W"), _f32(H, "H"), W.shape[0], W.shape[1], 0 if exchange else DIST_NO_EXCHANGE,
                  _stream()))
        return H

    def gcn_backward(self, dY, dX):
        """dX = (A^T dY) on this rank's shard rows, dY and dX float32 [rows, feat].  Collective: every rank calls it
        with the same width, as many times; needs backward=True at construction"""
        from . import _f32, _stream, check, lib

        check(lib().gnnagg_dist_gcn_backward(self.h, _f32(dY, "dY"), _f32(dX, "dX"), int(dY.shape[1]), _stream()))
        return dX

    def gcn_layer_host(self, hX, hW, hH, buf=0):
        """pinned host X shard (float32 or bfloat16) and W -> host H (or A*X when hW is None), float32; copies inside,
        synchronises the stream"""
        from . import _bf16, _f32, _is_bf16, _stream, check, lib

        fin = hX.shape[1]
        fout = fin if hW is None else hW.shape[1]
        if _is_bf16(hX):
            check(lib().gnnagg_dist_gcn_layer_host_bf16(self.h, int(buf), _bf16(hX, "hX", cuda=False), _f32(hW, "hW", cuda=False),
                                                        _f32(hH, "hH", cuda=False), fin, fout, _stream()))
        else:
            check(lib().gnnagg_dist_gcn_layer_host(self.h, int(buf), _f32(hX, "hX", cuda=False), _f32(hW, "hW", cuda=False),
                                                   _f32(hH, "hH", cuda=False), fin, fout, _stream()))
        return hH

    def profile(self, on=True):
        from . import check, lib

        check(lib().gnnagg_dist_profile_enable(self.h, int(on)))

    def profile_read(self):
        """ms of the last run: dict(exchange, step, stage0, dense)"""
        import ctypes as C

        from . import check, lib

        ms = (C.c_float * 4)()
        check(lib().gnnagg_dist_profile_read(self.h, ms))
        return {"exchange": ms[0], "step": ms[1], "stage0": ms[2], "dense": ms[3]}

    def check(self):
        from . import check, lib

        check(lib().gnnagg_dist_check(self.h))

    @property
    def launches(self):
        from . import lib

        return lib().gnnagg_dist_launch_count(self.h)

    def close(self):
        """collective when world > 1 and the rank was created here: everybody idle -> unmap the peers -> free"""
        from . import lib

        if getattr(self, "h", None) and self._owns:
            if self.world > 1:
                import torch
                import torch.distributed as dist

                torch.cuda.synchronize()
                dist.barrier(group=self.group)
                lib().gnnagg_dist_disconnect(self.h)
                dist.barrier(group=self.group)
            lib().gnnagg_dist_destroy(self.h)
        self.h = None


class LocalDist:
    """gnnagg_dist_create: ONE process drives `world` ranks (devices[r], default r; the same device may be given
    several times, which is how the single-GPU tests exercise the whole protocol).  set_graph for every rank, then
    connect()."""

    def __init__(self, bounds, feat_cap, devices=None):
        import ctypes as C

        from . import check, lib

        world = len(bounds) - 1
        self.world, self.bounds, self.feat_cap = world, [int(b) for b in bounds], feat_cap
        self.devices = list(range(world)) if devices is None else [int(d) for d in devices]
        self._hs = (C.c_void_p * world)()
        check(lib().gnnagg_dist_create(world, (C.c_int * world)(*self.devices), _bounds_array(self.bounds), feat_cap, self._hs))
        self.handles = [C.c_void_p(self._hs[r]) for r in range(world)]
        self.ranks = [None] * world

    def set_graph(self, rank, ptr, idx, val, remote_stages=1, backward=False):
        self.ranks[rank] = PeerHalo(ptr, idx, val, self.bounds, rank, self.world, self.feat_cap, remote_stages,
                                    handle=self.handles[rank], backward=backward)
        return self.ranks[rank]

    def connect(self):
        from . import check, lib

        check(lib().gnnagg_dist_connect_local(self._hs, self.world))
        for r in self.ranks:
            r.refresh_info()

    def close(self):
        import torch

        from . import lib

        torch.cuda.synchronize()
        for h in self.handles:
            lib().gnnagg_dist_disconnect(h)
        for h in self.handles:
            lib().gnnagg_dist_destroy(h)
        self.handles = []


_dist_gcn_fn = None


def _dist_gcn_function():
    """the autograd Function behind dist_gcn_aggregate, defined on first use (this module imports torch lazily)"""
    global _dist_gcn_fn
    if _dist_gcn_fn is None:
        import torch

        class DistGCNAggregate(torch.autograd.Function):
            @staticmethod
            def forward(ctx, ph, X, buf):
                F = X.shape[1]
                ph.x(buf, F, X.dtype).copy_(X)
                Y = torch.empty((ph.rows, F), device=X.device, dtype=torch.float32)
                ph.gcn_run(Y, buf, F, dtype=X.dtype)
                ctx.ph, ctx.x_dtype = ph, X.dtype
                return Y

            @staticmethod
            def backward(ctx, dY):
                dX = torch.empty(dY.shape, device=dY.device, dtype=torch.float32)
                ctx.ph.gcn_backward(dY.contiguous(), dX)
                return None, dX.to(ctx.x_dtype), None

        _dist_gcn_fn = DistGCNAggregate
    return _dist_gcn_fn


def dist_gcn_aggregate(ph, X, buf=0):
    """Y = A_block X across ranks as a differentiable op: X is this rank's shard [rows, F] (float32 or bfloat16), copied
    into shard buffer `buf` of the PeerHalo `ph` (made with backward=True); Y is float32.  The backward is
    gnnagg_dist_gcn_backward, dX computed in float32 and rounded once to X's dtype (a bf16 shard needs nothing else: the
    backward never reads X).  A layer is this op followed by torch.matmul with W.

    The op is collective in both directions: every rank runs its forward, and later its backward, the same number of
    times with the same width.  In one process driving several ranks (LocalDist), each rank's forward must run on its
    own stream, as gcn_run already requires; autograd runs each backward on the stream of its forward."""
    return _dist_gcn_function().apply(ph, X, buf)


def stage_ends(world, R):
    """[R+1] arrival positions at which the owner groups of the stage mode end (dist.cu): geometric growth -- 7 owners in
    3 stages are cut 1 + 2 + 4 -- with at least one owner per group"""
    ends = [0] * (R + 1)
    for s in range(1, R + 1):
        e = int(((1 << s) - 1) / float((1 << R) - 1) * (world - 1) + 0.5)
        e = max(e, s)
        e = min(e, world - 1 - (R - s))
        ends[s] = world - 1 if s == R else e
    return ends


def peer_plan(idx, bounds, rank, remote_stages, ptr=None):
    """numpy restatement of the index bookkeeping of gnnagg_dist_set_graph (csrc/dist.cu), for tests and for
    reasoning about traffic without a GPU.  remote_stages = R > 0: stages by owner; 0: one pass; < 0: row pipelining
    with K = -R edge-balanced row chunks (needs `ptr`).  Returns a dict:
      recv_rows   global ids of the distinct REMOTE sources of this block in receive-slot order: ascending id, or --
                  row-pipelined -- by the round (row chunk) that needs a row first, then ascending id
      recv_tab    [rounds, world+1] first slot of every owner's rows of a round; recv_tab[c][world] = end of round c
      recv_local  recv_rows as local row numbers inside their owner's shard (the rows that owner pushes)
      stage_of    [world] stage of every owner: 0 = this rank (and everybody when R <= 0), 1..R = groups of the owners
                  taken in the order rank+1, rank+2, ... (mod world), group sizes growing geometrically (stage_ends)
      recv_order  the world-1 remote owners in the order their rows arrive (owner p pushes to p-1, p-2, ...)
      chunk_rows  [rounds+1] row chunk boundaries
      idx_new     per edge: local row of the own shard, or rows_own + receive slot (one buffer: shard, then slots)
      stage       per edge: its stage"""
    bounds = np.asarray(bounds, np.int64)
    W = len(bounds) - 1
    g = np.asarray(idx, np.int64)
    own_lo, own_hi = int(bounds[rank]), int(bounds[rank + 1])
    rows_own = own_hi - own_lo
    remote = (g < own_lo) | (g >= own_hi)
    R = 0 if W == 1 else max(0, min(int(remote_stages), W - 1))
    K = 1 if (W == 1 or remote_stages >= 0) else min(-int(remote_stages), 16)
    chunk_rows = np.array([0] + [rows_own] * K, np.int64)
    U = np.unique(g[remote])
    first = np.zeros(len(U), np.int64)
    if K > 1:
        ptr = np.asarray(ptr, np.int64)
        m = int(ptr[-1])
        for c in range(1, K):
            chunk_rows[c] = max(min(int(np.searchsorted(ptr, (m * c) // K, side="left")), rows_own), chunk_rows[c - 1])
        row = np.repeat(np.arange(rows_own), np.diff(ptr))
        chunk_e = np.searchsorted(chunk_rows[1:K], row, side="right")          # chunk of every edge's row
        first = np.full(len(U), K, np.int64)
        np.minimum.at(first, np.searchsorted(U, g[remote]), chunk_e[remote])
        order_u = np.lexsort((U, first))                                         # by round, then id
        U, first = U[order_u], first[order_u]
    owner_u = np.searchsorted(bounds, U, side="right") - 1
    recv_tab = np.zeros((K, W + 1), np.int64)
    for c in range(K):
        lo = int(np.searchsorted(first, c, side="left")) if K > 1 else 0
        sel = U[first == c] if K > 1 else U
        recv_tab[c] = lo + np.searchsorted(sel, bounds, side="left")
    order = [(rank + 1 + k) % W for k in range(W - 1)]
    stage_of = np.zeros(W, np.int64)
    ends = stage_ends(W, R)
    for k, p in enumerate(order):
        stage_of[p] = 0 if R == 0 else 1 + int(np.searchsorted(ends[1:], k, side="right"))
    owner_e = np.clip(np.searchsorted(bounds, g, side="right") - 1, 0, W - 1)
    slot_of = np.empty(len(U), np.int64)
    by_id = np.argsort(U, kind="stable")
    slot_of[:] = 0
    slots_sorted = np.empty(len(U), np.int64)
    slots_sorted[:] = by_id                                                      # U[by_id] ascending -> slot = by_id
    Us = U[by_id]
    e_slot = slots_sorted[np.searchsorted(Us, g[remote])] if remote.any() else np.zeros(0, np.int64)
    idx_new = (g - own_lo).astype(np.int64)
    idx_new[remote] = rows_own + e_slot
    counts = np.bincount(owner_u, minlength=W) if len(U) else np.zeros(W, np.int64)
    return {"recv_rows": U, "recv_tab": recv_tab, "recv_off": recv_tab[0] if K == 1 else None, "recv_counts": counts,
            "recv_local": U - bounds[owner_u], "stage_of": stage_of, "recv_order": order, "num_stages": 1 + R, "rounds": K,
            "chunk_rows": chunk_rows, "idx_new": idx_new.astype(np.int32),
            "stage": np.where(remote, stage_of[owner_e], 0).astype(np.int32)}
