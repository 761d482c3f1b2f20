// agg_kernels.cuh -- the neighbour-aggregation kernel family (GCN SpMM and fused GAT), sm_100a.
//
// Replaces the reference kernels aggr_gcn / aggr_gcn_target (include/aggr_gcn.h:5-36,78-114) and
// aggr_gat / aggr_gat_fine (include/aggr_gat.h:116-205).  Not a port: the reference maps one warp
// to one row (or one neighbour group), F/32 y-warps re-read idx/val, every lane issues scalar
// 4-byte gathers and split rows are combined with float atomics.  Here:
//
//   * EDGE-BALANCED ITEMS.  The edge array is cut into fixed-size items; a "virtual warp" of
//     LPR = F/4 lanes (8/16/32) owns one item and walks the rows that intersect it.  A hub row
//     of 10^5..10^6 edges is therefore spread over thousands of virtual warps and a warp never
//     idles on a short row.  One 32-lane warp always stages 512 consecutive edges.
//   * TMA STAGING.  The 512 idx (and val) entries of a warp are brought into shared memory by
//     two 1-D bulk copies (cp.async.bulk -> UBLKCP) completing on an mbarrier; the walk then
//     reads them as conflict-free broadcasts instead of 2 SHFL per edge-lane.
//   * 128-BIT GATHERS, U-DEEP.  Each lane gathers float4 of the source row; U (8) independent
//     gathers are issued before the first FMA so every warp keeps 4 KB in flight.
//   * DETERMINISTIC SPLIT ROWS.  A row that crosses item boundaries leaves per-item partials in
//     a carry buffer; a small fix-up kernel adds them in item order (no float atomics, results
//     are run-to-run reproducible).  Only the scheduled mode -- whose group order is
//     arbitrary (locality slices) -- combines with 128-bit RED.ADD, like the reference.
//   * 64-bit addressing of X/Y (the reference overflows int at idx*F, aggr_gcn.h:23).
#pragma once
#include <climits>
#include <type_traits>

#include "common.cuh"

namespace gnnagg {

struct AggParams {
    // CSR (or scheduled group list): ptr has num_rows+1 entries, idx/val num_edges entries
    const int *__restrict__ ptr;
    const int *__restrict__ idx;
    const float *__restrict__ val;       // GCN edge values; unused for GAT
    const int *__restrict__ target;      // scheduled mode: output row of every group
    const int *__restrict__ item_row;    // row containing edge k*kFineItem
    const void *__restrict__ X;          // [*, F] fp32, or bf16 bit patterns for the XBF16 instances
    const float *__restrict__ att;       // GAT attention table [n,2]
    const float *__restrict__ P;         // MLP: projected features P = X*W, [n, F] (also the gather source); SDDMM: X2
    float *__restrict__ Y;               // [n, F]
    float *__restrict__ carry;           // [num_items, F] partials of rows entering an item
    float *__restrict__ den_row;         // GAT: [n] denominator of rows that start in an item and leave it
    float *__restrict__ carry_den;       // GAT: [num_items]
    float *__restrict__ newval;          // GAT scheduled: un-normalised edge weights (aggr_gat.h:192); SDDMM: the dot products
    // GAT backward (two traversals, see kModeGATBWD / kModeGATBWD2 below)
    const float2 *__restrict__ bwd_c;    // per destination row (1 / D_v, c_v = <Y[v], dY[v]>); pass 1 reads .y, pass 2 reads .x
    float2 *__restrict__ bwd_wt;         // per edge (w_e, t_e): un-normalised weight and w_e (g_e - c_v) lrelu'(s_e)
    float2 *__restrict__ bwd_part;       // pass 1: [n] (sum w, sum t) over the edges of row v inside the item where v starts
    float2 *__restrict__ bwd_carry;      // pass 1: [num_items] the same sums of the row that ENTERS an item
    float *__restrict__ rsum;            // pass 2: row sums of ds go to rsum[row * rsum_stride] (source half of d att)
    int rsum_stride;
    int num_rows;
    int num_edges;
    int F;
    float slope;
    int bulk_ok;                         // idx/val 16-byte aligned -> TMA staging allowed
    int num_fine_items;                  // entries of item_row
    int accumulate;                      // GCN un-scheduled: Y += A*X instead of Y = A*X
    const int *__restrict__ out_row;     // un-scheduled GCN over a COMPACTED sub-CSR (locality slices): row r of the CSR is
                                         // output row out_row[r]; NULL: identity.  Every output row occurs at most once.
    // row-range launch (un-scheduled only): rows [row_lo, row_hi) = edges [edge_lo, edge_hi); the whole graph is
    // (0, num_rows, 0, num_edges).  Items keep their global numbering, a range just clips them.
    int row_lo, row_hi, edge_lo, edge_hi;
};

// The GAT backward (aggr_gat_fine_bwd, aggr_gat.h:222-294) is two traversals with one row-parallel kernel between them:
// kModeGATBWD  (pass 1, the CSR): the SDDMM traversal with X2 = dY.  Its per-edge epilogue turns g_e = <X[u], dY[v]>
//   into (w_e, t_e) with w_e the UN-normalised softmax weight and t_e = w_e (g_e - c_v) lrelu'(s_e) (:266-290 before
//   the division by D_v), and sums both per row on the way (item/carry scheme, deterministic): D_v is not an input.
//   gat_bwd_rowfinal_kernel then closes the rows: 1 / D_v and d att[2v] = (sum t) / D_v.
// kModeGATBWD2 (pass 2, the TRANSPOSED CSR, rows = sources u): the aggregation dX[u] = sum_e alpha_e dY[v] whose
//   weight is formed on the fly, alpha_e = w_e / D_v with (w, t) fetched through t_perm (staged like GCN edge values),
//   and whose row scalar -- the GAT denominator slot -- is sum_e t_e / D_v = d att[2u+1].
enum { kModeGCN = 0, kModeGAT = 1, kModeMLP = 2, kModeSDDMM = 3, kModeGATBWD = 4, kModeGATBWD2 = 5 };
__host__ __device__ constexpr bool mode_emits_edges(int mode) { return mode == kModeSDDMM || mode == kModeGATBWD; }  // per-edge outputs, no row sums
__host__ __device__ constexpr bool mode_has_dst(int mode) { return mode == kModeMLP || mode_emits_edges(mode); }  // keeps P[dst,:] in registers
__host__ __device__ constexpr bool mode_stages_val(int mode) { return mode == kModeGCN; }
// the edge weight is computed per batch by lanes vl < U and shared by shuffle; a scalar per row travels with the sums
__host__ __device__ constexpr bool mode_gat_like(int mode) { return mode == kModeGAT || mode == kModeGATBWD2; }

// row that contains edge e0 (start of an item): direct lookup when items are aligned with the
// item_row table, bounded binary search otherwise (the small-graph variant uses 32..128-edge items)
__device__ __forceinline__ int item_start_row(const AggParams &p, int e0)
{
    if (e0 % kFineItem == 0) return __ldg(p.item_row + e0 / kFineItem);
    return row_of_edge(p.ptr, p.item_row, p.num_fine_items, p.num_rows, e0);
}

// four consecutive columns of the gathered row at x: a float4, or (XBF16) four bf16 in 8 bytes widened exactly to fp32
// (a bf16 is the high half of an fp32)
template <bool XBF16>
__device__ __forceinline__ float4 ldg_x4(const char *x)
{
    if (!XBF16) return __ldg(reinterpret_cast<const float4 *>(x));
    const uint2 h = __ldg(reinterpret_cast<const uint2 *>(x));
    return make_float4(__uint_as_float(h.x << 16), __uint_as_float(h.x & 0xffff0000u), __uint_as_float(h.y << 16),
                       __uint_as_float(h.y & 0xffff0000u));
}

// WE = edges staged per warp: 512 normally, 128 for small graphs (4x more warps, shorter walks)
// (5 resident CTAs per SM for the small-graph variant -- 48 registers -- measured on the arxiv shape: no change.)
// XBF16 (GCN, GAT, and pass 1 of the GAT backward): X holds bf16.  The lane mapping, items and carries are those of
// the fp32 run of the same width; each lane gathers 8 bytes where it gathered 16 and runs the same FMAs / dot products
// on the widened values, so the result equals the fp32 run on the widened X bit for bit.  The other operands (att, the
// dY row of pass 1) stay fp32.
template <int LPR, int NV, int MODE, bool SCHED, int WE, bool XBF16 = false>
__global__ void __launch_bounds__(kCtaThreads, (WE < 512) ? 4 : 3) agg_kernel(const AggParams p)
{
    static_assert(!XBF16 || MODE == kModeGCN || MODE == kModeGAT || (MODE == kModeGATBWD && !SCHED),
                  "bf16 X is an operand of the GCN and GAT aggregations and of pass 1 of the GAT backward");
    using XT = typename std::conditional<XBF16, uint16_t, float>::type;
    constexpr int kWarpEdges = WE;            // shadows the namespace-level default
    constexpr int VPW = 32 / LPR;             // virtual warps per warp
    constexpr int EB = kWarpEdges / VPW;      // edges per item
    // gathers in flight per lane = U*NV float4; the small-graph variant trades depth for residency
    constexpr int U = (WE < 512) ? 4 : ((NV == 1) ? 8 : 4);
    constexpr int CHUNK = LPR * 4 * NV;       // feature columns covered per pass
    static_assert(LPR >= 8 && U <= LPR && EB % U == 0, "virtual warp narrower than 8 lanes is not supported");

    // per warp: [0] = idx, [1] = val (float bits); one base address serves both (val = idx + kWarpEdges words)
    __shared__ __align__(16) int s_stage[kCtaWarps][2][kWarpEdges];
    __shared__ __align__(8) uint64_t s_bar[kCtaWarps];

    // the two passes of the GAT backward read what the kernel in front of them wrote and are launched with launch_dep
    if (MODE == kModeGATBWD || MODE == kModeGATBWD2) griddep_wait();
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int64_t gwarp = (int64_t)(p.edge_lo / kWarpEdges) + (int64_t)blockIdx.x * kCtaWarps + warp;
    const int64_t wbase64 = gwarp * kWarpEdges;
    if (wbase64 >= p.edge_hi) return;  // whole warp idle (warp-uniform)
    // (opaque in the per-edge-output modes: their long batch body otherwise re-derives it from %tid / %ctaid every time)
    const int wbase = mode_emits_edges(MODE) ? (int)opaque32((uint32_t)wbase64) : (int)wbase64;
    const int wcnt = min(kWarpEdges, p.num_edges - wbase);

    // ---------------- stage idx (+val) of this warp's edges ----------------
    int *const my_idx = s_stage[warp][0];
    float *const my_val = reinterpret_cast<float *>(my_idx + kWarpEdges);
    int first_row = 0, first_row_end = 0, first_row_begin = 0;
    {
        const int nb = p.bulk_ok ? (wcnt & ~3) : 0;  // bulk copies need 16-byte multiples
        // edge values travel with idx for GCN, and for the GAT backward when the weights are handed in (no table)
        // and for its second pass, whose "values" are the positions t_perm of the edges in CSR order
        const bool stage_val = (MODE == kModeGCN) || (MODE == kModeGATBWD && p.att == nullptr) || (MODE == kModeGATBWD2);
        const uint32_t bar = smem_u32(&s_bar[warp]);
        if (nb > 0) {
            if (lane == 0) {
                mbar_init(bar, 1);
                fence_proxy_async();  // init visible to the async proxy; CTA scope (no L1 invalidate)
                const uint32_t bytes = (uint32_t)nb * 4u;
                mbar_expect_tx(bar, stage_val ? 2u * bytes : bytes);  // GAT / MLP / SDDMM stage idx only
                bulk_g2s(smem_u32(my_idx), p.idx + wbase, bytes, bar);
                if (stage_val) bulk_g2s(smem_u32(my_val), p.val + wbase, bytes, bar);
            }
        }
        for (int i = nb + lane; i < wcnt; i += 32) {
            my_idx[i] = __ldg(p.idx + wbase + i);
            if (stage_val) my_val[i] = __ldg(p.val + wbase + i);
        }
        // the start row of this lane's item is looked up while the bulk copy is in flight
        {
            const int e0s = max(wbase + (lane / LPR) * EB, p.edge_lo);
            if (e0s < p.edge_hi) {
                first_row = (e0s == p.edge_lo) ? p.row_lo : item_start_row(p, e0s);
                first_row_end = __ldg(p.ptr + first_row + 1);
                first_row_begin = __ldg(p.ptr + first_row);
            }
        }
        __syncwarp();
        if (nb > 0) mbar_wait(bar, 0);
        // GAT: the source half of the attention logit, att[2u+1] (aggr_gat.h:138), is NOT staged here: a separate
        // gather phase per warp (16 dependent-free loads per lane, then the walk) left the walk without loads in flight
        // while it ran.  Lane u < U of a virtual warp fetches the term of edge u of each batch together with the batch's
        // row gathers instead, and the virtual warp shares it by shuffle.
    }

    // ---------------- the walk: one virtual warp per item ----------------
    const int vw = lane / LPR;
    const int vl = lane % LPR;
    // Mask of the shuffles below.  Their sources are always lanes of the caller's own virtual warp (width = LPR), whose
    // lanes never diverge from each other, so the lanes that currently execute together are a valid mask -- and the
    // right one: with the static per-virtual-warp mask, two or four virtual warps that run converged (the normal case)
    // present DIFFERENT mask values to one shfl.sync, which the hardware then executes once per distinct mask behind a
    // MATCH.ANY check (seen in the SASS of every LPR < 32 variant).  One common mask lets them share the instruction.
    auto vmask = [&]() -> unsigned { return (LPR == 32) ? 0xffffffffu : __activemask(); };
    const int e0 = max(wbase + vw * EB, p.edge_lo);            // item clipped to the launched edge range
    const int e1 = min(wbase + vw * EB + EB, p.edge_hi);
    if (e0 >= e1) return;  // below, only shuffles whose sources lie inside the caller's virtual warp (vmask)
    const int64_t item = gwarp * VPW + vw;
    const int F = p.F;

    for (int cb = 0; cb < F; cb += CHUNK) {
        const int col = cb + vl * 4;
        const bool act0 = col < F;
        const bool act1 = (NV > 1) && (col + LPR * 4 < F);

        int row = first_row;
        int row_end = first_row_end;
        bool carry_in = SCHED ? false : (first_row_begin < e0);
        float a_dst = 0.f;
        if (MODE == kModeGAT) a_dst = __ldg(p.att + 2 * (size_t)(SCHED ? __ldg(p.target + row) : row));

        float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
        float den = 0.f;
        // MLP: projected feature of the destination row, P[dst, col..] (aggr_nn.h:26 `cached`, after projection)
        // (Fetching it one row ahead, and carrying the row terms of the GAT backward in registers beside it, was measured
        // on the arxiv shape and lost: 0.162 against 0.154 ms for the whole backward -- the walk is bound by how many
        // warps an SM holds, 3 CTAs per SM cost another 0.015 ms, and the extra registers are not free.)
        float4 pd0 = make_float4(0.f, 0.f, 0.f, 0.f), pd1 = pd0;
        auto load_dst = [&](int r) {
            const float *q = p.P + (size_t)(SCHED ? __ldg(p.target + r) : r) * F + col;
            if (act0) pd0 = ldg_f4(q);
            if (act1) pd1 = ldg_f4(q + LPR * 4);
        };
        if (mode_has_dst(MODE)) load_dst(first_row);

        // closes `row`: writes / accumulates its result and moves to the next row
        auto flush = [&](bool at_item_end) {
            if (mode_emits_edges(MODE)) {
                // nothing is accumulated per row: the flush only advances to the next row / group
            } else if (SCHED) {
                const int t = __ldg(p.target + row);
                const bool merge = !at_item_end && (row + 1 < p.row_hi) && (__ldg(p.target + row + 1) == t);
                if (!merge) {  // consecutive groups of one target are summed in registers first
                    float *y = p.Y + (size_t)t * F + col;
                    if (act0) red_add_f4(y, acc0);
                    if (act1) red_add_f4(y + LPR * 4, acc1);
                    if (MODE == kModeGAT && vl == 0 && cb == 0) atomicAdd(p.den_row + t, den);
                    acc0 = make_float4(0.f, 0.f, 0.f, 0.f);
                    acc1 = acc0;
                    den = 0.f;
                }
            } else if (carry_in) {
                float *c = p.carry + (size_t)item * F + col;
                if (act0) stg_f4(c, acc0);
                if (act1) stg_f4(c + LPR * 4, acc1);
                if (mode_gat_like(MODE) && vl == 0 && cb == 0) p.carry_den[item] = den;
                carry_in = false;
            } else {
                float *y = p.Y + (size_t)((MODE == kModeGCN && p.out_row) ? __ldg(p.out_row + row) : row) * F + col;
                if (MODE == kModeGAT) {
                    // complete row: normalise here (aggr_gat.h:163); empty row -> 0 (documented)
                    const float inv = (den != 0.f) ? __fdividef(1.f, den) : 0.f;
                    acc0 = make_float4(acc0.x * inv, acc0.y * inv, acc0.z * inv, acc0.w * inv);
                    acc1 = make_float4(acc1.x * inv, acc1.y * inv, acc1.z * inv, acc1.w * inv);
                }
                if (MODE == kModeGATBWD2 && vl == 0 && cb == 0) p.rsum[(size_t)row * p.rsum_stride] = den;  // complete row
                if (MODE == kModeGCN && p.accumulate) {  // each row is stored by exactly one item: plain RMW is safe
                    // a lane whose partial sum is exactly zero has nothing to add: rows without edges in this sub-CSR
                    // (most rows of a source slice of a low-degree graph) cost no traffic on Y
                    // The add itself is a 128-bit reduction (RED.E.ADD.F32x4): nobody else touches this row during the
                    // launch, so the result is as deterministic as load-add-store, but the warp does not wait for Y to come
                    // back from memory at the end of every (short) row.
                    const bool z0 = !act0 || is_zero4(acc0), z1 = !act1 || is_zero4(acc1);
                    if (!z0) red_add_f4(y, acc0);
                    if (!z1) red_add_f4(y + LPR * 4, acc1);
                } else {
                    if (act0) stg_f4(y, acc0);
                    if (act1) stg_f4(y + LPR * 4, acc1);
                }
            }
            if (!SCHED) {
                acc0 = make_float4(0.f, 0.f, 0.f, 0.f);
                acc1 = acc0;
                den = 0.f;
            }
            ++row;
            if (row < p.row_hi) {
                row_end = __ldg(p.ptr + row + 1);
                if (MODE == kModeGAT) a_dst = __ldg(p.att + 2 * (size_t)(SCHED ? __ldg(p.target + row) : row));
                if (mode_has_dst(MODE)) load_dst(row);
            } else {
                row_end = INT_MAX;
            }
        };

        int e = e0;
        while (row_end == e) flush(false);  // leading empty rows (only item 0 can see any)

        // gather base of this lane: column `col` of row 0 (inactive lanes of a partial chunk read
        // column 0 instead of being predicated off; their results are never stored)
        const char *xb = reinterpret_cast<const char *>(
            opaque64(reinterpret_cast<uint64_t>(static_cast<const XT *>(p.X) + (act0 ? col : 0))));
        const uint32_t row_bytes = opaque32((uint32_t)F * (uint32_t)sizeof(XT));
        const uint32_t s_base = opaque32(smem_u32(my_idx));  // shared address of this warp's staged idx (val: + 4*kWarpEdges)
        const int second = act1 ? LPR * 4 * (int)sizeof(XT) : 0;  // byte offset of the second 4 columns (NV == 2)

        // per-edge outputs: lane emit_id * (LPR / U) of the virtual warp ends up with the total of edge emit_id of a batch
        const int emit_id = (int)opaque32((uint32_t)(vl / (LPR / U)));
        const bool emit_lane = (vl % (LPR / U)) == 0;
        // per-edge combination of the gathered row (u is a compile-time constant after unrolling)
        float dd[U];  // SDDMM: this lane's partial dot products of the batch
        int drow[U];  // GAT backward: destination row of every edge of the batch (uniform over the virtual warp)
        int my_row = 0;
        // GAT backward, pass 1: (sum w, sum t) of row `srow`.  Every writer lane keeps the part of its own edges; the
        // virtual warp adds the parts up (fixed butterfly order) only when the row changes or the item ends.  The row
        // that enters the item leaves the sums in bwd_carry[item], a row that starts here in bwd_part[row].
        float s_w = 0.f, s_t = 0.f;
        int srow = -1;
        const int item32 = (int)opaque32((uint32_t)item);  // fewer than 2^31 items; kept instead of re-derived per batch
        bool s_carry = carry_in;
        auto sum_flush = [&]() {
            if (srow >= 0) {
                float tw = s_w, tt = s_t;
                const unsigned m = vmask();
#pragma unroll
                for (int off = LPR / 2; off >= 1; off >>= 1) {
                    tw += __shfl_xor_sync(m, tw, off, LPR);
                    tt += __shfl_xor_sync(m, tt, off, LPR);
                }
                if (vl == 0) {
                    if (s_carry)
                        p.bwd_carry[item32] = make_float2(tw, tt);
                    else
                        p.bwd_part[srow] = make_float2(tw, tt);
                }
                s_carry = false;
            }
            s_w = s_t = 0.f;
        };
        // GAT backward, pass 2: (alpha_e, ds_e) of the staged edge k: (w, t) through the staged position of the edge in
        // CSR order, times 1 / D_v of its destination v = the column index of the transposed CSR
        auto edge_terms = [&](const int k, float &alpha, float &ds) {
            const int pe = __float_as_int(my_val[k]);
            const float2 wt = __ldg(reinterpret_cast<const float2 *>(p.bwd_wt) + pe);
            const float inv = __ldg(&p.bwd_c[my_idx[k]].x);
            alpha = wt.x * inv;
            ds = wt.y * inv;
        };
        auto combine = [&](const int u, const float wu, const float4 &a0, const float4 &a1) {
            if (MODE == kModeMLP) {
                relu_add4(acc0, pd0, a0);
                if (NV > 1) relu_add4(acc1, pd1, a1);
            } else if (mode_emits_edges(MODE)) {
                // pd0 / pd1 of a lane without columns stay zero (load_dst), so its product vanishes without a predicate
                dd[u] = (NV > 1) ? dot4(pd0, a0) + dot4(pd1, a1) : dot4(pd0, a0);
                if (MODE == kModeGATBWD) {
                    drow[u] = row;
                    if (emit_id == u) my_row = row;  // the row of the edge this lane will write
                }
            } else {
                fma4(acc0, wu, a0);
                if (NV > 1) fma4(acc1, wu, a1);
            }
        };
        // SDDMM: totals of the batch's dot products (reduce-scatter over the virtual warp) -> out[e .. e+nb)
        // same_row: all nb edges of the batch belong to the current `row` (no row ended inside the batch)
        auto sddmm_emit = [&](const int nb, const bool same_row) {
            const int id = emit_id;
            const bool writer = emit_lane && id < nb;
            // GAT backward: everything the epilogue needs besides g_e is fetched before the shuffles
            float sv = 0.f, a_v = 0.f;
            float2 ri = make_float2(0.f, 0.f);
            if (MODE == kModeGATBWD && writer && cb + CHUNK >= F) {
                sv = (p.att != nullptr) ? __ldg(p.att + 2 * (size_t)my_idx[e + id - wbase] + 1)  // source attention term
                                        : my_val[e + id - wbase];                                  // handed-in weight
                const int v = same_row ? row : my_row;  // row of this writer's edge
                ri = __ldg(p.bwd_c + v);
                if (p.att != nullptr) a_v = __ldg(p.att + 2 * (size_t)v);
            }
            VwReduceScatter<LPR, LPR / 2, U>::run(dd, vl, vmask());
            float mw = 0.f, mt = 0.f;  // GAT backward: (w, t) of this writer's edge
            if (writer) {
                if (MODE == kModeSDDMM) {
                    float *o = p.newval + e + id;
                    *o = (cb == 0) ? dd[0] : *o + dd[0];  // wide rows: column chunks accumulate
                } else {
                    float2 *o = p.bwd_wt + e + id;
                    const float g = (cb == 0) ? dd[0] : o->y + dd[0];
                    if (cb + CHUNK < F) {
                        o->y = g;  // more column chunks to come
                    } else {
                        mw = sv;              // handed in: newval of aggr_gat_fine; s > 0 <=> w > 1
                        bool pos = sv > 1.f;
                        if (p.att != nullptr) {
                            const float sc = a_v + sv;
                            pos = sc > 0.f;
                            mw = __expf(fmaxf(sc, sc * p.slope));  // aggr_gat.h:190
                        }
                        mt = mw * (g - ri.y) * (pos ? 1.f : p.slope);  // :287-289, times D_v
                        *o = make_float2(mw, mt);
                    }
                }
            }
            if (MODE == kModeGATBWD && cb + CHUNK >= F) {
                if (same_row) {
                    if (row != srow) {
                        sum_flush();
                        srow = row;
                    }
                    s_w += mw;  // zero on the lanes that hold no edge
                    s_t += mt;
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        if (u < nb) {
                            if (drow[u] != srow) {
                                sum_flush();
                                srow = drow[u];
                            }
                            if (writer && id == u) {
                                s_w += mw;
                                s_t += mt;
                            }
                        }
                    }
                }
            }
        };

        // a batch of nb < U edges starting at e (scalar shared loads, clamped): used to re-align the first item of a
        // clipped row range and for the ragged end of the last item
        auto short_batch = [&](const int nb) {
            int src[U];
            float w[U];
            float4 v0[U], v1[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int k = min(e + u, e1 - 1) - wbase;
                src[u] = my_idx[k];
                w[u] = (mode_has_dst(MODE) || mode_gat_like(MODE)) ? 0.f : my_val[k];
            }
            float a_src = 0.f;  // GAT: source attention term of edge min(e + vl, e1 - 1), lanes vl < U
            if (MODE == kModeGAT && vl < U) a_src = __ldg(p.att + 2 * (size_t)my_idx[min(e + vl, e1 - 1) - wbase] + 1);
            float ds_lane = 0.f;  // GAT backward, pass 2: lane vl < U forms (alpha, ds) of that edge; a_src carries alpha
            if (MODE == kModeGATBWD2 && vl < U) edge_terms(min(e + vl, e1 - 1) - wbase, a_src, ds_lane);
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const char *x = xb + (size_t)(uint32_t)src[u] * row_bytes;
                v0[u] = ldg_x4<XBF16>(x);
                if (NV > 1) v1[u] = ldg_x4<XBF16>(x + second);
            }
            float wout = 0.f;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                float wu = w[u];
                const unsigned m = mode_gat_like(MODE) ? vmask() : 0u;  // fresh: a flush may lie between two of these
                if (mode_gat_like(MODE)) wu = __shfl_sync(m, a_src, u, LPR);  // all lanes of the virtual warp, every u
                float du = 0.f;
                if (MODE == kModeGATBWD2) du = __shfl_sync(m, ds_lane, u, LPR);
                if (u < nb) {
                    while (row_end == e + u) flush(false);
                    if (MODE == kModeGATBWD2) den += du;
                    if (MODE == kModeGAT) {
                        const float sc = a_dst + wu;
                        wu = __expf(fmaxf(sc, sc * p.slope));
                        den += wu;
                        if (SCHED && vl == u % LPR) wout = wu;
                    }
                    combine(u, wu, v0[u], v1[u]);
                } else if (mode_emits_edges(MODE)) {
                    dd[u] = 0.f;
                }
            }
            if (MODE == kModeGAT && SCHED && cb == 0 && p.newval != nullptr) {
                if (vl < nb) p.newval[e + vl] = wout;
            }
            if (mode_emits_edges(MODE)) sddmm_emit(nb, false);
            e += nb;
        };

        {
            const int head = min((4 - ((e - wbase) & 3)) & 3, e1 - e);  // 128-bit shared loads below need e - wbase = 0 mod 4
            if (head > 0) short_batch(head);
        }

        // ---- full batches: U edges, idx/val fetched as 128-bit shared loads
        while (e + U <= e1) {
            const int k = e - wbase;
            int src[U];
            float w[U];
#pragma unroll
            for (int q = 0; q < U / 4; ++q) {
                const int4 i4 = lds_i4(s_base + 4u * (uint32_t)(k + 4 * q));
                const float4 w4 = (mode_has_dst(MODE) || mode_gat_like(MODE))
                                      ? make_float4(0.f, 0.f, 0.f, 0.f)
                                      : lds_f4(s_base + 4u * (uint32_t)(k + 4 * q + kWarpEdges));
                src[4 * q] = i4.x, src[4 * q + 1] = i4.y, src[4 * q + 2] = i4.z, src[4 * q + 3] = i4.w;
                w[4 * q] = w4.x, w[4 * q + 1] = w4.y, w[4 * q + 2] = w4.z, w[4 * q + 3] = w4.w;
            }
            float a_src = 0.f;  // GAT: source attention term of edge e + vl (lanes vl < U), in flight with the row gathers
            if (MODE == kModeGAT && vl < U) a_src = __ldg(p.att + 2 * (size_t)my_idx[k + vl] + 1);
            float ds_lane = 0.f;  // pass 2 of the GAT backward: (alpha, ds) of edge e + vl, a_src carries alpha
            if (MODE == kModeGATBWD2 && vl < U) edge_terms(k + vl, a_src, ds_lane);
            float4 v0[U], v1[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const char *x = xb + (size_t)(uint32_t)src[u] * row_bytes;  // one IMAD.WIDE.U32
                v0[u] = ldg_x4<XBF16>(x);
                if (NV > 1) v1[u] = ldg_x4<XBF16>(x + second);
            }
            float wout = 0.f;
            const bool whole = row_end - e >= U;  // no row ends inside the batch
            if (MODE == kModeGAT && row_end - e >= U) {
                // no row ends inside the batch: lane u of the virtual warp evaluates the weight of edge u once
                // (one MUFU per edge instead of one per edge-lane) and the virtual warp shares it by shuffle
                float wgt = 0.f;
                if (vl < U) {
                    const float sc = a_dst + a_src;
                    wgt = __expf(fmaxf(sc, sc * p.slope));  // aggr_gat.h:143
                }
                const unsigned m = vmask();
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const float wu = __shfl_sync(m, wgt, u, LPR);
                    den += wu;
                    fma4(acc0, wu, v0[u]);
                    if (NV > 1) fma4(acc1, wu, v1[u]);
                }
                wout = wgt;
            } else if (MODE == kModeGATBWD2 && row_end - e >= U) {
                // the batch is summed on its own, then added to the row: the duplicate edges of a (u, v) pair give the
                // row identical terms alpha dY[v] and ds, whose rounding errors add up along one fp32 chain instead of
                // cancelling -- EB of them (512) exceed the parity gate, EB / U + U additions stay well inside it
                const unsigned m = vmask();
                float4 b0 = make_float4(0.f, 0.f, 0.f, 0.f), b1 = b0;
                float bden = 0.f;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    bden += __shfl_sync(m, ds_lane, u, LPR);
                    const float wu = __shfl_sync(m, a_src, u, LPR);
                    fma4(b0, wu, v0[u]);
                    if (NV > 1) fma4(b1, wu, v1[u]);
                }
                den += bden;
                acc0 = add4(acc0, b0);
                if (NV > 1) acc1 = add4(acc1, b1);
            } else if (!mode_gat_like(MODE) && row_end - e >= U) {
                // no row ends inside the batch: straight FMA chain (per-edge outputs: the dot products, all of row `row`)
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (mode_emits_edges(MODE))
                        dd[u] = (NV > 1) ? dot4(pd0, v0[u]) + dot4(pd1, v1[u]) : dot4(pd0, v0[u]);
                    else
                        combine(u, w[u], v0[u], v1[u]);
                }
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    while (row_end == e + u) flush(false);
                    float wu = w[u];
                    const unsigned m = mode_gat_like(MODE) ? vmask() : 0u;  // fresh: flush() above may have run
                    if (MODE == kModeGATBWD2) {
                        wu = __shfl_sync(m, a_src, u, LPR);
                        den += __shfl_sync(m, ds_lane, u, LPR);
                    }
                    if (MODE == kModeGAT) {
                        const float sc = a_dst + __shfl_sync(m, a_src, u, LPR);
                        wu = __expf(fmaxf(sc, sc * p.slope));  // aggr_gat.h:143
                        den += wu;
                        if (SCHED && vl == u % LPR) wout = wu;
                    }
                    combine(u, wu, v0[u], v1[u]);
                }
            }
            if (MODE == kModeGAT && SCHED && cb == 0 && p.newval != nullptr) {
                // one coalesced store per batch instead of one per edge (U <= LPR always holds)
                if (vl < U) p.newval[e + vl] = wout;
            }
            if (mode_emits_edges(MODE)) sddmm_emit(U, whole);
            e += U;
        }

        if (e < e1) short_batch(e1 - e);

        // item end
        if (mode_emits_edges(MODE)) {
            // per-edge outputs were written batch by batch
            if (MODE == kModeGATBWD && cb + CHUNK >= F) sum_flush();
        } else if (row_end == e1) {
            while (row < p.row_hi && row_end == e1) flush(true);  // row closes here (+ trailing empty rows)
        } else if (SCHED) {
            flush(true);
        } else if (carry_in) {
            float *c = p.carry + (size_t)item * F + col;  // row spans the whole item
            if (act0) stg_f4(c, acc0);
            if (act1) stg_f4(c + LPR * 4, acc1);
            if (mode_gat_like(MODE) && vl == 0 && cb == 0) p.carry_den[item] = den;
        } else {
            // row starts here and continues: raw partial
            float *y = p.Y + (size_t)((MODE == kModeGCN && p.out_row) ? __ldg(p.out_row + row) : row) * F + col;
            if (MODE == kModeGCN && p.accumulate) {
                if (act0) red_add_f4(y, acc0);
                if (act1) red_add_f4(y + LPR * 4, acc1);
            } else {
                if (act0) stg_f4(y, acc0);
                if (act1) stg_f4(y + LPR * 4, acc1);
            }
            if (mode_gat_like(MODE) && vl == 0 && cb == 0) p.den_row[row] = den;
        }
    }
}

// Adds the carried partials of rows that cross item boundaries, in a fixed order (deterministic).
// One virtual warp of min(32, F/4) lanes per item (F = 32: four items per warp).  Two passes so that a hub row spanning thousands of items is not summed by a
// single warp:  PHASE 1 -- every kFixChunk-th carry item of a row ("chunk head") sums its chunk of up
// to kFixChunk consecutive partials; rows whose whole span fits one chunk are finished here.
// PHASE 2 -- one warp per long row adds the chunk heads and finishes the row.
constexpr int kFixChunk = 32;

// sums carry[b0], carry[b0+step], ... carry[<= b1] (and the denominators) in that order; `finish` adds the total to
// Y[row] (GAT: and normalises), otherwise the total replaces carry[item]
template <int MODE>
__device__ __forceinline__ void fixup_sum(const AggParams &p, int row, int64_t item, int64_t b0, int64_t b1, int64_t step,
                                          bool finish, int lane, int lanes = 32)
{
    const int F = p.F;
    float dsum = 0.f, inv = 1.f;
    if (mode_gat_like(MODE)) {
        for (int64_t b = b0; b <= b1; b += step) dsum += p.carry_den[b];
        if (finish) {
            dsum += p.den_row[row];
            inv = (dsum != 0.f) ? __fdividef(1.f, dsum) : 0.f;
            if (MODE == kModeGATBWD2 && lane == 0) p.rsum[(size_t)row * p.rsum_stride] = dsum;  // a plain row sum
        }
    }
    for (int col = lane * 4; col < F; col += lanes * 4) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int64_t b = b0;
        for (; b + 3 * step <= b1; b += 4 * step) {
            const float4 c0 = *reinterpret_cast<const float4 *>(p.carry + (size_t)b * F + col);
            const float4 c1 = *reinterpret_cast<const float4 *>(p.carry + (size_t)(b + step) * F + col);
            const float4 c2 = *reinterpret_cast<const float4 *>(p.carry + (size_t)(b + 2 * step) * F + col);
            const float4 c3 = *reinterpret_cast<const float4 *>(p.carry + (size_t)(b + 3 * step) * F + col);
            acc = add4(add4(add4(add4(acc, c0), c1), c2), c3);
        }
        for (; b <= b1; b += step) acc = add4(acc, *reinterpret_cast<const float4 *>(p.carry + (size_t)b * F + col));
        if (finish) {
            float *y = p.Y + (size_t)((MODE == kModeGCN && p.out_row) ? __ldg(p.out_row + row) : row) * F + col;
            if (MODE == kModeGCN || MODE == kModeGATBWD2) {
                red_add_f4(y, acc);  // one add per element and launch: deterministic, and no wait for Y
            } else {
                acc = add4(*reinterpret_cast<const float4 *>(y), acc);
                if (MODE == kModeGAT) acc = make_float4(acc.x * inv, acc.y * inv, acc.z * inv, acc.w * inv);
                stg_f4(y, acc);
            }
        } else {
            stg_f4(p.carry + (size_t)item * F + col, acc);  // chunk head now holds the chunk sum
        }
    }
    if (mode_gat_like(MODE) && !finish && lane == 0) p.carry_den[item] = dsum;
}

// PHASE 1: one warp per item of the launched range.  What an item has to do depends on the graph and the item size
// only, so it is looked up in a record built once (fixup_records_kernel): x = row entering the item if the item is a
// chunk head, else -1; y = number of partials in its chunk, negated when the chunk is the whole span (row finished here).
// One dependent load instead of the item_row -> ptr[row], ptr[row+1] chain in front of the carry loads.
template <int MODE>
__global__ void __launch_bounds__(256) agg_fixup_kernel(const AggParams p, int EB, int64_t num_items,
                                                        const int2 *__restrict__ records, int lanes)
{
    griddep_wait();
    // items of the launched edge range only; the first one is clipped at a row start, so nothing enters it
    const int64_t item = (int64_t)(p.edge_lo / EB) + ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / lanes;
    if (item < 1 || item >= num_items || item * EB >= p.edge_hi || item * EB <= p.edge_lo) return;
    const int2 rec = __ldg(records + item);
    if (rec.x < 0) return;  // no row enters this item, or it is not a chunk head
    const int size = rec.y < 0 ? -rec.y : rec.y;
    fixup_sum<MODE>(p, rec.x, item, item, item + size - 1, 1, rec.y < 0, threadIdx.x % lanes, lanes);
}

__global__ void __launch_bounds__(256) fixup_records_kernel(const AggParams p, int EB, int64_t num_items, int2 *__restrict__ records)
{
    const int64_t item = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (item >= num_items) return;
    int2 rec = make_int2(-1, 0);
    if (item >= 1) {
        const int e0 = (int)(item * EB);
        const int row = item_start_row(p, e0);
        const int rs = __ldg(p.ptr + row);
        if (rs < e0) {
            const int64_t first = (int64_t)(rs / EB) + 1;                       // first carry item of that row
            const int64_t last = (int64_t)(__ldg(p.ptr + row + 1) - 1) / EB;    // item holding the row's last edge
            if ((item - first) % kFixChunk == 0) {
                const int size = (int)(min(last, item + kFixChunk - 1) - item + 1);
                rec = make_int2(row, (last - first) < kFixChunk ? -size : size);
            }
        }
    }
    records[item] = rec;
}

// PHASE 2: one warp per LONG row (more than kFixChunk carry items; the list is built once per graph and item size by
// long_rows_kernel).  Launching it over all items cost 0.06 ms on C2 for a few hundred rows with work.
template <int MODE>
__global__ void __launch_bounds__(256) agg_fixup_long_kernel(const AggParams p, int EB, const int *__restrict__ long_rows,
                                                             int num_long)
{
    griddep_wait();
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= num_long) return;
    const int row = __ldg(long_rows + w);
    if (row < p.row_lo || row >= p.row_hi) return;
    const int64_t first = (int64_t)(__ldg(p.ptr + row) / EB) + 1;
    const int64_t last = (int64_t)(__ldg(p.ptr + row + 1) - 1) / EB;
    fixup_sum<MODE>(p, row, first, first, last, kFixChunk, true, threadIdx.x & 31);
}

// rows whose carry items number more than kFixChunk (any order)
__global__ void __launch_bounds__(256) long_rows_kernel(const int *__restrict__ ptr, int num_rows, int EB,
                                                        int *__restrict__ list, int *__restrict__ count)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= num_rows) return;
    const int rs = __ldg(ptr + r), re = __ldg(ptr + r + 1);
    if (re <= rs) return;
    const int64_t first = (int64_t)(rs / EB) + 1, last = (int64_t)(re - 1) / EB;
    if (last - first >= kFixChunk) list[atomicAdd(count, 1)] = r;
}

// scheduled GAT epilogue: Y[v,:] /= den[v] when den != 0  (scaleArray, aggr_gat.h:207-213)
__global__ void __launch_bounds__(256) gat_scale_kernel(float *__restrict__ Y, const float *__restrict__ den, int F,
                                                        int64_t total4)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int64_t row = (i * 4) / F;
    const float d = __ldg(den + row);
    if (d != 0.f) {
        float4 v = reinterpret_cast<float4 *>(Y)[i];
        const float inv = __fdividef(1.f, d);
        v = make_float4(v.x * inv, v.y * inv, v.z * inv, v.w * inv);
        reinterpret_cast<float4 *>(Y)[i] = v;
    }
}

// row containing edge k*kFineItem, for every k (one thread each)
__global__ void __launch_bounds__(256) item_row_kernel(const int *__restrict__ ptr, int num_rows, int num_edges,
                                                       int *__restrict__ item_row, int num_items)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= num_items) return;
    const int64_t e64 = (int64_t)k * kFineItem;
    const int e = (int)(e64 < num_edges ? e64 : num_edges - 1);
    int lo = 0, hi = num_rows - 1;  // last r with ptr[r] <= e
    while (lo < hi) {
        const int mid = (int)(((int64_t)lo + hi + 1) >> 1);
        if (__ldg(ptr + mid) <= e)
            lo = mid;
        else
            hi = mid - 1;
    }
    item_row[k] = lo;
}

}  // namespace gnnagg
