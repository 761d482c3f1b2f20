// dist.cu -- multi-GPU aggregation over NVLink peer memory (gnnagg_dist_*, SURVEY.md 8(e)).
//
// The reference is single-GPU: every driver asserts GPUNUM == 1 (Figure9/main.cu:19) and the multi-GPU
// leftovers (GPUNUM/gptrs/gidxs globals, syncAll: include/util.h:39-57,135-142; prepare*Multi prototypes:
// include/data.h:48-58) have no implementation.  What is built here: the graph is 1-D partitioned by
// destination row; rank r owns a row block and the matching shard of X.  The only exchange step is the
// source-feature halo.  It is NOT a library collective:
//
//   * at set-up each rank finds the distinct REMOTE source rows its block references (mark / scan / fill on the
//     GPU), re-indexes its CSR into [own shard rows | receive slots] coordinates -- the receive buffer sits right
//     behind the shard, so one base pointer serves both -- and splits it by the OWNER of the source into stages
//     (the slices of locality_schedule, graph_schedule.h:24-29, kept as CSRs).  Shard, receive buffer, the list
//     of wanted rows and a page of flags live in ONE peer-visible allocation (same process: peer access; one
//     process per GPU: a cudaIpc handle, exchanged once).  At connect time every owner copies, once, the lists
//     of rows its peers want from it;
//   * a step: every OWNER pushes.  halo_push_kernel gathers the wanted rows from its own shard (local HBM, local
//     TLB) and writes them with 128-bit stores straight into the receiver's buffer over NVLink -- posted writes
//     into a contiguous destination, no pack buffer, no NCCL, no read round trips (a first version PULLED the rows
//     with remote loads and reached 300-400 GB/s per GPU; profiles/r2_sweep_n8_pull.jsonl).  Owner p serves the
//     receivers in the order p-1, p-2, ..., so at any time every receiver is written by exactly one owner;
//   * the receiver aggregates stage 0 (edges whose source is local) meanwhile, and stage s as soon as the owners
//     of that stage have landed (gnnagg_gcn_run_acc, deterministic).  remote_stages = 0 runs ONE pass after all
//     arrivals: no extra pass over Y, for graphs whose rows are too short to pay for it.
//   Cross-GPU ordering is two epoch flags per pair in peer-visible memory: arrived[p] at the receiver ("owner p's
//   rows of epoch e are in your buffer": the last CTA of the push kernel, after a system-scope fence) and
//   consumed[q] at the owner ("receiver q has finished reading what you pushed in epoch e": write-after-read
//   protection of q's buffer).  Spins are one-warp kernels, bounded by globaltimer, and report through an error word.
#include <cub/cub.cuh>
#include <cuda_runtime.h>
#include <unistd.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "common.cuh"
#include "gnnagg.h"
#include "internal.h"

namespace gnnagg {

constexpr int kMaxWorld = GNNAGG_DIST_MAX_WORLD;
constexpr uint64_t kSpinLimitNs = 20ull * 1000 * 1000 * 1000;  // a peer that does not answer within 20 s is reported
constexpr size_t kFlagBytes = 512;
constexpr int kMaxRounds = 16;          // row chunks of the row-pipelined mode
constexpr size_t kMetaBytes = 1536;     // int recv_tab[kMaxRounds][kMaxWorld + 1] behind the flags, read by the owners at connect

struct HaloFlags {
    uint32_t arrived[kMaxWorld];   // arrived[p]: last epoch whose rows owner p has written into MY receive buffer (written by p)
    uint32_t consumed[kMaxWorld];  // consumed[q]: last epoch receiver q finished reading what I pushed to it (written by q)
    uint32_t push_cnt[kMaxWorld];  // local: CTAs of the running push kernel towards q that are done
    uint32_t err;                  // first protocol error seen by a kernel of this rank (0 = none)
};
static_assert(sizeof(HaloFlags) <= kFlagBytes, "flags page too small");

struct PeerTable {
    HaloFlags *flags[kMaxWorld];
};
struct Bounds {
    int64_t b[kMaxWorld + 1];
    int stage_of[kMaxWorld];
    int world;
};

#define DT_TRY(expr)                                                                                          \
    do {                                                                                                      \
        cudaError_t _e = (expr);                                                                              \
        if (_e != cudaSuccess) {                                                                              \
            char _buf[512];                                                                                   \
            snprintf(_buf, sizeof _buf, "%s:%d %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return set_error(GNNAGG_ERR_CUDA, _buf);                                                          \
        }                                                                                                     \
    } while (0)

__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint64_t global_ns()
{
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// waits until *flag has reached `epoch`; gives up after kSpinLimitNs and records `code` in *err
__device__ __forceinline__ bool spin_until(const uint32_t *flag, uint32_t epoch, uint32_t *err, uint32_t code)
{
    if ((int32_t)(ld_acquire_sys(flag) - epoch) >= 0) return true;
    const uint64_t t0 = global_ns();
    while ((int32_t)(ld_acquire_sys(flag) - epoch) < 0) {
        __nanosleep(128);
        if (global_ns() - t0 > kSpinLimitNs) {
            atomicCAS(err, 0u, code);
            return false;
        }
    }
    return true;
}

// start of a step at the OWNER: every receiver must have finished reading what was pushed to it in the previous epoch
// before its buffer is written again
__global__ void __launch_bounds__(32) halo_begin_kernel(HaloFlags *mine, int rank, int world, uint32_t epoch)
{
    const int q = threadIdx.x;
    if (q < world && q != rank) spin_until(&mine->consumed[q], epoch - 1u, &mine->err, 0x100u + (uint32_t)q);
}

// at the RECEIVER, in front of a stage: the rows of the owners in `mask` have landed
__global__ void __launch_bounds__(32) halo_wait_kernel(HaloFlags *mine, uint32_t mask, uint32_t epoch)
{
    const int p = threadIdx.x;
    if (p < kMaxWorld && ((mask >> p) & 1u)) spin_until(&mine->arrived[p], epoch, &mine->err, (uint32_t)p);
}

// end of a step at the RECEIVER: tell every owner that its rows of this epoch have been read
__global__ void __launch_bounds__(32) halo_consumed_kernel(PeerTable peers, int rank, int world, uint32_t epoch)
{
    const int p = threadIdx.x;
    if (p < world && p != rank) st_release_sys(&peers.flags[p]->consumed[rank], epoch);
}

// dst[i, :] = X[rows[i], :] for the `count` rows receiver q wants from this owner (in this round): X is the own shard
// (local gathers), dst the slice of q's receive slots reserved for them (peer memory: the stores travel over NVLink, or
// stay local when the "peer" lives on the same device).  The last CTA to finish publishes `value` in q's arrived[] flag.
// Built to run BESIDE the aggregation kernel, not instead of it: 128 threads and at most 32 registers, so a CTA fits
// into what three aggregation CTAs (3 x 256 threads x 80 registers) leave free on an SM; the first version (256 threads,
// 8 loads in flight per thread, 2 CTAs per SM) displaced one aggregation CTA per SM for as long as the exchange ran.
// Posted writes need no latency hiding; U loads per thread cover the local gather latency.
// The rows are copied in units of T, whatever they hold: float4 for fp32 rows and for bf16 rows of a width that is a
// multiple of 8; uint2 for bf16 rows of a width that is 4 mod 8 (F = 100: 200 bytes, 8-byte aligned only).  FU = units
// per row, fu_shift = log2(FU) when FU is a power of two (else -1), units = rows x FU.
template <typename T, int U, bool PREFETCH>
__global__ void __launch_bounds__(128, 16) halo_push_kernel(const T *__restrict__ X, const int *__restrict__ rows,
                                                            T *__restrict__ dst, int64_t units, int FU, int fu_shift,
                                                            uint32_t *done_cnt, uint32_t *arrived_flag, uint32_t value)
{
    const int64_t stride = (int64_t)gridDim.x * 128 * U;
    for (int64_t base = (int64_t)blockIdx.x * 128 * U + threadIdx.x; base < units; base += stride) {
        if (PREFETCH) {
            // the rows of the NEXT iteration are pulled into L2 now: prefetches hold no registers, so the kernel has twice
            // its load depth in flight where the memory system is busy with the aggregation's gathers
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t e = base + stride + (int64_t)u * 128;
                if (e < units && (e & (int64_t)(128 / sizeof(T) - 1)) == 0) {  // one prefetch per 128-byte line
                    const int64_t r = (fu_shift >= 0) ? (e >> fu_shift) : (e / FU);
                    const int c = (int)(e - r * FU);
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(X + (int64_t)__ldg(rows + r) * FU + c));
                }
            }
        }
        T v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t e = base + (int64_t)u * 128;
            if (e < units) {
                const int64_t r = (fu_shift >= 0) ? (e >> fu_shift) : (e / FU);
                const int c = (int)(e - r * FU);
                v[u] = __ldg(X + (int64_t)__ldg(rows + r) * FU + c);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t e = base + (int64_t)u * 128;
            if (e < units) dst[e] = v[u];
        }
    }
    // every thread's stores are ordered before this CTA's count, the count before the flag (system scope)
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t before = atomicAdd(done_cnt, 1u);
        if (before == gridDim.x - 1) {
            atomicExch(done_cnt, 0u);  // ready for the next launch towards this receiver (stream-ordered after this one)
            __threadfence_system();
            st_release_sys(arrived_flag, value);
        }
    }
}

// the same loop without the register diet: 256 threads, U = 8 loads in flight per thread (GNNAGG_PUSH_HEAVY=1; it displaces
// aggregation CTAs instead of running beside them)
template <int U>
__global__ void __launch_bounds__(256) halo_push_heavy_kernel(const float4 *__restrict__ X, const int *__restrict__ rows,
                                                            float4 *__restrict__ dst, int64_t count4, int F4, int f4_shift,
                                                            uint32_t *done_cnt, uint32_t *arrived_flag, uint32_t value)
{
    const int64_t stride = (int64_t)gridDim.x * 256 * U;
    for (int64_t base = (int64_t)blockIdx.x * 256 * U + threadIdx.x; base < count4; base += stride) {
        if (false) {
            // the rows of the NEXT iteration are pulled into L2 now: prefetches hold no registers, so the kernel has twice
            // its load depth in flight where the memory system is busy with the aggregation's gathers
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int64_t e = base + stride + (int64_t)u * 256;
                if (e < count4 && (e & 7) == 0) {  // one prefetch per 128-byte line
                    const int64_t r = (f4_shift >= 0) ? (e >> f4_shift) : (e / F4);
                    const int c = (int)(e - r * F4);
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(X + (int64_t)__ldg(rows + r) * F4 + c));
                }
            }
        }
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t e = base + (int64_t)u * 256;
            if (e < count4) {
                const int64_t r = (f4_shift >= 0) ? (e >> f4_shift) : (e / F4);
                const int c = (int)(e - r * F4);
                v[u] = __ldg(X + (int64_t)__ldg(rows + r) * F4 + c);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t e = base + (int64_t)u * 256;
            if (e < count4) dst[e] = v[u];
        }
    }
    // every thread's stores are ordered before this CTA's count, the count before the flag (system scope)
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t before = atomicAdd(done_cnt, 1u);
        if (before == gridDim.x - 1) {
            atomicExch(done_cnt, 0u);  // ready for the next launch towards this receiver (stream-ordered after this one)
            __threadfence_system();
            st_release_sys(arrived_flag, value);
        }
    }
}

// EXPERIMENT, off by default (GNNAGG_PUSH_TMA=1 selects it): the same push with the rows STAGED THROUGH SHARED MEMORY BY
// THE TMA ENGINE.  One warp per CTA keeps a ring of kPushBufs batches (<= 8 KB each) in flight -- every lane issues one
// 1-D bulk copy (cp.async.bulk, global -> shared) for one wanted row onto the batch's mbarrier; when the batch has
// landed ONE bulk copy (shared -> global) writes it to the receiver's contiguous slots over NVLink.  32 threads, 28
// registers, bytes in flight bounded by shared memory instead of registers.  Measured on 8 B200s it LOSES to the register
// version (profiles/r2_sweep_n8_push_v3_tma.jsonl vs r2_sweep_n8_push_v2_light.jsonl: reddit-shape step 4.20 vs 3.48 ms,
// RMAT-26 exchange alone 569 vs 615 GB/s): its 48 KB of shared memory per CTA changes the SM's L1 / shared-memory
// split, and the SM drains before kernels with different splits can share it -- the push stops running BESIDE the
// aggregation, which was the point.  Kept selectable as the evidence for that conclusion.
constexpr int kPushBufs = 6;        // ring depth
constexpr int kPushAhead = 4;       // batches of loads in flight per warp
constexpr int kPushBatchBytes = 8192;

__device__ __forceinline__ void bulk_s2g(void *dst, uint32_t src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read()
{
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__global__ void __launch_bounds__(32) halo_push_tma_kernel(const float *__restrict__ X, const int *__restrict__ rows,
                                                           float *__restrict__ dst, int64_t count, int F, int rows_per_batch,
                                                           uint32_t *done_cnt, uint32_t *arrived_flag, uint32_t value)
{
    extern __shared__ __align__(128) uint8_t push_smem[];
    __shared__ __align__(8) uint64_t bars[kPushBufs];
    const int lane = threadIdx.x;
    const uint32_t row_bytes = (uint32_t)F * 4u;
    const int64_t batches = (count + rows_per_batch - 1) / rows_per_batch;
    const int64_t mine = batches > blockIdx.x ? (batches - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;  // batches of this warp
    if (lane == 0) {
        for (int i = 0; i < kPushBufs; ++i) mbar_init(smem_u32(&bars[i]), 1);
        fence_mbar_init();
    }
    __syncwarp();
    // loads of this warp's j-th batch into ring slot j % kPushBufs
    auto issue = [&](int64_t j) {
        const int buf = (int)(j % kPushBufs);
        const int64_t r0 = (blockIdx.x + j * gridDim.x) * rows_per_batch;
        const int nr = (int)min((int64_t)rows_per_batch, count - r0);
        const uint32_t bar = smem_u32(&bars[buf]);
        if (lane == 0) mbar_expect_tx(bar, (uint32_t)nr * row_bytes);
        __syncwarp();
        if (lane < nr)
            bulk_g2s(smem_u32(push_smem) + (uint32_t)buf * kPushBatchBytes + (uint32_t)lane * row_bytes,
                     X + (size_t)__ldg(rows + r0 + lane) * F, row_bytes, bar);
    };
    for (int64_t j = 0; j < kPushAhead && j < mine; ++j) issue(j);
    for (int64_t it = 0; it < mine; ++it) {
        if (it + kPushAhead < mine) {
            // slot (it + kPushAhead) % kPushBufs was last stored from kPushBufs - kPushAhead iterations ago: that bulk store
            // must have finished READING shared memory (not the remote write) before the TMA overwrites it
            if (lane == 0) bulk_wait_read<kPushBufs - kPushAhead - 1>();
            __syncwarp();
            issue(it + kPushAhead);
        }
        const int buf = (int)(it % kPushBufs);
        mbar_wait(smem_u32(&bars[buf]), (uint32_t)((it / kPushBufs) & 1));
        if (lane == 0) {
            const int64_t r0 = (blockIdx.x + it * gridDim.x) * rows_per_batch;
            const int nr = (int)min((int64_t)rows_per_batch, count - r0);
            bulk_s2g(dst + (size_t)r0 * F, smem_u32(push_smem) + (uint32_t)buf * kPushBatchBytes, (uint32_t)nr * row_bytes);
            bulk_commit();
        }
    }
    if (lane == 0) {
        bulk_wait_all();  // every bulk store of this warp has been performed
        asm volatile("fence.proxy.async;" ::: "memory");
        __threadfence_system();
        const uint32_t before = atomicAdd(done_cnt, 1u);
        if (before == gridDim.x - 1) {
            atomicExch(done_cnt, 0u);
            __threadfence_system();
            st_release_sys(arrived_flag, value);
        }
    }
}

// ---- set-up kernels: which remote rows does this block reference, and where do they land -------------------
__device__ __forceinline__ int owner_of(const Bounds &b, int64_t g)
{
    int p = 0;
    while (p + 1 < b.world && g >= b.b[p + 1]) ++p;
    return p;
}

__global__ void __launch_bounds__(256) dist_mark_kernel(const int *__restrict__ idx, int64_t m, int64_t own_lo, int64_t own_hi,
                                                        int64_t total, int *__restrict__ mark, int *__restrict__ bad)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int64_t g = __ldg(idx + e);
    if (g < 0 || g >= total)
        *bad = 1;
    else if (g < own_lo || g >= own_hi)
        mark[g] = 1;
}

__global__ void __launch_bounds__(256) dist_fill_recv_kernel(const int *__restrict__ mark, const int *__restrict__ pos, int64_t total,
                                                             Bounds b, int *__restrict__ recv_local)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total || !mark[g]) return;
    recv_local[pos[g]] = (int)(g - b.b[owner_of(b, g)]);
}

// new index of every edge -- local row of the own shard, or `rows_own + receive slot` -- and its stage
__global__ void __launch_bounds__(256) dist_reindex_kernel(const int *__restrict__ idx, int64_t m, const int *__restrict__ pos,
                                                           int64_t own_lo, int64_t own_hi, int rows_own, Bounds b,
                                                           int *__restrict__ idx_new, int *__restrict__ keys)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int64_t g = __ldg(idx + e);
    if (g >= own_lo && g < own_hi) {
        idx_new[e] = (int)(g - own_lo);
        keys[e] = 0;
    } else {
        idx_new[e] = rows_own + __ldg(pos + g);
        keys[e] = b.stage_of[owner_of(b, g)];
    }
}

// ---- row-pipelined mode: the round (row chunk) in which every remote source is needed first
struct ChunkRows {
    int lo[kMaxRounds + 1];
    int rounds;
};

__global__ void __launch_bounds__(256) dist_first_use_kernel(const int *__restrict__ ptr, const int *__restrict__ idx,
                                                             const int *__restrict__ item_row, int num_items, int n, int64_t m,
                                                             int64_t own_lo, int64_t own_hi, int64_t total, ChunkRows cr,
                                                             int *__restrict__ first, int *__restrict__ bad)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int64_t g = __ldg(idx + e);
    if (g < 0 || g >= total) {
        *bad = 1;
        return;
    }
    if (g >= own_lo && g < own_hi) return;
    const int row = row_of_edge(ptr, item_row, num_items, n, (int)e);
    int c = 0;
    while (c + 1 < cr.rounds && row >= cr.lo[c + 1]) ++c;
    atomicMin(first + g, c);
}

__global__ void __launch_bounds__(256) dist_round_mark_kernel(const int *__restrict__ first, int64_t total, int round, int any,
                                                              int *__restrict__ mark)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g > total) return;
    mark[g] = (g < total && (any ? first[g] < kMaxRounds + 1 : first[g] == round)) ? 1 : 0;
}

// receive slots of round `round` start at `base`; inside a round ascending global id (owner by owner)
__global__ void __launch_bounds__(256) dist_round_fill_kernel(const int *__restrict__ mark, const int *__restrict__ pos, int64_t total,
                                                              Bounds b, int base, int *__restrict__ recv_local, int *__restrict__ slot)
{
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= total || !mark[g]) return;
    const int s = base + pos[g];
    recv_local[s] = (int)(g - b.b[owner_of(b, g)]);
    slot[g] = s;
}

__global__ void __launch_bounds__(256) dist_reindex_slot_kernel(const int *__restrict__ idx, int64_t m, const int *__restrict__ slot,
                                                                int64_t own_lo, int64_t own_hi, int rows_own,
                                                                int *__restrict__ idx_new, int *__restrict__ keys)
{
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int64_t g = __ldg(idx + e);
    idx_new[e] = (g >= own_lo && g < own_hi) ? (int)(g - own_lo) : rows_own + __ldg(slot + g);
    keys[e] = 0;
}

__global__ void __launch_bounds__(256) dist_fill_int_kernel(int *__restrict__ out, int64_t count, int value)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = value;
}

__global__ void __launch_bounds__(256) dist_gather_val_kernel(const float *__restrict__ val, const int *__restrict__ perm,
                                                              float *__restrict__ out, int count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = __ldg(val + __ldg(perm + i));
}

static inline unsigned nblocks(int64_t n) { return (unsigned)((n + 255) / 256); }
static inline size_t round512(size_t b) { return (b + 511) & ~(size_t)511; }

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard()
    {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

}  // namespace gnnagg

using namespace gnnagg;

constexpr int kMaxStages = kMaxWorld;

// what a rank publishes to its peers after gnnagg_dist_set_graph (gnnagg_dist_export): fits GNNAGG_DIST_BLOB_BYTES
struct DistBlob {
    uint32_t magic;
    int rank, world, device, pid;
    int feat_cap;
    int64_t rows;
    uint64_t raw_base;  // usable as is inside the exporting process
    uint64_t bytes;
    uint64_t off_x[2], off_req, off_meta;
    int rounds;  // 1, or the row chunks of the row-pipelined mode: rows of recv_tab (in the buffer, at off_meta) in use
    cudaIpcMemHandle_t mem;
};
static_assert(sizeof(DistBlob) <= GNNAGG_DIST_BLOB_BYTES, "blob too large");

struct gnnagg_dist {
    int rank = 0, world = 1, device = 0, pid = 0;
    int64_t bounds[kMaxWorld + 1] = {0};
    int rows = 0;  // rows of the own shard = rows of the CSR block
    int feat_cap = 0;
    // peer-visible allocation (made by set_graph): [flags | wanted-row list | x0 + receive 0 | x1 + receive 1]
    char *base = nullptr;
    size_t bytes = 0, off_x[2] = {0, 0}, off_req = 0, off_meta = 0;
    // peers as seen from this rank
    char *peer_base[kMaxWorld] = {nullptr};
    size_t peer_off_x[kMaxWorld][2] = {{0, 0}};
    int peer_rows[kMaxWorld] = {0};         // rows of q's shard: its receive buffer starts that many rows behind its x
    int peer_slot[kMaxWorld][kMaxRounds] = {{0}};  // first receive slot of q's buffer for this owner's rows of round c
    int send_cnt[kMaxWorld][kMaxRounds] = {{0}};   // rows q wants from this owner in round c
    int send_off[kMaxWorld][kMaxRounds] = {{0}};   // where they start inside send_rows[q]
    int *send_rows[kMaxWorld] = {nullptr};         // which ones (local row numbers; owned copy of q's lists, round by round)
    bool peer_ipc[kMaxWorld] = {false};
    bool connected = false;
    // plan
    int64_t num_e = 0;
    int remote_stages = 0, num_stages = 0;  // R = 0: one pass; else stage 0 = local sources, 1..R = groups of owners
    int stage_of[kMaxWorld] = {0};
    uint32_t stage_mask[kMaxStages] = {0};  // owners whose arrival a stage waits for
    int64_t num_recv = 0;
    // rounds = 1: receive slots ascending by global id (owner by owner).  Row-pipelined mode (rounds = K row chunks):
    // slots ordered by the round in which a row is needed first, then by id; recv_tab[c][p] = first slot of owner p's
    // rows of round c, recv_tab[c][world] = end of round c
    int rounds = 1;
    int recv_tab[kMaxRounds][kMaxWorld + 1] = {{0}};
    int chunk_rows[kMaxRounds + 1] = {0};
    int64_t recv_cnt[kMaxWorld] = {0};
    // sub-CSRs, one per stage
    int *sl_ptr = nullptr, *sl_idx = nullptr, *sl_perm = nullptr;
    float *sl_val = nullptr;
    int sl_off[kMaxStages] = {0}, sl_cnt[kMaxStages] = {0};
    gnnagg_aggregator *stage[kMaxStages] = {nullptr};
    float *ax = nullptr;
    size_t ax_cap = 0;
    // host-buffer entry point: device staging of W and of the result, copy-back stream
    float *st_w = nullptr, *st_out = nullptr;
    size_t st_w_cap = 0, st_out_cap = 0;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t chunk_done[4] = {nullptr, nullptr, nullptr, nullptr}, copies_done = nullptr;
    // step machinery
    cudaStream_t comm = nullptr;
    cudaEvent_t ev_sig = nullptr, ev_done = nullptr;
    cudaEvent_t t_m0 = nullptr, t_m1 = nullptr, t_m2 = nullptr, t_m3 = nullptr, t_c0 = nullptr, t_c1 = nullptr;
    bool prof = false;
    uint32_t epoch = 0;
    int sm_count = 148;
    int prepared_feat = 0;
    int push_heavy = 0;         // k > 0: 256-thread / 8-loads push kernel with up to k CTAs per SM (experiment)
    int push_prefetch = 0;      // 1: the register push kernel prefetches the next iteration's rows into L2
    int push_tma = 0;           // 1: rows staged through shared memory by bulk copies (halo_push_tma_kernel); 0: register version
    int same_device_ranks = 1;  // ranks (including this one) living on this rank's device: > 1 only in single-GPU tests
    int64_t launches = 0;
};

static HaloFlags *flags_of(char *base) { return reinterpret_cast<HaloFlags *>(base); }

static void close_peers(gnnagg_dist *d)
{
    for (int p = 0; p < d->world; ++p) {
        if (p != d->rank && d->peer_base[p] && d->peer_ipc[p]) cudaIpcCloseMemHandle(d->peer_base[p]);
        if (p != d->rank) d->peer_base[p] = nullptr;
        d->peer_ipc[p] = false;
        cudaFree(d->send_rows[p]);
        d->send_rows[p] = nullptr;
        for (int c = 0; c < kMaxRounds; ++c) d->send_cnt[p][c] = 0;
    }
    d->connected = d->world == 1 && d->base != nullptr;
}

static void free_graph(gnnagg_dist *d)
{
    close_peers(d);
    for (int s = 0; s < kMaxStages; ++s) {
        if (d->stage[s]) gnnagg_destroy(d->stage[s]);
        d->stage[s] = nullptr;
    }
    cudaFree(d->sl_ptr), cudaFree(d->sl_idx), cudaFree(d->sl_perm), cudaFree(d->sl_val);
    cudaFree(d->base);
    d->sl_ptr = d->sl_idx = d->sl_perm = nullptr;
    d->sl_val = nullptr;
    d->base = nullptr;
    d->bytes = 0;
    d->num_stages = 0;
    d->num_recv = 0;
    d->prepared_feat = 0;
    d->connected = false;
    d->peer_base[d->rank] = nullptr;
}

extern "C" {

int gnnagg_dist_create_rank(int rank, int world, const int64_t *shard_bounds, int feat_cap, gnnagg_dist **out)
{
    if (!out || !shard_bounds || world < 1 || world > kMaxWorld || rank < 0 || rank >= world || feat_cap < 4 || (feat_cap & 3))
        return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_create_rank: bad argument (world <= 16, feat_cap a multiple of 4)");
    for (int p = 0; p < world; ++p)
        if (shard_bounds[p + 1] < shard_bounds[p] || shard_bounds[0] != 0)
            return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_create_rank: shard_bounds must start at 0 and ascend");
    if (shard_bounds[world] > INT32_MAX) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_create_rank: source ids are int32");
    gnnagg_dist *d = new gnnagg_dist();
    d->rank = rank;
    d->world = world;
    d->pid = (int)getpid();
    d->feat_cap = feat_cap;
    memcpy(d->bounds, shard_bounds, sizeof(int64_t) * (size_t)(world + 1));
    d->rows = (int)(shard_bounds[rank + 1] - shard_bounds[rank]);
    auto fail = [&](cudaError_t e, const char *what) {
        char buf[256];
        snprintf(buf, sizeof buf, "gnnagg_dist_create_rank: %s: %s", what, cudaGetErrorString(e));
        delete d;
        return set_error(GNNAGG_ERR_CUDA, buf);
    };
    cudaError_t e = cudaGetDevice(&d->device);
    if (e != cudaSuccess) return fail(e, "cudaGetDevice");
    cudaDeviceGetAttribute(&d->sm_count, cudaDevAttrMultiProcessorCount, d->device);
    int lo = 0, hi = 0;
    cudaDeviceGetStreamPriorityRange(&lo, &hi);  // hi = numerically lowest = highest priority
    e = cudaStreamCreateWithPriority(&d->comm, cudaStreamNonBlocking, hi);
    if (e != cudaSuccess) return fail(e, "cudaStreamCreateWithPriority");
    cudaEventCreateWithFlags(&d->ev_sig, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&d->ev_done, cudaEventDisableTiming);
    {  // load the step's kernels now: a first launch while a peer's kernels spin on this rank could wait forever
        cudaFuncAttributes attr;
        if (cudaFuncGetAttributes(&attr, halo_begin_kernel) != cudaSuccess) cudaGetLastError();
        if (cudaFuncGetAttributes(&attr, halo_wait_kernel) != cudaSuccess) cudaGetLastError();
        if (cudaFuncGetAttributes(&attr, halo_consumed_kernel) != cudaSuccess) cudaGetLastError();
        if (cudaFuncGetAttributes(&attr, halo_push_kernel<float4, 4, false>) != cudaSuccess) cudaGetLastError();
        if (cudaFuncGetAttributes(&attr, halo_push_kernel<uint2, 4, false>) != cudaSuccess) cudaGetLastError();  // bf16, F = 4 mod 8
        if (cudaFuncGetAttributes(&attr, halo_push_kernel<float4, 4, true>) != cudaSuccess) cudaGetLastError();
        if (const char *env = getenv("GNNAGG_PUSH_PREFETCH")) d->push_prefetch = atoi(env) != 0;
        if (cudaFuncGetAttributes(&attr, halo_push_heavy_kernel<8>) != cudaSuccess) cudaGetLastError();
        if (const char *env = getenv("GNNAGG_PUSH_HEAVY")) d->push_heavy = atoi(env);
        if (cudaFuncGetAttributes(&attr, halo_push_tma_kernel) != cudaSuccess) cudaGetLastError();
        if (cudaFuncSetAttribute(halo_push_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kPushBufs * kPushBatchBytes) != cudaSuccess)
            cudaGetLastError();
        if (const char *env = getenv("GNNAGG_PUSH_TMA")) d->push_tma = atoi(env) != 0;
        dense_preload();
    }
    *out = d;
    return GNNAGG_OK;
}

int gnnagg_dist_create(int world, const int *devices, const int64_t *shard_bounds, int feat_cap, gnnagg_dist **out)
{
    if (!out || world < 1 || world > kMaxWorld) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_create: bad argument");
    int prev = 0;
    DT_TRY(cudaGetDevice(&prev));
    for (int r = 0; r < world; ++r) out[r] = nullptr;
    int rc = GNNAGG_OK;
    for (int r = 0; r < world && rc == GNNAGG_OK; ++r) {
        if (cudaSetDevice(devices ? devices[r] : r) != cudaSuccess) {
            rc = set_error(GNNAGG_ERR_CUDA, "gnnagg_dist_create: cudaSetDevice failed");
            break;
        }
        rc = gnnagg_dist_create_rank(r, world, shard_bounds, feat_cap, &out[r]);
    }
    if (rc != GNNAGG_OK)
        for (int r = 0; r < world; ++r) {
            if (out[r]) gnnagg_dist_destroy(out[r]);
            out[r] = nullptr;
        }
    cudaSetDevice(prev);
    return rc;
}

int gnnagg_dist_export(gnnagg_dist *d, void *blob)
{
    if (!d || !blob) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_export: NULL argument");
    if (!d->base) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_export: no graph yet (gnnagg_dist_set_graph comes first)");
    DeviceGuard guard(d->device);
    DistBlob b;
    memset(&b, 0, sizeof b);
    b.magic = 0x676e6e62u;
    b.rank = d->rank, b.world = d->world, b.device = d->device, b.pid = d->pid;
    b.feat_cap = d->feat_cap;
    b.rows = d->rows;
    b.raw_base = (uint64_t)(uintptr_t)d->base;
    b.bytes = d->bytes;
    b.off_x[0] = d->off_x[0], b.off_x[1] = d->off_x[1], b.off_req = d->off_req, b.off_meta = d->off_meta;
    b.rounds = d->rounds;
    // a handle is only needed by OTHER processes; a failure here (IPC not permitted) is reported at connect time
    if (cudaIpcGetMemHandle(&b.mem, d->base) != cudaSuccess) {
        cudaGetLastError();
        memset(&b.mem, 0, sizeof b.mem);
    }
    memset(blob, 0, GNNAGG_DIST_BLOB_BYTES);
    memcpy(blob, &b, sizeof b);
    return GNNAGG_OK;
}

int gnnagg_dist_connect(gnnagg_dist *d, const void *blobs)
{
    if (!d || !blobs) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_connect: NULL argument");
    if (!d->base) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_connect: no graph yet (gnnagg_dist_set_graph comes first)");
    DeviceGuard guard(d->device);
    close_peers(d);
    int same = 1;
    for (int p = 0; p < d->world; ++p) {
        if (p == d->rank) continue;
        DistBlob b;
        memcpy(&b, (const char *)blobs + (size_t)p * GNNAGG_DIST_BLOB_BYTES, sizeof b);
        if (b.magic != 0x676e6e62u || b.rank != p || b.world != d->world || b.feat_cap != d->feat_cap ||
            b.rows != d->bounds[p + 1] - d->bounds[p])
            return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_connect: blob does not describe the expected peer");
        if (b.pid == d->pid) {  // same process: the pointer is valid here once peer access is on
            if (b.device != d->device) {
                int can = 0;
                DT_TRY(cudaDeviceCanAccessPeer(&can, d->device, b.device));
                if (!can) return set_error(GNNAGG_ERR_CUDA, "gnnagg_dist_connect: no peer access between the devices");
                cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled)
                    cudaGetLastError();
                else if (e != cudaSuccess)
                    DT_TRY(e);
            }
            d->peer_base[p] = reinterpret_cast<char *>((uintptr_t)b.raw_base);
        } else {
            void *mapped = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&mapped, b.mem, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                cudaGetLastError();
                char buf[256];
                snprintf(buf, sizeof buf, "gnnagg_dist_connect: cudaIpcOpenMemHandle(rank %d): %s", p, cudaGetErrorString(e));
                return set_error(GNNAGG_ERR_CUDA, buf);
            }
            d->peer_base[p] = (char *)mapped;
            d->peer_ipc[p] = true;
        }
        d->peer_off_x[p][0] = b.off_x[0];
        d->peer_off_x[p][1] = b.off_x[1];
        d->peer_rows[p] = (int)b.rows;
        // the rows p wants from this owner: per round c the slots [tab[c][rank], tab[c][rank + 1]) of ITS list; copied once
        if (b.rounds != d->rounds) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_connect: ranks disagree on the pipelining mode");
        int tab[kMaxRounds][kMaxWorld + 1];
        DT_TRY(cudaMemcpy(tab, d->peer_base[p] + b.off_meta, sizeof tab, cudaMemcpyDefault));
        int total_rows = 0;
        for (int c = 0; c < d->rounds; ++c) {
            d->peer_slot[p][c] = tab[c][d->rank];
            d->send_cnt[p][c] = tab[c][d->rank + 1] - tab[c][d->rank];
            d->send_off[p][c] = total_rows;
            total_rows += d->send_cnt[p][c];
        }
        if (total_rows > 0) {
            DT_TRY(cudaMalloc((void **)&d->send_rows[p], (size_t)total_rows * sizeof(int)));
            for (int c = 0; c < d->rounds; ++c)
                if (d->send_cnt[p][c] > 0)
                    DT_TRY(cudaMemcpy(d->send_rows[p] + d->send_off[p][c],
                                      d->peer_base[p] + b.off_req + (size_t)d->peer_slot[p][c] * sizeof(int),
                                      (size_t)d->send_cnt[p][c] * sizeof(int), cudaMemcpyDefault));
        }
        if (b.device == d->device) ++same;
    }
    d->same_device_ranks = same;
    d->connected = true;
    return GNNAGG_OK;
}

int gnnagg_dist_connect_local(gnnagg_dist **ranks, int world)
{
    if (!ranks || world < 1 || world > kMaxWorld) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_connect_local: bad argument");
    char *blobs = new char[(size_t)world * GNNAGG_DIST_BLOB_BYTES];
    int rc = GNNAGG_OK;
    for (int r = 0; r < world && rc == GNNAGG_OK; ++r) {
        if (!ranks[r] || ranks[r]->rank != r || ranks[r]->world != world)
            rc = set_error(GNNAGG_ERR_ARG, "gnnagg_dist_connect_local: handles must be the ranks 0..world-1 of one group");
        else
            rc = gnnagg_dist_export(ranks[r], blobs + (size_t)r * GNNAGG_DIST_BLOB_BYTES);
    }
    for (int r = 0; r < world && rc == GNNAGG_OK; ++r) rc = gnnagg_dist_connect(ranks[r], blobs);
    delete[] blobs;
    return rc;
}

int gnnagg_dist_disconnect(gnnagg_dist *d)
{
    if (!d) return GNNAGG_OK;
    DeviceGuard guard(d->device);
    cudaDeviceSynchronize();
    close_peers(d);
    return GNNAGG_OK;
}

int gnnagg_dist_destroy(gnnagg_dist *d)
{
    if (!d) return GNNAGG_OK;
    DeviceGuard guard(d->device);
    cudaDeviceSynchronize();
    free_graph(d);
    cudaFree(d->ax);
    cudaFree(d->st_w);
    cudaFree(d->st_out);
    if (d->copy_stream) cudaStreamDestroy(d->copy_stream);
    for (cudaEvent_t e : d->chunk_done)
        if (e) cudaEventDestroy(e);
    if (d->copies_done) cudaEventDestroy(d->copies_done);
    if (d->comm) cudaStreamDestroy(d->comm);
    cudaEvent_t evs[] = {d->ev_sig, d->ev_done, d->t_m0, d->t_m1, d->t_m2, d->t_m3, d->t_c0, d->t_c1};
    for (cudaEvent_t e : evs)
        if (e) cudaEventDestroy(e);
    delete d;
    return GNNAGG_OK;
}

float *gnnagg_dist_x(gnnagg_dist *d, int buf)
{
    if (!d || !d->base || buf < 0 || buf > 1) return nullptr;
    return reinterpret_cast<float *>(d->base + d->off_x[buf]);
}

int gnnagg_dist_set_graph(gnnagg_dist *d, const int *d_ptr, const int *d_idx, const float *d_val, int64_t num_e,
                          int remote_stages, void *stream)
{
    if (!d || !d_ptr || (num_e > 0 && (!d_idx || !d_val)) || num_e < 0 || num_e > INT32_MAX)
        return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_set_graph: bad argument");
    if (d->base)
        return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_set_graph: this rank already has a graph (peers may have it mapped); "
                                           "create a new handle for a new graph");
    DeviceGuard guard(d->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int W = d->world, n = d->rows, m = (int)num_e;
    const int64_t total = d->bounds[W];
    const int64_t own_lo = d->bounds[d->rank], own_hi = d->bounds[d->rank + 1];
    // pipelining mode.  remote_stages = R > 0: stage 0 = local sources, the W-1 remote owners -- taken in the order
    // rank+1, rank+2, ... in which they push to this rank -- cut into R groups, one accumulating stage each.
    // R = 0: a single pass once everything has arrived.  R < 0: ROW pipelining with K = -R row chunks: the receive
    // slots are ordered by the chunk that needs a row first, the owners push round by round and chunk c (a row range
    // of the ONE CSR: no extra pass over Y) starts when round c has landed.
    int R = 0, K = 1;
    if (W > 1 && remote_stages > 0) R = remote_stages > W - 1 ? W - 1 : remote_stages;
    if (W > 1 && remote_stages < 0) K = -remote_stages > kMaxRounds ? kMaxRounds : -remote_stages;
    d->remote_stages = R;
    d->num_stages = 1 + R;
    d->rounds = K;
    for (int s = 0; s < kMaxStages; ++s) d->stage_mask[s] = 0;
    d->stage_of[d->rank] = 0;
    // groups grow geometrically (7 owners in 3 stages: 1 + 2 + 4): the first remote stage must not wait long after the
    // local one, and the later, larger ones amortise their launches; every group holds at least one owner
    int stage_end[kMaxStages + 1] = {0};  // stage s covers arrival positions [stage_end[s-1], stage_end[s])
    for (int s = 1; s <= R; ++s) {
        int e = (int)((double)((1 << s) - 1) / (double)((1 << R) - 1) * (W - 1) + 0.5);
        if (e < s) e = s;
        if (e > W - 1 - (R - s)) e = W - 1 - (R - s);
        stage_end[s] = s == R ? W - 1 : e;
    }
    for (int k = 0; k < W - 1; ++k) {
        const int p = (d->rank + 1 + k) % W;
        int stage = 0;
        if (R > 0) {
            stage = 1;
            while (stage < R && k >= stage_end[stage]) ++stage;
        }
        d->stage_of[p] = stage;
        d->stage_mask[stage] |= 1u << p;
    }
    Bounds b;
    memset(&b, 0, sizeof b);
    b.world = W;
    for (int p = 0; p <= W; ++p) b.b[p] = d->bounds[p];
    for (int p = 0; p < W; ++p) b.stage_of[p] = d->stage_of[p];

    int *mark = nullptr, *pos = nullptr, *bad = nullptr, *idx_new = nullptr, *keys = nullptr, *item_row = nullptr, *first = nullptr,
        *slot = nullptr;
    void *tmp = nullptr;
    size_t tmp_bytes = 0;
    int rc = GNNAGG_OK;
    auto cleanup = [&]() {
        cudaFree(mark), cudaFree(pos), cudaFree(bad), cudaFree(idx_new), cudaFree(keys), cudaFree(item_row), cudaFree(first),
            cudaFree(slot), cudaFree(tmp);
    };
#define SG_TRY(expr)                                                                             \
    do {                                                                                         \
        cudaError_t _e = (expr);                                                                 \
        if (_e != cudaSuccess) {                                                                 \
            char _buf[512];                                                                      \
            snprintf(_buf, sizeof _buf, "gnnagg_dist_set_graph: %s: %s", #expr, cudaGetErrorString(_e)); \
            cleanup();                                                                           \
            free_graph(d);                                                                       \
            return set_error(GNNAGG_ERR_CUDA, _buf);                                             \
        }                                                                                        \
    } while (0)
#define SG_FAIL(code, msg)      \
    do {                        \
        cleanup();              \
        free_graph(d);          \
        return set_error(code, msg); \
    } while (0)
    const size_t me = (size_t)(m > 0 ? m : 1);
    int items = 0;
    rc = build_item_rows_device(d_ptr, n, m, &item_row, &items, st);
    if (rc != GNNAGG_OK) {
        cleanup();
        free_graph(d);
        return rc;
    }
    SG_TRY(cudaMalloc((void **)&mark, ((size_t)total + 1) * sizeof(int)));
    SG_TRY(cudaMalloc((void **)&pos, ((size_t)total + 1) * sizeof(int)));
    SG_TRY(cudaMalloc((void **)&bad, sizeof(int)));
    SG_TRY(cudaMemsetAsync(bad, 0, sizeof(int), st));
    {
        size_t need = 0;
        SG_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, mark, pos, (int)(total + 1), st));
        SG_TRY(cudaMalloc(&tmp, need ? need : 1));
        tmp_bytes = need;
    }
    // row chunks (edge balanced, cut on a host mirror of the row pointers); K = 1: the whole block
    d->chunk_rows[0] = 0;
    for (int c = 1; c <= kMaxRounds; ++c) d->chunk_rows[c] = n;
    if (K > 1) {
        int *hp = new int[(size_t)n + 1];
        cudaError_t e = cudaMemcpyAsync(hp, d_ptr, ((size_t)n + 1) * sizeof(int), cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e == cudaSuccess)
            for (int c = 1; c < K; ++c) {
                const int64_t target = (int64_t)m * c / K;
                d->chunk_rows[c] = (int)(std::lower_bound(hp, hp + n + 1, (int)target) - hp);
                if (d->chunk_rows[c] > n) d->chunk_rows[c] = n;
                if (d->chunk_rows[c] < d->chunk_rows[c - 1]) d->chunk_rows[c] = d->chunk_rows[c - 1];
            }
        delete[] hp;
        SG_TRY(e);
    }
    // ---- which remote rows, and in which round each is needed first (first[g]; kMaxRounds + 1 = never)
    SG_TRY(cudaMalloc((void **)&first, ((size_t)total + 1) * sizeof(int)));
    dist_fill_int_kernel<<<nblocks(total + 1), 256, 0, st>>>(first, total + 1, kMaxRounds + 1);
    {
        ChunkRows cr;
        memset(&cr, 0, sizeof cr);
        cr.rounds = K;
        for (int c = 0; c <= kMaxRounds; ++c) cr.lo[c] = d->chunk_rows[c];
        if (m > 0)
            dist_first_use_kernel<<<nblocks(m), 256, 0, st>>>(d_ptr, d_idx, item_row, items, n, m, own_lo, own_hi, total, cr, first, bad);
    }
    int h_bad = 0, h_total = 0;
    dist_round_mark_kernel<<<nblocks(total + 1), 256, 0, st>>>(first, total, 0, 1, mark);
    SG_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, mark, pos, (int)(total + 1), st));
    SG_TRY(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, st));
    SG_TRY(cudaMemcpyAsync(&h_total, pos + total, sizeof(int), cudaMemcpyDeviceToHost, st));
    {
        int h_off[kMaxWorld + 1] = {0};
        for (int p = 0; p <= W; ++p) SG_TRY(cudaMemcpyAsync(&h_off[p], pos + d->bounds[p], sizeof(int), cudaMemcpyDeviceToHost, st));
        SG_TRY(cudaStreamSynchronize(st));
        for (int p = 0; p < W; ++p) d->recv_cnt[p] = h_off[p + 1] - h_off[p];
    }
    if (h_bad) SG_FAIL(GNNAGG_ERR_ARG, "gnnagg_dist_set_graph: a source id lies outside [0, shard_bounds[world])");
    d->num_recv = h_total;
    if ((int64_t)n + d->num_recv > INT32_MAX) SG_FAIL(GNNAGG_ERR_ARG, "gnnagg_dist_set_graph: shard rows + receive slots exceed int32");
    // ---- the peer-visible allocation: flags | slot table | wanted rows | 2 x (shard + receive slots)
    {
        const size_t req = round512((size_t)(d->num_recv > 0 ? d->num_recv : 1) * sizeof(int));
        const size_t xbuf = round512(((size_t)n + (size_t)d->num_recv) * d->feat_cap * sizeof(float) + 16);
        d->off_meta = kFlagBytes;
        d->off_req = kFlagBytes + kMetaBytes;
        d->off_x[0] = d->off_req + req;
        d->off_x[1] = d->off_x[0] + xbuf;
        d->bytes = d->off_x[1] + xbuf;
        SG_TRY(cudaMalloc((void **)&d->base, d->bytes));
        SG_TRY(cudaMemsetAsync(d->base, 0, kFlagBytes + kMetaBytes, st));
        d->peer_base[d->rank] = d->base;
        d->peer_off_x[d->rank][0] = d->off_x[0];
        d->peer_off_x[d->rank][1] = d->off_x[1];
    }
    // ---- receive slots round by round (one round unless row-pipelined), inside a round ascending global id
    SG_TRY(cudaMalloc((void **)&slot, ((size_t)total + 1) * sizeof(int)));
    {
        int base = 0;
        for (int c = 0; c < K; ++c) {
            dist_round_mark_kernel<<<nblocks(total + 1), 256, 0, st>>>(first, total, c, 0, mark);
            SG_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, mark, pos, (int)(total + 1), st));
            int h_off[kMaxWorld + 1] = {0};
            for (int p = 0; p <= W; ++p) SG_TRY(cudaMemcpyAsync(&h_off[p], pos + d->bounds[p], sizeof(int), cudaMemcpyDeviceToHost, st));
            if (total > 0)
                dist_round_fill_kernel<<<nblocks(total), 256, 0, st>>>(mark, pos, total, b, base, reinterpret_cast<int *>(d->base + d->off_req),
                                                                     slot);
            SG_TRY(cudaStreamSynchronize(st));
            for (int p = 0; p <= W; ++p) d->recv_tab[c][p] = base + h_off[p];
            base += h_off[W];
        }
        if (base != (int)d->num_recv) SG_FAIL(GNNAGG_ERR_STATE, "gnnagg_dist_set_graph: internal error (receive slots do not add up)");
        SG_TRY(cudaMemcpyAsync(d->base + d->off_meta, d->recv_tab, sizeof d->recv_tab, cudaMemcpyHostToDevice, st));
    }
    SG_TRY(cudaMalloc((void **)&idx_new, me * sizeof(int)));
    SG_TRY(cudaMalloc((void **)&keys, me * sizeof(int)));
    if (m > 0) {
        if (R == 0)
            dist_reindex_slot_kernel<<<nblocks(m), 256, 0, st>>>(d_idx, m, slot, own_lo, own_hi, n, idx_new, keys);
        else  // K = 1 here: the slot of a row is its rank among the marked ids, and edges carry the stage of their owner
            dist_reindex_kernel<<<nblocks(m), 256, 0, st>>>(d_idx, m, pos, own_lo, own_hi, n, b, idx_new, keys);
    }
    SG_TRY(cudaGetLastError());
    SG_TRY(cudaStreamSynchronize(st));
    cudaFree(mark), cudaFree(pos), cudaFree(tmp), cudaFree(first), cudaFree(slot);
    mark = pos = first = slot = nullptr;
    tmp = nullptr;
    // sub-CSR per stage (stable split: CSR order inside a stage), then one ordinary aggregator per stage
    rc = source_slices_build_device(d_ptr, idx_new, item_row, items, n, m, d->num_stages, 1, &d->sl_ptr, &d->sl_idx, &d->sl_perm,
                                    d->sl_off, d->sl_cnt, st, keys);
    if (rc != GNNAGG_OK) {
        cleanup();
        free_graph(d);
        return rc;
    }
    const size_t padded = me + 4 * (size_t)d->num_stages;
    SG_TRY(cudaMalloc((void **)&d->sl_val, padded * sizeof(float)));
    for (int s = 0; s < d->num_stages; ++s) {
        if (d->sl_cnt[s] > 0)
            dist_gather_val_kernel<<<nblocks(d->sl_cnt[s]), 256, 0, st>>>(d_val, d->sl_perm + d->sl_off[s], d->sl_val + d->sl_off[s],
                                                                        d->sl_cnt[s]);
    }
    SG_TRY(cudaGetLastError());
    SG_TRY(cudaStreamSynchronize(st));
    cleanup();
    mark = pos = bad = idx_new = keys = item_row = first = slot = nullptr;
    tmp = nullptr;
    cudaFree(d->sl_perm);  // only needed for the values
    d->sl_perm = nullptr;
    for (int s = 0; s < d->num_stages; ++s) {
        rc = gnnagg_create(d->sl_ptr + (size_t)s * ((size_t)n + 1), d->sl_idx + d->sl_off[s], nullptr, nullptr, n, d->sl_cnt[s],
                           &d->stage[s]);
        // stages run on their own CSR: the merged view of duplicate edges is not used across ranks (yet)
        if (rc == GNNAGG_OK) rc = gnnagg_set_merge_duplicates(d->stage[s], 1);
        if (rc == GNNAGG_OK) rc = gnnagg_set_val(d->stage[s], d->sl_val + d->sl_off[s]);
        if (rc != GNNAGG_OK) {
            free_graph(d);
            return rc;
        }
    }
    d->num_e = num_e;
    d->launches += 8 + 3 * d->num_stages + 3 * K;
    d->connected = W == 1;
    return gnnagg_dist_prepare(d, d->feat_cap, stream);
#undef SG_TRY
#undef SG_FAIL
}

int gnnagg_dist_prepare(gnnagg_dist *d, int feat, void *stream)
{
    if (!d || d->num_stages == 0) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_prepare: no graph (gnnagg_dist_set_graph)");
    if (feat < 4 || (feat & 3) || feat > d->feat_cap) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_prepare: bad feat");
    DeviceGuard guard(d->device);
    for (int s = 0; s < d->num_stages; ++s)
        if (int rc = gnnagg_prepare(d->stage[s], feat, stream)) return rc;
    // A*X of the fused layer: allocated here rather than inside the first step for the same reason
    const size_t need = (size_t)d->rows * feat;
    if (need > d->ax_cap) {
        cudaFree(d->ax);
        d->ax = nullptr;
        d->ax_cap = 0;
        DT_TRY(cudaMalloc((void **)&d->ax, (need ? need : 1) * sizeof(float)));
        d->ax_cap = need;
    }
    d->prepared_feat = feat;
    return GNNAGG_OK;
}

int gnnagg_dist_info(const gnnagg_dist *d, int64_t *num_recv, int64_t *recv_counts, int *num_stages, int64_t *stage_edges,
                     int64_t *send_counts)
{
    if (!d) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_info: NULL handle");
    if (num_recv) *num_recv = d->num_recv;
    if (recv_counts)
        for (int p = 0; p < d->world; ++p) recv_counts[p] = d->recv_cnt[p];
    if (num_stages) *num_stages = d->num_stages;
    if (stage_edges)
        for (int s = 0; s < d->num_stages; ++s) stage_edges[s] = d->sl_cnt[s];
    if (send_counts)
        for (int p = 0; p < d->world; ++p) {
            send_counts[p] = 0;
            for (int c = 0; c < d->rounds; ++c) send_counts[p] += d->send_cnt[p][c];
        }
    return GNNAGG_OK;
}

int gnnagg_dist_profile_enable(gnnagg_dist *d, int on)
{
    if (!d) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_profile_enable: NULL handle");
    DeviceGuard guard(d->device);
    if (on && !d->t_m0) {
        cudaEvent_t *evs[] = {&d->t_m0, &d->t_m1, &d->t_m2, &d->t_m3, &d->t_c0, &d->t_c1};
        for (cudaEvent_t *e : evs) DT_TRY(cudaEventCreate(e));
    }
    d->prof = on != 0;
    return GNNAGG_OK;
}

int gnnagg_dist_profile_read(gnnagg_dist *d, float *ms)
{
    if (!d || !ms || !d->t_m0) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_profile_read: profiling not enabled");
    DeviceGuard guard(d->device);
    DT_TRY(cudaEventSynchronize(d->t_m3));
    DT_TRY(cudaEventSynchronize(d->t_c1));
    DT_TRY(cudaEventElapsedTime(&ms[0], d->t_c0, d->t_c1));  // halo: first push issued .. last push complete (comm stream)
    DT_TRY(cudaEventElapsedTime(&ms[1], d->t_m0, d->t_m3));  // whole step
    DT_TRY(cudaEventElapsedTime(&ms[2], d->t_m0, d->t_m1));  // stage 0
    DT_TRY(cudaEventElapsedTime(&ms[3], d->t_m2, d->t_m3));  // dense combination
    return GNNAGG_OK;
}

int gnnagg_dist_check(gnnagg_dist *d)
{
    if (!d) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_check: NULL handle");
    if (!d->base) return GNNAGG_OK;
    DeviceGuard guard(d->device);
    uint32_t err = 0;
    DT_TRY(cudaMemcpy(&err, &flags_of(d->base)->err, sizeof err, cudaMemcpyDeviceToHost));
    if (err) {
        char buf[160];
        snprintf(buf, sizeof buf, "halo protocol: rank %d gave up waiting for rank %u (%s flag, code 0x%x)", d->rank, err & 0xffu,
                 (err & 0x100u) ? "consumed" : "arrived", err);
        return set_error(GNNAGG_ERR_STATE, buf);
    }
    return GNNAGG_OK;
}

int64_t gnnagg_dist_launch_count(const gnnagg_dist *d)
{
    if (!d) return 0;
    int64_t total = d->launches;
    for (int s = 0; s < d->num_stages; ++s) total += gnnagg_launch_count(d->stage[s]);
    return total;
}

// One step: Y = A_block * X with X = the shards `buf` of all ranks.  flags: GNNAGG_DIST_NO_EXCHANGE re-uses the
// receive buffer of the previous step (kernels-only timing).
// host_out != NULL: the LAST stage runs in kHostChunks row chunks; chunk c is aggregated (and combined) on `st` while
// the finished rows of chunk c-1 travel to host_out on a second stream (Y / H then are device staging).
// bf16: the shards and receive slots hold bf16 rows of stride feat_in (every address into them is computed in bytes);
// Y, AX and H stay fp32.
constexpr int kHostChunks = 4;

static int stage_run_acc(gnnagg_aggregator *a, bool bf16, const char *xs, float *Y, int feat, int accumulate, cudaStream_t st)
{
    return bf16 ? gnnagg_gcn_run_acc_bf16(a, reinterpret_cast<const uint16_t *>(xs), Y, feat, accumulate, st)
                : gnnagg_gcn_run_acc(a, reinterpret_cast<const float *>(xs), Y, feat, accumulate, st);
}

static int stage_run_rows(gnnagg_aggregator *a, bool bf16, const char *xs, float *Y, int feat, int accumulate, int r0, int r1,
                          cudaStream_t st)
{
    return bf16 ? gnnagg_gcn_run_rows_bf16(a, reinterpret_cast<const uint16_t *>(xs), Y, feat, accumulate, r0, r1, st)
                : gnnagg_gcn_run_rows(a, reinterpret_cast<const float *>(xs), Y, feat, accumulate, r0, r1, st);
}

static int dist_run(gnnagg_dist *d, int buf, bool bf16, float *Y, const float *W, float *H, int feat_in, int feat_out, int flags,
                    cudaStream_t st, float *host_out = nullptr)
{
    if (!d || (!Y && d->rows > 0) || buf < 0 || buf > 1) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_gcn_run: bad argument");
    if (d->num_stages == 0) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_gcn_run: no graph (gnnagg_dist_set_graph)");
    if (!d->connected) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_gcn_run: peers not connected (gnnagg_dist_connect)");
    if (feat_in < 4 || (feat_in & 3) || feat_in > d->feat_cap)
        return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_gcn_run: feat must be a multiple of 4, at most feat_cap");
    DeviceGuard guard(d->device);
    const int Wd = d->world;
    const bool exchange = Wd > 1 && !(flags & GNNAGG_DIST_NO_EXCHANGE);
    // per-stage fix-up tables for this feature width (set_graph builds them for feat_cap).  Building them waits for the
    // device, which is harmless with one process per GPU; a process that drives SEVERAL ranks must call
    // gnnagg_dist_prepare for every rank before the first step of a new width (a device-wide wait while another rank's
    // kernels spin on this rank's flags would never return)
    if (d->prepared_feat != feat_in)
        if (int rc = gnnagg_dist_prepare(d, feat_in, st)) return rc;
    const char *xs = d->base + d->off_x[buf];  // shard rows, then the receive slots
    const size_t row_bytes = (size_t)feat_in * (bf16 ? 2 : 4);
    HaloFlags *mine = flags_of(d->base);
    uint32_t epoch = d->epoch;
    // arrived[] counts completed pushes: round c of epoch e raises it to (e - 1) * rounds + c + 1
    uint32_t flag_base = 0;
    if (d->prof) DT_TRY(cudaEventRecord(d->t_m0, st));
    if (exchange) {
        epoch = ++d->epoch;
        flag_base = (epoch - 1u) * (uint32_t)d->rounds;
        // owner side: wait until every receiver has consumed the previous epoch, then push, receiver by receiver
        halo_begin_kernel<<<1, 32, 0, st>>>(mine, d->rank, Wd, epoch);
        DT_TRY(cudaPeekAtLastError());
        DT_TRY(cudaEventRecord(d->ev_sig, st));
        DT_TRY(cudaStreamWaitEvent(d->comm, d->ev_sig, 0));
        if (d->prof) DT_TRY(cudaEventRecord(d->t_c0, d->comm));
        // copy units of the push: 16 bytes, or 8 for bf16 rows of a width that is 4 mod 8 (8-byte aligned only)
        const bool narrow = bf16 && (feat_in & 7);
        const int FU = (int)(row_bytes / (narrow ? sizeof(uint2) : sizeof(float4)));
        int shift = -1;
        for (int s = 0; s < 16; ++s)
            if ((1 << s) == FU) shift = s;
        for (int c = 0; c < d->rounds; ++c) {
            for (int k = 0; k < Wd - 1; ++k) {
                const int q = (d->rank - 1 - k + 2 * Wd) % Wd;  // receiver q takes this owner as its k-th
                const int64_t units = (int64_t)d->send_cnt[q][c] * FU;
                // one light CTA per SM (two when the round is large) keeps the link busy; ranks sharing a device (tests) split that
                int64_t grid = (units + 128 * 4 - 1) / (128 * 4);
                const int64_t cap = d->same_device_ranks > 1 ? std::max(4, d->sm_count / (2 * d->same_device_ranks)) : 2 * d->sm_count;
                grid = grid < 1 ? 1 : (grid > cap ? cap : grid);  // an empty push still raises the flag
                char *dst = d->peer_base[q] + d->peer_off_x[q][buf] + ((size_t)d->peer_rows[q] + (size_t)d->peer_slot[q][c]) * row_bytes;
                const int *list = d->send_rows[q] ? d->send_rows[q] + d->send_off[q][c] : nullptr;
                uint32_t *flag = &flags_of(d->peer_base[q])->arrived[d->rank];
                // bf16 steps always take the default kernel: the GNNAGG_PUSH_* experiments are fp32 only
                if (!bf16 && d->push_tma && feat_in * 4 <= kPushBatchBytes) {
                    int rpb = kPushBatchBytes / (feat_in * 4);
                    rpb = rpb > 32 ? 32 : rpb;
                    int64_t g2 = (d->send_cnt[q][c] + rpb - 1) / rpb;
                    const int64_t cap2 = d->same_device_ranks > 1 ? std::max(4, d->sm_count / (2 * d->same_device_ranks)) : 2 * d->sm_count;
                    g2 = g2 < 1 ? 1 : (g2 > cap2 ? cap2 : g2);
                    halo_push_tma_kernel<<<(unsigned)g2, 32, kPushBufs * kPushBatchBytes, d->comm>>>(
                        reinterpret_cast<const float *>(xs), list, reinterpret_cast<float *>(dst), d->send_cnt[q][c], feat_in, rpb,
                        &mine->push_cnt[q], flag, flag_base + (uint32_t)c + 1u);
                } else if (!bf16 && d->push_heavy) {
                    int64_t gh = (units + 256 * 8 - 1) / (256 * 8);
                    const int64_t caph = d->same_device_ranks > 1 ? std::max(4, d->sm_count / (2 * d->same_device_ranks)) : (int64_t)d->push_heavy * d->sm_count;
                    gh = gh < 1 ? 1 : (gh > caph ? caph : gh);
                    halo_push_heavy_kernel<8><<<(unsigned)gh, 256, 0, d->comm>>>(reinterpret_cast<const float4 *>(xs), list,
                                                                               reinterpret_cast<float4 *>(dst), units, FU, shift,
                                                                               &mine->push_cnt[q], flag, flag_base + (uint32_t)c + 1u);
                } else if (!bf16 && d->push_prefetch) {
                    halo_push_kernel<float4, 4, true><<<(unsigned)grid, 128, 0, d->comm>>>(
                        reinterpret_cast<const float4 *>(xs), list, reinterpret_cast<float4 *>(dst), units, FU, shift, &mine->push_cnt[q],
                        flag, flag_base + (uint32_t)c + 1u);
                } else if (narrow) {
                    halo_push_kernel<uint2, 4, false><<<(unsigned)grid, 128, 0, d->comm>>>(
                        reinterpret_cast<const uint2 *>(xs), list, reinterpret_cast<uint2 *>(dst), units, FU, shift, &mine->push_cnt[q],
                        flag, flag_base + (uint32_t)c + 1u);
                } else {
                    halo_push_kernel<float4, 4, false><<<(unsigned)grid, 128, 0, d->comm>>>(
                        reinterpret_cast<const float4 *>(xs), list, reinterpret_cast<float4 *>(dst), units, FU, shift, &mine->push_cnt[q],
                        flag, flag_base + (uint32_t)c + 1u);
                }
                DT_TRY(cudaPeekAtLastError());
                ++d->launches;
            }
        }
        DT_TRY(cudaEventRecord(d->ev_done, d->comm));
        if (d->prof) DT_TRY(cudaEventRecord(d->t_c1, d->comm));
        d->launches += 1;
    } else if (d->prof) {
        DT_TRY(cudaEventRecord(d->t_c0, st));
        DT_TRY(cudaEventRecord(d->t_c1, st));
    }
    float *agg_out = W ? d->ax : Y;
    const int fo = W ? feat_out : feat_in;
    // receiver side.  Stage mode: stage by stage, each behind the arrival of its owners.  Row-pipelined mode: ONE stage,
    // row chunk c behind the arrival of round c from every owner.  With a host destination the last stage is cut into
    // row chunks in either mode, and every finished chunk is combined and sent on its way.
    const uint32_t all_owners = exchange ? (((Wd >= 32 ? 0u : (1u << Wd)) - 1u) & ~(1u << d->rank)) : 0u;
    for (int s = 0; s < d->num_stages; ++s) {
        const bool last = s == d->num_stages - 1;
        const bool by_rounds = last && d->rounds > 1;
        const bool by_chunks = last && host_out && d->rows >= 4096;
        if (exchange && d->stage_mask[s] && !by_rounds) {
            halo_wait_kernel<<<1, 32, 0, st>>>(mine, d->stage_mask[s], flag_base + 1u);
            DT_TRY(cudaPeekAtLastError());
            ++d->launches;
        }
        if (!by_rounds && !by_chunks) {
            if (int rc = stage_run_acc(d->stage[s], bf16, xs, agg_out, feat_in, s > 0, st)) return rc;
            if (s == 0 && d->prof) DT_TRY(cudaEventRecord(d->t_m1, st));
            continue;
        }
        const int chunks = by_rounds ? d->rounds : kHostChunks;
        float *out_dev = W ? H : Y;
        int copies = 0;
        for (int c = 0; c < chunks; ++c) {
            const int r0 = by_rounds ? d->chunk_rows[c] : (int)((int64_t)d->rows * c / chunks);
            const int r1 = by_rounds ? d->chunk_rows[c + 1] : (int)((int64_t)d->rows * (c + 1) / chunks);
            if (exchange && by_rounds) {
                halo_wait_kernel<<<1, 32, 0, st>>>(mine, all_owners, flag_base + (uint32_t)c + 1u);
                DT_TRY(cudaPeekAtLastError());
                ++d->launches;
            }
            if (r1 <= r0) continue;
            if (int rc = stage_run_rows(d->stage[s], bf16, xs, agg_out, feat_in, s > 0, r0, r1, st)) return rc;
            if (!host_out) continue;
            if (W) {
                if (int rc = gnnagg_dense_nn(d->ax + (size_t)r0 * feat_in, W, H + (size_t)r0 * feat_out, r1 - r0, feat_out, feat_in, st))
                    return rc;
                d->launches += 2;
            }
            // copy-back events are a small ring: a chunk's event is re-recorded only after the copy stream has consumed it
            cudaEvent_t ev = d->chunk_done[copies % 4];
            DT_TRY(cudaEventRecord(ev, st));
            DT_TRY(cudaStreamWaitEvent(d->copy_stream, ev, 0));
            DT_TRY(cudaMemcpyAsync(host_out + (size_t)r0 * fo, out_dev + (size_t)r0 * fo, (size_t)(r1 - r0) * fo * sizeof(float),
                                   cudaMemcpyDeviceToHost, d->copy_stream));
            ++copies;
        }
        if (host_out) {
            DT_TRY(cudaEventRecord(d->copies_done, d->copy_stream));
            host_out = nullptr;  // done: nothing left for the tail below
            W = nullptr;
        }
        if (s == 0 && d->prof) DT_TRY(cudaEventRecord(d->t_m1, st));
    }
    if (d->prof) DT_TRY(cudaEventRecord(d->t_m2, st));
    if (W && d->rows > 0) {
        if (int rc = gnnagg_dense_nn(d->ax, W, H, d->rows, feat_out, feat_in, st)) return rc;
        d->launches += 2;
    }
    if (host_out && d->rows > 0) {  // small shard: one copy after everything
        DT_TRY(cudaMemcpyAsync(host_out, agg_out == d->ax ? H : Y, (size_t)d->rows * fo * sizeof(float), cudaMemcpyDeviceToHost, st));
    }
    if (exchange) {
        PeerTable peers;
        memset(&peers, 0, sizeof peers);
        for (int p = 0; p < Wd; ++p) peers.flags[p] = flags_of(d->peer_base[p]);
        halo_consumed_kernel<<<1, 32, 0, st>>>(peers, d->rank, Wd, epoch);
        DT_TRY(cudaPeekAtLastError());
        ++d->launches;
        DT_TRY(cudaStreamWaitEvent(st, d->ev_done, 0));  // the caller's stream covers this rank's pushes too: X may be rewritten
    }
    if (d->prof) DT_TRY(cudaEventRecord(d->t_m3, st));
    return GNNAGG_OK;
}

int gnnagg_dist_gcn_run(gnnagg_dist *d, int buf, float *Y, int feat, int flags, void *stream)
{
    return dist_run(d, buf, false, Y, nullptr, nullptr, feat, feat, flags, (cudaStream_t)stream);
}

int gnnagg_dist_gcn_run_bf16(gnnagg_dist *d, int buf, float *Y, int feat, int flags, void *stream)
{
    return dist_run(d, buf, true, Y, nullptr, nullptr, feat, feat, flags, (cudaStream_t)stream);
}

static int dist_layer(gnnagg_dist *d, int buf, bool bf16, const float *W, float *H, int feat_in, int feat_out, int flags,
                      void *stream)
{
    if (!W || (!H && d && d->rows > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_gcn_layer: NULL argument");
    return dist_run(d, buf, bf16, H, W, H, feat_in, feat_out, flags, (cudaStream_t)stream);
}

int gnnagg_dist_gcn_layer(gnnagg_dist *d, int buf, const float *W, float *H, int feat_in, int feat_out, int flags, void *stream)
{
    return dist_layer(d, buf, false, W, H, feat_in, feat_out, flags, stream);
}

int gnnagg_dist_gcn_layer_bf16(gnnagg_dist *d, int buf, const float *W, float *H, int feat_in, int feat_out, int flags,
                               void *stream)
{
    return dist_layer(d, buf, true, W, H, feat_in, feat_out, flags, stream);
}

static int dist_layer_host(gnnagg_dist *d, int buf, bool bf16, const void *h_X, const float *h_W, float *h_out, int feat_in,
                           int feat_out, void *stream)
{
    if (!d || (d->rows > 0 && (!h_X || !h_out)) || buf < 0 || buf > 1)
        return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_gcn_layer_host: bad argument");
    if (!d->base) return set_error(GNNAGG_ERR_STATE, "gnnagg_dist_gcn_layer_host: no graph (gnnagg_dist_set_graph)");
    if (feat_in < 4 || (feat_in & 3) || feat_in > d->feat_cap) return set_error(GNNAGG_ERR_ARG, "gnnagg_dist_gcn_layer_host: bad feat");
    DeviceGuard guard(d->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int fo = h_W ? feat_out : feat_in;
    auto grow = [](float *&p, size_t &cap, size_t need) -> cudaError_t {
        if (need <= cap && p) return cudaSuccess;
        cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc((void **)&p, (need ? need : 1) * sizeof(float));
        if (e == cudaSuccess) cap = need;
        return e;
    };
    DT_TRY(grow(d->st_out, d->st_out_cap, (size_t)d->rows * fo));
    if (h_W) DT_TRY(grow(d->st_w, d->st_w_cap, (size_t)feat_in * feat_out));
    if (!d->copy_stream) {
        DT_TRY(cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking));
        for (cudaEvent_t &e : d->chunk_done) DT_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        DT_TRY(cudaEventCreateWithFlags(&d->copies_done, cudaEventDisableTiming));
    }
    DT_TRY(cudaEventRecord(d->copies_done, d->copy_stream));  // so that the wait below is defined when no chunk copy is issued
    if (d->rows > 0)
        DT_TRY(cudaMemcpyAsync(d->base + d->off_x[buf], h_X, (size_t)d->rows * feat_in * (bf16 ? 2 : 4), cudaMemcpyHostToDevice, st));
    if (h_W) DT_TRY(cudaMemcpyAsync(d->st_w, h_W, (size_t)feat_in * feat_out * sizeof(float), cudaMemcpyHostToDevice, st));
    if (int rc = dist_run(d, buf, bf16, d->st_out, h_W ? d->st_w : nullptr, d->st_out, feat_in, feat_out, 0, st, h_out)) return rc;
    DT_TRY(cudaStreamWaitEvent(st, d->copies_done, 0));
    DT_TRY(cudaStreamSynchronize(st));
    return GNNAGG_OK;
}

int gnnagg_dist_gcn_layer_host(gnnagg_dist *d, int buf, const float *h_X, const float *h_W, float *h_out, int feat_in,
                               int feat_out, void *stream)
{
    return dist_layer_host(d, buf, false, h_X, h_W, h_out, feat_in, feat_out, stream);
}

int gnnagg_dist_gcn_layer_host_bf16(gnnagg_dist *d, int buf, const uint16_t *h_X, const float *h_W, float *h_out, int feat_in,
                                    int feat_out, void *stream)
{
    return dist_layer_host(d, buf, true, h_X, h_W, h_out, feat_in, feat_out, stream);
}

}  // extern "C"
