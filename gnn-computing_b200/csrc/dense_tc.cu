// dense_tc.cu -- the dense combination C[M,N] = A[M,K] * B[K,N] (row-major fp32) on the 5th-gen
// tensor cores: tcgen05.mma kind::tf32 with the accumulator in TMEM, fp32-level accuracy through
// the 3xTF32 split  A*B ~= Ahi*Bhi + Alo*Bhi + Ahi*Blo.
//
// Replaces matmul_NN (include/dense.h:4-23: cublasSgemm + cublasSgeam transpose) and the
// shuffle-based 32-wide matvec inside aggr_gcn_nn (include/aggr_gcn.h:341-357, OUT <= 32 only).
//
// Shape of the problem: M = #vertices (10^5..10^8), K = feat_in, N = feat_out (32..256): a tall-skinny GEMM that
// is bound by streaming A in and C out, next to a gather-bound aggregation that takes 10-20x longer.  Design:
//   * persistent CTAs, one 128-row tile of A at a time, accumulator in TMEM (double-buffered: 2 x N columns);
//   * A cannot come in by TMA because of the hi/lo split: producer warps load fp32, split in registers
//     (cvt.rna.tf32) and store both operands into the canonical K-major no-swizzle layout, 32 values of K per
//     ring stage; W is split once per call by split_w_kernel and arrives by bulk copy;
//   * warp-specialised roles connected by mbarriers only (dense_tf32x3_ws_kernel below): 4 producer warps, one MMA
//     lane issuing 12 tcgen05.mma per stage (4 k-steps x 3 products), tcgen05.commit frees the stage, 4 epilogue
//     warps read TMEM with tcgen05.ld (32 lanes x 32 bit x 16 columns) and store rows straight to global memory.
#include <cuda.h>
#include <cuda_runtime.h>

#include <mutex>
#include <stdint.h>

#include <cstdio>
#include <cstdlib>

#include "common.cuh"
#include "gnnagg.h"
#include "internal.h"

namespace gnnagg {

constexpr int kTileM = 128;
constexpr int kChunkK = 32;                              // floats of K per pipeline stage
constexpr int kStageBytes = kTileM * kChunkK * 4;        // one operand (hi or lo) of one stage: 16 KB
constexpr int kMaxNK = 16384;                            // N_slab * K limit: Bhi+Blo <= 128 KB

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tc_commit(uint32_t bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void tc_mma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        :
        : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// K-major, no-swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// [0,14) start>>4, [16,30) leading byte offset>>4 (between the two 16-byte K chunks of one MMA),
// [32,46) stride byte offset>>4 (between 8-row core matrices), [46,48) version = 1, swizzle = 0
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo, uint32_t sbo)
{
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) |
           (1ull << 46);
}

__device__ __forceinline__ float tf32_round(float x)
{
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// ---------------------------------------------------------------------------------------------------------
// W is split ONCE per call into Whi / Wlo, laid out chunk by chunk (32 values of K per chunk) in the canonical
// K-major operand layout, so that the main kernel can bring it into shared memory with plain bulk copies (TMA,
// UBLKCP): all of it at the start when 2*K*N*4 <= 128 KB, else the two chunks of a stage per stage.
// ---------------------------------------------------------------------------------------------------------
// element (k, n) of W -> chunk kc = k/32:  kc*N*32 + (n/8)*256 + ((k%32)/4)*32 + (n%8)*4 + (k%4)   [floats]
__global__ void __launch_bounds__(256) split_w_kernel(const float *__restrict__ W, float *__restrict__ Whi,
                                                      float *__restrict__ Wlo, int K, int N)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= K * N) return;
    const int k = i / N, n = i % N;
    const float w = __ldg(W + i);
    const float hi = tf32_round(w);
    const size_t off = (size_t)(k >> 5) * N * 32 + (size_t)(n >> 3) * 256 + (size_t)((k & 31) >> 2) * 32 + (size_t)(n & 7) * 4 + (k & 3);
    Whi[off] = hi;
    Wlo[off] = w - hi;
}

// 16 consecutive accumulator columns of this thread's TMEM lane (row) into r[0..15]; completes at tcgen05.wait::ld
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t *r)
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

// ---------------------------------------------------------------------------------------------------------
// Warp-specialised kernel, A fed by the TMA engine.
//
// Round 1/2a versions loaded A with LDG into registers, split it there and stored hi and lo into shared memory.  ncu
// showed what bound them: l1tex__data_pipe_lsu_wavefronts at 78-89 % of peak -- every 128-bit global load that misses
// costs ~23 cycles of the LSU data pipe (one fill wavefront per sector), 4x what the tile's shared-memory traffic
// costs -- while DRAM ran at 2.4-3.1 TB/s and the tensor pipe at 23-44 % (profiles/r2_ncu_summary.md).  So A no longer
// goes through the LSU at all:
//   * the raw fp32 tile (128 rows x 32 floats) arrives by ONE 2-D bulk tensor copy per stage
//     (cp.async.bulk.tensor, CU_TENSOR_MAP_SWIZZLE_128B): it lands in exactly the 128-byte-swizzled K-major layout a
//     tcgen05 shared-memory descriptor can name, and rows beyond M are zero-filled by the engine;
//   * kind::tf32 reads the top 19 bits of each fp32 word, i.e. the raw tile IS the `hi` operand (hi = a truncated to
//     tf32); only lo = a - trunc(a) has to be produced -- 4 converter warps read the raw tile and write the lo tile at
//     the same swizzled offset (LDS.128 + 4 LOP + 4 FADD + STS.128 per 16 bytes; half the stores of the old split);
//   * A*B ~= lo*Bhi + a*Blo + a*Bhi as before (W is still pre-split with round-to-nearest by split_w_kernel).
//     With a truncated instead of rounded, |lo| < 2^-10 |a|; the dropped lo*Blo term and the tf32 truncation of lo
//     are both below 2^-20 |a b| per product, inside the 1e-5 gate with the same tests as before.
// Roles (mbarriers only inside the loop):
//   warp  9    loader    : waits empty[stage], arms full_raw[stage] with the byte count and issues the tensor copy of the
//                          A chunk (+ the two bulk copies of the stage's W chunks when W is streamed)
//   warps 4-7  converters: wait full_raw, write the lo tile, fence.proxy.async, arrive on full_lo[stage]
//   warp  8    MMA       : one lane waits full_lo, issues the 12 tcgen05.mma of the chunk into accumulator buffer
//                          tile&1, tcgen05.commit -> empty[stage]; after the last chunk commit -> acc_full[buffer]
//   warps 0-3  epilogue  : wait acc_full[buffer], tcgen05.ld 32 TMEM lanes x 32 columns, transpose the block through a
//                          padded shared-memory tile, store 4 rows x 128 B per instruction; arrive on acc_empty[buffer]
// The accumulator is double-buffered in TMEM (2 x N columns <= 512).  RESIDENT (2*K*N*4 <= 128 KB): W hi/lo sit in
// shared memory for the life of the CTA; otherwise the stage's W chunks are streamed from L2.
// ---------------------------------------------------------------------------------------------------------
constexpr int kWsThreads = 352;
constexpr int kConverterThreads = 128;
constexpr int kMaxRaw = 4;                                 // depth of the raw-tile ring (tensor copies in flight)
constexpr int kLoStages = 2;                               // depth of the lo (+ streamed W) ring
constexpr int kEpiRowBytes = (32 + 4) * 4;                 // 32 floats + 16 B of padding: conflict-free both ways
constexpr int kEpiBytes = 4 * 32 * kEpiRowBytes;           // one 32 x 32 tile per epilogue warp

// 128-byte-swizzled K-major operand (what the tensor copy writes): 8-row x 128-byte atoms, 1024 bytes apart
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t addr)
{
    return (uint64_t)((addr & 0x3FFFFu) >> 4) | ((uint64_t)1 << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void *tmap, int c0, int c1, uint32_t bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"(tmap), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}

// Two rings, because what has to be deep and what has to be wide differ: the RAW ring (RR x 16 KB, the tensor copies in
// flight -- HBM latency is hidden by its depth) and the LO ring (2 x [lo tile 16 KB + the stage's W chunks when W is
// streamed]).  Chunk c uses raw slot c % RR and lo slot c % 2.
template <bool RESIDENT>
__global__ void __launch_bounds__(kWsThreads, 1)
dense_tf32x3_ws_kernel(const __grid_constant__ CUtensorMap tmapA, const float *__restrict__ Whi, const float *__restrict__ Wlo,
                       float *__restrict__ C, int64_t M, int N, int K, int acc_cols, int RR, int LS)
{
    extern __shared__ __align__(1024) uint8_t smem[];
    __shared__ __align__(8) uint64_t s_full_raw[kMaxRaw], s_empty_raw[kMaxRaw], s_full_lo[kLoStages], s_full_w[kLoStages],
        s_empty_lo[kLoStages], s_acc_full[2], s_acc_empty[2], s_w_ready;
    __shared__ uint32_t s_tmem;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int chunks = K / kChunkK;
    const uint32_t b_chunk = (uint32_t)N * 128u;  // bytes of one 32-wide K chunk of Whi (or Wlo)
    const uint32_t w_bytes = RESIDENT ? 2u * (uint32_t)chunks * b_chunk : 0u;
    const uint32_t lo_stage = RESIDENT ? (uint32_t)kStageBytes : (uint32_t)kStageBytes + 2u * b_chunk;  // [A lo | (Bhi | Blo)]
    uint8_t *const raw_ring = smem + w_bytes;     // 1024-byte aligned: every piece is a multiple of 8 KB
    uint8_t *const lo_ring = raw_ring + (uint32_t)RR * kStageBytes;
    uint8_t *const epi = lo_ring + (uint32_t)LS * lo_stage;
    const uint32_t sbo = (kChunkK / 4) * 128;     // W operands: 1024 B between 8-row core-matrix groups (no swizzle)
    const int64_t tiles = (M + kTileM - 1) / kTileM;
    const int64_t my_tiles = tiles > blockIdx.x ? (tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    const uint32_t total = (uint32_t)(my_tiles * chunks);  // chunks this CTA processes

    if (warp == 8) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)),
                     "r"((uint32_t)(2 * acc_cols))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        for (int i = 0; i < RR; ++i) {
            mbar_init(smem_u32(&s_full_raw[i]), 1);
            mbar_init(smem_u32(&s_empty_raw[i]), 1);
        }
        for (int i = 0; i < LS; ++i) {
            mbar_init(smem_u32(&s_full_lo[i]), kConverterThreads);
            mbar_init(smem_u32(&s_full_w[i]), 1);
            mbar_init(smem_u32(&s_empty_lo[i]), 1);
        }
        for (int i = 0; i < 2; ++i) {
            mbar_init(smem_u32(&s_acc_full[i]), 1);
            mbar_init(smem_u32(&s_acc_empty[i]), 128);
        }
        mbar_init(smem_u32(&s_w_ready), 1);
        fence_mbar_init();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = s_tmem;

    if (warp == 9) {
        // ---------------------------------------------------------------- A loader (one lane): tensor copies, RR deep
        if (lane == 0) {
            uint32_t slot = 0, round = 0;
            for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
                for (int kc = 0; kc < chunks; ++kc) {
                    if (round > 0) mbar_wait(smem_u32(&s_empty_raw[slot]), (round - 1) & 1);  // MMAs of the previous use retired
                    const uint32_t full = smem_u32(&s_full_raw[slot]);
                    mbar_expect_tx(full, (uint32_t)kStageBytes);
                    tma_load_2d(smem_u32(raw_ring + slot * kStageBytes), &tmapA, kc * kChunkK, (int)(tile * kTileM), full);
                    if (++slot == (uint32_t)RR) {
                        slot = 0;
                        ++round;
                    }
                }
            }
        }
    } else if (warp == 10) {
        // ---------------------------------------------------------------- W loader (one lane)
        if (lane == 0) {
            if (RESIDENT) {
                // all of W (pre-split, chunk layout) into shared memory once: 2 * chunks bulk copies on one mbarrier
                const uint32_t ready = smem_u32(&s_w_ready);
                mbar_expect_tx(ready, w_bytes);
                for (int kc = 0; kc < chunks; ++kc) {
                    bulk_g2s(smem_u32(smem) + (uint32_t)kc * b_chunk, Whi + (size_t)kc * N * 32, b_chunk, ready);
                    bulk_g2s(smem_u32(smem) + (uint32_t)(chunks + kc) * b_chunk, Wlo + (size_t)kc * N * 32, b_chunk, ready);
                }
            } else {
                // the two W chunks of every K chunk into the lo-ring slot, as soon as the MMAs that read the slot retired
                for (uint32_t c = 0; c < total; ++c) {
                    const uint32_t l = c % (uint32_t)LS, round = c / (uint32_t)LS;
                    const int kc = (int)(c % (uint32_t)chunks);
                    if (round > 0) mbar_wait(smem_u32(&s_empty_lo[l]), (round - 1) & 1);
                    const uint32_t full = smem_u32(&s_full_w[l]);
                    const uint32_t dst = smem_u32(lo_ring + l * lo_stage) + (uint32_t)kStageBytes;
                    mbar_expect_tx(full, 2u * b_chunk);
                    bulk_g2s(dst, Whi + (size_t)kc * N * 32, b_chunk, full);
                    bulk_g2s(dst + b_chunk, Wlo + (size_t)kc * N * 32, b_chunk, full);
                }
            }
        }
    } else if (warp >= 4 && warp < 8) {
        // ---------------------------------------------------------------- converters: lo = a - trunc_tf32(a)
        const int t = tid - 128;
        uint32_t slot = 0, par_raw = 0;
        for (uint32_t c = 0; c < total; ++c) {
            const uint32_t l = c % (uint32_t)LS, round_l = c / (uint32_t)LS;
            mbar_wait(smem_u32(&s_full_raw[slot]), par_raw);
            if (round_l > 0) mbar_wait(smem_u32(&s_empty_lo[l]), (round_l - 1) & 1);  // MMAs that read this lo slot retired
            const uint8_t *raw = raw_ring + slot * kStageBytes;
            uint8_t *lo = lo_ring + l * lo_stage;
#pragma unroll
            for (int p = 0; p < 8; ++p) {
                // element-wise on the swizzled tile: offset in = offset out; 8 consecutive threads = one 128-byte row
                const uint32_t off = (uint32_t)(p * kConverterThreads + t) * 16u;
                const float4 v = *reinterpret_cast<const float4 *>(raw + off);
                float4 r;
                r.x = v.x - __uint_as_float(__float_as_uint(v.x) & 0xFFFFE000u);
                r.y = v.y - __uint_as_float(__float_as_uint(v.y) & 0xFFFFE000u);
                r.z = v.z - __uint_as_float(__float_as_uint(v.z) & 0xFFFFE000u);
                r.w = v.w - __uint_as_float(__float_as_uint(v.w) & 0xFFFFE000u);
                *reinterpret_cast<float4 *>(lo + off) = r;
            }
            fence_proxy_async();  // generic-proxy stores visible to the tensor core's async proxy
            mbar_arrive(smem_u32(&s_full_lo[l]));
            if (++slot == (uint32_t)RR) {
                slot = 0;
                par_raw ^= 1u;
            }
        }
    } else if (warp == 8) {
        // ---------------------------------------------------------------- MMA issue (one lane)
        if (lane == 0) {
            const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
            if (RESIDENT) mbar_wait(smem_u32(&s_w_ready), 0);
            uint32_t slot = 0, par_raw = 0, c = 0, t = 0;
            for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++t) {
                const uint32_t buf = t & 1;
                if (t >= 2) mbar_wait(smem_u32(&s_acc_empty[buf]), ((t >> 1) - 1) & 1);  // epilogue drained this buffer
                tc_fence_after();
                const uint32_t d_tmem = tmem + buf * (uint32_t)acc_cols;
                for (int kc = 0; kc < chunks; ++kc, ++c) {
                    const uint32_t l = c % (uint32_t)LS, par_l = (c / (uint32_t)LS) & 1;
                    mbar_wait(smem_u32(&s_full_raw[slot]), par_raw);  // the tensor copy landed
                    mbar_wait(smem_u32(&s_full_lo[l]), par_l);        // the lo tile is written
                    if (!RESIDENT) mbar_wait(smem_u32(&s_full_w[l]), par_l);
                    tc_fence_after();
                    const uint32_t a_hi = smem_u32(raw_ring + slot * kStageBytes), a_lo = smem_u32(lo_ring + l * lo_stage);
                    const uint32_t b_hi = RESIDENT ? smem_u32(smem) + (uint32_t)kc * b_chunk : a_lo + kStageBytes;
                    const uint32_t b_lo = RESIDENT ? b_hi + (uint32_t)chunks * b_chunk : b_hi + b_chunk;
#pragma unroll
                    for (int j = 0; j < kChunkK / 8; ++j) {  // one MMA consumes K = 8 tf32 = 32 bytes of every row
                        const uint64_t dah = smem_desc_sw128(a_hi + j * 32), dal = smem_desc_sw128(a_lo + j * 32);
                        const uint64_t dbh = smem_desc(b_hi + j * 256, 128, sbo), dbl = smem_desc(b_lo + j * 256, 128, sbo);
                        tc_mma_tf32(d_tmem, dal, dbh, idesc, (kc | j) ? 1u : 0u);  // small terms first
                        tc_mma_tf32(d_tmem, dah, dbl, idesc, 1u);
                        tc_mma_tf32(d_tmem, dah, dbh, idesc, 1u);
                    }
                    tc_commit(smem_u32(&s_empty_raw[slot]));  // both rings are released by the same MMAs
                    tc_commit(smem_u32(&s_empty_lo[l]));
                    if (++slot == (uint32_t)RR) {
                        slot = 0;
                        par_raw ^= 1u;
                    }
                }
                tc_commit(smem_u32(&s_acc_full[buf]));
            }
        }
    } else if (warp < 4) {
        // ---------------------------------------------------------------- warps 0-3: epilogue
        uint8_t *const my_tile = epi + warp * (32 * kEpiRowBytes);
        uint32_t t = 0;
        for (int64_t tile = blockIdx.x; tile < tiles; tile += gridDim.x, ++t) {
            const uint32_t buf = t & 1;
            mbar_wait(smem_u32(&s_acc_full[buf]), (t >> 1) & 1);
            tc_fence_after();
            const int64_t row0 = tile * kTileM + warp * 32;  // first of this warp's 32 rows
            const uint32_t taddr = tmem + buf * (uint32_t)acc_cols + ((uint32_t)(warp * 32) << 16);
            for (int col = 0; col < N; col += 32) {  // N is a multiple of 32: two 16-column TMEM loads per wait
                uint32_t r[32];
                tmem_ld16(taddr + (uint32_t)col, r);
                tmem_ld16(taddr + (uint32_t)col + 16u, r + 16);
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                // lane = row: write the row's 32 values, then read the block back 4 rows x 128 B at a time
                float4 *mine = reinterpret_cast<float4 *>(my_tile + lane * kEpiRowBytes);
#pragma unroll
                for (int i = 0; i < 8; ++i)
                    mine[i] = make_float4(__uint_as_float(r[4 * i]), __uint_as_float(r[4 * i + 1]), __uint_as_float(r[4 * i + 2]),
                                          __uint_as_float(r[4 * i + 3]));
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int rr = j * 4 + (lane >> 3);
                    const float4 v = *reinterpret_cast<const float4 *>(my_tile + rr * kEpiRowBytes + (lane & 7) * 16);
                    if (row0 + rr < M) stg_f4(C + (size_t)(row0 + rr) * N + col + (lane & 7) * 4, v);
                }
                __syncwarp();  // the tile is rewritten by the next column block
            }
            tc_fence_before();
            mbar_arrive(smem_u32(&s_acc_empty[buf]));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 8)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)(2 * acc_cols)) : "memory");
}

// cuTensorMapEncodeTiled through the runtime's driver entry point: libgnnagg.so does not link libcuda, so it still
// loads on a machine without a GPU (tests/test_abi.py)
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled()
{
    static std::mutex lock;
    static EncodeTiledFn fn = nullptr;
    std::lock_guard<std::mutex> guard(lock);
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            cudaGetLastError();
    }
    return fn;
}

// A [M, K] fp32 row-major, box = 32 floats x 128 rows, 128-byte swizzle, rows beyond M read as zero
static int make_a_tensor_map(CUtensorMap *map, const float *A, int64_t M, int K)
{
    EncodeTiledFn enc = encode_tiled();
    if (!enc) return set_error(GNNAGG_ERR_CUDA, "dense combination: cuTensorMapEncodeTiled is not available from this driver");
    const cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)M};
    const cuuint64_t gstride[1] = {(cuuint64_t)K * sizeof(float)};
    const cuuint32_t box[2] = {(cuuint32_t)kChunkK, (cuuint32_t)kTileM};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float *>(A), gdim, gstride, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        char buf[128];
        snprintf(buf, sizeof buf, "dense combination: cuTensorMapEncodeTiled failed (%d)", (int)r);
        return set_error(GNNAGG_ERR_CUDA, buf);
    }
    return GNNAGG_OK;
}

// Stream-ordered pool for the W split of the streamed kernel.  The device's default pool hands freed memory back to
// the driver at every synchronisation (release threshold 0), which made each call re-map its 2*K*N floats; a private
// pool that keeps what it has turns the allocation into a pointer bump.  One pool per device, created on first use.
static cudaMemPool_t split_pool(int dev)
{
    static std::mutex lock;
    static cudaMemPool_t pools[64] = {};
    if (dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> guard(lock);
    if (!pools[dev]) {
        cudaMemPoolProps props = {};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = dev;
        if (cudaMemPoolCreate(&pools[dev], &props) != cudaSuccess) {
            pools[dev] = nullptr;
            return nullptr;
        }
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(pools[dev], cudaMemPoolAttrReleaseThreshold, &keep);
    }
    return pools[dev];
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device (per-context) property of the function: remember what
// has been configured for EACH device, so that a process driving several GPUs (gnnagg_dist_create) opts in on all
template <class Kernel>
static cudaError_t ensure_dynamic_smem(Kernel kernel, int slot, int dev, size_t bytes)
{
    static std::mutex lock;
    static size_t configured[2][64] = {};
    if (dev < 0 || dev >= 64) return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    std::lock_guard<std::mutex> guard(lock);
    if (bytes <= configured[slot][dev]) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) configured[slot][dev] = bytes;
    return e;
}

// forces the (lazy) load of the combination kernels and creates the W-split pool; see capi.cu: preload
void dense_preload()
{
    cudaFuncAttributes attr;
    if (cudaFuncGetAttributes(&attr, split_w_kernel) != cudaSuccess) cudaGetLastError();
    if (cudaFuncGetAttributes(&attr, dense_tf32x3_ws_kernel<true>) != cudaSuccess) cudaGetLastError();
    if (cudaFuncGetAttributes(&attr, dense_tf32x3_ws_kernel<false>) != cudaSuccess) cudaGetLastError();
    int dev = 0;
    if (cudaGetDevice(&dev) == cudaSuccess) {
        split_pool(dev);
        // opt in to the largest dynamic shared memory either variant can ask for, now rather than at the first launch
        ensure_dynamic_smem(dense_tf32x3_ws_kernel<false>, 0, dev, 227 * 1024 - 1024);
        ensure_dynamic_smem(dense_tf32x3_ws_kernel<true>, 1, dev, 227 * 1024 - 1024);
        encode_tiled();
    }
}

// Shapes the tensor-core kernel does not take (K or N not a multiple of 32, or above 256): a plain fp32 tiled GEMM,
// 64 x 64 tile per CTA, 4 x 4 outputs per thread, K in steps of 16 through shared memory; sums in K order (fp32 FMA).
// matmul_NN of the reference (dense.h:4-23, cuBLAS) takes any size; the configs of BASELINE.json never come here.
__global__ void __launch_bounds__(256) dense_simt_kernel(const float *__restrict__ A, const float *__restrict__ B, float *__restrict__ C,
                                                         int64_t M, int N, int K)
{
    __shared__ float sA[16][64 + 1], sB[16][64];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t row0 = (int64_t)blockIdx.y * 64;
    const int col0 = blockIdx.x * 64;
    float acc[4][4] = {};
    for (int k0 = 0; k0 < K; k0 += 16) {
        for (int i = threadIdx.x; i < 64 * 16; i += 256) {
            const int r = i >> 4, k = i & 15;
            sA[k][r] = (row0 + r < M && k0 + k < K) ? __ldg(A + (size_t)(row0 + r) * K + k0 + k) : 0.f;
            const int kb = i >> 6, c = i & 63;
            sB[kb][c] = (k0 + kb < K && col0 + c < N) ? __ldg(B + (size_t)(k0 + kb) * N + col0 + c) : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            float a[4], b[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) a[i] = sA[k][ty * 4 + i], b[i] = sB[k][tx * 4 + i];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (row0 + ty * 4 + i < M && col0 + tx * 4 + j < N) C[(size_t)(row0 + ty * 4 + i) * N + col0 + tx * 4 + j] = acc[i][j];
}

// widths the tcgen05 kernel takes; every other product goes through dense_simt_kernel
static bool dense_on_tensor_cores(int N, int K) { return N >= 32 && K >= 32 && N <= 256 && K <= 256 && N % 32 == 0 && K % 32 == 0; }

int dense_nn_launches(int64_t M, int N, int K)
{
    if (M <= 0) return 0;
    return dense_on_tensor_cores(N, K) ? 2 : (int)((M + (int64_t)65535 * 64 - 1) / ((int64_t)65535 * 64));
}

int dense_nn_launch(const float *A, const float *B, float *C, int64_t M, int N, int K, void *stream)
{
    cudaStream_t st = (cudaStream_t)stream;
    if (N < 1 || K < 1) return set_error(GNNAGG_ERR_ARG, "dense combination: feat_in and feat_out must be positive");
    if (!dense_on_tensor_cores(N, K)) {
        if (M <= 0) return GNNAGG_OK;
        const dim3 grid((unsigned)((N + 63) / 64), (unsigned)((M + 63) / 64));
        if (grid.y > 65535u * 16u) return set_error(GNNAGG_ERR_ARG, "dense combination: too many rows for the generic kernel");
        for (int64_t r0 = 0; r0 < M; r0 += (int64_t)65535 * 64) {  // gridDim.y limit
            const int64_t rows = M - r0 < (int64_t)65535 * 64 ? M - r0 : (int64_t)65535 * 64;
            dense_simt_kernel<<<dim3(grid.x, (unsigned)((rows + 63) / 64)), 256, 0, st>>>(A + (size_t)r0 * K, B, C + (size_t)r0 * N, rows, N, K);
        }
        return cudaPeekAtLastError() == cudaSuccess ? GNNAGG_OK : set_error(GNNAGG_ERR_CUDA, "dense combination: launch failed");
    }
    if ((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(C)) & 15)
        return set_error(GNNAGG_ERR_ARG, "dense combination: A and C must be 16-byte aligned");
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return set_error(GNNAGG_ERR_CUDA, "dense combination: no CUDA device");
    if (M <= 0) return GNNAGG_OK;
    const int64_t tiles = (M + kTileM - 1) / kTileM;
    const unsigned grid = (unsigned)(tiles < sms ? tiles : sms);
    int acc_cols = 32;  // TMEM columns of one accumulator buffer (power of two >= N); two buffers are allocated
    while (acc_cols < N) acc_cols *= 2;
    // W split once per call into global memory (hi | lo, chunk layout), from a private stream-ordered pool
    float *wsplit = nullptr;
    cudaMemPool_t pool = split_pool(dev);
    if (!pool || cudaMallocFromPoolAsync((void **)&wsplit, (size_t)2 * K * N * sizeof(float), pool, st) != cudaSuccess)
        return set_error(GNNAGG_ERR_CUDA, "dense combination: cannot allocate the W split");
    float *whi = wsplit, *wlo = wsplit + (size_t)K * N;
    split_w_kernel<<<(K * N + 255) / 256, 256, 0, st>>>(B, whi, wlo, K, N);
    CUtensorMap tmapA;
    if (int rc = make_a_tensor_map(&tmapA, A, M, K)) {
        cudaFreeAsync(wsplit, st);
        return rc;
    }
    cudaError_t e = cudaSuccess;
    // static shared memory rounds up to 1 KB (the dynamic part is 1024-byte aligned); everything else goes to the rings
    constexpr size_t kSmemBudget = 227 * 1024 - 1024;
    if (N * K > kMaxNK) {  // W does not fit in shared memory next to the rings: stream it, two chunks per lo-ring slot
        const size_t fixed = (size_t)kLoStages * (kStageBytes + (size_t)2 * N * 128) + kEpiBytes;
        int RR = (int)((kSmemBudget - fixed) / kStageBytes);
        RR = RR > kMaxRaw ? kMaxRaw : RR;
        if (RR < 1) return set_error(GNNAGG_ERR_ARG, "dense combination: feat_out too large for the shared-memory rings");
        const size_t smem_s = fixed + (size_t)RR * kStageBytes;
        e = ensure_dynamic_smem(dense_tf32x3_ws_kernel<false>, 0, dev, smem_s);
        if (e == cudaSuccess) dense_tf32x3_ws_kernel<false><<<grid, kWsThreads, smem_s, st>>>(tmapA, whi, wlo, C, M, N, K, acc_cols, RR, kLoStages);
    } else {
        // (one lo slot and a fourth raw slot instead was measured: 0.074 ms against 0.0615 ms on C2 -- the converter <-> MMA
        // hand-over then serialises; two lo slots stay)
        const int LS = kLoStages;
        const size_t fixed = (size_t)2 * N * K * 4 + (size_t)LS * kStageBytes + kEpiBytes;  // W hi/lo resident
        int RR = (int)((kSmemBudget - fixed) / kStageBytes);
        RR = RR > kMaxRaw ? kMaxRaw : RR;
        const size_t smem = fixed + (size_t)RR * kStageBytes;
        e = ensure_dynamic_smem(dense_tf32x3_ws_kernel<true>, 1, dev, smem);
        if (e == cudaSuccess) dense_tf32x3_ws_kernel<true><<<grid, kWsThreads, smem, st>>>(tmapA, whi, wlo, C, M, N, K, acc_cols, RR, LS);
    }
    if (e == cudaSuccess) e = cudaPeekAtLastError();
    cudaFreeAsync(wsplit, st);
    return e == cudaSuccess ? GNNAGG_OK : set_error(GNNAGG_ERR_CUDA, cudaGetErrorString(e));
}

}  // namespace gnnagg
