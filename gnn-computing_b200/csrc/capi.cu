// capi.cu -- the C ABI of libgnnagg.so (include/gnnagg.h): aggregator object, launch logic.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "agg_kernels.cuh"
#include "edge_kernels.cuh"
#include "gnnagg.h"
#include "internal.h"

namespace gnnagg {

static thread_local std::string g_error;

int set_error(int code, const char *msg)
{
    g_error = msg ? msg : "";
    return code;
}

#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            char _buf[512];                                                                  \
            snprintf(_buf, sizeof _buf, "%s:%d %s: %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return set_error(GNNAGG_ERR_CUDA, _buf);                                         \
        }                                                                                    \
    } while (0)

#define LAUNCH_CHECK(a)                   \
    do {                                  \
        CUDA_TRY(cudaPeekAtLastError()); \
        ++(a)->launches;                  \
    } while (0)

template <class T>
static int ensure(T *&p, size_t &cap, size_t need)
{
    if (need <= cap && p) return GNNAGG_OK;
    if (p) CUDA_TRY(cudaFree(p));
    p = nullptr;
    cap = 0;
    CUDA_TRY(cudaMalloc((void **)&p, (need ? need : 1) * sizeof(T)));
    cap = need;
    return GNNAGG_OK;
}

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Programmatic dependent launch for the short kernels that follow a traversal (fix-up passes, the row-final kernel and
// the second pass of the GAT backward): the launch is processed and the grid scheduled while the predecessor's last
// CTAs drain; the kernel itself waits (griddep_wait) before it reads.  GNNAGG_PDL=0 turns the attribute off.
static bool pdl_enabled()
{
    static const bool on = [] {
        const char *e = getenv("GNNAGG_PDL");
        return e ? atoi(e) != 0 : true;
    }();
    return on;
}

template <class... KArgs, class... Args>
static void launch_dep(void (*kernel)(KArgs...), unsigned grid, unsigned block, cudaStream_t st, Args &&...args)
{
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(block);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);  // errors surface in the caller's LAUNCH_CHECK
}

}  // namespace gnnagg

using namespace gnnagg;

constexpr int kMaxSlices = 16;
// automatic locality slicing (gnnagg_set_locality_slices(a, 0)): X at least this many times the L2, slices of about
// kLocalitySliceL2Multiples x L2, average degree at least kLocalityMinDegree
constexpr double kLocalityMinL2Multiples = 8.0;
constexpr double kLocalitySliceL2Multiples = 2.5;
constexpr double kLocalityMinDegree = 20.0;
constexpr int kLocalityMaxAuto = 4;
// automatic merged view of duplicate edges (gnnagg_set_merge_duplicates(a, 0)), DESIGN.md §4.11: merging must remove at
// least kMergeMinFraction of the edges (reddit / proteins shapes: 34 %, 16-28 % faster layer; arxiv / products shapes:
// 5 %, no gain beyond the spread), on graphs of at least kMergeMinEdges edges -- the small-graph bound of
// kSmallGraphEdges, below which the aggregation is bound by the length of one warp's walk rather than by the L1 data
// path that merging relieves, and where the decision's host synchronisation would fall on every small aggregator
constexpr int64_t kMergeMinEdges = 4000000;
constexpr double kMergeMinFraction = 0.10;

struct gnnagg_aggregator {
    // borrowed graph
    const int *d_ptr = nullptr, *d_idx = nullptr;
    const int *h_ptr_user = nullptr, *h_idx_user = nullptr;
    std::vector<int> h_ptr, h_idx;  // lazily mirrored (aggregator.h:30-39)
    int n = 0, m = 0;
    const float *d_val = nullptr;
    // derived
    int *d_item_row = nullptr;
    int num_items = 0;  // ceil(m / kFineItem)
    // scratch (owned)
    float *carry = nullptr;
    size_t carry_cap = 0;
    float *den_row = nullptr;
    size_t den_row_cap = 0;
    float *carry_den = nullptr;
    size_t carry_den_cap = 0;
    float *newval = nullptr;
    size_t newval_cap = 0;
    float *ax = nullptr;
    size_t ax_cap = 0;
    // host-buffer entry points: device staging
    float *st_in = nullptr, *st_out = nullptr, *st_w = nullptr, *st_att = nullptr;
    size_t st_in_cap = 0, st_out_cap = 0, st_w_cap = 0, st_att_cap = 0;
    // schedule (owned device copies)
    int sched_kind = GNNAGG_SCHED_NOP;
    int num_target = 0, sched_edges = 0, sched_items = 0;
    int neighbor_group_size = 0, locality_partition_num = 0;
    int *s_ptr = nullptr, *s_idx = nullptr, *s_target = nullptr, *s_perm = nullptr, *s_item_row = nullptr;
    float *s_val = nullptr;  // owned only when s_perm != nullptr (locality kinds); NG aliases d_val
    bool s_idx_owned = false;  // neighbour grouping keeps the edge order: its idx aliases d_idx
    // rows spanning more than kFixChunk carry items, per item size (second fix-up pass; built on first use)
    struct LongRows {
        int item_edges = 0, count = 0;
        int *list = nullptr;
        int2 *records = nullptr;  // per item: what the first fix-up pass does there (fixup_records_kernel)
    };
    std::vector<LongRows> long_rows;
    int64_t launches = 0;
    int warp_edges = 0;  // 0 = automatic
    // backward pass (gnnagg_transpose_build): the transposed CSR and a child aggregator that runs over it
    int num_src = 0;
    int *t_ptr = nullptr, *t_idx = nullptr, *t_perm = nullptr;
    gnnagg_aggregator *tr = nullptr;
    float *t_val = nullptr;    // edge values in transposed order (owned, m floats)
    const float *t_val_of = nullptr;  // which d_val t_val currently mirrors (NULL: none / attention weights)
    // GAT backward scratch: per row (1 / D_v, c_v); per edge (w_e, t_e); pass-1 row sums per row / per entered item
    float2 *bwd_c = nullptr, *bwd_wt = nullptr, *bwd_part = nullptr, *bwd_carry = nullptr;
    size_t bwd_c_cap = 0, bwd_wt_cap = 0, bwd_part_cap = 0, bwd_carry_cap = 0;
    float *bwd_t = nullptr;  // large graphs: ds_e in transposed edge order (alpha_e goes to t_val)
    size_t bwd_t_cap = 0;
    // host-buffer entry points: the result is copied back per row chunk on a second stream while the next chunk computes
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t chunk_done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t copies_done = nullptr;
    // host-buffer entry points, large graphs: the CSR split by source-id ranges so that slice c can be aggregated while
    // the rows of X that slice c+1 gathers are still on their way from the host (source_slices_build_device)
    int host_slices = 0;  // 0 = automatic, > 0 forced slice count, < 0 row-chunk pipeline only (gnnagg_set_host_pipeline)
    int num_slices = 0, slice_width = 0;
    gnnagg_aggregator *slice[kMaxSlices] = {nullptr};
    int *sl_ptr = nullptr, *sl_idx = nullptr, *sl_perm = nullptr;
    float *sl_val = nullptr;
    const float *sl_val_of = nullptr;
    int sl_off[kMaxSlices] = {0}, sl_cnt[kMaxSlices] = {0};
    // locality slices of the device-resident path (gnnagg_set_locality_slices): when X is many times the L2, the
    // un-scheduled aggregation runs source slice by source slice (sub-CSRs in accumulate mode, deterministic) so that
    // the rows a slice gathers stay cache resident -- locality_schedule (graph_schedule.h:17-89) without its atomics.
    // `loc` borrows this aggregator's CSR and owns the slices.
    int loc_slices = 0;  // 0 = automatic, 1 = off, 2..kMaxSlices forced
    gnnagg_aggregator *loc = nullptr;
    // a slice compacted to its non-empty rows: d_ptr = c_ptr (owned), row r of it is output row out_row[r] (owned)
    int *c_ptr = nullptr, *out_row = nullptr;
    cudaStream_t in_stream = nullptr;
    cudaEvent_t in_done[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t in_free = nullptr;
    // merged view (gnnagg_set_merge_duplicates): runs of adjacent equal sources in a row as one entry each.  `mg` runs
    // over mg_ptr / mg_idx / mg_val (owned here) with its own item table, carry and long-row records; built on first use
    int merge_mode = 0;       // 0 = automatic, 1 = off, 2 = on
    int merge_auto = -1;      // automatic decision: -1 not taken yet, 0 off, 1 on
    gnnagg_aggregator *mg = nullptr;
    int *mg_ptr = nullptr, *mg_idx = nullptr, *mg_start = nullptr;  // mg_start[k]: CSR edge id of run k's first edge
    float *mg_val = nullptr;
    const float *mg_val_of = nullptr;  // which d_val mg_val currently sums (NULL: none / stale after gnnagg_set_val)
    // optional per-kernel timing (gnnagg_profile_enable)
    bool prof = false;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};  // begin, agg0, agg1, agg_end, end
};

#define PROF_RECORD(a, i, st)                                   \
    do {                                                        \
        if ((a)->prof) CUDA_TRY(cudaEventRecord((a)->ev[i], st)); \
    } while (0)

namespace gnnagg {

static EdgeParams edge_params(const gnnagg_aggregator *a)
{
    EdgeParams g;
    g.ptr = a->d_ptr;
    g.idx = a->d_idx;
    g.item_row = a->d_item_row;
    g.num_rows = a->n;
    g.num_edges = a->m;
    g.num_items = a->num_items;
    return g;
}

static int build_item_rows(gnnagg_aggregator *a, const int *d_ptr, int rows, int edges, int **out, int *items,
                           cudaStream_t st)
{
    *items = (int)cdiv(edges, kFineItem);
    if (*out) CUDA_TRY(cudaFree(*out));
    *out = nullptr;
    CUDA_TRY(cudaMalloc((void **)out, (size_t)(*items ? *items : 1) * sizeof(int)));
    if (*items > 0) {
        item_row_kernel<<<(unsigned)cdiv(*items, 256), 256, 0, st>>>(d_ptr, rows, edges, *out, *items);
        LAUNCH_CHECK(a);
    }
    return GNNAGG_OK;
}

int build_item_rows_device(const int *d_ptr, int rows, int edges, int **out, int *items, cudaStream_t st)
{
    *items = (int)cdiv(edges, kFineItem);
    *out = nullptr;
    CUDA_TRY(cudaMalloc((void **)out, (size_t)(*items ? *items : 1) * sizeof(int)));
    if (*items > 0) {
        item_row_kernel<<<(unsigned)cdiv(*items, 256), 256, 0, st>>>(d_ptr, rows, edges, *out, *items);
        CUDA_TRY(cudaPeekAtLastError());
    }
    return GNNAGG_OK;
}

static void free_schedule(gnnagg_aggregator *a)
{
    cudaFree(a->s_ptr);
    if (a->s_idx_owned) cudaFree(a->s_idx);
    a->s_idx_owned = false;
    cudaFree(a->s_target);
    cudaFree(a->s_item_row);
    if (a->s_perm) cudaFree(a->s_val);
    cudaFree(a->s_perm);
    a->s_ptr = a->s_idx = a->s_target = a->s_item_row = a->s_perm = nullptr;
    a->s_val = nullptr;
    a->num_target = a->sched_edges = a->sched_items = 0;
    a->sched_kind = GNNAGG_SCHED_NOP;
}

__global__ void gather_val_kernel(const float *__restrict__ val, const int *__restrict__ perm, float *__restrict__ out,
                                  int count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = __ldg(val + __ldg(perm + i));
}

// out[perm[i]] = in[i]: scheduled edge order back to CSR order
__global__ void scatter_val_kernel(const float *__restrict__ in, const int *__restrict__ perm, float *__restrict__ out, int count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[__ldg(perm + i)] = __ldg(in + i);
}

// val'[k] = sum of the values of run k in CSR order, in fp64, rounded once; one thread per run (deterministic)
__global__ void merge_val_kernel(const float *__restrict__ val, const int *__restrict__ start, float *__restrict__ out,
                                 int runs)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= runs) return;
    const int end = __ldg(start + k + 1);
    double s = 0.0;
    for (int e = __ldg(start + k); e < end; ++e) s += (double)__ldg(val + e);
    out[k] = (float)s;
}

static int check_feat(int F)
{
    if (F < 4 || F > 1024 || (F & 3)) return set_error(GNNAGG_ERR_ARG, "feat must be a multiple of 4 in [4,1024]");
    return GNNAGG_OK;
}

// lanes that cover one feature row with a float4 each: F/4 rounded up to 8, 16 or 32
static inline int lanes_for(int F) { return F <= 32 ? 8 : (F <= 64 ? 16 : 32); }

// lanes per virtual warp of the aggregation kernels for a feature width (agg_kernel<LPR, NV>).  Virtual warps HALF as
// wide with two float4 per lane for rows of 33..128 floats -- one broadcast load of the staged idx / val then serves
// twice as many items, and those loads take 18 % of the L1 data pipe on the reddit shape -- were measured and lost:
// aggregation 2.27 -> 2.43 ms on reddit F=128, 0.496 -> 0.537 ms on proteins F=64.
static inline int lpr_for(int F) { return lanes_for(F); }

// graphs below this many edges use the 128-edge-per-warp variant: with 512 there would be fewer than
// ~2 waves of CTAs on 148 SMs and the kernel would be bound by the length of one warp's walk
constexpr int64_t kSmallGraphEdges = 4000000;

static inline int warp_edges_for(const gnnagg_aggregator *a, int64_t num_edges)
{
    if (a->warp_edges) return a->warp_edges;
    return num_edges < kSmallGraphEdges ? 128 : kWarpEdges;
}
static inline int item_edges_for(const gnnagg_aggregator *a, int F, int64_t num_edges)
{
    return warp_edges_for(a, num_edges) / (32 / lpr_for(F));
}

template <int MODE, bool SCHED, int WE>
static void launch_agg_we(const AggParams &p, cudaStream_t st)
{
    const int F = p.F;
    const int64_t first = (int64_t)(p.edge_lo / WE) * WE;  // warps keep their global 512-edge alignment (TMA staging)
    const unsigned grid = (unsigned)cdiv(p.edge_hi - first, (int64_t)WE * kCtaWarps);
    auto go = [&](void (*kernel)(const AggParams)) {
        if (MODE == kModeGATBWD || MODE == kModeGATBWD2)
            launch_dep(kernel, grid, kCtaThreads, st, p);
        else
            kernel<<<grid, kCtaThreads, 0, st>>>(p);
    };
    if (F <= 32)
        go(agg_kernel<8, 1, MODE, SCHED, WE>);
    else if (F <= 64)
        go(agg_kernel<16, 1, MODE, SCHED, WE>);
    else if (F <= 128)
        go(agg_kernel<32, 1, MODE, SCHED, WE>);
    else
        go(agg_kernel<32, 2, MODE, SCHED, WE>);
}

// CUDA loads a kernel lazily at its first launch, and that load can wait for the device to go idle.  A process that
// drives several ranks must therefore never launch a kernel for the FIRST time while another rank's kernels spin on a
// flag this rank has yet to set (dist.cu).  cudaFuncGetAttributes forces the load.
template <class K>
static void preload(K kernel)
{
    cudaFuncAttributes attr;
    if (cudaFuncGetAttributes(&attr, kernel) != cudaSuccess) cudaGetLastError();
}

template <int WE>
static void preload_gcn_we(int F)
{
    if (F <= 32)
        preload(agg_kernel<8, 1, kModeGCN, false, WE>);
    else if (F <= 64)
        preload(agg_kernel<16, 1, kModeGCN, false, WE>);
    else if (F <= 128)
        preload(agg_kernel<32, 1, kModeGCN, false, WE>);
    else
        preload(agg_kernel<32, 2, kModeGCN, false, WE>);
}

// rows of a's CSR with more than kFixChunk carry items of EB edges, found once per item size (one host synchronisation)
static int long_rows_of(gnnagg_aggregator *a, const AggParams &p, int EB, cudaStream_t st, const int **list, int *count,
                        const int2 **records)
{
    for (auto &e : a->long_rows)
        if (e.item_edges == EB) {
            *list = e.list;
            *count = e.count;
            *records = e.records;
            return GNNAGG_OK;
        }
    gnnagg_aggregator::LongRows e;
    e.item_edges = EB;
    const size_t cap = (size_t)a->m / ((size_t)kFixChunk * EB) + 2;
    int *counter = nullptr;
    const int64_t items = cdiv(a->m, EB);
    CUDA_TRY(cudaMalloc((void **)&e.list, cap * sizeof(int)));
    if (cudaMalloc((void **)&counter, sizeof(int)) != cudaSuccess ||
        cudaMalloc((void **)&e.records, (size_t)(items + 1) * sizeof(int2)) != cudaSuccess) {
        cudaFree(e.list);
        cudaFree(counter);
        return set_error(GNNAGG_ERR_CUDA, "out of device memory");
    }
    cudaMemsetAsync(counter, 0, sizeof(int), st);
    long_rows_kernel<<<(unsigned)cdiv(a->n, 256), 256, 0, st>>>(a->d_ptr, a->n, EB, e.list, counter);
    fixup_records_kernel<<<(unsigned)cdiv(items, 256), 256, 0, st>>>(p, EB, items, e.records);
    cudaError_t err = cudaMemcpyAsync(&e.count, counter, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    cudaFree(counter);
    if (err != cudaSuccess) {
        cudaFree(e.list);
        cudaFree(e.records);
        return set_error(GNNAGG_ERR_CUDA, cudaGetErrorString(err));
    }
    a->launches += 2;
    a->long_rows.push_back(e);
    *list = e.list;
    *count = e.count;
    *records = e.records;
    return GNNAGG_OK;
}

template <int MODE, bool SCHED>
static int launch_agg(gnnagg_aggregator *a, AggParams p, cudaStream_t st)
{
    if (p.row_hi == 0 && p.edge_hi == 0) {  // callers that do not set a row range get the whole graph
        p.row_lo = 0, p.row_hi = p.num_rows, p.edge_lo = 0, p.edge_hi = p.num_edges;
    }
    if (p.edge_hi <= p.edge_lo) return GNNAGG_OK;
    PROF_RECORD(a, 1, st);
    if (warp_edges_for(a, p.num_edges) == 128)
        launch_agg_we<MODE, SCHED, 128>(p, st);
    else
        launch_agg_we<MODE, SCHED, kWarpEdges>(p, st);
    LAUNCH_CHECK(a);
    PROF_RECORD(a, 2, st);
    if (!SCHED && !mode_emits_edges(MODE)) {
        const int EB = item_edges_for(a, p.F, p.num_edges);
        const int64_t items = cdiv(p.num_edges, EB);
        const int64_t range_items = cdiv(p.edge_hi, EB) - p.edge_lo / EB;  // items touched by the launched range
        if (range_items > 1) {
            const int *list = nullptr;
            const int2 *records = nullptr;
            int num_long = 0;
            if (int rc = long_rows_of(a, p, EB, st, &list, &num_long, &records)) return rc;
            const int lanes = lanes_for(p.F);
            launch_dep(agg_fixup_kernel<MODE>, (unsigned)cdiv(range_items * lanes, 256), 256, st, p, EB, items, records, lanes);
            LAUNCH_CHECK(a);
            if (num_long > 0) {
                launch_dep(agg_fixup_long_kernel<MODE>, (unsigned)cdiv(num_long, 8), 256, st, p, EB, list, num_long);
                LAUNCH_CHECK(a);
            }
        }
    }
    return GNNAGG_OK;
}

static int aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// rows [row_lo, row_hi) of the un-scheduled aggregation (row_hi < 0: all rows); Y is indexed by GLOBAL row
static int gcn_run_core(gnnagg_aggregator *a, const float *X, float *Y, int F, int scheduled, cudaStream_t st,
                        int accumulate = 0, int row_lo = 0, int row_hi = -1, int edge_lo = 0, int edge_hi = 0)
{
    if (a && a->n == 0) return GNNAGG_OK;  // an empty row block (possible after edge-balanced partitioning)
    if (!a || !X || !Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run: NULL argument");
    if (int rc = check_feat(F)) return rc;
    if (!aligned16(X) || !aligned16(Y)) return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
    if (!a->d_val && a->m > 0) return set_error(GNNAGG_ERR_STATE, "gnnagg_gcn_run: edge values not set (gnnagg_set_val)");
    AggParams p{};
    p.X = X;
    p.Y = Y;
    p.F = F;
    if (scheduled) {
        if (a->sched_kind == GNNAGG_SCHED_NOP) return set_error(GNNAGG_ERR_STATE, "scheduled run before schedule");
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));  // aggr_gcn.h:393
        if (a->sched_edges == 0) return GNNAGG_OK;
        p.ptr = a->s_ptr;
        p.idx = a->s_idx;
        p.val = a->s_val;
        p.target = a->s_target;
        p.item_row = a->s_item_row;
        p.num_rows = a->num_target;
        p.num_edges = a->sched_edges;
        p.num_fine_items = a->sched_items;
        p.bulk_ok = aligned16(p.idx) && aligned16(p.val);
        return launch_agg<kModeGCN, true>(a, p, st);
    }
    if (a->m == 0) {
        if (!accumulate) CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(a, F, a->m);
    if (int rc = ensure(a->carry, a->carry_cap, (size_t)cdiv(a->m, EB) * F)) return rc;
    p.num_fine_items = a->num_items;
    p.accumulate = accumulate;
    p.out_row = a->out_row;
    p.ptr = a->d_ptr;
    p.idx = a->d_idx;
    p.val = a->d_val;
    p.item_row = a->d_item_row;
    p.carry = a->carry;
    p.num_rows = a->n;
    p.num_edges = a->m;
    p.bulk_ok = aligned16(p.idx) && aligned16(p.val);
    if (row_hi >= 0) {
        p.row_lo = row_lo, p.row_hi = row_hi, p.edge_lo = edge_lo, p.edge_hi = edge_hi;
        if (row_hi <= row_lo) return GNNAGG_OK;
        if (edge_hi <= edge_lo) {  // a chunk of empty rows
            if (!accumulate) CUDA_TRY(cudaMemsetAsync(Y + (size_t)row_lo * F, 0, (size_t)(row_hi - row_lo) * F * sizeof(float), st));
            return GNNAGG_OK;
        }
    }
    return launch_agg<kModeGCN, false>(a, p, st);
}

// host mirror of the row pointers (needed to cut row chunks)
static int host_ptr(gnnagg_aggregator *a, const int **out)
{
    if (a->h_ptr_user) {
        *out = a->h_ptr_user;
        return GNNAGG_OK;
    }
    if (a->h_ptr.empty()) {
        a->h_ptr.resize((size_t)a->n + 1);
        CUDA_TRY(cudaMemcpy(a->h_ptr.data(), a->d_ptr, a->h_ptr.size() * sizeof(int), cudaMemcpyDeviceToHost));
    }
    *out = a->h_ptr.data();
    return GNNAGG_OK;
}

// edge-balanced row chunk boundaries: bounds[0..chunks]
static void row_chunks(const int *hp, int n, int m, int chunks, int *bounds)
{
    bounds[0] = 0;
    for (int c = 1; c < chunks; ++c) {
        const int64_t target = (int64_t)m * c / chunks;
        int lo = bounds[c - 1], hi = n;  // first row with ptr[row] >= target
        while (lo < hi) {
            const int mid = lo + (hi - lo) / 2;
            if (hp[mid] >= target)
                hi = mid;
            else
                lo = mid + 1;
        }
        bounds[c] = lo;
    }
    bounds[chunks] = n;
}

static int ensure_copy_stream(gnnagg_aggregator *a)
{
    if (a->copy_stream) return GNNAGG_OK;
    CUDA_TRY(cudaStreamCreateWithFlags(&a->copy_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 8; ++i) CUDA_TRY(cudaEventCreateWithFlags(&a->chunk_done[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&a->copies_done, cudaEventDisableTiming));
    return GNNAGG_OK;
}

static int gat_run_core(gnnagg_aggregator *a, const float *X, const float *att, float *Y, int F, float slope,
                        int scheduled, cudaStream_t st)
{
    if (a && a->n == 0) return GNNAGG_OK;
    if (!a || !X || !Y || !att) return set_error(GNNAGG_ERR_ARG, "gnnagg_gat_run: NULL argument");
    if (int rc = check_feat(F)) return rc;
    if (!aligned16(X) || !aligned16(Y)) return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
    if (int rc = ensure(a->den_row, a->den_row_cap, (size_t)a->n)) return rc;
    AggParams p{};
    p.X = X;
    p.Y = Y;
    p.att = att;
    p.F = F;
    p.slope = slope;
    p.den_row = a->den_row;
    if (scheduled) {
        if (a->sched_kind == GNNAGG_SCHED_NOP) return set_error(GNNAGG_ERR_STATE, "scheduled run before schedule");
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));
        if (a->sched_edges == 0) return GNNAGG_OK;
        CUDA_TRY(cudaMemsetAsync(a->den_row, 0, (size_t)a->n * sizeof(float), st));
        if (int rc = ensure(a->newval, a->newval_cap, (size_t)a->sched_edges)) return rc;
        p.ptr = a->s_ptr;
        p.idx = a->s_idx;
        p.target = a->s_target;
        p.item_row = a->s_item_row;
        p.newval = a->newval;
        p.num_rows = a->num_target;
        p.num_edges = a->sched_edges;
        p.num_fine_items = a->sched_items;
        p.bulk_ok = aligned16(p.idx);
        if (int rc = launch_agg<kModeGAT, true>(a, p, st)) return rc;
        const int64_t total4 = (int64_t)a->n * F / 4;
        gat_scale_kernel<<<(unsigned)cdiv(total4, 256), 256, 0, st>>>(Y, a->den_row, F, total4);
        LAUNCH_CHECK(a);
        return GNNAGG_OK;
    }
    if (a->m == 0) {
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(a, F, a->m);
    if (int rc = ensure(a->carry, a->carry_cap, (size_t)cdiv(a->m, EB) * F)) return rc;
    if (int rc = ensure(a->carry_den, a->carry_den_cap, (size_t)cdiv(a->m, EB))) return rc;
    p.num_fine_items = a->num_items;
    p.ptr = a->d_ptr;
    p.idx = a->d_idx;
    p.item_row = a->d_item_row;
    p.carry = a->carry;
    p.carry_den = a->carry_den;
    p.num_rows = a->n;
    p.num_edges = a->m;
    p.bulk_ok = aligned16(p.idx);
    return launch_agg<kModeGAT, false>(a, p, st);
}

static int mlp_run_core(gnnagg_aggregator *a, const float *P, float *Y, int F, int scheduled, cudaStream_t st)
{
    AggParams p{};
    p.X = P;
    p.P = P;
    p.Y = Y;
    p.F = F;
    if (scheduled) {
        if (a->sched_kind == GNNAGG_SCHED_NOP) return set_error(GNNAGG_ERR_STATE, "scheduled run before schedule");
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));  // aggr_nn.h:314
        if (a->sched_edges == 0) return GNNAGG_OK;
        p.ptr = a->s_ptr;
        p.idx = a->s_idx;
        p.target = a->s_target;
        p.item_row = a->s_item_row;
        p.num_rows = a->num_target;
        p.num_edges = a->sched_edges;
        p.num_fine_items = a->sched_items;
        p.bulk_ok = aligned16(p.idx);
        return launch_agg<kModeMLP, true>(a, p, st);
    }
    if (a->m == 0) {
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(a, F, a->m);
    if (int rc = ensure(a->carry, a->carry_cap, (size_t)cdiv(a->m, EB) * F)) return rc;
    p.num_fine_items = a->num_items;
    p.ptr = a->d_ptr;
    p.idx = a->d_idx;
    p.item_row = a->d_item_row;
    p.carry = a->carry;
    p.num_rows = a->n;
    p.num_edges = a->m;
    p.bulk_ok = aligned16(p.idx);
    return launch_agg<kModeMLP, false>(a, p, st);
}

static void free_slices(gnnagg_aggregator *a);
static int merged_view(gnnagg_aggregator *a, cudaStream_t st, gnnagg_aggregator **out);

// builds the source slices on first use and (re)mirrors the edge values into slice order
static int ensure_slices(gnnagg_aggregator *a, int want, cudaStream_t st, bool compact = false)
{
    if (a->num_slices != want) {
        free_slices(a);
        const int width = (int)cdiv(a->n, want);
        if (int rc = source_slices_build_device(a->d_ptr, a->d_idx, a->d_item_row, a->num_items, a->n, a->m, want, width,
                                                &a->sl_ptr, &a->sl_idx, &a->sl_perm, a->sl_off, a->sl_cnt, st))
            return rc;
        const size_t padded = (size_t)a->m + 4 * (size_t)want;
        if (cudaMalloc((void **)&a->sl_val, padded * sizeof(float)) != cudaSuccess) {
            free_slices(a);
            return set_error(GNNAGG_ERR_CUDA, "host pipeline: out of device memory for the source slices");
        }
        for (int c = 0; c < want; ++c) {
            gnnagg_aggregator *s = new gnnagg_aggregator();
            a->slice[c] = s;
            s->d_ptr = a->sl_ptr + (size_t)c * ((size_t)a->n + 1);
            s->d_idx = a->sl_idx + a->sl_off[c];
            s->d_val = a->sl_val + a->sl_off[c];
            s->n = a->n;
            s->m = a->sl_cnt[c];
            s->warp_edges = a->warp_edges ? a->warp_edges : (a->m < kSmallGraphEdges ? 128 : kWarpEdges);  // as the whole graph
            if (compact && c > 0) {
                // slices behind the first only ADD to rows that have edges in them: keep those rows only (slice 0 stays
                // complete: it is the pass that writes every row, zeros included)
                int rows = 0;
                if (int rc = compact_rows_device(s->d_ptr, a->n, &s->c_ptr, &s->out_row, &rows, st)) {
                    free_slices(a);
                    return rc;
                }
                s->d_ptr = s->c_ptr;
                s->n = rows;
            }
            if (int rc = build_item_rows(s, s->d_ptr, s->n, s->m, &s->d_item_row, &s->num_items, st)) {
                free_slices(a);
                return rc;
            }
        }
        a->num_slices = want;
        a->slice_width = width;
        a->launches += 6 + 3 * want;
    }
    if (a->sl_val_of != a->d_val) {
        for (int c = 0; c < want; ++c) {
            if (a->sl_cnt[c] == 0) continue;
            gather_val_kernel<<<(unsigned)cdiv(a->sl_cnt[c], 256), 256, 0, st>>>(a->d_val, a->sl_perm + a->sl_off[c],
                                                                              a->sl_val + a->sl_off[c], a->sl_cnt[c]);
            LAUNCH_CHECK(a);
        }
        a->sl_val_of = a->d_val;
    }
    return GNNAGG_OK;
}


// how many source slices the device-resident un-scheduled aggregation uses for this feature width (1 = none)
static int locality_slices_for(const gnnagg_aggregator *a, int F)
{
    if (a->loc_slices >= 1) return a->loc_slices < kMaxSlices ? a->loc_slices : kMaxSlices;
    // automatic: worth it when X is many times the L2 (the gathers of a slice then stay resident where those of the
    // whole graph do not) and rows are long enough that the extra passes over Y stay small next to the gathers
    int dev = 0, l2 = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev) != cudaSuccess || l2 <= 0)
        return 1;
    const double x_bytes = 4.0 * (double)a->n * F;
    if (x_bytes < kLocalityMinL2Multiples * (double)l2 || a->m < kSmallGraphEdges) return 1;
    if ((double)a->m < kLocalityMinDegree * (double)a->n) return 1;
    int S = (int)(x_bytes / (kLocalitySliceL2Multiples * (double)l2) + 0.999);
    return S < 2 ? 1 : (S > kLocalityMaxAuto ? kLocalityMaxAuto : S);
}

// Y (+)= A X slice by slice over the source ranges; same result as the un-sliced run up to fp32 summation order
static int gcn_run_sliced(gnnagg_aggregator *a, const float *X, float *Y, int F, int S, cudaStream_t st, int accumulate)
{
    if (!a->loc) {
        a->loc = new gnnagg_aggregator();
        a->loc->d_ptr = a->d_ptr;
        a->loc->d_idx = a->d_idx;
        a->loc->n = a->n;
        a->loc->m = a->m;
        a->loc->d_item_row = a->d_item_row;  // borrowed
        a->loc->num_items = a->num_items;
    }
    a->loc->warp_edges = a->warp_edges;
    a->loc->d_val = a->d_val;
    const int64_t before_build = a->loc->launches;
    if (int rc = ensure_slices(a->loc, S, st, true)) return rc;
    a->launches += a->loc->launches - before_build;
    PROF_RECORD(a, 1, st);
    for (int c = 0; c < S; ++c) {
        gnnagg_aggregator *s = a->loc->slice[c];
        const int64_t before = s->launches;
        if (int rc = gcn_run_core(s, X, Y, F, 0, st, accumulate || c > 0)) return rc;
        a->launches += s->launches - before;
    }
    PROF_RECORD(a, 2, st);
    return GNNAGG_OK;
}

// timing brackets: ev[0] call entry, ev[3] end of the aggregation part, ev[4] end of the call
static int gcn_run_impl(gnnagg_aggregator *a, const float *X, float *Y, int F, int scheduled, cudaStream_t st,
                        bool last = true, int accumulate = 0)
{
    if (a) PROF_RECORD(a, 0, st);
    if (a && a->prof) {  // so that a call that launches no aggregation kernel still reads as 0 ms
        CUDA_TRY(cudaEventRecord(a->ev[1], st));
        CUDA_TRY(cudaEventRecord(a->ev[2], st));
    }
    int S = 1;
    if (a && !scheduled && a->n > 0 && a->m > 0 && X && Y && check_feat(F) == GNNAGG_OK && a->d_val) S = locality_slices_for(a, F);
    if (S > 1) {
        if (!aligned16(X) || !aligned16(Y)) return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
        if (int rc = gcn_run_sliced(a, X, Y, F, S, st, accumulate)) return rc;
    } else {
        gnnagg_aggregator *t = a;
        if (a && !scheduled)
            if (int rc = merged_view(a, st, &t)) return rc;
        const int64_t before = t ? t->launches : 0;
        const int rc = gcn_run_core(t, X, Y, F, scheduled, st, accumulate);
        if (t != a) a->launches += t->launches - before;
        if (rc) return rc;
    }
    PROF_RECORD(a, 3, st);
    if (last) PROF_RECORD(a, 4, st);
    return GNNAGG_OK;
}

static int gat_run_impl(gnnagg_aggregator *a, const float *X, const float *att, float *Y, int F, float slope,
                        int scheduled, cudaStream_t st)
{
    if (a) PROF_RECORD(a, 0, st);
    if (a && a->prof) {
        CUDA_TRY(cudaEventRecord(a->ev[1], st));
        CUDA_TRY(cudaEventRecord(a->ev[2], st));
    }
    if (int rc = gat_run_core(a, X, att, Y, F, slope, scheduled, st)) return rc;
    PROF_RECORD(a, 3, st);
    PROF_RECORD(a, 4, st);
    return GNNAGG_OK;
}

// out[v * ostride] = sum over row v of in[e], rows and edges as described by g; deterministic.
// `a` owns the carry scratch (sized for ITS item count: g must describe a's graph).
template <int SRC = kSumArray>
static int rowsum_impl(gnnagg_aggregator *a, const float *in, float *out, cudaStream_t st, int ostride = 1, float slope = 0.f)
{
    if (a->m == 0) {
        if (ostride == 1)
            CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)a->n * sizeof(float), st));
        else if (a->n > 0)
            CUDA_TRY(cudaMemset2DAsync(out, (size_t)ostride * sizeof(float), 0, sizeof(float), (size_t)a->n, st));
        return GNNAGG_OK;
    }
    const int64_t items = cdiv(a->m, kRowsumItem);
    if (int rc = ensure(a->carry_den, a->carry_den_cap, (size_t)items)) return rc;
    const EdgeParams g = edge_params(a);
    const unsigned grid = (unsigned)cdiv(items, 256);
    rowsum_kernel<SRC><<<grid, 256, 0, st>>>(g, in, slope, out, a->carry_den, ostride);
    LAUNCH_CHECK(a);
    if (items > 1) {
        rowsum_fixup_kernel<1><<<grid, 256, 0, st>>>(g, out, a->carry_den, ostride);
        LAUNCH_CHECK(a);
        if (items > kRowsumChunk + 1) {
            rowsum_fixup_kernel<2><<<grid, 256, 0, st>>>(g, out, a->carry_den, ostride);
            LAUNCH_CHECK(a);
        }
    }
    return GNNAGG_OK;
}

static void free_long_rows(gnnagg_aggregator *a)
{
    for (auto &e : a->long_rows) cudaFree(e.list), cudaFree(e.records);
    a->long_rows.clear();
}

static void free_slices(gnnagg_aggregator *a)
{
    for (int c = 0; c < kMaxSlices; ++c) {
        if (!a->slice[c]) continue;
        cudaFree(a->slice[c]->d_item_row);
        cudaFree(a->slice[c]->carry);
        cudaFree(a->slice[c]->c_ptr);
        cudaFree(a->slice[c]->out_row);
        free_long_rows(a->slice[c]);
        delete a->slice[c];
        a->slice[c] = nullptr;
    }
    cudaFree(a->sl_ptr), cudaFree(a->sl_idx), cudaFree(a->sl_perm), cudaFree(a->sl_val);
    a->sl_ptr = a->sl_idx = a->sl_perm = nullptr;
    a->sl_val = nullptr;
    a->sl_val_of = nullptr;
    a->num_slices = 0;
}

static void free_transpose(gnnagg_aggregator *a)
{
    if (a->tr) {
        cudaFree(a->tr->d_item_row);
        cudaFree(a->tr->carry);
        cudaFree(a->tr->carry_den);
        cudaFree(a->tr->den_row);
        free_long_rows(a->tr);
        delete a->tr;
        a->tr = nullptr;
    }
    cudaFree(a->t_ptr), cudaFree(a->t_idx), cudaFree(a->t_perm), cudaFree(a->t_val);
    a->t_ptr = a->t_idx = a->t_perm = nullptr;
    a->t_val = nullptr;
    a->t_val_of = nullptr;
    a->num_src = 0;
}

static void free_merged(gnnagg_aggregator *a)
{
    if (a->mg) {
        cudaFree(a->mg->d_item_row);
        cudaFree(a->mg->carry);
        free_long_rows(a->mg);
        delete a->mg;  // its timing events are the parent's
        a->mg = nullptr;
    }
    cudaFree(a->mg_ptr), cudaFree(a->mg_idx), cudaFree(a->mg_start), cudaFree(a->mg_val);
    a->mg_ptr = a->mg_idx = a->mg_start = nullptr;
    a->mg_val = nullptr;
    a->mg_val_of = nullptr;
}

// whether the un-scheduled, un-sliced GCN aggregation runs on the merged view (after ensure_merged)
static bool merged_in_use(const gnnagg_aggregator *a)
{
    return a->mg && (a->merge_mode == 2 || (a->merge_mode == 0 && a->merge_auto == 1));
}

// builds the merged view when the setting asks for it; automatic: takes the decision once (kMergeMin*) from a count of
// m', so that a graph the rule leaves alone pays one counting pass and no m-sized allocation
static int ensure_merged(gnnagg_aggregator *a, cudaStream_t st)
{
    if (a->merge_mode == 1 || a->n == 0 || a->m == 0) return GNNAGG_OK;
    if (a->merge_mode == 0 && a->merge_auto < 0) {
        int mm = a->m;
        if (a->m >= kMergeMinEdges) {
            if (int rc = merge_count_device(a->d_ptr, a->d_idx, a->n, a->m, &mm, st)) return rc;
            a->launches += 2;
        }
        a->merge_auto = (double)(a->m - mm) >= kMergeMinFraction * (double)a->m && a->m >= kMergeMinEdges;
    }
    if (a->merge_mode == 0 && a->merge_auto == 0) return GNNAGG_OK;
    if (!a->mg) {
        int mm = 0;
        if (int rc = merge_build_device(a->d_ptr, a->d_idx, a->n, a->m, &a->mg_ptr, &a->mg_idx, &a->mg_start, &mm, st))
            return rc;
        a->launches += 5;  // run heads, row heads, scan (counted once), compaction, row pointers
        if (cudaMalloc((void **)&a->mg_val, (size_t)(mm ? mm : 1) * sizeof(float)) != cudaSuccess) {
            free_merged(a);
            return set_error(GNNAGG_ERR_CUDA, "merged view: out of device memory");
        }
        gnnagg_aggregator *g = new gnnagg_aggregator();
        g->d_ptr = a->mg_ptr;
        g->d_idx = a->mg_idx;
        g->d_val = a->mg_val;
        g->n = a->n;
        g->m = mm;
        g->merge_mode = 1;
        a->mg = g;
        if (int rc = build_item_rows(g, g->d_ptr, g->n, g->m, &g->d_item_row, &g->num_items, st)) {
            free_merged(a);
            return rc;
        }
        a->launches += g->launches;
        g->launches = 0;
    }
    return GNNAGG_OK;
}

// the aggregator the un-scheduled, un-sliced GCN aggregation of `a` runs on: the merged view when it is in use (its
// values re-summed on `st` when the edge values changed), else `a` itself
static int merged_view(gnnagg_aggregator *a, cudaStream_t st, gnnagg_aggregator **out)
{
    *out = a;
    if (a->merge_mode == 1 || !a->d_val) return GNNAGG_OK;
    if (int rc = ensure_merged(a, st)) return rc;
    if (!merged_in_use(a)) return GNNAGG_OK;
    gnnagg_aggregator *g = a->mg;
    if (a->mg_val_of != a->d_val) {
        merge_val_kernel<<<(unsigned)cdiv(g->m, 256), 256, 0, st>>>(a->d_val, a->mg_start, a->mg_val, g->m);
        LAUNCH_CHECK(a);
        a->mg_val_of = a->d_val;
    }
    g->warp_edges = a->warp_edges;
    g->prof = a->prof;  // the aggregation kernel's events are the parent's (gnnagg_profile_read)
    for (int i = 0; i < 5; ++i) g->ev[i] = a->ev[i];
    *out = g;
    return GNNAGG_OK;
}

// t_val[j] = src[t_perm[j]]: edge data into transposed order
static int to_transposed(gnnagg_aggregator *a, const float *src, float *dst, cudaStream_t st)
{
    if (a->m == 0) return GNNAGG_OK;
    gather_val_kernel<<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(src, a->t_perm, dst, a->m);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

}  // namespace gnnagg

extern "C" {

int gnnagg_version(void) { return 100; }
const char *gnnagg_last_error(void) { return g_error.c_str(); }

int gnnagg_device_info(int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len)
{
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, dev));
    if (sm_count) *sm_count = prop.multiProcessorCount;
    if (cc_major) *cc_major = prop.major;
    if (cc_minor) *cc_minor = prop.minor;
    if (name && name_len > 0) {
        strncpy(name, prop.name, (size_t)name_len - 1);
        name[name_len - 1] = 0;
    }
    return GNNAGG_OK;
}

int gnnagg_create(const int *d_ptr, const int *d_idx, const int *h_ptr, const int *h_idx, int num_v, int num_e,
                  gnnagg_aggregator **out)
{
    // legacy-stream variant (what the reference's constructors do): returns with the set-up kernel complete, so a run
    // issued on ANY stream right afterwards is ordered behind it
    const int rc = gnnagg_create_on(d_ptr, d_idx, h_ptr, h_idx, num_v, num_e, out, nullptr);
    if (rc == GNNAGG_OK) CUDA_TRY(cudaStreamSynchronize(0));
    return rc;
}

int gnnagg_create_on(const int *d_ptr, const int *d_idx, const int *h_ptr, const int *h_idx, int num_v, int num_e,
                     gnnagg_aggregator **out, void *stream)
{
    if (!out || !d_ptr || (num_e > 0 && !d_idx) || num_v < 0 || num_e < 0)
        return set_error(GNNAGG_ERR_ARG, "gnnagg_create: bad argument");
    gnnagg_aggregator *a = new gnnagg_aggregator();
    a->d_ptr = d_ptr;
    a->d_idx = d_idx;
    a->h_ptr_user = h_ptr;
    a->h_idx_user = h_idx;
    a->n = num_v;
    a->m = num_e;
    const int rc = build_item_rows(a, d_ptr, num_v, num_e, &a->d_item_row, &a->num_items, (cudaStream_t)stream);
    if (rc != GNNAGG_OK) {
        delete a;
        return rc;
    }
    *out = a;
    return GNNAGG_OK;
}

int gnnagg_destroy(gnnagg_aggregator *a)
{
    if (!a) return GNNAGG_OK;
    free_schedule(a);
    free_transpose(a);
    free_slices(a);
    if (a->loc) {
        free_slices(a->loc);  // its CSR and item table are this aggregator's
        delete a->loc;
        a->loc = nullptr;
    }
    free_merged(a);
    free_long_rows(a);
    for (int i = 0; i < 8; ++i)
        if (a->in_done[i]) cudaEventDestroy(a->in_done[i]);
    if (a->in_free) cudaEventDestroy(a->in_free);
    if (a->in_stream) cudaStreamDestroy(a->in_stream);
    cudaFree(a->bwd_c);
    cudaFree(a->bwd_wt);
    cudaFree(a->bwd_part);
    cudaFree(a->bwd_carry);
    cudaFree(a->bwd_t);
    cudaFree(a->d_item_row);
    cudaFree(a->carry);
    cudaFree(a->den_row);
    cudaFree(a->carry_den);
    cudaFree(a->newval);
    cudaFree(a->ax);
    cudaFree(a->st_in);
    cudaFree(a->st_out);
    cudaFree(a->st_w);
    cudaFree(a->st_att);
    for (int i = 0; i < 5; ++i)
        if (a->ev[i]) cudaEventDestroy(a->ev[i]);
    for (int i = 0; i < 8; ++i)
        if (a->chunk_done[i]) cudaEventDestroy(a->chunk_done[i]);
    if (a->copies_done) cudaEventDestroy(a->copies_done);
    if (a->copy_stream) cudaStreamDestroy(a->copy_stream);
    delete a;
    return GNNAGG_OK;
}

int gnnagg_set_val(gnnagg_aggregator *a, const float *d_val)
{
    const int rc = gnnagg_set_val_on(a, d_val, nullptr);
    if (rc == GNNAGG_OK && a->s_perm) CUDA_TRY(cudaStreamSynchronize(0));  // the permuted copy is complete on return
    return rc;
}

int gnnagg_set_val_on(gnnagg_aggregator *a, const float *d_val, void *stream)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_set_val: NULL aggregator");
    a->d_val = d_val;
    a->t_val_of = nullptr;  // same pointer, possibly new contents (aggr_gcn.h:540-544): re-mirror on the next backward
    a->sl_val_of = nullptr;
    a->mg_val_of = nullptr;
    if (a->loc) a->loc->sl_val_of = nullptr;
    if (a->sched_kind == GNNAGG_SCHED_NOP) return GNNAGG_OK;
    if (a->s_perm) {  // locality kinds keep a permuted copy (aggr_gcn.h:522-537)
        if (!a->s_val) CUDA_TRY(cudaMalloc((void **)&a->s_val, (size_t)(a->sched_edges ? a->sched_edges : 1) * sizeof(float)));
        if (d_val && a->sched_edges > 0) {
            gather_val_kernel<<<(unsigned)cdiv(a->sched_edges, 256), 256, 0, (cudaStream_t)stream>>>(d_val, a->s_perm, a->s_val,
                                                                                                  a->sched_edges);
            LAUNCH_CHECK(a);
        }
    } else {
        a->s_val = const_cast<float *>(d_val);  // d_val_scheduled = d_val (aggr_gcn.h:506,542)
    }
    return GNNAGG_OK;
}

int gnnagg_schedule_apply(gnnagg_aggregator *a, int kind, const int *params, int nparams, int total_num_v)
{
    if (!a || !params || nparams < 1) return set_error(GNNAGG_ERR_ARG, "gnnagg_schedule_apply: bad argument");
    if (kind == GNNAGG_SCHED_LOCALITY_NEIGHBOR_GROUPING && nparams < 2)
        return set_error(GNNAGG_ERR_ARG, "locality_neighbor_grouping needs {par_num, neighbor_num}");
    int par = 0, ng = 0;
    if (kind == GNNAGG_SCHED_NEIGHBOR_GROUPING)
        ng = params[0];
    else if (kind == GNNAGG_SCHED_LOCALITY)
        par = params[0];
    else if (kind == GNNAGG_SCHED_LOCALITY_NEIGHBOR_GROUPING)
        par = params[0], ng = params[1];
    else
        return set_error(GNNAGG_ERR_ARG, "gnnagg_schedule_apply: unknown kind");

    // built on the device (sched_device.cu); bit-identical to the host builders of gnnagg_schedule_build.
    // Neighbour grouping keeps the CSR edge order (graph_schedule.h:123-124): idx and val are aliased, not copied.
    int *sp = nullptr, *si = nullptr, *stg = nullptr, *sperm = nullptr, nt = 0, se = 0;
    if (int rc = schedule_build_device(kind, a->d_ptr, a->d_idx, a->d_item_row, a->num_items, a->n, a->m, par, ng,
                                       total_num_v, &sp, &si, &stg, &sperm, &nt, &se, 0))
        return rc;
    free_schedule(a);
    a->sched_kind = kind;
    a->neighbor_group_size = ng;
    a->locality_partition_num = par;
    a->num_target = nt;
    a->sched_edges = se;
    a->s_ptr = sp;
    a->s_target = stg;
    a->s_perm = sperm;
    if (si) {
        a->s_idx = si;
        a->s_idx_owned = true;
    } else {
        a->s_idx = const_cast<int *>(a->d_idx);
    }
    if (int rc = build_item_rows(a, a->s_ptr, a->num_target, a->sched_edges, &a->s_item_row, &a->sched_items, 0))
        return rc;
    if (int rc = gnnagg_set_val(a, a->d_val)) return rc;
    CUDA_TRY(cudaStreamSynchronize(0));
    return GNNAGG_OK;
}

int gnnagg_schedule_kind(const gnnagg_aggregator *a) { return a ? a->sched_kind : GNNAGG_SCHED_NOP; }

int gnnagg_sched_to_csr_order(gnnagg_aggregator *a, const float *in_sched, float *out_csr, void *stream)
{
    if (!a || (a->m > 0 && (!in_sched || !out_csr))) return set_error(GNNAGG_ERR_ARG, "gnnagg_sched_to_csr_order: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (!a->s_perm) {  // no schedule, or neighbour grouping: the scheduled order IS the CSR order
        if (in_sched != out_csr) CUDA_TRY(cudaMemcpyAsync(out_csr, in_sched, (size_t)a->m * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return GNNAGG_OK;
    }
    if (in_sched == out_csr) return set_error(GNNAGG_ERR_ARG, "gnnagg_sched_to_csr_order: in place is not possible after a locality schedule");
    if (a->sched_edges != a->m)
        return set_error(GNNAGG_ERR_STATE, "gnnagg_sched_to_csr_order: the schedule dropped edges (sources outside the slice range)");
    scatter_val_kernel<<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(in_sched, a->s_perm, out_csr, a->m);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_num_target(const gnnagg_aggregator *a) { return a ? a->num_target : 0; }
const int *gnnagg_sched_dev_ptr(const gnnagg_aggregator *a) { return a ? a->s_ptr : nullptr; }
const int *gnnagg_sched_dev_idx(const gnnagg_aggregator *a) { return a ? a->s_idx : nullptr; }
const int *gnnagg_sched_dev_target(const gnnagg_aggregator *a) { return a ? a->s_target : nullptr; }
const float *gnnagg_sched_dev_val(const gnnagg_aggregator *a) { return a ? a->s_val : nullptr; }
const float *gnnagg_gat_edge_weights(const gnnagg_aggregator *a) { return a ? a->newval : nullptr; }
int64_t gnnagg_launch_count(const gnnagg_aggregator *a) { return a ? a->launches : 0; }

int gnnagg_set_warp_edges(gnnagg_aggregator *a, int warp_edges)
{
    if (!a || (warp_edges != 0 && warp_edges != 128 && warp_edges != 512))
        return set_error(GNNAGG_ERR_ARG, "gnnagg_set_warp_edges: 0, 128 or 512");
    a->warp_edges = warp_edges;
    if (a->tr) a->tr->warp_edges = warp_edges;
    return GNNAGG_OK;
}

int gnnagg_set_locality_slices(gnnagg_aggregator *a, int slices)
{
    if (!a || slices < 0 || slices > kMaxSlices) return set_error(GNNAGG_ERR_ARG, "gnnagg_set_locality_slices: 0 (automatic), 1 (off) .. 16");
    a->loc_slices = slices;
    return GNNAGG_OK;
}

int gnnagg_set_merge_duplicates(gnnagg_aggregator *a, int mode)
{
    if (!a || mode < 0 || mode > 2) return set_error(GNNAGG_ERR_ARG, "gnnagg_set_merge_duplicates: 0 (automatic), 1 (off), 2 (on)");
    a->merge_mode = mode;  // a view already built stays until gnnagg_destroy: switching back costs no rebuild
    return GNNAGG_OK;
}

int gnnagg_merged_edges(gnnagg_aggregator *a)
{
    if (!a) return set_error(-1, "gnnagg_merged_edges: NULL aggregator");
    if (ensure_merged(a, nullptr) != GNNAGG_OK) return -1;
    return merged_in_use(a) ? a->mg->m : a->m;
}

int gnnagg_merged_dev(const gnnagg_aggregator *a, const int **ptr, const int **idx, const float **val)
{
    if (!a || !merged_in_use(a)) return set_error(GNNAGG_ERR_STATE, "gnnagg_merged_dev: the merged view is not in use");
    if (ptr) *ptr = a->mg_ptr;
    if (idx) *idx = a->mg_idx;
    if (val) *val = a->mg_val;
    return GNNAGG_OK;
}

int gnnagg_profile_enable(gnnagg_aggregator *a, int on)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_profile_enable: NULL aggregator");
    if (on && !a->ev[0])
        for (int i = 0; i < 5; ++i) CUDA_TRY(cudaEventCreate(&a->ev[i]));
    a->prof = on != 0;
    return GNNAGG_OK;
}

int gnnagg_profile_read(gnnagg_aggregator *a, float *ms)
{
    if (!a || !ms || !a->ev[0]) return set_error(GNNAGG_ERR_STATE, "gnnagg_profile_read: profiling not enabled");
    CUDA_TRY(cudaEventSynchronize(a->ev[4]));
    float agg = 0.f, agg_total = 0.f, dense = 0.f, total = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&agg, a->ev[1], a->ev[2]));
    CUDA_TRY(cudaEventElapsedTime(&agg_total, a->ev[0], a->ev[3]));
    CUDA_TRY(cudaEventElapsedTime(&dense, a->ev[3], a->ev[4]));
    CUDA_TRY(cudaEventElapsedTime(&total, a->ev[0], a->ev[4]));
    ms[0] = agg;
    ms[1] = agg_total - agg;
    ms[2] = dense;
    ms[3] = total;
    return GNNAGG_OK;
}

int gnnagg_memcpy_d2h(void *h_dst, const void *d_src, uint64_t bytes)
{
    if (bytes == 0) return GNNAGG_OK;
    if (!h_dst || !d_src) return set_error(GNNAGG_ERR_ARG, "gnnagg_memcpy_d2h: NULL argument");
    CUDA_TRY(cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return GNNAGG_OK;
}

int gnnagg_prepare(gnnagg_aggregator *a, int feat, void *stream)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_prepare: NULL aggregator");
    if (int rc = check_feat(feat)) return rc;
    if (a->m == 0 || a->n == 0) return GNNAGG_OK;
    gnnagg_aggregator *t = a;
    if (int rc = merged_view(a, (cudaStream_t)stream, &t)) return rc;
    if (t != a) {
        const int64_t before = t->launches;
        const int rc = gnnagg_prepare(t, feat, stream);
        a->launches += t->launches - before;
        return rc;
    }
    const int EB = item_edges_for(a, feat, a->m);
    if (int rc = ensure(a->carry, a->carry_cap, (size_t)cdiv(a->m, EB) * feat)) return rc;
    if (warp_edges_for(a, a->m) == 128)
        preload_gcn_we<128>(feat);
    else
        preload_gcn_we<kWarpEdges>(feat);
    preload(agg_fixup_kernel<kModeGCN>);
    preload(agg_fixup_long_kernel<kModeGCN>);
    AggParams p{};
    p.ptr = a->d_ptr;
    p.item_row = a->d_item_row;
    p.num_rows = a->n;
    p.num_edges = a->m;
    p.num_fine_items = a->num_items;
    const int *list = nullptr;
    const int2 *records = nullptr;
    int num_long = 0;
    if (int rc = long_rows_of(a, p, EB, (cudaStream_t)stream, &list, &num_long, &records)) return rc;
    const int *hp = nullptr;
    return host_ptr(a, &hp);  // row-range launches (gnnagg_gcn_run_rows) cut edge ranges on the host
}

int gnnagg_gcn_run_rows(gnnagg_aggregator *a, const float *X, float *Y, int feat, int accumulate, int row_lo, int row_hi,
                        void *stream)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run_rows: NULL aggregator");
    if (row_lo < 0 || row_hi > a->n || row_lo > row_hi) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run_rows: bad row range");
    if (row_lo == row_hi) return GNNAGG_OK;
    gnnagg_aggregator *t = a;
    if (int rc = merged_view(a, (cudaStream_t)stream, &t)) return rc;
    const int *hp = nullptr;
    if (int rc = host_ptr(t, &hp)) return rc;
    const int64_t before = t->launches;
    const int rc = gcn_run_core(t, X, Y, feat, 0, (cudaStream_t)stream, accumulate != 0, row_lo, row_hi, hp[row_lo], hp[row_hi]);
    if (t != a) a->launches += t->launches - before;
    return rc;
}

int gnnagg_gcn_run(gnnagg_aggregator *a, const float *X, float *Y, int feat, int scheduled, void *stream)
{
    return gcn_run_impl(a, X, Y, feat, scheduled, (cudaStream_t)stream);
}

int gnnagg_gcn_run_acc(gnnagg_aggregator *a, const float *X, float *Y, int feat, int accumulate, void *stream)
{
    return gcn_run_impl(a, X, Y, feat, 0, (cudaStream_t)stream, true, accumulate != 0);
}

int gnnagg_gat_run(gnnagg_aggregator *a, const float *X, const float *att, float *Y, int feat, float slope,
                   int scheduled, void *stream)
{
    return gat_run_impl(a, X, att, Y, feat, slope, scheduled, (cudaStream_t)stream);
}

int gnnagg_dense_nn(const float *A, const float *B, float *C, int64_t M, int N, int K, void *stream)
{
    if (!A || !B || !C || M < 0) return set_error(GNNAGG_ERR_ARG, "gnnagg_dense_nn: bad argument");
    if (M == 0) return GNNAGG_OK;
    return dense_nn_launch(A, B, C, M, N, K, stream);
}

int gnnagg_gcn_layer(gnnagg_aggregator *a, const float *X, const float *W, float *H, float *AX, int feat_in,
                     int feat_out, int scheduled, void *stream)
{
    if (!a || !X || !W || !H) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_layer: NULL argument");
    float *ax = AX;
    if (!ax) {
        if (int rc = ensure(a->ax, a->ax_cap, (size_t)a->n * feat_in)) return rc;
        ax = a->ax;
    }
    if (int rc = gcn_run_impl(a, X, ax, feat_in, scheduled, (cudaStream_t)stream, false)) return rc;
    if (a->n > 0) {
        if (int rc = dense_nn_launch(ax, W, H, a->n, feat_out, feat_in, stream)) return rc;
        a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
    }
    PROF_RECORD(a, 4, (cudaStream_t)stream);
    return GNNAGG_OK;
}

int gnnagg_mlp_run(gnnagg_aggregator *a, const float *X, const float *W, float *Y, int feat, int scheduled,
                   void *stream)
{
    if (a && a->n == 0) return GNNAGG_OK;
    if (!a || !X || !W || !Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_mlp_run: NULL argument");
    if (!aligned16(X) || !aligned16(Y)) return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = ensure(a->ax, a->ax_cap, (size_t)a->n * feat)) return rc;
    PROF_RECORD(a, 0, st);
    if (int rc = dense_nn_launch(X, W, a->ax, a->n, feat, feat, stream)) return rc;  // P = X W, once per call
    a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
    if (a->prof) {
        CUDA_TRY(cudaEventRecord(a->ev[1], st));
        CUDA_TRY(cudaEventRecord(a->ev[2], st));
    }
    if (int rc = mlp_run_core(a, a->ax, Y, feat, scheduled, st)) return rc;
    PROF_RECORD(a, 3, st);
    PROF_RECORD(a, 4, st);
    return GNNAGG_OK;
}

int gnnagg_gcn_run_edgewise(gnnagg_aggregator *a, const float *X, float *Y, int feat, void *stream)
{
    if (!a || !X || !Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run_edgewise: NULL argument");
    if (int rc = check_feat(feat)) return rc;
    if (!a->d_val && a->m > 0) return set_error(GNNAGG_ERR_STATE, "edge values not set");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * feat * sizeof(float), st));  // aggr_gcn.h:447
    if (a->m == 0) return GNNAGG_OK;
    const EdgeParams g = edge_params(a);
    const int lpr = lanes_for(feat);
    const unsigned grid = (unsigned)cdiv(cdiv(a->m, 32 / lpr), 8);
    if (lpr == 8)
        gcn_edgewise_kernel<8><<<grid, 256, 0, st>>>(g, a->d_val, X, Y, feat);
    else if (lpr == 16)
        gcn_edgewise_kernel<16><<<grid, 256, 0, st>>>(g, a->d_val, X, Y, feat);
    else
        gcn_edgewise_kernel<32><<<grid, 256, 0, st>>>(g, a->d_val, X, Y, feat);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_csr2edgelist(gnnagg_aggregator *a, int *d_edgelist, void *stream)
{
    if (!a || (!d_edgelist && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_csr2edgelist: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    csr2edgelist_kernel<<<(unsigned)cdiv(a->m, 256), 256, 0, (cudaStream_t)stream>>>(edge_params(a), d_edgelist);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_u_add_v(gnnagg_aggregator *a, const float *att, float *out_val, void *stream)
{
    if (!a || !att || (!out_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_u_add_v: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    edge_map_kernel<kEdgeUAddV><<<(unsigned)cdiv(a->m, 256), 256, 0, (cudaStream_t)stream>>>(edge_params(a), att, out_val, 0.f);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_add_to_center(gnnagg_aggregator *a, const float *in_val, float *out_center, void *stream)
{
    if (!a || !out_center || (!in_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_add_to_center: NULL argument");
    return rowsum_impl(a, in_val, out_center, (cudaStream_t)stream);
}

int gnnagg_each_div(gnnagg_aggregator *a, const float *in_center, float *inout_val, void *stream)
{
    if (!a || !in_center || (!inout_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_each_div: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    edge_map_kernel<kEdgeDiv><<<(unsigned)cdiv(a->m, 256), 256, 0, (cudaStream_t)stream>>>(edge_params(a), in_center, inout_val, 0.f);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_edge_softmax(gnnagg_aggregator *a, const float *att, float *out_val, float slope, void *stream)
{
    if (!a || !att || (!out_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_edge_softmax: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = ensure(a->den_row, a->den_row_cap, (size_t)a->n)) return rc;
    const EdgeParams g = edge_params(a);
    edge_map_kernel<kEdgeWeight><<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(g, att, out_val, slope);
    LAUNCH_CHECK(a);
    if (int rc = rowsum_impl(a, out_val, a->den_row, st)) return rc;
    edge_map_kernel<kEdgeDiv><<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(g, a->den_row, out_val, 0.f);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_sddmm(gnnagg_aggregator *a, const float *X1, const float *X2, float *out_val, int feat, int scheduled,
                 void *stream)
{
    if (!a || !X1 || !X2 || (!out_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_sddmm: NULL argument");
    if (int rc = check_feat(feat)) return rc;
    if (!aligned16(X1) || !aligned16(X2)) return set_error(GNNAGG_ERR_ARG, "X1 and X2 must be 16-byte aligned");
    // same edge-balanced traversal as the aggregation (agg_kernel, MODE = SDDMM): X1 rows are gathered per edge,
    // the X2 row of the destination stays in registers, per-edge dot products leave through a reduce-scatter
    AggParams p{};
    p.X = X1;
    p.P = X2;
    p.newval = out_val;
    p.F = feat;
    cudaStream_t st = (cudaStream_t)stream;
    if (scheduled) {
        if (a->sched_kind != GNNAGG_SCHED_NEIGHBOR_GROUPING)  // aggr_sddmm.h:100
            return set_error(GNNAGG_ERR_STATE, "scheduled SDDMM needs a neighbor_grouping schedule");
        if (a->sched_edges == 0) return GNNAGG_OK;
        p.ptr = a->s_ptr;
        p.idx = a->s_idx;
        p.target = a->s_target;
        p.item_row = a->s_item_row;
        p.num_rows = a->num_target;
        p.num_edges = a->sched_edges;
        p.num_fine_items = a->sched_items;
        p.bulk_ok = aligned16(p.idx);
        return launch_agg<kModeSDDMM, true>(a, p, st);
    }
    if (a->m == 0) return GNNAGG_OK;
    p.ptr = a->d_ptr;
    p.idx = a->d_idx;
    p.item_row = a->d_item_row;
    p.num_rows = a->n;
    p.num_edges = a->m;
    p.num_fine_items = a->num_items;
    p.bulk_ok = aligned16(p.idx);
    return launch_agg<kModeSDDMM, false>(a, p, st);
}

int gnnagg_transpose_build(gnnagg_aggregator *a, int num_src, void *stream)
{
    if (!a || num_src < 0) return set_error(GNNAGG_ERR_ARG, "gnnagg_transpose_build: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    free_transpose(a);
    if (int rc = transpose_build_device(a->d_ptr, a->d_idx, a->d_item_row, a->num_items, a->n, a->m, num_src, &a->t_ptr,
                                        &a->t_idx, &a->t_perm, st))
        return rc;
    a->num_src = num_src;
    a->tr = new gnnagg_aggregator();
    a->tr->d_ptr = a->t_ptr;
    a->tr->d_idx = a->t_idx;
    a->tr->n = num_src;
    a->tr->m = a->m;
    a->tr->warp_edges = a->warp_edges;
    int rc = build_item_rows(a->tr, a->t_ptr, num_src, a->m, &a->tr->d_item_row, &a->tr->num_items, st);
    if (rc == GNNAGG_OK && cudaMalloc((void **)&a->t_val, (size_t)(a->m ? a->m : 1) * sizeof(float)) != cudaSuccess)
        rc = set_error(GNNAGG_ERR_CUDA, "gnnagg_transpose_build: out of device memory");
    if (rc != GNNAGG_OK) {
        free_transpose(a);  // never leave a half-built transpose behind
        return rc;
    }
    a->tr->d_val = a->t_val;
    a->launches += 5;  // iota, radix sort (counted once), rows, pointers, item table
    return GNNAGG_OK;
}

int gnnagg_transpose_dev(const gnnagg_aggregator *a, int *num_src, const int **t_ptr, const int **t_idx, const int **t_perm)
{
    if (!a || !a->tr) return set_error(GNNAGG_ERR_STATE, "gnnagg_transpose_dev: gnnagg_transpose_build has not run");
    if (num_src) *num_src = a->num_src;
    if (t_ptr) *t_ptr = a->t_ptr;
    if (t_idx) *t_idx = a->t_idx;
    if (t_perm) *t_perm = a->t_perm;
    return GNNAGG_OK;
}

int gnnagg_gcn_backward(gnnagg_aggregator *a, const float *dY, float *dX, int feat, void *stream)
{
    if (!a || !dY || !dX) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_backward: NULL argument");
    if (!a->tr) return set_error(GNNAGG_ERR_STATE, "gnnagg_gcn_backward: gnnagg_transpose_build has not run");
    if (!a->d_val && a->m > 0) return set_error(GNNAGG_ERR_STATE, "gnnagg_gcn_backward: edge values not set (gnnagg_set_val)");
    cudaStream_t st = (cudaStream_t)stream;
    if (a->t_val_of != a->d_val) {
        if (int rc = to_transposed(a, a->d_val, a->t_val, st)) return rc;
        a->t_val_of = a->d_val;
    }
    const int64_t before = a->tr->launches;
    const int rc = gcn_run_core(a->tr, dY, dX, feat, 0, st);
    a->launches += a->tr->launches - before;
    return rc;
}

int gnnagg_gat_backward(gnnagg_aggregator *a, const float *X, const float *att, const float *w, const float *den,
                        const float *Y, const float *dY, float *dX, float *datt, int feat, float slope, void *stream)
{
    if (!a || !X || !Y || !dY || !dX || !datt || (!att && !w))
        return set_error(GNNAGG_ERR_ARG, "gnnagg_gat_backward: NULL argument (att or w must be given)");
    if (!a->tr) return set_error(GNNAGG_ERR_STATE, "gnnagg_gat_backward: gnnagg_transpose_build has not run");
    if (int rc = check_feat(feat)) return rc;
    if (!aligned16(X) || !aligned16(Y) || !aligned16(dY) || !aligned16(dX))
        return set_error(GNNAGG_ERR_ARG, "X, Y, dY and dX must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    // every row < n gets its destination half and every row < num_src its source half from the kernels below; only a
    // rectangular block leaves entries of the [max(n, num_src), 2] table that nobody writes
    const int rows = a->n > a->num_src ? a->n : a->num_src;
    if (a->n != a->num_src || a->m == 0) CUDA_TRY(cudaMemsetAsync(datt, 0, (size_t)rows * 2 * sizeof(float), st));
    if (a->m == 0) {
        CUDA_TRY(cudaMemsetAsync(dX, 0, (size_t)a->num_src * feat * sizeof(float), st));
        return GNNAGG_OK;
    }
    gnnagg_aggregator *t = a->tr;
    const int EB = item_edges_for(a, feat, a->m);
    const int EBt = item_edges_for(t, feat, a->m);
    if (int rc = ensure(a->bwd_c, a->bwd_c_cap, (size_t)a->n)) return rc;
    if (int rc = ensure(a->bwd_wt, a->bwd_wt_cap, (size_t)a->m)) return rc;
    if (int rc = ensure(a->bwd_part, a->bwd_part_cap, (size_t)a->n)) return rc;
    if (int rc = ensure(a->bwd_carry, a->bwd_carry_cap, (size_t)cdiv(a->m, EB) + 1)) return rc;
    if (int rc = ensure(t->carry, t->carry_cap, (size_t)cdiv(a->m, EBt) * feat)) return rc;
    if (int rc = ensure(t->carry_den, t->carry_den_cap, (size_t)cdiv(a->m, EBt))) return rc;
    if (int rc = ensure(t->den_row, t->den_row_cap, (size_t)a->num_src)) return rc;
    const bool large = a->m >= kSmallGraphEdges;  // (w, t) of the graph does not stay in L2: see step 4
    if (large)
        if (int rc = ensure(a->bwd_t, a->bwd_t_cap, (size_t)a->m)) return rc;
    // 1. per destination row: c_v = <Y[v], dY[v]>
    gat_bwd_rowinfo_kernel<<<(unsigned)cdiv((int64_t)a->n * 8, 256), 256, 0, st>>>(Y, dY, a->bwd_c, a->n, feat);
    LAUNCH_CHECK(a);
    // 2. pass 1 over the CSR: g_e = <X[u], dY[v]> (the SDDMM traversal), per edge (w_e, t_e), per row their sums
    {
        AggParams p{};
        p.X = X;
        p.P = dY;
        p.att = att;
        p.val = w;
        p.bwd_c = a->bwd_c;
        p.bwd_wt = a->bwd_wt;
        p.bwd_part = a->bwd_part;
        p.bwd_carry = a->bwd_carry;
        p.F = feat;
        p.slope = slope;
        p.ptr = a->d_ptr;
        p.idx = a->d_idx;
        p.item_row = a->d_item_row;
        p.num_rows = a->n;
        p.num_edges = a->m;
        p.num_fine_items = a->num_items;
        p.bulk_ok = aligned16(p.idx) && (att || aligned16(w));
        if (int rc = launch_agg<kModeGATBWD, false>(a, p, st)) return rc;
    }
    // 3. rows closed: 1 / D_v and the destination half of the attention gradient
    launch_dep(gat_bwd_rowfinal_kernel, (unsigned)cdiv((int64_t)a->n * 8, 256), 256, st, a->d_ptr, a->bwd_part, a->bwd_carry,
               den, a->bwd_c, datt, a->n, EB);
    LAUNCH_CHECK(a);
    if (large) {
        // 4a. large graphs: (w, t) permuted into transposed order by a streaming kernel, then the source half as a row sum
        //     and dX as the plain aggregation over the transposed CSR with edge values alpha
        launch_dep(gat_bwd_permute_kernel, (unsigned)cdiv(a->m, 256), 256, st, (const float2 *)a->bwd_wt, (const int *)a->t_perm,
                   (const int *)a->t_idx, (const float2 *)a->bwd_c, a->t_val, a->bwd_t, a->m);
        LAUNCH_CHECK(a);
        a->t_val_of = nullptr;  // t_val no longer mirrors the GCN edge values
        const int64_t before = t->launches;
        int rc = rowsum_impl(t, a->bwd_t, datt + 1, st, 2);
        if (rc == GNNAGG_OK) rc = gcn_run_core(t, dY, dX, feat, 0, st);
        a->launches += t->launches - before;
        return rc;
    }
    // 4b. pass 2 over the transposed CSR: dX[u] = sum_e alpha_e dY[v] and the source half sum_e ds_e, weights formed on
    //     the fly from (w, t) through t_perm and 1 / D_v ((w, t) of a small graph stays in L2)
    {
        AggParams p{};
        p.X = dY;
        p.Y = dX;
        p.val = reinterpret_cast<const float *>(a->t_perm);
        p.bwd_c = a->bwd_c;
        p.bwd_wt = a->bwd_wt;
        p.rsum = datt + 1;
        p.rsum_stride = 2;
        p.F = feat;
        p.ptr = t->d_ptr;
        p.idx = t->d_idx;
        p.item_row = t->d_item_row;
        p.carry = t->carry;
        p.carry_den = t->carry_den;
        p.den_row = t->den_row;
        p.num_rows = t->n;
        p.num_edges = t->m;
        p.num_fine_items = t->num_items;
        p.bulk_ok = aligned16(p.idx) && aligned16(p.val);
        const int64_t before = t->launches;
        const int rc = launch_agg<kModeGATBWD2, false>(t, p, st);
        a->launches += t->launches - before;
        return rc;
    }
}

int gnnagg_sample_subgraph(gnnagg_aggregator *a, int *d_active, int fanout, int layer_num, uint64_t seed, int **d_vertexset,
                           int **d_sub_ptr, int **d_sub_idx, int *num_v, int *num_e, void *stream)
{
    if (!a || (!d_active && a->n > 0) || !d_vertexset || !d_sub_ptr || !d_sub_idx || !num_v || !num_e || layer_num < 1)
        return set_error(GNNAGG_ERR_ARG, "gnnagg_sample_subgraph: bad argument");
    const int rc = sample_subgraph_device(a->d_ptr, a->d_idx, a->d_item_row, a->num_items, a->n, a->m, d_active, fanout,
                                          layer_num, seed, d_vertexset, d_sub_ptr, d_sub_idx, num_v, num_e, (cudaStream_t)stream);
    if (rc == GNNAGG_OK) a->launches += 5 + 2 * (layer_num - 1);
    return rc;
}

int gnnagg_device_free(void *d_ptr)
{
    CUDA_TRY(cudaFree(d_ptr));
    return GNNAGG_OK;
}

int gnnagg_gather_rows(const float *X, const int64_t *rows, float *out, int64_t count, int feat, void *stream)
{
    if (count == 0) return GNNAGG_OK;
    if (!X || !rows || !out || count < 0) return set_error(GNNAGG_ERR_ARG, "gnnagg_gather_rows: bad argument");
    if (int rc = check_feat(feat)) return rc;
    if (!aligned16(X) || !aligned16(out)) return set_error(GNNAGG_ERR_ARG, "X and out must be 16-byte aligned");
    const int64_t total4 = count * (feat / 4);
    gather_rows_kernel<<<(unsigned)cdiv(total4, 256), 256, 0, (cudaStream_t)stream>>>(X, rows, out, total4, feat / 4);
    CUDA_TRY(cudaPeekAtLastError());
    return GNNAGG_OK;
}

int gnnagg_spmm_naive(int num_v, const int *d_ptr, const int *d_idx, const float *d_val, const float *X, float *Y,
                      int feat, void *stream)
{
    if (!d_ptr || !X || !Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_spmm_naive: NULL argument");
    if (int rc = check_feat(feat)) return rc;
    if (num_v == 0) return GNNAGG_OK;
    spmm_naive_kernel<<<(unsigned)cdiv(num_v, 128), 128, 0, (cudaStream_t)stream>>>(num_v, d_ptr, d_idx, d_val, X, Y, feat);
    CUDA_TRY(cudaPeekAtLastError());
    return GNNAGG_OK;
}

static int count_diff(int *diffnum, cudaStream_t st, int *d_cnt)
{
    CUDA_TRY(cudaPeekAtLastError());
    CUDA_TRY(cudaMemcpyAsync(diffnum, d_cnt, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaFree(d_cnt));
    return GNNAGG_OK;
}

int gnnagg_validate(const float *d_ref, const float *d_ans, int64_t num, int *diffnum, void *stream)
{
    if (!d_ref || !d_ans || !diffnum) return set_error(GNNAGG_ERR_ARG, "gnnagg_validate: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    int *d_cnt = nullptr;
    CUDA_TRY(cudaMalloc((void **)&d_cnt, sizeof(int)));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(int), st));
    if (num > 0) validate_kernel<<<(unsigned)cdiv(num, 128), 128, 0, st>>>(d_ref, d_ans, num, d_cnt);
    return count_diff(diffnum, st, d_cnt);
}

int gnnagg_validate_reordered(const float *d_ref, const float *d_ans, const int *d_map, int num_v, int feat,
                              int *diffnum, void *stream)
{
    if (!d_ref || !d_ans || !diffnum) return set_error(GNNAGG_ERR_ARG, "gnnagg_validate_reordered: NULL argument");
    if (!d_map) return gnnagg_validate(d_ref, d_ans, (int64_t)num_v * feat, diffnum, stream);  // spmm.h:73-74
    cudaStream_t st = (cudaStream_t)stream;
    int *d_cnt = nullptr;
    CUDA_TRY(cudaMalloc((void **)&d_cnt, sizeof(int)));
    CUDA_TRY(cudaMemsetAsync(d_cnt, 0, sizeof(int), st));
    const int64_t num = (int64_t)num_v * feat;
    if (num > 0) validate_reordered_kernel<<<(unsigned)cdiv(num, 128), 128, 0, st>>>(d_ref, d_ans, d_map, num_v, feat, d_cnt);
    return count_diff(diffnum, st, d_cnt);
}

// ------------------------------------------------------------------ host-buffer entry points
constexpr int kHostChunks = 4;
constexpr int kHostSlices = 4;

static int ensure_in_stream(gnnagg_aggregator *a)
{
    if (a->in_stream) return GNNAGG_OK;
    CUDA_TRY(cudaStreamCreateWithFlags(&a->in_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 8; ++i) CUDA_TRY(cudaEventCreateWithFlags(&a->in_done[i], cudaEventDisableTiming));
    CUDA_TRY(cudaEventCreateWithFlags(&a->in_free, cudaEventDisableTiming));
    return GNNAGG_OK;
}

// Host-buffer GCN aggregation / layer.  Three regimes:
//   * scheduled runs and tiny graphs: copy in, run, copy out;
//   * medium graphs: one input copy, then edge-balanced ROW chunks -- chunk c is aggregated (and combined) on `stream`
//     while the finished rows of chunk c-1 travel back on a second stream;
//   * large graphs (>= kSmallGraphEdges edges, or forced): SOURCE slices on top of that.  X arrives in S row blocks on a
//     third stream; slice c (the edges whose source lies in block c) is accumulated into the output as soon as block c
//     is resident, so the aggregation hides behind the input copy; the last two slices run row chunk by row chunk, each
//     chunk followed by its combination and its copy back, so the output copy starts soon after the input copy ends.
static int gcn_host_pipeline(gnnagg_aggregator *a, const float *h_X, const float *h_W, float *h_out, int feat_in,
                             int feat_out, int scheduled, cudaStream_t st)
{
    const bool layer = h_W != nullptr;
    const int fo = layer ? feat_out : feat_in;
    const size_t cin = (size_t)a->n * feat_in, cout = (size_t)a->n * fo;
    if (int rc = ensure(a->st_in, a->st_in_cap, cin)) return rc;
    if (int rc = ensure(a->st_out, a->st_out_cap, cout)) return rc;
    if (layer) {
        if (int rc = ensure(a->st_w, a->st_w_cap, (size_t)feat_in * feat_out)) return rc;
        if (int rc = ensure(a->ax, a->ax_cap, cin)) return rc;
        CUDA_TRY(cudaMemcpyAsync(a->st_w, h_W, (size_t)feat_in * feat_out * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    float *agg_out = layer ? a->ax : a->st_out;
    if (scheduled || a->n < 4096) {  // scheduled order is not row-contiguous; tiny graphs are not worth chunking
        CUDA_TRY(cudaMemcpyAsync(a->st_in, h_X, cin * sizeof(float), cudaMemcpyHostToDevice, st));
        if (int rc = gcn_run_impl(a, a->st_in, agg_out, feat_in, scheduled, st, !layer)) return rc;
        if (layer && a->n > 0) {
            if (int rc = dense_nn_launch(a->ax, a->st_w, a->st_out, a->n, feat_out, feat_in, st)) return rc;
            a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
        }
        CUDA_TRY(cudaMemcpyAsync(h_out, a->st_out, cout * sizeof(float), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        return GNNAGG_OK;
    }
    if (int rc = check_feat(feat_in)) return rc;
    if (!a->d_val && a->m > 0) return set_error(GNNAGG_ERR_STATE, "edge values not set (gnnagg_set_val)");
    if (int rc = ensure_copy_stream(a)) return rc;
    const int S = a->host_slices > 0 ? a->host_slices : (a->host_slices == 0 && a->m >= kSmallGraphEdges ? kHostSlices : 1);
    // the aggregators whose rows are chunked for the copy back: the graph itself, or the trailing slices
    gnnagg_aggregator *tail[2] = {a, nullptr};
    int tail_first = 0, tail_count = 1;
    if (S > 1) {
        if (int rc = ensure_slices(a, S, st)) return rc;
        if (int rc = ensure_in_stream(a)) return rc;
        // input blocks on their own stream, after everything already queued on `st` (a previous call may still read st_in)
        CUDA_TRY(cudaEventRecord(a->in_free, st));
        CUDA_TRY(cudaStreamWaitEvent(a->in_stream, a->in_free, 0));
        for (int c = 0; c < S; ++c) {
            const int64_t r0 = std::min<int64_t>((int64_t)c * a->slice_width, a->n), r1 = std::min<int64_t>(r0 + a->slice_width, a->n);
            if (r1 > r0)
                CUDA_TRY(cudaMemcpyAsync(a->st_in + (size_t)r0 * feat_in, h_X + (size_t)r0 * feat_in,
                                         (size_t)(r1 - r0) * feat_in * sizeof(float), cudaMemcpyHostToDevice, a->in_stream));
            CUDA_TRY(cudaEventRecord(a->in_done[c], a->in_stream));
        }
        // The aggregation is longer than the input copy, so when the last block lands part of the second-to-last slice
        // is still to do: the last TWO slices run row chunk by row chunk (both slices of a chunk, its combination, its
        // copy back), the slices before them over all rows as their block arrives.
        tail_count = 2;
        tail_first = S - tail_count;
        for (int c = 0; c < tail_first; ++c) {
            CUDA_TRY(cudaStreamWaitEvent(st, a->in_done[c], 0));
            gnnagg_aggregator *s = a->slice[c];
            const int64_t before = s->launches;
            if (int rc = gcn_run_core(s, a->st_in, agg_out, feat_in, 0, st, c > 0)) return rc;
            a->launches += s->launches - before;
        }
        tail[0] = a->slice[tail_first];
        tail[1] = a->slice[tail_first + 1];
    } else {
        CUDA_TRY(cudaMemcpyAsync(a->st_in, h_X, cin * sizeof(float), cudaMemcpyHostToDevice, st));
        if (int rc = merged_view(a, st, &tail[0])) return rc;  // the rows gcn_run aggregates, chunk by chunk
    }
    const int *hp[2] = {nullptr, nullptr};
    for (int t = 0; t < tail_count; ++t)
        if (int rc = host_ptr(tail[t], &hp[t])) return rc;
    int bounds[kHostChunks + 1];
    if (S > 1) {  // equal ROW counts: the chunks are sized for the copy back
        for (int c = 0; c <= kHostChunks; ++c) bounds[c] = (int)((int64_t)a->n * c / kHostChunks);
    } else {
        row_chunks(hp[0], a->n, tail[0]->m, kHostChunks, bounds);
    }
    for (int c = 0; c < kHostChunks; ++c) {
        const int r0 = bounds[c], r1 = bounds[c + 1];
        if (r1 <= r0) continue;
        for (int t = 0; t < tail_count; ++t) {
            if (S > 1 && c == 0) CUDA_TRY(cudaStreamWaitEvent(st, a->in_done[tail_first + t], 0));
            const int64_t before = tail[t]->launches;
            if (int rc = gcn_run_core(tail[t], a->st_in, agg_out, feat_in, 0, st, S > 1 && (tail_first + t) > 0, r0, r1,
                                      hp[t][r0], hp[t][r1]))
                return rc;
            if (tail[t] != a) a->launches += tail[t]->launches - before;
        }
        if (layer) {
            if (int rc = dense_nn_launch(a->ax + (size_t)r0 * feat_in, a->st_w, a->st_out + (size_t)r0 * fo, r1 - r0, feat_out,
                                         feat_in, st))
                return rc;
            a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
        }
        CUDA_TRY(cudaEventRecord(a->chunk_done[c], st));
        CUDA_TRY(cudaStreamWaitEvent(a->copy_stream, a->chunk_done[c], 0));
        CUDA_TRY(cudaMemcpyAsync(h_out + (size_t)r0 * fo, a->st_out + (size_t)r0 * fo, (size_t)(r1 - r0) * fo * sizeof(float),
                                 cudaMemcpyDeviceToHost, a->copy_stream));
    }
    CUDA_TRY(cudaEventRecord(a->copies_done, a->copy_stream));
    CUDA_TRY(cudaStreamWaitEvent(st, a->copies_done, 0));  // the caller's stream is ordered after the copies as well
    CUDA_TRY(cudaStreamSynchronize(st));
    return GNNAGG_OK;
}

int gnnagg_set_host_pipeline(gnnagg_aggregator *a, int slices)
{
    if (!a || slices > 8) return set_error(GNNAGG_ERR_ARG, "gnnagg_set_host_pipeline: at most 8 source slices");
    a->host_slices = slices;
    return GNNAGG_OK;
}

int gnnagg_gcn_run_host(gnnagg_aggregator *a, const float *h_X, float *h_Y, int feat, int scheduled, void *stream)
{
    if (!a || !h_X || !h_Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run_host: NULL argument");
    return gcn_host_pipeline(a, h_X, nullptr, h_Y, feat, feat, scheduled, (cudaStream_t)stream);
}

int gnnagg_gcn_layer_host(gnnagg_aggregator *a, const float *h_X, const float *h_W, float *h_H, int feat_in,
                          int feat_out, int scheduled, void *stream)
{
    if (!a || !h_X || !h_W || !h_H) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_layer_host: NULL argument");
    return gcn_host_pipeline(a, h_X, h_W, h_H, feat_in, feat_out, scheduled, (cudaStream_t)stream);
}

int gnnagg_gat_run_host(gnnagg_aggregator *a, const float *h_X, const float *h_att, float *h_Y, int feat,
                        float slope, int scheduled, void *stream)
{
    if (!a || !h_X || !h_att || !h_Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_gat_run_host: NULL argument");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t cnt = (size_t)a->n * feat;
    if (int rc = ensure(a->st_in, a->st_in_cap, cnt)) return rc;
    if (int rc = ensure(a->st_out, a->st_out_cap, cnt)) return rc;
    if (int rc = ensure(a->st_att, a->st_att_cap, (size_t)a->n * 2)) return rc;
    CUDA_TRY(cudaMemcpyAsync(a->st_in, h_X, cnt * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(a->st_att, h_att, (size_t)a->n * 2 * sizeof(float), cudaMemcpyHostToDevice, st));
    if (int rc = gat_run_impl(a, a->st_in, a->st_att, a->st_out, feat, slope, scheduled, st)) return rc;
    CUDA_TRY(cudaMemcpyAsync(h_Y, a->st_out, cnt * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return GNNAGG_OK;
}
}
