// capi.cu -- the C ABI of libgnnagg.so (include/gnnagg.h): aggregator object, launch logic.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <string>
#include <utility>
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

// an owned device array, freed with its owner
template <class T>
struct DevBuf {
    T *p = nullptr;
    size_t cap = 0;

    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf(DevBuf &&o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr, o.cap = 0; }
    DevBuf &operator=(DevBuf o) noexcept
    {
        std::swap(p, o.p), std::swap(cap, o.cap);
        return *this;
    }
    ~DevBuf()
    {
        if (p) cudaFree(p);
    }

    // at least `need` elements; grows only, and does not keep the contents
    int ensure(size_t need)
    {
        if (need <= cap && p) return GNNAGG_OK;
        if (p) CUDA_TRY(cudaFree(p));
        p = nullptr;
        cap = 0;
        CUDA_TRY(cudaMalloc((void **)&p, (need ? need : 1) * sizeof(T)));
        cap = need;
        return GNNAGG_OK;
    }
    // takes over an array cudaMalloc'ed elsewhere (the *_build_device functions)
    void adopt(T *q) { *this = DevBuf(), p = q; }
};

// events created together and destroyed with their owner
template <int N>
struct Events {
    cudaEvent_t e[N] = {};

    Events() = default;
    Events(const Events &) = delete;
    ~Events()
    {
        for (cudaEvent_t x : e)
            if (x) cudaEventDestroy(x);
    }
    cudaEvent_t operator[](int i) const { return e[i]; }
    bool created() const { return e[0] != nullptr; }
    int create(unsigned flags)
    {
        for (cudaEvent_t &x : e) CUDA_TRY(cudaEventCreateWithFlags(&x, flags));
        return GNNAGG_OK;
    }
};

// a second stream that overlaps copies with the work on the caller's stream, created on first use: ev[0..7] per chunk
// or slice, ev[8] once per call
struct SideStream {
    cudaStream_t stream = nullptr;
    Events<9> ev;

    SideStream() = default;
    SideStream(const SideStream &) = delete;
    ~SideStream()
    {
        if (stream) cudaStreamDestroy(stream);
    }
    int ensure()
    {
        if (stream) return GNNAGG_OK;
        CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        return ev.create(cudaEventDisableTiming);
    }
};

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

// rows spanning more than kFixChunk carry items, per item size (second fix-up pass; built on first use)
struct LongRows {
    int item_edges = 0, count = 0;
    DevBuf<int> list;
    DevBuf<int2> records;  // per item: what the first fix-up pass does there (fixup_records_kernel)
};

// What one traversal runs on: a CSR, its item table, the scratch sized for them, and the aggregator whose launch
// counter and timing events it reports to.  The aggregator is the view of the user's CSR; the graphs it derives from
// it (source slices, transposed CSR, merged view) own their arrays and hold a view of them.
struct View {
    gnnagg_aggregator *root = nullptr;
    const int *d_ptr = nullptr, *d_idx = nullptr;
    const float *d_val = nullptr;
    int n = 0, m = 0;
    const int *d_item_row = nullptr;
    int num_items = 0;   // ceil(m / kFineItem)
    int warp_edges = 0;  // 0 = automatic
    bool records = false;          // its aggregation kernel is bracketed by the root's ev[1] / ev[2]
    const int *out_row = nullptr;  // a slice compacted to its non-empty rows: row r of it is output row out_row[r]
    DevBuf<float> carry, carry_den, den_row;
    std::vector<LongRows> long_rows;
    const int *h_ptr_user = nullptr;
    std::vector<int> h_ptr;  // lazily mirrored (aggregator.h:30-39)
};

// The CSR split by source-id ranges into sub-CSRs over the same rows (source_slices_build_device).  Edge values are
// mirrored into slice order.
struct Slices {
    struct Slice {
        DevBuf<int> item_row, c_ptr, out_row;  // c_ptr / out_row: compacted slices only
        View v;
    };
    DevBuf<int> ptr, idx, perm;
    DevBuf<float> val;
    uint64_t val_gen = 0;  // the root's edge-value generation `val` mirrors (0: none)
    int off[kMaxSlices] = {0}, cnt[kMaxSlices] = {0};
    int width = 0;
    std::vector<Slice> slice;
};

// the transposed CSR of the backward passes (gnnagg_transpose_build)
struct Transpose {
    DevBuf<int> ptr, idx, perm, item_row;
    DevBuf<float> val;     // edge values in transposed order, or the GAT backward's alpha
    uint64_t val_gen = 0;  // the root's edge-value generation `val` mirrors (0: none)
    View v;
};

// the merged view of duplicate edges (gnnagg_set_merge_duplicates): runs of adjacent equal sources in a row as one
// entry each
struct Merged {
    DevBuf<int> ptr, idx, start, item_row;  // start[k]: CSR edge id of run k's first edge
    DevBuf<float> val;                      // run sums of the edge values
    uint64_t val_gen = 0;                   // the root's edge-value generation `val` sums (0: none)
    View v;
};

// a schedule (sched_device.cu).  Neighbour grouping keeps the CSR edge order: idx and val are the CSR's, and only the
// locality kinds fill own_idx / own_val.
struct Schedule {
    int kind = GNNAGG_SCHED_NOP;
    int num_target = 0, edges = 0, items = 0;
    DevBuf<int> ptr, target, perm, item_row, own_idx;
    DevBuf<float> own_val;
    const int *idx = nullptr;
    const float *val = nullptr;
};

struct gnnagg_aggregator : View {
    int64_t launches = 0;
    uint64_t val_gen = 0;  // counts gnnagg_set_val_on calls: the derived value arrays compare theirs with it
    DevBuf<int> item_row;
    // scratch
    DevBuf<float> newval, ax;
    // host-buffer entry points: device staging
    DevBuf<float> st_in, st_out, st_w, st_att;
    Schedule sched;
    // backward pass (gnnagg_transpose_build)
    std::unique_ptr<Transpose> tr;
    // GAT backward scratch: per row (1 / D_v, c_v); per edge (w_e, t_e); pass-1 row sums per row / per entered item
    DevBuf<float2> bwd_c, bwd_wt, bwd_part, bwd_carry;
    DevBuf<float> bwd_t;  // large graphs: ds_e in transposed edge order (alpha_e goes to tr->val)
    // host-buffer entry points: the result is copied back per row chunk on `copy` while the next chunk computes; on
    // large graphs the CSR is split by source-id ranges so that slice c can be aggregated while the rows of X that
    // slice c+1 gathers are still on their way from the host on `in`
    SideStream copy, in;
    int host_slices = 0;  // 0 = automatic, > 0 forced slice count, < 0 row-chunk pipeline only (gnnagg_set_host_pipeline)
    std::unique_ptr<Slices> host;
    // locality slices of the device-resident path (gnnagg_set_locality_slices): when X is many times the L2, the
    // un-scheduled aggregation runs source slice by source slice (sub-CSRs in accumulate mode, deterministic) so that
    // the rows a slice gathers stay cache resident -- locality_schedule (graph_schedule.h:17-89) without its atomics
    int loc_slices = 0;  // 0 = automatic, 1 = off, 2..kMaxSlices forced
    std::unique_ptr<Slices> loc;
    // merged view, built on first use
    int merge_mode = 0;   // 0 = automatic, 1 = off, 2 = on
    int merge_auto = -1;  // automatic decision: -1 not taken yet, 0 off, 1 on
    std::unique_ptr<Merged> mg;
    // optional per-kernel timing (gnnagg_profile_enable)
    bool prof = false;
    Events<5> ev;  // begin, agg0, agg1, agg_end, end
};

#define PROF_RECORD(a, i, st)                                   \
    do {                                                        \
        if ((a)->prof) CUDA_TRY(cudaEventRecord((a)->ev[i], st)); \
    } while (0)

namespace gnnagg {

static EdgeParams edge_params(const View &v)
{
    EdgeParams g;
    g.ptr = v.d_ptr;
    g.idx = v.d_idx;
    g.item_row = v.d_item_row;
    g.num_rows = v.n;
    g.num_edges = v.m;
    g.num_items = v.num_items;
    return g;
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

// the item table of a CSR into `buf`; its launch is counted by the caller
static int item_table(DevBuf<int> &buf, const int *d_ptr, int rows, int edges, int *items, cudaStream_t st)
{
    int *out = nullptr;
    const int rc = build_item_rows_device(d_ptr, rows, edges, &out, items, st);
    buf.adopt(out);  // also when the launch failed
    return rc;
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

// lanes that cover one feature row with a float4 each: F/4 rounded up to 8, 16 or 32.  Also the lanes per virtual
// warp of the aggregation kernels (agg_kernel<LPR, NV>).  Virtual warps HALF as wide with two float4 per lane for rows
// of 33..128 floats -- one broadcast load of the staged idx / val then serves twice as many items, and those loads take
// 18 % of the L1 data pipe on the reddit shape -- were measured and lost: aggregation 2.27 -> 2.43 ms on reddit F=128,
// 0.496 -> 0.537 ms on proteins F=64.
static inline int lanes_for(int F) { return F <= 32 ? 8 : (F <= 64 ? 16 : 32); }

// graphs below this many edges use the 128-edge-per-warp variant: with 512 there would be fewer than
// ~2 waves of CTAs on 148 SMs and the kernel would be bound by the length of one warp's walk
constexpr int64_t kSmallGraphEdges = 4000000;

static inline int warp_edges_for(const View &v, int64_t num_edges)
{
    if (v.warp_edges) return v.warp_edges;
    return num_edges < kSmallGraphEdges ? 128 : kWarpEdges;
}
static inline int item_edges_for(const View &v, int F, int64_t num_edges)
{
    return warp_edges_for(v, num_edges) / (32 / lanes_for(F));
}

using AggKernel = void (*)(const AggParams);

// the aggregation kernel for a mode, edges per warp, feature width and element type of X
template <int MODE, bool SCHED, bool XBF16 = false>
static AggKernel agg_kernel_for(int WE, int F)
{
    if (WE == 128)
        return F <= 32 ? agg_kernel<8, 1, MODE, SCHED, 128, XBF16>
             : F <= 64 ? agg_kernel<16, 1, MODE, SCHED, 128, XBF16>
             : F <= 128 ? agg_kernel<32, 1, MODE, SCHED, 128, XBF16>
                        : agg_kernel<32, 2, MODE, SCHED, 128, XBF16>;
    return F <= 32 ? agg_kernel<8, 1, MODE, SCHED, kWarpEdges, XBF16>
         : F <= 64 ? agg_kernel<16, 1, MODE, SCHED, kWarpEdges, XBF16>
         : F <= 128 ? agg_kernel<32, 1, MODE, SCHED, kWarpEdges, XBF16>
                    : agg_kernel<32, 2, MODE, SCHED, kWarpEdges, XBF16>;
}
template <int MODE, bool SCHED>
static AggKernel agg_kernel_for(int WE, int F, bool xbf16)
{
    if constexpr (MODE == kModeGCN)
        if (xbf16) return agg_kernel_for<MODE, SCHED, true>(WE, F);
    return agg_kernel_for<MODE, SCHED>(WE, F);
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

// rows of v's CSR with more than kFixChunk carry items of EB edges, found once per item size (one host synchronisation)
static const LongRows *long_rows_of(View &v, const AggParams &p, int EB, cudaStream_t st)
{
    for (const LongRows &e : v.long_rows)
        if (e.item_edges == EB) return &e;
    LongRows e;
    e.item_edges = EB;
    const int64_t items = cdiv(v.m, EB);
    if (e.list.ensure((size_t)v.m / ((size_t)kFixChunk * EB) + 2)) return nullptr;
    int *counter = nullptr;
    if (cudaMalloc((void **)&counter, sizeof(int)) != cudaSuccess || e.records.ensure((size_t)items + 1)) {
        cudaFree(counter);
        set_error(GNNAGG_ERR_CUDA, "out of device memory");
        return nullptr;
    }
    cudaMemsetAsync(counter, 0, sizeof(int), st);
    long_rows_kernel<<<(unsigned)cdiv(v.n, 256), 256, 0, st>>>(v.d_ptr, v.n, EB, e.list.p, counter);
    fixup_records_kernel<<<(unsigned)cdiv(items, 256), 256, 0, st>>>(p, EB, items, e.records.p);
    cudaError_t err = cudaMemcpyAsync(&e.count, counter, sizeof(int), cudaMemcpyDeviceToHost, st);
    if (err == cudaSuccess) err = cudaStreamSynchronize(st);
    cudaFree(counter);
    if (err != cudaSuccess) {
        set_error(GNNAGG_ERR_CUDA, cudaGetErrorString(err));
        return nullptr;
    }
    v.root->launches += 2;
    v.long_rows.push_back(std::move(e));
    return &v.long_rows.back();
}

// xbf16: p.X holds bf16 (GCN only)
template <int MODE, bool SCHED>
static int launch_agg(View &v, AggParams p, cudaStream_t st, bool xbf16 = false)
{
    if (p.row_hi == 0 && p.edge_hi == 0) {  // callers that do not set a row range get the whole graph
        p.row_lo = 0, p.row_hi = p.num_rows, p.edge_lo = 0, p.edge_hi = p.num_edges;
    }
    if (p.edge_hi <= p.edge_lo) return GNNAGG_OK;
    gnnagg_aggregator *a = v.root;
    if (v.records) PROF_RECORD(a, 1, st);
    const int WE = warp_edges_for(v, p.num_edges);
    const int64_t first = (int64_t)(p.edge_lo / WE) * WE;  // warps keep their global 512-edge alignment (TMA staging)
    const unsigned grid = (unsigned)cdiv(p.edge_hi - first, (int64_t)WE * kCtaWarps);
    const AggKernel kernel = agg_kernel_for<MODE, SCHED>(WE, p.F, xbf16);
    if (MODE == kModeGATBWD || MODE == kModeGATBWD2)
        launch_dep(kernel, grid, kCtaThreads, st, p);
    else
        kernel<<<grid, kCtaThreads, 0, st>>>(p);
    LAUNCH_CHECK(a);
    if (v.records) PROF_RECORD(a, 2, st);
    if (!SCHED && !mode_emits_edges(MODE)) {
        const int EB = item_edges_for(v, p.F, p.num_edges);
        const int64_t items = cdiv(p.num_edges, EB);
        const int64_t range_items = cdiv(p.edge_hi, EB) - p.edge_lo / EB;  // items touched by the launched range
        if (range_items > 1) {
            const LongRows *lr = long_rows_of(v, p, EB, st);
            if (!lr) return GNNAGG_ERR_CUDA;
            const int lanes = lanes_for(p.F);
            launch_dep(agg_fixup_kernel<MODE>, (unsigned)cdiv(range_items * lanes, 256), 256, st, p, EB, items,
                       (const int2 *)lr->records.p, lanes);
            LAUNCH_CHECK(a);
            if (lr->count > 0) {
                launch_dep(agg_fixup_long_kernel<MODE>, (unsigned)cdiv(lr->count, 8), 256, st, p, EB, (const int *)lr->list.p,
                           lr->count);
                LAUNCH_CHECK(a);
            }
        }
    }
    return GNNAGG_OK;
}

static int aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// the gathered operand of a GCN aggregation: fp32 X (16-byte aligned), or bf16 bit patterns (8-byte aligned) that the
// kernel widens exactly to fp32
struct GatherX {
    const void *p;
    bool bf16;
    GatherX(const float *x) : p(x), bf16(false) {}
    GatherX(const uint16_t *x) : p(x), bf16(true) {}
    int elem_bytes() const { return bf16 ? 2 : 4; }
};

static int check_xy(const GatherX &X, const float *Y)
{
    if (X.bf16) {
        if ((reinterpret_cast<uintptr_t>(X.p) & 7) || !aligned16(Y))
            return set_error(GNNAGG_ERR_ARG, "X (bf16) must be 8-byte aligned and Y 16-byte aligned");
    } else if (!aligned16(X.p) || !aligned16(Y)) {
        return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
    }
    return GNNAGG_OK;
}

// the traversal fields of AggParams: a view's CSR, or the root's schedule
static void set_view(AggParams &p, const View &v)
{
    p.ptr = v.d_ptr;
    p.idx = v.d_idx;
    p.item_row = v.d_item_row;
    p.num_rows = v.n;
    p.num_edges = v.m;
    p.num_fine_items = v.num_items;
}
static void set_sched(AggParams &p, const gnnagg_aggregator *a)
{
    p.ptr = a->sched.ptr.p;
    p.idx = a->sched.idx;
    p.target = a->sched.target.p;
    p.item_row = a->sched.item_row.p;
    p.num_rows = a->sched.num_target;
    p.num_edges = a->sched.edges;
    p.num_fine_items = a->sched.items;
}

// scheduled GCN, GAT and MLP runs: Y zeroed (rows no target reaches stay 0), then the schedule's traversal fields;
// nothing is left to launch when p.num_edges == 0
static int sched_prologue(gnnagg_aggregator *a, float *Y, int F, cudaStream_t st, AggParams &p)
{
    if (a->sched.kind == GNNAGG_SCHED_NOP) return set_error(GNNAGG_ERR_STATE, "scheduled run before schedule");
    CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));  // aggr_gcn.h:393, aggr_nn.h:314
    set_sched(p, a);
    return GNNAGG_OK;
}

// rows [row_lo, row_hi) of the un-scheduled aggregation over v (row_hi < 0: all rows); Y is indexed by GLOBAL row.
// Scheduled runs use v.root's schedule.
static int gcn_run_core(View &v, GatherX X, float *Y, int F, int scheduled, cudaStream_t st, int accumulate = 0,
                        int row_lo = 0, int row_hi = -1, int edge_lo = 0, int edge_hi = 0)
{
    if (v.n == 0) return GNNAGG_OK;  // an empty row block (possible after edge-balanced partitioning)
    if (!X.p || !Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run: NULL argument");
    if (int rc = check_feat(F)) return rc;
    if (int rc = check_xy(X, Y)) return rc;
    if (!v.d_val && v.m > 0) return set_error(GNNAGG_ERR_STATE, "gnnagg_gcn_run: edge values not set (gnnagg_set_val)");
    AggParams p{};
    p.X = X.p;
    p.Y = Y;
    p.F = F;
    if (scheduled) {
        if (int rc = sched_prologue(v.root, Y, F, st, p)) return rc;
        if (p.num_edges == 0) return GNNAGG_OK;
        p.val = v.root->sched.val;
        p.bulk_ok = aligned16(p.idx) && aligned16(p.val);
        return launch_agg<kModeGCN, true>(v, p, st, X.bf16);
    }
    if (v.m == 0) {
        if (!accumulate) CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)v.n * F * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(v, F, v.m);
    if (int rc = v.carry.ensure((size_t)cdiv(v.m, EB) * F)) return rc;
    set_view(p, v);
    p.accumulate = accumulate;
    p.out_row = v.out_row;
    p.val = v.d_val;
    p.carry = v.carry.p;
    p.bulk_ok = aligned16(p.idx) && aligned16(p.val);
    if (row_hi >= 0) {
        p.row_lo = row_lo, p.row_hi = row_hi, p.edge_lo = edge_lo, p.edge_hi = edge_hi;
        if (row_hi <= row_lo) return GNNAGG_OK;
        if (edge_hi <= edge_lo) {  // a chunk of empty rows
            if (!accumulate) CUDA_TRY(cudaMemsetAsync(Y + (size_t)row_lo * F, 0, (size_t)(row_hi - row_lo) * F * sizeof(float), st));
            return GNNAGG_OK;
        }
    }
    return launch_agg<kModeGCN, false>(v, p, st, X.bf16);
}

// host mirror of the row pointers (needed to cut row chunks)
static int host_ptr(View &v, const int **out)
{
    if (v.h_ptr_user) {
        *out = v.h_ptr_user;
        return GNNAGG_OK;
    }
    if (v.h_ptr.empty()) {
        v.h_ptr.resize((size_t)v.n + 1);
        CUDA_TRY(cudaMemcpy(v.h_ptr.data(), v.d_ptr, v.h_ptr.size() * sizeof(int), cudaMemcpyDeviceToHost));
    }
    *out = v.h_ptr.data();
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

static int gat_run_core(gnnagg_aggregator *a, const float *X, const float *att, float *Y, int F, float slope,
                        int scheduled, cudaStream_t st)
{
    if (a && a->n == 0) return GNNAGG_OK;
    if (!a || !X || !Y || !att) return set_error(GNNAGG_ERR_ARG, "gnnagg_gat_run: NULL argument");
    if (int rc = check_feat(F)) return rc;
    if (!aligned16(X) || !aligned16(Y)) return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
    if (int rc = a->den_row.ensure((size_t)a->n)) return rc;
    AggParams p{};
    p.X = X;
    p.Y = Y;
    p.att = att;
    p.F = F;
    p.slope = slope;
    p.den_row = a->den_row.p;
    if (scheduled) {
        if (int rc = sched_prologue(a, Y, F, st, p)) return rc;
        if (p.num_edges == 0) return GNNAGG_OK;
        CUDA_TRY(cudaMemsetAsync(a->den_row.p, 0, (size_t)a->n * sizeof(float), st));
        if (int rc = a->newval.ensure((size_t)a->sched.edges)) return rc;
        p.newval = a->newval.p;
        p.bulk_ok = aligned16(p.idx);
        if (int rc = launch_agg<kModeGAT, true>(*a, p, st)) return rc;
        const int64_t total4 = (int64_t)a->n * F / 4;
        gat_scale_kernel<<<(unsigned)cdiv(total4, 256), 256, 0, st>>>(Y, a->den_row.p, F, total4);
        LAUNCH_CHECK(a);
        return GNNAGG_OK;
    }
    if (a->m == 0) {
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(*a, F, a->m);
    if (int rc = a->carry.ensure((size_t)cdiv(a->m, EB) * F)) return rc;
    if (int rc = a->carry_den.ensure((size_t)cdiv(a->m, EB))) return rc;
    set_view(p, *a);
    p.carry = a->carry.p;
    p.carry_den = a->carry_den.p;
    p.bulk_ok = aligned16(p.idx);
    return launch_agg<kModeGAT, false>(*a, p, st);
}

static int mlp_run_core(gnnagg_aggregator *a, const float *P, float *Y, int F, int scheduled, cudaStream_t st)
{
    AggParams p{};
    p.X = P;
    p.P = P;
    p.Y = Y;
    p.F = F;
    if (scheduled) {
        if (int rc = sched_prologue(a, Y, F, st, p)) return rc;
        if (p.num_edges == 0) return GNNAGG_OK;
        p.bulk_ok = aligned16(p.idx);
        return launch_agg<kModeMLP, true>(*a, p, st);
    }
    if (a->m == 0) {
        CUDA_TRY(cudaMemsetAsync(Y, 0, (size_t)a->n * F * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(*a, F, a->m);
    if (int rc = a->carry.ensure((size_t)cdiv(a->m, EB) * F)) return rc;
    set_view(p, *a);
    p.carry = a->carry.p;
    p.bulk_ok = aligned16(p.idx);
    return launch_agg<kModeMLP, false>(*a, p, st);
}

// builds the source slices of `a` on first use and (re)mirrors the edge values into slice order
static int ensure_slices(gnnagg_aggregator *a, std::unique_ptr<Slices> &set, int want, cudaStream_t st, bool compact = false)
{
    if (!set || (int)set->slice.size() != want) {
        set.reset();
        auto s = std::make_unique<Slices>();
        const int width = (int)cdiv(a->n, want);
        int *sp = nullptr, *si = nullptr, *sq = nullptr;
        if (int rc = source_slices_build_device(a->d_ptr, a->d_idx, a->d_item_row, a->num_items, a->n, a->m, want, width,
                                                &sp, &si, &sq, s->off, s->cnt, st))
            return rc;
        s->ptr.adopt(sp), s->idx.adopt(si), s->perm.adopt(sq);
        if (s->val.ensure((size_t)a->m + 4 * (size_t)want))
            return set_error(GNNAGG_ERR_CUDA, "host pipeline: out of device memory for the source slices");
        s->slice.resize(want);
        for (int c = 0; c < want; ++c) {
            Slices::Slice &sl = s->slice[c];
            View &v = sl.v;
            v.root = a;
            v.d_ptr = s->ptr.p + (size_t)c * ((size_t)a->n + 1);
            v.d_idx = s->idx.p + s->off[c];
            v.d_val = s->val.p + s->off[c];
            v.n = a->n;
            v.m = s->cnt[c];
            v.warp_edges = a->warp_edges ? a->warp_edges : (a->m < kSmallGraphEdges ? 128 : kWarpEdges);  // as the whole graph
            if (compact && c > 0) {
                // slices behind the first only ADD to rows that have edges in them: keep those rows only (slice 0 stays
                // complete: it is the pass that writes every row, zeros included)
                int *cp = nullptr, *rows = nullptr;
                const int rc = compact_rows_device(v.d_ptr, a->n, &cp, &rows, &v.n, st);
                if (rc) return rc;
                sl.c_ptr.adopt(cp), sl.out_row.adopt(rows);
                v.d_ptr = cp;
                v.out_row = rows;
            }
            if (int rc = item_table(sl.item_row, v.d_ptr, v.n, v.m, &v.num_items, st)) return rc;
            v.d_item_row = sl.item_row.p;
        }
        s->width = width;
        set = std::move(s);
        a->launches += 6 + 3 * want;
    }
    if (set->val_gen != a->val_gen) {
        for (int c = 0; c < want; ++c) {
            if (set->cnt[c] == 0) continue;
            gather_val_kernel<<<(unsigned)cdiv(set->cnt[c], 256), 256, 0, st>>>(a->d_val, set->perm.p + set->off[c],
                                                                                set->val.p + set->off[c], set->cnt[c]);
            LAUNCH_CHECK(a);
        }
        set->val_gen = a->val_gen;
    }
    return GNNAGG_OK;
}


// how many source slices the device-resident un-scheduled aggregation uses for this feature width (1 = none)
// x_elem_bytes: bytes per element of X as stored (4 fp32, 2 bf16); the constants were tuned on fp32 runs only
static int locality_slices_for(const gnnagg_aggregator *a, int F, int x_elem_bytes)
{
    if (a->loc_slices >= 1) return a->loc_slices < kMaxSlices ? a->loc_slices : kMaxSlices;
    // automatic: worth it when X is many times the L2 (the gathers of a slice then stay resident where those of the
    // whole graph do not) and rows are long enough that the extra passes over Y stay small next to the gathers
    int dev = 0, l2 = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev) != cudaSuccess || l2 <= 0)
        return 1;
    const double x_bytes = (double)x_elem_bytes * (double)a->n * F;
    if (x_bytes < kLocalityMinL2Multiples * (double)l2 || a->m < kSmallGraphEdges) return 1;
    if ((double)a->m < kLocalityMinDegree * (double)a->n) return 1;
    int S = (int)(x_bytes / (kLocalitySliceL2Multiples * (double)l2) + 0.999);
    return S < 2 ? 1 : (S > kLocalityMaxAuto ? kLocalityMaxAuto : S);
}

// Y (+)= A X slice by slice over the source ranges; same result as the un-sliced run up to fp32 summation order
static int gcn_run_sliced(gnnagg_aggregator *a, GatherX X, float *Y, int F, int S, cudaStream_t st, int accumulate)
{
    if (int rc = ensure_slices(a, a->loc, S, st, true)) return rc;
    PROF_RECORD(a, 1, st);
    for (int c = 0; c < S; ++c)
        if (int rc = gcn_run_core(a->loc->slice[c].v, X, Y, F, 0, st, accumulate || c > 0)) return rc;
    PROF_RECORD(a, 2, st);
    return GNNAGG_OK;
}

// ev[1] / ev[2] back to back ahead of the aggregation, so that a call that launches no aggregation kernel still reads
// as 0 ms
static int prof_agg_empty(gnnagg_aggregator *a, cudaStream_t st)
{
    if (a->prof) {
        CUDA_TRY(cudaEventRecord(a->ev[1], st));
        CUDA_TRY(cudaEventRecord(a->ev[2], st));
    }
    return GNNAGG_OK;
}

static int merged_view(gnnagg_aggregator *a, cudaStream_t st, View **out);

// timing brackets: ev[0] call entry, ev[3] end of the aggregation part, ev[4] end of the call
static int gcn_run_impl(gnnagg_aggregator *a, GatherX X, float *Y, int F, int scheduled, cudaStream_t st,
                        bool last = true, int accumulate = 0)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run: NULL argument");
    PROF_RECORD(a, 0, st);
    if (int rc = prof_agg_empty(a, st)) return rc;
    int S = 1;
    if (!scheduled && a->n > 0 && a->m > 0 && X.p && Y && check_feat(F) == GNNAGG_OK && a->d_val)
        S = locality_slices_for(a, F, X.elem_bytes());
    if (S > 1) {
        if (int rc = check_xy(X, Y)) return rc;
        if (int rc = gcn_run_sliced(a, X, Y, F, S, st, accumulate)) return rc;
    } else {
        View *t = a;
        if (!scheduled)
            if (int rc = merged_view(a, st, &t)) return rc;
        if (int rc = gcn_run_core(*t, X, Y, F, scheduled, st, accumulate)) return rc;
    }
    PROF_RECORD(a, 3, st);
    if (last) PROF_RECORD(a, 4, st);
    return GNNAGG_OK;
}

static int gat_run_impl(gnnagg_aggregator *a, const float *X, const float *att, float *Y, int F, float slope,
                        int scheduled, cudaStream_t st)
{
    if (a) {
        PROF_RECORD(a, 0, st);
        if (int rc = prof_agg_empty(a, st)) return rc;
    }
    if (int rc = gat_run_core(a, X, att, Y, F, slope, scheduled, st)) return rc;
    PROF_RECORD(a, 3, st);
    PROF_RECORD(a, 4, st);
    return GNNAGG_OK;
}

// out[v * ostride] = sum over row v of in[e], rows and edges as those of view v; deterministic
template <int SRC = kSumArray>
static int rowsum_impl(View &v, const float *in, float *out, cudaStream_t st, int ostride = 1, float slope = 0.f)
{
    if (v.m == 0) {
        if (ostride == 1)
            CUDA_TRY(cudaMemsetAsync(out, 0, (size_t)v.n * sizeof(float), st));
        else if (v.n > 0)
            CUDA_TRY(cudaMemset2DAsync(out, (size_t)ostride * sizeof(float), 0, sizeof(float), (size_t)v.n, st));
        return GNNAGG_OK;
    }
    const int64_t items = cdiv(v.m, kRowsumItem);
    if (int rc = v.carry_den.ensure((size_t)items)) return rc;
    const EdgeParams g = edge_params(v);
    const unsigned grid = (unsigned)cdiv(items, 256);
    rowsum_kernel<SRC><<<grid, 256, 0, st>>>(g, in, slope, out, v.carry_den.p, ostride);
    LAUNCH_CHECK(v.root);
    if (items > 1) {
        rowsum_fixup_kernel<1><<<grid, 256, 0, st>>>(g, out, v.carry_den.p, ostride);
        LAUNCH_CHECK(v.root);
        if (items > kRowsumChunk + 1) {
            rowsum_fixup_kernel<2><<<grid, 256, 0, st>>>(g, out, v.carry_den.p, ostride);
            LAUNCH_CHECK(v.root);
        }
    }
    return GNNAGG_OK;
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
        auto g = std::make_unique<Merged>();
        int *mp = nullptr, *mi = nullptr, *ms = nullptr;
        View &v = g->v;
        if (int rc = merge_build_device(a->d_ptr, a->d_idx, a->n, a->m, &mp, &mi, &ms, &v.m, st)) return rc;
        g->ptr.adopt(mp), g->idx.adopt(mi), g->start.adopt(ms);
        a->launches += 5;  // run heads, row heads, scan (counted once), compaction, row pointers
        if (g->val.ensure((size_t)v.m)) return set_error(GNNAGG_ERR_CUDA, "merged view: out of device memory");
        v.root = a;
        v.d_ptr = mp;
        v.d_idx = mi;
        v.d_val = g->val.p;
        v.n = a->n;
        v.records = true;  // the aggregation kernel's events are the root's (gnnagg_profile_read)
        if (int rc = item_table(g->item_row, mp, v.n, v.m, &v.num_items, st)) return rc;
        v.d_item_row = g->item_row.p;
        a->launches += v.num_items > 0;
        a->mg = std::move(g);
    }
    return GNNAGG_OK;
}

// the view the un-scheduled, un-sliced GCN aggregation of `a` runs on: the merged view when it is in use (its values
// re-summed on `st` when the edge values changed), else `a` itself
static int merged_view(gnnagg_aggregator *a, cudaStream_t st, View **out)
{
    *out = a;
    if (a->merge_mode == 1 || !a->d_val) return GNNAGG_OK;
    if (int rc = ensure_merged(a, st)) return rc;
    if (!merged_in_use(a)) return GNNAGG_OK;
    Merged &g = *a->mg;
    if (g.val_gen != a->val_gen) {
        merge_val_kernel<<<(unsigned)cdiv(g.v.m, 256), 256, 0, st>>>(a->d_val, g.start.p, g.val.p, g.v.m);
        LAUNCH_CHECK(a);
        g.val_gen = a->val_gen;
    }
    g.v.warp_edges = a->warp_edges;  // the setting follows the root's; automatic decides on m'
    *out = &g.v;
    return GNNAGG_OK;
}

static int gcn_layer_impl(gnnagg_aggregator *a, GatherX X, const float *W, float *H, float *AX, int feat_in, int feat_out,
                          int scheduled, void *stream)
{
    if (!a || !X.p || !W || !H) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_layer: NULL argument");
    float *ax = AX;
    if (!ax) {
        if (int rc = a->ax.ensure((size_t)a->n * feat_in)) return rc;
        ax = a->ax.p;
    }
    if (int rc = gcn_run_impl(a, X, ax, feat_in, scheduled, (cudaStream_t)stream, false)) return rc;
    if (a->n > 0) {
        if (int rc = dense_nn_launch(ax, W, H, a->n, feat_out, feat_in, stream)) return rc;
        a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
    }
    PROF_RECORD(a, 4, (cudaStream_t)stream);
    return GNNAGG_OK;
}

static int gcn_backward_impl(gnnagg_aggregator *a, GatherX dY, float *dX, int feat, cudaStream_t st)
{
    if (!a || !dY.p || !dX) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_backward: NULL argument");
    if (!a->tr) return set_error(GNNAGG_ERR_STATE, "gnnagg_gcn_backward: gnnagg_transpose_build has not run");
    if (!a->d_val && a->m > 0) return set_error(GNNAGG_ERR_STATE, "gnnagg_gcn_backward: edge values not set (gnnagg_set_val)");
    Transpose &t = *a->tr;
    if (t.val_gen != a->val_gen) {  // t.val[j] = val[perm[j]]: the edge values in transposed order
        if (a->m > 0) {
            gather_val_kernel<<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(a->d_val, t.perm.p, t.val.p, a->m);
            LAUNCH_CHECK(a);
        }
        t.val_gen = a->val_gen;
    }
    return gcn_run_core(t.v, dY, dX, feat, 0, st);
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
    std::unique_ptr<gnnagg_aggregator> a(new gnnagg_aggregator());
    a->root = a.get();
    a->records = true;
    a->d_ptr = d_ptr;
    a->d_idx = d_idx;
    a->h_ptr_user = h_ptr;
    a->n = num_v;
    a->m = num_e;
    if (int rc = item_table(a->item_row, d_ptr, num_v, num_e, &a->num_items, (cudaStream_t)stream)) return rc;
    a->d_item_row = a->item_row.p;
    a->launches += a->num_items > 0;
    *out = a.release();
    return GNNAGG_OK;
}

int gnnagg_destroy(gnnagg_aggregator *a)
{
    delete a;
    return GNNAGG_OK;
}

int gnnagg_set_val(gnnagg_aggregator *a, const float *d_val)
{
    const int rc = gnnagg_set_val_on(a, d_val, nullptr);
    if (rc == GNNAGG_OK && a->sched.perm.p) CUDA_TRY(cudaStreamSynchronize(0));  // the permuted copy is complete on return
    return rc;
}

int gnnagg_set_val_on(gnnagg_aggregator *a, const float *d_val, void *stream)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_set_val: NULL aggregator");
    a->d_val = d_val;
    ++a->val_gen;  // same pointer, possibly new contents (aggr_gcn.h:540-544): the derived copies are stale
    Schedule &s = a->sched;
    if (s.kind == GNNAGG_SCHED_NOP) return GNNAGG_OK;
    if (s.perm.p) {  // locality kinds keep a permuted copy (aggr_gcn.h:522-537)
        if (int rc = s.own_val.ensure((size_t)s.edges)) return rc;
        s.val = s.own_val.p;
        if (d_val && s.edges > 0) {
            gather_val_kernel<<<(unsigned)cdiv(s.edges, 256), 256, 0, (cudaStream_t)stream>>>(d_val, s.perm.p, s.own_val.p, s.edges);
            LAUNCH_CHECK(a);
        }
    } else {
        s.val = d_val;  // d_val_scheduled = d_val (aggr_gcn.h:506,542)
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
    Schedule &s = a->sched;
    s = Schedule();
    s.kind = kind;
    s.num_target = nt;
    s.edges = se;
    s.ptr.adopt(sp), s.target.adopt(stg), s.perm.adopt(sperm), s.own_idx.adopt(si);
    s.idx = si ? si : a->d_idx;
    if (int rc = item_table(s.item_row, sp, nt, se, &s.items, 0)) return rc;
    a->launches += s.items > 0;
    if (int rc = gnnagg_set_val(a, a->d_val)) return rc;
    CUDA_TRY(cudaStreamSynchronize(0));
    return GNNAGG_OK;
}

int gnnagg_schedule_kind(const gnnagg_aggregator *a) { return a ? a->sched.kind : GNNAGG_SCHED_NOP; }

int gnnagg_sched_to_csr_order(gnnagg_aggregator *a, const float *in_sched, float *out_csr, void *stream)
{
    if (!a || (a->m > 0 && (!in_sched || !out_csr))) return set_error(GNNAGG_ERR_ARG, "gnnagg_sched_to_csr_order: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (!a->sched.perm.p) {  // no schedule, or neighbour grouping: the scheduled order IS the CSR order
        if (in_sched != out_csr) CUDA_TRY(cudaMemcpyAsync(out_csr, in_sched, (size_t)a->m * sizeof(float), cudaMemcpyDeviceToDevice, st));
        return GNNAGG_OK;
    }
    if (in_sched == out_csr) return set_error(GNNAGG_ERR_ARG, "gnnagg_sched_to_csr_order: in place is not possible after a locality schedule");
    if (a->sched.edges != a->m)
        return set_error(GNNAGG_ERR_STATE, "gnnagg_sched_to_csr_order: the schedule dropped edges (sources outside the slice range)");
    scatter_val_kernel<<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(in_sched, a->sched.perm.p, out_csr, a->m);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_num_target(const gnnagg_aggregator *a) { return a ? a->sched.num_target : 0; }
const int *gnnagg_sched_dev_ptr(const gnnagg_aggregator *a) { return a ? a->sched.ptr.p : nullptr; }
const int *gnnagg_sched_dev_idx(const gnnagg_aggregator *a) { return a ? a->sched.idx : nullptr; }
const int *gnnagg_sched_dev_target(const gnnagg_aggregator *a) { return a ? a->sched.target.p : nullptr; }
const float *gnnagg_sched_dev_val(const gnnagg_aggregator *a) { return a ? a->sched.val : nullptr; }
const float *gnnagg_gat_edge_weights(const gnnagg_aggregator *a) { return a ? a->newval.p : nullptr; }
int64_t gnnagg_launch_count(const gnnagg_aggregator *a) { return a ? a->launches : 0; }

int gnnagg_set_warp_edges(gnnagg_aggregator *a, int warp_edges)
{
    if (!a || (warp_edges != 0 && warp_edges != 128 && warp_edges != 512))
        return set_error(GNNAGG_ERR_ARG, "gnnagg_set_warp_edges: 0, 128 or 512");
    a->warp_edges = warp_edges;
    if (a->tr) a->tr->v.warp_edges = warp_edges;
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
    return merged_in_use(a) ? a->mg->v.m : a->m;
}

int gnnagg_merged_dev(const gnnagg_aggregator *a, const int **ptr, const int **idx, const float **val)
{
    if (!a || !merged_in_use(a)) return set_error(GNNAGG_ERR_STATE, "gnnagg_merged_dev: the merged view is not in use");
    if (ptr) *ptr = a->mg->ptr.p;
    if (idx) *idx = a->mg->idx.p;
    if (val) *val = a->mg->val.p;
    return GNNAGG_OK;
}

int gnnagg_profile_enable(gnnagg_aggregator *a, int on)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_profile_enable: NULL aggregator");
    if (on && !a->ev.created())
        if (int rc = a->ev.create(cudaEventDefault)) return rc;
    a->prof = on != 0;
    return GNNAGG_OK;
}

int gnnagg_profile_read(gnnagg_aggregator *a, float *ms)
{
    if (!a || !ms || !a->ev.created()) return set_error(GNNAGG_ERR_STATE, "gnnagg_profile_read: profiling not enabled");
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
    View *t = a;
    if (int rc = merged_view(a, (cudaStream_t)stream, &t)) return rc;
    View &v = *t;
    const int EB = item_edges_for(v, feat, v.m);
    if (int rc = v.carry.ensure((size_t)cdiv(v.m, EB) * feat)) return rc;
    preload(agg_kernel_for<kModeGCN, false>(warp_edges_for(v, v.m), feat));
    preload(agg_kernel_for<kModeGCN, false, true>(warp_edges_for(v, v.m), feat));  // gnnagg_gcn_run_bf16
    preload(agg_fixup_kernel<kModeGCN>);
    preload(agg_fixup_long_kernel<kModeGCN>);
    AggParams p{};
    set_view(p, v);
    if (!long_rows_of(v, p, EB, (cudaStream_t)stream)) return GNNAGG_ERR_CUDA;
    const int *hp = nullptr;
    return host_ptr(v, &hp);  // row-range launches (gnnagg_gcn_run_rows) cut edge ranges on the host
}

static int gcn_run_rows_impl(gnnagg_aggregator *a, GatherX X, float *Y, int feat, int accumulate, int row_lo, int row_hi,
                             cudaStream_t st)
{
    if (!a) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run_rows: NULL aggregator");
    if (row_lo < 0 || row_hi > a->n || row_lo > row_hi) return set_error(GNNAGG_ERR_ARG, "gnnagg_gcn_run_rows: bad row range");
    if (row_lo == row_hi) return GNNAGG_OK;
    View *t = a;
    if (int rc = merged_view(a, st, &t)) return rc;
    const int *hp = nullptr;
    if (int rc = host_ptr(*t, &hp)) return rc;
    return gcn_run_core(*t, X, Y, feat, 0, st, accumulate != 0, row_lo, row_hi, hp[row_lo], hp[row_hi]);
}

int gnnagg_gcn_run_rows(gnnagg_aggregator *a, const float *X, float *Y, int feat, int accumulate, int row_lo, int row_hi,
                        void *stream)
{
    return gcn_run_rows_impl(a, X, Y, feat, accumulate, row_lo, row_hi, (cudaStream_t)stream);
}

int gnnagg_gcn_run_rows_bf16(gnnagg_aggregator *a, const uint16_t *X, float *Y, int feat, int accumulate, int row_lo,
                             int row_hi, void *stream)
{
    return gcn_run_rows_impl(a, X, Y, feat, accumulate, row_lo, row_hi, (cudaStream_t)stream);
}

int gnnagg_gcn_run(gnnagg_aggregator *a, const float *X, float *Y, int feat, int scheduled, void *stream)
{
    return gcn_run_impl(a, X, Y, feat, scheduled, (cudaStream_t)stream);
}

int gnnagg_gcn_run_bf16(gnnagg_aggregator *a, const uint16_t *X, float *Y, int feat, int scheduled, void *stream)
{
    return gcn_run_impl(a, X, Y, feat, scheduled, (cudaStream_t)stream);
}

int gnnagg_gcn_run_acc(gnnagg_aggregator *a, const float *X, float *Y, int feat, int accumulate, void *stream)
{
    return gcn_run_impl(a, X, Y, feat, 0, (cudaStream_t)stream, true, accumulate != 0);
}

int gnnagg_gcn_run_acc_bf16(gnnagg_aggregator *a, const uint16_t *X, float *Y, int feat, int accumulate, void *stream)
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
    return gcn_layer_impl(a, X, W, H, AX, feat_in, feat_out, scheduled, stream);
}

int gnnagg_gcn_layer_bf16(gnnagg_aggregator *a, const uint16_t *X, const float *W, float *H, float *AX, int feat_in,
                          int feat_out, int scheduled, void *stream)
{
    return gcn_layer_impl(a, X, W, H, AX, feat_in, feat_out, scheduled, stream);
}

int gnnagg_mlp_run(gnnagg_aggregator *a, const float *X, const float *W, float *Y, int feat, int scheduled,
                   void *stream)
{
    if (a && a->n == 0) return GNNAGG_OK;
    if (!a || !X || !W || !Y) return set_error(GNNAGG_ERR_ARG, "gnnagg_mlp_run: NULL argument");
    if (!aligned16(X) || !aligned16(Y)) return set_error(GNNAGG_ERR_ARG, "X and Y must be 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = a->ax.ensure((size_t)a->n * feat)) return rc;
    PROF_RECORD(a, 0, st);
    if (int rc = dense_nn_launch(X, W, a->ax.p, a->n, feat, feat, stream)) return rc;  // P = X W, once per call
    a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
    if (int rc = prof_agg_empty(a, st)) return rc;
    if (int rc = mlp_run_core(a, a->ax.p, Y, feat, scheduled, st)) return rc;
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
    const EdgeParams g = edge_params(*a);
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
    csr2edgelist_kernel<<<(unsigned)cdiv(a->m, 256), 256, 0, (cudaStream_t)stream>>>(edge_params(*a), d_edgelist);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_u_add_v(gnnagg_aggregator *a, const float *att, float *out_val, void *stream)
{
    if (!a || !att || (!out_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_u_add_v: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    edge_map_kernel<kEdgeUAddV><<<(unsigned)cdiv(a->m, 256), 256, 0, (cudaStream_t)stream>>>(edge_params(*a), att, out_val, 0.f);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_add_to_center(gnnagg_aggregator *a, const float *in_val, float *out_center, void *stream)
{
    if (!a || !out_center || (!in_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_add_to_center: NULL argument");
    return rowsum_impl(*a, in_val, out_center, (cudaStream_t)stream);
}

int gnnagg_each_div(gnnagg_aggregator *a, const float *in_center, float *inout_val, void *stream)
{
    if (!a || !in_center || (!inout_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_each_div: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    edge_map_kernel<kEdgeDiv><<<(unsigned)cdiv(a->m, 256), 256, 0, (cudaStream_t)stream>>>(edge_params(*a), in_center, inout_val, 0.f);
    LAUNCH_CHECK(a);
    return GNNAGG_OK;
}

int gnnagg_edge_softmax(gnnagg_aggregator *a, const float *att, float *out_val, float slope, void *stream)
{
    if (!a || !att || (!out_val && a->m > 0)) return set_error(GNNAGG_ERR_ARG, "gnnagg_edge_softmax: NULL argument");
    if (a->m == 0) return GNNAGG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = a->den_row.ensure((size_t)a->n)) return rc;
    const EdgeParams g = edge_params(*a);
    edge_map_kernel<kEdgeWeight><<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(g, att, out_val, slope);
    LAUNCH_CHECK(a);
    if (int rc = rowsum_impl(*a, out_val, a->den_row.p, st)) return rc;
    edge_map_kernel<kEdgeDiv><<<(unsigned)cdiv(a->m, 256), 256, 0, st>>>(g, a->den_row.p, out_val, 0.f);
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
        if (a->sched.kind != GNNAGG_SCHED_NEIGHBOR_GROUPING)  // aggr_sddmm.h:100
            return set_error(GNNAGG_ERR_STATE, "scheduled SDDMM needs a neighbor_grouping schedule");
        if (a->sched.edges == 0) return GNNAGG_OK;
        set_sched(p, a);
        p.bulk_ok = aligned16(p.idx);
        return launch_agg<kModeSDDMM, true>(*a, p, st);
    }
    if (a->m == 0) return GNNAGG_OK;
    set_view(p, *a);
    p.bulk_ok = aligned16(p.idx);
    return launch_agg<kModeSDDMM, false>(*a, p, st);
}

int gnnagg_transpose_build(gnnagg_aggregator *a, int num_src, void *stream)
{
    if (!a || num_src < 0) return set_error(GNNAGG_ERR_ARG, "gnnagg_transpose_build: bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    a->tr.reset();
    auto t = std::make_unique<Transpose>();
    int *tp = nullptr, *ti = nullptr, *tq = nullptr;
    if (int rc = transpose_build_device(a->d_ptr, a->d_idx, a->d_item_row, a->num_items, a->n, a->m, num_src, &tp, &ti, &tq, st))
        return rc;
    t->ptr.adopt(tp), t->idx.adopt(ti), t->perm.adopt(tq);
    View &v = t->v;
    v.root = a;
    v.d_ptr = tp;
    v.d_idx = ti;
    v.n = num_src;
    v.m = a->m;
    v.warp_edges = a->warp_edges;
    int rc = item_table(t->item_row, tp, num_src, a->m, &v.num_items, st);
    if (rc == GNNAGG_OK && t->val.ensure((size_t)a->m) != GNNAGG_OK)
        rc = set_error(GNNAGG_ERR_CUDA, "gnnagg_transpose_build: out of device memory");
    if (rc != GNNAGG_OK) return rc;  // never leave a half-built transpose behind
    v.d_item_row = t->item_row.p;
    v.d_val = t->val.p;
    a->tr = std::move(t);
    a->launches += 5;  // iota, radix sort (counted once), rows, pointers, item table
    return GNNAGG_OK;
}

int gnnagg_transpose_dev(const gnnagg_aggregator *a, int *num_src, const int **t_ptr, const int **t_idx, const int **t_perm)
{
    if (!a || !a->tr) return set_error(GNNAGG_ERR_STATE, "gnnagg_transpose_dev: gnnagg_transpose_build has not run");
    if (num_src) *num_src = a->tr->v.n;
    if (t_ptr) *t_ptr = a->tr->ptr.p;
    if (t_idx) *t_idx = a->tr->idx.p;
    if (t_perm) *t_perm = a->tr->perm.p;
    return GNNAGG_OK;
}

int gnnagg_gcn_backward(gnnagg_aggregator *a, const float *dY, float *dX, int feat, void *stream)
{
    return gcn_backward_impl(a, dY, dX, feat, (cudaStream_t)stream);
}

int gnnagg_gcn_backward_bf16(gnnagg_aggregator *a, const uint16_t *dY, float *dX, int feat, void *stream)
{
    return gcn_backward_impl(a, dY, dX, feat, (cudaStream_t)stream);
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
    Transpose &tr = *a->tr;
    View &t = tr.v;
    // every row < n gets its destination half and every row < num_src its source half from the kernels below; only a
    // rectangular block leaves entries of the [max(n, num_src), 2] table that nobody writes
    const int rows = a->n > t.n ? a->n : t.n;
    if (a->n != t.n || a->m == 0) CUDA_TRY(cudaMemsetAsync(datt, 0, (size_t)rows * 2 * sizeof(float), st));
    if (a->m == 0) {
        CUDA_TRY(cudaMemsetAsync(dX, 0, (size_t)t.n * feat * sizeof(float), st));
        return GNNAGG_OK;
    }
    const int EB = item_edges_for(*a, feat, a->m);
    const int EBt = item_edges_for(t, feat, a->m);
    if (int rc = a->bwd_c.ensure((size_t)a->n)) return rc;
    if (int rc = a->bwd_wt.ensure((size_t)a->m)) return rc;
    if (int rc = a->bwd_part.ensure((size_t)a->n)) return rc;
    if (int rc = a->bwd_carry.ensure((size_t)cdiv(a->m, EB) + 1)) return rc;
    if (int rc = t.carry.ensure((size_t)cdiv(a->m, EBt) * feat)) return rc;
    if (int rc = t.carry_den.ensure((size_t)cdiv(a->m, EBt))) return rc;
    if (int rc = t.den_row.ensure((size_t)t.n)) return rc;
    const bool large = a->m >= kSmallGraphEdges;  // (w, t) of the graph does not stay in L2: see step 4
    if (large)
        if (int rc = a->bwd_t.ensure((size_t)a->m)) return rc;
    // 1. per destination row: c_v = <Y[v], dY[v]>
    gat_bwd_rowinfo_kernel<<<(unsigned)cdiv((int64_t)a->n * 8, 256), 256, 0, st>>>(Y, dY, a->bwd_c.p, a->n, feat);
    LAUNCH_CHECK(a);
    // 2. pass 1 over the CSR: g_e = <X[u], dY[v]> (the SDDMM traversal), per edge (w_e, t_e), per row their sums
    {
        AggParams p{};
        p.X = X;
        p.P = dY;
        p.att = att;
        p.val = w;
        p.bwd_c = a->bwd_c.p;
        p.bwd_wt = a->bwd_wt.p;
        p.bwd_part = a->bwd_part.p;
        p.bwd_carry = a->bwd_carry.p;
        p.F = feat;
        p.slope = slope;
        set_view(p, *a);
        p.bulk_ok = aligned16(p.idx) && (att || aligned16(w));
        if (int rc = launch_agg<kModeGATBWD, false>(*a, p, st)) return rc;
    }
    // 3. rows closed: 1 / D_v and the destination half of the attention gradient
    launch_dep(gat_bwd_rowfinal_kernel, (unsigned)cdiv((int64_t)a->n * 8, 256), 256, st, a->d_ptr, a->bwd_part.p,
               a->bwd_carry.p, den, a->bwd_c.p, datt, a->n, EB);
    LAUNCH_CHECK(a);
    if (large) {
        // 4a. large graphs: (w, t) permuted into transposed order by a streaming kernel, then the source half as a row sum
        //     and dX as the plain aggregation over the transposed CSR with edge values alpha
        launch_dep(gat_bwd_permute_kernel, (unsigned)cdiv(a->m, 256), 256, st, (const float2 *)a->bwd_wt.p,
                   (const int *)tr.perm.p, (const int *)tr.idx.p, (const float2 *)a->bwd_c.p, tr.val.p, a->bwd_t.p, a->m);
        LAUNCH_CHECK(a);
        tr.val_gen = 0;  // tr.val no longer mirrors the GCN edge values
        if (int rc = rowsum_impl(t, a->bwd_t.p, datt + 1, st, 2)) return rc;
        return gcn_run_core(t, dY, dX, feat, 0, st);
    }
    // 4b. pass 2 over the transposed CSR: dX[u] = sum_e alpha_e dY[v] and the source half sum_e ds_e, weights formed on
    //     the fly from (w, t) through tr.perm and 1 / D_v ((w, t) of a small graph stays in L2)
    AggParams p{};
    p.X = dY;
    p.Y = dX;
    p.val = reinterpret_cast<const float *>(tr.perm.p);
    p.bwd_c = a->bwd_c.p;
    p.bwd_wt = a->bwd_wt.p;
    p.rsum = datt + 1;
    p.rsum_stride = 2;
    p.F = feat;
    set_view(p, t);
    p.carry = t.carry.p;
    p.carry_den = t.carry_den.p;
    p.den_row = t.den_row.p;
    p.bulk_ok = aligned16(p.idx) && aligned16(p.val);
    return launch_agg<kModeGATBWD2, false>(t, p, st);
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
    if (int rc = a->st_in.ensure(cin)) return rc;
    if (int rc = a->st_out.ensure(cout)) return rc;
    if (layer) {
        if (int rc = a->st_w.ensure((size_t)feat_in * feat_out)) return rc;
        if (int rc = a->ax.ensure(cin)) return rc;
        CUDA_TRY(cudaMemcpyAsync(a->st_w.p, h_W, (size_t)feat_in * feat_out * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    float *st_in = a->st_in.p, *st_out = a->st_out.p, *agg_out = layer ? a->ax.p : st_out;
    if (scheduled || a->n < 4096) {  // scheduled order is not row-contiguous; tiny graphs are not worth chunking
        CUDA_TRY(cudaMemcpyAsync(st_in, h_X, cin * sizeof(float), cudaMemcpyHostToDevice, st));
        if (int rc = gcn_run_impl(a, st_in, agg_out, feat_in, scheduled, st, !layer)) return rc;
        if (layer && a->n > 0) {
            if (int rc = dense_nn_launch(a->ax.p, a->st_w.p, st_out, a->n, feat_out, feat_in, st)) return rc;
            a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
        }
        CUDA_TRY(cudaMemcpyAsync(h_out, st_out, cout * sizeof(float), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        return GNNAGG_OK;
    }
    if (int rc = check_feat(feat_in)) return rc;
    if (!a->d_val && a->m > 0) return set_error(GNNAGG_ERR_STATE, "edge values not set (gnnagg_set_val)");
    if (int rc = a->copy.ensure()) return rc;
    const int S = a->host_slices > 0 ? a->host_slices : (a->host_slices == 0 && a->m >= kSmallGraphEdges ? kHostSlices : 1);
    // the views whose rows are chunked for the copy back: the graph itself (or its merged view), or the trailing slices
    View *tail[2] = {a, nullptr};
    int tail_first = 0, tail_count = 1;
    if (S > 1) {
        if (int rc = ensure_slices(a, a->host, S, st)) return rc;
        if (int rc = a->in.ensure()) return rc;
        const Events<9> &in_ev = a->in.ev;
        const int width = a->host->width;
        // input blocks on their own stream, after everything already queued on `st` (a previous call may still read st_in)
        CUDA_TRY(cudaEventRecord(in_ev[8], st));
        CUDA_TRY(cudaStreamWaitEvent(a->in.stream, in_ev[8], 0));
        for (int c = 0; c < S; ++c) {
            const int64_t r0 = std::min<int64_t>((int64_t)c * width, a->n), r1 = std::min<int64_t>(r0 + width, a->n);
            if (r1 > r0)
                CUDA_TRY(cudaMemcpyAsync(st_in + (size_t)r0 * feat_in, h_X + (size_t)r0 * feat_in,
                                         (size_t)(r1 - r0) * feat_in * sizeof(float), cudaMemcpyHostToDevice, a->in.stream));
            CUDA_TRY(cudaEventRecord(in_ev[c], a->in.stream));
        }
        // The aggregation is longer than the input copy, so when the last block lands part of the second-to-last slice
        // is still to do: the last TWO slices run row chunk by row chunk (both slices of a chunk, its combination, its
        // copy back), the slices before them over all rows as their block arrives.
        tail_count = 2;
        tail_first = S - tail_count;
        for (int c = 0; c < tail_first; ++c) {
            CUDA_TRY(cudaStreamWaitEvent(st, in_ev[c], 0));
            if (int rc = gcn_run_core(a->host->slice[c].v, st_in, agg_out, feat_in, 0, st, c > 0)) return rc;
        }
        tail[0] = &a->host->slice[tail_first].v;
        tail[1] = &a->host->slice[tail_first + 1].v;
    } else {
        CUDA_TRY(cudaMemcpyAsync(st_in, h_X, cin * sizeof(float), cudaMemcpyHostToDevice, st));
        if (int rc = merged_view(a, st, &tail[0])) return rc;  // the rows gcn_run aggregates, chunk by chunk
    }
    const int *hp[2] = {nullptr, nullptr};
    for (int t = 0; t < tail_count; ++t)
        if (int rc = host_ptr(*tail[t], &hp[t])) return rc;
    int bounds[kHostChunks + 1];
    if (S > 1) {  // equal ROW counts: the chunks are sized for the copy back
        for (int c = 0; c <= kHostChunks; ++c) bounds[c] = (int)((int64_t)a->n * c / kHostChunks);
    } else {
        row_chunks(hp[0], a->n, tail[0]->m, kHostChunks, bounds);
    }
    const Events<9> &copy_ev = a->copy.ev;
    for (int c = 0; c < kHostChunks; ++c) {
        const int r0 = bounds[c], r1 = bounds[c + 1];
        if (r1 <= r0) continue;
        for (int t = 0; t < tail_count; ++t) {
            if (S > 1 && c == 0) CUDA_TRY(cudaStreamWaitEvent(st, a->in.ev[tail_first + t], 0));
            if (int rc = gcn_run_core(*tail[t], st_in, agg_out, feat_in, 0, st, S > 1 && (tail_first + t) > 0, r0, r1,
                                      hp[t][r0], hp[t][r1]))
                return rc;
        }
        if (layer) {
            if (int rc = dense_nn_launch(a->ax.p + (size_t)r0 * feat_in, a->st_w.p, st_out + (size_t)r0 * fo, r1 - r0, feat_out,
                                         feat_in, st))
                return rc;
            a->launches += 2;  // split_w_kernel + dense_tf32x3_ws_kernel
        }
        CUDA_TRY(cudaEventRecord(copy_ev[c], st));
        CUDA_TRY(cudaStreamWaitEvent(a->copy.stream, copy_ev[c], 0));
        CUDA_TRY(cudaMemcpyAsync(h_out + (size_t)r0 * fo, st_out + (size_t)r0 * fo, (size_t)(r1 - r0) * fo * sizeof(float),
                                 cudaMemcpyDeviceToHost, a->copy.stream));
    }
    CUDA_TRY(cudaEventRecord(copy_ev[8], a->copy.stream));
    CUDA_TRY(cudaStreamWaitEvent(st, copy_ev[8], 0));  // the caller's stream is ordered after the copies as well
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
    if (int rc = a->st_in.ensure(cnt)) return rc;
    if (int rc = a->st_out.ensure(cnt)) return rc;
    if (int rc = a->st_att.ensure((size_t)a->n * 2)) return rc;
    CUDA_TRY(cudaMemcpyAsync(a->st_in.p, h_X, cnt * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(a->st_att.p, h_att, (size_t)a->n * 2 * sizeof(float), cudaMemcpyHostToDevice, st));
    if (int rc = gat_run_impl(a, a->st_in.p, a->st_att.p, a->st_out.p, feat, slope, scheduled, st)) return rc;
    CUDA_TRY(cudaMemcpyAsync(h_Y, a->st_out.p, cnt * sizeof(float), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return GNNAGG_OK;
}
}
