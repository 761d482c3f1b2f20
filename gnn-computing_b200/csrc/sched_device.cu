// sched_device.cu -- the three schedules of include/graph_schedule.h built ON THE GPU, bit-identical to the
// host builders (host_prep.cpp / the reference), for gnnagg_schedule_apply.
//
// The reference builds schedules on the host from a device->host mirror of the CSR and uploads three vectors
// (aggregator.h:67-99); its locality variants rescan all edges once per slice (graph_schedule.h:24-63).  Here:
//   neighbour grouping : groups per row = ceil(deg/NG) -> exclusive scan -> one thread per row writes its groups;
//                        idx (and val) are NOT copied: the schedule keeps the CSR edge order (:123-124).
//   locality (+NG)     : key(e) = slice(src(e)) * n + row(e); a STABLE radix sort of the edge ids by key is
//                        exactly "for every slice, for every row, neighbours in CSR order" (:24-43); runs of equal
//                        keys are the (slice,row) groups (:54-57), cut every NG edges in the combined variant
//                        (:182-190, :202-209); edges whose source lies outside [0,total) get the largest key
//                        and are dropped, as the range test of the reference drops them (:37).
// Scans / sort / run-length encoding come from CUB (part of the CUDA toolkit, like the Thrust the reference uses
// in sample.h).
#include <cub/cub.cuh>

#include "common.cuh"
#include "gnnagg.h"
#include "internal.h"

namespace gnnagg {

#define SD_TRY(expr)                                                          \
    do {                                                                      \
        cudaError_t _e = (expr);                                              \
        if (_e != cudaSuccess) {                                              \
            set_error(GNNAGG_ERR_CUDA, cudaGetErrorString(_e));               \
            goto fail;                                                        \
        }                                                                     \
    } while (0)

__global__ void __launch_bounds__(256) ng_count_kernel(const int *__restrict__ ptr, int n, int ng, int *__restrict__ groups)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) groups[r] = (ptr[r + 1] - ptr[r] + ng - 1) / ng;
}

__global__ void __launch_bounds__(256) ng_fill_kernel(const int *__restrict__ ptr, const int *__restrict__ gstart, int n, int ng,
                                                      int *__restrict__ out_ptr, int *__restrict__ out_target)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int end = ptr[r + 1];
    int g = gstart[r];
    for (int b = ptr[r]; b < end; b += ng, ++g) {
        out_ptr[g + 1] = min(b + ng, end);
        out_target[g] = r;
    }
    if (r == 0) out_ptr[0] = 0;
}

// key of every edge: slice * n + row, or the sentinel for sources outside [0,total)
__global__ void __launch_bounds__(256) loc_key_kernel(const int *__restrict__ ptr, const int *__restrict__ idx,
                                                      const int *__restrict__ item_row, int num_items, int n, int m, int par_num,
                                                      int total, uint64_t sentinel, uint64_t *__restrict__ keys,
                                                      int *__restrict__ edge_id)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int row = row_of_edge(ptr, item_row, num_items, n, e);
    const int src = idx[e];
    const int w = total / par_num;
    uint64_t key = sentinel;
    if (src >= 0 && src < total) {
        int p = (w == 0) ? par_num - 1 : src / w;  // graph_schedule.h:26-29: slices of floor(total/par), the last one runs to total
        if (p >= par_num) p = par_num - 1;
        key = (uint64_t)p * (uint64_t)n + (uint64_t)row;
    }
    keys[e] = key;
    edge_id[e] = e;
}

__global__ void __launch_bounds__(256) run_groups_kernel(const int *__restrict__ run_len, int num_runs, int ng,
                                                         const uint64_t *__restrict__ run_key, uint64_t sentinel,
                                                         int *__restrict__ groups)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= num_runs) return;
    groups[k] = (run_key[k] == sentinel) ? 0 : (ng > 0 ? (run_len[k] + ng - 1) / ng : 1);
}

__global__ void __launch_bounds__(256) run_fill_kernel(const int *__restrict__ run_len, const int *__restrict__ run_start,
                                                       const int *__restrict__ gstart, const uint64_t *__restrict__ run_key,
                                                       int num_runs, int ng, int n, uint64_t sentinel, int *__restrict__ out_ptr,
                                                       int *__restrict__ out_target)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k == 0) out_ptr[0] = 0;
    if (k >= num_runs || run_key[k] == sentinel) return;
    const int begin = run_start[k], end = begin + run_len[k];
    const int row = (int)(run_key[k] % (uint64_t)n);
    const int step = ng > 0 ? ng : run_len[k];
    int g = gstart[k];
    for (int b = begin; b < end; b += step, ++g) {
        out_ptr[g + 1] = min(b + step, end);
        out_target[g] = row;
    }
}

__global__ void __launch_bounds__(256) gather_idx_kernel(const int *__restrict__ idx, const int *__restrict__ perm,
                                                         int *__restrict__ out, int count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = __ldg(idx + __ldg(perm + i));
}

static inline unsigned blocks(int64_t n) { return (unsigned)((n + 255) / 256); }

// Device schedule build.  Outputs are cudaMalloc'ed here and owned by the caller:
//   *s_ptr [G+1], *s_target [G]; locality kinds additionally *s_idx [E'] and *s_perm [E'] (CSR edge id at every
//   scheduled position; neighbour grouping leaves both NULL: its order is the CSR order).
int schedule_build_device(int kind, const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                          int par_num, int ng, int total, int **s_ptr, int **s_idx, int **s_target, int **s_perm,
                          int *num_target, int *sched_edges, cudaStream_t st)
{
    *s_ptr = *s_idx = *s_target = *s_perm = nullptr;
    *num_target = 0;
    *sched_edges = 0;
    int *groups = nullptr, *gstart = nullptr, *edge_id = nullptr, *perm = nullptr, *run_len = nullptr, *run_start = nullptr,
        *num_runs_d = nullptr;
    uint64_t *keys = nullptr, *keys_sorted = nullptr, *run_key = nullptr;
    void *tmp = nullptr;
    size_t tmp_bytes = 0, need = 0;
    int G = 0;
    auto scratch = [&](size_t bytes) -> cudaError_t {
        if (bytes <= tmp_bytes) return cudaSuccess;
        if (tmp) cudaFree(tmp);
        tmp = nullptr;
        tmp_bytes = 0;
        cudaError_t e = cudaMalloc(&tmp, bytes ? bytes : 1);
        if (e == cudaSuccess) tmp_bytes = bytes;
        return e;
    };

    if (kind == GNNAGG_SCHED_NEIGHBOR_GROUPING) {
        if (ng <= 0) return set_error(GNNAGG_ERR_ARG, "neighbor_num must be > 0");
        SD_TRY(cudaMalloc((void **)&groups, (size_t)(n + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&gstart, (size_t)(n + 1) * sizeof(int)));
        SD_TRY(cudaMemsetAsync(groups, 0, (size_t)(n + 1) * sizeof(int), st));
        if (n > 0) ng_count_kernel<<<blocks(n), 256, 0, st>>>(d_ptr, n, ng, groups);
        SD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, groups, gstart, n + 1, st));
        SD_TRY(scratch(need));
        SD_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, groups, gstart, n + 1, st));
        SD_TRY(cudaMemcpyAsync(&G, gstart + n, sizeof(int), cudaMemcpyDeviceToHost, st));
        SD_TRY(cudaStreamSynchronize(st));
        SD_TRY(cudaMalloc((void **)s_ptr, (size_t)(G + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)s_target, (size_t)(G > 0 ? G : 1) * sizeof(int)));
        SD_TRY(cudaMemsetAsync(*s_ptr, 0, sizeof(int), st));
        if (n > 0) ng_fill_kernel<<<blocks(n), 256, 0, st>>>(d_ptr, gstart, n, ng, *s_ptr, *s_target);
        *num_target = G;
        *sched_edges = m;
    } else {
        if (par_num <= 0 || (kind == GNNAGG_SCHED_LOCALITY_NEIGHBOR_GROUPING && ng <= 0))
            return set_error(GNNAGG_ERR_ARG, "par_num, neighbor_num must be > 0");
        if (kind == GNNAGG_SCHED_LOCALITY) ng = 0;
        const uint64_t sentinel = (uint64_t)par_num * (uint64_t)(n > 0 ? n : 1);  // larger than every real key
        int end_bit = 1;
        while (end_bit < 64 && (sentinel >> end_bit) != 0) ++end_bit;
        const size_t me = (size_t)(m > 0 ? m : 1);
        SD_TRY(cudaMalloc((void **)&keys, me * sizeof(uint64_t)));
        SD_TRY(cudaMalloc((void **)&keys_sorted, me * sizeof(uint64_t)));
        SD_TRY(cudaMalloc((void **)&edge_id, me * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&perm, me * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&run_key, me * sizeof(uint64_t)));
        SD_TRY(cudaMalloc((void **)&run_len, (me + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&run_start, (me + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&groups, (me + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&gstart, (me + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&num_runs_d, sizeof(int)));
        int num_runs = 0, last_len = 0, E = m;
        uint64_t last_key = 0;
        if (m > 0) {
            loc_key_kernel<<<blocks(m), 256, 0, st>>>(d_ptr, d_idx, d_item_row, num_items, n, m, par_num, total, sentinel, keys,
                                                     edge_id);
            SD_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, keys, keys_sorted, edge_id, perm, m, 0, end_bit, st));
            SD_TRY(scratch(need));
            SD_TRY(cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, keys_sorted, edge_id, perm, m, 0, end_bit, st));  // stable
            SD_TRY(cub::DeviceRunLengthEncode::Encode(nullptr, need, keys_sorted, run_key, run_len, num_runs_d, m, st));
            SD_TRY(scratch(need));
            SD_TRY(cub::DeviceRunLengthEncode::Encode(tmp, tmp_bytes, keys_sorted, run_key, run_len, num_runs_d, m, st));
            SD_TRY(cudaMemcpyAsync(&num_runs, num_runs_d, sizeof(int), cudaMemcpyDeviceToHost, st));
            SD_TRY(cudaStreamSynchronize(st));
            // dropped edges form the last run (sentinel key)
            SD_TRY(cudaMemcpyAsync(&last_key, run_key + (num_runs - 1), sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
            SD_TRY(cudaMemcpyAsync(&last_len, run_len + (num_runs - 1), sizeof(int), cudaMemcpyDeviceToHost, st));
            SD_TRY(cudaStreamSynchronize(st));
            if (last_key == sentinel) E = m - last_len;
            SD_TRY(cudaMemsetAsync(run_len + num_runs, 0, sizeof(int), st));
            SD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, run_len, run_start, num_runs + 1, st));
            SD_TRY(scratch(need));
            SD_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, run_len, run_start, num_runs + 1, st));
            run_groups_kernel<<<blocks(num_runs), 256, 0, st>>>(run_len, num_runs, ng, run_key, sentinel, groups);
            SD_TRY(cudaMemsetAsync(groups + num_runs, 0, sizeof(int), st));
            SD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, groups, gstart, num_runs + 1, st));
            SD_TRY(scratch(need));
            SD_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, groups, gstart, num_runs + 1, st));
            SD_TRY(cudaMemcpyAsync(&G, gstart + num_runs, sizeof(int), cudaMemcpyDeviceToHost, st));
            SD_TRY(cudaStreamSynchronize(st));
        }
        SD_TRY(cudaMalloc((void **)s_ptr, (size_t)(G + 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)s_target, (size_t)(G > 0 ? G : 1) * sizeof(int)));
        SD_TRY(cudaMalloc((void **)s_idx, (size_t)(E > 0 ? E : 1) * sizeof(int)));
        SD_TRY(cudaMemsetAsync(*s_ptr, 0, sizeof(int), st));
        if (num_runs > 0)
            run_fill_kernel<<<blocks(num_runs), 256, 0, st>>>(run_len, run_start, gstart, run_key, num_runs, ng, n, sentinel,
                                                             *s_ptr, *s_target);
        if (E > 0) gather_idx_kernel<<<blocks(E), 256, 0, st>>>(d_idx, perm, *s_idx, E);
        *s_perm = perm;  // first E entries are the scheduled order
        perm = nullptr;
        *num_target = G;
        *sched_edges = E;
    }
    SD_TRY(cudaGetLastError());
    SD_TRY(cudaStreamSynchronize(st));
    cudaFree(groups), cudaFree(gstart), cudaFree(edge_id), cudaFree(perm), cudaFree(run_len), cudaFree(run_start),
        cudaFree(num_runs_d), cudaFree(keys), cudaFree(keys_sorted), cudaFree(run_key), cudaFree(tmp);
    return GNNAGG_OK;
fail:
    cudaFree(groups), cudaFree(gstart), cudaFree(edge_id), cudaFree(perm), cudaFree(run_len), cudaFree(run_start),
        cudaFree(num_runs_d), cudaFree(keys), cudaFree(keys_sorted), cudaFree(run_key), cudaFree(tmp);
    cudaFree(*s_ptr), cudaFree(*s_idx), cudaFree(*s_target), cudaFree(*s_perm);
    *s_ptr = *s_idx = *s_target = *s_perm = nullptr;
    return GNNAGG_ERR_CUDA;
}


// ---------------------------------------------------------------------------------------------------------
// Transposed CSR for the backward pass (gnnagg_transpose_build): edges grouped by SOURCE, inside a source in
// CSR order (a stable sort), so the gradient w.r.t. the gathered rows is again a gather-side aggregation
//   dX[u,:] = sum over edges (v <- u) of w_e dY[v,:]
// that runs through the same deterministic agg_kernel instead of the float atomics of the reference's
// aggr_gat_fine_bwd (aggr_gat.h:264).
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) iota_kernel(int *__restrict__ out, int count)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = i;
}

__global__ void __launch_bounds__(256) edge_rows_kernel(const int *__restrict__ ptr, const int *__restrict__ item_row,
                                                        int num_items, int n, const int *__restrict__ perm, int m,
                                                        int *__restrict__ out)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) out[j] = row_of_edge(ptr, item_row, num_items, n, __ldg(perm + j));
}

// row pointers from the sorted keys: t_ptr[u] = first position whose key is >= u
__global__ void __launch_bounds__(256) ptr_from_sorted_kernel(const int *__restrict__ keys, int m, int num_src,
                                                              int *__restrict__ t_ptr)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j > m) return;
    const int lo = (j == 0) ? 0 : __ldg(keys + j - 1) + 1;
    const int hi = (j == m) ? num_src : __ldg(keys + j);
    for (int u = lo; u <= hi; ++u) t_ptr[u] = j;
}

int transpose_build_device(const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                           int num_src, int **t_ptr, int **t_idx, int **t_perm, cudaStream_t st)
{
    *t_ptr = *t_idx = *t_perm = nullptr;
    int *edge_id = nullptr, *keys_sorted = nullptr;
    void *tmp = nullptr;
    size_t need = 0;
    int ends[2] = {0, 0};
    const size_t me = (size_t)(m > 0 ? m : 1);
    SD_TRY(cudaMalloc((void **)t_ptr, ((size_t)num_src + 1) * sizeof(int)));
    SD_TRY(cudaMalloc((void **)t_idx, me * sizeof(int)));
    SD_TRY(cudaMalloc((void **)t_perm, me * sizeof(int)));
    if (m == 0) {
        SD_TRY(cudaMemsetAsync(*t_ptr, 0, ((size_t)num_src + 1) * sizeof(int), st));
    } else {
        SD_TRY(cudaMalloc((void **)&edge_id, me * sizeof(int)));
        SD_TRY(cudaMalloc((void **)&keys_sorted, me * sizeof(int)));
        iota_kernel<<<blocks(m), 256, 0, st>>>(edge_id, m);
        SD_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, d_idx, keys_sorted, edge_id, *t_perm, m, 0, 32, st));
        SD_TRY(cudaMalloc(&tmp, need ? need : 1));
        SD_TRY(cub::DeviceRadixSort::SortPairs(tmp, need, d_idx, keys_sorted, edge_id, *t_perm, m, 0, 32, st));  // stable
        SD_TRY(cudaMemcpyAsync(&ends[0], keys_sorted, sizeof(int), cudaMemcpyDeviceToHost, st));
        SD_TRY(cudaMemcpyAsync(&ends[1], keys_sorted + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, st));
        SD_TRY(cudaStreamSynchronize(st));
        if (ends[0] < 0 || ends[1] >= num_src) {
            set_error(GNNAGG_ERR_ARG, "gnnagg_transpose_build: a source id lies outside [0, num_src)");
            goto fail_keep_error;
        }
        edge_rows_kernel<<<blocks(m), 256, 0, st>>>(d_ptr, d_item_row, num_items, n, *t_perm, m, *t_idx);
        ptr_from_sorted_kernel<<<blocks((int64_t)m + 1), 256, 0, st>>>(keys_sorted, m, num_src, *t_ptr);
    }
    SD_TRY(cudaGetLastError());
    SD_TRY(cudaStreamSynchronize(st));
    cudaFree(edge_id), cudaFree(keys_sorted), cudaFree(tmp);
    return GNNAGG_OK;
fail:
    cudaFree(edge_id), cudaFree(keys_sorted), cudaFree(tmp);
    cudaFree(*t_ptr), cudaFree(*t_idx), cudaFree(*t_perm);
    *t_ptr = *t_idx = *t_perm = nullptr;
    return GNNAGG_ERR_CUDA;
fail_keep_error:
    cudaFree(edge_id), cudaFree(keys_sorted), cudaFree(tmp);
    cudaFree(*t_ptr), cudaFree(*t_idx), cudaFree(*t_perm);
    *t_ptr = *t_idx = *t_perm = nullptr;
    return GNNAGG_ERR_ARG;
}


// ---------------------------------------------------------------------------------------------------------
// Source slices for the host-buffer pipeline (capi.cu: gcn_host_pipeline): the CSR split by ranges of the SOURCE
// id into S sub-CSRs over the same rows -- the locality slices of graph_schedule.h:24-29, kept as complete CSRs so
// that each one runs through the deterministic un-scheduled kernel in accumulate mode.  Slice c only gathers rows
// [src_bounds[c], src_bounds[c+1]) of X, so its aggregation can start as soon as that part of X has arrived from
// the host.  Edge order inside a slice is CSR order (stable sort).  Outputs (cudaMalloc'ed, owned by the caller):
//   *sl_ptr  [S*(n+1)]  row pointers of every slice, relative to the slice's own edge array
//   *sl_idx, *sl_perm   source ids / CSR edge ids; slice c occupies [edge_off[c], edge_off[c] + edge_cnt[c]),
//                       edge_off[c] a multiple of 4 (16-byte aligned slices keep the bulk-copy staging usable)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) slice_key_kernel(const int *__restrict__ idx, int m, int num_slices, int width,
                                                        int *__restrict__ keys, int *__restrict__ edge_id)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    keys[e] = min(__ldg(idx + e) / width, num_slices - 1);
    edge_id[e] = e;
}

int source_slices_build_device(const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                               int num_slices, int width, int **sl_ptr, int **sl_idx, int **sl_perm, int *edge_off,
                               int *edge_cnt, cudaStream_t st, const int *d_edge_keys)
{
    *sl_ptr = *sl_idx = *sl_perm = nullptr;
    int *keys = nullptr, *keys_sorted = nullptr, *edge_id = nullptr, *perm = nullptr, *rows_sorted = nullptr, *bounds_d = nullptr;
    void *tmp = nullptr;
    size_t need = 0;
    int bounds[65] = {0};
    const size_t me = (size_t)(m > 0 ? m : 1);
    const size_t padded = me + 4 * (size_t)num_slices;
    int end_bit = 1;
    while ((1 << end_bit) < num_slices) ++end_bit;
    if (num_slices < 1 || num_slices > 64 || width < 1) return set_error(GNNAGG_ERR_ARG, "source slices: bad slice count");
    SD_TRY(cudaMalloc((void **)sl_ptr, (size_t)num_slices * ((size_t)n + 1) * sizeof(int)));
    SD_TRY(cudaMalloc((void **)sl_idx, padded * sizeof(int)));
    SD_TRY(cudaMalloc((void **)sl_perm, padded * sizeof(int)));
    SD_TRY(cudaMemsetAsync(*sl_perm, 0, padded * sizeof(int), st));
    if (!d_edge_keys) SD_TRY(cudaMalloc((void **)&keys, me * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&keys_sorted, me * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&edge_id, me * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&perm, me * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&rows_sorted, me * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&bounds_d, ((size_t)num_slices + 1) * sizeof(int)));
    if (m > 0) {
        // slice of every edge: source id / width, or handed in by the caller (dist.cu: stage of the source's owner)
        const int *sort_keys = d_edge_keys ? d_edge_keys : keys;
        if (d_edge_keys)
            iota_kernel<<<blocks(m), 256, 0, st>>>(edge_id, m);
        else
            slice_key_kernel<<<blocks(m), 256, 0, st>>>(d_idx, m, num_slices, width, keys, edge_id);
        SD_TRY(cub::DeviceRadixSort::SortPairs(nullptr, need, sort_keys, keys_sorted, edge_id, perm, m, 0, end_bit, st));
        SD_TRY(cudaMalloc(&tmp, need ? need : 1));
        SD_TRY(cub::DeviceRadixSort::SortPairs(tmp, need, sort_keys, keys_sorted, edge_id, perm, m, 0, end_bit, st));  // stable
        ptr_from_sorted_kernel<<<blocks((int64_t)m + 1), 256, 0, st>>>(keys_sorted, m, num_slices, bounds_d);
        edge_rows_kernel<<<blocks(m), 256, 0, st>>>(d_ptr, d_item_row, num_items, n, perm, m, rows_sorted);
        SD_TRY(cudaMemcpyAsync(bounds, bounds_d, ((size_t)num_slices + 1) * sizeof(int), cudaMemcpyDeviceToHost, st));
        SD_TRY(cudaStreamSynchronize(st));
    }
    {
        int off = 0;
        for (int c = 0; c < num_slices; ++c) {
            const int cnt = bounds[c + 1] - bounds[c];
            edge_off[c] = off;
            edge_cnt[c] = cnt;
            int *ptr_c = *sl_ptr + (size_t)c * ((size_t)n + 1);
            if (cnt > 0) {
                ptr_from_sorted_kernel<<<blocks((int64_t)cnt + 1), 256, 0, st>>>(rows_sorted + bounds[c], cnt, n, ptr_c);
                gather_idx_kernel<<<blocks(cnt), 256, 0, st>>>(d_idx, perm + bounds[c], *sl_idx + off, cnt);
                SD_TRY(cudaMemcpyAsync(*sl_perm + off, perm + bounds[c], (size_t)cnt * sizeof(int), cudaMemcpyDeviceToDevice, st));
            } else {
                SD_TRY(cudaMemsetAsync(ptr_c, 0, ((size_t)n + 1) * sizeof(int), st));
            }
            off += (cnt + 3) & ~3;
        }
    }
    SD_TRY(cudaGetLastError());
    SD_TRY(cudaStreamSynchronize(st));
    cudaFree(keys), cudaFree(keys_sorted), cudaFree(edge_id), cudaFree(perm), cudaFree(rows_sorted), cudaFree(bounds_d), cudaFree(tmp);
    return GNNAGG_OK;
fail:
    cudaFree(keys), cudaFree(keys_sorted), cudaFree(edge_id), cudaFree(perm), cudaFree(rows_sorted), cudaFree(bounds_d), cudaFree(tmp);
    cudaFree(*sl_ptr), cudaFree(*sl_idx), cudaFree(*sl_perm);
    *sl_ptr = *sl_idx = *sl_perm = nullptr;
    return GNNAGG_ERR_CUDA;
}


// ---------------------------------------------------------------------------------------------------------
// Compaction of a sub-CSR to its non-empty rows (locality slices of the device-resident path, capi.cu): a source
// slice of a low-degree graph leaves most rows without an edge, and walking them costs more than the slice's
// edges.  Outputs (cudaMalloc'ed, owned by the caller): *c_row [*n_out] the rows that have edges, ascending, and
// *c_ptr [*n_out + 1] their row pointers -- the (ptr, target) pair of a schedule whose groups are whole rows
// (graph_schedule.h:54-57 emits exactly these (slice, row) groups), so every output row occurs at most once.
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) row_flag_kernel(const int *__restrict__ ptr, int n, char *__restrict__ flag)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n) flag[r] = ptr[r + 1] > ptr[r];
}

__global__ void __launch_bounds__(256) compact_ptr_kernel(const int *__restrict__ ptr, const int *__restrict__ rows, int count, int n,
                                                          int *__restrict__ out)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) out[i] = ptr[rows[i]];
    if (i == count) out[count] = ptr[n];
}

int compact_rows_device(const int *d_ptr, int n, int **c_ptr, int **c_row, int *n_out, cudaStream_t st)
{
    *c_ptr = *c_row = nullptr;
    *n_out = 0;
    char *flag = nullptr;
    int *count_d = nullptr, *ids = nullptr;
    void *tmp = nullptr;
    size_t need = 0;
    int count = 0;
    SD_TRY(cudaMalloc((void **)&flag, (size_t)(n > 0 ? n : 1)));
    SD_TRY(cudaMalloc((void **)&ids, (size_t)(n > 0 ? n : 1) * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&count_d, sizeof(int)));
    SD_TRY(cudaMalloc((void **)c_row, (size_t)(n > 0 ? n : 1) * sizeof(int)));
    if (n > 0) {
        row_flag_kernel<<<blocks(n), 256, 0, st>>>(d_ptr, n, flag);
        iota_kernel<<<blocks(n), 256, 0, st>>>(ids, n);
        SD_TRY(cub::DeviceSelect::Flagged(nullptr, need, ids, flag, *c_row, count_d, n, st));
        SD_TRY(cudaMalloc(&tmp, need ? need : 1));
        SD_TRY(cub::DeviceSelect::Flagged(tmp, need, ids, flag, *c_row, count_d, n, st));
        SD_TRY(cudaMemcpyAsync(&count, count_d, sizeof(int), cudaMemcpyDeviceToHost, st));
        SD_TRY(cudaStreamSynchronize(st));
    }
    SD_TRY(cudaMalloc((void **)c_ptr, ((size_t)count + 1) * sizeof(int)));
    compact_ptr_kernel<<<blocks((int64_t)count + 1), 256, 0, st>>>(d_ptr, *c_row, count, n, *c_ptr);
    SD_TRY(cudaGetLastError());
    SD_TRY(cudaStreamSynchronize(st));
    *n_out = count;
    cudaFree(flag), cudaFree(count_d), cudaFree(ids), cudaFree(tmp);
    return GNNAGG_OK;
fail:
    cudaFree(flag), cudaFree(count_d), cudaFree(ids), cudaFree(tmp);
    cudaFree(*c_ptr), cudaFree(*c_row);
    *c_ptr = *c_row = nullptr;
    return GNNAGG_ERR_CUDA;
}


// ---------------------------------------------------------------------------------------------------------
// Merged view of a CSR (capi.cu: merged_view): every run of ADJACENT equal sources inside a row becomes one entry,
// so the aggregation gathers each (row, source) pair once.  No sort, no reordering: a CSR sorted within its rows
// merges every duplicate, an unsorted one the adjacent ones only.  The structure depends on ptr / idx alone; the
// values are summed per run by merge_val_kernel whenever the edge values change.  Outputs (cudaMalloc'ed, owned by
// the caller):
//   *mg_ptr   [n+1]  merged row pointers, mg_ptr[r] = merged position of ptr[r]
//   *mg_idx   [m']   the source of every run
//   *mg_start [m'+1] CSR edge id of the first edge of every run; mg_start[m'] = m
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) run_head_kernel(const int *__restrict__ idx, int m, int *__restrict__ head)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < m) head[e] = (e == 0 || __ldg(idx + e) != __ldg(idx + e - 1)) ? 1 : 0;
    if (e == m) head[m] = 0;  // the exclusive scan then ends in the run count
}

// the first edge of every non-empty row starts a run (runs never cross a row boundary); after run_head_kernel
__global__ void __launch_bounds__(256) row_head_kernel(const int *__restrict__ ptr, int n, int *__restrict__ head)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n && ptr[r] < ptr[r + 1]) head[ptr[r]] = 1;
}

__global__ void __launch_bounds__(256) run_compact_kernel(const int *__restrict__ idx, const int *__restrict__ head,
                                                          const int *__restrict__ pos, int m, int *__restrict__ mg_idx,
                                                          int *__restrict__ mg_start)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < m && head[e]) {
        mg_idx[pos[e]] = __ldg(idx + e);
        mg_start[pos[e]] = e;
    }
    if (e == m) mg_start[pos[m]] = m;
}

__global__ void __launch_bounds__(256) merged_ptr_kernel(const int *__restrict__ ptr, const int *__restrict__ pos, int n,
                                                         int *__restrict__ mg_ptr)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r <= n) mg_ptr[r] = pos[ptr[r]];
}

// m' without building anything: adjacent source changes, plus the first edge, plus the row starts whose source equals
// the previous edge's (a run never crosses a row boundary).  Integer counts: the atomics are exact.
__global__ void __launch_bounds__(256) count_changes_kernel(const int *__restrict__ idx, int m, int *__restrict__ count)
{
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    const int c = (e < m && (e == 0 || __ldg(idx + e) != __ldg(idx + e - 1))) ? 1 : 0;
    const int s = __syncthreads_count(c);
    if (threadIdx.x == 0 && s) atomicAdd(count, s);
}

__global__ void __launch_bounds__(256) count_row_splits_kernel(const int *__restrict__ ptr, const int *__restrict__ idx, int n,
                                                               int *__restrict__ count)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int c = 0;
    if (r < n) {
        const int e = ptr[r];
        c = (e > 0 && e < ptr[r + 1] && __ldg(idx + e) == __ldg(idx + e - 1)) ? 1 : 0;
    }
    const int s = __syncthreads_count(c);
    if (threadIdx.x == 0 && s) atomicAdd(count, s);
}

int merge_count_device(const int *d_ptr, const int *d_idx, int n, int m, int *merged_edges, cudaStream_t st)
{
    *merged_edges = 0;
    int *count = nullptr;
    SD_TRY(cudaMalloc((void **)&count, sizeof(int)));
    SD_TRY(cudaMemsetAsync(count, 0, sizeof(int), st));
    if (m > 0) count_changes_kernel<<<blocks(m), 256, 0, st>>>(d_idx, m, count);
    if (n > 0 && m > 0) count_row_splits_kernel<<<blocks(n), 256, 0, st>>>(d_ptr, d_idx, n, count);
    SD_TRY(cudaGetLastError());
    SD_TRY(cudaMemcpyAsync(merged_edges, count, sizeof(int), cudaMemcpyDeviceToHost, st));
    SD_TRY(cudaStreamSynchronize(st));
    cudaFree(count);
    return GNNAGG_OK;
fail:
    cudaFree(count);
    return GNNAGG_ERR_CUDA;
}

int merge_build_device(const int *d_ptr, const int *d_idx, int n, int m, int **mg_ptr, int **mg_idx, int **mg_start,
                       int *merged_edges, cudaStream_t st)
{
    *mg_ptr = *mg_idx = *mg_start = nullptr;
    *merged_edges = 0;
    int *head = nullptr, *pos = nullptr;
    void *tmp = nullptr;
    size_t need = 0;
    int mm = 0;
    SD_TRY(cudaMalloc((void **)&head, ((size_t)m + 1) * sizeof(int)));
    SD_TRY(cudaMalloc((void **)&pos, ((size_t)m + 1) * sizeof(int)));
    run_head_kernel<<<blocks((int64_t)m + 1), 256, 0, st>>>(d_idx, m, head);
    if (n > 0) row_head_kernel<<<blocks(n), 256, 0, st>>>(d_ptr, n, head);
    SD_TRY(cub::DeviceScan::ExclusiveSum(nullptr, need, head, pos, m + 1, st));
    SD_TRY(cudaMalloc(&tmp, need ? need : 1));
    SD_TRY(cub::DeviceScan::ExclusiveSum(tmp, need, head, pos, m + 1, st));
    SD_TRY(cudaMemcpyAsync(&mm, pos + m, sizeof(int), cudaMemcpyDeviceToHost, st));
    SD_TRY(cudaStreamSynchronize(st));
    SD_TRY(cudaMalloc((void **)mg_ptr, ((size_t)n + 1) * sizeof(int)));
    SD_TRY(cudaMalloc((void **)mg_idx, (size_t)(mm > 0 ? mm : 1) * sizeof(int)));
    SD_TRY(cudaMalloc((void **)mg_start, ((size_t)mm + 1) * sizeof(int)));
    run_compact_kernel<<<blocks((int64_t)m + 1), 256, 0, st>>>(d_idx, head, pos, m, *mg_idx, *mg_start);
    merged_ptr_kernel<<<blocks((int64_t)n + 1), 256, 0, st>>>(d_ptr, pos, n, *mg_ptr);
    SD_TRY(cudaGetLastError());
    SD_TRY(cudaStreamSynchronize(st));
    *merged_edges = mm;
    cudaFree(head), cudaFree(pos), cudaFree(tmp);
    return GNNAGG_OK;
fail:
    cudaFree(head), cudaFree(pos), cudaFree(tmp);
    cudaFree(*mg_ptr), cudaFree(*mg_idx), cudaFree(*mg_start);
    *mg_ptr = *mg_idx = *mg_start = nullptr;
    return GNNAGG_ERR_CUDA;
}

}  // namespace gnnagg
