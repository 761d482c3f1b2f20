// internal.h -- private declarations shared by the translation units of libgnnagg.so
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

struct gnnagg_schedule {
    int kind = 3;
    bool has_val = false;
    std::vector<int> ptr, idx, target;
    std::vector<float> val;
};

namespace gnnagg {

// records a thread-local message and returns `code`
int set_error(int code, const char *msg);

// host schedule builder (host_prep.cpp)
int schedule_build(int kind, const int *ptr, const int *idx, const float *val, int num_v, int num_e, int par_num,
                   int neighbor_num, int total_num_v, gnnagg_schedule *s);

// schedules built on the GPU, bit-identical to schedule_build (sched_device.cu); outputs are cudaMalloc'ed
int schedule_build_device(int kind, const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                          int par_num, int ng, int total, int **s_ptr, int **s_idx, int **s_target, int **s_perm,
                          int *num_target, int *sched_edges, cudaStream_t st);

// transposed CSR (edges stably sorted by source) for the backward pass (sched_device.cu); outputs are cudaMalloc'ed
int transpose_build_device(const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                           int num_src, int **t_ptr, int **t_idx, int **t_perm, cudaStream_t st);

// the CSR split by source-id ranges into num_slices sub-CSRs over the same rows (sched_device.cu)
int source_slices_build_device(const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                               int num_slices, int width, int **sl_ptr, int **sl_idx, int **sl_perm, int *edge_off,
                               int *edge_cnt, cudaStream_t st, const int *d_edge_keys = nullptr);

// non-empty rows of a sub-CSR and their row pointers (sched_device.cu); outputs are cudaMalloc'ed
int compact_rows_device(const int *d_ptr, int n, int **c_ptr, int **c_row, int *n_out, cudaStream_t st);

// runs of adjacent equal sources inside a row merged into one entry each (sched_device.cu); outputs are cudaMalloc'ed
int merge_build_device(const int *d_ptr, const int *d_idx, int n, int m, int **mg_ptr, int **mg_idx, int **mg_start,
                       int *merged_edges, cudaStream_t st);

// m' of that merge, counted without building it (sched_device.cu)
int merge_count_device(const int *d_ptr, const int *d_idx, int n, int m, int *merged_edges, cudaStream_t st);

// item_row table of a CSR (row containing edge k*128), cudaMalloc'ed into *out (capi.cu)
int build_item_rows_device(const int *d_ptr, int rows, int edges, int **out, int *items, cudaStream_t st);

// sub-graph samplers of include/sample.h (sample_device.cu); outputs are cudaMalloc'ed
int sample_subgraph_device(const int *d_ptr, const int *d_idx, const int *d_item_row, int num_items, int n, int m,
                           int *d_active, int fanout, int layer_num, uint64_t seed, int **vertexset, int **sub_ptr,
                           int **sub_idx, int *num_v, int *num_e, cudaStream_t st);

// dense combination on tcgen05 (dense_tc.cu); stream is a cudaStream_t
int dense_nn_launch(const float *A, const float *B, float *C, int64_t M, int N, int K, void *stream);
// loads the combination kernels and their per-device state ahead of the first launch (dense_tc.cu)
void dense_preload();

}  // namespace gnnagg
