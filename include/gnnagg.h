/*
 * gnnagg.h -- C ABI of the B200-native neighbour-aggregation library (libgnnagg.so).
 *
 * Drop-in boundary for the aggregation hot path of xxcclong/GNN-Computing.  Every entry point
 * names the reference interface it replaces (paths relative to the reference tree).  The
 * existing flat boundary of the reference is Figure7/kernel_generated.cu:15-74
 * (GCN_init_impl / GCN_run_impl / GCN_schedule_impl / GAT_*_impl: plain device pointers, ints
 * and an int64 handle); this header keeps that shape and adds what the C++ aggregator classes
 * (include/aggregator.h, aggr_gcn.h, aggr_gat.h, aggr_sddmm.h) expose beyond it.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes only.  Return value: 0 = ok, <0 = error;
 *     gnnagg_last_error() returns a thread-local message.  Nothing aborts the process (the
 *     reference calls exit(1) + cudaDeviceReset(), include/util.h:82-104; the C++ shim headers
 *     in include/ reproduce that on top of this ABI).
 *   - CSR row = destination vertex, idx = source ids, int32 indices, fp32 values, dense
 *     matrices row-major [rows, feat]; feat must be a multiple of 4 (the reference requires a
 *     multiple of 32, aggr_gcn.h:386) and at most 1024.
 *   - All `d_*`/device arguments are DEVICE pointers on the current device and are BORROWED:
 *     the library frees only what it allocated (the reference aggregator cudaFree()s its
 *     inputs, aggregator.h:58-66; the shim emulates that where a driver relies on it).
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream, which is what
 *     every reference launch uses).  Calls are asynchronous unless stated otherwise.
 *   - There is no CPU fallback: device entry points fail with GNNAGG_ERR_CUDA when no GPU is
 *     present.  Host entry points (schedules, reorder, loader) never touch the GPU.
 */
#ifndef GNNAGG_H
#define GNNAGG_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GNNAGG_OK 0
#define GNNAGG_ERR_ARG (-1)   /* bad argument (NULL, feat not supported, schedule missing ...) */
#define GNNAGG_ERR_CUDA (-2)  /* a CUDA runtime call or launch failed */
#define GNNAGG_ERR_IO (-3)    /* file missing / malformed */
#define GNNAGG_ERR_STATE (-4) /* call order (e.g. scheduled run before schedule) */

/* enum Schedule of include/graph_schedule.h:8-14, same numeric values */
#define GNNAGG_SCHED_LOCALITY 0
#define GNNAGG_SCHED_NEIGHBOR_GROUPING 1
#define GNNAGG_SCHED_LOCALITY_NEIGHBOR_GROUPING 2
#define GNNAGG_SCHED_NOP 3

typedef struct gnnagg_aggregator gnnagg_aggregator; /* opaque; replaces `Aggregator*` cast to int64 */
typedef struct gnnagg_schedule gnnagg_schedule;     /* opaque host-side schedule result */

int gnnagg_version(void);
const char *gnnagg_last_error(void);
/* number of SMs / device name of the current device; GNNAGG_ERR_CUDA without a GPU */
int gnnagg_device_info(int *sm_count, int *cc_major, int *cc_minor, char *name, int name_len);

/* ------------------------------------------------------------------------------------------
 * Host preprocessing -- bit-exact with the reference, no GPU involved
 * ------------------------------------------------------------------------------------------ */

/* Builds one of the three schedules on host arrays.
 *   kind GNNAGG_SCHED_NEIGHBOR_GROUPING           replaces neighbor_grouping_schedule  (graph_schedule.h:91-154)
 *   kind GNNAGG_SCHED_LOCALITY                    replaces locality_schedule            (graph_schedule.h:17-89)
 *   kind GNNAGG_SCHED_LOCALITY_NEIGHBOR_GROUPING  replaces localityNeighborGrouping     (graph_schedule.h:156-243)
 * val may be NULL (then no val vector is produced; neighbor grouping never produces one).
 * total_num_v is the source-id range the locality slices divide (the reference passes the
 * global `n`, aggregator.h:79,87). */
int gnnagg_schedule_build(int kind, const int *ptr, const int *idx, const float *val, int num_v, int num_e,
                          int par_num, int neighbor_num, int total_num_v, gnnagg_schedule **out);
int64_t gnnagg_schedule_num_target(const gnnagg_schedule *s); /* == target_vec.size(), aggregator.h:94 */
int64_t gnnagg_schedule_num_edges(const gnnagg_schedule *s);  /* == idx_vec.size() */
const int *gnnagg_schedule_ptr(const gnnagg_schedule *s);     /* num_target+1 entries */
const int *gnnagg_schedule_idx(const gnnagg_schedule *s);
const int *gnnagg_schedule_target(const gnnagg_schedule *s);
const float *gnnagg_schedule_val(const gnnagg_schedule *s);   /* NULL when no val vector */
void gnnagg_schedule_free(gnnagg_schedule *s);

/* replaces reorderCSR (src/data.cu:4-29): map[i] = old id placed at new position i,
 * reverse_map[old] = new; newptr[num_v+1] and newidx[num_e] are caller-allocated. */
int gnnagg_reorder_csr(const int *ptr, const int *idx, const int *map, const int *reverse_map, int num_v, int num_e,
                       int *newptr, int *newidx);

/* replaces load_graph (src/data.cu:31-139), split in the two steps a C caller needs:
 *   gnnagg_graph_config : reads "<datadir><dset>.config"                       (:38-44)
 *   gnnagg_graph_load   : fills indptr[num_v+1] / indices[num_e] from the .ptrdump/.edgedump
 *                         caches or the text .graph (writing the caches)       (:46-93);
 *                         if reorder_path is non-NULL/non-empty and exists the permutation is
 *                         read into rows/reverse_rows (caller-allocated, num_v each) and
 *                         applied (:96-133); *reordered tells whether that happened.
 * datadir must end with '/' (the reference hard-codes "../data/", :34). */
int gnnagg_graph_config(const char *datadir, const char *dset, int *num_v, int *num_e);
int gnnagg_graph_load(const char *datadir, const char *dset, const char *reorder_path, int num_v, int num_e,
                      int *indptr, int *indices, int *rows, int *reverse_rows, int *reordered);
/* writes <datadir><dset>.config and .graph in the reference's text format (test/bench helper,
 * the reference only reads these files: README.md:45-54) */
int gnnagg_graph_write(const char *datadir, const char *dset, int num_v, int num_e, const int *indptr,
                       const int *indices);

/* locality-aware reordering: deterministic re-statement of script/cluster2.py (MinHash-LSH
 * candidates -> exact Jaccard -> greedy size-capped union-find clustering).  Writes the
 * permutation rows[num_v] (entry k = old id placed at new position k) -- the content of a
 * <dset>.reorder<suffix> file.  num_perm/bands/rows_per_band/cap: cluster2.py uses 64 perms,
 * threshold 0.2 (-> b=28,r=2 in datasketch) and cap 64; pass 0 for these defaults. */
int gnnagg_lsh_reorder(const int *ptr, const int *idx, int num_v, int num_e, int num_perm, int bands,
                       int rows_per_band, int cluster_cap, uint64_t seed, int *rows);
int gnnagg_reorder_write(const char *path, const int *rows, int num_v); /* cluster2.py:168-171 format */

/* ------------------------------------------------------------------------------------------
 * Aggregator object -- replaces class Aggregator and its subclasses
 * ------------------------------------------------------------------------------------------ */

/* replaces Aggregator::Aggregator (aggregator.h:28-57) / GCN_init_impl, GAT_init_impl
 * (kernel_generated.cu:15-19,41-45).  h_ptr/h_idx may be NULL: they are then mirrored from the
 * device when a host schedule needs them (aggregator.h:30-39). */
int gnnagg_create(const int *d_ptr, const int *d_idx, const int *h_ptr, const int *h_idx, int num_v, int num_e,
                  gnnagg_aggregator **out);
/* same, with the set-up kernel (a row lookup table) issued on `stream` instead of the legacy stream: use it when
 * d_ptr / d_idx are still being produced on that stream, or when runs follow on a non-blocking stream.
 * gnnagg_create itself returns with the set-up complete. */
int gnnagg_create_on(const int *d_ptr, const int *d_idx, const int *h_ptr, const int *h_idx, int num_v, int num_e,
                     gnnagg_aggregator **out, void *stream);
int gnnagg_destroy(gnnagg_aggregator *a);

/* edge values of the GCN aggregator: ctor argument of Aggregator_GCN (aggr_gcn.h:365-374) and
 * Aggregator_GCN::updateval (aggr_gcn.h:540-544) / GCN_update_val_impl.  Borrowed. */
int gnnagg_set_val(gnnagg_aggregator *a, const float *d_val);
/* same on `stream` (after a locality schedule the values are permuted by a kernel: gnnagg_set_val waits for it,
 * this variant orders it on the caller's stream) */
int gnnagg_set_val_on(gnnagg_aggregator *a, const float *d_val, void *stream);

/* replaces Aggregator::schedule / Aggregator_GCN::schedule (aggregator.h:67-99,
 * aggr_gcn.h:501-538) / GCN_schedule_impl, GAT_schedule_impl.  params[0] = par_num or
 * neighbor_num, params[1] = neighbor_num for the combined schedule.  Builds on the host with
 * gnnagg_schedule_build and uploads; for the locality kinds the current val (if set) is
 * permuted alongside as in aggr_gcn.h:522-537. */
int gnnagg_schedule_apply(gnnagg_aggregator *a, int kind, const int *params, int nparams, int total_num_v);
int gnnagg_num_target(const gnnagg_aggregator *a); /* public field Aggregator::num_target */
int gnnagg_schedule_kind(const gnnagg_aggregator *a); /* GNNAGG_SCHED_* of the schedule in force (NOP before any) */
/* per-edge data from SCHEDULED edge order (what the scheduled GAT run leaves in gnnagg_gat_edge_weights, like
 * aggr_gat_fine's newval, aggr_gat.h:192) back to CSR order, the order gnnagg_gat_backward indexes `w` in.  The two
 * orders coincide for `nop` and `neighbor_grouping` (then this is a copy); after a locality schedule they do not. */
int gnnagg_sched_to_csr_order(gnnagg_aggregator *a, const float *in_sched, float *out_csr, void *stream);
/* device views of the uploaded schedule (d_ptr_scheduled, d_idx_scheduled, d_target_scheduled,
 * d_val_scheduled of aggregator.h:132-134 / aggr_gcn.h:549); NULL before a schedule */
const int *gnnagg_sched_dev_ptr(const gnnagg_aggregator *a);
const int *gnnagg_sched_dev_idx(const gnnagg_aggregator *a);
const int *gnnagg_sched_dev_target(const gnnagg_aggregator *a);
const float *gnnagg_sched_dev_val(const gnnagg_aggregator *a);

/* Optional: builds, now, the per-graph tables the FIRST un-scheduled run for this feature width would otherwise build
 * (which rows cross item boundaries; one host synchronisation).  After it, runs of that width never synchronise the
 * host: required before CUDA-graph capture, and used by the multi-GPU path, where a host wait in the middle of a step
 * could deadlock a process that drives several ranks. */
int gnnagg_prepare(gnnagg_aggregator *a, int feat, void *stream);

/* GCN aggregation Y = A*X.  replaces Aggregator_GCN::run / run_with_feat (aggr_gcn.h:379-444)
 * / GCN_run_impl and the kernels aggr_gcn (:5-36) [scheduled=0] and aggr_gcn_target (:78-114)
 * [scheduled=1].  Y is fully overwritten in both modes (the reference memsets, :393). */
int gnnagg_gcn_run(gnnagg_aggregator *a, const float *X, float *Y, int feat, int scheduled, void *stream);

/* Y += A*X (accumulate != 0) or Y = A*X on the un-scheduled CSR.  Building block of the multi-GPU
 * pipeline: a rank's row block is split by SOURCE shard (the slices of locality_schedule,
 * graph_schedule.h:24-29) and every slice is accumulated as soon as its shard of X has arrived.  With
 * accumulate = 0 it is gnnagg_gcn_run(scheduled = 0).  Deterministic (no atomics). */
int gnnagg_gcn_run_acc(gnnagg_aggregator *a, const float *X, float *Y, int feat, int accumulate, void *stream);

/* the same for the destination rows [row_lo, row_hi) only (Y is still indexed by global row): lets a caller
 * pipeline the aggregation of one row chunk with the copy-out / combination of the previous one.  Cuts the edge
 * range on a host mirror of the row pointers (copied once; gnnagg_prepare does it ahead of time). */
int gnnagg_gcn_run_rows(gnnagg_aggregator *a, const float *X, float *Y, int feat, int accumulate, int row_lo, int row_hi,
                        void *stream);

/* out[i,:] = X[rows[i],:] for i < count (feat a multiple of 4).  Packs the rows of the local X shard that
 * another rank's row block references before the pruned halo exchange (multi-GPU path, new functionality:
 * the reference is single-GPU). */
int gnnagg_gather_rows(const float *X, const int64_t *rows, float *out, int64_t count, int feat, void *stream);

/* edge-parallel variant: replaces Aggregator_GCN::runEdgeWise + aggr_gcn_edgewise
 * (aggr_gcn.h:291-302,445-460) and Aggregator::csr2edgelist (aggregator.h:115-122).
 * Any feat (the reference is F=32 only). */
int gnnagg_gcn_run_edgewise(gnnagg_aggregator *a, const float *X, float *Y, int feat, void *stream);
int gnnagg_csr2edgelist(gnnagg_aggregator *a, int *d_edgelist /* 2*num_e */, void *stream);

/* fused aggregation + combination  AX = A*X ; H = AX*W,  W row-major [feat_in, feat_out].
 * replaces Aggregator_GCN::run_with_nn + aggr_gcn_nn (aggr_gcn.h:304-359,491-499) and the
 * un-fused aggr_gcn_target + matmul_NN baseline (dense.h:4-23, Figure10/main_b.cu:89-90).
 * AX may be NULL (not materialised for the caller).  Outputs are overwritten (the reference
 * accumulates into never-zeroed buffers, SURVEY 4).  feat_in, feat_out multiples of 32 up to 256 run on the tensor
 * cores; any other size goes through a plain fp32 kernel (matmul_NN takes any size, dense.h:4-23).
 * The combination runs on tcgen05 tensor cores in 3xTF32 (fp32-level accuracy). */
int gnnagg_gcn_layer(gnnagg_aggregator *a, const float *X, const float *W, float *H, float *AX, int feat_in,
                     int feat_out, int scheduled, void *stream);
/* the dense combination alone: C[M,N] = A[M,K]*B[K,N] row-major; replaces matmul_NN (dense.h:4-23) */
int gnnagg_dense_nn(const float *A, const float *B, float *C, int64_t M, int N, int K, void *stream);

/* fused GAT aggregation  Y[v] = sum_u w X[u] / sum_u w,  w = exp(max(s, slope*s)),
 * s = att[2v] + att[2u+1].  replaces Aggregator_GAT::run / run_with_feat (aggr_gat.h:317-394)
 * / GAT_run_impl and the kernels aggr_gat (:116-164) [scheduled=0] and aggr_gat_fine +
 * scaleArray (:167-213) [scheduled=1; additionally leaves the un-normalised w in the
 * aggregator's edge buffer, gnnagg_gat_edge_weights()].  Empty rows yield 0 (reference: NaN /
 * untouched, documented deviation).  slope: the reference hard-codes 0.2 (:339,347). */
int gnnagg_gat_run(gnnagg_aggregator *a, const float *X, const float *att, float *Y, int feat, float slope,
                   int scheduled, void *stream);
const float *gnnagg_gat_edge_weights(const gnnagg_aggregator *a); /* d_newval of aggr_gat.h:306, scheduled order */

/* un-fused GAT pieces on the un-scheduled CSR:
 *   gnnagg_edge_softmax   replaces run_att + attGat                (aggr_gat.h:5-31,395-401)
 *   gnnagg_u_add_v        replaces run_u_add_v + u_add_v           (aggr_gat.h:33-48,402-409)
 *   gnnagg_add_to_center  replaces run_add_to_center               (aggr_gat.h:50-74,410-417; out[v], stride 1)
 *   gnnagg_each_div       replaces run_div_each + each_div         (aggr_gat.h:76-92,418-425) */
int gnnagg_edge_softmax(gnnagg_aggregator *a, const float *att, float *out_val, float slope, void *stream);
int gnnagg_u_add_v(gnnagg_aggregator *a, const float *att, float *out_val, void *stream);
int gnnagg_add_to_center(gnnagg_aggregator *a, const float *in_val, float *out_center, void *stream);
int gnnagg_each_div(gnnagg_aggregator *a, const float *in_center, float *inout_val, void *stream);

/* per-edge MLP aggregation  Y[v,:] = sum_{u in N(v)} ReLU((X[v,:] + X[u,:]) * W),  W row-major [feat, feat].
 * replaces Aggregator_MLP::run + aggr_mlp / aggr_mlp_target (include/aggr_nn.h:51-341; there feat = 32 only and
 * a 32x32 mat-vec per EDGE).  Here the projection is hoisted out of the edge loop: (x_v + x_u) W = P[v] + P[u]
 * with P = X W computed once on the tensor cores (gnnagg_dense_nn), so an edge costs one gathered row and
 * `feat` adds.  feat a multiple of 32 <= 256; scheduled = 1 uses the current schedule (RED combination). */
int gnnagg_mlp_run(gnnagg_aggregator *a, const float *X, const float *W, float *Y, int feat, int scheduled,
                   void *stream);

/* SDDMM  val[e] = <X1[idx[e],:], X2[row(e),:]>.  replaces Aggregator_SDDMM::run + aggr_sddmm /
 * aggr_sddmm_target (aggr_sddmm.h:5-117); scheduled=1 requires a neighbor-grouping schedule
 * (:100) and writes in scheduled edge order (identical to CSR order for that schedule).
 * Any feat multiple of 4 (the reference is F=32 only, :21). */
int gnnagg_sddmm(gnnagg_aggregator *a, const float *X1, const float *X2, float *out_val, int feat, int scheduled,
                 void *stream);

/* ---- backward of the aggregation (SURVEY §8(f) rank 3) ---------------------------------------------------
 * The reference has one experimental backward kernel, aggr_gat_fine_bwd behind Aggregator_GAT::run_bwd
 * (include/aggr_gat.h:222-294, :426-434): float atomics into d_feat (:264), F = 32 only (:245), LeakyReLU
 * derivative keyed on `newval < 0` (never true, :289), source half of the attention gradient only (:290).
 * These entry points compute the full, deterministic derivative of gnnagg_gcn_run / gnnagg_gat_run instead.
 *
 * gnnagg_transpose_build  once per graph: the CSR transposed ON THE GPU (edges stably sorted by source;
 *                         num_src = number of source rows, = num_v for a square graph), kept in the handle.
 * gnnagg_transpose_dev    device views of it: t_ptr[num_src+1], t_idx[m] = destination rows,
 *                         t_perm[m] = CSR edge id at every transposed position.
 * gnnagg_gcn_backward     dX[u,:] = sum over edges (v <- u) of val_e dY[v,:]   (= A^T dY), dX is [num_src, feat].
 * gnnagg_gat_backward     for Y = gnnagg_gat_run(X, att) and dL/dY = dY:
 *                           alpha_e = w_e / D_v, ds_e = alpha_e (<X[u],dY[v]> - <Y[v],dY[v]>) * (s_e > 0 ? 1 : slope)
 *                           dX[u,:] = sum_e alpha_e dY[v,:]            (:264)
 *                           datt[2v] = sum_e ds_e,  datt[2u+1] = sum_e ds_e   (:287-290; att/datt have max(num_v,num_src) rows)
 *                         Either `att` is given (w, den may be NULL: weights are recomputed), or w[m] (un-normalised
 *                         weights in CSR order, what aggr_gat_fine leaves in newval, :193) -- then att may be NULL and
 *                         the sign of s_e is read from w_e > 1.  den[num_v] (`div` of run_bwd) is optional: when NULL
 *                         the row sums D_v are formed on the way (they cost nothing extra), when given it is used as is.
 *                         Outputs are overwritten (the reference accumulates into caller-zeroed arrays). */
int gnnagg_transpose_build(gnnagg_aggregator *a, int num_src, void *stream);
int gnnagg_transpose_dev(const gnnagg_aggregator *a, int *num_src, const int **t_ptr, const int **t_idx, const int **t_perm);
int gnnagg_gcn_backward(gnnagg_aggregator *a, const float *dY, float *dX, int feat, void *stream);
int gnnagg_gat_backward(gnnagg_aggregator *a, const float *X, const float *att, const float *w, const float *den,
                        const float *Y, const float *dY, float *dX, float *datt, int feat, float slope, void *stream);

/* ---- GCN aggregation from bf16 features ------------------------------------------------------------------
 * The same operations as gnnagg_gcn_run, gnnagg_gcn_layer and gnnagg_gcn_backward with the GATHERED operand (X, or dY
 * of the backward) stored in bf16: X / dY are bf16 bit patterns, 8-byte aligned, [rows, feat] row-major.  Edge values,
 * accumulation and every output (Y, H, AX, dX) stay fp32, outputs 16-byte aligned; feat is a multiple of 4 in
 * [4, 1024] as for fp32.  Each bf16 value is widened exactly to fp32 on load and then summed as in the fp32 run, so
 * the result equals the fp32 entry point run on the widened X, bit for bit for un-scheduled runs (CSR, merged view,
 * locality slices) and up to the arbitrary RED.ADD order of scheduled runs.  Routing, the settings, profiling
 * (gnnagg_profile_read) and the launch count are those of the fp32 entry point; gnnagg_prepare also readies the bf16
 * kernel.  The automatic locality-slice rule sizes X from the bytes stored (2 per element); its constants were tuned
 * on fp32 runs and are not re-tuned for bf16.  gnnagg_gcn_layer_bf16 uses the same fp32 combination as
 * gnnagg_gcn_layer on the fp32 AX. */
int gnnagg_gcn_run_bf16(gnnagg_aggregator *a, const uint16_t *X, float *Y, int feat, int scheduled, void *stream);
int gnnagg_gcn_layer_bf16(gnnagg_aggregator *a, const uint16_t *X, const float *W, float *H, float *AX, int feat_in,
                          int feat_out, int scheduled, void *stream);
int gnnagg_gcn_backward_bf16(gnnagg_aggregator *a, const uint16_t *dY, float *dX, int feat, void *stream);
/* bf16 forms of gnnagg_gcn_run_acc and gnnagg_gcn_run_rows (the stages of the multi-GPU step), same contract */
int gnnagg_gcn_run_acc_bf16(gnnagg_aggregator *a, const uint16_t *X, float *Y, int feat, int accumulate, void *stream);
int gnnagg_gcn_run_rows_bf16(gnnagg_aggregator *a, const uint16_t *X, float *Y, int feat, int accumulate, int row_lo,
                             int row_hi, void *stream);

/* ---- sub-graph samplers (SURVEY §8(f) rank 4) -------------------------------------------------------------
 * replaces sampleVertex (include/sample.h:131-200) and sampleVertexSampleNeighbor (:274-357).
 * d_active [num_v]: non-zero marks the seed vertices; on return it holds the 0/1 set after layer_num - 1 hops
 * (the reference updates its `int *&active_vertex` the same way).  The rows of the active vertices are extracted in
 * ascending vertex order: *d_vertexset [*num_v] their ids, *d_sub_ptr [*num_v + 1], *d_sub_idx [*num_e] GLOBAL source
 * ids -- the three arrays of a CSRSubGraph (util.h:15-36), cudaMalloc'ed here and owned by the caller
 * (gnnagg_device_free, or hand them to an aggregator shim that frees them as the reference's does).
 *   fanout <= 0 : complete neighbour lists; bit-identical to sampleVertex.
 *   fanout  > 0 : rows longer than fanout keep exactly fanout neighbours, the j-th drawn uniformly from the j-th of
 *                 fanout equal strata of the row as a pure function of (seed, vertex, j) -- CSR order kept, inclusion
 *                 probability fanout/deg, reproducible on CPU and GPU.  This RE-SPECIFIES sampleVertexSampleNeighbor,
 *                 whose mark test is inverted / matches nothing for rows longer than the limit (sample.h:97-104 vs
 *                 :229-246) and which no driver calls; see gnn-computing_b200/csrc/sample_device.cu. */
int gnnagg_sample_subgraph(gnnagg_aggregator *a, int *d_active, int fanout, int layer_num, uint64_t seed, int **d_vertexset,
                           int **d_sub_ptr, int **d_sub_idx, int *num_v, int *num_e, void *stream);
int gnnagg_device_free(void *d_ptr);

/* naive reference-style SpMM + validators of include/spmm.h:
 *   gnnagg_spmm_naive        replaces spmm<LENFEATURE> (spmm.h:223-265; thread per row; rows
 *                            with no edge are left untouched as there, :236-237)
 *   gnnagg_validate          replaces valid()/validate2 (spmm.h:11-21,35-69): #elements with
 *                            |(ref-ans)/ref| > 1e-2
 *   gnnagg_validate_reordered replaces validReordered()/validateReordered (spmm.h:23-33,71-91)
 * The two validators synchronise and return the count through *diffnum. */
int gnnagg_spmm_naive(int num_v, const int *d_ptr, const int *d_idx, const float *d_val, const float *X, float *Y,
                      int feat, void *stream);
int gnnagg_validate(const float *d_ref, const float *d_ans, int64_t num, int *diffnum, void *stream);
int gnnagg_validate_reordered(const float *d_ref, const float *d_ans, const int *d_map, int num_v, int feat,
                              int *diffnum, void *stream);

/* ------------------------------------------------------------------------------------------
 * Multi-GPU: 1-D row partition by destination, source-feature halo over NVLink peer memory.
 * The reference is single-GPU: every driver asserts GPUNUM == 1 (Figure9/main.cu:19); what it
 * sketched and never built are the per-GPU globals GPUNUM / gptrs / gidxs (include/util.h:39-57),
 * syncAll (include/util.h:135-142) and the prepare*Multi prototypes (include/data.h:48-58).
 * These entry points are that missing piece.  Rank r owns the destination rows
 * [shard_bounds[r], shard_bounds[r+1]) and the matching rows of X; its CSR block keeps GLOBAL
 * source ids.  A gnnagg_dist handle is ONE rank (one GPU).  Life cycle:
 *   1. create   single process : gnnagg_dist_create(world, devices, ...) -> world handles (the shape SURVEY
 *                                8(b) names; per-rank calls may come from one thread, no step call blocks the host)
 *               process per GPU: gnnagg_dist_create_rank on the current device
 *   2. gnnagg_dist_set_graph on every rank: finds the distinct remote rows the block references, builds the
 *      per-stage CSRs and allocates the rank's ONE peer-visible buffer (flags | wanted rows | 2 x [X shard +
 *      receive slots])
 *   3. connect  single process : gnnagg_dist_connect_local(handles, world)
 *               process per GPU: gnnagg_dist_export a GNNAGG_DIST_BLOB_BYTES blob, all-gather the blobs with
 *                                whatever the caller has (MPI, torch.distributed, a file), gnnagg_dist_connect
 *                                (cudaIpc mapping; every owner copies the lists of rows its peers want, once)
 *   4. steps    write the X shard into gnnagg_dist_x(d, buf) on `stream`, then gnnagg_dist_gcn_run / _gcn_layer.
 *               Two shard buffers: a layer may write the next layer's input into the other one.  A shard stored in
 *               bf16 goes through the _bf16 forms of the steps (below): half the halo bytes, fp32 outputs.
 *   5. teardown all ranks idle -> gnnagg_dist_disconnect on every rank -> (barrier) -> gnnagg_dist_destroy
 * A step: every OWNER pushes the rows each peer wants from its shard straight into that peer's receive slots with
 * 128-bit stores over NVLink (local gathers, posted remote writes, contiguous destination; owner p serves receivers
 * p-1, p-2, ... so each receiver is written by one owner at a time).  What the receiver overlaps with the pushes
 * depends on `remote_stages`:
 *    R > 0  stages by OWNER: stage 0 (edges with local sources) at once, then one accumulating stage per group of owners
 *           as it lands -- for long rows (reddit-shape: 490 edges per row), where R extra passes over Y cost little;
 *    R = 0  a single pass after all arrivals;
 *    R < 0  ROW pipelining with K = -R (<= 16) edge-balanced row chunks: receive slots are ordered by the chunk that
 *           needs a row first, the owners push round by round and chunk c -- a row range of the ONE CSR, no extra pass
 *           over Y -- starts when round c has landed.  For short rows (R-MAT: 16 edges per row).
 * Deterministic: no atomics, a fixed summation order per (world, remote_stages).  No NCCL, no pack buffer.
 * ------------------------------------------------------------------------------------------ */
#define GNNAGG_DIST_MAX_WORLD 16
#define GNNAGG_DIST_BLOB_BYTES 256
#define GNNAGG_DIST_NO_EXCHANGE 1 /* run flag: re-use the receive slots of the previous run (kernels-only timing) */
typedef struct gnnagg_dist gnnagg_dist;
int gnnagg_dist_create(int world, const int *devices /* NULL: 0..world-1 */, const int64_t *shard_bounds /* world+1 */,
                       int feat_cap, gnnagg_dist **out /* [world] */);
int gnnagg_dist_create_rank(int rank, int world, const int64_t *shard_bounds, int feat_cap, gnnagg_dist **out);
/* the rank's row block (borrowed only during the call: the library keeps its own re-indexed per-stage CSRs);
 * synchronises `stream`.  remote_stages: see above (clamped to world-1 / 16 chunks).  Once per handle; all ranks of a
 * group must use the same value. */
int gnnagg_dist_set_graph(gnnagg_dist *d, const int *d_ptr, const int *d_idx, const float *d_val, int64_t num_e,
                          int remote_stages, void *stream);
int gnnagg_dist_export(gnnagg_dist *d, void *blob /* GNNAGG_DIST_BLOB_BYTES */);
int gnnagg_dist_connect(gnnagg_dist *d, const void *blobs /* world * GNNAGG_DIST_BLOB_BYTES, indexed by rank */);
int gnnagg_dist_connect_local(gnnagg_dist **ranks, int world); /* export + connect of all ranks of one process */
int gnnagg_dist_disconnect(gnnagg_dist *d); /* unmaps the peers; the rank cannot step afterwards */
int gnnagg_dist_destroy(gnnagg_dist *d);
/* builds the per-stage tables for a feature width other than feat_cap (set_graph prepares feat_cap).  Waits for the
 * device: with one process per GPU the first run of a new width does it by itself; a process driving several ranks
 * must call it for EVERY rank before the first step of that width. */
int gnnagg_dist_prepare(gnnagg_dist *d, int feat, void *stream);
float *gnnagg_dist_x(gnnagg_dist *d, int buf); /* [rows of the shard, feat] row-major, feat <= feat_cap; NULL before set_graph */
/* Y = A_block * X  /  H = (A_block * X) * W, with X = buffer `buf` of every rank (all ranks must call with the same
 * buf and feat).  Asynchronous on `stream`. */
int gnnagg_dist_gcn_run(gnnagg_dist *d, int buf, float *Y, int feat, int flags, void *stream);
int gnnagg_dist_gcn_layer(gnnagg_dist *d, int buf, const float *W, float *H, int feat_in, int feat_out, int flags,
                          void *stream);
/* host-buffer variants (bench.py's e2e number at N > 1): X shard host -> peer-visible buffer, the step, result ->
 * host; the last stage runs row chunk by row chunk so the copy back overlaps it.  Synchronise `stream`.  Pinned host
 * memory makes the copies asynchronous.  h_W NULL: aggregation only (h_out is [rows, feat_in]). */
int gnnagg_dist_gcn_layer_host(gnnagg_dist *d, int buf, const float *h_X, const float *h_W, float *h_out, int feat_in,
                               int feat_out, void *stream);
/* the three steps with the shard stored in bf16: gnnagg_dist_x(d, buf) (or h_X) holds bf16 bit patterns, row stride
 * `feat` (a multiple of 4, at most feat_cap), so a shard takes half of the buffer and the halo pushes -- and the H2D copy
 * of the host variant -- move half the bytes.  The stages gather with gnnagg_gcn_run_acc_bf16 / _rows_bf16; edge values,
 * sums, Y, AX, the combination and H stay fp32 (as gnnagg_gcn_layer_bf16), and the result equals the fp32 step on the
 * widened X bit for bit.  Launches, gnnagg_dist_profile_read and gnnagg_dist_prepare are those of the fp32 step; the
 * push is always the default register kernel (the GNNAGG_PUSH_* experiments apply to fp32 steps only).  Every rank of a
 * step must use the same dtype, buf and feat. */
int gnnagg_dist_gcn_run_bf16(gnnagg_dist *d, int buf, float *Y, int feat, int flags, void *stream);
int gnnagg_dist_gcn_layer_bf16(gnnagg_dist *d, int buf, const float *W, float *H, int feat_in, int feat_out, int flags,
                               void *stream);
int gnnagg_dist_gcn_layer_host_bf16(gnnagg_dist *d, int buf, const uint16_t *h_X, const float *h_W, float *h_out,
                                    int feat_in, int feat_out, void *stream);
/* distinct remote source rows this rank receives per step (in total / per owner), stages and their edge counts,
 * rows this rank pushes to every peer (after connect); any pointer may be NULL */
int gnnagg_dist_info(const gnnagg_dist *d, int64_t *num_recv, int64_t *recv_counts /* [world] */, int *num_stages,
                     int64_t *stage_edges /* [num_stages] */, int64_t *send_counts /* [world] */);
/* device timing of the last run: ms[0] halo pushes of this rank (first issued .. last complete, comm stream),
 * ms[1] whole step, ms[2] stage 0, ms[3] dense combination */
int gnnagg_dist_profile_enable(gnnagg_dist *d, int on);
int gnnagg_dist_profile_read(gnnagg_dist *d, float *ms /* [4] */);
/* GNNAGG_ERR_STATE if a kernel of this rank gave up waiting for a peer (bounded spin, 20 s); synchronous */
int gnnagg_dist_check(gnnagg_dist *d);
int64_t gnnagg_dist_launch_count(const gnnagg_dist *d);

/* ------------------------------------------------------------------------------------------
 * Host-buffer entry points (what a caller holding HOST arrays uses; bench.py's e2e number).
 * They copy inputs host->device, run, copy the result back and synchronise `stream`.
 * Pinned host memory makes the copies asynchronous with respect to the host.
 * ------------------------------------------------------------------------------------------ */
int gnnagg_gcn_run_host(gnnagg_aggregator *a, const float *h_X, float *h_Y, int feat, int scheduled, void *stream);
int gnnagg_gcn_layer_host(gnnagg_aggregator *a, const float *h_X, const float *h_W, float *h_H, int feat_in,
                          int feat_out, int scheduled, void *stream);
int gnnagg_gat_run_host(gnnagg_aggregator *a, const float *h_X, const float *h_att, float *h_Y, int feat,
                        float slope, int scheduled, void *stream);

/* how the two GCN host-buffer entry points overlap copies and kernels (X must be [num_v, feat], square graph):
 *   0  automatic: graphs of >= 4M edges use 4 SOURCE slices -- X travels in 4 row blocks and the sub-CSR of the edges
 *      whose source lies in block c (built once on the GPU, the locality slices of graph_schedule.h:24-29 kept as CSRs)
 *      is accumulated as soon as block c is resident; the last slice runs in row chunks so the copy back starts one
 *      chunk after the input copy ends.  Smaller graphs: one input copy, then row chunks.
 *  >0  force that many source slices (<= 8);   <0  row chunks only.
 * Results are deterministic for a given setting; slices change the fp32 summation order (slice by slice). */
int gnnagg_set_host_pipeline(gnnagg_aggregator *a, int slices);

/* Locality slices of the device-resident, un-scheduled GCN aggregation / layer -- the idea of locality_schedule
 * (graph_schedule.h:17-89: process the edges source range by source range so that the gathered rows stay in cache)
 * without its float atomics: the CSR is split once, on the GPU, into `slices` sub-CSRs by source range and the
 * deterministic kernel accumulates them one after the other; lanes whose partial sum is zero skip the pass over Y.
 *   0  automatic (default): when X is >= 8x the L2 and the average degree is >= 20: ceil(X bytes / 2.5 L2) slices, at
 *      most 4.  The first slice covers every row (it writes the zeros of empty rows too); the others are compacted to
 *      the rows that have edges in them and ADD with 128-bit reductions (one add per element and launch: deterministic).
 *      Products-shape (25 edges per row, F=256, X = 20x L2): 4.48 ms un-sliced, 4.27 / 4.29 / 4.82 ms with 2 / 4 / 8
 *      slices -- the gain is bounded because every slice still costs a pass over the rows it touches; the reddit /
 *      proteins / arxiv shapes (X within a few L2 sizes) run un-sliced
 *   1  off;  2..16  forced.   Square graphs (sources in [0, num_v)); out-of-range sources fall into the last slice.
 * Results are deterministic for a given setting; slices change the fp32 summation order (slice by slice). */
int gnnagg_set_locality_slices(gnnagg_aggregator *a, int slices);

/* Merged view of duplicate edges for the un-scheduled, un-sliced GCN aggregation (gnnagg_gcn_run, gnnagg_gcn_run_acc,
 * gnnagg_gcn_layer, gnnagg_gcn_run_rows and the row-chunk host pipeline): every run of ADJACENT edges of a row with the
 * same source becomes one entry whose value is the run's sum (summed in fp64 in CSR order, rounded once to fp32), so
 * each (row, source) pair is gathered once.  The same matrix A; built once on the GPU from ptr / idx (no sort, no
 * reordering: rows sorted by source merge every duplicate), its values re-summed on the run's stream after
 * gnnagg_set_val.  Scheduled runs, locality and source slices, GAT, SDDMM, MLP and the backward passes keep the CSR.
 *   0  automatic (default): on when the graph has >= 4M edges and merging removes >= 10 % of them
 *   1  off (the CSR as given);  2  on.
 * Results are deterministic for a given setting; merging changes the fp32 summation order. */
int gnnagg_set_merge_duplicates(gnnagg_aggregator *a, int mode);

/* edges the GCN aggregation walks under the current setting: m' of the merged view, or num_e when it is off (builds
 * the view, or takes the automatic decision, on the legacy stream if that has not happened yet); -1 on error */
int gnnagg_merged_edges(gnnagg_aggregator *a);

/* device arrays of the merged view (row pointers [num_v+1], sources [m'], values [m']) as the last run left them;
 * GNNAGG_ERR_STATE when the view is not in use */
int gnnagg_merged_dev(const gnnagg_aggregator *a, const int **ptr, const int **idx, const float **val);

/* tuning knob (the reference's analogue is the BLOCK_SIZE argument of run(), aggr_gcn.h:381-386):
 * edges staged per warp by the aggregation kernels: 0 = automatic (128 below 4M edges, else 512),
 * or force 128 / 512.  Results do not depend on it beyond fp32 summation order. */
int gnnagg_set_warp_edges(gnnagg_aggregator *a, int warp_edges);

/* per-kernel device timing of the LAST gnnagg_gcn_run / gnnagg_gat_run / gnnagg_gcn_layer call:
 * when enabled the library brackets its launches with CUDA events on the caller's stream.
 * gnnagg_profile_read synchronises on those events and returns milliseconds in
 * ms[0] = aggregation kernel, ms[1] = split-row fix-up (or memset+scale in scheduled mode),
 * ms[2] = dense combination, ms[3] = whole call.  Used by bench.py for the roofline line
 * (the reference's analogue is run_clock / aggr_gcn_clock, aggr_gcn.h:159-248,462-489). */
int gnnagg_profile_enable(gnnagg_aggregator *a, int on);
int gnnagg_profile_read(gnnagg_aggregator *a, float *ms /* [4] */);

/* synchronous device->host copy of `bytes` bytes (binding helper: lets a ctypes/cgo caller read
 * the scheduled arrays returned by gnnagg_sched_dev_* without linking the CUDA runtime itself;
 * the reference does this with cudaMemcpy in its drivers) */
int gnnagg_memcpy_d2h(void *h_dst, const void *d_src, uint64_t bytes);

/* number of kernels the library launched on behalf of this aggregator since creation
 * (bench.py's gpu_launches claim) */
int64_t gnnagg_launch_count(const gnnagg_aggregator *a);

#ifdef __cplusplus
}
#endif
#endif /* GNNAGG_H */
