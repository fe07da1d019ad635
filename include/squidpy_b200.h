/*
 * squidpy_b200.h — C ABI of libsquidpy_b200.so: B200 (sm_100a) kernels for squidpy's spatial-statistics hot
 * path.  Plain pointers and sizes only (no torch / numpy types).  All array arguments are HOST pointers owned
 * by the caller unless a parameter is documented as a device pointer; the library never frees caller memory.
 *
 * Conventions
 *   - every function returns 0 (SQB_OK) or a negative sqb_status; sqb_last_error() returns a thread-local
 *     human-readable message for the last failure on the calling thread;
 *   - a sqb_ctx binds one CUDA device and one stream (caller-supplied cudaStream_t, or library-owned);
 *     object handles (sqb_nhood, sqb_autocorr) belong to the ctx they were created on; handles are not
 *     thread-safe, distinct ctx/handles may be used concurrently (one per GPU);
 *   - calls are synchronous with respect to the host unless the name ends in _async.
 *
 * Each entry point replaces one internal seam of the reference (paths relative to the squidpy tree):
 *   sqb_nhood_count            <- _test(indices, indptr, clustering)          src/squidpy/gr/_nhood.py:60-61,208-209
 *   sqb_nhood_permute*         <- _nhood_enrichment_helper(...)               src/squidpy/gr/_nhood.py:516-547
 *                                 (+ rng.shuffle / _shuffle_group             src/squidpy/gr/_utils.py:185-213,
 *                                    spawn_generators                         src/squidpy/_utils.py:240-241)
 *   sqb_interaction_matrix     <- _interaction_matrix(data, indices, indptr, cats, out) src/squidpy/gr/_nhood.py:401,412-429
 *   sqb_autocorr_*             <- scanpy.metrics.morans_i / gearys_c call     src/squidpy/gr/_ppatterns.py:216,267-272
 *   sqb_cooc_counts            <- _occur_count(x, y, thresholds, labs, n,k,l) src/squidpy/gr/_ppatterns.py:283-310
 *   sqb_pair_counts_f64        <- KDTree.two_point_correlation(points, r)     src/squidpy/gr/_ripley.py:218-223
 *   sqb_ligrec_counts          <- _score_permutations(data, clustering, generators, ...)  src/squidpy/gr/_ligrec.py:616-676
 *   sqb_sepal                  <- _diffusion(conc, use_hex, n_iter, sat, sat_idx, unsat, unsat_idx, dt, thresh)  src/squidpy/gr/_sepal.py:186-233
 *   sqb_knn_2d / sqb_radius_2d <- NearestNeighbors.kneighbors / radius_neighbors src/squidpy/gr/neighbors.py:192-209,253-270,395-419
 *   sqb_interaction_matrix     <- _interaction_matrix(data, indices, indptr, cats, out)  src/squidpy/gr/_nhood.py:412-429
 */
#ifndef SQUIDPY_B200_H
#define SQUIDPY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SQB_ABI_VERSION 3

typedef enum {
    SQB_OK = 0,
    SQB_ERR_INVALID = -1, /* bad argument (message says which) */
    SQB_ERR_CUDA = -2,    /* CUDA runtime / launch failure */
    SQB_ERR_OOM = -3,     /* device allocation failed */
    SQB_ERR_UNSUPPORTED = -4,
    SQB_ERR_STATE = -5 /* call sequence error (e.g. run before upload) */
} sqb_status;

typedef struct sqb_ctx sqb_ctx;
typedef struct sqb_nhood sqb_nhood;
typedef struct sqb_autocorr sqb_autocorr;

/* ---- library / context --------------------------------------------------------------------------- */
int sqb_abi_version(void);
const char* sqb_last_error(void);
int sqb_device_count(int* count);

/* stream: a cudaStream_t to launch on (e.g. torch's current stream), or NULL for a library-owned stream. */
int sqb_ctx_create(int device, void* stream, sqb_ctx** out);
int sqb_ctx_destroy(sqb_ctx* ctx);
int sqb_ctx_sync(sqb_ctx* ctx);
int sqb_ctx_stream(sqb_ctx* ctx, void** stream);
int sqb_ctx_sm_count(sqb_ctx* ctx, int* sm_count);
/* number of kernels this library launched on ctx so far */
int sqb_ctx_launch_count(sqb_ctx* ctx, int64_t* launches);
/* per-kernel-class event timing (synchronises every launch; for roofline passes, not for throughput runs) */
int sqb_ctx_profile(sqb_ctx* ctx, int enable);
int sqb_ctx_profile_reset(sqb_ctx* ctx);
/* kclass: 0 fill, 1 shuffle, 2 transpose, 3 count, 4 autocorr prep, 5 autocorr main, 6 autocorr final, 7 pairs, 8 misc */
int sqb_ctx_profile_get(sqb_ctx* ctx, int kclass, double* ms, int64_t* launches);

/* page-locked host memory for the host-facing API (so H2D/D2H copies run at full PCIe rate) */
int sqb_host_alloc(size_t bytes, void** ptr);
int sqb_host_free(void* ptr);

/* ---- nhood_enrichment ------------------------------------------------------------------------------
 * Graph = CSR of obsp['spatial_connectivities'] (data ignored; entries counted as stored; reference dtypes
 * uint32, _nhood.py:52,205).  n_cls = number of categories (labels in [0, n_cls)).                       */
int sqb_nhood_create(sqb_ctx* ctx, int64_t n, int64_t nnz, const uint32_t* indptr, const uint32_t* indices,
                     int n_cls, sqb_nhood** out);
int sqb_nhood_destroy(sqb_nhood* h);

/* observed count: out[a*n_cls+b] = #stored entries (i->j) with labels[i]=a, labels[j]=b   (uint32)       */
int sqb_nhood_count(sqb_nhood* h, const uint32_t* labels, uint32_t* out);

/* Base labels for the permutation test and the optional library partition (lib_codes[i] in [0,n_libs),
 * NULL/0 for none).  With libraries each category is shuffled separately, in category order, by the same
 * generator (gr/_utils.py:208-212).                                                                      */
int sqb_nhood_set_base(sqb_nhood* h, const uint32_t* base_labels, const int32_t* lib_codes, int n_libs);

/* Permutation test.  states: n_perms x 6 uint64 = numpy PCG64 state of generator p
 *   {state_hi, state_lo, inc_hi, inc_lo, has_uint32, uinteger}  (has_uint32 must be 0: fresh generators).
 * Permutation p replays numpy Generator.shuffle bit-exactly on the device and counts.
 * out_counts: n_perms x n_cls x n_cls uint32.                                                            */
int sqb_nhood_permute(sqb_nhood* h, const uint64_t* states, int64_t n_perms, uint32_t* out_counts);

/* The same in three steps, for measurement with inputs resident in HBM:
 * upload (H2D of the generator states), run (kernels only, asynchronous on the ctx stream, results stay on
 * the device), download (D2H of the counts, synchronises).                                               */
int sqb_nhood_permute_upload(sqb_nhood* h, const uint64_t* states, int64_t n_perms);
int sqb_nhood_permute_run_async(sqb_nhood* h);
int sqb_nhood_permute_download(sqb_nhood* h, uint32_t* out_counts);
/* Fast RNG mode (NOT the reference's permutations): permutation p (global index first_perm + p) of every library
 * segment is a keyed bijection — 4-round Feistel network with cycle walking, round keys = splitmix64(seed, global
 * permutation index, segment, round) — applied to the segment's labels sorted by class; labels are written straight into
 * the permutation-minor matrix the count kernel reads (no stream replay, no Fisher-Yates, no transposition).  Same
 * null distribution as numpy's shuffle, different draws: z-scores agree with the exact mode to O(n_perms^-1/2)
 * (SURVEY.md 8d "Fast-RNG validation"); tests/philox_ref.py is the executable specification.  After this upload,
 * run_async / download / stats / sums / var_chain / shuffled_labels work as in the exact mode.                     */
int sqb_nhood_permute_upload_philox(sqb_nhood* h, uint64_t seed, int64_t first_perm, int64_t n_perms);
/* Mean and standard deviation over the permutations of every count bin (n_cls x n_cls float64 each), computed on the
 * device in the operation order of numpy's perms.mean(axis=0) / perms.std(axis=0) on the float64 counts
 * (_nhood.py:231), i.e. bit-identical to the reference's host computation; saves the download of all counts.          */
int sqb_nhood_permute_stats(sqb_nhood* h, double* mean_out, double* std_out);
/* The same statistics when the permutations are sharded over several GPUs (contiguous shards in rank order):
 * sums: exact integer per-bin sums of this handle's permutations (all-reduce them, mean = sum / P_total);
 * var_chain: acc_out = acc_in continued with numpy's sequential sum((x - mean)^2) over this handle's permutations; rank r
 * passes acc_out to rank r+1, std = sqrt(acc_last / P_total): bit-identical to perms.std(axis=0) on the gathered counts.  */
int sqb_nhood_permute_sums(sqb_nhood* h, int64_t* sums_out);
int sqb_nhood_permute_var_chain(sqb_nhood* h, const double* mean, const double* acc_in, double* acc_out);

/* The same statistics with DEVICE pointers (n_cls*n_cls elements each), asynchronous on the ctx stream: for callers that
 * hand the buffers straight to a collective (torch tensors + NCCL) — no host round trip between count kernel and all-reduce. */
int sqb_nhood_permute_stats_dev(sqb_nhood* h, double* d_mean, double* d_std);
int sqb_nhood_permute_sums_dev(sqb_nhood* h, int64_t* d_sums);
int sqb_nhood_permute_var_chain_dev(sqb_nhood* h, const double* d_mean, const double* d_acc_in, double* d_acc_out);
/* Multi-GPU statistics by gathering (what squidpy_b200._dist does under NCCL): the per-permutation counts [n_perms][n_cls^2] as an
 * asynchronous device-to-device copy on the context's stream into a caller-owned buffer (the block a collective sends), and the
 * mean / std over the rows of any device array of counts (the gathered blocks, rows in global permutation order) -- the kernel of
 * sqb_nhood_permute_stats, i.e. `perms.mean(0)` / `perms.std(0)` of gr/_nhood.py:231 in numpy's operation order.          */
int sqb_nhood_permute_counts_dev(sqb_nhood* h, uint32_t* d_dst);
int sqb_nhood_stats_rows_dev(sqb_ctx* ctx, const uint32_t* d_counts, int64_t rows, int n_cls, double* d_mean, double* d_std);

/* Test hook: shuffled label vectors of permutations [p0, p1) of the last upload, recomputed on the device
 * (original node order), out: (p1-p0) x n uint32.                                                        */
int sqb_nhood_shuffled_labels(sqb_nhood* h, int64_t p0, int64_t p1, uint32_t* out);

/* Tuning / test options (all variants produce bit-identical results).
 *   "shuffle_algo"   -1 auto [default]: two-kernel list replay (7) for many permutations of large arrays, else 1 / 2;
 *                    1 CTA per permutation; 2 warp per permutation; 7 two kernels (swap-target generation + list apply);
 *                    any other value is rejected with SQB_ERR_INVALID.
 *   "shuffle_threads" 128/256/512/1024 (algos 1, 7), "shuffle_r" 2/4/8 steps per thread (7),
 *   "shuffle_q"      1/2/4/8 PCG64 outputs per lane and batch (2, and the target generation of 7),
 *   "shuffle_low"    elements of every label array kept in shared memory by the apply kernel of 7 (-1 all that fits, 0 off),
 *   "shuffle_ctas"   persistent grid size = permutations in flight (0 = occupancy x SM count),
 *   "shuffle_stagger_us" start-up stagger of the persistent CTAs, "shuffle_wfactor_x100" window = min(i/4, f*sqrt(i)),
 *   "perm_chunk"     permutations resident at once (read at the next upload), "count_algo" 0 auto / 1 shared-memory histograms /
 *                    2 global atomics, "count_sym" -1 auto (row-record kernel; structurally symmetric graphs are counted from the entries with j >= i) /
 *                    0 always the CSR-row kernel on the full CSR, "count_un" row records (three entries each) a warp takes per pass in the count kernel (1 / 2 / 3 / 4),
 *   "count_single"   sqb_nhood_count: 1 dedicated single-vector kernel [default] / 0 the batched kernels (test hook). */
int sqb_nhood_set_option(sqb_nhood* h, const char* key, int64_t value);
/* algorithmic bytes per permutation, SURVEY.md 8(d): 4*nnz + 4*(n+1) + 8*n + 4*n_cls^2                   */
int sqb_nhood_bytes_per_perm(sqb_nhood* h, int64_t* bytes);

/* ---- interaction_matrix ------------------------------------------------------------------------------
 * Replaces _interaction_matrix(data, indices, indptr, cats, output) (src/squidpy/gr/_nhood.py:401,412-429) and the NaN
 * masking of interaction_matrix (:386-395).  codes[i] in [0, n_cls) or < 0 for an observation without label: stored
 * entries with an unlabelled end point are skipped (== restricting the graph to the labelled observations).
 * data == NULL (weights=False): out_counts[a*n_cls+b] = number of stored entries (i->j) with code(i)=a, code(j)=b (int64).
 * data != NULL (weights=True, data_dtype 0 = f32, 1 = f64): out_weighted[a*n_cls+b] = float64 sum of their values.       */
int sqb_interaction_matrix(sqb_ctx* ctx, int64_t n, int64_t nnz, const uint32_t* indptr, const uint32_t* indices,
                           const void* data, int data_dtype, const int32_t* codes, int n_cls, double* out_weighted,
                           int64_t* out_counts);

/* ---- ligrec permutation test ------------------------------------------------------------------------------
 * _score_permutations of the reference (src/squidpy/gr/_ligrec.py:616-676) for a handle whose base labels are the cells'
 * cluster codes (sqb_nhood_set_base on a graph-less handle: nnz = 0) and whose numpy generator states are uploaded
 * (sqb_nhood_permute_upload).  data: n x n_genes float64 row-major; inv_counts: n_cls; mean_obs: n_cls x n_genes;
 * interactions: n_inter x 2 gene indices; inter_clusters: n_cpairs x 2 cluster indices; valid: n_inter x n_cpairs (uint8).
 * out_counts[i, j] = #permutations with  mean_perm[a, g0] + mean_perm[b, g1] > mean_obs[a, g0] + mean_obs[b, g1]
 * (int64; same float64 operation order as the reference, so the decisions are identical).                          */
int sqb_ligrec_counts(sqb_nhood* h, const double* data, int64_t n_genes, const double* inv_counts, const double* mean_obs,
                      const int32_t* interactions, int64_t n_inter, const int32_t* inter_clusters, int64_t n_cpairs,
                      const uint8_t* valid, int64_t* out_counts);

/* ---- spatial_autocorr (Moran's I / Geary's C) -------------------------------------------------------
 * W = obsp[connectivity_key] (after optional float32 row normalisation on the host) as CSR; w_dtype 0 = f32,
 * 1 = f64 (cast to f64 like scanpy does).  mode 0 = Moran's I, 1 = Geary's C.
 * X layout 0: features x obs (row-major dense, or CSR by feature); layout 1: obs x features (row-major
 * dense, or CSR by observation == CSC of the features x obs matrix, AnnData's native X).
 * x_dtype 0 = f32, 1 = f64.  row_perm (or NULL): length-n permutation p; row r of the permuted W is row p[r]
 * (g[idx_shuffle, :], _ppatterns.py:271-272).  out: n_features float64 (NaN for constant features).
 * Sparse X must not store an observation twice for one feature (scipy: sum_duplicates()); indices need not be
 * sorted.  Index ranges, indptr monotonicity and duplicates are checked on the device (SQB_ERR_INVALID).   */
int sqb_autocorr_create(sqb_ctx* ctx, int64_t n, int64_t nnz, const int32_t* w_indptr, const int32_t* w_indices,
                        const void* w_data, int w_dtype, sqb_autocorr** out);
int sqb_autocorr_destroy(sqb_autocorr* h);
int sqb_autocorr_load_dense(sqb_autocorr* h, const void* x, int x_dtype, int layout, int64_t n_features);
int sqb_autocorr_load_csr(sqb_autocorr* h, const int64_t* x_indptr, const int32_t* x_indices, const void* x_data,
                          int x_dtype, int layout, int64_t n_features);
/* Feature shard of a CSR-by-observation matrix (multi-GPU: every rank takes a contiguous range of features): uploads only
 * the columns col_lo <= c < col_hi of every row (rows must hold ascending column indices — scipy's sorted indices; the
 * slices are found with two binary searches per row and packed into pinned staging buffers by host threads) and loads them
 * as features 0 .. col_hi - col_lo.                                                                          */
int sqb_autocorr_load_csr_cols(sqb_autocorr* h, const int64_t* x_indptr, const int32_t* x_indices, const void* x_data,
                               int x_dtype, int64_t n_features_total, int64_t col_lo, int64_t col_hi);
int sqb_autocorr_run_async(sqb_autocorr* h, int mode, const int64_t* row_perm);
int sqb_autocorr_download(sqb_autocorr* h, double* out);
/* The permutation variant in one call (_score_helper, _ppatterns.py:258-280): row_perms = n_perms x n int64 (row p is
 * idx_shuffle of permutation p), out = n_perms x n_features float64.  X stays resident; the permutations are validated
 * on the device (one error flag per batch) and every permutation is one kernel launch.                      */
int sqb_autocorr_run_perms(sqb_autocorr* h, int mode, const int64_t* row_perms, int64_t n_perms, double* out);
/* load + run + download */
int sqb_autocorr_dense(sqb_autocorr* h, int mode, const void* x, int x_dtype, int layout, int64_t n_features,
                       const int64_t* row_perm, double* out);
int sqb_autocorr_csr(sqb_autocorr* h, int mode, const int64_t* x_indptr, const int32_t* x_indices,
                     const void* x_data, int x_dtype, int layout, int64_t n_features, const int64_t* row_perm,
                     double* out);

/* ---- co_occurrence ------------------------------------------------------------------------------------
 * out[(a*k+b)*L + r] = #{ordered (i,j), i != j : labs[i]=a, labs[j]=b, d2_ij <= thr[r]}  (int64, cumulative in
 * r), float32 arithmetic with d2 = fma(dy,dy,dx*dx) (use_fma=1, what the reference's JIT emits on x86-64 with
 * FMA) or dx*dx+dy*dy (use_fma=0).  thr ascending.  Only tiles t with t % shard_count == shard_index are
 * evaluated (multi-GPU sharding; pass 0,1 for everything); partial results add up across shards.          */
int sqb_cooc_counts(sqb_ctx* ctx, const float* x, const float* y, int64_t n, const int32_t* labs, int k,
                    const float* thr, int L, int use_fma, int shard_index, int shard_count, int64_t* out);

/* ---- ripley L -------------------------------------------------------------------------------------------
 * For every group g (points group_ptr[g]..group_ptr[g+1] of pts, interleaved x,y float64):
 * out[g*S + s] = #{ordered (i,j) in group g, INCLUDING i == j : sqrt(dx*dx + dy*dy) <= support[s]}  (int64),
 * i.e. sklearn KDTree.two_point_correlation(points_g, support).  support ascending.                        */
int sqb_pair_counts_f64(sqb_ctx* ctx, const double* pts, const int64_t* group_ptr, int n_groups,
                        const double* support, int S, int shard_index, int shard_count, int64_t* out);

/* ---- sepal ---------------------------------------------------------------------------------------------------------
 * `_diffusion` for every gene (src/squidpy/gr/_sepal.py:186-289): vals = n_genes x n float64 (one row per gene), sat / unsat =
 * saturated / unsaturated node ids, sat_idx = n_sat x max_neighs neighbour ids, unsat_idx = nearest saturated node of every
 * unsaturated node (`_compute_idxs`, :292-306).  out[g] = dt * (first iteration whose entropy change is <= thresh), NaN if
 * n_iter iterations do not converge.                                                                                  */
int sqb_sepal(sqb_ctx* ctx, const double* vals, int64_t n_genes, int64_t n, const int32_t* sat, int64_t n_sat,
              const int32_t* sat_idx, int max_neighs, const int32_t* unsat, const int32_t* unsat_idx, int64_t n_unsat,
              int n_iter, double dt, double thresh, double* out);

/* ---- spatial neighbour graphs (what runs right before every hot-path call) ------------------------------------------
 * Exact k nearest neighbours of every observation among the others (2-D float64 coordinates, interleaved x,y), the query
 * itself excluded: NearestNeighbors(n_neighbors=k).fit(xy).kneighbors() of KNNBuilder.build_graph / GridBuilder._base_adjacency
 * (src/squidpy/gr/neighbors.py:192-209, :395-419).  out_idx / out_dist: n x k, every row ordered by ASCENDING NEIGHBOUR INDEX
 * (CSR-ready: indptr = k * arange(n + 1)); distances = sqrt(dx*dx + dy*dy) in float64 like sklearn's kd_tree.  Ties at the k-th
 * distance go to the smaller index.  median_out (or NULL): np.median of the n*k distances (GridBuilder's cut = 1.3 x that).   */
int sqb_knn_2d(sqb_ctx* ctx, const double* xy, int64_t n, int k, int32_t* out_idx, double* out_dist, double* median_out);
/* All neighbours within `radius` (dx*dx + dy*dy <= radius*radius, self excluded): radius_neighbors() of RadiusBuilder.build_graph
 * (neighbors.py:253-270).  Two calls: with out_idx == NULL only out_indptr (n + 1) and *nnz_out are produced; with buffers of
 * `capacity` >= nnz entries the rows are filled in ascending column order.                                                 */
int sqb_radius_2d(sqb_ctx* ctx, const double* xy, int64_t n, double radius, int64_t* out_indptr, int32_t* out_idx,
                  double* out_dist, int64_t capacity, int64_t* nnz_out);

#ifdef __cplusplus
}
#endif
#endif /* SQUIDPY_B200_H */
