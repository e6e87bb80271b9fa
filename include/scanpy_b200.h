/* scanpy_b200.h — C ABI of libscanpy_b200.so: the B200-native (sm_100a) kernels behind
 * scanpy's  sc.pp.pca -> sc.pp.neighbors -> sc.tl.leiden  hot path.
 *
 * The reference (scverse/scanpy @ fabadb94) is pure Python and has no FFI of its own: its hot
 * path is three call sites into third-party native code.  Each entry point below replaces one of
 * those call sites and is what a reference-side binding (ctypes, see INTEGRATION.md) would bind:
 *
 *   sb2_pca_csr_f32            <- sklearn PCA(svd_solver='arpack').fit_transform(csr)
 *                                 src/scanpy/preprocessing/_pca/__init__.py:282-291,308
 *                                 (solver 1: the covariance_eigh route, _pca/_dask.py:143-213 +
 *                                  _pca/_kernels.py:14-58)
 *   sb2_knn_l2_f32             <- KNeighborsTransformer(algorithm='brute').fit_transform(x)
 *                                 src/scanpy/neighbors/__init__.py:754-768,638
 *   sb2_fuzzy_simplicial_set_f32 <- umap.umap_.fuzzy_simplicial_set(...).tocsr()
 *                                 src/scanpy/neighbors/_connectivity.py:124-138
 *   sb2_leiden_csr_f32         <- leidenalg.find_partition / Graph.community_leiden
 *                                 src/scanpy/tools/_leiden.py:184-187,195-196 (graph build
 *                                 src/scanpy/_utils/__init__.py:278-306 is eliminated: CSR in)
 *
 * Conventions
 *   - every function returns int32: 0 ok, <0 error (SB2_E_*); sb2_last_error() gives the text
 *     (thread-local, library-owned, valid until the next failing call on that thread).
 *   - pointers prefixed d_ are DEVICE pointers into memory the caller owns (the Python host
 *     allocates them as torch CUDA tensors); h_ are HOST pointers.  No torch types cross the ABI.
 *   - work is enqueued on the ctx's CUDA stream.  Functions that return host-visible scalars
 *     (nnz, counters, modularity) synchronise that stream before returning; the others are async.
 *   - a ctx is bound to one device and is not thread-safe.  No callbacks, no exceptions.
 *   - indptr is int64 (10M x 4k at 5 % has > 2^31 non-zeros), column / neighbour indices int32.
 */
#ifndef SCANPY_B200_H
#define SCANPY_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SB2_OK 0
#define SB2_E_BADARG (-1)
#define SB2_E_CUDA (-2)
#define SB2_E_NCCL (-3)
#define SB2_E_OOM (-4)
#define SB2_E_NOTCONV (-5)
#define SB2_E_UNSUPPORTED (-6)

typedef struct sb2_ctx sb2_ctx;

typedef struct sb2_device_info {
  int32_t device;
  int32_t sm_count;
  int32_t cc_major, cc_minor;
  int32_t clock_khz;        /* max SM clock */
  int32_t mem_clock_khz;
  int32_t l2_bytes;
  int32_t smem_per_block_optin;
  int64_t total_mem;
  char name[64];
} sb2_device_info;

/* per-call statistics (all optional: pass NULL) */
typedef struct sb2_pca_info {
  int32_t iterations;       /* operator applications */
  int32_t converged;        /* 1 if residual test met */
  double max_rel_residual;  /* max_j ||A v_j - theta_j v_j|| / theta_1 over the k kept pairs */
  double total_var;         /* sum of per-gene variances (ddof=1) */
} sb2_pca_info;

typedef struct sb2_knn_info {
  int64_t n_uncertified;    /* query rows that needed the exact fallback */
  float max_norm;
  float pass1_ms;           /* CUDA-event duration of all first-pass sweep launches on the ctx stream */
  double pass1_flops;       /* 2 * n_query * n_points * d: the algorithmic flops of that launch */
  double pass1_issued_flops; /* flops actually issued (tensor path: padded tiles x split-precision K axis) */
  int32_t pass1_tensor;     /* 2 = knn_sweep2_kernel (tcgen05 N=256, default), 1 = knn_pass1_tc_kernel (first-generation tcgen05
                               sweep: SB2_KNN_V=1 or K axes too wide for generation 2), 0 = knn_pass1_kernel (fp32 FFMA) */
  int64_t n_resweep;        /* rows the fp16 tier left uncertified, swept again in split precision (tensor path) */
} sb2_knn_info;

typedef struct sb2_leiden_info {
  int32_t passes;           /* whole Leiden iterations run */
  int32_t levels;           /* aggregation levels of the last pass */
  int64_t moves;            /* accepted local moves, all levels */
} sb2_leiden_info;

int32_t sb2_version(void);
const char* sb2_last_error(void);

/* stream: the cudaStream_t (as void*) to enqueue on; NULL means the legacy default stream unless
 * flags has SB2_CTX_PRIVATE_STREAM, in which case the ctx creates its own non-blocking stream. */
#define SB2_CTX_PRIVATE_STREAM 1u
int32_t sb2_ctx_create(int32_t device, void* stream, uint32_t flags, sb2_ctx** out);
int32_t sb2_ctx_destroy(sb2_ctx* ctx);
int32_t sb2_ctx_sync(sb2_ctx* ctx);
int32_t sb2_device_info_get(sb2_ctx* ctx, sb2_device_info* out);
/* number of kernel launches this ctx has enqueued so far (bench.py's gpu_launches) */
int64_t sb2_ctx_launch_count(sb2_ctx* ctx);

/* Multi-GPU (one process per GPU): rank 0 calls sb2_comm_unique_id, the 128 bytes travel to the
 * other ranks through the host's own rendezvous (torch.distributed broadcast), every rank calls
 * sb2_comm_init.  With a communicator attached, sb2_pca_csr_f32 treats its CSR as the rank's row
 * shard and all-reduces its small dense reductions. */
int32_t sb2_comm_unique_id(void* h_id128);
int32_t sb2_comm_init(sb2_ctx* ctx, int32_t n_ranks, int32_t rank, const void* h_id128);
int32_t sb2_comm_allgather(sb2_ctx* ctx, const void* d_send, void* d_recv, int64_t bytes_per_rank);
int32_t sb2_comm_allreduce_f64(sb2_ctx* ctx, double* d_buf, int64_t count);

/* ---- PCA: top-k principal components of the implicitly centred CSR matrix (A1 in SURVEY.md) ----
 * solver 0: block subspace iteration driven by CSR x dense SpMM passes (replaces ARPACK).
 * solver 1: exact Gram route  G = X^T X (one CSR pass) -> covariance -> dense block iteration.
 * n_total = number of rows over ALL ranks (== n when no communicator is attached).
 * Outputs: d_x_pca [n x k] float32 row-major, d_components [k x g] float32 (rows = PCs, sign fixed by
 * svd_flip(u_based_decision=False)), h_var[k], h_var_ratio[k], h_mean[g] (host, float64). */
int32_t sb2_pca_csr_f32(sb2_ctx* ctx, int64_t n, int64_t n_total, int32_t g, const int64_t* d_indptr,
                        const int32_t* d_indices, const float* d_data, int32_t k, int32_t solver,
                        int32_t max_iter, double tol, uint64_t seed, float* d_x_pca, float* d_components,
                        double* h_var, double* h_var_ratio, double* h_mean, sb2_pca_info* info);

/* building blocks of the above, exported for tests / profiling */
int32_t sb2_csr_col_stats(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                          const float* d_data, double* d_col_sum, double* d_col_sumsq);
/* Y[n x l] = X * B[g x l] - 1 * shift[l]  (shift may be NULL) */
int32_t sb2_spmm_csr(sb2_ctx* ctx, int64_t n, int32_t g, int32_t l, const int64_t* d_indptr,
                     const int32_t* d_indices, const float* d_data, const float* d_b, const float* d_shift,
                     float* d_y);
/* Z[g x l] (float64) = X^T * Y[n x l] */
int32_t sb2_spmm_csr_t(sb2_ctx* ctx, int64_t n, int32_t g, int32_t l, const int64_t* d_indptr,
                       const int32_t* d_indices, const float* d_data, const float* d_y, double* d_z);
/* G[g x g] (float64, full symmetric) = X^T X */
int32_t sb2_csr_gram(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                     const float* d_data, double* d_gram);

/* sc.pp.pca(zero_center=False): replaces sklearn.decomposition.TruncatedSVD (src/scanpy/preprocessing/_pca/__init__.py:309-336).
 * Top-k singular triplets of X itself: d_x_pca = X V (= U Sigma), d_components = V^T with svd_flip(u_based_decision=False)
 * signs, h_var = np.var(X V, axis=0) (ddof 0), h_var_ratio = h_var / sum of per-gene variances (ddof 0). */
int32_t sb2_tsvd_csr_f32(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                         const float* d_data, int32_t k, int32_t solver, int32_t max_iter, double tol, uint64_t seed,
                         float* d_x_pca, float* d_components, double* h_var, double* h_var_ratio, sb2_pca_info* info);

/* ---- out-of-core / chunked PCA: sc.pp.pca(chunked=True) (src/scanpy/preprocessing/_pca/__init__.py:245-271) ----
 * The reference streams row chunks through sklearn.decomposition.IncrementalPCA and asserts the result equals the full PCA
 * (tests/test_pca.py:357-386).  Here the chunks stream through the exact Gram route: device memory = one chunk + 2 g^2
 * doubles, independent of n.
 *   pass 1: sb2_pca_stream_accumulate_f32 adds the chunk's column sums / sums of squares into d_stats fp64 [2g] and its
 *           X^T X into d_gram fp64 [g x g] (caller zero-fills both before the first chunk);
 *   solve : sb2_pca_stream_solve_f32 -> d_components [k x g], h_var, h_var_ratio, h_mean as sb2_pca_csr_f32, plus the
 *           projection operator d_proj fp32 [g x 128] (first g * *h_l entries used), d_shift fp32 [128], *h_l (32/64/128);
 *   pass 2: sb2_pca_stream_project_f32 -> d_x_pca [n_chunk x k] = X_chunk U - mu^T U. */
int32_t sb2_pca_stream_accumulate_f32(sb2_ctx* ctx, int64_t n_chunk, int32_t g, const int64_t* d_indptr,
                                      const int32_t* d_indices, const float* d_data, double* d_stats, double* d_gram);
int32_t sb2_pca_stream_solve_f32(sb2_ctx* ctx, int64_t n_total, int32_t g, const double* d_stats, const double* d_gram,
                                 int32_t k, int32_t max_iter, double tol, uint64_t seed, float* d_components, double* h_var,
                                 double* h_var_ratio, double* h_mean, float* d_proj, float* d_shift, int32_t* h_l,
                                 sb2_pca_info* info);
int32_t sb2_pca_stream_project_f32(sb2_ctx* ctx, int64_t n_chunk, int32_t g, const int64_t* d_indptr,
                                   const int32_t* d_indices, const float* d_data, int32_t k, int32_t l, const float* d_proj,
                                   const float* d_shift, float* d_x_pca);

/* ---- exact brute-force kNN (euclidean) -----------------------------------------------------
 * points: d_x [n_points x d] float32 row-major.  Queries are rows [q0, q0+n_query) of the same
 * array (q0 % 128 == 0 unless n_query == n_points).  k includes the query itself: column 0 of
 * the outputs is the query row with distance 0 (src/scanpy/neighbors/_common.py:74-98).
 * Outputs [n_query x k]: d_idx int32 (global row ids), d_dist float64, ascending by (distance, id).
 * d <= 150, k <= 56.  Exactness: a fast first pass (tcgen05 fp16 / split-fp16 sweeps; SB2_KNN_PASS1=ffma selects the
 * fp32 CUDA-core sweep, k <= 30) proposes 32 (k <= 24) or 64 candidates per query, an fp64 re-score certifies the top-k
 * against a rounding-error bound, uncertified rows are recomputed exactly. */
int32_t sb2_knn_l2_f32(sb2_ctx* ctx, int64_t n_points, int32_t d, const float* d_x, int64_t q0, int64_t n_query,
                       int32_t k, int32_t* d_idx, double* d_dist, sb2_knn_info* info);

/* test / debug entry: raw proposals (scores in the sweep's scaled units + ids, 64 per point) of ONE cold-start tensor-core
 * sweep in the operand format `terms` (1: fp16, 3: split fp16) and the quantities its rounding-error certificate uses:
 * h_meta[6] = { inv_s2 (score_true = score * inv_s2), largest squared norm R^2, max_p |x_p - fp16(x_p)|, c_q, c_n, list_m };
 * the certificate bounds |score * inv_s2 - (q.c - |c|^2/2)| by  c_n R^2/2 + c_q |q| R  (+ for terms = 1:
 * dnorm[q] R + (|q| + dnorm[q]) max dnorm).  d_dnorm [n_points] may be NULL. */
int32_t sb2_knn_debug_proposals_f32(sb2_ctx* ctx, int64_t n_points, int32_t d, const float* d_x, int32_t terms,
                                    float* d_score, int32_t* d_idx, float* d_dnorm, double* h_meta);

/* ---- UMAP fuzzy simplicial set -> symmetric connectivities CSR -------------------------------
 * d_knn_idx/d_knn_dist [n x k] (column 0 = self), as produced by sb2_knn_l2_f32; 2 <= k <= 64.
 * Output CSR: d_indptr int64[n+1], d_indices int32[cap], d_data float32[cap]; cap >= 2*n*(k-1) is
 * always enough.  Rows sorted by column, no explicit zeros, zero diagonal. */
int32_t sb2_fuzzy_simplicial_set_f32(sb2_ctx* ctx, int64_t n, int32_t k, const int32_t* d_knn_idx,
                                     const double* d_knn_dist, float set_op_mix_ratio, float local_connectivity,
                                     int64_t* d_indptr, int32_t* d_indices, float* d_data, int64_t cap,
                                     int64_t* h_nnz, float* d_sigmas, float* d_rhos);

/* method='gauss' (method 1) / 'jaccard' (method 2) connectivities from the same k-lists (SURVEY.md 8f row f3;
 * src/scanpy/neighbors/_connectivity.py:17-100 sparse kNN branch, :141-186).  float64 values like the reference. */
int32_t sb2_knn_connectivities_f64(sb2_ctx* ctx, int64_t n, int32_t k, const int32_t* d_knn_idx, const double* d_knn_dist,
                                   int32_t method, int64_t* d_indptr, int32_t* d_indices, double* d_data, int64_t cap,
                                   int64_t* h_nnz);

/* ---- Leiden on a symmetric weighted CSR graph ------------------------------------------------
 * n_iterations < 0: iterate until a whole pass moves nothing.  Output membership int32[n]
 * renumbered by decreasing community size; *h_modularity at the given resolution. */
int32_t sb2_leiden_csr_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                           const float* d_weights, double resolution, int32_t n_iterations, uint64_t seed,
                           int32_t* d_membership, double* h_modularity, int32_t* h_n_comms, sb2_leiden_info* info);
int32_t sb2_modularity_csr_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                               const float* d_weights, double resolution, const int32_t* d_membership,
                               double* h_modularity);
/* Louvain (SURVEY.md 8f row f3): local moving + aggregation, no refinement, one pass to its fixed point - replaces
 * `louvain.find_partition(g, RBConfigurationVertexPartition, ...)` / `g.community_multilevel(weights)` at
 * src/scanpy/tools/_louvain.py:150-176.  Outputs as sb2_leiden_csr_f32. */
int32_t sb2_louvain_csr_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                            const float* d_weights, double resolution, uint64_t seed, int32_t* d_membership,
                            double* h_modularity, int32_t* h_n_comms, sb2_leiden_info* info);

/* ---- preprocessing passes in front of the path (SURVEY.md 8f, row f2): normalize_total, log1p, HVG statistics ----
 * sb2_csr_row_sums_f32      <- numba `_normalize_csr` (src/scanpy/preprocessing/_normalization.py:29-66): per-cell
 *                              totals; with d_skip_cols only columns whose flag is 0 are summed
 * sb2_csr_hiexpr_count_f32  <- same function, the `exclude_highly_expressed` branch: per-gene count of entries
 *                              exceeding max_fraction * cell total
 * sb2_csr_scale_rows_f32    <- axis_mul_or_truediv(x, counts_per_cell, op=truediv, allow_divide_by_zero=False)
 *                              (src/scanpy/_utils/__init__.py:623-660), in place
 * sb2_log1p_f32             <- np.log1p(x.data) [/ log(base)] (src/scanpy/preprocessing/_simple.py:359-380), in place
 * sb2_csr_col_sums_f32      <- stats.mean_var(expm1(x), axis=0) inside highly_variable_genes(flavor='seurat')
 *                              (src/scanpy/preprocessing/_highly_variable_genes.py:337-346): per-gene sum and sum of
 *                              squares (fp64) of expm1(x * log_scale) (apply_expm1 = 1) or of x */
int32_t sb2_csr_row_sums_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                             const float* d_data, const int32_t* d_skip_cols, float* d_out);
int32_t sb2_csr_hiexpr_count_f32(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                 const float* d_data, const float* d_row_sums, double max_fraction,
                                 int32_t* d_counts_per_col);
int32_t sb2_csr_scale_rows_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, float* d_data, const float* d_scale);
int32_t sb2_log1p_f32(sb2_ctx* ctx, int64_t nnz, float* d_data, double base);
int32_t sb2_csr_col_sums_f32(sb2_ctx* ctx, int64_t nnz, int32_t g, const int32_t* d_indices, const float* d_data,
                             int32_t apply_expm1, double log_scale, double* d_sum, double* d_sumsq);


/* ---- extreme eigenpairs of diag(s) A diag(s), A symmetric fp32 CSR (csrc/eigs.cu: thick-restart Lanczos, fp64) ----
 * Replaces `scipy.sparse.linalg.eigsh(matrix.astype(float64), k=n_comps, which='LM', v0=...)` in
 * Neighbors.compute_eigen (src/scanpy/neighbors/__init__.py:832-884; sc.tl.diffmap) and the eigsh of umap's spectral
 * initialisation (sc.tl.umap).  d_scale may be NULL (s = 1).  which: 0 largest algebraic, 1 largest magnitude, 2 smallest
 * algebraic.  ncv <= 0 / tol <= 0 / max_restarts <= 0 pick defaults (max(2 nev + 16, 40), 1e-10, 400).  h_evals ascending
 * like eigsh; d_evecs fp64 [nev x n], row e = unit eigenvector of h_evals[e] (sign arbitrary, as with ARPACK). */
typedef struct sb2_eigs_info {
  int32_t restarts, matvecs, n_converged, reserved;
  double max_residual;
} sb2_eigs_info;
int32_t sb2_eigsh_csr_scaled(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                             const float* d_weights, const double* d_scale, int32_t nev, int32_t which, int32_t ncv,
                             double tol, int32_t max_restarts, const double* d_v0, double* h_evals, double* d_evecs,
                             sb2_eigs_info* info);
/* d_scale fp64[n] with T_sym = diag(d_scale) W diag(d_scale): the symmetrised transition matrix of
 * Neighbors.compute_transitions (src/scanpy/neighbors/__init__.py:791-830; density_normalize as there). */
int32_t sb2_transition_scale_f64(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                                 const float* d_weights, int32_t density_normalize, double* d_scale);

/* ---- sc.tl.umap layout (SURVEY.md 8f row f1; csrc/umap.cu) ----
 * Replaces `umap.umap_.simplicial_set_embedding` as called at src/scanpy/tools/_umap.py:196-215.
 * sb2_umap_spectral_init_f32: init='spectral' (eigenvectors 2..dim+1 of D^-1/2 A D^-1/2, expanded to max|x| = 10, N(0,1e-4)
 *   jitter) into d_init fp32 [n x dim].
 * sb2_umap_layout_f32: d_embedding fp32 [n x dim] holds the initialisation on entry (rescaled to [0,10]^dim first, like the
 *   reference) and the optimised layout on return; graph = symmetric connectivities CSR (not modified); a, b from
 *   find_ab_params(spread, min_dist); deterministic in (graph, init, seed). */
int32_t sb2_umap_spectral_init_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                                   const float* d_weights, int32_t dim, uint64_t seed, float* d_init);
int32_t sb2_umap_layout_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices, const float* d_weights,
                            int32_t dim, int32_t n_epochs, double a, double b, double gamma, double initial_alpha,
                            int32_t negative_sample_rate, uint64_t seed, float* d_embedding);

/* ---- sc.tl.paga aggregation (SURVEY.md 8f row f3): d_counts int64 [G x G], counts[gi*G + gj] = stored arcs i -> j with
 * d_group[i] = gi, d_group[j] = gj.  Replaces igraph's VertexClustering.cluster_graph / subgraph(i).ecount() at
 * src/scanpy/tools/_paga.py:177-208 (inner-cluster edge counts are the diagonal). */
int32_t sb2_group_arc_counts(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices,
                             const int32_t* d_group, int32_t n_groups, int64_t* d_counts);

/* ---- sc.pp.scale (SURVEY.md 8f row f2 tail; src/scanpy/preprocessing/_scale.py:150-296) ----
 * sb2_csr_col_stats_rows_f32 <- mean_var(x[mask_obs, :], axis=0, correction=1): per-gene sum / sum of squares (fp64) over
 *                               the rows with d_mask[row] != 0 (d_mask == NULL: every row)
 * sb2_csr_scale_cols_f32     <- numba `scale_and_clip_csr` (:267-283): data[j] = min(max_value, data[j] / std[col]) on the
 *                               masked rows, in place (zero_center=False keeps the matrix sparse)
 * sb2_csr_scale_dense_f64    <- `x -= mean; x /= std; clip` on a CSR (:203-222): the dense float64 [n x g] result; rows
 *                               outside d_mask keep their values
 * sb2_dense_col_stats / sb2_dense_scale <- the same two steps for a dense float32 (is_f64 = 0) / float64 [n x g] input,
 *                               in place; d_mean == NULL means zero_center=False (then only the upper clip applies) */
int32_t sb2_csr_col_stats_rows_f32(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                   const float* d_data, const uint8_t* d_mask, double* d_sum, double* d_sumsq);
int32_t sb2_csr_scale_cols_f32(sb2_ctx* ctx, int64_t n, const int64_t* d_indptr, const int32_t* d_indices, float* d_data,
                               const double* d_std, const uint8_t* d_mask, int32_t has_max, double max_value);
int32_t sb2_csr_scale_dense_f64(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                const float* d_data, const double* d_mean, const double* d_std, const uint8_t* d_mask,
                                int32_t has_max, double max_value, double* d_out);
int32_t sb2_dense_col_stats(sb2_ctx* ctx, int64_t n, int32_t g, const void* d_x, int32_t is_f64, const uint8_t* d_mask,
                            double* d_sum, double* d_sumsq);
int32_t sb2_dense_scale(sb2_ctx* ctx, int64_t n, int32_t g, void* d_x, int32_t is_f64, const double* d_mean,
                        const double* d_std, const uint8_t* d_mask, int32_t has_max, double max_value);

/* ---- sc.tl.rank_genes_groups (src/scanpy/tools/_rank_genes_groups.py; csrc/rank_genes.cu) ----
 * Cells carry a group code 0..n_codes-1; code n_codes-1 is the remainder (cells in no selected group).  At most
 * SB2_RANK_GENES_MAX_GROUPS selected groups (n_codes <= SB2_RANK_GENES_MAX_GROUPS + 1), else SB2_E_UNSUPPORTED.
 * sb2_rank_genes_group_stats <- the grouped mean / var / count_nonzero of `_basic_stats` (:319-452): for every code q and
 *   gene j, d_sum = sum of x', d_m2 = sum of (x' - mean)^2 over all n_q cells (implicit zeros included), d_nnz = count of
 *   x != 0, with x' = expm1(x * expm1_scale) (expm1_scale != 0) or x.  d_rows int32 [n]: the rows ordered by code (stable),
 *   h_group_offsets int64 [n_codes + 1]: code q owns d_rows[off[q] : off[q + 1]].  Outputs [n_codes x g], bit-reproducible.
 * sb2_rank_genes_wilcoxon <- the rank sums and tie terms of `wilcoxon` (:505-579), exact integers.  d_codes int32 [n],
 *   d_group_sizes int64 [n_codes].  ref < 0: ranks over all cells; d_rank2[q][j] = 2 x rank sum of code q, d_tie[q][j] =
 *   sum over tie runs of gene j of t^3 - t (the same for every q).  ref >= 0: for each q (not ref, not the remainder) ranks
 *   over the cells of q and ref only; d_rank2[q][j] = 2 x rank sum of q, d_tie[q][j] over those cells; remainder cells take
 *   no part, rows ref and n_codes-1 are 0.  d_tie uint64 [n_codes x g x 2] = (low, high) 64-bit halves of the 128-bit sum.
 *   h_stage_ms (may be NULL): float[2] = device ms of the sort and of the rank walk (synchronises the stream). */
#define SB2_RANK_GENES_MAX_GROUPS 1024
int32_t sb2_rank_genes_group_stats(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                   const float* d_data, const int32_t* d_rows, const int64_t* h_group_offsets,
                                   int32_t n_codes, double expm1_scale, double* d_sum, double* d_m2, int64_t* d_nnz);
int32_t sb2_rank_genes_wilcoxon(sb2_ctx* ctx, int64_t n, int32_t g, const int64_t* d_indptr, const int32_t* d_indices,
                                const float* d_data, int64_t nnz, const int32_t* d_codes, const int64_t* d_group_sizes,
                                int32_t n_codes, int32_t ref, int64_t* d_rank2, uint64_t* d_tie, float* h_stage_ms);

#ifdef __cplusplus
}
#endif
#endif /* SCANPY_B200_H */
