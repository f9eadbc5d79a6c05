/*
 * b200rec.h -- C ABI of libb200rec.so, the B200 (sm_100a) compute core that replaces the reference's
 * three Cython extension classes and the inline numpy hot loops of IALS / EASE_R / P3alpha / RP3beta.
 *
 * Boundary (SURVEY.md section 8(b)).  Every entry point below names the reference interface it replaces
 * (paths relative to the reference checkout).  Conventions:
 *   - every function returns 0 on success or a negative B200_E_* code; b200_last_error() gives the text
 *     (thread-local).  No C++ exception crosses the boundary.
 *   - plain pointers and sizes only; the caller owns every buffer it passes; handles own their device memory.
 *   - pointers named h_* are HOST pointers (pageable or pinned), d_* are DEVICE pointers on the current
 *     CUDA device; `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - the library uses the calling thread's current CUDA device (one process per GPU).
 *   - there is no CPU fallback: without a usable CUDA device every call fails with B200_E_CUDA.
 */
#ifndef B200REC_H_
#define B200REC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_E_INVALID (-1) /* bad argument (the Python shim raises ValueError with the reference's text) */
#define B200_E_CUDA (-2)    /* CUDA runtime / launch failure (RuntimeError) */
#define B200_E_NOMEM (-3)   /* device or host allocation failed */
#define B200_E_UNSUPPORTED (-4)

const char* b200_last_error(void);
int b200_version(void);
/* number of kernels of this library launched by the calling process so far (bench.py "gpu_launches") */
int64_t b200_launch_count(void);
/* fills name (<=256 bytes), SM count, and total device memory of the current device */
int b200_device_info(char* name, int name_len, int* sm_count, int64_t* total_mem);

/* ------------------------------------------------------------------------------------------------
 * K1: sparse column-column similarity with top-K  (hot path i)
 * replaces  Base/Similarity/Cython/Compute_Similarity_Cython.pyx:52-611
 *           (ctor :73-216, computeItemSimilarities :327-408, compute_similarity :413-611)
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200_sim_s* b200_sim_t;

enum b200_sim_kind {
  B200_SIM_COSINE = 0,     /* pyx:138, :484-485 / :505-507 */
  B200_SIM_ADJUSTED = 1,   /* pyx:119, :277-312 */
  B200_SIM_ASYMMETRIC = 2, /* pyx:121, :176-180, :479-481 */
  B200_SIM_PEARSON = 3,    /* pyx:123, :236-273 */
  B200_SIM_JACCARD = 4,    /* jaccard == tanimoto, pyx:125-128, :488-491 */
  B200_SIM_DICE = 5,       /* pyx:130-132, :493-496 */
  B200_SIM_TVERSKY = 6,    /* pyx:134-136, :498-503 */
  B200_SIM_EUCLIDEAN = 7   /* Compute_Similarity_Euclidean.py; created through b200_sim_create_euclidean only */
};

/* Build the device-side representation of dataMatrix (n_rows x n_cols CSR, int32 indices sorted per row,
 * fp32 data, no explicit zeros -- what BaseRecommender.__init__ guarantees, Base/BaseRecommender.py:23-24).
 * Does what the reference constructor does (pyx:147-209): TopK=min(topK,n_cols), the per-kind data
 * transform, column norms, row weights, CSR + CSC copies -- on the GPU.
 *   shrink      : already truncated to an integer value by the caller if it mirrors pyx:65
 *   normalize   : ignored (forced 0) for the set kinds, as pyx:128,132,136
 *   h_row_weights: NULL or n_rows floats (pyx:184-194)
 * topK must be >= 1 here; the dense (TopK==0, pyx:510-513) and full-Gram (EASE_R, topK=n_cols) outputs go
 * through b200_sim_compute_dense(). */
int b200_sim_create(b200_sim_t* out, int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* h_indptr,
                    const int32_t* h_indices, const float* h_data, int kind, int topK, float shrink,
                    int normalize, float asymmetric_alpha, float tversky_alpha, float tversky_beta,
                    const float* h_row_weights, void* stream);
int b200_sim_destroy(b200_sim_t h);

/* P3alpha / RP3beta product (GraphBased/P3alphaRecommender.py:54-117, GraphBased/RP3betaRecommender.py:54-104):
 * for target item i and neighbour j,  value = A[i] * B[j] * sum over users u of item i of data[u, j], with
 * data = (r_uj / rowsum_u)^alpha (Pui), A[i] = (1/deg_i)^alpha (the constant row of Piu), B[j] = deg_j^-beta
 * (RP3beta; all ones for P3alpha).  The same accumulate/top-K kernel as the similarities (formula "scale");
 * b200_sim_compute* then returns per TARGET item i its topK (j, value) -- row i of the reference's W_sparse. */
int b200_sim_create_scaled(b200_sim_t* out, int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* h_indptr,
                           const int32_t* h_indices, const float* h_data, const float* h_A, const float* h_B,
                           int topK, void* stream);

/* Euclidean similarity (Base/Similarity/Compute_Similarity_Euclidean.py:17-223): for target column i and EVERY other
 * column j (co-rated or not)  d2 = |i|^2 + |j|^2 - 2 i.j (:144-149), optionally / (|i| |j|) where that is non-zero
 * (normalize, :152-154) and / n_rows (normalize_avg_row, :156-157), d = sqrt(d2) where d2 > 0 (:159-160),
 * similarity = 1 / (g(d) + shrink + 1e-9) with g = exp, identity or log(1 + .) (:162-169); the K largest over all
 * columns except i itself (:172-186).  Same accumulate kernel as b200_sim_create, every cell of the neighbour axis
 * evaluated; b200_sim_compute* return the top-K table.  row_weights (:152, only well defined for square matrices in
 * the reference) are not supported. */
enum b200_euclid_mode { B200_EUCLID_EXP = 0, B200_EUCLID_LIN = 1, B200_EUCLID_LOG = 2 };
int b200_sim_create_euclidean(b200_sim_t* out, int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* h_indptr,
                              const int32_t* h_indices, const float* h_data, int topK, float shrink, int normalize,
                              int normalize_avg_row, int distance_mode, void* stream);

/* effective K (min(topK, n_cols)), window geometry and path chosen at create time */
int b200_sim_info(b200_sim_t h, int* K, int* n_windows, int* window_cells, int* binary_path, int* signed_data);

/* compute_similarity(start_col, end_col) (pyx:413-611) for columns [start_col, end_col):
 * for local column c = col - start_col, slots [c*K, c*K + cnt[c]) of idx/val hold the neighbours j and
 * similarities W[j, col]; unused slots hold idx -1 / val 0.  Neighbours are the K largest similarities
 * among all columns (zeros outrank negatives and are not emitted -- Compute_Similarity_Python.py:335-345),
 * ties broken by ascending neighbour index.  Slot order within a column is unspecified.
 * The d_ variant leaves results on the device (the NCCL all-gather send buffer in multi-GPU runs). */
int b200_sim_compute_device(b200_sim_t h, int start_col, int end_col, int32_t* d_idx, float* d_val,
                            int32_t* d_cnt, void* stream);
int b200_sim_compute(b200_sim_t h, int start_col, int end_col, int32_t* h_idx, float* h_val, int32_t* h_cnt);
/* Multi-GPU, item-sharded (SURVEY.md 8(e) K1): like b200_sim_compute_device for the columns [start_col, end_col) this rank
 * owns, but every finished column is written into n_tables FULL tables -- d_tables[0] the local one, the others the peers'
 * copies of the same allocation, mapped into this process (symmetric memory over NVLink / NVSwitch) -- by the CTA that
 * computed it, so the kernel is the all-gather and no collective follows it (a barrier across the ranks does).
 * Each table is one int32 allocation: idx rows [n_columns, K] at idx_offset, val rows (fp32 bits) at val_offset, cnt
 * [n_columns] at cnt_offset (offsets in 4-byte elements); row = ORIGINAL column index.  n_tables <= 8. */
int b200_sim_compute_peers_device(b200_sim_t h, int start_col, int end_col, int n_tables, void* const* d_tables,
                                  int64_t idx_offset, int64_t val_offset, int64_t cnt_offset, void* stream);
/* Dense output (TopK == 0, pyx:510-513,597-599; and the full Gram EASE_R asks for with topK = n_items,
 * EASE_R/EASE_R_Recommender.py:55-56): d_out is [end_col - start_col, n_cols] row-major fp32,
 * d_out[target - start_col, neighbour] = W[neighbour, target]; zero where the columns share no row. */
int b200_sim_compute_dense_device(b200_sim_t h, int start_col, int end_col, float* d_out, void* stream);

/* Assemble the scipy-canonical CSR of W (n_cols x n_cols, row j = neighbour, column = target column, sorted
 * column indices per row, fp32 -- what pyx:603-611 returns) from a top-K table holding ALL columns
 * (e.g. after the all-gather).  Two calls: _count returns nnz; _fill writes indptr[n_cols+1], indices[nnz],
 * data[nnz] into host buffers.  d_idx/d_val/d_cnt are device pointers of shape [n_cols*K],[n_cols*K],[n_cols]. */
int b200_topk_table_to_csr_count(int n_cols, int K, const int32_t* d_cnt, int64_t* nnz_out, void* stream);
int b200_topk_table_to_csr_fill(int n_cols, int K, const int32_t* d_idx, const float* d_val,
                                const int32_t* d_cnt, int64_t nnz, int32_t* h_indptr, int32_t* h_indices,
                                float* h_data, void* stream);

/* TEST HOOK: shrink the logical capacity of the candidate buffer (K < cap <= allocated) so that small inputs
 * exercise the overflow / rescan path of the selection. */
int b200_sim_debug_set_cap(b200_sim_t h, int cap);

/* TEST/BENCH HOOK: per-phase SM-cycle counters of the top-K kernel, summed over CTAs (thread 0's clock):
 * [0] stage  [1] accumulate  [2] bootstrap histogram  [3] scan+clear  [4] evaluate+compact  [5] select
 * [6] emit (window kernel); the bitmap kernel reports [1] accumulate  [2] level >= 3  [3] level 2  [4] level 1  [6] emit+clear.  enable!=0 turns counting on for later launches; out8 (nullable) receives and resets the counters. */
int b200_sim_debug_phase_cycles(b200_sim_t h, int enable, uint64_t* out8);

/* TEST/BENCH HOOK for the 4-bit-counter kernel of the binary path (csrc/sim_k1d.cuh; chosen at create time for binary data
 * with many columns, B200REC_K1C=0 disables it): reports whether the handle uses it, how many of its CTAs share an SM, and
 * how the last launch was routed (columns it took / columns the window kernel computed, including the ones handed back
 * because a counter overflowed).  set_fail_every > 0 makes it hand back every n-th local column (exercises the redo path);
 * 0 switches that off. */
int b200_sim_debug_k1c(b200_sim_t h, int set_fail_every, int* enabled, int* ctas_per_sm, int* n_bitmap_cols, int* n_window_cols);

/* duration in milliseconds of the last top-K kernel launched through this handle, measured with CUDA
 * events on the launching stream (bench.py roofline leg) */
int b200_sim_last_kernel_ms(b200_sim_t h, float* ms);
/* sum over columns [start,end) of the gathered-entry count  sum_{u in col} len_u  (SURVEY 8(d) bytes model) */
int b200_sim_work(b200_sim_t h, int start_col, int end_col, int64_t* gathered_entries);
/* the same quantity per (original) column, n_cols int64 values: the weights of the multi-GPU column partition */
int b200_sim_col_work(b200_sim_t h, int64_t* out_n_cols);

/* ------------------------------------------------------------------------------------------------
 * K2: matrix-factorisation SGD epochs, BPR-MF and FunkSVD  (hot path ii)
 * replaces  MatrixFactorization/Cython/MatrixFactorization_Cython_Epoch.pyx:51-987
 *           (ctor :96-151, epochIteration_Cython :276-286, BPR :583-678, FunkSVD :289-390,
 *            apply :773-832, adaptive_gradient :838-876, samplers :881-987, getters :688-705)
 * AsySVD (:396-578) has its own handle below (K2b).
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200_mf_s* b200_mf_t;

enum b200_mf_algorithm { B200_MF_BPR = 0, B200_MF_FUNK_SVD = 1 };
enum b200_sgd_mode { B200_SGD = 0, B200_ADAGRAD = 1, B200_RMSPROP = 2, B200_ADAM = 3 };
enum b200_sampler { B200_SAMPLER_GLIBC = 0, /* host replay of srand(seed)/rand(), the reference's stream */
                    B200_SAMPLER_PHILOX = 1 /* Philox4x32-10 on the device, same acceptance rules */ };

/* URM: CSR, sorted indices (pyx:118-119).  h_user_factors / h_item_factors: the initial factors, row-major
 * [n_users x f] / [n_items x f] doubles -- the caller draws them exactly as pyx:177-178 does (numpy legacy RNG)
 * so that parity runs start from the reference's own initial point.  has_seed == 0 mirrors random_seed=None.
 * hogwild != 0: no mini-batch barrier, every sample updates at once (batch_size is then only used for the
 * per-epoch sample count, pyx:586 / :292). */
int b200_mf_create(b200_mf_t* out, int64_t n_users, int64_t n_items, int64_t nnz, const int32_t* h_indptr,
                   const int32_t* h_indices, const float* h_data, int n_factors, int algorithm, int batch_size,
                   float negative_interactions_quota, float learning_rate, int use_bias, float user_reg,
                   float item_reg, float bias_reg, float positive_reg, float negative_reg, int sgd_mode,
                   float gamma, float beta_1, float beta_2, const double* h_user_factors,
                   const double* h_item_factors, int has_seed, uint32_t random_seed, int sampler, int hogwild);
int b200_mf_destroy(b200_mf_t h);
/* epochIteration_Cython() (pyx:276-286): (n_users or nnz)/batch_size + 1 mini-batches */
int b200_mf_epoch(b200_mf_t h, void* stream);
/* multi-GPU data parallelism: this rank's device sampler draws users from [user_lo, user_hi) only (so user rows are
 * never shared between ranks) and an epoch consumes samples_per_epoch samples (0 = the reference's epoch length); stream_id (the rank)
 * selects a distinct Philox stream */
int b200_mf_set_user_shard(b200_mf_t h, int user_lo, int user_hi, int64_t samples_per_epoch, uint32_t stream_id);
int b200_mf_samples_last_epoch(b200_mf_t h, int64_t* n);
/* the (user, item, neg item | rating) stream the last epoch consumed (for replaying it through the oracle) */
int b200_mf_get_samples(b200_mf_t h, int32_t* u, int32_t* i, int32_t* j, float* r);
/* get_USER_factors / get_ITEM_factors / get_USER_bias / get_ITEM_bias / get_GLOBAL_bias (pyx:688-705);
 * any pointer may be NULL; doubles like the reference's arrays */
int b200_mf_get_factors(b200_mf_t h, double* user_factors, double* item_factors, double* user_bias,
                        double* item_bias, double* global_bias);
/* device pointers of the fp32 factor matrices (scoring without a host round trip) */
int b200_mf_device_factors(b200_mf_t h, float** d_user_factors, float** d_item_factors);
/* device time of the last epoch (sampling kernel + epoch kernel), CUDA events on the launching stream */
int b200_mf_last_epoch_ms(b200_mf_t h, float* ms);
/* Multi-GPU exchange of a replicated factor table (SURVEY.md 8(e), K2: "V (item factors) replicated"; the reference has
 * no distributed path).  n = elements (a multiple of 4), all pointers on the device, fp32.
 *   snapshot:  own = V - B;  sum = own (the caller all-reduces `sum` in place);  B = V
 *   apply:     t = sum - own (the other ranks' movement);  V += t (RED.ADD: the trainer may be writing V);  B += t */
int b200_mf_delta_snapshot_device(const float* d_V, float* d_B, float* d_own, float* d_sum, int64_t n, void* stream);
int b200_mf_delta_apply_device(float* d_V, float* d_B, const float* d_sum, const float* d_own, int64_t n, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K2b: AsymmetricSVD epochs  (SURVEY.md 8(f).4)
 * replaces  MatrixFactorization_Cython_Epoch.pyx:396-578 epochIteration_Cython_ASY_SVD_SGD (algorithm_name="ASY_SVD",
 *           batch size 1 :399) with sampleMSE_Cython :881-938 and adaptive_gradient :838-876
 * Both factor tables have one row per ITEM (pyx:163-166): h_profile_factors is the reference's USER_factors (the Y of the
 * paper, summed over a user's profile), h_item_factors its ITEM_factors; row-major [n_items x n_factors] doubles drawn by the
 * caller exactly as pyx:177-178 does.  The sample stream is the reference's own: srand(random_seed) / rand() replayed on the
 * host (has_seed == 0: glibc's default stream, seed 1).  One epoch = nnz + 1 samples (pyx:402), strictly in order.
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200_asysvd_s* b200_asysvd_t;
int b200_asysvd_create(b200_asysvd_t* out, int64_t n_users, int64_t n_items, int64_t nnz, const int32_t* h_indptr,
                       const int32_t* h_indices, const float* h_data, int n_factors, double negative_interactions_quota,
                       float learning_rate, int use_bias, float user_reg, float item_reg, float bias_reg, int sgd_mode,
                       float gamma, float beta_1, float beta_2, const double* h_profile_factors,
                       const double* h_item_factors, int has_seed, uint32_t random_seed);
int b200_asysvd_destroy(b200_asysvd_t h);
int b200_asysvd_epoch(b200_asysvd_t h, void* stream);
/* the (user, item, rating) stream of the last epoch, nnz + 1 entries each */
int b200_asysvd_get_samples(b200_asysvd_t h, int32_t* u, int32_t* i, float* r);
/* get_USER_factors (= Y, n_items rows) / get_ITEM_factors / get_USER_bias / get_ITEM_bias / get_GLOBAL_bias; any may be NULL */
int b200_asysvd_get_factors(b200_asysvd_t h, double* profile_factors, double* item_factors, double* user_bias,
                            double* item_bias, double* global_bias);
int b200_asysvd_last_epoch_ms(b200_asysvd_t h, float* ms);

/* ------------------------------------------------------------------------------------------------
 * K3: SLIM-BPR epochs on a dense / symmetric item-item matrix  (hot path ii)
 * replaces  SLIM_BPR/Cython/SLIM_BPR_Cython_Epoch.pyx:60-480  (ctor :88-134, epochIteration_Cython :211-335,
 *           sampleBPR_Cython :436-480, adaptive_gradient :395-433, get_S :340-388, Triangular_Matrix :1223-1415)
 * The tree-sparse training mode (train_with_sparse_weights, Sparse_Matrix_Tree_CSR :579-1031) keeps its semantics on the
 * dense array: b200_slim_enable_tree / b200_slim_tree_prune below.
 * ------------------------------------------------------------------------------------------------ */
typedef struct b200_slim_s* b200_slim_t;

/* URM_mask: CSR, sorted indices (pyx:100-119).  S starts at zero.  hogwild == 0: the batch-1 recursion in stream
 * order on one CTA (the reference's semantics); hogwild != 0: all SMs, atomics, no ordering between samples. */
int b200_slim_create(b200_slim_t* out, int64_t n_users, int64_t n_items, int64_t nnz, const int32_t* h_indptr,
                     const int32_t* h_indices, float learning_rate, float li_reg, float lj_reg, int symmetric,
                     int sgd_mode, float gamma, float beta_1, float beta_2, int has_seed, uint32_t random_seed,
                     int sampler, int hogwild);
int b200_slim_destroy(b200_slim_t h);
/* epochIteration_Cython() (pyx:211-335): n_users samples */
int b200_slim_epoch(b200_slim_t h, void* stream);
int b200_slim_get_samples(b200_slim_t h, int32_t* u, int32_t* i, int32_t* j);
/* the full n_items x n_items view get_S() starts from (diagonal zeroed pyx:345-355, symmetric mode mirrored
 * pyx:1363-1372), row-major fp32, to a host buffer and/or a device buffer (either may be NULL) */
int b200_slim_get_S_dense(b200_slim_t h, float* h_out, float* d_out);
int b200_slim_last_epoch_ms(b200_slim_t h, float* ms);
/* train_with_sparse_weights=True (pyx:111-134): call once after b200_slim_create (symmetric = 0, hogwild = 0) and before the
 * first epoch.  A byte map records the cells the reference's row trees would hold (add_value, pyx:617-680); every epoch cuts
 * the rows that hold >= topK cells back to their topK largest after the samples n with n % (n_users / 5) == 0
 * (rebalance_tree, pyx:318-319, :782-802; ties keep the higher column like the reference's stable qsort, :991).
 * topK = 0 is the reference's topK=False: nothing is ever removed. */
int b200_slim_enable_tree(b200_slim_t h, int topK);
/* the selection get_S() applies IN PLACE before it emits the rows (get_scipy_csr(TopK), pyx:762-763); touch_diagonal != 0
 * first creates the diagonal cells with value 0 like get_S does (pyx:349-350) -- they count towards a row's length */
int b200_slim_tree_prune(b200_slim_t h, int touch_diagonal, void* stream);
/* Column-sharded S for catalogues whose dense S does not fit one GPU (SURVEY.md 8(e) K3; the reference's answer to that is
 * the tree-sparse mode, pyx:509-1031): this handle owns S[:, col_lo:col_hi) as an [n_items, col_hi - col_lo] slab (full
 * matrix, not the triangular storage).  Every rank creates one with the SAME random_seed and draws the same Philox sample
 * stream (n_users samples per epoch, pyx:231).  A step over samples [first, first + n_batch) of the epoch:
 *   partial: d_x[n] = sum over this rank's columns of S[i, s] - S[j, s], s in the user's profile   (pyx:242-255)
 *   (the caller adds the ranks' d_x: one all-reduce of n_batch floats)
 *   apply:   gradient from the summed x (pyx:258-263), update of the cells this rank owns            (pyx:266-304)
 * n_batch = 1 is the reference's recursion exactly; the apply that completes the epoch advances it. */
int b200_slim_create_sharded(b200_slim_t* out, int64_t n_users, int64_t n_items, int64_t nnz, const int32_t* h_indptr,
                             const int32_t* h_indices, float learning_rate, float li_reg, float lj_reg, int sgd_mode,
                             float gamma, float beta_1, float beta_2, uint32_t random_seed, int col_lo, int col_hi);
int b200_slim_shard_partial_device(b200_slim_t h, int64_t first, int n_batch, float* d_x, void* stream);
int b200_slim_shard_apply_device(b200_slim_t h, int64_t first, int n_batch, const float* d_x_sum, void* stream);
/* the slab on the device and its column range */
int b200_slim_shard_device(b200_slim_t h, float** d_S, int* col_lo, int* col_hi);

/* ------------------------------------------------------------------------------------------------
 * K1b: top-K along the rows / columns of a dense fp32 n x n matrix on the device
 * replaces  Base/Recommender_utils.py:55-122 similarityMatrixTopK            (along_columns=1, mode 0)
 *           SLIM_BPR_Cython_Epoch.pyx:1335-1415 / :371,386 row top-K of get_S (along_columns=0, mode 1 / 0)
 * mode 0: the K largest of the non-zero values; mode 1: the K largest over all cells, zeros then dropped.
 * Output table [n, K] like b200_sim_compute_device (line = row or column, idx = position along it).
 * ------------------------------------------------------------------------------------------------ */
enum b200_topk_mode { B200_TOPK_NONZERO = 0, B200_TOPK_ZEROS_OUTRANK = 1,
                      /* SLIMElasticNetRecommender.py:99-107: the min(nnz - 1, K) largest non-zero values of a line */
                      B200_TOPK_NONZERO_DROP_LAST = 2 };
int b200_dense_topk_device(const float* d_matrix, int n, int K, int along_columns, int mode, int32_t* d_idx,
                           float* d_val, int32_t* d_cnt, void* stream);
/* mode 0 over the lines of a rectangular dense matrix (line l starts at l * stride_line, its cells are stride_inner apart);
 * reported positions are cell index + index_offset -- the per-row top-K of one column slab of a sharded matrix */
int b200_dense_topk_rect_device(const float* d_matrix, int n_lines, int n_inner, int64_t stride_line, int64_t stride_inner,
                                int index_offset, int K, int mode, int32_t* d_idx, float* d_val, int32_t* d_cnt, void* stream);
/* the same selection over the lines of a compressed sparse n x n matrix on the device (CSC columns or CSR rows):
 * line l holds entries d_ptr[l]..d_ptr[l+1] with positions d_line_idx[] and values d_vals[] */
int b200_sparse_topk_device(int n, const int32_t* d_ptr, const int32_t* d_line_idx, const float* d_vals, int K,
                            int mode, int32_t* d_idx, float* d_val, int32_t* d_cnt, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K6: batch scoring behind _compute_item_score / recommend
 * replaces  Base/BaseSimilarityMatrixRecommender.py:73-92 (and :97-116)   URM[users] . W_sparse -> dense block
 *           Base/BaseMatrixFactorizationRecommender.py:38-70              U[users] . V^T (+ biases)
 *           Base/BaseRecommender.py:164-169, :189-196                      seen -> -inf, per-row top-`cutoff`
 * All pointers are DEVICE pointers; d_out / d_scores are dense row-major [n_users_block, n_items] fp32.
 * ------------------------------------------------------------------------------------------------ */
/* d_out[b, :] = sum over (i, r) in row d_users[b] of CSR A of r * (row i of B); B is CSR, or -- with d_b_ptr and
 * d_b_idx NULL -- a dense row-major [*, n_out_cols] matrix in d_b_val (EASE_R's dense W, EASE_R_Recommender.py:87-106) */
int b200_score_spmm_device(const int32_t* d_users, int n_users_block, const int32_t* d_a_ptr, const int32_t* d_a_idx,
                           const float* d_a_val, const int32_t* d_b_ptr, const int32_t* d_b_idx, const float* d_b_val,
                           int n_out_cols, float* d_out, void* stream);
/* d_out[cols, rows] = transpose of d_in[rows, cols] (item factors are scored from their transpose) */
int b200_transpose_device(const float* d_in, int rows, int cols, float* d_out, void* stream);
/* d_out[b, j] = U[d_users[b], :] . VT[:, j] (+ global + user + item bias when the three pointers are non-NULL) */
int b200_score_mf_device(const int32_t* d_users, int n_users_block, const float* d_user_factors,
                         const float* d_item_factors_T, int n_factors, int n_items, const float* d_user_bias,
                         const float* d_item_bias, const float* d_global_bias, float* d_out, void* stream);
/* -inf on items outside d_items_keep (nullable, n_items bytes) and on the seen items of each user (nullable URM) */
int b200_score_mask_device(const int32_t* d_users, int n_users_block, const int32_t* d_urm_ptr, const int32_t* d_urm_idx,
                           const unsigned char* d_items_keep, int n_items, float* d_scores, void* stream);
/* per row the `cutoff` (<= 1024) best items, best first, ties by ascending item index: [n_rows, cutoff] tables */
int b200_score_topn_device(const float* d_scores, int n_rows, int n_items, int cutoff, int32_t* d_items,
                           float* d_item_scores, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K7: SLIM ElasticNet  (SURVEY.md 8(f).4)
 * replaces  SLIM_ElasticNet/SLIMElasticNetRecommender.py:77-131 -- one sklearn ElasticNet(precompute=True, fit_intercept=False,
 *           selection='random', max_iter=100, tol=1e-4).fit(URM with column j zeroed, URM[:, j]) per item
 * d_G: the Gram matrix X^T X, [n_items x n_items] fp32 (its diagonal is not read), d_diag: the sum of squares of every column.
 * For item j the coordinate descent runs on Q = G without row / column j, q = G[:, j], with sklearn's stopping rule
 * (max|dw| / max|w| < tol -> duality gap < tol * ||y||^2) in CYCLIC coordinate order (the reference's order is drawn from an
 * unseeded generator).  d_coef_T[j, :] receives the coefficients of item j (dense; top-K selection: b200_dense_topk_device,
 * mode B200_TOPK_NONZERO_DROP_LAST), d_n_iter (nullable) the passes used.
 * ------------------------------------------------------------------------------------------------ */
int b200_slim_enet_device(const float* d_G, const float* d_diag, int n_items, int64_t n_users, double l1_ratio, double alpha,
                          int positive_only, int max_iter, float tol, float* d_coef_T, int32_t* d_n_iter, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K5: EASE^R closed form  (hot path iii)
 * replaces  EASE_R/EASE_R_Recommender.py:55-69
 * ------------------------------------------------------------------------------------------------ */
/* In-place inverse of a symmetric positive definite matrix on the device through a blocked Cholesky factorisation
 * (replaces np.linalg.inv, EASE_R_Recommender.py:65).  d_A: [n_pad, n_pad] row-major fp32, n_pad a multiple of 128
 * (pad with an identity block); d_work: 2 * n_pad * n_pad floats. */
int b200_spd_inverse_device(float* d_A, int n_pad, float* d_work, void* stream);
/* TEST HOOK: one GEMM of the blocked inverse through tensor-core GEMM version 1 (the default, gemm_tc.cuh) or 2
 * (gemm_tc2.cuh: pre-packed hi/lo TF32 operands fed by cp.async.bulk, opt-in via B200REC_GEMM=2).
 * kind 0: C = alpha A B^T + beta C (A [M,K], B [N,K]); kind 1: C = alpha A B + beta C (B [K,N]);
 * kind 2: C = alpha A^T B + beta C with k >= max(row block, column block) only (A [K,M], B [K,N]; the L^T L product).
 * Row-major device pointers; M, N multiples of 128, K a multiple of 32. */
int b200_debug_gemm_device(int version, int kind, int M, int N, int K, float alpha, const float* d_A, int lda,
                           const float* d_B, int ldb, float beta, float* d_C, int ldc, void* stream);
/* d_G: dense [n_items, n_items] Gram block X^T X (b200_sim_compute_dense_device with normalize=0, shrink=0); the
 * diagonal is replaced by item popularity (stored-entry count per column of the URM, :62-63) + l2_norm, the matrix is
 * inverted, and B[i, j] = P[i, j] / (-P[j, j]), B[j, j] = 0 is written to h_B (host) and/or d_B (device). */
int b200_ease_from_gram_device(const float* d_G, int n_items, const int32_t* d_urm_indices, int64_t nnz, float l2_norm,
                               float* h_B, float* d_B, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K4: implicit ALS half epoch  (hot path iii)
 * replaces  MatrixFactorization/IALSRecommender.py:137-201 (_run_epoch user loop or item loop + _update_row)
 * For every row r in d_rows (the warm users, or the warm items): profile = d_idx[d_ptr[r] .. d_ptr[r+1]),
 * confidences c = d_conf[...] (the C or C_csc matrix, :99-123), Y = the other side's factors [n_other, f] fp64:
 *     X[r, :] = (Y^T Y + Y_p^T diag(c - 1) Y_p + reg I)^-1  Y_p^T c
 * Rows not listed keep their previous contents (cold rows, :143).  d_YtY_work: f * f doubles of scratch.
 * n_factors <= 256 (up to 208 the packed fp64 system lives in shared memory; above, its last rows spill to a per-CTA
 * slab of global memory and the Gram accumulation takes two passes over the profile).
 * ------------------------------------------------------------------------------------------------ */
int b200_ials_half_epoch_device(const int32_t* d_rows, int n_solve, const int32_t* d_ptr, const int32_t* d_idx,
                                const float* d_conf, const double* d_Y, int n_other, int n_factors, double reg,
                                double* d_X, double* d_YtY_work, void* stream);

/* ------------------------------------------------------------------------------------------------
 * URM feature weighting in front of the KNN similarity  (SURVEY.md 8(f).3)
 * replaces  Base/IR_feature_weighting.py:13-51 okapi_BM_25 and :56-78 TF_IDF as KNN/ItemKNNCFRecommender.py:42-50 and
 *           KNN/UserKNNCFRecommender.py:43-51 apply them: weighting(URM.T).T -- items are the documents, users the terms.
 * d_data (the CSR values of the n_users x n_items URM on the device) is rewritten in place.
 * ------------------------------------------------------------------------------------------------ */
enum b200_weighting { B200_WEIGHT_BM25 = 0, B200_WEIGHT_TFIDF = 1 };
int b200_feature_weighting_device(int mode, int n_users, int n_items, int64_t nnz, const int32_t* d_indptr,
                                  const int32_t* d_indices, float* d_data, float K1, float B, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Evaluation inner loop on the device  (SURVEY.md 8(f).1)
 * replaces  Base/Evaluation/Evaluator.py:305-388 _compute_metrics_on_recommendation_list and the per-user metric
 *           functions of Base/Evaluation/metrics.py (:65-287, :615-716) for one block of users.
 * d_rec_items / d_rec_scores: the [n_block, max_cutoff] tables of b200_score_topn_device (a -inf score ends a list);
 * test URM in CSR with sorted indices; d_cutoffs: n_cutoffs ascending list lengths; d_idcg: [n_users, n_cutoffs] ideal
 * DCG of every user (metrics.py:268); d_item_novelty / d_item_pop_norm: the per-item terms of Novelty (:651) and
 * AveragePopularity (:686).  Accumulates (atomically, across calls) into d_acc [n_cutoffs, B200_EVAL_NACC] doubles
 * and the per-item counters d_rec_count / d_hit_count [n_cutoffs, n_items] (times recommended / recommended and
 * relevant), from which the global-distribution metrics (coverage, Gini, Shannon, Herfindahl, mean inter-list) follow.
 * ------------------------------------------------------------------------------------------------ */
enum b200_eval_slot {
  B200_EVAL_PRECISION = 0, B200_EVAL_PRECISION_RECALL_MIN_DEN = 1, B200_EVAL_RECALL = 2, B200_EVAL_MAP = 3,
  B200_EVAL_MAP_MIN_DEN = 4, B200_EVAL_MRR = 5, B200_EVAL_NDCG = 6, B200_EVAL_HIT_RATE = 7, B200_EVAL_ARHR = 8,
  B200_EVAL_NOVELTY = 9, B200_EVAL_AVERAGE_POPULARITY = 10, B200_EVAL_USERS_WITH_RECS = 11, B200_EVAL_N_USERS = 12,
  B200_EVAL_NACC = 16
};
int b200_eval_accumulate_device(const int32_t* d_users, int n_block, const int32_t* d_rec_items, const float* d_rec_scores,
                                int max_cutoff, const int32_t* d_test_ptr, const int32_t* d_test_idx,
                                const float* d_test_val, const int32_t* d_cutoffs, int n_cutoffs, const double* d_idcg,
                                const double* d_item_novelty, const double* d_item_pop_norm, int n_items, double* d_acc,
                                int32_t* d_rec_count, int32_t* d_hit_count, void* stream);

/* ------------------------------------------------------------------------------------------------
 * K8: randomized truncated SVD (PureSVD)
 * replaces  MatrixFactorization/PureSVDRecommender.py:36-55 -- sklearn.utils.extmath.randomized_svd(URM_train,
 *           n_components=num_factors, random_state=random_seed) with its defaults (n_oversamples=10, n_iter='auto',
 *           power_iteration_normalizer='auto', transpose='auto', flip_sign=True)
 * Dense blocks are row-major fp32 [rows, ld] with ld a multiple of 4 (<= 512) and l active columns; columns l..ld-1 are zero.
 * A (n_rows x n_cols) is the URM, or its transpose (sklearn's transpose rule: the URM when it is not wide).
 * ------------------------------------------------------------------------------------------------ */
/* d_Y[r, :] = sum over the stored entries (r, c, v) of the CSR matrix of v * d_X[c, :], all ld columns (the safe_sparse_dot
 * products A @ Q and A.T @ Q of sklearn's _randomized_range_finder; A.T through the CSR of b200_csr_transpose_device) */
int b200_csr_spmm_dense_device(int64_t n_rows, const int32_t* d_ptr, const int32_t* d_idx, const float* d_val, const float* d_X,
                               int ld, float* d_Y, void* stream);
/* CSR of the transpose (scipy's tocsc(): inside a column the rows ascend); d_t_ptr: n_cols + 1, d_t_idx / d_t_val: nnz */
int b200_csr_transpose_device(int64_t n_rows, int64_t n_cols, int64_t nnz, const int32_t* d_ptr, const int32_t* d_idx,
                              const float* d_val, int32_t* d_t_ptr, int32_t* d_t_idx, float* d_t_val, void* stream);
/* In place: the n x l block d_Y becomes an orthonormal basis of its column span (the LU / QR normalisers of
 * _randomized_range_finder; shifted CholeskyQR3 here).  Deficient columns are refilled with seeded Gaussian columns;
 * *h_breakdowns (nullable) receives how many were.  l <= min(n, 512). */
int b200_orthonormalize_device(int64_t n, int l, int ld, float* d_Y, uint32_t seed, int32_t* h_breakdowns, void* stream);
/* _randomized_range_finder + the projection B = Q^T A of randomized_svd: from d_omega [n_cols, ld] (the Gaussian start),
 * n_iter x (A Q, normalise, A^T Q, normalise), then d_Q [n_rows, ld] = orthonormal basis of A Q, and B^T = A^T Q = Qb Rb with
 * d_Qb [n_cols, ld] orthonormal and d_Rb [l, l] fp64 row-major.  h_ms (nullable, 2 floats): device ms in SpMM / in
 * orthonormalisation; h_breakdowns (nullable): deficient columns refilled over the whole call. */
int b200_rsvd_range_device(int64_t n_rows, int64_t n_cols, const int32_t* d_ptr, const int32_t* d_idx, const float* d_val,
                           const int32_t* d_t_ptr, const int32_t* d_t_idx, const float* d_t_val, const float* d_omega, int l, int ld,
                           int n_iter, uint32_t seed, float* d_Q, float* d_Qb, double* d_Rb, float* h_ms, int32_t* h_breakdowns,
                           void* stream);
/* With svd(Rb^T) = W diag(sigma) Z^T computed on the host (h_W, h_Z: [l, l] fp64 row-major, h_sigma: the first k values):
 * A's left factor Q W[:, :k] and right factor Qb Z[:, :k] go to d_user_factors [n_users, k] / d_item_factors [n_items, k]
 * (swapped when `transpose`, A = URM^T), svd_flip makes the largest-magnitude entry of every user-side column positive (first
 * row on ties), and `scale_item_side` multiplies the item-side columns by sigma (PureSVD's ITEM_factors = (diag(s) Vt)^T). */
int b200_rsvd_finish_device(int64_t n_rows, int64_t n_cols, const float* d_Q, const float* d_Qb, int l, int ld, const double* h_W,
                            const double* h_Z, const float* h_sigma, int k, int transpose, int scale_item_side,
                            float* d_user_factors, float* d_item_factors, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200REC_H_ */
