/* cubecobra_b200.h -- C ABI of libcubecobra_b200.so (sm_100a only).
 *
 * The reference (CubeArtisan/CubeCobraRecommender) is pure Python and defines no FFI;
 * these entry points are what a ctypes binding inside the reference's own functions
 * would call (INTEGRATION.md shows the stubs).  Each group cites the reference code it
 * replaces as file:line relative to the reference repository root.
 *
 * Conventions
 *   - every function returns int: CC_OK (0) or a negative CC_ERR_*; the message is
 *     available per host thread from cc_last_error();
 *   - unless a name ends in `_host`, every pointer is a DEVICE pointer on the current
 *     CUDA device; the caller owns every buffer, including workspaces (sizes from the
 *     matching *_bytes() helper); nothing is allocated, freed or synchronised behind the
 *     caller's back (the `_host` entry points are the exception: they own their device
 *     scratch and return after their stream has drained);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it;
 *   - matrices are row-major with an explicit leading dimension in ELEMENTS;
 *   - re-entrant across devices: one host thread (or process) per GPU, no global state.
 */
#ifndef CUBECOBRA_B200_H
#define CUBECOBRA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CC_VERSION 100
#define CC_OK 0
#define CC_ERR_ARGUMENT (-1)
#define CC_ERR_CUDA (-2)
#define CC_ERR_DEVICE (-3)
#define CC_ERR_UNSUPPORTED (-4)

const char* cc_last_error(void);
int cc_version(void);
int cc_device_check(void);

/* ------------------------------------------------------------------------------------
 * (1) Co-occurrence / conditional-probability graph
 *     replaces utils.create_adjacency_matrix          src/non_ml/utils.py:75-92
 *              y_mtx (M-hat) construction             src/ml/train.py:69-71
 *              DataGenerator.neg_sampler              src/ml/generator.py:30
 * Cubes arrive as CSR (indptr int64 [K+1], indices int32 [nnz]) instead of the dense
 * float64 (K, C) matrix of utils.build_cubes (src/non_ml/utils.py:57-73).
 * ---------------------------------------------------------------------------------- */
int64_t cc_bits_words(int64_t num_cubes);   /* rows  of the bit matrix (32 cubes per word, padded) */
int64_t cc_bits_cpad(int32_t num_cards);    /* columns of the bit matrix (cards, padded to the tile) */
/* bits: uint32 [cc_bits_words(K)][cc_bits_cpad(C)], zeroed and filled; *bad_flag != 0 afterwards
 * if a card index was outside [0, C). */
int cc_bitpack_cubes(const int64_t* indptr, const int32_t* indices, int64_t num_cubes, int32_t num_cards,
                     uint32_t* bits, int* bad_flag, void* stream);
/* counts[i][j] (int32, ld >= C) = number of cubes containing both i and j; accumulate != 0 adds. */
int cc_cooc_count(const uint32_t* bits, int64_t num_cubes, int32_t num_cards, int32_t* counts, int64_t ld,
                  int accumulate, void* stream);
/* The same counts on the tensor cores: cubes are expanded to a K-major 0/1 byte matrix X^T [C][chunk] (in the
 * caller's workspace, cc_cooc_tc_workspace_bytes) and contracted as X^T X with tcgen05.mma kind::i8 (int32
 * accumulators, exact), upper-triangle 256x256 tiles mirrored by the epilogue; cubes are processed in chunks of
 * cc_cooc_tc_chunk_cubes.  counts: 16-byte aligned, ldc % 4 == 0.  bad (optional) is set to 1 on an
 * out-of-range card id.  Duplicate ids inside a cube collapse, as in utils.build_cubes (utils.py:66-71). */
int64_t cc_cooc_tc_chunk_cubes(int64_t num_cubes);
int64_t cc_cooc_tc_workspace_bytes(int64_t num_cubes, int32_t num_cards);
int cc_cooc_count_tc(const int64_t* indptr, const int32_t* indices, int64_t num_cubes, int32_t num_cards,
                     void* workspace, int64_t workspace_bytes, int32_t* counts, int64_t ldc, int accumulate,
                     int32_t* bad, void* stream);
/* From counts: M (float64, nullable), M-hat (float32, nullable), rowsum of y (float64, nullable). */
int cc_row_normalise(const int32_t* counts, int64_t ld, int32_t num_cards, double* m64, int64_t ld_m,
                     float* mhat, int64_t ld_mhat, double* rowsum, int has_force_diag, double force_diag,
                     void* stream);
/* The same on a ROW BLOCK: counts / m64 / mhat / rowsum hold rows [row0, row0 + nrows) of the (C, C) matrices -- a
 * rank's shard after the int32 counts of a cube-sharded build were reduce-scattered by row block over NVLink instead
 * of all_reduced (a row of M needs nothing but its own counts row, whose diagonal element sits in column row0 + i). */
int cc_row_normalise_rows(const int32_t* counts, int64_t ld, int32_t row0, int32_t nrows, int32_t num_cards, double* m64,
                          int64_t ld_m, float* mhat, int64_t ld_mhat, double* rowsum, int has_force_diag,
                          double force_diag, void* stream);
int64_t cc_col_mass_workspace_bytes(int32_t num_cards);
/* neg_sampler[j] = sum_i Mhat[i][j] / sum(Mhat), float64, deterministic order. */
int cc_col_mass(const int32_t* counts, int64_t ld, int32_t num_cards, const double* rowsum, double* workspace,
                double* neg_sampler, void* stream);
/* Row-block form: col_mass[j] = sum of M-hat[i][j] over the block's rows, not normalised; the blocks' vectors are summed
 * over the ranks (an all_reduce of C doubles) and cc_col_mass_scale divides by the total (generator.py:30). */
int cc_col_mass_rows(const int32_t* counts, int64_t ld, int32_t row0, int32_t nrows, int32_t num_cards, const double* rowsum,
                     double* workspace, double* col_mass, void* stream);
int cc_col_mass_scale(double* col_mass, int32_t num_cards, void* stream);
/* Host-buffer drop-in for utils.create_adjacency_matrix: CSR in, float64 (C, C) out
 * (and the int32 counts if counts_host != NULL).  H2D + kernels + D2H inside the call. */
int cc_create_adjacency_matrix_host(const int64_t* indptr_host, const int32_t* indices_host, int64_t num_cubes,
                                    int32_t num_cards, int has_force_diag, double force_diag, double* m_host,
                                    int32_t* counts_host);

/* ------------------------------------------------------------------------------------
 * (2) Graph scoring and masked top-N
 *     replaces simple_recs                            src/scripts/recommend.py:7-18
 *              simple_cuts                            src/scripts/cut_cards.py:7-18
 *              ranking walk of ml_recommend           src/scripts/ml_recommend.py:87-104
 *                                                     web/ml_recommend_web.py:46-60
 * Scores are summed in NumPy's pairwise order so float64 scores are bit-identical.
 * Tie rule: descending -> larger index first; ascending -> smaller index first
 * (== numpy argsort(kind='stable'), reversed for descending).
 * ---------------------------------------------------------------------------------- */
int64_t cc_pairwise_leaf_count(int64_t n_rows);
/* plan_host: int32 [total_leaves][4]; leaf_ptr_host: int32 [batch+1] */
int cc_pairwise_plan_host(const int64_t* row_ptr_host, int32_t batch, int32_t* plan_host, int32_t* leaf_ptr_host);
/* scores[b][j] = sum over rows[row_ptr[b]..row_ptr[b+1]) of M[row][j]  (M[i][i] read as 0 if zero_diag);
 * partial_ws: float64 [total_leaves][C]. */
int cc_score_gather_f64(const double* m, int64_t ld, int32_t num_cards, const int32_t* rows, const int64_t* row_ptr,
                        int32_t batch, const int32_t* plan, const int32_t* leaf_ptr, int32_t total_leaves,
                        int zero_diag, double* partial_ws, double* scores, int64_t ld_scores, void* stream);
int64_t cc_topn_workspace_bytes(int32_t num_cards, int32_t batch, int32_t n, int is_f64);
/* Per cube b: rank the cards NOT listed in mask (mode_only_listed == 0) or ONLY the listed ones (== 1);
 * out_ids int32 [batch][n] (-1 padded), out_vals [batch][n] (nullable), out_count int32 [batch] (nullable). */
int cc_topn_masked_f32(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                       const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n, void* workspace,
                       int64_t workspace_bytes, int32_t* out_ids, float* out_vals, int32_t* out_count, void* stream);
/* float32 with n <= 128 runs as a CTA-per-cube row select (the row is staged in shared memory by bulk asynchronous
 * copies, double-buffered; needs ld % 4 == 0, a 16-byte aligned base and C <= ~26 000) or, for rows that do not
 * qualify, as a warp-per-cube streaming select (one pass over the row); larger n and float64 use the radix select /
 * full bitonic ranking.  All of them implement one total order on (score, index).  NaN scores: the row select never
 * selects them.  cc_topn_set_algo: 0 = automatic (default: the row select with two CTAs per SM when the rows qualify --
 * in its register form when the whole row is ranked and holds at most 22 528 cards: group extremes kept in registers,
 * one diverged block per warp in the second sweep, counting ranks summed over neighbouring lanes; 92 us per 4096 rows of
 * 20 884 scores against 103 us), 1 = streaming select, 2 / 3 = row select with both sweeps over shared memory (one CTA
 * per SM with two row buffers / two CTAs per SM), 4 = the register form (tests compare all of them).
 * cc_topn_masked_sigmoid_f32 takes LOGITS, ranks sigmoid(logit) (the float32
 * probabilities the reference ranks, ml_recommend.py:78-104) and returns the winners' probabilities; n <= 128.
 * cc_topn_set_force_radix(1) pins float32 top-N to the radix kernel (tests compare the two). */
int cc_topn_masked_sigmoid_f32(const float* logits, int64_t ld, int32_t num_cards, int32_t batch,
                               const int64_t* mask_ptr, const int32_t* mask_idx, int mode_only_listed, int descending,
                               int32_t n, int32_t* out_ids, float* out_probs, int32_t* out_count, void* stream);
int cc_topn_set_force_radix(int on);
int cc_topn_set_algo(int algo);
/* Diagnostic build of the row select (fused sigmoid, descending): same results, plus per-phase clock64() sums of each
 * CTA's thread 0 in prof (int64 [cc_topn_rowselect_profile_grid(batch, variant)][10], device memory).  variant 0 = one
 * CTA per SM with two row buffers, 1 = two CTAs per SM with one, 2 = the next revision (algo 4) in the shape of 1. */
int64_t cc_topn_rowselect_profile_grid(int32_t batch, int variant);
int cc_topn_rowselect_profile(const float* logits, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                              const int32_t* mask_idx, int32_t n, int variant, int32_t* out_ids, float* out_probs,
                              int32_t* out_count, long long* prof, void* stream);
/* In-cube ("cuts") scores for a batch (src/scripts/ml_recommend.py:105-108, web/ml_recommend_web.py:61-64: results[idx] for
 * every in-cube idx): out[p] = scores[b][idx[p]] for the CSR entries p in [row_ptr[b], row_ptr[b+1]) of cube b, through
 * the float32 sigmoid when apply_sigmoid != 0 (scores are logits then).  out: float32 [row_ptr[batch]]. */
int cc_cuts_gather_f32(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* row_ptr,
                       const int32_t* idx, int apply_sigmoid, float* out, void* stream);
/* Target ranks for leave-k-out evaluation.  Per cube b the candidates are the cards of [0, C) NOT listed in mask row b;
 * for every entry p in [target_ptr[b], target_ptr[b+1]), out_rank[p] is the 0-based position of card target_idx[p]
 * among them in the descending order of cc_topn_masked_f32(descending = 1) / cc_topn_masked_sigmoid_f32: larger
 * score first, ties -> larger index first, with apply_sigmoid != 0 the float32 sigmoid of the logits.  So a target of
 * rank r < n is the one those selects return at slot r.  Targets are candidates too (a hidden card ranks behind the
 * other hidden cards that beat it); a target listed in the mask or outside [0, C) gets -1; duplicate entries get the
 * same rank.  Any number of targets per row.  NaN scores are outside the contract.  One CTA per cube: the row is read
 * once per 1024 targets.  out_rank: int32 [target_ptr[batch]]. */
int cc_rank_targets_f32(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                        const int32_t* mask_idx, const int64_t* target_ptr, const int32_t* target_idx, int apply_sigmoid,
                        int32_t* out_rank, void* stream);
/* The same ranks for float64 scores, in the order of cc_topn_masked_f64(descending = 1): larger score first, ties ->
 * larger index first (so a target of rank r < n is the one that select returns at slot r).  No sigmoid.  ld == 0 means
 * one score row shared by every cube (e.g. a popularity ranking); otherwise ld >= C.  Masked, out-of-range and
 * duplicate targets as in cc_rank_targets_f32; NaN scores are outside the contract.  out_rank: int32
 * [target_ptr[batch]]. */
int cc_rank_targets_f64(const double* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                        const int32_t* mask_idx, const int64_t* target_ptr, const int32_t* target_idx,
                        int32_t* out_rank, void* stream);
/* Cut ranks for offline evaluation of the cut list.  Per cube b the candidates are the distinct cards of [0, C) listed
 * in row b of list (duplicate entries count once, out-of-range entries are ignored): exactly the set
 * cc_topn_masked_*(mode_only_listed = 1) ranks.  For every entry p in [target_ptr[b], target_ptr[b+1]), out_rank[p]
 * is the 0-based position of card target_idx[p] among them in the ascending order of
 * cc_topn_masked_*(mode_only_listed = 1, descending = 0): smaller score first, ties -> smaller index first, with
 * apply_sigmoid != 0 the float32 sigmoid of the logits (saturated probabilities tie).  So a target of rank r < n is
 * the one that select returns at slot r.  A target not listed in row b, or outside [0, C), gets -1; duplicate target
 * entries get the same rank.  Any number of listed cards and targets per row; C up to 100 000 and beyond (the list
 * bitmap takes C / 8 bytes of shared memory).  NaN scores are outside the contract.  One CTA per cube, reading only
 * the row's listed scores.  out_rank: int32 [target_ptr[batch]]. */
int cc_rank_cuts_f32(const float* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* list_ptr,
                     const int32_t* list_idx, const int64_t* target_ptr, const int32_t* target_idx, int apply_sigmoid,
                     int32_t* out_rank, void* stream);
/* The same ranks for float64 scores, in the order of cc_topn_masked_f64(mode_only_listed = 1, descending = 0).  No
 * sigmoid.  ld == 0 means one score row shared by every cube (a popularity ranking); otherwise ld >= C. */
int cc_rank_cuts_f64(const double* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* list_ptr,
                     const int32_t* list_idx, const int64_t* target_ptr, const int32_t* target_idx, int32_t* out_rank,
                     void* stream);
/* Card similarity (src/scripts/similarity.py:25-29): out[r] = -cos(emb[r], emb[query]) with Keras' l2_normalize
 * (epsilon 1e-12), emb float32 [rows][ld >= dim]; rank ascending with cc_topn_masked_f32. */
int cc_cosine_neg_f32(const float* emb, int64_t ld, int32_t rows, int32_t dim, int32_t query, float* out, void* stream);
/* Card / cube similarity for many queries at once: out[q * ldo + r] = -cos(queries[q], cands[r]) with Keras'
 * l2_normalize (epsilon 1e-12), bit for bit the value cc_cosine_neg_f32 writes for that pair.  dim must be 64
 * (the encoder's width).  num_queries == 0 is a no-op.  Rank each row ascending with cc_topn_masked_f32.
 * queries float32 [num_queries][ldq], cands float32 [num_cands][ldc]: both 16-byte aligned with ldq and ldc multiples
 * of 4 (the rows are read as float4).  out float32 [num_queries][ldo >= num_cands], any alignment (16-byte aligned
 * rows, ldo % 4 == 0, are written as float4); columns [num_cands, ldo) are not written. */
int cc_cosine_neg_many_f32(const float* queries, int64_t ldq, int32_t num_queries,
                           const float* cands, int64_t ldc, int32_t num_cands, int32_t dim,
                           float* out, int64_t ldo, void* stream);
int cc_topn_masked_f64(const double* scores, int64_t ld, int32_t num_cards, int32_t batch, const int64_t* mask_ptr,
                       const int32_t* mask_idx, int mode_only_listed, int descending, int32_t n, void* workspace,
                       int64_t workspace_bytes, int32_t* out_ids, double* out_vals, int32_t* out_count, void* stream);

/* ------------------------------------------------------------------------------------
 * (3) Noise function F and batch assembly
 *     replaces DataGenerator.generate_data            src/ml/generator.py:74-103
 *              reg_indices draw                       src/ml/generator.py:47-51
 * ---------------------------------------------------------------------------------- */
int cc_alias_build_host(const double* p_host, int32_t n, float* prob_host, int32_t* alias_host);
int64_t cc_noise_smem_bytes(int32_t num_cards, int32_t max_size);
/* batch_ids (nullable): which cubes of the CSR form this batch.  Outputs: x_idx int32 [batch][x_stride],
 * x_len int32 [batch], y_bits uint32 [batch][y_words] (nullable), flips_out int32 [batch] (nullable),
 * *overflow_flag != 0 if a cube exceeded max_size (1) or x_stride (2).  step_ptr: device int64 step counter
 * (nullable = 0) mixed into the Philox counter so CUDA-graph replays draw fresh noise. */
int cc_noise(const int64_t* indptr, const int32_t* indices, const int32_t* batch_ids, int32_t batch,
             int32_t num_cards, const float* alias_prob, const int32_t* alias_idx, float noise_mean, float noise_std,
             uint64_t seed, const int64_t* step_ptr, int32_t max_size, int32_t x_stride, int32_t* x_idx,
             int32_t* x_len, uint32_t* y_bits, int64_t y_words, int32_t* flips_out, int* overflow_flag,
             float* x_dense /* nullable: dense 0/1 rows of x, [batch][ld_dense] */, int64_t ld_dense, void* stream);
/* Same, with the dense 0/1 rows optionally written as bf16 (dense_bf16 != 0; x_dense then points at bf16 rows of
 * ld_dense elements) for the bf16 form of the dW1 = x^T g1 GEMM. */
int cc_noise_ex(const int64_t* indptr, const int32_t* indices, const int32_t* batch_ids, int32_t batch,
                int32_t num_cards, const float* alias_prob, const int32_t* alias_idx, float noise_mean, float noise_std,
                uint64_t seed, const int64_t* step_ptr, int32_t max_size, int32_t x_stride, int32_t* x_idx,
                int32_t* x_len, uint32_t* y_bits, int64_t y_words, int32_t* flips_out, int* overflow_flag,
                void* x_dense, int64_t ld_dense, int dense_bf16, void* stream);
int cc_sample_reg_rows(const float* alias_prob, const int32_t* alias_idx, int32_t num_cards, int32_t n, uint64_t seed,
                       const int64_t* step_ptr, int32_t* rows, void* stream);
int cc_cubes_to_bits(const int32_t* idx, const int64_t* row_start, const int32_t* row_len, int32_t batch,
                     int32_t num_cards, uint32_t* bits, int64_t words, void* stream);
int cc_step_increment(int64_t* step_ptr, void* stream);

/* ------------------------------------------------------------------------------------
 * (4) Encoder first layer on sparse cubes (embedding bag)
 *     replaces Dense(512)(x) on 0/1 rows              src/ml/model.py:27,36 (and :122 for I[r])
 * ---------------------------------------------------------------------------------- */
int cc_bag_fwd(const float* w, int64_t ldw, int32_t hidden, const int32_t* idx, const int64_t* row_start,
               const int32_t* row_len, int32_t batch, const float* bias, float* out, int64_t ldo, int relu,
               int round_tf32, void* stream);
int cc_bag_bwd(const float* g, int64_t ldg, int32_t hidden, const int32_t* idx, const int64_t* row_start,
               const int32_t* row_len, int32_t batch, float* dw, int64_t ldw, void* stream);

/* ------------------------------------------------------------------------------------
 * (5) Dense layers
 *     replaces Dense layers of Encoder / Decoder      src/ml/model.py:27-33, 58-64
 * C[M,N] = epi(op(A) op(B)); transa: A given as [K,M]; transb: B given as [N,K].
 * epilogue order: + bias[N], relu, * (mask[M,N] > 0), then store or accumulate.
 * ---------------------------------------------------------------------------------- */
int cc_gemm_f32_simt(int transa, int transb, int m, int n, int k, const float* a, int64_t lda, const float* b,
                     int64_t ldb, float* c, int64_t ldc, const float* bias, int relu, const float* mask,
                     int64_t ldmask, int accumulate, void* stream);
/* tcgen05 tensor-core GEMM (TMA + TMEM, TMA-store epilogue).  precision: 1 = tf32 (float operands),
 * 2 = bf16 (__nv_bfloat16 operands; C, bias and mask stay float).  split_k: 0 = choose tile width and
 * K split automatically, > 1 = spread the reduction over CTAs (TMA reduce-add into C; a non-linear
 * epilogue then runs as a second elementwise pass).  tile_n: 0 (auto) | 128 | 256.  A, B and C need
 * 16-byte aligned bases and leading dimensions that are multiples of 16 bytes. */
int cc_gemm_tc(int precision, int transa, int transb, int m, int n, int k, const void* a, int64_t lda, const void* b,
               int64_t ldb, float* c, int64_t ldc, const float* bias, int relu, const float* mask, int64_t ldmask,
               int accumulate, int split_k, int tile_n, int round_tf32, void* stream);
/* Fused decoder output layer + sigmoid-BCE (model.py:64,94 + train.py:85): z = A[M,K] W[K,N] + bias is
 * never stored; dz[M][lddz] = (sigmoid(z) - y)/count (columns [N, lddz) zeroed, lddz % 32 == 0), loss_partial
 * float64 [cc_gemm_bce_partial_count(m, lddz)] holds per-(tile, warp) loss sums for cc_loss_finalize.  dbias (nullable,
 * float [n]) receives the column sums of dz, i.e. the gradient of the layer's bias (zeroed, then accumulated with float
 * atomics by the epilogue: summation order, hence the last bits, can differ between runs).  dz_bf16 != 0 (precision 2
 * only): dz is a bf16 matrix (lddz in elements), the form the bf16 dW / dX GEMMs consume.  dz == NULL: loss only
 * (evaluation) -- the same partials, nothing else written; lddz still sizes loss_partial, and dbias must be NULL and
 * dz_bf16 0 (anything else is rejected). */
int cc_gemm_bce_tc(int precision, int m, int n, int k, const void* a, int64_t lda, const void* w, int64_t ldw,
                   const float* bias, const uint32_t* ybits, int64_t ywords, double count, void* dz, int64_t lddz,
                   double* loss_partial, float* dbias, int round_tf32, int dz_bf16, void* stream);
/* The same with Keras' binary_accuracy (metrics=['accuracy'], src/ml/train.py:87) counted on the way: acc_partial
 * (nullable, float64, sized and laid out like loss_partial) receives per-(tile, warp) counts of the cells with
 * round(sigmoid(z)) == y; their sum / (B*C) is the metric Keras reports as output_1_accuracy. */
int cc_gemm_bce_tc_ex(int precision, int m, int n, int k, const void* a, int64_t lda, const void* w, int64_t ldw,
                      const float* bias, const uint32_t* ybits, int64_t ywords, double count, void* dz, int64_t lddz,
                      double* loss_partial, float* dbias, int round_tf32, int dz_bf16, double* acc_partial,
                      void* stream);
int64_t cc_gemm_bce_partial_count(int m, int lddz);
/* CTA-pair tiling of the tcgen05 GEMMs (256 x 256 tiles on two SMs, tcgen05.mma.cta_group::2):
 * -1 = the planner decides per problem (default), 0 = never, 1 = whenever the shape allows it. */
int cc_gemm_tc_set_pair_mode(int mode);
/* The planner cc_gemm_tc uses (host logic, no device work): plan[0] = tile width (128 | 256), plan[1] = K split,
 * plan[2] = CTAs per tile (1, or 2 = a 256 x 256 CTA-pair tile), from a wave-quantisation model over the SM count. */
int cc_gemm_tc_plan(int precision, int m, int n, int k, int tile_n, int split_k, int* plan);
/* plan4 = {tile width, K split, CTAs per tile, hybrid stream-K (0 | 1)}.  Hybrid stream-K: whole waves of output tiles
 * stay data-parallel, the tiles that would leave a ragged last wave are cut along K into one contiguous span of k-blocks
 * per CTA (pair) and TMA-reduce-added -- only those tiles pay read-modify-write traffic. */
int cc_gemm_tc_plan_ex(int precision, int m, int n, int k, int tile_n, int split_k, int* plan4);
/* -1 = the planner decides between split-K and hybrid stream-K (default), 0 = never stream-K, 1 = whenever possible. */
int cc_gemm_tc_set_stream_k(int mode);
/* Tile scheduling of the persistent tcgen05 GEMMs: 0 (default) = static round-robin, 1 = tiles drawn at run time from
 * a global atomic counter, so CTAs that start late or lose their SM to a concurrent kernel (an NCCL all_reduce
 * overlapping backward) take fewer tiles instead of stretching the GEMM. */
int cc_gemm_tc_set_dynamic_tiles(int on);
/* Programmatic dependent launch between consecutive tcgen05 GEMMs of a stream (default on): a GEMM's CTAs may be
 * scheduled and run their prologue while the previous kernel drains; they wait (griddepcontrol.wait) for its
 * completion before touching global memory. */
int cc_gemm_tc_set_pdl(int on);
/* MN-major tf32 operands ([K][MN] row-major: Keras kernels in forward, activations / dlogits in the weight-gradient
 * GEMMs) are fetched by ONE 3-D TMA per k-block instead of 4-8 two-dimensional boxes (CC_GEMM_MN3=0 restores the boxes);
 * this returns how many operands took the 3-D form since the library was loaded. */
int64_t cc_gemm_tc_mn3_count(void);
/* Declares [base, base + bytes) readable in full (bytes = 0 forgets the range starting at base): an MN-major tf32
 * operand whose rows are NOT padded to 32 floats (a 512 x 20 884 Keras kernel) may take the 3-D form only if the up to
 * 124 bytes its last column group reads past a row's end are known to exist -- true inside the flat parameter buffer,
 * where a kernel's last row is followed by its bias.  The ML model registers its parameter shadow. */
int cc_gemm_tc_register_readable(const void* base, int64_t bytes);
/* Up to three consecutive small Dense layers in ONE launch (the 512 -> 256 -> 128 -> 64 -> 128 -> 256 -> 512 stack of
 * model.py:27-33, 58-64 and its input gradients): a CTA takes 128 rows through the chain with the intermediate
 * activations kept in tensor memory (tcgen05.mma with the A operand in TMEM); every layer's output is also stored.
 * widths = {k0, n1, ..., n_layers} (k multiples of 32, n multiples of 64, <= 512; only the last layer may be 512 wide);
 * layer l: out_l[m][n_l] = epi(in_l W_l), in_1 = a, in_{l+1} = out_l.  w_is_kn[l] = 1: W_l is the Keras kernel [K][N]
 * (forward); 0: [N][K] (a kernel used transposed: backward).  bias / mask: arrays of `layers` nullable pointers (either
 * array itself nullable); relu applies to layers with a bias, mask keeps values where mask[row][col] > 0 (ReLU's
 * backward).  bits_out[l] (nullable): a (m, n_l / 32) uint32 matrix that receives one bit per output element (set where
 * the output is positive); mask_bits[l] (nullable, takes precedence over mask[l]): such a matrix used as the ReLU mask --
 * a 32-column chunk then costs a row 4 bytes of mask instead of 128.  Results are bit-identical to the same layers as
 * separate cc_gemm_tc calls. */
int cc_chain_tc(int m, int layers, const int32_t* widths, const float* a, int64_t lda, const float* const* w,
                const int64_t* ldw, const int32_t* w_is_kn, const float* const* bias, const float* const* mask,
                const int64_t* ldmask, const uint32_t* const* mask_bits, uint32_t* const* bits_out, int relu,
                float* const* out, const int64_t* ldout, int round_tf32, void* stream);
int64_t cc_colsum_workspace_bytes(int m, int n);
int cc_colsum_f32(const float* x, int64_t ld, int m, int n, float* workspace, float* out, int accumulate,
                  void* stream);
int cc_relu_mask_f32(float* x, int64_t ldx, const float* act, int64_t lda, int m, int n, void* stream);

/* ------------------------------------------------------------------------------------
 * (6) Losses and optimiser (Keras 2.5 conventions)
 *     replaces compile(adam, [bce, kld], loss_weights) src/ml/train.py:83-88
 * ---------------------------------------------------------------------------------- */
/* row_loss[b] = sum_c bce(z[b][c], y[b][c]); dz = (sigmoid(z) - y)/count (nullable); columns
 * [num_cards, ncols_pad) of dz are zeroed. */
int cc_bce_logits_fwd_bwd(const float* z, int64_t ldz, const uint32_t* ybits, int64_t ywords, int32_t batch,
                          int32_t num_cards, int32_t ncols_pad, double count, float* dz, int64_t lddz,
                          double* row_loss, void* stream);
/* row_correct[b] = number of cells with (z > 0) == y: the numerator of Keras' binary_accuracy (metrics=['accuracy'],
 * src/ml/train.py:87) for the exact-fp32 mode, which keeps its logits in memory (the fused GEMM counts in its epilogue). */
int cc_binary_accuracy_rows(const float* z, int64_t ldz, const uint32_t* ybits, int64_t ywords, int32_t batch,
                            int32_t num_cards, double* row_correct, void* stream);
/* row r uses target row target_rows[r] (nullable = r); dz = grad_scale*(q*S - t'*1[unclipped]).
 * dbias (nullable, float [num_cards]): also emit the column sums of dz, i.e. the softmax layer's bias gradient, from
 * the persistent form of the kernel (one CTA per SM walks the rows, next row prefetched with cp.async, column sums
 * kept in registers and added with float atomics at the end).  Only where cc_softmax_kl_fuses_dbias(...) != 0. */
int cc_softmax_kl_fuses_dbias(int32_t num_cards, int32_t ncols_pad, int64_t ldz, int64_t ldt, int64_t lddz);
int cc_softmax_kl_fwd_bwd(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                          int32_t rows, int32_t num_cards, int32_t ncols_pad, double grad_scale, float* dz,
                          int64_t lddz, double* row_loss, int round_tf32, float* dbias, void* stream);
/* Same with the dlogits written as bf16 into dz_bf16 [rows][lddz_bf16] instead of dz (needs dbias != NULL, i.e. the
 * persistent kernel); dz may then be NULL.  tlogt (nullable, float64 [rows of target]; persistent kernel only): the
 * table written by cc_kl_target_table -- with it the kernel evaluates no logarithm per element. */
int cc_softmax_kl_fwd_bwd_ex(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                             int32_t rows, int32_t num_cards, int32_t ncols_pad, double grad_scale, float* dz,
                             int64_t lddz, double* row_loss, int round_tf32, float* dbias, void* dz_bf16,
                             int64_t lddz_bf16, const double* tlogt, void* stream);
/* The same with Keras' categorical_accuracy counted on the way (metrics=['accuracy'], src/ml/train.py:87): row_hit[r] = 1
 * where the first maximal logit of row r sits in column target_argmax[target row] (cc_kl_target_argmax builds that table:
 * first maximal column of every row of M-hat, like tf.argmax).  Persistent kernels only (dbias != NULL). */
int cc_softmax_kl_fwd_bwd_metrics(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                                  int32_t rows, int32_t num_cards, int32_t ncols_pad, double grad_scale, float* dz,
                                  int64_t lddz, double* row_loss, int round_tf32, float* dbias, void* dz_bf16,
                                  int64_t lddz_bf16, const double* tlogt, const int32_t* target_argmax, int32_t* row_hit,
                                  void* stream);
int cc_kl_target_argmax(const float* target, int64_t ldt, int32_t target_rows, int32_t num_cards, int32_t* out, void* stream);
/* Loss only (evaluation): row_loss[r] and, with target_argmax, row_hit[r] (the two are nullable together), computed
 * exactly as cc_softmax_kl_fwd_bwd_metrics computes them with the same tlogt (nullable) and fast (its round_tf32); no
 * dlogits, no bias gradient, z is only read.  The register-resident kernel's shapes only (num_cards % 4 == 0, at most
 * 22 528 cards, 16-byte aligned rows): anything else returns CC_ERR_ARGUMENT. */
int cc_softmax_kl_loss(const float* z, int64_t ldz, const float* target, int64_t ldt, const int32_t* target_rows,
                       int32_t rows, int32_t num_cards, int32_t ncols_pad, const double* tlogt,
                       const int32_t* target_argmax, double* row_loss, int32_t* row_hit, int fast, void* stream);
/* Which persistent kernel serves dbias != NULL: 0 = choose (512 threads with the target row and the column sums in
 * registers when num_cards <= 22 528, else the 1024-thread form), 1 = always the 1024-thread form (tests, A/B runs). */
int cc_softmax_kl_set_variant(int variant);
/* tlogt[i] = sum_c t' log t', t' = clip(target[i][c], 1e-7, 1), float64: the model-independent half of Keras'
 * kullback_leibler_divergence (src/ml/train.py:85) for every row of M-hat; built once per graph. */
int cc_kl_target_table(const float* target, int64_t ldt, int32_t target_rows, int32_t num_cards, double* tlogt,
                       void* stream);
/* out3 (float64 [3]) = { sum(bce_rows)/bce_div, sum(kl_rows)/kl_div, bce + reg*kl } */
int cc_loss_finalize(const double* bce_rows, int32_t nb, double bce_div, const double* kl_rows, int32_t nr,
                     double kl_div, double reg, double* out3, void* stream);
/* TF-style Adam over flat buffers; the step number is *step_ptr + 1 (device int64).  shadow_tf32 (nullable)
 * receives the updated weights rounded to tf32 (round-to-nearest) for the tensor-core GEMMs.
 * round_tf32 flags elsewhere: outputs that feed a kind::tf32 GEMM are rounded to nearest where they are
 * produced, because the tensor core itself truncates (biased). */
int cc_adam_step(float* params, const float* grads, float* m, float* v, int64_t n, const int64_t* step_ptr, float lr,
                 float beta1, float beta2, float eps, float* shadow_tf32, void* stream);
/* Data-parallel form: Adam fused with the gradient exchange over NVLink peer memory.  Rank `rank` owns the slice
 * [lo, hi) (multiples of 4) of the flat buffers: it sums that slice of the gradient buffers of ALL ranks
 * (grads_ptrs[world]: device pointers, peers mapped through symmetric memory; summed in rank order), applies the Adam
 * update to its slice of m, v and params, and stores the updated parameters into every rank's parameter buffer
 * (params_ptrs[world]).  m and v are this rank's full-size buffers (only [lo, hi) is touched).  The caller puts a
 * cross-rank barrier before (all gradients written) and after (all slices delivered) the call.  world <= 16.
 * grads_multicast / params_multicast (both or neither): NVLS multicast mappings of the same two buffers; when given,
 * the sum is one multimem.ld_reduce (reduced inside the NVSwitch, order chosen by the hardware) and the broadcast one
 * multimem.st, instead of world peer loads and world peer stores. */
int cc_adam_step_p2p(const void* const* grads_ptrs, void* const* params_ptrs, int world, int rank, float* m, float* v,
                     int64_t lo, int64_t hi, const int64_t* step_ptr, float lr, float beta1, float beta2, float eps,
                     const void* grads_multicast, void* params_multicast, void* stream);
/* fp32 [rows][ld_src] -> bf16 [rows][ld_dst], round to nearest even (cols, ld_src, ld_dst multiples of 4). */
int cc_convert_f32_bf16(const float* src, int64_t ld_src, void* dst, int64_t ld_dst, int32_t rows, int32_t cols, void* stream);
int cc_round_tf32(const float* x, float* out, int64_t n, void* stream);
int cc_sigmoid_f32(const float* z, float* out, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CUBECOBRA_B200_H */
