/* mi_b200.h — C ABI of libmi_b200.so: the B200-native (sm_100a) MI critic / estimator hot path.
 *
 * The reference (vnoz/Mutual-Information-MultiModal) is pure Python and has no FFI; its hot path is
 * three attribute lookups inside MultiModalManager.train (mutual_info_img_txt/main_utils.py:220-226):
 *
 *     mi_input  = self.create_mi_pairs(embedding_img, embedding_txt, study_id, device)   # :80-110
 *     mi_output = self.mi_discriminator(mi_input)                                          # :222, model.py:18-32
 *     loss      = mi_critic(mi_output, args.batch_size, device)                            # :224, mi_critics.py:3-23
 *     loss.backward()                                                                      # :226
 *
 * The entry points below are what a binding for that sequence calls (see INTEGRATION.md for the
 * ctypes stub).  Conventions: all pointers are DEVICE pointers owned by the caller (except where a
 * name ends in _host); row-major; bf16 operands; fp32 / fp64 results; nothing is allocated or freed
 * inside; work is enqueued on `stream` and the call returns without synchronising; return value is
 * 0 on success or a negative mi_status.  Re-entrant across host threads / streams (per-call state is thread-local;
 * the mi_set_* knobs are process-wide and meant to be set once, before the first call); one call per workspace at a
 * time.  Study ids: any int32 value is a legal id (no reserved values).
 *
 * Score block:   S[q,k] = scale * <Q[q,:], K[k,:]>,   q in [0,Bq), k in [0,Bk)
 * Sample of row q is column (q_offset + q)  (the positive pair / diagonal).
 * Negatives mask (main_utils.py:105):  M[q,k] = sid_q[q] != sid_k[k]   (the diagonal has equal ids).
 */
#ifndef MI_B200_H_
#define MI_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* mi_stream_t;   /* == cudaStream_t */

enum mi_status {
  MI_OK = 0,
  MI_ERR_BAD_ARG = -1,        /* null pointer, non-positive size, D % 8 != 0, misaligned pointer */
  MI_ERR_WORKSPACE = -2,      /* workspace too small: call the matching *_workspace_bytes */
  MI_ERR_CUDA = -3,           /* a CUDA runtime / driver call failed (see mi_last_cuda_error) */
  MI_ERR_NO_DEVICE = -4,      /* no sm_100 device: there is NO CPU fallback */
  MI_ERR_NO_NEGATIVES = -5,   /* reported by the host layer when N_neg == 0 (reference yields nan/-inf) */
  MI_GUARD_TRIPPED = 1        /* mi_sharded_critic_loss_fwd_bwd only: the sampled references left the safe window on some rank
                                 (every rank returns this together); the outputs are NOT valid — repeat on the exact path */
};

enum mi_critic { MI_CRITIC_DOT = 0, MI_CRITIC_BILINEAR = 1 };

/* estimator codes.  DV and INFONCE_REF restate mi_critics.py:3-12 and :14-23 (the reference's
 * "infonce" is DV + log N_neg); INFONCE_ROW / INFONCE_SYM are the true row / symmetric InfoNCE
 * bounds the north star adds (no counterpart in the reference).  JS and NWJ are the f-divergence
 * bounds (no counterpart in the reference either; minimised, i.e. minus the bound; M = the negatives mask):
 *   JS   (Jensen-Shannon, Deep InfoMax / f-GAN):  L = mean_{M} softplus(S) + mean_i softplus(-S_ii)
 *   NWJ  (Nguyen-Wainwright-Jordan, "MINE-f"):    L = e^{-1} mean_{M} e^{S} - mean_i S_ii = e^{LSE_M - ln N_neg - 1} - pos_mean
 * JS and NWJ run only in the single-GPU separable-critic entries (mi_critic_loss_fwd_bwd and its host forms); every other
 * entry that takes an estimator rejects them (MI_ERR_BAD_ARG, or a size of 0 from its planner). */
enum mi_estimator { MI_EST_DV = 0, MI_EST_INFONCE_REF = 1, MI_EST_INFONCE_ROW = 2, MI_EST_INFONCE_SYM = 3,
                    MI_EST_JS = 4, MI_EST_NWJ = 5 };

enum mi_precision { MI_PREC_BF16_FAST = 0,   /* dS panel rounded once to bf16 */
                    MI_PREC_BF16_STRICT = 1, /* dS = hi + lo bf16 split (fp32-accumulate mode) */
                    MI_PREC_TWO_PASS = 2     /* flag (OR it in): exact softmax references (a statistics pass over EVERY
                                                column before the gradient pass) instead of sampled ones
                                                (mi_critic_loss_fwd_bwd) */ };

const char* mi_status_string(int status);
const char* mi_last_cuda_error(void);
int mi_abi_version(void);
/* 0 when a compute-capability-10.x device is current, MI_ERR_NO_DEVICE otherwise */
int mi_device_check(void);

/* ---- building blocks --------------------------------------------------------------------------- */

/* hi/lo split operands ("strict", fp32-accumulate mode): a *_split argument of 2 means the bf16 matrix
 * is a pair stored as [hi | lo] in each row, lo starting at column round_up(D, 128) (D = the logical
 * width) with zeros in between; value = hi + lo (16 significant bits).  1 = plain bf16. */

/* C[M,N] = alpha * ( A[M,K] * B[N,K]^T - gamma * SUB[M,N] ), bf16 operands (K contiguous), fp32
 * accumulate on tcgen05.  out_f32 and/or out_bf16 may be NULL; SUB may be NULL; out_split = 2 writes
 * out_bf16 as a [hi | lo] pair.  Replaces the nn.Linear-style contractions around the critic
 * (T = X W, dX = dT W^T, dW = X^T dT). */
int mi_gemm_bf16(const void* A, int64_t lda, int a_split, const void* B, int64_t ldb, int b_split,
                 int64_t M, int64_t N, int64_t K, float alpha, float gamma, const void* sub, int64_t ld_sub,
                 float* out_f32, int64_t ld_out, void* out_bf16, int64_t ld_out16, int out_split,
                 mi_stream_t stream);

/* C[M,N] = sum_k A(m,k) B(n,k) where an operand with *_mn = 1 is given as the row-major [K, rows] matrix
 * (A(m,k) = A[k*lda + m]) and read IN PLACE through MN-major UMMA shared-memory descriptors — X^T dT, X W and
 * dA W1 need no transposed copies.  *_split = 2: hi/lo pair, lo at column round_up(K,128) (K-major) or
 * round_up(rows,128) (MN-major).  fp32 outputs of few tiles and long K use split-K (partials in `workspace`). */
size_t mi_gemm_bf16_mn_workspace_bytes(int64_t M, int64_t N, int64_t K, int a_split, int a_mn, int b_split, int b_mn);
int mi_gemm_bf16_mn(const void* A, int64_t lda, int a_split, int a_mn, const void* B, int64_t ldb, int b_split, int b_mn,
                    int64_t M, int64_t N, int64_t K, float* out_f32, int64_t ld_out, void* out_bf16, int64_t ld_out16, int out_split,
                    void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* out[C,R] = in[R,C]^T (bf16) */
int mi_transpose_bf16(const void* in, int64_t ld_in, void* out, int64_t ld_out, int64_t R, int64_t C, mi_stream_t stream);
/* out = bf16(in), n elements */
int mi_cast_f32_to_bf16(const float* in, void* out, int64_t n, mi_stream_t stream);

/* Score statistics without materialising S (replaces create_mi_pairs + critic + the reductions of
 * mi_critics.py:7-10 / :18-20):
 *   row_out[q] = { lse_neg, n_neg, diag, lse_all }   natural log; lse_neg = LSE_k M[q,k] S[q,k],
 *                                                    lse_all = logaddexp(lse_neg, diag)
 *   scal_out   = { m = max_q lse_neg, sum_q exp(lse_neg - m), sum_q n_neg, sum_q diag,
 *                  sum_q (lse_all - diag), #rows without negatives, 0, 0 }          (fp64) */
size_t mi_score_stats_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D);
int mi_score_stats(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                   const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                   int64_t Bq, int64_t Bk, int64_t D, float scale,
                   float* row_out /*[Bq,4]*/, double* scal_out /*[8]*/,
                   void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* Row statistics as mi_score_stats AND, from the same score tiles, the column statistics of the row block: col_lse_out[c]
 * (c < Bk) = log-sum-exp over the block's rows r with sid_q[r] != sid_k[c] of S[r, c] (-inf if there is none).  This is the
 * statistics pass of the symmetric InfoNCE estimator in the batch-sharded step (a rank holds Bq rows at q_offset of the
 * [Bk, Bk] score matrix): the ranks' col_lse vectors are merged with a log-sum-exp by the caller, so the columns cost no
 * second pass and no all-gather of the projected image embeddings (mi_critics.py has no symmetric form; BASELINE config 3). */
size_t mi_score_stats_rc_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D);
int mi_score_stats_rc(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                      const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                      int64_t Bq, int64_t Bk, int64_t D, float scale, float* row_out, double* scal_out, float* col_lse_out,
                      void* workspace, size_t workspace_bytes, mi_stream_t stream);
/* mi_score_stats_rc with the schedule and output of the batch-sharded symmetric step (mi_score_stats_rc is this call with
 * NULL, 0, 0; same workspace size):
 *   event_k_ready / k_local_valid as in mi_score_single_pass: with k_local_valid = 1, q_offset and Bq multiples of 256 and
 *     Bq < Bk, the tiles of the own column block [q_offset, q_offset + Bq) are scored before the wait for the event;
 *     otherwise the call waits before the first tile.
 *   include_pos = 1: the block's positive pairs are folded into its own columns, col_lse_out[q_offset + r] =
 *     logaddexp(col_lse_out[q_offset + r], S[r, q_offset + r]).  Column j of the batch is then the plain log-sum-exp of the
 *     ranks' col_lse_out[j] (mi_merge_sym_stats). */
int mi_score_stats_rc_ex(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                         const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                         int64_t Bq, int64_t Bk, int64_t D, float scale, float* row_out, double* scal_out, float* col_lse_out,
                         void* event_k_ready, int k_local_valid, int include_pos,
                         void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* Fused gradient pass (replaces loss.backward() through mi_critics.py and the pair tensor,
 * main_utils.py:226): recomputes score tiles, forms
 *   G[q,k] = incl[q,k] * ( wq * exp(S - refq[q]) + wk * exp(S - refk[k]) )
 *   incl   = M  (include_diag = 0, DV)   or   M + diagonal  (include_diag = 1, InfoNCE)
 * and returns  Oq[q,:] = alpha * ( sum_k G[q,k] K[k,:] - gamma * K[q_offset+q,:] )  (fp32 and/or bf16,
 * optionally hi/lo)  and, when outk_f32 != NULL,
 *              Ok[k,:] = alpha * ( sum_q G[q,k] Q[q,:] - gamma * [0 <= k-q_offset < Bq] Q[k-q_offset,:] )
 * from the same score recompute (gamma is the weight of the positive pair, 1/B).
 * refq / refk may be NULL (term unused).  Ok is finished before Oq (event_after_outk marks that point, so a
 * caller can start the reduce-scatter of Ok under the remaining work).  The B x B matrix never exists: G is staged as a bounded bf16
 * row panel in `workspace` and consumed by the two tensor-core contractions. */
size_t mi_score_grad_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D, int precision);
int mi_score_grad(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                  const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                  int64_t Bq, int64_t Bk, int64_t D, float scale,
                  const float* refq, float wq, const float* refk, float wk,
                  int include_diag, int precision, float alpha, float gamma,
                  float* outq_f32, void* outq_bf16, int64_t ld_outq16, int outq_split, float* outk_f32,
                  void* event_after_outk /* cudaEvent_t or NULL: recorded on `stream` once Ok is complete */,
                  void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* Single-pass form of statistics + gradients for dv / infonce / row InfoNCE: ONE score computation instead of two.
 * The pass writes P~ = incl e^{S - ref[q]} before the exact row statistics exist, so it needs a per-row reference close
 * enough to the row's log-sum-exp for P~ and its row sum to stay inside the fp32 / bf16 range (+-87 in the exponent).
 *
 * mi_score_ref_sample produces it: ref[q] = log-sum-exp of row q over the SAMPLED columns col0 + s * stride (s * stride <
 * n_cols) of K — the statistics epilogue run on a strided view of K (TMA row pitch = stride * ldk, no gather);
 * include_diag = 1 adds the positive pair.  stride = 1 samples every column: the references are then the exact row
 * log-sum-exps and the pass cannot leave the safe window.  stride = 0 picks mi_ref_sample_stride(Bq, n_cols, D) (about
 * mi_set_ref_sample_columns() columns per row, default 2048, i.e. ~1 % of the step at B = 65536).  Also returned:
 * diag_out[q] = the positive-pair score S[q, q_offset + q], lambda_out[0] = the largest sample log-sum-exp (may be NULL).
 * Sampled references (stride > 1) are lifted 48 nats above the sample's log-sum-exp: the true value can only lie above it.
 *
 * mi_score_single_pass: the same tiles give the row sums (=> row_out / scal_out exactly as mi_score_stats; for
 * include_diag = 1 the sums include the positive pair) and
 *   oq_raw[q,:] = sum_k P~[q,k] K[k,:]                 ok_raw[k,:] = sum_q P~[q,k] wrow[q] Q[q,:]
 * with wrow = e^{ref - lambda[0]} (include_diag = 0; lambda = ONE constant near the largest reference, the same on every
 * rank whose ok_raw is summed) or inv_bg / rowsum (include_diag = 1; lambda unused, may be NULL).
 * Any reference is mathematically valid.  flag_out (and scal_out[6]) count the rows whose reference left the numerically
 * safe window (row sum outside [1e-30, 1e30], or ref - lambda > 80): must be 0, else repeat with stride = 1 references.
 * The gradients follow from mi_single_finalize_q / _k once the (global) log-sum-exp is known:
 *   Oq = alpha (c_q oq_raw - gamma Kdiag),  c_q = e^{ref_q - lse} (dv_like) or wrow_q
 *   Ok = alpha (kappa ok_raw - gamma Qdiag), kappa = e^{lambda - lse} (dv_like) or 1     (in place) */
size_t mi_score_ref_sample_workspace_bytes(int64_t Bq, int64_t n_cols, int64_t D, int64_t stride);
int64_t mi_ref_sample_stride(int64_t Bq, int64_t n_cols, int64_t D);
int mi_score_ref_sample(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                        const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                        int64_t Bq, int64_t Bk, int64_t D, float scale, int include_diag,
                        int64_t col0, int64_t n_cols, int64_t stride,
                        int subset /* 1: K holds only PART of the row's columns (a rank's own block): margin even at stride 1 */,
                        float* ref_out /*[Bq]*/, float* diag_out /*[Bq]*/, float* lambda_out /*[1] or NULL*/,
                        void* workspace, size_t workspace_bytes, mi_stream_t stream);
size_t mi_score_single_pass_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D, int precision);
int mi_row_norm_max(const void* A, int64_t lda, int a_split, int64_t rows, int64_t D, float* norm_out, float* max_out, mi_stream_t stream);
int mi_score_single_pass(const void* Q, int64_t ldq, int q_split, const void* K, int64_t ldk, int k_split,
                         const int32_t* sid_q, const int32_t* sid_k, int64_t q_offset,
                         int64_t Bq, int64_t Bk, int64_t D, float scale, int include_diag, int precision, float inv_bg,
                         const float* ref /*[Bq]*/, const float* lambda /*[1]*/, const float* diag /*[Bq]*/,
                         float* row_out /*[Bq,4]*/, double* scal_out /*[8]*/,
                         float* oq_raw /*[Bq,D]*/, float* ok_raw /*[Bk,D] or NULL*/,
                         float* wrow /*[Bq]*/, int32_t* flag_out /*[1]*/,
                         void* event_after_outk,
                         void* event_after_scal /* cudaEvent_t or NULL: recorded once row_out / scal_out are final, i.e. BEFORE the
                                                   last panel's two contractions — exchange the loss scalars under them */,
                         void* event_k_ready /* cudaEvent_t or NULL: the K rows (an all-gather in flight) are complete once this
                                                event fires; the mask pre-pass is enqueued BEFORE the wait */,
                         int k_local_valid /* 1: rows [q_offset, q_offset + Bq) of K (this rank's own text embeddings) are valid
                                              already — the score tiles of the own column block also run before the wait */,
                         void* workspace, size_t workspace_bytes, mi_stream_t stream);
/* Multi-GPU glue: the ranks' scal_out rows [world][8] (all-gathered) -> loss_out (fp64[8], layout of mi_critic_loss_fwd_bwd,
 * global batch B_global, estimators DV / INFONCE_REF / INFONCE_ROW) and the global log-sum-exp as a float (lse_out[1]).
 * loss_out[7] = the ranks' guard counts summed (+1 if e^{lambda - lse} would leave the fp32 range; lambda may be NULL).
 * Two tiny kernels instead of a chain of framework ops.  scratch8: 8 doubles of device scratch. */
int mi_merge_scalars(const double* scal_all, int world, int64_t B_global, int estimator, const float* lambda,
                     double* loss_out, float* lse_out, double* scratch8, mi_stream_t stream);
/* The symmetric estimator's merge (the one the batch-sharded step runs, fp64): the ranks' scalar rows scal_all [world][8]
 * (mi_score_stats_rc_ex) and column partials col_all [world][col_pitch] (include_pos = 1, first B_global floats of each row
 * used) -> c_out [B_global] fp32 = the fp64 log-sum-exp of column j over the ranks, rounded once (the column references of
 * the gradient pass), and loss_out (fp64[8]) in the layout of the single-GPU symmetric call: slot 0 = (row + col) / 2,
 * 4 = loss_row, 5 = loss_col = (sum_j c_j - sum_i S_ii) / B_global, 7 = 0.  Sums run in a fixed order (no atomics): the
 * same inputs give the same bits.  scratch: mi_merge_sym_stats_scratch_doubles(B_global) doubles of device scratch. */
int64_t mi_merge_sym_stats_scratch_doubles(int64_t B_global);
int mi_merge_sym_stats(const double* scal_all, const float* col_all, int64_t col_pitch, int world, int64_t B_global,
                       double* loss_out, float* c_out, double* scratch, mi_stream_t stream);
int mi_single_finalize_q(const float* oq_raw, int64_t rows, int64_t D, const float* ref, const float* wrow, const float* lse,
                         int dv_like, float alpha, float gamma, const void* kdiag, int64_t ldk, int k_split,
                         float* out_f32, void* out_bf16, int64_t ld16, int out_split, mi_stream_t stream);
int mi_single_finalize_k(float* ok, int64_t rows, int64_t D, const float* lambda, const float* lse, int dv_like,
                         float alpha, float gamma, const void* qdiag, int64_t ldq, int q_split, mi_stream_t stream);

/* ---- the whole path, one GPU ------------------------------------------------------------------- */

/* loss_out (fp64[8]) = { loss, pos_mean, lse_neg, n_neg, loss_row, loss_col, #rows w/o negatives, guard }.
 * X = image embeddings [B,D], Y = text embeddings [B,D], W = [D,D] (NULL for the dot critic),
 * S = inv_tau * X W Y^T.  dX, dY (fp32 [B,D]) and dW (fp32 [D,D]) may all be NULL (forward only).
 *
 * dv / infonce / row InfoNCE run the single pass with SAMPLED references (mi_score_ref_sample).  If any row's reference
 * leaves the safe window the library repeats the step itself with exact references: the repeat is enqueued on the same
 * stream behind a device-side predicate (a handful of empty launches when the guard stayed clear), so the call stays
 * asynchronous and CUDA-graph capturable, and the results are ALWAYS those of a pass whose guard was clear.
 * guard (loss_out[7]) = number of rows that tripped the sampled pass: > 0 only says that the exact repeat produced the
 * results.  MI_PREC_TWO_PASS asks for exact references from the start.  The symmetric estimator always runs the
 * statistics passes + one gradient pass with exact references.
 *
 * MI_EST_NWJ runs DV's single pass (same references, guard and exact repeat; MI_PREC_TWO_PASS = exact references) and
 * differs only in its scalar: G = kappa softmax_M(S) - I/B, kappa = e^{LSE_M - ln N_neg - 1} (ln N_neg in fp64).  A kappa
 * outside the fp32 range is NOT a guard condition (an exact repeat could not change it): the fp64 loss stays finite and the
 * gradients overflow as an fp32 computation of the same formula would.
 * MI_EST_JS needs no normaliser: ONE score pass per row panel writes M sigma(S) into the dS panel and sums M softplus(S) per
 * row; G = M sigma(S) / N_neg - diag(sigma(-S_ii)) / B.  No reference sample, no guard (loss_out[7] = 0), MI_PREC_TWO_PASS
 * changes nothing.  Forward-only calls run the same pass without the panel.
 * loss_out of the two:     slot   0     1          2                       3       4                       5   6                  7
 *                          NWJ    loss  pos_mean   LSE_M                   n_neg   0                       0   rows w/o neg.      guard (as DV)
 *                          JS     loss  pos_mean   mean_M softplus(S)      n_neg   mean_i softplus(-S_ii)  0   rows w/o neg.      0
 * Without any negative pair the loss of both is NaN. */
size_t mi_critic_workspace_bytes(int64_t B, int64_t D, int critic, int estimator, int precision, int need_grads);
int mi_critic_loss_fwd_bwd(const void* X, const void* Y, const void* W, const int32_t* sid,
                           int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                           double* loss_out, float* dX, float* dY, float* dW,
                           void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* Same call with HOST buffers (fp32 embeddings as the encoders produce them): copies X, Y, W, sid
 * to the device, runs the path, copies loss and gradients back, synchronises; a tripped guard is handled on the host
 * (the step is repeated with exact references before the call returns; loss_out[7] as above).
 * dev_scratch is a device buffer of mi_critic_host_scratch_bytes(...) bytes.  Uses one internal copy stream per device:
 * concurrent calls on the same device are serialised inside the library. */
size_t mi_critic_host_scratch_bytes(int64_t B, int64_t D, int critic, int estimator, int precision, int need_grads);
int mi_critic_loss_fwd_bwd_host(const float* X_host, const float* Y_host, const float* W_host, const int32_t* sid_host,
                                int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                                double* loss_out_host, float* dX_host, float* dY_host, float* dW_host,
                                void* dev_scratch, size_t dev_scratch_bytes, mi_stream_t stream);

/* The data-loader form: embeddings arrive in HOST buffers (host_dtype 0 = fp32, 1 = bf16: copied straight into the operand
 * buffers), the loss goes back to the host, the gradients stay on the DEVICE (dX_dev, dY_dev, dW_dev: fp32 device buffers or
 * NULL) where the encoders' backward consumes them.  Same streaming of the image-embedding panels under the pass, same guard
 * handling and scratch size as mi_critic_loss_fwd_bwd_host; synchronises before it returns. */
int mi_critic_loss_fwd_bwd_from_host(const void* X_host, const void* Y_host, const void* W_host, const int32_t* sid_host, int host_dtype,
                                     int64_t B, int64_t D, int critic, int estimator, int precision, float inv_tau,
                                     double* loss_out_host, float* dX_dev, float* dY_dev, float* dW_dev,
                                     void* dev_scratch, size_t dev_scratch_bytes, mi_stream_t stream);

/* ---- the whole path, batch-sharded over the GPUs of one node (SURVEY 8e) --------------------------------------- */

/* One host call per step and rank: rank r passes its row shard (X_local, Y_local [B_local, D] bf16, sid_local int32; all ranks
 * the same B_local) and receives the GLOBAL-batch loss (loss_out fp64[8], device, identical on every rank) and the gradients
 * of its rows (dX, dY fp32 [B_local, D]) plus dW (fp32 [D, D], already summed over ranks).  Every estimator; for DV /
 * INFONCE_REF / INFONCE_ROW inside: all-gather of the ids and of Y
 * (in place, the own column block is scored while the others arrive), references from a sample of the OWN column block and
 * an all-reduce(max) of lambda, the single pass, all-gather of the 8 loss scalars, reduce-scatter of the dY contributions
 * under the dT contraction, all-reduce of dW under the dX GEMM — NCCL called directly on `nccl_comm` (an ncclComm_t, e.g.
 * torch.distributed's ProcessGroupNCCL._comm_ptr()) from ONE internal communication stream per context; libnccl.so.2 is
 * resolved from the running process.  check_guard = 1: the host waits (an event, not a stream) until the merged guard count
 * is known — right after the score tiles — and returns MI_GUARD_TRIPPED on every rank when it is non-zero; 0: never
 * synchronises, the count is left in loss_out[7].  A context is bound to one device / communicator and serves one call at a
 * time; the collectives it issues must not interleave with other collectives on the same communicator from other threads.
 * MI_EST_INFONCE_SYM uses exact statistics (no guard: loss_out[7] = 0, never MI_GUARD_TRIPPED, check_guard ignored, no host
 * read) with the loss_out layout of the single-GPU symmetric call: all-gather of the ids and of Y, the row + column
 * statistics pass (own column block first, own positive pairs folded into the column partials), ONE all-gather of each
 * rank's packed record {8 fp64 scalars | B fp32 column partials}, the fp64 merge (mi_merge_sym_stats) on every rank, the
 * gradient pass with row and column references, then the same reduce-scatter / all-reduce as above. */
typedef struct mi_dist_ctx mi_dist_ctx;
int mi_dist_ctx_create(void* nccl_comm, mi_dist_ctx** out);
void mi_dist_ctx_destroy(mi_dist_ctx* ctx);
int mi_dist_ctx_info(const mi_dist_ctx* ctx, int* rank, int* world);
size_t mi_sharded_critic_workspace_bytes(int64_t B_local, int world, int64_t D, int critic, int estimator, int precision);
int mi_sharded_critic_loss_fwd_bwd(mi_dist_ctx* ctx, const void* X_local, const void* Y_local, const void* W, const int32_t* sid_local,
                                   int64_t B_local, int64_t D, int critic, int estimator, int precision, float inv_tau,
                                   double* loss_out, float* dX, float* dY, float* dW,
                                   void* workspace, size_t workspace_bytes, int check_guard, mi_stream_t stream);

/* ---- the reference's own critic: make_mlp(2D, [H1, H2]) on every pair (SURVEY 8f-1) ---------------- */

/* Replaces, for the critic the reference ships (main_utils.py:77: mi_discriminator = make_mlp(1536, [1024, 512]),
 * model.py:18-32), the sequence  create_mi_pairs -> mi_discriminator -> dv/infonce_bound_loss -> backward
 * (main_utils.py:220-226) without building the [B + N_neg, 2D] pair tensor.  All tensors fp32, row-major, on the
 * device, in nn.Linear layout:  W1 [H1, 2D] (columns [0,D) act on the image embedding, [D,2D) on the text
 * embedding), b1 [H1], W2 [H2, H1], b2 [H2], W3 [1, H2], b3 [1].   D, H1, H2 multiples of 8, H2 <= 512.
 * estimator: MI_EST_DV, MI_EST_INFONCE_REF, MI_EST_INFONCE_ROW or MI_EST_INFONCE_SYM.  precision: MI_PREC_BF16_FAST
 * (bf16 operands of the tensor-core contractions, fp32 accumulate) or MI_PREC_BF16_STRICT (hi/lo bf16 pairs, 16
 * significant bits).  loss_out (fp64[8]) as mi_critic_loss_fwd_bwd (slot 4 = loss_row, slot 5 = loss_col of
 * MI_EST_INFONCE_SYM).  dv / infonce with gradients run as a single pass (softmax weights against
 * the maximum logit of a sample of pairs, Z2 formed once; see mi_set_mlp_mode); if its guard trips, the two-pass sequence
 * repeats the step behind a device-side predicate and loss_out[7] > 0 reports it.  infonce_row and infonce_sym always run
 * the two-pass sequence (their row / column normalisers need every logit first).  The call never synchronises.
 * S_out (optional, [B, B]) receives the logit of EVERY pair
 * (S[i,j] = mlp([x_i ; y_j]); the reference's logits are its diagonal followed by its negatives in gap-major
 * order).  Every gradient pointer may be NULL; all NULL = forward only. */
size_t mi_mlp_critic_workspace_bytes(int64_t B, int64_t D, int64_t H1, int64_t H2, int precision);
int mi_mlp_critic_loss_fwd_bwd(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                               const float* W3, const float* b3, const int32_t* sid,
                               int64_t B, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                               double* loss_out, float* S_out, float* dX, float* dY, float* dW1, float* db1, float* dW2, float* db2,
                               float* dW3, float* db3, void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* The MLP critic over a ROW BLOCK: the stage ops of the batch-sharded step (DESIGN 8.4; mi_b200.dist drives them with
 * its own collectives).  Rank r holds image rows X [Bq, D] at global rows [q_offset, q_offset + Bq) and has all-gathered
 * the Bk text rows Y [Bk, D] of the batch (Bk = B_global) and their ids sid_k [Bk]; sid_q [Bq] = the ids of its own rows.
 * The six parameters are replicated.  Every call is asynchronous on `stream` and never synchronises.  Per step:
 *   1. mi_mlp_block_ref_logit  (single pass only) -> ref_out[1]: the maximum logit of a sample of the block's OWN pairs
 *      (image rows x the text rows at the same global indices); the caller takes the maximum over the ranks.
 *   2. mi_mlp_block_fwd        the block's pass over its Bq x Bk pairs -> scal_out[8], the block's scalar row in the
 *      mi_score_stats layout (slot 7: the block's sum of the softmax weights in reference units, single pass only).
 *      two_pass = 0: the single pass against `ref` (same value on every rank); 1: the logits are formed first (exact).
 *      mi_mlp_block_fwd_rc (MI_EST_INFONCE_SYM, two_pass = 1 only) also writes col_lse_out [Bk]: for every text row j the
 *      log-sum-exp of the block's logits S[i, j] over its negatives and, when j = q_offset + i lies in the block, the
 *      positive pair (-inf if the set is empty).  The column of the batch is the log-sum-exp of the ranks' values.
 *   3. (caller) all-gather of the scalar rows -> scal_all [world, 8] (MI_EST_INFONCE_SYM: and of the column partials)
 *   4. mi_mlp_block_merge      -> loss_out[8] of the batch (mi_mlp_critic_loss_fwd_bwd's layout) and merged[8] (the merged
 *      row, slot 7 summed).  Single pass: loss_out[7] != 0 when the global weight sum left [1e-30, 1e30] while negatives
 *      exist — the same verdict on every rank; the caller then repeats the step with two_pass = 1.
 *      MI_EST_INFONCE_SYM (two_pass = 1 only): every slot as for MI_EST_INFONCE_ROW; the caller completes slot 5
 *      (loss_col = (sum_j c_j - B_global * slot 1) / B_global, c = the merged columns) and slot 0 (= (slot 4 + slot 5) / 2).
 *   5. mi_mlp_block_bwd        -> dX of the block's rows, dC_part [Bk, H1] (the block's contribution to dL/dC for EVERY
 *      text row, to be summed over ranks), the image half of dW1 ([H1, 2D] pitch, columns [0, D)), db1, dW2, db2, dW3,
 *      db3: the block's shares (sum over ranks = the gradient of the global loss).  mi_mlp_block_bwd_rc takes col_lse [Bk],
 *      the merged columns of the batch (MI_EST_INFONCE_SYM; NULL otherwise).
 *   6. (caller) reduce-scatter of dC_part -> dC [Bq, H1] of the own text rows;
 *      mi_mlp_input_grad(dC, Y_own, W1, side = 1) -> dY of the own rows and the text half of dW1; all-reduce of the
 *      parameter gradients.
 * `state` (mi_mlp_block_state_bytes) is caller-owned and carries the block from fwd to bwd; `workspace`
 * (mi_mlp_block_workspace_bytes, covers every stage and mi_mlp_input_grad with R = Bq) is scratch that may be reused in
 * between.  Sizes are 0 for unsupported shapes (D, H1, H2 multiples of 8, H2 <= 512). */
size_t mi_mlp_block_workspace_bytes(int64_t Bq, int64_t Bk, int64_t D, int64_t H1, int64_t H2, int precision);
size_t mi_mlp_block_state_bytes(int64_t Bq, int64_t Bk, int64_t D, int64_t H1, int64_t H2, int precision);
int mi_mlp_block_ref_logit(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                           const float* W3, const float* b3, int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2,
                           int precision, float* ref_out, void* workspace, size_t workspace_bytes, mi_stream_t stream);
int mi_mlp_block_fwd(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                     const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                     int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                     const float* ref, int two_pass, double* scal_out, void* state, size_t state_bytes,
                     void* workspace, size_t workspace_bytes, mi_stream_t stream);
int mi_mlp_block_fwd_rc(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                        const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                        int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                        const float* ref, int two_pass, double* scal_out, float* col_lse_out, void* state, size_t state_bytes,
                        void* workspace, size_t workspace_bytes, mi_stream_t stream);
int mi_mlp_block_merge(const double* scal_all, int world, int64_t B_global, int estimator, int two_pass, double* loss_out,
                       double* merged, mi_stream_t stream);
int mi_mlp_block_bwd(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                     const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                     int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                     int two_pass, const double* loss, const double* merged, void* state, size_t state_bytes,
                     float* dX, float* dC_part, float* dW1, float* db1, float* dW2, float* db2, float* dW3, float* db3,
                     void* workspace, size_t workspace_bytes, mi_stream_t stream);
int mi_mlp_block_bwd_rc(const float* X, const float* Y, const float* W1, const float* b1, const float* W2, const float* b2,
                        const float* W3, const float* b3, const int32_t* sid_q, const int32_t* sid_k,
                        int64_t Bq, int64_t Bk, int64_t q_offset, int64_t D, int64_t H1, int64_t H2, int estimator, int precision,
                        int two_pass, const double* loss, const double* merged, const float* col_lse, void* state, size_t state_bytes,
                        float* dX, float* dC_part, float* dW1, float* db1, float* dW2, float* db2, float* dW3, float* db3,
                        void* workspace, size_t workspace_bytes, mi_stream_t stream);
/* Layer-1 backward of one side of the MLP critic over R rows: dZ [R, H1] = dL/d(W1side in), In [R, D], W1 the full [H1, 2D]
 * weight; side 0 = image (W1x, columns [0, D)), 1 = text (W1y, columns [D, 2D)).  dIn = dZ W1side [R, D], the side's
 * half of dW1 [H1, 2D] = dZ^T In, db1 (optional) = column sums of dZ.  Any output may be NULL. */
size_t mi_mlp_input_grad_workspace_bytes(int64_t R, int64_t D, int64_t H1, int precision);
int mi_mlp_input_grad(const float* dZ, const float* In, const float* W1, int side, int64_t R, int64_t D, int64_t H1, int precision,
                      float* dIn, float* dW1, float* db1, void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* ---- Generalised Discrimination Value (validate.py:16-49, gdv_calculation; SURVEY 8f-3) ----------------- */

/* pos [Np, D], neg [Nn, D]: fp32 device matrices of the two classes' embeddings (validate.py:118-127).  Each class is
 * z-scored per feature (StandardScaler semantics incl. its constant-feature rule), then the sums of ALL pairwise
 * Euclidean distances inside each class and between the classes are formed on the tile engine with a
 * sqrt(|a|^2 + |b|^2 - 2 a.b) epilogue (no N x N matrix).  out (fp64[4]) = { gdv, intra_pos, intra_neg, inter } with the
 * reference's normalisers (which count N * D elements, validate.py:25,31-33).  D multiple of 8; Np, Nn >= 2. */
size_t mi_gdv_workspace_bytes(int64_t Np, int64_t Nn, int64_t D, int precision);
int mi_gdv(const float* pos, const float* neg, int64_t Np, int64_t Nn, int64_t D, int precision, double* out /*[4]*/,
           void* workspace, size_t workspace_bytes, mi_stream_t stream);

/* Introspection of host-side scheduling decisions (used by the CPU tests; no device needed).
 * mi_plan_ksplit: the K splits a GEMM with `tiles` output tiles and `k_blocks` K blocks is given (>= min_ks).
 * mi_plan_mlp_walk: the (unit, M block, N tile) work items of the MLP critic's fused dZ1 kernel for a panel of `rr` image
 * rows at batch B, hidden width H1, in the order the CTA pairs walk them; returns the item count. */
int mi_plan_ksplit(int64_t tiles, int k_blocks, int64_t min_ks);
int64_t mi_plan_mlp_walk(int64_t rr, int64_t B, int64_t H1, int32_t* out /*[max_items][3]*/, int64_t max_items);

/* number of kernels this library has launched since load (bench.py's gpu_launches) */
int64_t mi_launch_count(void);

/* Optional CUDA-event timing of every tile-engine launch (records events on the launch stream).
 * mi_profile_read drains the records: ms[k] / launches[k], k = 0 score statistics, 1 dS panel, 2 GEMM. */
void mi_set_profiling(int on);
int mi_profile_read(double* ms /*[3]*/, int64_t* launches /*[3]*/);
/* the same with n_kinds <= 6 buckets: 3 = MLP-critic single pass (forward + dZ2), 4 = MLP-critic dZ1 contraction with fused
 * reductions, 5 = MLP-critic two-pass epilogues (logits / dZ2) */
int mi_profile_read_kinds(double* ms, int64_t* launches, int n_kinds);

/* bring-up / A-B knob: 2 (default) = CTA pairs, cta_group::2 MMAs with M = 256; 1 = single-CTA M = 128.
 * Also settable through the environment variable MI_CTA_GROUP before the first call. */
void mi_set_cta_group(int group);
void mi_set_mlp_panel_pairs(int64_t pairs); /* pairs per row panel of the MLP-critic path (default 2^20; tests use small values) */
/* MLP-critic A/B knob.  bit 0: dv / infonce run as a single pass (reference logit from a sample of pairs, Z2 formed once,
 * device-predicated two-pass repeat if the guard trips); bit 1: the dZ1 reductions are fused into their GEMM's epilogue.
 * Default 3; 0 = the two-pass sequence for every estimator; negative = default. */
void mi_set_mlp_mode(int mode);
int mi_get_mlp_mode(void);                  /* the current MLP-critic mode (0..3) */
/* Multi-GPU overlap: the tile-engine launches that follow `event_after_outk` inside mi_score_single_pass / mi_score_grad
 * use (SM count - n) SMs, so the collective the caller starts at that event (reduce-scatter of the dY contributions)
 * finds free SMs instead of queueing behind a persistent 148-CTA grid.  0 (default) = use every SM. */
void mi_set_overlap_reserve_sms(int n);
/* Columns sampled per row for the single pass's references (default 2048; <= 0: always every column).  Tests use small
 * values to exercise the sampled path and its guard at small B. */
void mi_set_ref_sample_columns(int64_t n);
int mi_get_cta_group(void);

#ifdef __cplusplus
}
#endif
#endif /* MI_B200_H_ */
