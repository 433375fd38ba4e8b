/*
 * coper.h — C ABI of libcoper_sm100.so: the B200 (sm_100a) kernels behind the CoPER-ConvE hot path.
 *
 * The reference (otiliastr/coper, CoPER_ConvE/qa_cpg) has no FFI: its "operators" are the TensorFlow-1
 * stock ops called from models.py / metrics.py.  Each entry point below therefore cites the reference
 * call site (file:line under /root/reference/CoPER_ConvE/qa_cpg/) whose arithmetic it replaces.
 *
 * Conventions
 *   - every function returns 0 (COPER_OK) or a negative coper_status; no exceptions, no allocation:
 *     all buffers (inputs, outputs, workspaces) are caller-owned DEVICE pointers; workspace sizes come
 *     from the matching *_workspace_bytes function.
 *   - `stream` is a cudaStream_t passed as void*; work is enqueued on it and the call returns
 *     immediately (no host synchronisation) -> every entry point is CUDA-graph capturable.
 *   - tensors are dense row-major fp32 unless stated; index tensors are int64 (TF's e1/e2/rel dtype,
 *     models.py:141-143) or int32 where noted.
 *   - `prec` selects the arithmetic of the GEMM-shaped kernels: COPER_PREC_FP32 = CUDA-core FFMA,
 *     fp32 operands and accumulation (parity path, <=1e-5 rel); COPER_PREC_BF16 = tcgen05 kind::f16 with
 *     bf16 operands / fp32 TMEM accumulators; COPER_PREC_TF32X3 = tcgen05 kind::tf32 with 3-term error
 *     compensation (hi*hi + hi*lo + lo*hi), fp32-class accuracy on the tensor pipe; COPER_PREC_FP16X3 = the same
 *     3-term compensation on IEEE fp16 (hi, lo) planes (kind::f16: twice the MMA rate and half the operand bytes of
 *     tf32; fp16 has tf32's 11-bit significand, its 5-bit exponent is handled by one power-of-two scale per
 *     operand, chosen from the operand's max |x| when it is prepared and removed again in the epilogue).
 *   - dropout is a counter-based hash of (seed, element index): keep iff hash32 < keep * 2^32
 *     (coper_dropout_mask exports the same mask for the oracle).  keep >= 1 disables it.  The seed is
 *     (*seed_dev + salt): seed_dev is a device uint64 the step-state kernel bumps once per step (so a
 *     captured CUDA graph draws fresh masks on every replay); seed_dev may be NULL (= 0).
 */
#ifndef COPER_H_
#define COPER_H_

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* coper_stream_t; /* cudaStream_t */

typedef enum {
  COPER_OK = 0,
  COPER_ERR_INVALID_ARG = -1,
  COPER_ERR_CUDA = -2,
  COPER_ERR_UNSUPPORTED = -3,
  COPER_ERR_WORKSPACE = -4
} coper_status;

enum { COPER_PREC_FP32 = 0, COPER_PREC_BF16 = 1, COPER_PREC_TF32X3 = 2, COPER_PREC_FP16X3 = 3 };

int coper_version(void);
const char* coper_status_string(int status);
/* last cudaError_t observed by a failing call on this thread (0 if none) */
int coper_last_cuda_error(void);
/* number of kernels this library has launched in this process (bench.py reports the per-step delta) */
long long coper_launch_count(void);
/* Programmatic dependent launch between consecutive kernels of a stream (every kernel of the library is launched with
 * the programmatic-stream-serialization attribute and begins with griddepcontrol.launch_dependents / .wait): on by
 * default; worth ~8 % on the launch-bound evaluation step of the named datasets, and measured to COST ~10 % on the
 * HBM-bound 10 M-entity step (DESIGN 4.6) - a caller with tables of that size switches it off. */
int coper_set_pdl(int on);
/* 1 if the running device is compute capability 10.x (tcgen05 paths usable), 0 otherwise, <0 on error */
int coper_device_is_sm100(void);

/* ------------------------------------------------------------------------------------------------
 * a2 / K1 — tf.nn.embedding_lookup (models.py:176,178): out[i,:] = table[idx[i],:]
 * With [row_lo,row_hi) != [0,n_rows) only locally-owned rows are written, others are zero-filled
 * (entity-sharded lookup: an all-reduce(sum) of the outputs then delivers every row exactly). */
int coper_gather_rows(const float* table, int64_t row_lo, int64_t row_hi, int width,
                      const int64_t* idx, int n_idx, float* out, coper_stream_t stream);
/* The two lookups that open a step (models.py:176 head entities, :178 relations) in ONE launch; n_b == 0: only table a.
 * step_state != NULL: the launch also performs coper_step_state_advance(step_state, seed_dev, lr, beta1, beta2)
 * (nothing in the lookups reads that state) - a training step then starts with one kernel instead of three. */
int coper_gather_rows2(const float* table_a, int64_t lo_a, int64_t hi_a, int width_a, const int64_t* idx_a, int n_a,
                       float* out_a, const float* table_b, int64_t lo_b, int64_t hi_b, int width_b,
                       const int64_t* idx_b, int n_b, float* out_b, float* step_state, uint64_t* seed_dev, float lr,
                       float beta1, float beta2, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * a5 / K4 — tf.nn.conv2d NHWC, 1 input channel, stride 1, VALID (+ bias) (models.py:355,382-385;
 * per-query filters: models.py:375-380).  x0 [B, H*W] -> z [B, OH*OW*C] in (h,w,c) order.
 * wc [KH,KW,C] / bc [C], or [B,KH,KW,C] / [B,C] when per_query != 0. */
int coper_conv_fwd(const float* x0, int B, int H, int W, const float* wc, const float* bc, int KH, int KW,
                   int C, int per_query, float* z, coper_stream_t stream);
/* backward of the above (what TF autodiff derives for models.py:375-385 at models.py:198):
 * dz [B,OH*OW*C] -> dx0 [B,H*W]; shared filters: per-sample partials
 * dwc_part [S, KH*KW*C], dbc_part [S, C] with S = coper_conv_bwd_slabs(...) <= B slabs (reduce over S with
 * coper_reduce_partials; the 3x3 x 32-channel fast path emits one slab per 4 images);
 * per_query: S = B and the same buffers ARE the per-query gradients. */
int coper_conv_bwd_slabs(int B, int H, int W, int KH, int KW, int C, int per_query);
int coper_conv_bwd(const float* dz, const float* x0, int B, int H, int W, const float* wc, int KH, int KW,
                   int C, int per_query, float* dx0, float* dwc_part, float* dbc_part, coper_stream_t stream);
/* coper_bn_act_bwd_apply (with keep_pre = 1) + coper_conv_bwd in one call, for the Conv1BN block that follows the conv
 * (models.py:386-391): dout [B, OH*OW*C] is the gradient w.r.t. the block's OUTPUT, z the conv output, a .. c2 as in
 * coper_bn_act_bwd_apply.  Shared 3x3 x 32-channel filters: one kernel - the block's input gradient is formed while the
 * tile is staged in shared memory and never written to HBM; other shapes run the two kernels through dz_scratch
 * [B, OH*OW*C].  Same bits either way. */
int coper_conv_bwd_bn(const float* dout, const float* z, const float* x0, int B, int H, int W, const float* wc, int KH,
                      int KW, int C, int per_query, const float* a, const float* b, const float* mean,
                      const float* invstd, const float* c1, const float* c2, int relu, float keep_post,
                      const uint64_t* seed_dev, uint64_t salt_post, float* dx0, float* dwc_part, float* dbc_part,
                      float* dz_scratch, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * K5 — tf.layers.batch_normalization (+relu, +dropout) on x [R, C] with C fastest
 * (Conv1BN models.py:386-391 with R=B*OH*OW; FCBN :416-419 with R=B; CPG hidden BN :60-68).
 *   coper_colstats      : per-column partial (sum, sumsq) -> partials [nchunk, C, 2]; nchunk = coper_colstats_chunks(R)
 *   coper_bn_finalize   : use_batch_stats ? batch mean / biased var : moving stats  -> affine a,b
 *                         (out = a*x + b), mean, invstd; optionally updates moving stats in place with
 *                         TF semantics moving = moving*momentum + batch*(1-momentum)
 *                         (bessel != 0: unbiased variance for the moving update, the fused 4-D path).
 *   coper_bn_stats_finalize : coper_colstats + coper_bn_finalize(use_batch_stats = 1) in ONE launch - the block that
 *                         arrives last at *sync_word (a device word, zero before the first call, left zero) finalises
 *                         every channel from the chunk partials (fp64, fixed order: run-to-run identical; the
 *                         two-call form adds the same partials in another fixed order - last-bit differences).
 *                         (The two-call form remains for synchronised batch statistics: partials of all ranks are
 *                         all-gathered between the calls.)  coper_bn_act_bwd_stats_finalize: the same for the backward pair.
 *   coper_bn_act_fwd    : out = dropout_post(relu?(a[c]*x + b[c]))
 *   coper_bn_act_bwd_*  : g1 = dout * dropout_post * relu'(a*x+b); stats (sum g1, sum g1*xhat) ->
 *                         dgamma, dbeta, and dx = a*(g1 - c1 - xhat*c2) [* dropout_pre]. */
int coper_colstats_chunks(int64_t R);
int coper_colstats(const float* x, int64_t R, int C, float* partials, coper_stream_t stream);
int coper_bn_finalize(const float* partials, int nchunk, int64_t R, int C, const float* gamma, const float* beta,
                      float* moving_mean, float* moving_var, float momentum, float eps, int use_batch_stats,
                      int update_moving, int bessel, float* a, float* b, float* mean, float* invstd,
                      coper_stream_t stream);
int coper_bn_stats_finalize(const float* x, int64_t R, int C, float* partials, unsigned int* sync_word,
                            const float* gamma, const float* beta, float* moving_mean, float* moving_var,
                            float momentum, float eps, int update_moving, int bessel, float* a, float* b, float* mean,
                            float* invstd, coper_stream_t stream);
int coper_bn_act_fwd(const float* x, int64_t R, int C, const float* a, const float* b, int relu,
                     float keep_post, const uint64_t* seed_dev, uint64_t salt_post, float* out, coper_stream_t stream);
/* inference (training=False: moving statistics, no dropout): coper_bn_finalize(use_batch_stats = 0) +
 * coper_bn_act_fwd in one launch; same bits */
int coper_bn_act_fwd_moving(const float* x, int64_t R, int C, const float* gamma, const float* beta,
                            const float* moving_mean, const float* moving_var, float eps, int relu, float* out,
                            coper_stream_t stream);
int coper_bn_act_bwd_stats(const float* dout, const float* x, int64_t R, int C, const float* a, const float* b,
                           const float* mean, const float* invstd, int relu, float keep_post,
                           const uint64_t* seed_dev, uint64_t salt_post, float* partials, coper_stream_t stream);
int coper_bn_act_bwd_finalize(const float* partials, int nchunk, int64_t R, int C, int use_batch_stats,
                              float* dgamma, float* dbeta, float* c1, float* c2, coper_stream_t stream);
int coper_bn_act_bwd_stats_finalize(const float* dout, const float* x, int64_t R, int C, const float* a, const float* b,
                                    const float* mean, const float* invstd, int relu, float keep_post,
                                    const uint64_t* seed_dev, uint64_t salt_post, float* partials,
                                    unsigned int* sync_word, int use_batch_stats, float* dgamma, float* dbeta, float* c1,
                                    float* c2, coper_stream_t stream);
int coper_bn_act_bwd_apply(const float* dout, const float* x, int64_t R, int C, const float* a, const float* b,
                           const float* mean, const float* invstd, const float* c1, const float* c2, int relu,
                           float keep_post, const uint64_t* seed_dev, uint64_t salt_post, float keep_pre,
                           uint64_t salt_pre, float* dx, coper_stream_t stream);
/* mask[i] = 1.0f if element i is kept (same hash as the kernels) — the tf.nn.dropout draws of models.py:67-68,
 * 390-391,414-415 made reproducible; exported for the oracle/tests */
int coper_dropout_mask(int64_t n, float keep, const uint64_t* seed_dev, uint64_t salt, float* mask,
                       coper_stream_t stream);
/* x[i] = x[i] * mask(i)/keep (used for the CPG hidden-layer dropout, models.py:67-68) */
int coper_dropout_apply(float* x, int64_t n, float keep, const uint64_t* seed_dev, uint64_t salt,
                        coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * a3+a6 / K2+K3 — fused contextual-parameter generate-and-apply (models.py:70-73 + :412):
 *     y[b,:] = f[b,:] . reshape(c[b,:] . P, [F,d]) + cb[b,:] . Pb   ==   (c (x) f) . P^ + cb . Pb
 * c [B,dc] (relation embedding, or last CPG hidden activation), f [B,F], P [dc, F*d] (viewed [dc,F,d]),
 * cb [B,dcb], Pb [dcb,d].  The per-query weights [B,F,d] are never formed.  Output-dropout
 * (models.py:414-415) is applied to y when keep_out < 1.  workspace: coper_cpg_fc_fwd_workspace_bytes.
 * P_prepared (optional, tensor-pipe precisions): the operand form of P viewed [dc*F, d] (coper_prepare_operand, or
 * kept current by coper_mt_amsgrad); NULL = converted from P inside the call. */
size_t coper_cpg_fc_fwd_workspace_bytes(int B, int dc, int F, int d, int prec);
int coper_cpg_fc_fwd(const float* c, const float* f, const float* P, const void* P_prepared, const float* cb,
                     const float* Pb, int B, int dc, int F, int d, int dcb, float keep_out, const uint64_t* seed_dev,
                     uint64_t salt_out, float* y, void* workspace, size_t workspace_bytes, int prec,
                     coper_stream_t stream);
/* backward (models.py:198 autodiff of the above): given dy [B,d] (already through the dropout mask)
 *   dP [dc,F*d], dPb [dcb,d], df [B,F], dc_out [B,dc], dcb_out [B,dcb].
 * flags (bit mask):
 *   COPER_CPG_BWD_REUSE_FWD (tensor-pipe precisions only): `workspace` is the buffer the matching coper_cpg_fc_fwd
 *     call used and still holds its prepared f and P operands (f, P unchanged since).
 *   COPER_CPG_BWD_INPUT_GRADS_ONLY: compute df, dc_out, dcb_out and leave dP, dPb untouched; the workspace keeps
 *     the operands the weight-gradient half needs.
 *   COPER_CPG_BWD_WEIGHT_GRADS_ONLY: compute only dP, dPb from the operands an INPUT_GRADS_ONLY call with the same
 *     arguments left in `workspace` - the two halves are independent given those operands, so a caller may run
 *     the second on another stream while the backward chain through df / dc_out continues (models.py:198's graph
 *     has no edge between them either). */
#define COPER_CPG_BWD_REUSE_FWD 1
#define COPER_CPG_BWD_INPUT_GRADS_ONLY 2
#define COPER_CPG_BWD_WEIGHT_GRADS_ONLY 4
/* dcb_out += instead of = (a caller whose two generators read the same context - the reference's g_linear setup, context =
 * relation embedding for weights and bias - passes the same [B, dc] buffer as dc_out and dcb_out and gets their sum) */
#define COPER_CPG_BWD_DCB_ACCUMULATE 8
size_t coper_cpg_fc_bwd_workspace_bytes(int B, int dc, int F, int d, int prec);
int coper_cpg_fc_bwd(const float* c, const float* f, const float* P, const void* P_prepared, const float* cb,
                     const float* Pb, const float* dy, int B, int dc, int F, int d, int dcb, float* dP, float* dPb, float* df,
                     float* dc_out, float* dcb_out, void* workspace, size_t workspace_bytes, int prec,
                     int flags, coper_stream_t stream);

/* plain C = op(A) . op(B) (+C) for the small dense layers around the path (CPG hidden projections,
 * models.py:60): row-major; transX != 0 means the stored matrix is the transpose of the operand. */
int coper_sgemm(int transA, int transB, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                float* C, int ldc, int accumulate, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * a7 / K6 — 1-N scorer logits (models.py:433-437): scores[b,n] = q[b,:].E[n,:] + bias[n]
 * E is this rank's shard [Ns, d] (rows of the entity table), scores [B, ld_scores]. */
size_t coper_score1n_workspace_bytes(int B, int64_t Ns, int d, int prec);
int coper_score1n_fwd(const float* q, const float* E, const float* bias, int B, int64_t Ns, int d, float* scores,
                      int64_t ld_scores, void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream);

/* Tensor-pipe operand preparation (COPER_PREC_BF16 / COPER_PREC_TF32X3) for the operands of the tf.matmul calls
 * at models.py:70-73,412,433-437.  The tcgen05 kernels consume operands in
 * "prepared" form: a bf16 copy [rows, ldp] (ldp = cols rounded up to 8), or two fp32 planes (hi = tf32-rounded value,
 * lo = x - hi) of [rows, ldp] (ldp = cols rounded up to 4), or (FP16X3) two fp16 planes of [rows, ldp] (ldp = cols
 * rounded up to 8) holding hi / lo of x * 2^e followed by a 256-byte trailer whose first int32 is e.  Prepare the entity table once per evaluation pass /
 * optimizer step and reuse it across calls with coper_score1n_fwd_prepared (coper_score1n_fwd prepares per call). */
size_t coper_prepared_bytes(int64_t rows, int cols, int prec);
int coper_prepare_operand(const float* src, int64_t rows, int cols, int64_t ld_src, int prec, void* dst,
                          coper_stream_t stream);
int coper_score1n_fwd_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                               float* scores, int64_t ld_scores, int prec, coper_stream_t stream);

/* C = op(A).op(B) on the tensor pipe (tcgen05, fp32 accumulate in TMEM); same layout flags as coper_sgemm
 * (tf.matmul, models.py:60, and its autodiff twins).
 * Operands are prepared into the workspace on every call (bf16 copy or tf32 hi/lo planes). */
size_t coper_tc_gemm_workspace_bytes(int M, int N, int K, int prec);
int coper_tc_gemm(int transA, int transB, int M, int N, int K, const float* A, int lda, const float* B, int ldb,
                  float* C, int ldc, int prec, void* workspace, size_t workspace_bytes, coper_stream_t stream);

/* a7+a9+a10 / K6-K8 — scorer + label-smoothed sigmoid-BCE + its gradient (models.py:433-437,448-453,198):
 *   s = q.E^T + bias;  z' = bit ? pos_target : neg_target   (pos = (1-eps)+1/N, neg = 1/N; models.py:450)
 *   loss_sum = sum_{b,n} max(s,0) - s z' + log1p(exp(-|s|))   (caller divides by B*N_total)
 *   G[b,n]   = (sigmoid(s) - z') * inv_count                    (inv_count = 1/(B*N_total))
 *   dq = G.E, dE = G^T.q, dbias = sum_b G.
 * label_bits: FP32 engine - query-major rows [B, ceil(Ns/32)] (coper_csr_to_bits: bit n of row b = 1 iff entity n
 * is a positive of query b); tensor-pipe engines - the ENTITY-MAJOR matrix [Ns, ceil(B/32)] (coper_csr_to_bits_t);
 * G is caller-provided scratch of coper_score1n_bce_G_bytes (never read by the host; 128-byte aligned) holding
 * dL/dS with row pitch ldG (a multiple of 32, >= Ns): fp32 [B, ldG] (FP32), bf16 [B, ldG] (BF16) or tf32
 * hi/lo planes 2 x fp32 [B, ldG] (TF32X3) - on the tensor-pipe paths G is written by the scorer epilogue
 * directly in operand form and consumed by the dq / dE GEMMs through TMA.  workspace must be 256-byte
 * aligned.  loss_sum is a device double.  E_prepared (optional, tensor-pipe precisions): operand form of E
 * [Ns, d]; NULL = converted from E inside the call. */
size_t coper_score1n_bce_workspace_bytes(int B, int64_t Ns, int d, int prec);
size_t coper_score1n_bce_G_bytes(int B, int64_t Ns, int prec);
int coper_score1n_bce_fwd_bwd(const float* q, const float* E, const void* E_prepared, const float* bias,
                              const uint32_t* label_bits,
                              int B, int64_t Ns, int d, float pos_target, float neg_target, float inv_count,
                              double* loss_sum, void* G, int64_t ldG, float* dq, float* dE, float* dbias,
                              void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream);

/* coper_score1n_bce_fwd_bwd that additionally writes *dE_sumsq = sum of the squares of the dE it stored (fp64, fixed
 * order; tensor-pipe precisions only - the dE GEMM epilogue accumulates it): the global-norm clip (models.py:199) then
 * does not re-read the [Ns, d] gradient.  See COPER_GRAD_NORM_EXTERNAL. */
int coper_score1n_bce_fwd_bwd_norm(const float* q, const float* E, const void* E_prepared, const float* bias,
                                   const uint32_t* label_bits, int B, int64_t Ns, int d, float pos_target,
                                   float neg_target, float inv_count, double* loss_sum, void* G, int64_t ldG, float* dq,
                                   float* dE, float* dbias, double* dE_sumsq, void* workspace, size_t workspace_bytes,
                                   int prec, coper_stream_t stream);

/* The split form of coper_score1n_bce_fwd_bwd_norm (tensor-pipe precisions): call it with dE == NULL - loss, dq and G
 * are produced; the entity-gradient GEMM and the reduction of the dbias slabs are skipped (`dbias` is not written) - and
 * then coper_score1n_bce_dE with the same G / workspace (which still holds the prepared q and the dbias slabs):
 * dE = G^T . q (+ *dE_sumsq, optional) and dbias.  Neither depends on dq, and nothing the rest of the backward pass
 * (models.py:198 through the FC / conv layers) does depends on them, so the host may enqueue this call on a second
 * stream: the HBM-bound GEMM then runs under the latency-bound backward chain. */
int coper_score1n_bce_dE(const void* G, int B, int64_t Ns, int d, float inv_count, float* dE, double* dE_sumsq,
                         float* dbias, void* workspace, size_t workspace_bytes, int prec, coper_stream_t stream);

/* a8 / SURVEY §8f-2 — SAMPLED-label scorer (models.py:438-443), loss (:448-453) and gradients: what the shipped
 * big-dataset configs train with (training.num_labels = 100 / 1000).  lookup int32 [B, L] entity ids
 * (batch['lookup_values'], models.py:165), labels fp32 [B, L] (batch['e2_multi'] in sampled mode):
 *   s[b,l] = q[b].E[lookup[b,l]] + bias[lookup[b,l]]        (scores [B, L], optional output)
 *   z'     = one_minus_eps * label + inv_num_ent             (models.py:450: + 1/num_ent, also in sampled mode)
 *   loss_sum = sum BCE(s, z');  g[b,l] = (sigmoid(s) - z') * inv_count   (inv_count = 1/(B*L))
 *   dq[b]  = sum_l g[b,l] E[lookup[b,l]]
 * TF's gradient of the two gathers is an IndexedSlices (values g[b,l]*q[b] / g[b,l] at row lookup[b,l]); the sparse
 * AMSGrad rule and the slice-wise global norm need per entity row the SUM of its slices and the sum of their SQUARES:
 *   dE_sum, dE_sq [N, d], dbias_sum, dbias_sq [N] are ACCUMULATED (zero them first; the e1-gather slices are added on
 *   top with coper_segscatter_add).  Exact fp32 (gather-bound, no tensor-pipe variant); deterministic. */
size_t coper_score_sampled_workspace_bytes(int B, int L);

/* SURVEY §8f-2, on-device label sampling — replaces the input pipeline's _sample_negatives map (data.py:228-277) and
 * its [B, L] host->device copies.  Per query row b, from the CSR list of its known-true tails (rowptr int32 [B+1],
 * col int32 [nnz]; the e2_multi id lists, data.py:574-594), with n_pos_needed = int(1/(1+prop_negatives) * L):
 *   P <= n_pos_needed : all P positives in random order, then L - P sampled entities            (data.py:244-251)
 *   P >  n_pos_needed : n_pos = L - min(N, L - n_pos_needed) randomly chosen positives, then the rest (data.py:253-263)
 * The sampled entities are the prefix of a keyed pseudorandom PERMUTATION of [0, N) (4-round Feistel network + cycle
 * walking; key = *seed_dev + salt, row): distinct within a row and, as in the reference, positives are not removed
 * from them - a sampled entity that is a true tail gets label 1.  lookup int32 [B, L], labels fp32 [B, L] are the
 * batch['lookup_values'] / batch['e2_multi'] of models.py:135-152,165.  Needs L <= N < 2^31. */
int coper_sample_labels(const int32_t* rowptr, const int32_t* col, int B, int64_t N, int L, int n_pos_needed,
                        const uint64_t* seed_dev, uint64_t salt, int32_t* lookup, float* labels, coper_stream_t stream);
int coper_score_sampled_bce_fwd_bwd(const float* q, const float* E, const float* bias, const int32_t* lookup,
                                    const float* labels, int B, int L, int64_t N, int d, float one_minus_eps,
                                    float inv_num_ent, float inv_count, double* loss_sum, float* scores, float* g,
                                    float* dq, float* dE_sum, float* dE_sq, float* dbias_sum, float* dbias_sq,
                                    void* workspace, size_t workspace_bytes, coper_stream_t stream);

/* The same step on ONE entity shard (the entity-sharded multi-GPU schedules): lookup holds GLOBAL ids [B, L]; E / bias
 * are this rank's rows [row_hi - row_lo, d] / [row_hi - row_lo] of the [N, d] / [N] table.  Only positions whose id lies
 * in [row_lo, row_hi) are scored: their scores / g entries are written with exactly the values the unsharded call
 * writes for the same q; the entries of all other positions are LEFT UNTOUCHED.  loss_sum and dq [B, d] are this rank's
 * PARTIALS (a query none of whose lookups the rank owns gets dq = 0): summed over the shards of a partition of [0, N)
 * they are the unsharded values up to fp32 summation order.  dE_sum, dE_sq [row_hi - row_lo, d] and dbias_sum, dbias_sq
 * [row_hi - row_lo] are shard-local and accumulated as above; each row equals, bit for bit, the matching row of the
 * unsharded result (its slices are summed in the same position order).  Workspace:
 * coper_score_sampled_sharded_workspace_bytes (the [B*L] local sort keys on top of the unsharded layout).  Needs
 * 0 <= row_lo < row_hi <= N < 2^31, B*L < 2^31, d <= 256. */
size_t coper_score_sampled_sharded_workspace_bytes(int B, int L);
int coper_score_sampled_bce_fwd_bwd_sharded(const float* q, const float* E, const float* bias, const int32_t* lookup,
                                            const float* labels, int B, int L, int64_t N, int d, float one_minus_eps,
                                            float inv_num_ent, float inv_count, double* loss_sum, float* scores,
                                            float* g, float* dq, float* dE_sum, float* dE_sq, float* dbias_sum,
                                            float* dbias_sq, int64_t row_lo, int64_t row_hi, void* workspace,
                                            size_t workspace_bytes, coper_stream_t stream);

/* a8, forward only — scores of GIVEN candidate entities (models.py:438-443, predictions_lookup for arbitrary ids) and
 * the filtered rank of the gold tail among them; the [B, N] logits are never formed.  cand int32 [B, C] holds GLOBAL
 * entity ids; E / bias are this rank's rows [row_hi - row_lo, d] / [row_hi - row_lo] of the table.
 *   coper_score_candidates: scores fp32 [B, C]; a position whose id lies in [row_lo, row_hi) gets
 *       s = q[b].E[id] + bias[id], bit-identical to the score coper_score_sampled_bce_fwd_bwd writes for the same q,
 *       table and id (the same lane-strided fp32 fmaf chain, warp reduction and bias add); every other position
 *       (padding -1, ids outside the table, ids another shard owns) gets exactly 0 and reads nothing - summed over the
 *       shards of a partition of [0, N) the scores are the unsharded ones.  The gold logit of coper_candidate_rank is
 *       this call with C = 1 and cand = e2 (summed over the shards).
 *   coper_candidate_rank: counts ACCUMULATED into n_greater / n_equal int32 [B] (zero them first):
 *       n_greater[b] += #{j : cand[b,j] owned, cand[b,j] != e2[b], !filtered(b, cand[b,j]), s(b,j) >  gold[b]}
 *       n_equal[b]   += the same with ==.   rank = 1 + sum over shards of n_greater; duplicates count once per
 *       occurrence.  filter_bits: the shard's query-major rows of coper_csr_to_bits (entity_major = 0) or the
 *       entity-major matrix of coper_csr_to_bits_t (entity_major = 1); NULL = unfiltered.  e2 int32 [B].
 * Exact fp32 from the master table for every engine (gather-bound, no tensor-pipe variant); deterministic.  Needs
 * 1 <= B, 1 <= C, B*C < 2^31, 0 <= row_lo < row_hi < 2^31 (COPER_ERR_INVALID_ARG), d <= 256 (COPER_ERR_UNSUPPORTED). */
int coper_score_candidates(const float* q, const float* E, const float* bias, const int32_t* cand, int B, int C, int d,
                           int64_t row_lo, int64_t row_hi, float* scores, coper_stream_t stream);
int coper_candidate_rank(const float* q, const float* E, const float* bias, const int32_t* cand, const int32_t* e2,
                         int B, int C, int d, int64_t row_lo, int64_t row_hi, const float* gold,
                         const uint32_t* filter_bits, int entity_major, int32_t* n_greater, int32_t* n_equal,
                         coper_stream_t stream);

/* labels / filters: CSR positives (rowptr int32 [B+1], col int32 [nnz], global entity ids) -> bit rows for
 * the shard [ent_lo, ent_hi); replaces the dense fp32 multi-hot of data.py:182-186,318-322. */
int coper_csr_to_bits(const int32_t* rowptr, const int32_t* col, int B, int64_t ent_lo, int64_t ent_hi,
                      uint32_t* bits, coper_stream_t stream);
/* dense fp32 multi-hot [B, N] (the reference batch schema, models.py:144) -> bits (value == 1.0f) */
int coper_dense_to_bits(const float* dense, int B, int64_t N, uint32_t* bits, coper_stream_t stream);
/* ENTITY-MAJOR bit matrix (the multi-hot e2_multi of models.py:144 / the filter of metrics.py:44-46, one bit per
 * pair) used by the tensor-pipe scorers (one entity per epilogue thread):
 *   bits_t [ent_hi - ent_lo, ceil(B/32)]: bit (b & 31) of word (n, b >> 5) = 1 iff entity ent_lo + n is a positive /
 *   filtered tail of query b.  coper_bits_t_set ORs in the bits (ent[b], b) - used to add the gold entity to the
 *   filter set so the fused ranking kernel needs no per-element identity test. */
int coper_csr_to_bits_t(const int32_t* rowptr, const int32_t* col, int B, int64_t ent_lo, int64_t ent_hi,
                        uint32_t* bits_t, coper_stream_t stream);
int coper_dense_to_bits_t(const float* dense, int B, int64_t N, int64_t ld_dense, uint32_t* bits_t,
                          coper_stream_t stream);
int coper_bits_t_set(const int64_t* ent, int B, int64_t ent_lo, int64_t ent_hi, uint32_t* bits_t,
                     coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * a11 / K10 — filtered rank (metrics.py:44-51): for each query b over this shard's scores [B, ld]
 *   n_greater[b] += #{n : n != gold, !filter[b,n], s[b,n] >  gold_score[b]}
 *   n_equal[b]   += #{n : n != gold, !filter[b,n], s[b,n] == gold_score[b]}
 * rank = 1 + sum over shards of n_greater.  gold_local[b] = e2[b] - ent_lo (may be out of range).
 * coper_gold_scores extracts gold_score[b] = scores[b, gold_local[b]] (0 if not owned). Counts are
 * ACCUMULATED into n_greater / n_equal (zero them first). */
int coper_gold_scores(const float* scores, int64_t ld, int B, int64_t Ns, const int64_t* e2, int64_t ent_lo,
                      float* gold, coper_stream_t stream);
int coper_filtered_rank(const float* scores, int64_t ld, int B, int64_t Ns, const int64_t* e2, int64_t ent_lo,
                        const float* gold, const uint32_t* filter_bits, int32_t* n_greater, int32_t* n_equal,
                        coper_stream_t stream);

/* a7 + a11 fused (tensor-pipe precisions): filtered-rank counts taken straight from the scorer's TMEM
 * accumulators - the [B, Ns] logits are never written.  Operands in prepared form (coper_prepare_operand).
 *   coper_score1n_gold_prepared: gold[b] = q[b].E[e2[b]-ent_lo] + bias[...] if this shard owns e2[b], else 0;
 *       computed by the same tcgen05 instruction sequence as the ranking pass, so it is bit-identical to the
 *       logit that pass sees (sum gold over shards before ranking).  workspace: coper_score1n_rank_workspace_bytes.
 *   coper_score1n_rank_prepared: counts ACCUMULATED into n_greater / n_equal exactly as coper_filtered_rank does;
 *       filter_bits_t is the entity-major matrix (coper_csr_to_bits_t) and must contain the gold entity of every
 *       query (coper_bits_t_set) - metrics.py:44-46 excludes it from the comparison. */
size_t coper_score1n_rank_workspace_bytes(int B, int d, int prec);
int coper_score1n_gold_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                                const int64_t* e2, int64_t ent_lo, float* gold, void* workspace,
                                size_t workspace_bytes, int prec, coper_stream_t stream);
int coper_score1n_rank_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                                const float* gold, const uint32_t* filter_bits_t, int32_t* n_greater,
                                int32_t* n_equal, int prec, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * Top-k link prediction: for each query b the k best entities n of this shard [ent_lo, ent_lo + Ns) under
 *   score s[b, n] = q[b].E[n] + bias[n]   (the fp32 logits the engine's own scorer writes, bit for bit),
 *   eligible: every entity, or (filter bits != NULL) every entity whose filter bit is clear,
 *   order: score descending, then global entity id ascending (a total order: the result does not depend on tile
 *          schedule, grid size, shard count or list order; -0 and +0 compare equal).  Scores are assumed finite.
 * Output: out_scores fp32 [B, k], out_ids int64 [B, k] (global ids ent_lo + n), sorted by that order; a query with
 * fewer than k eligible entities is padded with (-inf, -1).  1 <= k <= COPER_TOPK_MAX, ent_lo + Ns < 2^31 - 1.
 *   coper_score1n_topk_prepared: tensor-pipe engines, fused with the scorer (the logits never leave TMEM); same
 *       operands and configuration choice as coper_score1n_fwd_prepared.  filter_bits_t: the entity-major matrix
 *       (coper_csr_to_bits_t), NULL = unfiltered.  workspace: coper_score1n_topk_workspace_bytes (256-byte aligned).
 *   coper_topk_scores: logits already in HBM, scores [B, ld] (fp32 engine: coper_score1n_fwd); filter_bits: the
 *       query-major rows of coper_csr_to_bits, NULL = unfiltered.  workspace: coper_topk_scores_workspace_bytes.
 *   coper_topk_merge: [n_lists, B, k] lists padded with (-inf, -1) -> [B, k] (e.g. the per-shard results of a
 *       sharded model).  Deterministic and independent of the order of the lists. */
#define COPER_TOPK_MAX 128
size_t coper_score1n_topk_workspace_bytes(int B, int64_t Ns, int d, int k, int prec);
int coper_score1n_topk_prepared(const void* q_prep, const void* E_prep, const float* bias, int B, int64_t Ns, int d,
                                const uint32_t* filter_bits_t, int64_t ent_lo, int k, float* out_scores,
                                int64_t* out_ids, void* workspace, size_t workspace_bytes, int prec,
                                coper_stream_t stream);
size_t coper_topk_scores_workspace_bytes(int B, int64_t Ns, int k);
int coper_topk_scores(const float* scores, int64_t ld, int B, int64_t Ns, const uint32_t* filter_bits, int64_t ent_lo,
                      int k, float* out_scores, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                      coper_stream_t stream);
int coper_topk_merge(const float* in_scores, const int64_t* in_ids, int n_lists, int B, int k, float* out_scores,
                     int64_t* out_ids, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * a10 scatter / K8(3) — gradient of the embedding gathers (IndexedSlices -> dense, models.py:198):
 *   dst[idx[i] - row_lo, :] += src[i, :] for row_lo <= idx[i] < row_hi; one writer per destination row
 *   (sort by key, warp per segment, fixed summation order) -> deterministic. */
size_t coper_segscatter_workspace_bytes(int M);
/* M <= 4096 (one batch of gathers): sort-free variant that can also accumulate the per-row sums of the SQUARED source
 * rows into dst_sq (NULL = skip) - the IndexedSlices bookkeeping of the sparse AMSGrad rule (utils/amsgrad.py:161-189)
 * and of tf.clip_by_global_norm's slice-wise norm (models.py:199).
 * Same summation order (index order) as coper_segscatter_add, which uses this path for small M. */
int coper_segscatter_add_sq(const int64_t* idx, int M, const float* src, int width, float* dst, float* dst_sq,
                            int64_t row_lo, int64_t row_hi, coper_stream_t stream);
/* Two independent small scatters of one step in ONE launch, each with coper_segscatter_add_sq's arguments (the
 * head-entity and relation gathers' gradients, models.py:176-178).  M_b == 0: job a alone (idx_b, src_b, dst_b may be
 * NULL).  norm_delta_a (NULL = skip) receives, per position i of idx_a, norm_delta_a[i] = sum_c (new^2 - old^2) over
 * the destination row position i updated (0 for non-heads / rows of other shards): the correction of a squared
 * gradient norm that was taken before this scatter (tf.clip_by_global_norm over the dense ent_emb gradient,
 * models.py:198-199). */
int coper_segscatter_add_pair(const int64_t* idx_a, int M_a, const float* src_a, int width_a, float* dst_a,
                              float* dst_sq_a, int64_t lo_a, int64_t hi_a, double* norm_delta_a, const int64_t* idx_b,
                              int M_b, const float* src_b, int width_b, float* dst_b, float* dst_sq_b, int64_t lo_b,
                              int64_t hi_b, coper_stream_t stream);
int coper_segscatter_add(const int64_t* idx, int M, const float* src, int width, float* dst, int64_t row_lo,
                         int64_t row_hi, void* workspace, size_t workspace_bytes, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * generic deterministic reductions
 *   coper_reduce_partials: out[n] = (accumulate ? out[n] : 0) + scale * sum_s in[s, n]   (fixed order, fp64 acc)
 *   coper_sumsq          : partials[slot*COPER_SUMSQ_BLOCKS + blk] = sum of squares of a strided chunk of x
 *   coper_clip_scale     : norm = sqrt(sum of partials[0 .. n_slots*COPER_SUMSQ_BLOCKS)); out[0] = clip / max(norm, clip);
 *                          out[1] = norm  (tf.clip_by_global_norm, models.py:199). */
#define COPER_SUMSQ_BLOCKS 256
int coper_reduce_partials(const float* in, int S, int64_t n, float scale, int accumulate, float* out,
                          coper_stream_t stream);
/* two reductions with the same slab count in one launch (the conv filter / bias gradient slabs of coper_conv_bwd) */
int coper_reduce_partials2(const float* in_a, int64_t n_a, float* out_a, const float* in_b, int64_t n_b, float* out_b,
                           int S, float scale, int accumulate, coper_stream_t stream);
int coper_sumsq(const float* x, int64_t n, int slot, double* partials, coper_stream_t stream);
int coper_clip_scale(const double* partials, int n_slots, float clip_norm, float* out2, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * f-1 — AMSGrad dense apply (utils/amsgrad.py:130-159) with the clip scale read from device memory:
 *   g = grad * clip_scale[0];
 *   bug_compat != 0 (reference as written: m, v slots never accumulate; m/v may be NULL):
 *       vhat = max(vhat, (1-b2) g^2);  theta -= lr_t * (1-b1) g / (sqrt(vhat) + eps)
 *   else (textbook): m = b1 m + (1-b1) g; v = b2 v + (1-b2) g^2; vhat = max(vhat, v); theta -= lr_t m/(sqrt(vhat)+eps)
 * lr_t = lr * sqrt(1-b2^t)/(1-b1^t) (amsgrad.py:137) is read from step_state[0] on the device.
 * coper_step_state_advance (1 thread): step_state = {lr_t, beta1_power, beta2_power, unused};
 *   lr_t <- lr*sqrt(1-b2p)/(1-b1p); then b1p *= b1, b2p *= b2 (amsgrad.py:230-241; powers start at b1, b2);
 *   *seed_dev += 1 (fresh dropout masks).  Call once per step BEFORE the update kernels. */
int coper_step_state_advance(float* step_state, uint64_t* seed_dev, float lr, float beta1, float beta2,
                             coper_stream_t stream);
int coper_amsgrad_step(float* theta, const float* grad, float* m, float* v, float* vhat, int64_t n,
                       const float* step_state, float beta1, float beta2, float eps, const float* clip_scale,
                       int bug_compat, coper_stream_t stream);

/* ------------------------------------------------------------------------------------------------
 * multi-tensor form of the clip + AMSGrad tail (models.py:199, utils/amsgrad.py:130-159): the whole
 * variable list is processed by ONE launch per phase instead of one per variable.
 *   descs         device array [n_tensors] describing every trainable (pointers as in coper_amsgrad_step);
 *                 `prepared` (optional) is refreshed with the tensor-pipe operand form of the UPDATED variable
 *                 (bf16 copy, or tf32 hi plane followed by the lo plane; requires row pitch == row length),
 *                 so the next step's GEMMs need no separate conversion pass.
 *                 mode = COPER_GRAD_DENSE: the dense rule of coper_amsgrad_step.  mode = COPER_GRAD_INDEXED_SLICES: the
 *                 variable is read only through tf.nn.embedding_lookup (rel_emb, models.py:178), TF hands the
 *                 optimizer an IndexedSlices and runs _apply_sparse_shared (utils/amsgrad.py:161-189), where the
 *                 slots DO accumulate: `grad` = sum of the slices per row, `grad_sq` = sum of the SQUARED slices
 *                 per row (each slice squared on its own); m <- b1 m + (1-b1) c grad; v <- b2 v + (1-b2) c^2 grad_sq;
 *                 vhat <- max(vhat, v); theta -= lr_t m / (sqrt(vhat) + eps) on the whole variable (c = clip scale;
 *                 m, v required).  The squared norm such a variable contributes to tf.clip_by_global_norm is
 *                 sum(grad_sq) - slices sharing an index are not summed first (clip_ops.global_norm on .values).
 *   chunks        device int32 [n_chunks][2] = (tensor id, chunk index); chunk = COPER_MT_CHUNK elements;
 *                 sorted by tensor id; chunk_offsets int32 [n_tensors + 1] = first chunk of each tensor.
 *   coper_mt_sumsq   -> tensor_sumsq[t] = |grad_t|^2 (fp64, fixed order; chunk_partials is scratch [n_chunks])
 *   coper_clip_scale_n(tensor_sumsq, n_tensors, ...) -> {clip / max(norm, clip), norm}
 *   coper_mt_amsgrad -> the update of coper_amsgrad_step for every tensor. */
#define COPER_MT_CHUNK 16384
/* COPER_GRAD_NORM_EXTERNAL (OR-ed into mode): coper_mt_sumsq does not read this gradient - its squared norm is written
 * into tensor_sumsq[t] by coper_sumsq_combine AFTER coper_mt_sumsq, from the partial sums the kernel that produced the
 * gradient emitted (coper_score1n_bce_fwd_bwd_norm) and the corrections of the scatter that touched it afterwards
 * (coper_segscatter_add_pair's norm_delta_a): the [N, d] entity gradient is then read once (by the update), not twice. */
enum { COPER_GRAD_DENSE = 0, COPER_GRAD_INDEXED_SLICES = 1, COPER_GRAD_NORM_EXTERNAL = 2 };
typedef struct {
  float* theta;
  const float* grad;
  float* m;
  float* v;
  float* vhat;
  void* prepared;
  const float* grad_sq;
  int64_t n;
  int32_t prepared_prec;
  int32_t mode;
} coper_param_desc;
/* out[0] = sum(parts) + sum(deltas), fp64, fixed order, clamped at 0 (tf.clip_by_global_norm, models.py:199: the
 * squared norm of one gradient assembled from its producers' partial sums). */
int coper_sumsq_combine(const double* parts, int n_parts, const double* deltas, int n_deltas, double* out,
                        coper_stream_t stream);
int coper_mt_sumsq(const coper_param_desc* descs, int n_tensors, const int32_t* chunks, int n_chunks,
                   const int32_t* chunk_offsets, double* chunk_partials, double* tensor_sumsq, coper_stream_t stream);
int coper_clip_scale_n(const double* sums, int n, float clip_norm, float* out2, coper_stream_t stream);
/* coper_mt_sumsq + coper_sumsq_combine (into tensor_sumsq[ext_tensor]; ext_tensor < 0: none) + coper_clip_scale_n
 * (clip_out == NULL: skipped - a multi-GPU caller all-reduces the sharded tensors' sums first) as two launches instead
 * of four; same summation orders, same bits.  n_chunks == 0: every norm is external, only the finishing launch runs. */
int coper_mt_sumsq_clip(const coper_param_desc* descs, int n_tensors, const int32_t* chunks, int n_chunks,
                        const int32_t* chunk_offsets, double* chunk_partials, double* tensor_sumsq, int ext_tensor,
                        const double* ext_parts, int n_ext_parts, const double* ext_deltas, int n_ext_deltas,
                        float clip_norm, float* clip_out, coper_stream_t stream);
int coper_mt_amsgrad(const coper_param_desc* descs, const int32_t* chunks, int n_chunks, const float* step_state,
                     float beta1, float beta2, float eps, const float* clip_scale, int bug_compat,
                     coper_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* COPER_H_ */
