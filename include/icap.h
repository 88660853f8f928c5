/*
 * libicap.so -- C ABI of the B200-native caption-generator hot path.
 *
 * The reference (shao-chi/Image-Caption) is pure Python/PyTorch and has NO native boundary
 * (SURVEY.md section 2.1); this header is the boundary a native port of its hot path binds to.
 * Each entry point names the reference code whose arithmetic it replaces (file:line relative to
 * the reference repo).  INTEGRATION.md shows the ctypes stub a maintainer adds on the reference
 * side.
 *
 * Conventions
 *   - plain C: raw DEVICE pointers (tensor.data_ptr()), int64 sizes / leading dimensions in
 *     ELEMENTS, dtype enums, and a cudaStream_t passed as void*.  No torch types.
 *   - return value: 0 = OK, >0 = cudaError_t of the failed launch, <0 = argument/shape error.
 *     icap_last_error() returns a thread-local description.  Nothing throws.
 *   - every function only enqueues work on `stream` (no host sync, no allocation) and is therefore
 *     CUDA-graph capturable.  The caller owns all memory.
 *   - sm_100a only; icap_sm_check() refuses anything else.  There is no CPU fallback.
 */
#ifndef ICAP_H_
#define ICAP_H_
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define ICAP_F32 0
#define ICAP_BF16 1

/* epilogues of icap_gemm */
#define ICAP_EPI_NONE 0
#define ICAP_EPI_RELU 1      /* C = relu(AB + bias)            FeedForward position_wise_1 + ReLU, modules.py:113-114 */
#define ICAP_EPI_RELU_MASK 2 /* C = (AB) * (aux > 0)           backward of that ReLU                                   */
/* C = AB + bias as usual (bf16 C), and aux = fp32 statistics OUT: per row and per 128 columns a float4 (largest value,
 * second largest, sum of exp(x - largest), 0) of the ROUNDED values that were stored; ldaux >= 8 * ceil(N / 256) floats.
 * The classifier of a beam-search step (model.py:176-186): icap_beam_select takes the buffer instead of making its own
 * statistics pass over the V logits of every row. */
#define ICAP_EPI_ROWSTATS 3
/* flag, OR-ed into `epilogue`: B and bias are WEIGHTS; the tcgen05 kernels then fetch their first B stages before their
 * grid dependency has resolved.  Such a pre-wait read may overlap every kernel of the stream back to, and including, the
 * nearest earlier kernel that waits before it lets its dependents start (every kernel of this library except the
 * tcgen05 GEMMs of icap_gemm and icap_gemm_ln, which let them start first; a kernel launched without PDL also counts):
 * none of those kernels may write the data read early. */
#define ICAP_EPI_B_STATIC 16

int icap_version(void);
const char* icap_last_error(void);
int icap_sm_check(int device);
/* on=1: tcgen05 GEMMs are launched with programmatic stream serialization (PDL): their per-CTA setup overlaps
 * the tail of the previous kernel in the stream (griddepcontrol.wait guards every dependent access). */
int icap_set_pdl(int on);

/* C[M,N] (+)= op(A)[M,K] . op(B)[K,N] (+ bias[N]) with an optional activation epilogue.
 *   a_kmajor=1: A stored [M][K]; 0: stored [K][M].   b_kmajor=1: B stored [N][K]; 0: stored [K][N].
 *   ab_dtype ICAP_F32 : true-fp32 SIMT kernel (fp32 parity mode), C fp32.
 *   ab_dtype ICAP_BF16: TMA + tcgen05.mma + TMEM kernel, C fp32 or bf16 (c_dtype).
 *   accumulate=1: C += ...; split_k>1 (needs accumulate=1, fp32 C, no bias) reduces K-slices with red.add;
 *   split_k<=0 (bf16): the kernel picks the split that fills the SMs (1 unless accumulate=1 and C is fp32).
 *   bf16 C with accumulate=1: C = bf16(C + bf16(v)), v = the fp32 result of the epilogue; the TMA reduce-add and the
 *   direct stores (C not 16-byte aligned, or rows of ldc or N elements not whole 16-byte chunks) both round v first, so
 *   the bits of C do not depend on its alignment.  fp32 C: C + v, rounded once.
 *   Nothing outside the [M, N] block of C is written, whatever ldc (C's rows leave through TMA stores only when N
 *   elements fill whole 16-byte chunks).  ICAP_EPI_ROWSTATS takes any N.  The fp32 kernel takes any M < 2^31.
 * Replaces every nn.Linear / torch.matmul weight contraction of the path and their autograd
 * backward: modules.py:42-44,59-60,72-77,86,100-101,113-116; model.py:68,93,235,246,295-306,392-394,433. */
int icap_gemm(int ab_dtype, int a_kmajor, int b_kmajor, int64_t M, int64_t N, int64_t K, const void* A, int64_t lda,
              const void* B, int64_t ldb, void* C, int64_t ldc, int c_dtype, const float* bias, int epilogue,
              const void* aux, int64_t ldaux, int accumulate, int split_k, void* stream);
/* The library reads its ICAP_* environment switches once; call this after changing the environment of the running
 * process (tests, tools).  icap_debug_trace (tools/, not used by the product path): record %globaltimer stamps of CTA 0
 * of every following tcgen05 GEMM launch into buf (device memory, 16 x uint64 per slot, slot = launch number % nslots;
 * buf = NULL: off). */
int icap_reload_env(void);
/* Width of the persistent grid of the following icap_gemm(bf16) launches (0 = all SMs): data parallel training leaves a
 * few SMs to the NCCL all-reduce kernels that overlap the backward.  A 256x256 CTA pair needs two SMs: with n = 1 (or
 * ICAP_GEMM_SMS=1) every GEMM runs on 128-row tiles, even when ICAP_GEMM_BN=pair asks for the pair. */
int icap_set_gemm_sms(int n);
int icap_debug_trace(unsigned long long* buf, int nslots);

/* Fused multi-head attention over packed projections (one CTA per (batch, head)).
 *   q rows b*Lq+i at q + row*ldq + h*dk; k/v rows b*Lk+j likewise; o rows at o + row*ldo + h*dv.
 *   key j of batch b is masked iff (kvalid && !kvalid[b*Lk+j]) || (causal && j > i).
 *   p_drop / seed: dropout on the probabilities (fixed 0.1 in the reference, modules.py:8,24); the effective
 *   seed is seed + seed_dev[0] * golden-ratio (seed_dev nullable) so a replayed CUDA graph gets fresh masks.
 *   Probability (b, h, i, j) is dropout element ((b*H + h)*Lq + i) * ld + j with ld = 16, 32, 48, 64 or 128 (the
 *   smallest of these >= Lk) for Lk <= 128 and (Lk + 3) & ~3 above.  Every kernel that icap_mha_fwd and icap_mha_bwd
 *   may choose uses this index, so the backward regenerates the forward's mask whichever kernel runs each of them.
 *   attn_mean (nullable, fp32 [B,Lq,Lk], pre-zeroed): += P / H  (greedy visualisation, model.py:123).
 * Replaces ScaledDotProductAttention.forward and the head split/merge, modules.py:16-27,72-84. */
int icap_mha_fwd(int dtype, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv, const void* q,
                 int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o, int64_t ldo,
                 const uint8_t* kvalid, int causal, float p_drop, uint64_t seed, const int* seed_dev, float* attn_mean,
                 void* stream);
int icap_mha_bwd(int dtype, int64_t B, int64_t H, int64_t Lq, int64_t Lk, int64_t dk, int64_t dv, const void* q,
                 int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, const void* dout, int64_t lddo,
                 void* dq, int64_t lddq, void* dk_out, int64_t lddk, void* dv_out, int64_t lddv,
                 const uint8_t* kvalid, int causal, float p_drop, uint64_t seed, const int* seed_dev, void* stream);

/* y = (LayerNorm(dropout(a) + res[row % res_rows]) * gamma + beta) * rowscale[row]   (eps given).
 *   a: [M,d] of a_dtype (the GEMM output); res/y: act_dtype; write_sum=1 stores the pre-norm sum
 *   back into a (needed by the backward); mean/rstd: fp32 [M] (nullable in inference).
 *   Dropout element index of a[row, col]: row*d + col (same seed rule as icap_mha_fwd); icap_add_ln_bwd(_rows)
 *   regenerates the mask from the same seed / seed_dev.
 * Replaces Dropout + residual + LayerNorm of modules.py:86-90,117-120, the embedding norms
 * model.py:307-309,433-436 and `output *= non_pad_mask`, modules.py:154-155,203-204. */
int icap_add_ln_fwd(int a_dtype, int act_dtype, int64_t M, int64_t d, void* a, const void* res, int64_t res_rows,
                    const float* gamma, const float* beta, const float* rowscale, void* y, float* mean_out,
                    float* rstd_out, int write_sum, float p_drop, uint64_t seed, const int* seed_dev, float eps,
                    void* stream);
/* dy = dy1 (+ dy2); ds -> residual branch, da = dropout-masked ds -> GEMM branch (nullable: use ds when p=0);
 * dgamma/dbeta/dbias2 (fp32 [d], accumulated; dbias2 = column sums of da, nullable). */
int icap_add_ln_bwd(int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                    const float* mean, const float* rstd, const float* gamma, const float* rowscale, void* ds, void* da,
                    float* dgamma, float* dbeta, float* dbias2, float p_drop, uint64_t seed, const int* seed_dev,
                    void* stream);

/* The two halves of icap_add_ln_bwd as separate launches: _rows writes ds / da (critical path of the backward),
 * _params accumulates dgamma / dbeta / dbias2 from the same inputs plus the ds / da written by _rows (may run later,
 * on another stream). */
int icap_add_ln_bwd_rows(int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                         const float* mean, const float* rstd, const float* gamma, const float* rowscale, void* ds, void* da,
                         float p_drop, uint64_t seed, const int* seed_dev, void* stream);
int icap_add_ln_bwd_params(int act_dtype, int64_t M, int64_t d, const void* dy1, const void* dy2, const void* s,
                           const float* mean, const float* rstd, const float* rowscale, const void* ds, const void* da,
                           float* dgamma, float* dbeta, float* dbias2, void* stream);

/* y = (LayerNorm(dropout(A[M,K] . W[N,K]^T + bias) + res) * gamma + beta) * rowscale in ONE tcgen05 kernel (bf16, N = d in
 * {128, 256, 512, 1024}): the N columns of a 128-row block are split over a thread-block cluster of N/128 CTAs, each
 * with its own TMA -> tcgen05.mma main loop; the row statistics are exchanged through distributed shared memory.
 * sum_out (nullable) receives the pre-norm sum, mean_out / rstd_out (nullable, fp32 [M]) the statistics: exactly
 * what icap_add_ln_fwd(write_sum=1) leaves for icap_add_ln_bwd, with the same dropout decisions: the dropout element
 * index of output (row, col) is row*N + col, as in icap_add_ln_fwd.
 * W, bias, gamma, beta are model parameters: the kernel requests its first W stages before its grid dependency has
 * resolved, so the pre-wait rule of ICAP_EPI_B_STATIC applies to them.
 * Returns -2 (nothing launched) for other shapes / unaligned rows: call icap_gemm + icap_add_ln_fwd instead.
 * Replaces joint_linear / position_wise_2 -> Dropout -> LayerNorm(out + residual) [-> *= non_pad_mask],
 * modules.py:86-90,117-120,154-155,203-204. */
int icap_gemm_ln(int64_t M, int64_t N, int64_t K, const void* A, int64_t lda, const void* W, int64_t ldw,
                 const float* bias, const void* res, int64_t ldr, const float* gamma, const float* beta,
                 const float* rowscale, void* y, int64_t ldy, void* sum_out, int64_t lds, float* mean_out,
                 float* rstd_out, float eps, float p_drop, uint64_t seed, const int* seed_dev, void* stream);
/* Fused log-softmax + NLL per row; with write_grad=1 the logits are overwritten IN PLACE by
 * (softmax - onehot) * inv_count[0] (zero rows for ignored targets).  row_loss: fp32 [M].
 * Replaces CrossEntropyLoss(ignore_index=pad_idx, 'mean'), model.py:76,93-96.  Rows of stride ldl >= V; M, V < 2^31. */
int icap_xent(int dtype, int64_t M, int64_t V, void* logits, int64_t ldl, const int* targets, int ignore_index,
              const float* inv_count, float* row_loss, int write_grad, void* stream);
/* out2[0] = mean loss (focal=1: (1-exp(-ce))^2 * ce, loss.py:20-28); out2[1] = d loss / d ce. */
int icap_xent_finalize(int64_t M, const float* row_loss, const float* inv_count, int focal, float* out2, void* stream);

/* out[row*out_stride] = argmax_j logits[row][j] (lowest index on ties); gap = top1 - top2 (nullable).
 * Replaces argmax(Softmax(classifer(.))), model.py:125-128.  Rows of stride ldl >= V; M, V < 2^31. */
int icap_argmax(int dtype, int64_t M, int64_t V, const void* logits, int64_t ldl, int* out, int64_t out_stride,
                float* gap, void* stream);
/* Sampled decoding step for M rows (row r = image * n + sample; tokens / logp rows of stride Tmax / ldp):
 *   finished row: t >= 1 and tokens[r, t] is end_idx or pad_idx  ->  tokens[r, t+1] = pad_idx, logp[r, t] = 0
 *                 (the mask rule of StructureCriterion, loss.py);
 *   otherwise     tokens[r, t+1] = the smallest j whose running sum of w_j = exp((x_j - max x) / tau), over the row's V
 *                 logits x as stored (bf16 or fp32), in column order, exceeds u * sum_j w_j (none after rounding: the last
 *                 j with w_j > 0), with the uniform
 *                   u = ((rand32(seed_fold(seed + seed_dev[0] * golden), r * Tmax + t) >> 8) + 0.5) * 2^-24
 *                 (icap_common.cuh; seed_dev nullable = 0);
 *                 logp[r, t] = log_softmax(x)[token] at tau = 1 (fp32): the model's log-probability of the token.
 * inv_temperature = 1 / tau must be finite and > 0.  The kernel reads nothing before its grid dependency has resolved.
 * Same seed, seed_dev[0] and logits -> bitwise-identical tokens and logp. */
int icap_sample_tokens(int dtype, int64_t M, int64_t V, const void* logits, int64_t ldl, float inv_temperature,
                       uint64_t seed, const int* seed_dev, int64_t t, int64_t Tmax, int* tokens, float* logp, int64_t ldp,
                       int end_idx, int pad_idx, void* stream);
/* Beam step for B images: candidates (beam r, token j) score softmax(logits[b*kin+r])[j] + prev[b,r]
 * (log_domain=1: log-softmax, the PolicyNetwork variant); writes the kout best in DESCENDING order:
 * score, parent = r, token = j; gap[b] = score_k - score_{k+1} (nullable).
 * stats (nullable): the ICAP_EPI_ROWSTATS buffer of the classifier GEMM that produced `logits` (row stride stats_ld
 * floats): replaces the kernel's own statistics pass over the logits.
 * Replaces Softmax + cat + topk + // and % of model.py:160-166,181-198 (model_RL.py:157,182). */
int icap_beam_select(int dtype, int64_t B, int64_t kin, int64_t V, const void* logits, int64_t ldl,
                     const float* prev_score, int64_t kout, float* out_score, int* out_parent, int* out_token,
                     float* gap, int log_domain, const float* stats, int64_t stats_ld, void* stream);
/* Beam step of a search that stops at <END> (not in the reference, which extends every beam to max_length and scores it
 * by summed probabilities, model.py:160-198).  Arguments as icap_beam_select, plus the hypotheses' token rows
 * tokens[b*kin + r, 0..Tmax) (positions 0..t filled), the step t and the <END> / <NULL> ids:
 *   - hypothesis r is FINISHED if t >= 1 and tokens[b*kin + r, t] is end_idx or pad_idx (the rule of icap_sample_tokens);
 *   - an unfinished r offers every token j with score prev[b,r] + log_softmax(x_r)[j], x_r its logits as stored (bf16
 *     or fp32): the arithmetic, in the same order, of icap_beam_select with log_domain = 1;
 *   - a finished r offers exactly one candidate: token pad_idx with score prev[b,r], unchanged;
 *   - the kout best candidates survive, written in descending order; ties go to the lower r*V + j; gap[b] = score_k -
 *     score_{k+1} (+inf when there are only k candidates).
 * A finished row reads no logits (no statistics either, with `stats`).  log_domain must be 1; 0 <= pad_idx < V;
 * 0 <= t < Tmax - 1; at t = 0 kin*V > kout, at t >= 1 kin >= kout (every row offers at least one candidate). */
int icap_beam_select_eos(int dtype, int64_t B, int64_t kin, int64_t V, const void* logits, int64_t ldl,
                         const float* prev_score, int64_t kout, float* out_score, int* out_parent, int* out_token,
                         float* gap, int log_domain, const float* stats, int64_t stats_ld, const int* tokens, int64_t Tmax,
                         int64_t t, int end_idx, int pad_idx, void* stream);
/* Final order of an <END>-aware beam search over k hypotheses per image (tokens rows b*k + s of Tmax ids, position 0 =
 * <START>; score [B, k] accumulated log-probabilities), one warp per image:
 *   len_s  = generated tokens up to and including the first end_idx; the tokens before a first pad_idx; Tmax - 1 if
 *            neither occurs;
 *   norm_s = score_s / ((5 + len_s) / 6)^alpha   (fp32; alpha finite and >= 0; alpha = 0 orders by log-probability);
 *   the n best by norm (ties: lower s) in descending order: out_ids [B, n, Tmax] (the token rows), out_score [B, n]
 *   (score_s, not normalised), out_len [B, n].  1 <= n <= k <= 8. */
int icap_beam_finalize(int64_t B, int64_t k, int64_t Tmax, const int* tokens, const float* score, int end_idx, int pad_idx,
                       float alpha, int64_t n, int* out_ids, float* out_score, int* out_len, void* stream);
/* PolicyNetwork.sample (model_RL.py:93-97) on fp32 logits [M, V]: logp = log_softmax(x) per row, idx[row] (int64,
 * nullable) = arg-max (lowest index on ties, as torch.argmax on the CPU).  icap_log_softmax_bwd is its backward:
 * dx = dlogp - exp(logp) * rowsum(dlogp)  (the self-critical loss gathers log-probabilities, loss.py:90-103,145-158). */
int icap_log_softmax_argmax(int64_t M, int64_t V, const float* x, int64_t ldx, float* logp, int64_t ldo, long long* idx,
                            void* stream);
int icap_log_softmax_bwd(int64_t M, int64_t V, const float* logp, int64_t ldp, const float* dlogp, int64_t ldd, float* dx,
                         int64_t ldx, void* stream);

/* Start of a KV-cached decode step in one launch: (parent != NULL) the beam bookkeeping of the previous step exactly as
 * icap_beam_reorder(B = rows / k, k, Tmax, t - 1, ...) does it -- position t receives `token` -- and then, for every row,
 * y = LayerNorm(table[token of position t] + pos_row) * gamma + beta and rowscale = (token != pad_idx): the decoder
 * input of position t (word embedding folded with word_embedding_linear, positional row, decoder.norm; model.py:432-436)
 * with the arithmetic of icap_embed_fwd + icap_add_ln_fwd.  parent == NULL: tokens are read from tok_in[row, t].
 * table / pos_row / y: act_dtype rows of width d (multiple of 8, <= 1024). */
int icap_decode_embed_ln(int act_dtype, int64_t rows, int64_t d, int64_t k, int64_t Tmax, int64_t t, const int* parent,
                         const int* token, const int* tok_in, int* tok_out, const int* slot_in, int* slot_out,
                         const void* table, const void* pos_row, const float* gamma, const float* beta, void* y,
                         float* rowscale, int pad_idx, float eps, void* stream);
/* Reorder token buffer (and KV-cache slot table) by parent and append the new token: model.py:194-198. */
int icap_beam_reorder(int64_t B, int64_t k, int64_t Tmax, int64_t t, const int* parent, const int* token,
                      const int* tok_in, int* tok_out, const int* slot_in, int* slot_out, void* stream);

/* KV-cached single-position attention for decoding (M = B*k rows, one query each).
 *   self-attention (tokens != NULL): keys/values of positions 0..Lk-1 live in the cache at physical row
 *                    slot[row*slot_ld+j] (own row when slot == NULL); position j is masked iff
 *                    tokens[row*tok_ld+j] == pad_idx  (model.py:421-430).
 *   cross-attention (tokens == NULL): keys are the Lk regions of image row / rows_per_image, masked by kvalid;
 *                    kc / vc / kvalid are produced once per decode: the kernel may fetch them before its grid
 *                    dependency has resolved, so the pre-wait rule of ICAP_EPI_B_STATIC applies to them.
 *   cache rows: k at kc + (slot*Tmax_or_Lk + j)*ldk + h*dk. */
int icap_mha_decode(int dtype, int64_t rows, int64_t H, int64_t Lk, int64_t dk, int64_t dv, const void* q, int64_t ldq,
                    const void* kc, int64_t ldk, const void* vc, int64_t ldv, int64_t kv_rows_per_seq, void* o,
                    int64_t ldo, const int* slot, int64_t slot_ld, const int* tokens, int64_t tok_ld, int pad_idx,
                    const uint8_t* kvalid, int64_t rows_per_image, float* attn_mean, void* stream);

/* Self-attention decode step with the KV-cache append fused in: the key / value of position `pos` (rows of k_new /
 * v_new, leading dimension ld_new) are written to the row's own cache line (kc/vc + (row*kv_rows_per_seq + pos)*ld)
 * and attended together with the cached positions 0..pos-1 (slot table / pad-token mask as in icap_mha_decode).
 * rows_per_image (>= 1, beam width): consecutive rows that belong to one image -- a scheduling hint only (their cache
 * lines overlap through the slot table, so they are processed by one thread block).  tokens, slot and the cache are
 * in ordinary stream order: before its grid dependency has resolved the kernel only prefetches the cached positions into
 * L2 from a provisional lookup of tokens / slot, and it reads both tables again after the wait.
 * Replaces the per-step prefix recomputation of model.py:114-122,169-180 (decoder self-attention, modules.py:190-194). */
int icap_mha_decode_self(int dtype, int64_t rows, int64_t H, int64_t pos, int64_t dk, int64_t dv, const void* q,
                         int64_t ldq, const void* k_new, const void* v_new, int64_t ld_new, void* kc, int64_t ldk, void* vc,
                         int64_t ldv, int64_t kv_rows_per_seq, void* o, int64_t ldo, const int* slot, int64_t slot_ld,
                         const int* tokens, int64_t tok_ld, int pad_idx, int64_t rows_per_image, void* stream);

/* dst[r][c] (+)= convert(src[r][c]) : operand packing / dtype casts / gradient unpacking.
 * accumulate: 0 = store, 1 = dst += src, 2 = atomic dst += src (fp32 dst; concurrent accumulation from several streams). */
int icap_copy2d(const void* src, int src_dtype, int64_t src_ld, void* dst, int dst_dtype, int64_t dst_ld, int64_t rows,
                int64_t cols, int accumulate, void* stream);
/* dst[r,:] = (base ? base[r,:] : 0) + src[(r / div) * mul + off, :]  -- row broadcast: the "whole image" token
 * repeated per region (split_image_objects, model.py:262-271) and `decode_output + encode_output[:, 0]`
 * (move_first_image_feature, model.py:452-453).  icap_rows_segsum_add is its adjoint:
 * dst[s * mul + off, :] += sum_{t < seg_len} src[s * seg_len + t, :]. */
int icap_rows_gather_add(int dtype, const void* src, int64_t src_ld, const void* base, int64_t base_ld, void* dst,
                         int64_t dst_ld, int64_t rows, int64_t cols, int64_t div, int64_t mul, int64_t off,
                         void* stream);
int icap_rows_segsum_add(int dtype, const void* src, int64_t src_ld, void* dst, int64_t dst_ld, int64_t nseg,
                         int64_t seg_len, int64_t cols, int64_t mul, int64_t off, void* stream);
/* kvalid[row] = rowscale[row] = any(pos[row,:] != 0) : get_attention_key_pad_mask / get_non_pad_mask,
 * model.py:202-209,354-358. */
int icap_region_valid(const float* pos, int64_t M, int64_t Dp, uint8_t* kvalid, float* rowscale, void* stream);
/* Device-resident region cache -> one batch (SURVEY.md 8f #2).  The reference gathers
 * `features[image_idx]` / `positions[image_idx]` on the HOST for every caption (core/dataset.py:12-18, five captions
 * per image) and ships [B, R, 2048] fp32 over PCIe every step.  Here the packed encoder input rows
 * [features | positions | 0-pad] (width Kc, the A operand of the embedding GEMM, in the compute dtype) and the
 * per-region validity byte live in HBM for the whole data set; a step sends only `idx` (B image numbers).
 * xcat[(b, r), :] = cache[(idx[b], r), :]; kvalid / rowscale as icap_region_valid.  *err (nullable) is set to 1 when
 * an index is outside [0, n_images) (that row then reads image 0). */
int icap_gather_regions(int dtype, const void* cache, const uint8_t* valid_cache, int64_t n_images, const void* idx,
                        int idx_is_int64, int64_t B, int64_t R, int64_t Kc, void* xcat, uint8_t* kvalid,
                        float* rowscale, int* err, void* stream);
/* inp = cap[:, :-1], tgt = cap[:, 1:], tok_valid/rowscale = inp != pad, count_f2 = {n, 1/n} with n the
 * number of non-pad targets (model.py:88-89,421-430; the 'mean' denominator of model.py:76). */
int icap_caption_prep(const void* captions, int cap_is_int64, int64_t B, int64_t L, int pad_idx, int* inp, int* tgt,
                      uint8_t* tok_valid, float* rowscale, int* count_i, float* count_f2, void* stream);
/* out[r,:] = table[tokens[r*tok_stride],:]  (nn.Embedding, model.py:432); rowscale[r] = token != pad (nullable);
 * and the scatter-add backward (row pad_idx untouched). */
int icap_embed_fwd(int table_dtype, int out_dtype, const int* tokens, int64_t tok_stride, int64_t M, int64_t E,
                   const void* table, void* out, float* rowscale, int pad_idx, void* stream);
int icap_embed_bwd(int dtype, const int* tokens, int64_t M, int64_t E, int pad_idx, const void* dout, float* dtable,
                   void* stream);
/* out[c] += sum_r x[r][c]  (bias gradients). */
int icap_colsum(int dtype, int64_t M, int64_t N, const void* x, int64_t ld, float* out, void* stream);
/* torch.optim.Adam step over flat fp32 buffers (+ bf16 shadow refresh); step counter on the device: tick=1
 * increments it first, tick=0 uses it as is, tick=2 uses step+1 WITHOUT incrementing (slices of the parameter
 * buffer updated during the backward, while the dropout seeds of the step still read the old counter; finish with
 * icap_step_tick); gradients are pre-multiplied by gscale * gscale_dev[0].
 * Replaces optimizer.step(), core/models.py:111-113,126. */
int icap_adam_step(int64_t n, float* p, const float* g, float* m, float* v, void* shadow_bf16, float lr, float beta1,
                   float beta2, float eps, int* step_dev, int tick, const float* gscale_dev, float gscale,
                   void* stream);
int icap_step_tick(int* step_dev, void* stream);
int icap_scale(float* x, int64_t n, const float* s_dev, float s, void* stream);
/* out[0] = numerator / x[0]  (data parallel: 1 / all-reduced token count, consumed by icap_adam_step as gscale_dev). */
int icap_reciprocal(const float* x, float* out, float numerator, void* stream);

/* ---- gradient all-reduce over NVLink peer memory (data parallel, SURVEY.md 8e): load/store kernels without shared
 * memory, co-resident with the backward's GEMM CTAs.  `flag_ptrs` / `buf_ptrs`: host arrays of nranks device pointers,
 * entry q = rank q's flag words (>= nranks uint32, zero-initialised once) / fp32 buffer as mapped into THIS process (CUDA
 * IPC for q != rank).  One bucket [lo, hi) (element offsets, multiples of 4) is reduced by
 *   icap_p2p_barrier; icap_p2p_reduce_scatter; icap_p2p_barrier; icap_p2p_all_gather
 * on one stream, with one more icap_p2p_barrier after the last bucket of a step.  The barrier (a one-warp kernel) bumps
 * the device-side `epoch`, publishes it into every rank's flag words and waits for all peers; after ~2 s without a peer it
 * stores 1 + the missing rank into `err` and returns instead of hanging.  Every rank must issue the same call sequence. */
int icap_p2p_barrier(void* const* flag_ptrs, int rank, int nranks, unsigned int* epoch, int* err, void* stream);
int icap_p2p_reduce_scatter(void* const* buf_ptrs, int rank, int nranks, int64_t lo, int64_t hi, int ctas, void* stream);
int icap_p2p_all_gather(void* const* buf_ptrs, int rank, int nranks, int64_t lo, int64_t hi, int ctas, void* stream);
/* NVSwitch in-switch reduction: `mc_base` is the multicast mapping of the same symmetric buffer (all ranks' copies behind
 * one address range).  Rank r runs multimem.ld_reduce (sum over the ranks, computed in the switch) + multimem.st
 * (broadcast) over chunk r of [lo, hi): a one-pass all-reduce.  Sequence per bucket: icap_p2p_barrier;
 * icap_p2p_allreduce_nvls; one more icap_p2p_barrier before anybody reads the result. */
int icap_p2p_allreduce_nvls(void* mc_base, int rank, int nranks, int64_t lo, int64_t hi, int ctas, void* stream);

/* ---- region feature extractor (SURVEY.md 8f #4: ResNet-101 trunk over the region crops, core/preprocess.py:26-62).
 * Activations are NHWC matrices [N*H*W, C]; every convolution is icap_gemm over the activation matrix itself (1x1) or
 * over the patch matrix gathered by icap_im2col_nhwc (3x3, 7x7, strided 1x1):
 *   out[(n, ho, wo), (ky, kx, c)] = x[n, ho*stride - pad + ky, wo*stride - pad + kx, c], zero outside the image and in
 *   the columns kh*kw*C .. ldo-1 (ldo = kh*kw*C rounded up to 8 so that TMA can read the rows).
 * icap_bn_scale_shift: per-channel scale = gamma / sqrt(var + eps), shift = beta - mean * scale.  train != 0: mean / var
 *   are the statistics of the M rows of x (what the reference's extractor uses: it never calls .eval(),
 *   preprocess.py:35-40), accumulated in the zero-initialised fp64 scratch sums[2*C] (left zeroed again), running
 *   statistics updated with `momentum` like nn.BatchNorm2d; train == 0: running statistics.
 * icap_bn_act: y = act(x * scale[c] + shift[c] + residual) (residual nullable, act = ReLU when relu != 0).
 * icap_maxpool_nhwc / icap_avgpool_nhwc: the 3x3/2 max pool after the stem and the global average pool (fp32 out). */
int icap_im2col_nhwc(int dtype, const void* x, int64_t N, int64_t H, int64_t W, int64_t C, int kh, int kw, int stride,
                     int pad, void* out, int64_t ldo, void* stream);
int icap_bn_scale_shift(int dtype, const void* x, int64_t M, int64_t C, double* sums, const float* gamma, const float* beta,
                        float* running_mean, float* running_var, float momentum, float eps, int train, float* scale,
                        float* shift, void* stream);
int icap_bn_act(int dtype, const void* x, int64_t M, int64_t C, const float* scale, const float* shift, const void* residual,
                int relu, void* y, void* stream);
int icap_maxpool_nhwc(int dtype, const void* x, int64_t N, int64_t H, int64_t W, int64_t C, int k, int stride, int pad,
                      void* y, void* stream);
int icap_avgpool_nhwc(int dtype, const void* x, int64_t N, int64_t HW, int64_t C, float* y, void* stream);

/* ---- caption metrics on token ids: BLEU-1..4, ROUGE-L, CIDEr, CIDEr-D, the scores of core/evaluations.py:12-34 (coco-
 * caption / pyciderevalcap arithmetic, METEOR and SPICE excluded) and the self-critical reward of loss.py:160-186.
 * A row of W <= 128 ids (int32 or int64, leading dimension ld) is read like core/utils.py::decode_captions: a <START> (1)
 * at position 0 is skipped, <NULL> (0) dropped, the row ends at the first <END> (2), which counts as a token.  Ids must
 * be < 32768: an n-gram (n = 1..4) is the key n << 60 | t0 << 45 | t1 << 30 | t2 << 15 | t3.
 * icap_caption_cook: per row the distinct keys ascending (keys / counts [N, 4W], zero-filled), their number nkeys[N],
 *   the token count lens[N] and the tokens after the cut toks [N, W].
 * icap_caption_df: document frequencies over a cooked reference set grouped by image (rows img_off[i] .. img_off[i+1]-1
 *   belong to image i): a key counts once per image.  table_keys / table_df (cap slots, power of two, zeroed by the
 *   caller; 0 = empty) receive the counts by linear probing; n_unique (nullable, int64) += the number of counted
 *   (image, key) pairs -- size the table from it (cap >= 1.5 x n_unique leaves no overflow path).  table_keys = NULL:
 *   count only.
 * icap_caption_ref_prep: norms [N, 4] fp64 = per-order L2 norms of count * (log(n_img) - log(max(1, df))).
 * icap_caption_score: one candidate row per image cand_img[m] (int64; outside [0, n_img) or without refs: 0).
 *   scores [M, 7] fp32 (nullable) = CIDEr-D, CIDEr, ROUGE-L, sentence BLEU-1..4; reward [M] (nullable) =
 *   cider_weight * CIDEr-D + bleu_weight * BLEU-4; corpus (nullable, int64 [10]) += BLEU's correct[1..4], guess[1..4],
 *   candidate length, closest reference length, so corpus BLEU is exact. */
int icap_caption_cook(const void* tokens, int tok_is_int64, int64_t N, int64_t W, int64_t ld, uint64_t* keys, int* counts,
                      int* nkeys, int* lens, int* toks, void* stream);
int icap_caption_df(int64_t n_img, const int64_t* img_off, int64_t W, const uint64_t* keys, const int* nkeys,
                    uint64_t* table_keys, int* table_df, int64_t cap, long long* n_unique, void* stream);
int icap_caption_ref_prep(int64_t N, int64_t W, const uint64_t* keys, const int* counts, const int* nkeys, int64_t n_img,
                          const uint64_t* table_keys, const int* table_df, int64_t cap, double* norms, void* stream);
int icap_caption_score(const void* cand, int cand_is_int64, int64_t M, int64_t Wc, int64_t ldc, const int64_t* cand_img,
                       int64_t n_img, const int64_t* img_off, int64_t W, const uint64_t* keys, const int* counts,
                       const int* nkeys, const int* lens, const int* toks, const double* norms, const uint64_t* table_keys,
                       const int* table_df, int64_t cap, float* scores, float* reward, float cider_weight,
                       float bleu_weight, long long* corpus, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ICAP_H_ */
