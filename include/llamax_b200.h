/*
 * llamax_b200 — C ABI of the B200-native (sm_100a) fine-tuning hot path of gau-nernst/llama-x.
 *
 * Every entry point replaces one Python/PyTorch seam of the reference (cited per function as file:line,
 * relative to the reference repo).  Conventions:
 *   - plain pointers + sizes, no torch types; all pointers are DEVICE pointers owned by the caller
 *   - `stream` is a cudaStream_t passed as void*; all work is asynchronous on it
 *   - return 0 on success, a negative LLAMAX_ERR_* code otherwise; llamax_last_error() gives the text
 *     (thread-local), so the Python seam can raise
 *   - no allocation inside; scratch / workspace buffers are passed in by the caller
 *   - bf16 tensors are row-major with an explicit leading dimension (elements) where noted
 *   - thread-safe: forward (caller thread) and backward (autograd engine thread) may call concurrently
 */
#ifndef LLAMAX_B200_H_
#define LLAMAX_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LLAMAX_B200_VERSION 102

#define LLAMAX_OK 0
#define LLAMAX_ERR_ARG (-1)  /* bad argument (shape / alignment / null) */
#define LLAMAX_ERR_CUDA (-2) /* CUDA runtime or driver error */

const char* llamax_last_error(void);
int llamax_version(void);
/* Select the device for subsequent calls of this thread (the library carries its own CUDA runtime). */
int llamax_set_device(int device);
/* 1 = single-CTA UMMA 128x256 tiles, 2 (default) = CTA pairs, UMMA 256x256 (tcgen05 cta_group::2). */
int llamax_set_gemm_cta_group(int cg);

/* Optional fused GEMM epilogue terms:  C = dequant(acc) + lora_scale * lora_h @ lora_b^T + resid
 *   LoRA up-projection  : modelling/lora.py:43   (lora_h = x @ lora_a^T computed by the caller)
 *   residual connection : modelling/llama.py:172-173 */
typedef struct {
  const void* lora_h; /* bf16 [M, lora_rank], row pitch ldh; NULL = no LoRA term */
  int64_t ldh;
  const void* lora_b; /* bf16 [N, lora_rank] contiguous */
  int32_t lora_rank;  /* multiple of 4, <= 16 */
  float lora_scale;   /* alpha / rank */
  const void* resid;  /* bf16 [M, N], row pitch ldr; NULL = none */
  int64_t ldr;
  /* Column segments for row-concatenated weights that share an input (q | k | v in one launch): output columns
   * [0, seg_n0) take LoRA-h columns [0, rank), [seg_n0, seg_n1) take [rank, 2 rank), [seg_n1, N) take [2 rank, 3 rank)
   * of lora_h (whose rows then hold 3 * rank values); lora_b is the row-concatenation [N, rank] of the three B matrices.
   * seg_n0 = 0: one segment. seg_n0, seg_n1 must be multiples of 256 (the tile width). */
  int32_t seg_n0, seg_n1;
  /* RoPE in the epilogue (llamax_int8_gemm_dequant only; modelling/llama.py:63-73 applied to the projection's bf16 output,
   * bit-identical to llamax_rope_inplace on the stored result): rope fp32 [rope_S, 64, 2] (cos, sin), 32-byte aligned,
   * head_dim 128; output columns [0, rope_cols) are rotated (rope_cols a multiple of 256: the q | k block of a q | k | v
   * launch), position = row % rope_S. NULL = none. Not combinable with resid; LoRA rank 0 or 8. */
  const void* rope;
  int32_t rope_S, rope_cols;
} llamax_epilogue_t;

/* ---- K3: int8 x int8 -> int32 GEMM with row/column-scale dequant --------------------------------
 * Replaces torch.ops.torchao.int8_mm_dequant (subclasses/int8_mm.py:121-149, Triton kernel :50-118).
 *   C[m,n] = bf16( (f32(sum_k A[m,k]*B[n,k]) * f32(a_scale[m])) * f32(b_scale[n]) )  [+ epilogue terms]
 * A int8 [M,K] pitch lda; B int8 [N,K] pitch ldb (the reference passes weight.int_data.T, i.e. this
 * matrix viewed as [K,N] with strides (1,K)); scales bf16 [M] / [N]; C bf16 [M,N] pitch ldc.
 * The int32 accumulators are exact (|acc| <= K*127^2 < 2^31 for K <= 133143). */
int llamax_int8_gemm_dequant(const void* A, int64_t lda, const void* B, int64_t ldb, const void* a_scale,
                             const void* b_scale, void* C, int64_t ldc, int64_t M, int64_t N, int64_t K,
                             const llamax_epilogue_t* epi, void* stream);
/* Same GEMM, raw int32 accumulators written to C (int32 [M,N]); parity/debug entry. */
int llamax_int8_gemm_s32(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t M,
                         int64_t N, int64_t K, void* stream);

/* ---- K4/K5/K6: bf16 x bf16 -> fp32 GEMM -----------------------------------------------------------
 *   C[m,n] = bf16( acc[m,n] (* col_scale[n]) ) [+ epilogue terms],  acc = sum_k A[m,k]*B[n,k]
 * weight-only forward   (subclasses/int8.py:118): B = bf16(int_data), col_scale = weight scale,
 *                        round_before_scale = 1 reproduces the reference's two roundings
 * grad_input            (subclasses/int8.py:127): B = (scale * int_data)^T from llamax_dequant_weight
 * LoRA down / dh        (modelling/lora.py:43)  : N = rank (any multiple of 8) */
int llamax_bf16_gemm(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t M,
                     int64_t N, int64_t K, const void* col_scale, int round_before_scale,
                     const llamax_epilogue_t* epi, void* stream);
/* grad_input GEMM of w2 with the SwiGLU backward as its epilogue (modelling/llama.py:152 differentiated):
 *   dg[m,n] = bf16( sum_k A[m,k]*B[n,k] + lora term )            (never written)
 *   da | db = swiglu_bwd(dg, a, b)   with a = ab[:, 0:N], b = ab[:, N:2N]  -> dab[:, 0:N] | dab[:, N:2N]
 *   g       = bf16(silu(a)) * b      -> g [M,N] contiguous, optional (NULL = not needed)
 * Same arithmetic as llamax_bf16_gemm followed by llamax_swiglu_bwd (identical results); N % 16 == 0,
 * ld_ab / ld_dab multiples of 8 and >= 2N, pointers 16-byte aligned. epi: LoRA term only (no residual). */
int llamax_bf16_gemm_swiglu_bwd(const void* A, int64_t lda, const void* B, int64_t ldb, int64_t M, int64_t N, int64_t K,
                                const llamax_epilogue_t* epi, const void* ab, int64_t ld_ab, void* dab, int64_t ld_dab,
                                void* g, void* stream);
/* llamax_bf16_gemm that also returns, per row and group of 128 output columns, the dot product of the bf16-ROUNDED
 * outputs with a second matrix:  dot_out[(m / S) * (N / 128) + g][m % S] = sum_{c in group g} C[m,c] * other[m,c]
 * (fp32, layout [M / S, N / 128, S]). With C = dO = grad_input of wo (int8.py:127 + the LoRA term) and other = O this is
 * the attention backward's delta[b, h, s] (head_dim 128) for free in the epilogue that writes dO: pass it to
 * llamax_attn_bwd with o = NULL. N % 256 == 0, M % S == 0, other bf16 [M,N] pitch ld_other (must not alias C); epi:
 * LoRA term only. */
int llamax_bf16_gemm_rowdot(const void* A, int64_t lda, const void* B, int64_t ldb, void* C, int64_t ldc, int64_t M,
                            int64_t N, int64_t K, const llamax_epilogue_t* epi, const void* other, int64_t ld_other,
                            void* dot_out, int64_t S, void* stream);

/* ---- K4/K5 mixed-input: bf16 activations x frozen INT8 weight, converted inside the GEMM ---------------------------
 * The int8 weight is read by TMA as stored and expanded to bf16 in shared memory by converter warps (exact: every int8
 * value is a bf16 value), so neither a de-quantised nor a transposed copy of the weight exists in HBM.
 *   b_layout = 0, weight-only forward (subclasses/int8.py:118): B8 int8 [N,K] pitch ldb8 (the weight as stored),
 *     C[m,n] = bf16( bf16(sum_k A[m,k]*B8[n,k]) * b_scale[n] ) [+ epilogue terms]; tail = NULL, K1 = K.
 *   b_layout = 1, grad_input (subclasses/int8.py:127): B8 int8 [K1,N] pitch ldb8 (the weight as stored: its rows are the
 *     contraction index; row-concatenated weights that share an input form one operand), b_scale bf16 [K1] folded into
 *     the operand as bf16(f32(w) * f32(s)) exactly like llamax_dequant_weight(transpose = 1, apply_scale = 1);
 *     tail: NULL (K1 = K) or bf16 [K-K1, N] pitch ldt (K - K1 <= 64): the LoRA A rows that multiply the dh columns
 *     A[:, K1:K];  C[m,n] = bf16( sum_{k<K1} A[m,k]*bf16(B8[k,n]*s[k]) + sum_{k>=K1} A[m,k]*tail[k-K1,n] ) [+ LoRA term].
 * K1 % 64 == 0. Results are bit-identical to llamax_dequant_weight + llamax_bf16_gemm on the same operands. */
int llamax_bf16_int8_gemm(const void* A, int64_t lda, const void* B8, int64_t ldb8, const void* b_scale, int b_layout,
                          const void* tail, int64_t ldt, void* C, int64_t ldc, int64_t M, int64_t N, int64_t K,
                          int64_t K1, const llamax_epilogue_t* epi, void* stream);
/* llamax_bf16_gemm_swiglu_bwd with the b_layout = 1 operand above (B8 = w2 as stored, [K, N] int8; k_scale bf16 [K]). */
int llamax_bf16_int8_gemm_swiglu_bwd(const void* A, int64_t lda, const void* B8, int64_t ldb8, const void* k_scale,
                                     int64_t M, int64_t N, int64_t K, const llamax_epilogue_t* epi, const void* ab,
                                     int64_t ld_ab, void* dab, int64_t ld_dab, void* g, void* stream);
/* Weight-gradient form: C[m,n] = bf16( sum_k At[k,m] * Bt[k,n] ), At bf16 [K,M] pitch ldat, Bt bf16 [K,N] pitch ldbt
 * (M, N indices contiguous; M % 8 == 0, N % 8 == 0). Both tensors are consumed as stored (MN-major UMMA operands):
 * dW[out,in] = dY[tokens,out]^T X[tokens,in] needs no transposed copies. Rows of Bt may overlap (pitch < N), which is
 * how the audio stem's im2col view is read. Used for the conv-stem weight gradients and a trainable LM head. */
int llamax_bf16_gemm_tn(const void* At, int64_t ldat, const void* Bt, int64_t ldbt, void* C, int64_t ldc, int64_t M,
                        int64_t N, int64_t K, void* stream);

/* De-quantise a frozen weight into a bf16 GEMM operand (scratch owned by the caller).
 *   transpose = 0: out[n,k] = bf16(w8[n,k]) (* scale[n] if apply_scale)          out [N,K], row pitch ldo
 *   transpose = 1: out[k,n] = bf16(f32(w8[n,k]) * f32(scale[n])) (or unscaled)    out [K,N], row pitch ldo
 * Reference: weight.int_data.T.to(dtype) (int8.py:118), weight_i8.to(dtype) and grad*scale (int8.py:127). */
int llamax_dequant_weight(const void* w8, const void* scale, void* out, int64_t ldo, int64_t N, int64_t K,
                          int transpose, int apply_scale, void* stream);

/* ---- K2: row-wise int8 quantisation (subclasses/int8.py:10-16) ------------------------------------
 *   s = amax(|x_f32|) / 127;  q = rint(x_f32 / max(s, 1e-12));  scale_out = bf16(s)        bit-exact */
int llamax_rowquant_int8(const void* x, int64_t ldx, void* q8, void* scale_out, int64_t M, int64_t K,
                         void* stream);
/* Same quantiser applied to x[m,c] * col_scale[c] (fp32 product; col_scale bf16 [K]). Used only by the OPT-IN,
 * non-parity INT8 grad_input mode (the reference author's TODO at subclasses/int8.py:105): grad_output * weight_scale
 * is quantised row-wise so that grad_input = q(dY * s) @ W_int8 runs on the int8 tensor path. */
int llamax_rowquant_int8_colscale(const void* x, int64_t ldx, const void* col_scale, void* q8, void* scale_out,
                                  int64_t M, int64_t K, void* stream);

/* ---- K1: RMSNorm (nn.RMSNorm(eps) at modelling/llama.py:158,160,182) ------------------------------
 *   y = bf16( (x_f32 * rsqrt(mean(x_f32^2) + eps)) * w_f32 )
 * optional outputs: rstd fp32 [M]; q8/qscale = rowquant_int8(y) fused (feeds the int8 GEMM). */
int llamax_rmsnorm_fwd(const void* x, const void* w, void* y, void* rstd, void* q8, void* qscale, int64_t M,
                       int64_t D, float eps, void* stream);
/* dx = [dres +] rmsnorm_backward(dy; x, w, rstd);  dw_partial fp32 [nparts, D] (summed by the caller or
 * by llamax_reduce_partials).  nparts is chosen by the caller (<= 1024). */
int llamax_rmsnorm_bwd(const void* dy, const void* x, const void* w, const void* rstd, const void* dres, void* dx,
                       void* dw_partial, int32_t nparts, int64_t M, int64_t D, void* stream);
/* out[d] (bf16) = sum_p partial[p, d] */
int llamax_reduce_partials(const void* partial, void* out, int32_t nparts, int64_t D, void* stream);

/* ---- K10: SwiGLU (modelling/llama.py:152) ---------------------------------------------------------
 *   g = bf16( bf16(silu_f32(a)) * b );  optional g (bf16), q8/qscale = rowquant_int8(g) */
int llamax_swiglu_fwd(const void* a, const void* b, int64_t ld, void* g, void* q8, void* qscale, int64_t M,
                      int64_t F, void* stream);
/* da, db (row pitch ldd) from dg; optionally re-materialises g (needed for the LoRA-A gradient of w2). */
int llamax_swiglu_bwd(const void* dg, const void* a, const void* b, int64_t ld, void* da, void* db, int64_t ldd,
                      void* g, int64_t M, int64_t F, void* stream);

/* ---- K7: RoPE (modelling/llama.py:63-73), interleaved pairs, fp32 math, in place ------------------
 * x bf16 [B*S, ...] row pitch ld; rotates `nheads` heads of width D starting at column 0.
 * rope fp32 [S, D/2, 2] (cos, sin) (build_rope, llama.py:54-60).  inverse = 1 applies the transpose
 * (the backward of apply_rope).  x 16-byte aligned, ld and D multiples of 8, fewer than 2^31 rows; anything else
 * returns LLAMAX_ERR_ARG. */
int llamax_rope_inplace(void* x, int64_t ld, const void* rope, int64_t B, int64_t S, int32_t nheads, int32_t D,
                        int inverse, void* stream);

/* ---- K8/K9: prefix-LM attention (modelling/llama.py:129-137) --------------------------------------
 * mask(q, kv) = (kv < prefix_len) | (q >= kv);  prefix_len = 0 is plain causal.
 * prefix_len_b: NULL, or int32 [B] with one prefix length per sequence of the batch (then prefix_len is ignored): the
 * LibriSpeech-shaped batches of train_librispeech.py:36-124 pack utterances of different durations.
 * Optional packed-sequence document-causal mask (train_metamathqa.py:67-70): doc_start / doc_end int32 [B, S] hold the
 * first / last position of the document containing each position (documents are contiguous); visible pairs are
 * additionally restricted to kv >= doc_start[q].  NULL = no document structure.
 * q bf16 [B,S,Hq,D] with row pitch ldq (elements between consecutive positions), k/v [B,S,Hkv,D] pitch
 * ldk/ldv, o [B,S,Hq,D] pitch ldo, lse fp32 [B,Hq,S] (natural-log-sum-exp of scaled scores).
 * GQA native: Hq % Hkv == 0, no K/V expansion.  D = 128, or 64 (run as zero-padded 128-wide tiles: the TMA
 * descriptor zero-fills the missing half, at half the tensor-core efficiency).  scale = 1/sqrt(D). */
int llamax_attn_fwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv, void* o,
                    int64_t ldo, void* lse, int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D,
                    int64_t prefix_len, const void* prefix_len_b, const void* doc_start, float scale, void* stream);
/* dq/dk/dv bf16 with pitches lddq/lddk/lddv; dq_accum fp32 workspace [B,S,Hq,D] (zeroed by the call);
 * delta fp32 workspace [B,Hq,S]; o = NULL: delta already holds sum_d dO * O (e.g. from llamax_bf16_gemm_rowdot) and
 * the pass over o / dout that computes it is skipped. rope_inverse: null, or the fp32 [>= S, D/2, 2] (cos, sin) table of K7: dq and dk then
 * leave the call already rotated back through RoPE (the autograd of apply_rope, llama.py:63-73), which saves the
 * separate in-place pass over the q|k gradient columns. */
int llamax_attn_bwd(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                    const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                    int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* dq_accum, void* delta,
                    int64_t B, int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                    const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                    const void* rope_inverse, void* stream);
/* Deterministic form (torch.use_deterministic_algorithms): same arguments without dq_accum, bitwise identical results
 * from run to run. dq comes from a kernel that owns 128 query rows of one head and sums over the kv tiles in ascending
 * order in tensor memory (no fp32 atomics, no workspace); dk / dv are bitwise those of llamax_attn_bwd. */
int llamax_attn_bwd_deterministic(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                                  const void* o, int64_t ldo, const void* lse, const void* dout, int64_t lddo, void* dq,
                                  int64_t lddq, void* dk, int64_t lddk, void* dv, int64_t lddv, void* delta, int64_t B,
                                  int64_t S, int32_t Hq, int32_t Hkv, int32_t D, int64_t prefix_len,
                                  const void* prefix_len_b, const void* doc_start, const void* doc_end, float scale,
                                  const void* rope_inverse, void* stream);

/* ---- audio stem (modelling/audio.py:26-31,51-60): Conv1d(k3,s1)+GELU, Conv1d(k3,s2)+GELU -------------------------
 * The convolutions run on llamax_bf16_gemm: with channels-last activations padded by one zero row on each side of a
 * batch slab, output row t of a k = 3 convolution is the dot product of the weights with 3C CONSECUTIVE elements
 * starting at padded row stride*t, i.e. the im2col matrix is a view with OVERLAPPING rows (lda = stride * C < K = 3C)
 * that TMA walks directly — no im2col copy. These entries are the elementwise ends of that GEMM:
 *   gelu_bias_fwd: z (in place) = bf16(z + bias[col]); y = bf16(gelu_erf(z)); rows with (row % period) outside [lo, hi)
 *                  are padding: z = y = 0.        gelu_bwd: dz = bf16(dy * gelu'(z)), 0 on padding rows.
 *   conv_s2k3_col2im: dxp[b, i, :] = sum_{2t + j = i} dcol[b, t, j, :]  (dcol [B, Tp/2, 3, C], dxp [B, Tp, C]) */
int llamax_gelu_bias_fwd(void* z, const void* bias, void* y, int64_t rows, int64_t C, int32_t period, int32_t lo,
                         int32_t hi, void* stream);
int llamax_gelu_bwd(const void* dy, const void* z, void* dz, int64_t rows, int64_t C, int32_t period, int32_t lo,
                    int32_t hi, void* stream);
int llamax_conv_s2k3_col2im(const void* dcol, void* dxp, int64_t B, int64_t Tp, int64_t C, void* stream);

/* ---- LoRA bookkeeping: many small strided copies in ONE launch -----------------------------------------------
 * The LoRA backward needs a few dozen tiny re-layouts per decoder block (scale * B^T, A^T into the grad_input operand,
 * h^T, fp32 dA^T / dB -> bf16 parameter gradients; modelling/lora.py:43 under autograd). As separate elementwise
 * launches they cost more than their bytes; this entry runs up to LLAMAX_MAX_COPY_JOBS of them in one grid.
 *   dst[c, r] (transpose) or dst[r, c] = bf16( scale * src[r, c] ),   src bf16 or fp32 [rows, cols] with pitch src_ld */
#define LLAMAX_MAX_COPY_JOBS 64
typedef struct {
  const void* src;
  void* dst;          /* bf16 */
  int64_t src_ld;     /* elements */
  int64_t dst_ld;     /* elements */
  int32_t rows, cols; /* of src */
  float scale;
  int32_t flags;      /* bit 0: src is fp32 (else bf16); bit 1: transpose */
} llamax_copy_job_t;
int llamax_batched_copy(const llamax_copy_job_t* jobs, int32_t n_jobs, void* stream);

/* ---- K6 backward: LoRA weight gradients (autograd of modelling/lora.py:43) ------------------------
 *   out[p, r] (fp32) = alpha * sum_m X[m, p] * H[m, r]       X bf16 [M,P] pitch ldx;  Ht = H^T bf16 [R, M] pitch ldht
 * used for dB = scale * dY^T h and dA^T = x^T dh.  tcgen05 GEMM with X read as an MN-major operand (no transpose
 * of the big tensor); rank <= 32; `out` is zeroed by the call, token-dimension splits are reduced with fp32 red.add. */
int llamax_lora_wgrad(const void* X, int64_t ldx, const void* Ht, int64_t ldht, void* out, int64_t M, int64_t P,
                      int32_t R, float alpha, void* stream);
/* Deterministic form: each token split stores its fp32 partial into workspace [LLAMAX_LORA_WGRAD_MAX_SPLITS, P, R]
 * (caller-provided; only the first `splits` slices are written) and the splits are summed in split order into `out`.
 * Same arguments as llamax_lora_wgrad plus the workspace. */
#define LLAMAX_LORA_WGRAD_MAX_SPLITS 32
int llamax_lora_wgrad_deterministic(const void* X, int64_t ldx, const void* Ht, int64_t ldht, void* out,
                                    void* workspace, int64_t M, int64_t P, int32_t R, float alpha, void* stream);

/* Fused pair for one LoRA linear's backward (autograd of modelling/lora.py:43), ONE pass over dY [M,N] (pitch lddy):
 *   dh [M,R] bf16 (pitch lddh) = dY . Bt^T            Bt = lora_scale * B^T, bf16 [R,N] pitch ldbt
 *   dB [N,R] fp32 (zeroed by the call) = alpha * dY^T . h       Ht = h^T, bf16 [R,M] pitch ldht
 * rank in {8,16,24,32}. dh_accum: fp32 workspace [M,R] (used when the column range is split across CTAs).
 * dht: NULL, or bf16 [R,M] (pitch lddht) that also receives dh^T — the H^T operand llamax_lora_wgrad needs for dA. */
int llamax_lora_bwd_pair(const void* dY, int64_t lddy, const void* Bt, int64_t ldbt, const void* Ht, int64_t ldht,
                         void* dh, int64_t lddh, void* dht, int64_t lddht, void* dh_accum, void* dB, int64_t M,
                         int64_t N, int32_t R, float alpha, void* stream);


/* ---- K12 (next row): cross-entropy over bf16 logits, forward + backward in place -------------------
 * F.cross_entropy(logits.float(), labels) (modelling/llama.py:216-218, audio.py:74-76), ignore_index = -100:
 *   loss_sum[0] += sum_rows (logsumexp(f32(logits[m,:])) - logits[m, label]);
 *   if write_grad: logits[m,:] <- (softmax(logits[m,:]) - onehot(label)) * inv_n[0]   (0 for ignored rows)
 * logits bf16 [M, V] pitch ld; labels int64 [M]; loss_sum, inv_n: fp32 device scalars. */
int llamax_cross_entropy(void* logits, int64_t ld, const void* labels, void* loss_sum, const void* inv_n, int64_t M,
                         int64_t V, int write_grad, void* stream);
/* Deterministic form: loss_rows fp32 [M] receives each row's loss (0 for ignored rows) instead of an atomic sum into one
 * scalar; the caller sums the rows in a fixed order. The gradient written into the logits is that of llamax_cross_entropy. */
int llamax_cross_entropy_rows(void* logits, int64_t ld, const void* labels, void* loss_rows, const void* inv_n,
                              int64_t M, int64_t V, int write_grad, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LLAMAX_B200_H_ */
