/*
 * mxprune.h - C ABI of libmxprune.so: the MXINT8 exponent-sign pruned-attention hot path
 * of d9bjo0522/mx_quantization, rebuilt as sm_100a CUDA.
 *
 * Every entry point is `extern "C"`, takes raw DEVICE pointers, explicit element strides and a
 * CUDA stream (passed as void*, i.e. a cudaStream_t), allocates nothing, never synchronises the
 * host and keeps no device state.  Work is enqueued asynchronously on `stream`, like the
 * PyTorch ops it replaces.  Return value: 0 on success, <0 on error (MXP_E_*); the message of the
 * last error on the calling thread is available from mxp_last_error().
 *
 * Tensors named q/k/v/x/out are fp32 "(B,H,N,hd)" views: element (b,h,n,d) lives at
 * ptr[b*sB + h*sH + n*sN + d] (strides in ELEMENTS, innermost stride 1).  This covers the three
 * layouts the reference's attention modules produce:
 *   - fused qkv buffer, permuted view   workloads/deit/scripts/main.py:87-88, DiT models.py:156-157
 *   - separate (B,N,H*hd) projections   workloads/PixArt/models/MX_transformer_block.py:637-639
 *   - plain contiguous (B,H,N,hd)       benchmarks / tests
 * Requirements: hd % 4 == 0, 4 <= hd <= 128, base pointers and row strides 16-byte aligned.
 *
 * 16-bit activations (the *_dt entry points, MXP_DT_BF16 / MXP_DT_F16): q, k and v share one element type, and the
 * result is the result of the same call on the exactly widened fp32 values - identical masks, indices, codes and
 * exponents, and the same fp32 output before its final store.  A1 (bfloat 16) and the subnormal flush act on the
 * widened values.  out is fp32 or the input type; a 16-bit out is the fp32 result rounded to nearest even.  There is
 * no conversion pass: a 16-bit call enqueues the launches of the fp32 call of the same shape and needs the same
 * workspace.  Views: strides in elements, base pointers and the three strides 16-byte aligned (strides % 8 == 0).
 * Scope: the exponent-sign predictor with the default path switches (the tensor-core predictor and attention; any
 * fused-path mode), head_dim a multiple of 8 in [32, 128], every Nk the fp32 path accepts, with or without key_bias;
 * anything else returns MXP_E_UNSUPPORTED.  key_bias stays fp32.
 *
 * Compact MXINT8 format shared by all entry points (SURVEY.md section 8a):
 *   code  int8  in [-127,127]   (sign-magnitude semantics; -128 never produced)
 *   exp   int8  in [-127,127]   one per 32 elements of head_dim; -126 marks an all-zero block
 *   value = code * 2^(exp-6);   predictor value = (code<0 ? -1 : +1) * 2^exp
 *
 * mx_specs (microxscaling/mx/specs.py:61-181) reaches this ABI as two integers:
 *   bfloat_bits  16 or 32   mx_specs["bfloat"]  (bf16 pre-rounding, half away from zero)
 *   flush        0 or 1     mx_specs["mx_flush_fp32_subnorms"]
 * every other key is validated host-side to the only combination on the path
 * (int8 / block 32 / round nearest / shared_exp max / scale_bits 8).
 */
#ifndef MXPRUNE_H_
#define MXPRUNE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MXP_ABI_VERSION 8

/*
 * Element types of q/k/v/x and out for the *_dt entry points.  The fp32 entry points are the *_dt ones with
 * MXP_DT_F32 everywhere.
 */
#define MXP_DT_F32  0
#define MXP_DT_BF16 1
#define MXP_DT_F16  2

#define MXP_OK             0
#define MXP_E_BADARG      -1   /* null pointer, bad shape/stride/alignment, k out of range */
#define MXP_E_UNSUPPORTED -2   /* shape outside what the kernels cover (see mxp_limits)     */
#define MXP_E_CUDA        -3   /* launch / runtime error reported by CUDA                   */

int mxp_abi_version(void);
const char* mxp_last_error(void);           /* thread-local, never NULL */

/* Largest key count and head_dim the kernels accept.  Every entry point that takes keys (predict_scores, predict_topk*,
 * sparse_attention*, pruned_attention*) returns MXP_E_UNSUPPORTED for more keys before it launches anything; the
 * quantizer takes any number of rows. */
void mxp_limits(int* max_keys, int* max_head_dim);

/*
 * MX block quantizer.  Replaces
 *   quantize_mx_op(quantize_elemwise_op(x, mx_specs, round), mx_specs, elem_format="int8",
 *                  axes=[-1], round="nearest")
 *   microxscaling/mx/mx_ops.py:309-341 (+ :180-306), elemwise_ops.py:243-277
 * but emits the integer codes/exponents instead of fake-quantised fp32.
 *   codes  int8  [B,H,N,hd]  contiguous           (required)
 *   exps   int8  [B,H,N,nb]  nb = ceil(hd/32)     (required)
 *   signs  u32   [B,H,N,nb]  bit d of word b = (code[b*32+d] < 0); may be NULL
 */
int mxp_quantize_mxint8(const float* x, int64_t sB, int64_t sH, int64_t sN,
                        int B, int H, int N, int hd, int bfloat_bits, int flush,
                        int8_t* codes, int8_t* exps, uint32_t* signs, void* stream);
/* x of element type x_dtype (MXP_DT_*); 16-bit x: head_dim a multiple of 8 (any such head_dim of the fp32 call) */
int mxp_quantize_mxint8_dt(const void* x, int x_dtype, int64_t sB, int64_t sH, int64_t sN,
                           int B, int H, int N, int hd, int bfloat_bits, int flush,
                           int8_t* codes, int8_t* exps, uint32_t* signs, void* stream);

/*
 * Dense exponent-sign approximation, (code<0 ? -1 : +1) * 2^exp per element, fp32 contiguous
 * [B,H,N,hd].  Replaces funcs.exponent_approximation(Q,K,mx_specs).exponent_based_sign()
 *   funcs/exponent_based_prediction.py:12-38,44-94 (call once per tensor).
 * Parity / debugging aid: the fused kernels never materialise this.
 */
int mxp_exp_sign_approx(const float* x, int64_t sB, int64_t sH, int64_t sN,
                        int B, int H, int N, int hd, int bfloat_bits, int flush,
                        float* approx, void* stream);

/*
 * Dense predicted scores, fp32 contiguous [B,H,Nq,Nk]:
 *   score[i,j] = sum_b 2^(eq[i,b]+ek[j,b]) * (n_b - 2*popc(sq[i,b]^sk[j,b]))
 * Replaces `pred_scores = ex_quant_q @ ex_quant_k.transpose(-2,-1)`
 *   workloads/deit/scripts/main.py:118, DiT models.py:186, MX_transformer_block.py:673.
 * Parity aid (O(N^2) output); the product path is mxp_predict_topk.
 */
int mxp_predict_scores(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                       const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                       int B, int H, int Nq, int Nk, int hd, int bfloat_bits, int flush,
                       float* scores, void* stream);

/*
 * Fused quantize + exponent-sign predictor + per-row top-k.  Q and K are read once; the
 * Nq x Nk score matrix is never written.  Replaces lines 107-123 of
 * workloads/deit/scripts/main.py (exponent_approximation ctor, exponent_based_sign, `@`,
 * torch.topk) and the same sequence in DiT models.py:178-194 /
 * PixArt MX_transformer_block.py:659-678.
 * Tie rule: descending score, ascending key index (first top_k of a stable descending sort).
 *   mask     u32 [B,H,Nq,ceil(Nk/32)]  bit (j%32) of word j/32 set iff key j is kept (required)
 *   idx      i32 [B,H,Nq,top_k]        kept keys in ascending key order; may be NULL
 *   q_codes  int8 [B,H,Nq,hd], q_exps int8 [B,H,Nq,nb]   may be NULL (both or neither)
 *   k_codes  int8 [B,H,Nk,hd], k_exps int8 [B,H,Nk,nb]   may be NULL (both or neither)
 * workspace: mxp_predict_topk_workspace_bytes() bytes of device memory (may be NULL if 0).
 */
size_t mxp_predict_topk_workspace_bytes(int B, int H, int Nq, int Nk, int hd);
int mxp_predict_topk(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                     const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                     int B, int H, int Nq, int Nk, int hd, int top_k,
                     int bfloat_bits, int flush,
                     uint32_t* mask, int32_t* idx,
                     int8_t* q_codes, int8_t* q_exps, int8_t* k_codes, int8_t* k_exps,
                     void* workspace, size_t workspace_bytes, void* stream);
/* q and k of element type in_dtype (MXP_DT_*) */
int mxp_predict_topk_dt(const void* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                        const void* k, int64_t k_sB, int64_t k_sH, int64_t k_sN, int in_dtype,
                        int B, int H, int Nq, int Nk, int hd, int top_k,
                        int bfloat_bits, int flush,
                        uint32_t* mask, int32_t* idx,
                        int8_t* q_codes, int8_t* q_exps, int8_t* k_codes, int8_t* k_exps,
                        void* workspace, size_t workspace_bytes, void* stream);

/*
 * Exact MXINT8 attention over the kept keys.  Replaces
 *   true_scores = mx.matmul(q, k^T) * scale ; vals = gather(idx) ; softmax ; scatter_ ;
 *   x = mx.matmul(attn, v)            workloads/deit/scripts/main.py:101-102,124,147-152
 * given Q/K already in compact form and the row bitmask of kept keys.  V (fp32) is quantised
 * along TOKENS in blocks of 32 (microxscaling/mx/matmul.py:76-83, axes=[-2]); P is quantised
 * along keys in 32-aligned windows of original key positions.
 *   out  fp32 (B,H,Nq,hd) view with element strides o_sB,o_sH,o_sN (innermost 1)
 */
size_t mxp_sparse_attention_workspace_bytes(int B, int H, int Nq, int Nk, int hd);
int mxp_sparse_attention(const int8_t* q_codes, const int8_t* q_exps,
                         const int8_t* k_codes, const int8_t* k_exps,
                         const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                         const uint32_t* mask,
                         int B, int H, int Nq, int Nk, int hd,
                         float scale, int bfloat_bits, int flush,
                         float* out, int64_t o_sB, int64_t o_sH, int64_t o_sN,
                         void* workspace, size_t workspace_bytes, void* stream);
/* v of element type v_dtype, out of element type out_dtype (MXP_DT_*; fp32 or v_dtype) */
int mxp_sparse_attention_dt(const int8_t* q_codes, const int8_t* q_exps,
                            const int8_t* k_codes, const int8_t* k_exps,
                            const void* v, int64_t v_sB, int64_t v_sH, int64_t v_sN, int v_dtype,
                            const uint32_t* mask,
                            int B, int H, int Nq, int Nk, int hd,
                            float scale, int bfloat_bits, int flush,
                            void* out, int64_t o_sB, int64_t o_sH, int64_t o_sN, int out_dtype,
                            void* workspace, size_t workspace_bytes, void* stream);

/*
 * The whole path in one call: q,k,v -> out.  Replaces lines 101-152 of
 * workloads/deit/scripts/main.py (and DiT models.py:168-225, PixArt
 * MX_transformer_block.py:647-710) for mx_quant && top_k && approx_flag && pred_mode=="ex_pred".
 *   mask_out  optional u32 [B,H,Nq,ceil(Nk/32)] copy of the kept-key bitmask (may be NULL)
 * workspace: mxp_pruned_attention_workspace_bytes() bytes, 256-byte aligned.
 */
size_t mxp_pruned_attention_workspace_bytes(int B, int H, int Nq, int Nk, int hd);
int mxp_pruned_attention(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                         const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                         const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                         int B, int H, int Nq, int Nk, int hd, int top_k,
                         float scale, int bfloat_bits, int flush,
                         float* out, int64_t o_sB, int64_t o_sH, int64_t o_sN,
                         uint32_t* mask_out,
                         void* workspace, size_t workspace_bytes, void* stream);

/*
 * Cross-attention with an additive key bias (SURVEY 8 f1): PixArt-alpha's MXCrossAttention adds the
 * text-token mask to BOTH the true and the predicted scores before top-k and softmax
 * (workloads/PixArt/models/MX_transformer_block.py:794-803, 821-822):
 *     true_scores += attn_bias ;  pred_scores = ex_q @ ex_k^T + attn_bias
 * key_bias[b * kb_sB + j] is that bias for key j of batch element b (the reference's (B,1,1,S) mask,
 * the same for every head and query row; finite values, e.g. (1 - mask) * -10000).  Nq and Nk may
 * differ; every Nk of mxp_pruned_attention (up to mxp_limits' max_keys).  Beyond 256 keys the tensor-core
 * selection adds the bias to its integer keys; rows it cannot rank exactly (a bias no integer key carries, a threshold
 * among keys below its window) are ranked by the CUDA-core kernel on fp32 keys fl32(pred + bias_j), exact for any
 * finite bias, and the streamed attention kernel adds bias_j after score * scale.  Everything else as mxp_pruned_attention.
 */
int mxp_pruned_attention_biased(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                                const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                                const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                                int B, int H, int Nq, int Nk, int hd, int top_k,
                                float scale, int bfloat_bits, int flush,
                                float* out, int64_t o_sB, int64_t o_sH, int64_t o_sN,
                                const float* key_bias, int64_t kb_sB,
                                uint32_t* mask_out,
                                void* workspace, size_t workspace_bytes, void* stream);
/* mxp_pruned_attention / mxp_pruned_attention_biased with q, k, v of element type in_dtype and out of element type
 * out_dtype (MXP_DT_*; fp32 or in_dtype); key_bias may be NULL */
int mxp_pruned_attention_dt(const void* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                            const void* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                            const void* v, int64_t v_sB, int64_t v_sH, int64_t v_sN, int in_dtype,
                            int B, int H, int Nq, int Nk, int hd, int top_k,
                            float scale, int bfloat_bits, int flush,
                            void* out, int64_t o_sB, int64_t o_sH, int64_t o_sN, int out_dtype,
                            const float* key_bias, int64_t kb_sB,
                            uint32_t* mask_out,
                            void* workspace, size_t workspace_bytes, void* stream);

/*
 * The reference's other sources of the top-k ranking (SURVEY 8 f3), behind the same call:
 *   MXP_PRED_EXP_SIGN   pred_mode == "ex_pred"     both sides +-2^e                 (== mxp_pruned_attention)
 *   MXP_PRED_PARTIAL_Q  pred_mode == "partial_Q"   Q = MXINT8 value, K = +-2^e      funcs/exponent_based_prediction.py:300-318
 *   MXP_PRED_PARTIAL_K  pred_mode == "partial_K"   Q = +-2^e, K = MXINT8 value      funcs/exponent_based_prediction.py:274-298
 *   MXP_PRED_EXACT      approx_flag == False       top-k of the true scores mx.matmul(q, k^T) * scale
 *                                                   workloads/deit/scripts/main.py:101-102,130
 *   MXP_PRED_MXINT4     pred_mode == "MXINT4"      both sides MXINT4 values (Sanger)    funcs/exponent_based_prediction.py:179-199
 *   MXP_PRED_TWO_STEP   pred_mode == "two_step_leading_ones" (EXION)  sign * e * (2^f1 + 2^f2) / 64
 *                                                                       funcs/exponent_based_prediction.py:96-177
 *   MXP_PRED_TRUE_EX    pred_mode == "true_ex"     sign * 2^floor(log2 |element|) per element
 *                                                   microxscaling/examples/deit/exponent_based_prediction.py:163-178
 * (callers: main.py:107-123, DiT models.py:178-194, MX_transformer_block.py:659-673).  Modes 1-6 need Nk <= 256 and head_dim a multiple
 * of 8, >= 32 (MXP_E_UNSUPPORTED otherwise); `scale` ranks the exact mode and scales the attention in
 * every mode.  key_bias (may be NULL) is the additive cross-attention bias of mxp_pruned_attention_biased, added
 * in fp32 to the ranked value of every mode (MX_transformer_block.py:803,822); modes 1-6 keep their Nk <= 256 limit
 * with a bias too (mode 0 takes it up to max_keys).  mxp_predict_topk_mode is the
 * selection alone (mask / idx as mxp_predict_topk).
 */
#define MXP_PRED_EXP_SIGN  0
#define MXP_PRED_PARTIAL_Q 1
#define MXP_PRED_PARTIAL_K 2
#define MXP_PRED_EXACT     3
#define MXP_PRED_MXINT4    4
#define MXP_PRED_TWO_STEP  5
#define MXP_PRED_TRUE_EX   6
int mxp_pruned_attention_mode(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                              const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                              const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                              int B, int H, int Nq, int Nk, int hd, int top_k, int pred_mode,
                              float scale, int bfloat_bits, int flush,
                              float* out, int64_t o_sB, int64_t o_sH, int64_t o_sN,
                              const float* key_bias, int64_t kb_sB,
                              uint32_t* mask_out,
                              void* workspace, size_t workspace_bytes, void* stream);
int mxp_predict_topk_mode(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                          const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                          int B, int H, int Nq, int Nk, int hd, int top_k, int pred_mode,
                          float scale, int bfloat_bits, int flush,
                          const float* key_bias, int64_t kb_sB,
                          uint32_t* mask, int32_t* idx,
                          void* workspace, size_t workspace_bytes, void* stream);

/*
 * ELSA ranking (funcs/elsa_approximation.py:60-145, workloads/deit/scripts/main.py:119-121): keys are ranked per
 * query row on  ||K_i|| * cos(max(pi/d * h - 0.127, 0)),  h = Hamming distance of the d-bit sign hashes of the MXINT8
 * rows of Q and K under the d x d orthogonal matrix `proj` (fp32 row-major on the device, 16-byte aligned; hash j =
 * (x . proj[j] >= 0)).  Inside a row that is the order of min(d - 2h, rank_cap), rank_cap = d - 2 h_c with h_c the
 * largest h the reference's fp32 clamp maps to angle 0 (the caller evaluates that clamp; mx_quantization_b200.ops
 * does).  Nq == Nk = N as in the reference, d = head_dim <= 80, N <= 256.  Hash bits of projections within fp32
 * rounding distance of 0 depend on the summation order (the reference's BLAS vs. this library).
 */
int mxp_pruned_attention_elsa(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                              const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                              const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                              int B, int H, int N, int hd, int top_k, const float* proj, float rank_cap,
                              float scale, int bfloat_bits, int flush,
                              float* out, int64_t o_sB, int64_t o_sH, int64_t o_sN,
                              uint32_t* mask_out,
                              void* workspace, size_t workspace_bytes, void* stream);
int mxp_predict_topk_elsa(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                          const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                          int B, int H, int N, int hd, int top_k, const float* proj, float rank_cap,
                          int bfloat_bits, int flush, uint32_t* mask, int32_t* idx, void* stream);

/*
 * MX Linear (SURVEY 8 f2, the step either side of the attention core): the forward of the
 * reference's mx.Linear (microxscaling/mx/linear.py:20-103) for MXINT8 activations and weights,
 *     y = A1( A1( MXq(A1(x)) . MXq(A1(W))^T ) + A1(bias) )
 * both operands MX-quantized along in_features in blocks of 32 (quantize_mx_op, axes=[-1]),
 * A1 = quantize_elemwise_op (bf16 half-away rounding for bfloat 16, identity for 32).
 *   x     fp32 (M, K) rows with stride ldx      W   fp32 (N, K) rows with stride ldw
 *   out   fp32 (M, N) rows with stride ldo      bias fp32 (N) or NULL
 * The weight is quantized once into the GEMM's operand order (mxp_mx_linear_prepare_weight ->
 * w_op, mxp_mx_linear_weight_bytes bytes); mxp_mx_linear quantizes the activations into the
 * workspace and runs the bf16 x bf16 -> fp32 GEMM on the tensor cores (the MXINT8 values are exact
 * in bf16).  K must be a multiple of 64, N a multiple of 4.
 */
size_t mxp_mx_linear_weight_bytes(int N, int K);
size_t mxp_mx_linear_workspace_bytes(int M, int N, int K);
int mxp_mx_linear_prepare_weight(const float* w, int64_t ldw, int N, int K, int bfloat_bits, int flush,
                                 void* w_op, void* stream);
int mxp_mx_linear(const float* x, int64_t ldx, int M, int K, const void* w_op, int N, const float* bias,
                  int bfloat_bits, int flush, float* out, int64_t ldo,
                  void* workspace, size_t workspace_bytes, void* stream);
/*
 * 16-bit MX Linear: W (w_dtype), x (x_dtype) and bias (bias_dtype) are each MXP_DT_F32, MXP_DT_BF16 or MXP_DT_F16,
 * independently; out has x_dtype.  The result is the fp32 call on the exactly widened W, x and bias, rounded to
 * nearest even when out is 16-bit (with bfloat 16 the fp32 result is already a bf16 value, so a bf16 out is
 * lossless).  A w_op prepared from a 16-bit W is byte-equal to the one of the widened W.  No conversion pass: a
 * 16-bit call enqueues the launches of the fp32 call and needs the same workspace.  A 16-bit x or W needs a 16-byte
 * aligned base and a row stride that is a multiple of 8 elements; a 16-bit out needs an 8-byte aligned base and a
 * row stride that is a multiple of 4 elements.  The fp32 entry points are these with MXP_DT_F32 everywhere.
 */
int mxp_mx_linear_prepare_weight_dt(const void* w, int w_dtype, int64_t ldw, int N, int K, int bfloat_bits,
                                    int flush, void* w_op, void* stream);
int mxp_mx_linear_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N,
                     const void* bias, int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo,
                     void* workspace, size_t workspace_bytes, void* stream);

/*
 * Fused MX MLP (a transformer block's fc1 -> activation -> fc2, timm Mlp):
 *     out = mx_linear(act(mx_linear(x, W1, b1)), W2, b2)
 * as the library computes the composition, bit for bit: fc1's output is rounded to x's type (as mxp_mx_linear_dt
 * stores it), the activation is torch.nn.functional.gelu on CUDA in fp32 opmath (bit-identical for every input)
 * rounded to x's type again, and fc2 quantizes that along N1.  The fp32 rounding steps are identities.  The hidden
 * activation is never written in a float type: fc1's epilogue applies the activation, quantizes each 32-element MX
 * block in registers and writes fc2's bf16 operand into the workspace.
 *   act      MXP_ACT_GELU (approximate='none', DeiT) or MXP_ACT_GELU_TANH (approximate='tanh', DiT, PixArt)
 *   x        (M, K) rows of x_dtype with stride ldx (the rules of mxp_mx_linear_dt)
 *   w1_op    fc1's prepared weight (N1, K);  w2_op  fc2's prepared weight (N2, N1)  (mxp_mx_linear_prepare_weight_dt)
 *   b1, b2   N1 / N2 biases of any MXP_DT_* type each, or NULL
 *   out      (M, N2) of x_dtype, row stride ldo (the rules of mxp_mx_linear_dt's out)
 * K and N1 multiples of 64, N2 a multiple of 4.  Launches, in order: x's quantizer, the rounding of b1 and of b2 (each
 * only when present), fc1 with the activation epilogue, fc2: 3 to 5 kernels.  workspace: mxp_mx_mlp_workspace_bytes
 * bytes, 256-byte aligned (x's operand, the hidden operand ceil(M/128)*128 x N1 bf16, the rounded biases).
 */
#define MXP_ACT_GELU      0
#define MXP_ACT_GELU_TANH 1
size_t mxp_mx_mlp_workspace_bytes(int M, int K, int N1, int N2);
int mxp_mx_mlp_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1,
                  const void* b1, int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype,
                  int bfloat_bits, int flush, void* out, int64_t ldo,
                  void* workspace, size_t workspace_bytes, void* stream);
/*
 * Parity aid: the fused MLP's activation applied elementwise to n contiguous elements of type dtype (MXP_DT_*), the
 * result in the same type (rounded to nearest even from fp32 for 16-bit types).  Equals torch.nn.functional.gelu on
 * CUDA bit for bit for every non-NaN input (NaN in, NaN out).
 */
int mxp_activation_dt(const void* x, int dtype, int64_t n, int act, void* out, void* stream);

/*
 * adaLN-modulated MX Linear / MLP (DiT's DiTBlock, PixArt's adaLN-single block):
 *     out = residual + gate * mx_linear(x * (1 + scale) + shift, W, bias)
 * mxp_mx_linear_adaln_dt takes the arguments of mxp_mx_linear_dt; mxp_mx_mlp_adaln_dt those of mxp_mx_mlp_dt, with the
 * modulation applied to x (fc1's operand) and the gated residual to fc2's output.  The M rows are B = M / tokens batch
 * entries of `tokens` rows each; row r belongs to entry b = r / tokens.  Every added tensor has x_dtype.
 *   shift, scale      (B, K) rows with strides ld_shift / ld_scale (the rules of x); both NULL, or both given.  The GEMM
 *                     operand is quantized from v = rd(rd(x * rd(1 + scale[b])) + shift[b]) instead of x.
 *   residual          (M, N) rows with stride ld_residual;  gate  (B, N) rows with stride ld_gate (both the rules of
 *                     out); both NULL, or both given.  The stored value is rd(residual + rd(gate[b] * y)), where y is
 *                     the value mxp_mx_linear_dt stores (already rounded to x_dtype).
 * Each operation is one fp32 add or multiply (no contraction), rd rounds to nearest even in x_dtype (the identity for
 * fp32): the expressions as eager torch evaluates them on tensors of x_dtype, so the result equals the torch
 * composition with the plain entry point bit for bit.  shift / scale / gate may be column slices of one (B, 6C) row
 * (DiT's adaLN_modulation(c).chunk(6, dim=1)), read in place.  Padding rows of a partial 128-row tile read none of
 * them.  tokens must divide M.  The launches and the workspace are those of the plain call.
 */
int mxp_mx_linear_adaln_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N,
                           const void* bias, int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo,
                           int tokens, const void* shift, int64_t ld_shift, const void* scale, int64_t ld_scale,
                           const void* residual, int64_t ld_residual, const void* gate, int64_t ld_gate,
                           void* workspace, size_t workspace_bytes, void* stream);
int mxp_mx_mlp_adaln_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1,
                        const void* b1, int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype,
                        int bfloat_bits, int flush, void* out, int64_t ldo, int tokens, const void* shift,
                        int64_t ld_shift, const void* scale, int64_t ld_scale, const void* residual,
                        int64_t ld_residual, const void* gate, int64_t ld_gate, void* workspace,
                        size_t workspace_bytes, void* stream);

/*
 * Pre-norm MX Linear / MLP with every block addition optional (DeiT's timm Block, DiT, PixArt-alpha):
 *     out = add(f(modulate(layer_norm(x))))
 * mxp_mx_linear_ex_dt takes the arguments of mxp_mx_linear_adaln_dt, mxp_mx_mlp_ex_dt those of mxp_mx_mlp_adaln_dt,
 * with three differences:
 *   layer_norm        1: the operand is quantized from torch.nn.functional.layer_norm(x, (K,), ln_weight, ln_bias,
 *                     ln_eps) on CUDA, bit for bit (mxp_layer_norm_dt's y, rounded to x_dtype), before the
 *                     modulation; 0: no norm (ln_weight / ln_bias must be NULL).
 *   ln_weight, ln_bias  K elements of x_dtype each, 16-byte (fp32) or 8-byte (16-bit) aligned; both or neither.
 *   residual without gate  a plain add: the stored value is rd(residual + y) (DeiT's x + attn(norm1(x))).  With the
 *                     gate it is the gated residual of the adaLN entry points.  gate without residual is an error.
 * Without shift / scale / gate, tokens only has to divide M (pass M).  Launches, in order: with the norm, the row
 * statistics kernel (k_layer_norm: one warp per row of x, writing each row's fp32 mean and rstd to the
 * workspace); then exactly the launches of the plain call (x's quantizer applies the norm and the modulation as it
 * loads x; the last GEMM's store applies the residual).  workspace: mxp_mx_linear_ex_workspace_bytes /
 * mxp_mx_mlp_ex_workspace_bytes bytes, 256-byte aligned: the plain call's workspace followed by the statistics,
 * 2 * align256(4 * M) bytes (without the norm the plain call's size suffices).
 */
size_t mxp_mx_linear_ex_workspace_bytes(int M, int N, int K);
size_t mxp_mx_mlp_ex_workspace_bytes(int M, int K, int N1, int N2);
int mxp_mx_linear_ex_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w_op, int N,
                        const void* bias, int bias_dtype, int bfloat_bits, int flush, void* out, int64_t ldo,
                        int layer_norm, const void* ln_weight, const void* ln_bias, float ln_eps, int tokens,
                        const void* shift, int64_t ld_shift, const void* scale, int64_t ld_scale, const void* residual,
                        int64_t ld_residual, const void* gate, int64_t ld_gate, void* workspace,
                        size_t workspace_bytes, void* stream);
int mxp_mx_mlp_ex_dt(const void* x, int x_dtype, int64_t ldx, int M, int K, const void* w1_op, int N1, const void* b1,
                     int b1_dtype, int act, const void* w2_op, int N2, const void* b2, int b2_dtype, int bfloat_bits,
                     int flush, void* out, int64_t ldo, int layer_norm, const void* ln_weight, const void* ln_bias,
                     float ln_eps, int tokens, const void* shift, int64_t ld_shift, const void* scale, int64_t ld_scale,
                     const void* residual, int64_t ld_residual, const void* gate, int64_t ld_gate, void* workspace,
                     size_t workspace_bytes, void* stream);
/*
 * Parity aid: the LayerNorm the _ex entry points apply, on (M, K) rows of x (dtype MXP_DT_*, row stride ldx):
 * torch.native_layer_norm(x, (K,), weight, bias, eps) on CUDA bit for bit - y (contiguous (M, K) of dtype), and the
 * fp32 mean and rstd of each row.  weight and bias: K elements of dtype each, or both NULL.  K a multiple of 4 up to
 * 2^24 (the rows torch's vectorized kernel takes); x, y, weight and bias 16-byte (fp32) or 8-byte (16-bit) aligned,
 * ldx a multiple of 4.  One launch (k_layer_norm), no workspace.
 */
int mxp_layer_norm_dt(const void* x, int dtype, int64_t ldx, int M, int K, const void* weight, const void* bias,
                      float eps, void* y, float* mean, float* rstd, void* stream);

/*
 * Measurement aid: same as mxp_pruned_attention (tcgen05 path), but brackets the three kernels
 * (predict+top-k, V operand prep, exact attention) with CUDA events on `stream`, SYNCHRONISES, and
 * returns their durations in milliseconds in kernel_ms[0..2].  bench.py's roofline uses this.
 */
int mxp_pruned_attention_profile(const float* q, int64_t q_sB, int64_t q_sH, int64_t q_sN,
                                 const float* k, int64_t k_sB, int64_t k_sH, int64_t k_sN,
                                 const float* v, int64_t v_sB, int64_t v_sH, int64_t v_sN,
                                 int B, int H, int Nq, int Nk, int hd, int top_k,
                                 float scale, int bfloat_bits, int flush,
                                 float* out, int64_t o_sB, int64_t o_sH, int64_t o_sN,
                                 uint32_t* mask_out,
                                 void* workspace, size_t workspace_bytes, void* stream, float* kernel_ms);

/*
 * Which implementation mxp_sparse_attention / mxp_pruned_attention use for the exact stage:
 *   0 (default)  tcgen05 tensor cores: bf16 operands (exact for MXINT8 values), fp32 TMEM accumulators
 *   1            CUDA-core dp4a gather path (kept for A/B measurement; needs head_dim % 4 == 0 only)
 * Process-wide; returns MXP_E_BADARG for any other value.
 */
int mxp_set_attention_path(int path);

/*
 * Which kernel scores the predictor (funcs/exponent_based_prediction.py:44-94 + the caller's
 * `ex_q @ ex_k^T`, workloads/deit/scripts/main.py:118) when Nk <= 256:
 *   0 (default)  +-2^e bf16 operands on the tcgen05 tensor cores (exact inside the integer-key window),
 *                keys selected in registers; needs head_dim % 8 == 0 and head_dim >= 32
 *   1            XOR/POPC on CUDA cores (also used automatically outside the domain of path 0)
 * Both return identical masks.  Process-wide; returns MXP_E_BADARG for any other value.
 */
int mxp_set_predict_path(int path);

/*
 * The round-2 kernels behind mxp_pruned_attention (same results as the three-kernel path they replace;
 * workloads/deit/scripts/main.py:101-152 as one launch):
 *   1 (default)  k_fused_pruned_attention - quantizer, predictor, top-k, V preparation and exact attention in ONE
 *                persistent launch - when top_k / Nk <= 0.35 (129 <= Nk <= 256, >= 64 heads, no key bias), where the
 *                exact stage runs on the k gathered entries only (main.py:124,147-152) and the launch is measured
 *                faster than the three kernels; the cost-follows-k attention kernel alone for smaller problems;
 *                everything else on the three-kernel path
 *   2            the fused launch wherever the shape is in its domain, dense epilogue included (tests, A/B)
 *   0            always the three-kernel path with the dense-epilogue attention kernels (A/B aid); for Nk > 256, where
 *                the attention kernel is the same in every mode, the long-sequence selection with its radix levels
 *                alone (no sampled window)
 * Process-wide; returns MXP_E_BADARG for any other value.
 */
int mxp_set_fused_path(int path);

/* Debug aid: per-phase cycle accounting of the fused kernel.  device_buffer = 320 * 32 uint64 of device memory
 * (zeroed by the caller), or NULL to switch the accounting off; the next fused launches add, per 256-thread group,
 * the clock64() cycles its thread 0 spent in each phase (slot meanings: tools/fused_timing.py). */
int mxp_debug_fused_timing(void* device_buffer);
/* Debug / A-B aid: 1 (default) = the two groups of a fused CTA take turns in phase 1 (quantize + select), 0 = unsynchronised. */
int mxp_debug_fused_pingpong(int on);

/* Number of kernel launches the last successful call on this thread enqueued (bench.py's
 * gpu_launches claim is counted from this). */
int mxp_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* MXPRUNE_H_ */
