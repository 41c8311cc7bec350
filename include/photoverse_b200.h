/* photoverse_b200.h -- C ABI of libphotoverse_b200.so (sm_100a only).
 *
 * B200-native replacement for the arithmetic of PhotoVerse's dual-branch conditioning hot path:
 *   reference  models/attention_processor.py:245-435  PhotoVerseAttnProcessor2_0.__call__
 *   reference  models/adapters.py:30-44               PhotoVerseAdapter.forward
 *   reference  models/unet.py:38-47                   get_visual_cross_attention_values_norm (side output)
 *   dependency peft 0.10.0 lora.Linear.forward        (LoRA on attn2.to_q/to_k/to_v, train.py:348-354)
 *
 * The reference has no FFI (it is pure PyTorch); these entry points are what a binding for this path
 * binds instead of the library calls listed in SURVEY.md section 2.2 (P1-P15, A1-A9).  INTEGRATION.md shows the
 * ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch); the library allocates nothing
 *     persistent except cached TMA descriptors; all tensors are dense row-major unless strides are given
 *   - all calls are asynchronous on `stream` (a cudaStream_t passed as void*), perform no host sync and
 *     no allocation, and are CUDA-graph capturable
 *   - return value: PV_OK or an error code; pv_last_error() gives the message; nothing throws
 *   - pv_dtype selects the arithmetic path:
 *        PV_BF16  bf16 storage, tcgen05 tensor-core MMAs with fp32 accumulation in TMEM (throughput mode)
 *        PV_F32   fp32 storage, fp32 FFMA arithmetic (parity mode: <= 1e-4 of the fp32 reference)
 *        PV_F16   fp16 storage, the PV_BF16 kernels with fp16 operands (kind::f16 MMAs, fp32 accumulation), for models
 *                 run in float16.  Inference only: pv_pack_weight, pv_linear_fwd, pv_kv_tile_bytes, pv_kv_pack_fwd,
 *                 pv_dual_attn_fwd, pv_dual_attn_core_fwd, pv_ln_lrelu_fwd and pv_group_mean_fwd accept it (wherever
 *                 they say PV_BF16 below, the same holds for PV_F16); every other entry point returns PV_ERR_UNSUPPORTED.
 *                 Values are rounded to fp16 (to nearest) exactly where the PV_BF16 path rounds to bf16.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point returns PV_ERR_CUDA
 */
#ifndef PHOTOVERSE_B200_H_
#define PHOTOVERSE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PV_ABI_VERSION 2

enum { PV_OK = 0, PV_ERR_INVALID = 1, PV_ERR_CUDA = 2, PV_ERR_UNSUPPORTED = 3 };
typedef enum { PV_F32 = 0, PV_BF16 = 1, PV_F16 = 2 } pv_dtype;

/* Keys are zero-padded to this many rows per (sample, head) in the packed K/V tiles. */
#define PV_KEYS_PAD 96
/* PV_BF16 tiles: text keys occupy slots [0,Lt), image keys slots [PV_IMG_KEY_OFFSET, PV_IMG_KEY_OFFSET+Li).
 * Limits of the fused kernel: 1 <= Lt <= 80 (CLIP: 77), 1 <= Li <= 16.                                    */
#define PV_IMG_KEY_OFFSET 80

int pv_version(void);
const char* pv_last_error(void);
/* Number of kernels this library has launched since it was loaded (bench.py: "gpu_launches"). */
unsigned long long pv_launch_count(void);
/* TEST-ONLY process-wide switches (not thread-safe; production code never calls this).  Every value selects among
 * kernels that compute the same result ("sattn_poly": to within the bf16 rounding of P):
 *   "fuse_out" 2|1|0      out projection as the second phase of the attention launch for every S > 128 shape | where it
 *                         is at least as fast as two launches (default: C <= 320) | always a separate GEMM launch
 *   "gemm_persistent" 1|0 persistent CTA-pair GEMM for out-projection-shaped pv_linear_fwd calls | single-CTA kernel
 *   "gemm_two_cta" 1|0, "force_bn" 0|64|128|160|256, "epi_swizzle" 1|0   tile choices of the single-CTA GEMM
 *   "pdl" 1|0             programmatic dependent launch of the persistent kernels
 *   "bwd_mma" 1|0         bf16 attention backward on tensor cores | the fp32-accurate SIMT kernel
 *   "bwd_tc" 1|0          ... on tcgen05 with TMEM accumulators where supported (head_dim 40 / 80) | the mma.sync kernel
 *   "sattn_poly" 0|2|4    pv_self_attn_fwd: exponentials out of every 8 pairs computed by a degree-3 polynomial on the FMA
 *                         pipe instead of MUFU (default 2; 7.5e-5 relative, below the bf16 rounding of P)
 *   "trace_block" n       which leader CTA writes the debug timeline (PV_TRACE builds)
 * Unknown names return PV_ERR_INVALID.                                                                         */
int pv_set_option(const char* name, int value);
/* Debug builds only (PV_TRACE=1 python -m photoverse_b200.build --force): device buffer of 4 + 3*capacity uint64
 * (zeroed by the caller) that one CTA of the persistent attention kernels fills with (event, index, SM clock)
 * triples; NULL switches it off.  Release builds return PV_ERR_INVALID for a non-NULL buffer.                    */
int pv_debug_trace(void* buf, int capacity_events);

/* ---- weights ---------------------------------------------------------------------------------------
 * W_eff[out,in] = W[out,in] + scaling * B[out,r] * A[r,in]   (peft lora.Linear merged form; r == 0 -> cast)
 * fp32 masters in, `out_dt` out.  Replaces the two skinny GEMMs + scale + add per projection (SURVEY 2.2 a5)
 * for every call in which the weights did not change.                                                   */
int pv_pack_weight(pv_dtype out_dt, const float* W, const float* lora_A, const float* lora_B, float scaling,
                   void* W_eff, int out_features, int in_features, int r, void* stream);

/* ---- generic projection -----------------------------------------------------------------------------
 * D[b] = A[b] * W[b]^T + bias[b]     A:[batch,M,K] (row stride lda, batch stride strideA, elements)
 *                                    W:[batch,N,K] (ldw, strideW; strideW == 0 -> one shared weight)
 *                                    bias fp32 [batch,N] (strideBias) or NULL;  D:[batch,M,N] (ldd, strideD)
 * dt is the type of A and W; out_dt the type of D (dt or, for PV_BF16 / PV_F16, PV_F32).  PV_BF16 / PV_F16: K % 8 == 0
 * and 16-byte aligned rows.
 * Replaces nn.Linear (attention_processor.py:297,304,305,392,393,423; adapters.py:14-28).
 * Stream-ordering precondition: W and bias must not be the OUTPUT of the kernel enqueued immediately before this
 * call on `stream` (they are weights: the persistent kernels fetch them before their programmatic-dependent-launch
 * wait; A and D are only touched after it).  Weights written two or more kernels earlier are fine.            */
int pv_linear_fwd(pv_dtype dt, pv_dtype out_dt, const void* A, const void* W, const float* bias, void* D,
                  int64_t M, int64_t N, int64_t K, int64_t batch, int64_t lda, int64_t ldw, int64_t ldd,
                  int64_t strideA, int64_t strideW, int64_t strideBias, int64_t strideD, void* stream);

/* ---- K/V projection + pack (attention_processor.py:304-313, 392-397) --------------------------------
 * text:[B,Lt,Dc]  img:[B,Li,Dc]  (dt)      Wkv_text:[2C,Dc] = [to_k_eff ; to_v_eff]   Wkv_img:[2C,Dc] = [to_k_ip ; to_v_ip]
 * kv_text_ws:[B*Lt,2C] fp32, kv_img_ws:[B*Li,2C] fp32   (outputs; also saved for backward)
 * Kp, Vp: packed per-(sample,head) key / value tiles consumed by pv_dual_attn_fwd:
 *     PV_BF16: Kp[b][h] = UMMA K-major core-matrix image of [PV_KEYS_PAD x d_pad], Vp[b][h] = image of V^T
 *              [d_pad x PV_KEYS_PAD]; d_pad = round_up(C/H,16); pv_kv_tile_bytes() each
 *     PV_F32 : Kp, Vp = [B,H,Lt+Li,d] fp32
 * v_ip_norm:[B,H,Li] fp32 = ||V_img||_2 over head_dim  (the processor's `to_v_ip_norm` side output)     */
int64_t pv_kv_tile_bytes(pv_dtype dt, int C, int H, int Lt, int Li);
int pv_kv_pack_fwd(pv_dtype dt, const void* text, const void* img, const void* Wkv_text, const void* Wkv_img,
                   float* kv_text_ws, float* kv_img_ws, void* Kp, void* Vp, float* v_ip_norm, int B, int Lt, int Li,
                   int Dc, int C, int H, void* stream);

/* ---- the dual-branch cross-attention (attention_processor.py:297, 307-322, 400-425) -----------------
 * Y = (w_text * softmax(Q K_t^T / sqrt(d)) V_t + w_img * softmax(Q K_i^T / sqrt(d)) V_i) Wo^T + bo,  Q = X Wq^T
 * X,Y:[B,S,C] (dt)   Wq,Wo:[C,C] (dt, Wq already LoRA-merged)   bo:[C] fp32   Kp,Vp from pv_kv_pack_fwd
 * ws_q : PV_F32 only, [B,S,C] fp32 scratch for Q (may be NULL for PV_BF16: Q never leaves the SM)
 * ws_o : [B,S,C] (dt) attention output before the out projection (saved for backward)
 * stats: optional [B,H,S,4] fp32 = (max_text, sum_text, max_img, sum_img) of the scaled logits, for backward
 * ws_sync: PV_BF16, optional: pv_dual_attn_sync_words(B, S) uint32 words, ZERO on entry and left zero on return
 *          (row-block counters; one buffer may serve any number of calls that are ordered on one stream).
 * PV_BF16 path with ws_sync, S > 128 (and, by default, C <= 320: see pv_set_option "fuse_out"): ONE persistent tcgen05
 * launch per processor call -- per CTA pair:
 * Q-projection -> QK^T over the concatenated keys -> per-segment softmax with the branch weights folded in -> ONE PV
 * contraction -> O to global memory; then, in the same launch, the pair's share of the out-projection tiles
 * (Wo + bias), each tile starting as soon as the row block's head groups have announced their O rows on ws_sync.
 * Without ws_sync (or S <= 128, a single row tile per sample) the out projection is a second tcgen05 GEMM launch.
 * Same precondition on Wq / Wo / bo as pv_linear_fwd (weights, not outputs of the immediately preceding kernel).
 * Supported head dims: 40, 80, 160 (C = 320, 640, 1280 with H = 8); 1 <= Lt <= 80; 1 <= Li <= 16.                */
int64_t pv_dual_attn_sync_words(int B, int S);
int pv_dual_attn_fwd(pv_dtype dt, const void* X, const void* Wq, const void* Kp, const void* Vp, const void* Wo,
                     const float* bo, void* Y, float* ws_q, void* ws_o, float* stats, unsigned int* ws_sync, int B, int S,
                     int C, int H, int Lt, int Li, float w_text, float w_img, void* stream);

/* The fused kernel alone (no out projection): PV_BF16: XorQ = X [B,S,C] bf16 and Wq is used (Q-projection fused);
 * PV_F32: XorQ = Q [B,S,C] fp32 (already projected) and Wq is ignored.  O:[B,S,C] (dt).  Used by the roofline
 * measurement in bench.py and by the backward pass (recompute).                                               */
int pv_dual_attn_core_fwd(pv_dtype dt, const void* XorQ, const void* Wq, const void* Kp, const void* Vp, void* O,
                          float* stats, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                          void* stream);

/* ---- adapter epilogues (adapters.py:15-16,18-19: LayerNorm(1024) -> LeakyReLU(0.01)) ----------------
 * y = leaky_relu(layer_norm(x) * gamma + beta); x:[rows,cols] fp32 (row stride ldx), y:[rows,cols] out_dt
 * (row stride ldy; PV_F32, PV_BF16 or PV_F16); cols % 128 == 0, cols <= 4096.  Optional mean / rstd [rows] fp32 saved for backward.
 * gamma/beta:[groups,cols]; row i uses group i / rows_per_group (rows_per_group <= 0: one shared gamma/beta) --
 * the T token heads of an adapter are normalised in one launch.
 * One warp per row, 16-byte vector loads, warp-shuffle reductions.                                        */
int pv_ln_lrelu_fwd(pv_dtype out_dt, const float* x, const float* gamma, const float* beta, void* y,
                    float* save_mean, float* save_rstd, int64_t rows, int cols, int64_t ldx, int64_t ldy,
                    int64_t rows_per_group, float eps, float slope, void* stream);
/* y[g, :] = mean over the P rows of group g: x:[groups,P,cols] (in_dt) -> y:[groups,cols] (out_dt, row stride ldy)
 * (adapters.py:36,41 `.mean(dim=1, keepdim=True)` over the 256 patch tokens, commuted in front of the last
 * Linear: mean(L3(h)) == L3(mean(h)), SURVEY 2.2 A8).  A 16-bit in_dt and a 16-bit out_dt must be the same type.   */
int pv_group_mean_fwd(pv_dtype in_dt, pv_dtype out_dt, const void* x, void* y, int64_t groups, int P, int cols,
                      int64_t ldy, void* stream);

/* ============================== backward (training step, reference train.py:495-538) ==============================
 * Trainable set of the path: adapters, to_k_ip / to_v_ip, LoRA A/B on attn2.to_q/to_k/to_v (train.py:348-370).  Input
 * gradients flow through every attn2 layer into the frozen UNet (accelerator.backward, train.py:538).
 * All reductions are two-pass and deterministic.  Workspaces are caller-owned; sizes from the *_ws_bytes queries.   */

/* W_eff^T[in,out] = (W + scaling * B A)^T in `out_dt`: the weight of an input-gradient GEMM  dX = dY W_eff, which is
 * pv_linear_fwd(dY, W_eff^T).  (autograd of attention_processor.py:297,304,305,392,393,423 and adapters.py:14-28)     */
int pv_pack_weight_t(pv_dtype out_dt, const float* W, const float* lora_A, const float* lora_B, float scaling,
                     void* W_eff_t, int out_features, int in_features, int r, void* stream);

/* out[c, r] = in[r, c]  (in:[rows,cols] row stride ldi; out:[cols, ldo] with columns [rows, ldo) zero-filled).  Turns the
 * packed forward weights into the weights of the input-gradient GEMMs without touching the fp32 masters again.       */
int pv_transpose_2d(pv_dtype dt, const void* in, void* out, int64_t rows, int64_t cols, int64_t ldi, int64_t ldo, void* stream);

/* dW[N,K] (fp32, dense) = alpha * sum_m G[m,n] X[m,k] + beta * dW    G:[M,N] (row stride ldg), X:[M,K] (ldx), both dt.
 * bf16 with M >= 512, N,K >= 128: transposes + tcgen05 GEMM over K' = M; otherwise fp32 SIMT split-M.                */
int64_t pv_linear_bwd_weight_ws_bytes(pv_dtype dt, int64_t M, int64_t N, int64_t K);
int pv_linear_bwd_weight(pv_dtype dt, const void* G, const void* X, float* dW, void* ws, int64_t M, int64_t N, int64_t K,
                         int64_t ldg, int64_t ldx, float alpha, float beta, void* stream);

/* Both LoRA factor gradients of one projection y = W x + scaling * B (A x) (peft 0.10.0 lora.Linear; train.py:348-354) in
 * one pass over the activations:  dA = scaling * (G B)^T X  [r,in],  dB = scaling * G^T (X A^T)  [out,r],
 * X:[M,in] (row stride ldx), G = dL/dy:[M,out] (ldg) in dt; lora_A:[r,in], lora_B:[out,r] fp32 masters;
 * dAB: fp32 [r*in + out*r] = dA then dB.  1 <= r <= 16 and in, out <= 1280: pv_lora_bwd_ws_bytes returns the workspace
 * size, or -1 when the shape is outside the kernel (rank 128: use pv_linear_fwd + pv_linear_bwd_weight).
 * Deterministic (per-block partials summed in a fixed order).                                                        */
int64_t pv_lora_bwd_ws_bytes(int64_t M, int in_features, int out_features, int r);
int pv_lora_bwd(pv_dtype dt, const void* X, const void* G, const float* lora_A, const float* lora_B, float scaling, float* dAB,
                void* ws, int64_t M, int in_features, int out_features, int r, int64_t ldx, int64_t ldg, void* stream);

/* out[n] = sum_m G[m,n]  (bias gradients) */
int64_t pv_col_sum_ws_bytes(int64_t M, int64_t N);
int pv_col_sum(pv_dtype dt, const void* G, float* out, void* ws, int64_t M, int64_t N, int64_t ldg, void* stream);

/* Backward of pv_ln_lrelu_fwd.  da, dx:[groups*rows_per_group, cols] (dt, dense); x fp32 pre-normalisation input and
 * mean / rstd as saved by the forward; gamma/beta:[groups,cols]; dgamma/dbeta:[groups,cols] fp32.  cols == 1024.      */
int64_t pv_ln_lrelu_bwd_ws_bytes(int64_t groups, int64_t rows_per_group, int cols);
int pv_ln_lrelu_bwd(pv_dtype dt, const void* da, const float* x, const float* mean, const float* rstd, const float* gamma,
                    const float* beta, void* dx, float* dgamma, float* dbeta, void* ws, int64_t groups,
                    int64_t rows_per_group, int cols, float slope, void* stream);

/* Backward of pv_group_mean_fwd: dx[g,p,:] = dy[g,:] / P   (dy row stride ldy; dx dense [groups,P,cols]) */
int pv_group_mean_bwd(pv_dtype dt, const void* dy, void* dx, int64_t groups, int P, int cols, int64_t ldy, void* stream);

/* Backward of the attention core (autograd of attention_processor.py:307-322, 400-420 with the two normalisers).
 * dO, Q, dQ:[B,S,C] (dt); kv_text:[B*Lt,2C], kv_img:[B*Li,2C] fp32 projections and stats:[B,H,S,4] from the forward;
 * ws receives per-query-chunk partial dK / dV, reduced by pv_kv_pack_bwd into dkv_text:[B*Lt,2C], dkv_img:[B*Li,2C]
 * (dt; columns [0,C) dK, [C,2C) dV) together with the backward of the `to_v_ip_norm` side output
 * (d_v_ip_norm:[B,H,Li] fp32 or NULL; models/unet.py:38-47, train.py:512-513).                                         */
int64_t pv_dual_attn_bwd_ws_bytes(int B, int S, int C, int H, int Lt, int Li);
int pv_dual_attn_bwd(pv_dtype dt, const void* dO, const void* Q, const float* kv_text, const float* kv_img,
                     const float* stats, void* dQ, void* ws, int B, int S, int C, int H, int Lt, int Li, float w_text,
                     float w_img, void* stream);
int pv_kv_pack_bwd(pv_dtype dt, const void* ws, const float* kv_img, const float* v_ip_norm, const float* d_v_ip_norm,
                   void* dkv_text, void* dkv_img, int B, int S, int Lt, int Li, int C, int H, void* stream);

/* ---- concept-token injection (models/clip.py:17-24 `_inject_concept_embeddings`; SURVEY 8 f2) -----------------------
 * out[b,l] = in[b,l] (l < idx_b) | concept[b,l-idx_b] (idx_b <= l < idx_b+T) | in[b,l-T+1] (l >= idx_b+T)
 * inputs_embeds, out:[B,L,cols]; concept:[B,T,cols] (dt); placeholder_idx:[B] int32 (device), 0 <= idx_b, idx_b + T <= L.
 * Backward: d_inputs_embeds:[B,L,cols] (zero at the dropped placeholder and at the truncated tail), d_concept:[B,T,cols]. */
int pv_inject_concept_fwd(pv_dtype dt, const void* inputs_embeds, const void* concept, const int* placeholder_idx,
                          void* out, int B, int L, int T, int cols, void* stream);
int pv_inject_concept_bwd(pv_dtype dt, const void* d_out, const int* placeholder_idx, void* d_inputs_embeds,
                          void* d_concept, int B, int L, int T, int cols, void* stream);

/* ---- training objective (train.py:509-535; SURVEY 8 f4) ---------------------------------------------------------------
 * loss = mean((noise_pred - noise)^2) + w_text * mean|concept| + w_vis * mean(v_ip_norms)     (reference: 0.01 / 0.001)
 * noise_pred, noise: n elements; concept: m elements (text adapter output, :509); v_ip_norms: k elements (the stacked
 * `to_v_ip_norm` side outputs of the attn2 processors, models/unet.py:38-47), all dt.  out4 (fp32, device) = {loss,
 * l_mse, l_text, l_vis}.  Two launches, fixed summation order.  Backward: d_loss is a device scalar (fp32);
 * d_noise_pred [n], d_concept [m], d_v_ip_norms [k] in dt.                                                              */
int64_t pv_train_loss_ws_bytes(void);
int pv_train_loss_fwd(pv_dtype dt, const void* noise_pred, const void* noise, int64_t n, const void* concept, int64_t m,
                      const void* v_ip_norms, int64_t k, float w_text, float w_vis, float* out4, void* ws, void* stream);
int pv_train_loss_bwd(pv_dtype dt, const void* noise_pred, const void* noise, int64_t n, const void* concept, int64_t m, int64_t k,
                      float w_text, float w_vis, const float* d_loss, void* d_noise_pred, void* d_concept, void* d_v_ip_norms,
                      void* stream);

/* ---- self-attention of the `attn1` layers (reference models/unet.py:20-24 installs diffusers' stock AttnProcessor2_0
 * there: O = softmax(Q K^T / sqrt(d)) V per (sample, head); SURVEY 8 row f4) -----------------------------------------
 * q, k, v: bf16 [B, S, *] views with a common row stride `ld` (elements; e.g. three slices of one fused [B,S,3C]
 * projection, ld = 3C), head h in columns [h*d, (h+1)*d); out: bf16 [B,S,C] contiguous.  d = C / heads in {40, 80, 160}.
 * ws: pv_self_attn_ws_bytes(B,S,C,heads) bytes of scratch (operand images).  Inference only (no statistics saved).  */
int64_t pv_self_attn_ws_bytes(int B, int S, int C, int heads);
int pv_self_attn_fwd(const void* q, const void* k, const void* v, int64_t ld, void* out, void* ws, int B, int S, int C,
                     int heads, void* stream);

/* ---- LoRA dropout backward (peft==0.10.0 lora.Linear.forward `lora_B(lora_A(dropout(x))) * scaling`, configured at
 * train.py:264-269, 348-354; SURVEY 8 a6) --------------------------------------------------------------------------
 * dst[i] += keep_mask[i] ? alpha * src[i] : 0, alpha = 1/(1-p).  dst, src: n elements (dt), n % 8 == 0;
 * keep_mask: n bytes (the boolean keep-mask drawn in the forward pass).                                            */
int pv_dropout_bwd_acc(pv_dtype dt, void* dst, const void* src, const uint8_t* keep_mask, float alpha, int64_t n,
                       void* stream);

/* ---- HBM-bound epilogues of the UNet evaluation that calls the path (SURVEY 8 row f1; reference models/infer.py:103-116
 * runs diffusers' UNet2DConditionModel: ResnetBlock2D `norm -> SiLU -> conv`, Transformer2DModel `norm -> proj_in`,
 * FeedForward GEGLU).  Inference only, bf16. ---------------------------------------------------------------------------
 * pv_group_norm_nhwc_fwd: y = [SiLU](GroupNorm_groups(x + add) * gamma + beta) on a CHANNELS-LAST activation: x, y are
 * [B, HW, C] dense (the memory of a torch.channels_last [B, C, H, W] tensor), gamma / beta fp32 [C]; add_bc: optional fp32
 * [B, C] addend broadcast over the pixels (NULL = none) -- ResnetBlock2D's `conv1 bias + time_emb_proj(temb)` between
 * conv1 and norm2; statistics in fp32 over the HW * C / groups elements of a (sample, group), biased variance, `eps`
 * inside the square root (torch.nn.GroupNorm).  C % 8 == 0, C % groups == 0, groups <= 64, C <= 4096.
 * ws: pv_group_norm_nhwc_ws_bytes(...) bytes of scratch (partial sums; -1 = unsupported shape).  Two launches, fixed
 * summation order.  save_stats: optional fp32 [B, groups, 2] = (mean, rstd) kept for the backward pass (NULL in inference).
 * pv_group_norm_nhwc_bwd: dx = d loss / d x of the same expression from dy (layout of x), x, add_bc and the saved stats;
 * gamma / beta are frozen on the PhotoVerse path (train.py:348-370 trains adapters, to_k_ip / to_v_ip and LoRA factors
 * only), so no affine gradients are produced.  Same workspace size, two launches.
 * pv_add_bias_nhwc_fwd: out[r, c] = a[r, c] + b[r, c] + bias[c] (rows x C dense, bias fp32, C % 8 == 0; out may alias a
 * or b) -- a block's residual sum together with the bias of its last convolution.
 * pv_layer_norm_fwd: y = LayerNorm(s) * gamma + beta over the last dimension, s = x [rows, C] dense, C % 8 == 0, C <= 1280,
 * gamma / beta fp32 (BasicTransformerBlock norm1 / norm2 / norm3).  With `residual` (and `sum_out`, both or neither):
 * s = x + residual, rounded to bf16 and written to sum_out -- the block's `x = attn(...) + x` in the pass of the norm
 * that follows it.  pv_layer_norm_bwd: its input gradient from dy and x
 * (frozen affine; mean / rstd are recomputed from the row).
 * pv_geglu_fwd: y[m, n] = h[m, n] * gelu(h[m, N + n]) with the exact (erf) GELU, gelu(.) rounded to bf16 before the
 * product like the two-kernel torch sequence; h: [M, 2N] with row stride ldh (elements), y: [M, N] dense; N % 8 == 0.
 * pv_geglu_bwd: dh [M, 2N] dense = [dy * gelu(gate) | dy * hidden * gelu'(gate)] from h and dy [M, N] dense.
 * pv_linear_geglu_fwd: y[m, n] = h[m, n] * gelu(h[m, N + n]) for the projection h = x W^T + b of an nn.Linear(K, 2N), in one
 * launch without writing h: x [M, K] bf16 (row stride ldx), y [M, N] bf16 (row stride ldy).  w_packed [2N, K] bf16 dense and
 * b_packed fp32 [2N] (or NULL) are W and b with their rows regrouped per 80 output columns: packed rows [160 j, 160 j + 80)
 * are rows [80 j, 80 j + 80) of W, packed rows [160 j + 80, 160 j + 160) are rows N + [80 j, 80 j + 80).  h is rounded
 * to bf16 after the bias and the rest rounds like pv_geglu_fwd.  N % 80 == 0, K % 64 == 0; a row's result does not
 * depend on M.  The packed weight must not be written by the kernel launched just before (it is read ahead of it). */
int64_t pv_group_norm_nhwc_ws_bytes(int64_t B, int64_t HW, int C, int groups);
int pv_group_norm_nhwc_fwd(pv_dtype dt, const void* x, const float* add_bc, const float* gamma, const float* beta, void* y,
                           float* save_stats, void* ws, int64_t B, int64_t HW, int C, int groups, float eps, int silu,
                           void* stream);
int pv_group_norm_nhwc_bwd(pv_dtype dt, const void* x, const float* add_bc, const void* dy, const float* stats,
                           const float* gamma, const float* beta, void* dx, void* ws, int64_t B, int64_t HW, int C, int groups,
                           int silu, void* stream);
int pv_add_bias_nhwc_fwd(pv_dtype dt, const void* a, const void* b, const float* bias, void* out, int64_t rows, int C,
                         void* stream);
int pv_layer_norm_fwd(pv_dtype dt, const void* x, const void* residual, void* sum_out, const float* gamma, const float* beta,
                      void* y, int64_t rows, int C, float eps, void* stream);
int pv_layer_norm_bwd(pv_dtype dt, const void* x, const void* dy, const float* gamma, void* dx, int64_t rows, int C, float eps,
                      void* stream);
int pv_geglu_fwd(pv_dtype dt, const void* h, void* y, int64_t M, int N, int64_t ldh, void* stream);
int pv_geglu_bwd(pv_dtype dt, const void* h, const void* dy, void* dh, int64_t M, int N, int64_t ldh, void* stream);
int pv_linear_geglu_fwd(pv_dtype dt, const void* x, const void* w_packed, const float* b_packed, void* y, int64_t M, int64_t N,
                        int64_t K, int64_t ldx, int64_t ldy, void* stream);

/* ---- activation dtype conversion (torch.autocast over a float32 model, DESIGN.md 4.9) -------------------------------
 * dst[i] = src[i] converted from in_dt to out_dt, n elements, both dense.  Pairs: PV_F32 -> PV_BF16, PV_F32 -> PV_F16,
 * PV_BF16 -> PV_F32, PV_F16 -> PV_F32; any other pair returns PV_ERR_UNSUPPORTED.  Round to nearest even: bit-identical to
 * torch.Tensor.to for every finite input; fp16 overflow gives +-inf; NaN stays NaN (payload not preserved).  Pointers need
 * only element alignment (vector accesses start at the first common 32-byte / 16-byte boundary).  n == 0 launches nothing. */
int pv_convert_fwd(pv_dtype in_dt, pv_dtype out_dt, const void* src, void* dst, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PHOTOVERSE_B200_H_ */
