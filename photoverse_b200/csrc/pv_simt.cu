// photoverse_b200 -- fp32 "parity mode" kernels (PV_F32): plain FFMA arithmetic, fp32 storage.
//
// The reference runs this path in fp32 by default (train.py:422, generate.py:73-78); north_star asks for
// <= 1e-4 max-abs against it.  A single-pass TF32 tensor-core product is marginal at K = 320..1280
// (SURVEY.md 7.3), so the fp32 mode keeps full fp32 products and accumulation on the CUDA cores.  It is the
// accuracy mode, not the throughput mode; the bf16 tcgen05 kernels (pv_gemm.cu / pv_attn.cu) are the fast path.
#include "pv_common.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

// ------------------------------------------------------------------------------------------------
// D[b] = A[b] W[b]^T + bias     (64x64 tile, BK=16, 256 threads, 4x4 micro-tile)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
simt_gemm_tn_f32_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ bias,
                        float* __restrict__ D, int M, int N, int K, long long lda, long long ldw, long long ldd,
                        long long strideA, long long strideW, long long strideBias, long long strideD) {
  __shared__ float As[16][64 + 4];
  __shared__ float Ws[16][64 + 4];
  const int b = blockIdx.z;
  A += strideA * b;
  W += strideW * b;
  D += strideD * b;
  const float* bias_b = bias ? bias + strideBias * b : nullptr;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;   // 16 x 16 threads
  const int lr = threadIdx.x >> 2;                           // 0..63 : tile row loaded by this thread
  const int lk = (threadIdx.x & 3) * 4;                      // 0,4,8,12 : first k of its float4
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f), wv = av;
    const int am = m0 + lr, wn = n0 + lr;
    if (am < M) {
      const float* src = A + am * lda + k0 + lk;
      if (k0 + lk + 3 < K && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) av = *reinterpret_cast<const float4*>(src);
      else {
        if (k0 + lk + 0 < K) av.x = src[0];
        if (k0 + lk + 1 < K) av.y = src[1];
        if (k0 + lk + 2 < K) av.z = src[2];
        if (k0 + lk + 3 < K) av.w = src[3];
      }
    }
    if (wn < N) {
      const float* src = W + wn * ldw + k0 + lk;
      if (k0 + lk + 3 < K && ((reinterpret_cast<uintptr_t>(src) & 15) == 0)) wv = *reinterpret_cast<const float4*>(src);
      else {
        if (k0 + lk + 0 < K) wv.x = src[0];
        if (k0 + lk + 1 < K) wv.y = src[1];
        if (k0 + lk + 2 < K) wv.z = src[2];
        if (k0 + lk + 3 < K) wv.w = src[3];
      }
    }
    As[lk + 0][lr] = av.x; As[lk + 1][lr] = av.y; As[lk + 2][lr] = av.z; As[lk + 3][lr] = av.w;
    Ws[lk + 0][lr] = wv.x; Ws[lk + 1][lr] = wv.y; Ws[lk + 2][lr] = wv.z; Ws[lk + 3][lr] = wv.w;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = Ws[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n < N) D[m * ldd + n] = acc[i][j] + (bias_b ? bias_b[n] : 0.f);
    }
  }
}

int gemm_f32(const float* A, const float* W, const float* bias, float* D, long long M, long long N, long long K,
             long long batch, long long lda, long long ldw, long long ldd, long long strideA, long long strideW,
             long long strideBias, long long strideD, cudaStream_t stream) {
  PV_REQUIRE(M > 0 && N > 0 && K > 0 && batch > 0, "empty problem");
  PV_REQUIRE(batch <= 65535 && (M + 63) / 64 <= 65535, "grid too large");
  dim3 grid((N + 63) / 64, (M + 63) / 64, batch);
  simt_gemm_tn_f32_kernel<<<grid, 256, 0, stream>>>(A, W, bias, D, (int)M, (int)N, (int)K, lda, ldw, ldd, strideA,
                                                    strideW, strideBias, strideD);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// fp32 dual-branch attention core: Q:[B,S,C]  K,V:[B,H,L,d]  ->  O:[B,S,C]
// block = (32 queries, head h, sample b); 4 warps, one query per warp at a time.
// ------------------------------------------------------------------------------------------------
constexpr int SA_QPB = 32;

// MASK: the image segment of query row s is weighted w_img * img_row_weight[b, s] (ip_adapter_masks)
template <bool MASK>
__global__ void __launch_bounds__(128)
simt_dual_attn_f32_kernel(const float* __restrict__ Q, const float* __restrict__ Kg, const float* __restrict__ Vg,
                          float* __restrict__ O, float* __restrict__ stats, int S, int C, int H, int d, int Lt, int Li,
                          float w_text, float w_img, float scale_log2e, const float* __restrict__ img_row_weight) {
  extern __shared__ float sm[];
  const int L = Lt + Li;
  const int dk = d + 1;                     // padded K row: conflict-free when lanes walk keys
  float* Ks = sm;                           // [L][d+1]
  float* Vs = Ks + L * dk;                  // [L][d]
  float* qs = Vs + L * d;                   // [4][d]
  float* ps = qs + 4 * d;                   // [4][96]
  const int b = blockIdx.z, h = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* Kb = Kg + (static_cast<size_t>(b) * H + h) * L * d;
  const float* Vb = Vg + (static_cast<size_t>(b) * H + h) * L * d;
  for (int i = threadIdx.x; i < L * d; i += blockDim.x) {
    const int k = i / d, c = i % d;
    Ks[k * dk + c] = Kb[i];
    Vs[i] = Vb[i];
  }
  __syncthreads();
  float* q_w = qs + warp * d;
  float* p_w = ps + warp * PV_KEYS_PAD;
  for (int qi = warp; qi < SA_QPB; qi += 4) {
    const int srow = blockIdx.x * SA_QPB + qi;
    if (srow >= S) break;                   // warp-uniform
    const float* qg = Q + (static_cast<size_t>(b) * S + srow) * C + h * d;
    for (int c = lane; c < d; c += 32) q_w[c] = qg[c];
    __syncwarp();
    float sc[3];
    float mt = -INFINITY, mi = -INFINITY;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int k = lane + 32 * t;
      float a = 0.f;
      if (k < L) {
        const float* kr = Ks + k * dk;
        for (int c = 0; c < d; ++c) a = fmaf(q_w[c], kr[c], a);
        if (k < Lt) mt = fmaxf(mt, a); else mi = fmaxf(mi, a);
      }
      sc[t] = a;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      mt = fmaxf(mt, __shfl_xor_sync(0xffffffffu, mt, o));
      mi = fmaxf(mi, __shfl_xor_sync(0xffffffffu, mi, o));
    }
    const float mts = mt * scale_log2e, mis = mi * scale_log2e;
    float lt = 0.f, li = 0.f;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int k = lane + 32 * t;
      float e = 0.f;
      if (k < Lt) { e = exp2f(fmaf(sc[t], scale_log2e, -mts)); lt += e; }
      else if (k < L) { e = exp2f(fmaf(sc[t], scale_log2e, -mis)); li += e; }
      sc[t] = e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lt += __shfl_xor_sync(0xffffffffu, lt, o);
      li += __shfl_xor_sync(0xffffffffu, li, o);
    }
    const float at = w_text / lt;
    const float wi = MASK ? w_img * __ldg(img_row_weight + static_cast<size_t>(b) * S + srow) : w_img;
    const float ai = (Li > 0) ? wi / li : 0.f;
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const int k = lane + 32 * t;
      if (k < L) p_w[k] = sc[t] * ((k < Lt) ? at : ai);
    }
    if (stats != nullptr && lane == 0) {
      const size_t idx = (static_cast<size_t>(b) * H + h) * S + srow;
      reinterpret_cast<float4*>(stats)[idx] = make_float4(mts, lt, mis, li);
    }
    __syncwarp();
    float* og = O + (static_cast<size_t>(b) * S + srow) * C + h * d;
    for (int c = lane; c < d; c += 32) {
      float a = 0.f;
      for (int k = 0; k < L; ++k) a = fmaf(p_w[k], Vs[k * d + c], a);
      og[c] = a;
    }
    __syncwarp();
  }
}

int dual_attn_core_f32(const float* Q, const float* Kp, const float* Vp, float* O, float* stats, int B, int S, int C,
                       int H, int Lt, int Li, float w_text, float w_img, cudaStream_t stream, const float* img_row_weight) {
  PV_REQUIRE(B > 0 && S > 0 && H > 0 && C % H == 0, "bad shape");
  PV_REQUIRE(Lt >= 1 && Li >= 1 && Lt + Li <= PV_KEYS_PAD, "need 1 <= Lt, 1 <= Li, Lt+Li <= %d", PV_KEYS_PAD);
  const int d = C / H, L = Lt + Li;
  const size_t smem = (static_cast<size_t>(L) * (d + 1) + static_cast<size_t>(L) * d + 4 * d + 4 * PV_KEYS_PAD) * sizeof(float);
  PV_REQUIRE(smem <= 200 * 1024, "head_dim %d too large for the fp32 kernel", d);
  const bool mask = img_row_weight != nullptr;
  auto kern = mask ? simt_dual_attn_f32_kernel<true> : simt_dual_attn_f32_kernel<false>;
  static size_t attr_smem[2] = {0, 0};
  if (smem > attr_smem[mask]) {
    PV_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_smem[mask] = smem;
  }
  PV_REQUIRE(B <= 65535 && H <= 65535, "grid too large");
  dim3 grid((S + SA_QPB - 1) / SA_QPB, H, B);
  kern<<<grid, 128, smem, stream>>>(Q, Kp, Vp, O, stats, S, C, H, d, Lt, Li, w_text, w_img,
                                    1.4426950408889634f / sqrtf(static_cast<float>(d)), img_row_weight);
  PV_LAUNCHED();
  return PV_OK;
}

}  // namespace pv
