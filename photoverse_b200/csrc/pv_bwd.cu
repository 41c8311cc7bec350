// photoverse_b200 -- backward kernels of the dual-branch conditioning path (training: reference train.py:495-538).
//
// Weight gradients flow only into the small trainable set (to_k_ip / to_v_ip, LoRA A/B on to_q/to_k/to_v, the two
// adapters); input gradients flow through every attn2 layer back into the frozen UNet.  Division of labour:
//   * dense, well-shaped contractions (dO = dY Wo, dX = dQ Wq, d text = dKV Wkv, adapter dX / dW)   -> the tcgen05 GEMM
//     of pv_gemm.cu, fed with transposed weights (pack_weight_t) or transposed activations (transpose2d)
//   * the attention core (two-normaliser softmax backward, deterministic dK / dV reduction over the queries) and
//     the skinny LoRA / K-V weight gradients                                                         -> fp32 SIMT kernels here
//   * LayerNorm+LeakyReLU backward, column sums, patch-mean backward                                  -> HBM-bound kernels here
// All reductions are two-pass (per-block partials, then an ordered sum): results are run-to-run deterministic.
#include "pv_common.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

int gemm_bf16(const void* A, const void* W, const float* bias, void* D, bool out_f32, long long M, long long N,
              long long K, long long batch, long long lda, long long ldw, long long ldd, long long strideA,
              long long strideW, long long strideBias, long long strideD, cudaStream_t stream, bool w_static = false,
              bool f16 = false);

template <typename T> __device__ __forceinline__ float ldf(const T* p);
template <> __device__ __forceinline__ float ldf<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) { return __bfloat162float(*p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v);
template <> __device__ __forceinline__ void stf<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }

// ------------------------------------------------------------------------------------------------
// W_eff^T[in, out] = (W + scaling * B A)^T  -> the "weight" of an input-gradient GEMM  dX = dY W_eff
// ------------------------------------------------------------------------------------------------
template <typename TO>
__global__ void __launch_bounds__(256)
pack_weight_t_kernel(const float* __restrict__ W, const float* __restrict__ A, const float* __restrict__ Bm,
                     float scaling, TO* __restrict__ out, int out_f, int in_f, int r) {
  __shared__ float tile[32][33];
  const int o0 = blockIdx.y * 32, i0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;     // 32 x 8
  for (int rr = ty; rr < 32; rr += 8) {
    const int o = o0 + rr, i = i0 + tx;
    float v = 0.f;
    if (o < out_f && i < in_f) {
      v = W[static_cast<size_t>(o) * in_f + i];
      if (r > 0) {
        float dlt = 0.f;
        for (int k = 0; k < r; ++k) dlt = fmaf(Bm[static_cast<size_t>(o) * r + k], A[static_cast<size_t>(k) * in_f + i], dlt);
        v = fmaf(scaling, dlt, v);
      }
    }
    tile[rr][tx] = v;
  }
  __syncthreads();
  for (int rr = ty; rr < 32; rr += 8) {
    const int i = i0 + rr, o = o0 + tx;
    if (i < in_f && o < out_f) stf(out + static_cast<size_t>(i) * out_f + o, tile[tx][rr]);
  }
}

int pack_weight_t(bool out_bf16, const float* W, const float* A, const float* Bm, float scaling, void* out, int out_f,
                  int in_f, int r, cudaStream_t stream) {
  PV_REQUIRE(out_f > 0 && in_f > 0 && r >= 0, "bad shape out=%d in=%d r=%d", out_f, in_f, r);
  PV_REQUIRE(r == 0 || (A != nullptr && Bm != nullptr), "LoRA rank %d without A/B", r);
  dim3 grid((in_f + 31) / 32, (out_f + 31) / 32);
  if (out_bf16) pack_weight_t_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(W, A, Bm, scaling, static_cast<__nv_bfloat16*>(out), out_f, in_f, r);
  else pack_weight_t_kernel<float><<<grid, 256, 0, stream>>>(W, A, Bm, scaling, static_cast<float*>(out), out_f, in_f, r);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// out[c, r] = in[r, c]   (rows r < R, cols c < Cc; out row stride ldo >= R, columns [R, ldo) zero-filled)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
transpose2d_kernel(const T* __restrict__ in, T* __restrict__ out, long long R, long long Cc, long long ldi, long long ldo) {
  __shared__ T tile[32][33];
  const long long r0 = static_cast<long long>(blockIdx.y) * 32, c0 = static_cast<long long>(blockIdx.x) * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int rr = ty; rr < 32; rr += 8) {
    const long long r = r0 + rr, c = c0 + tx;
    tile[rr][tx] = (r < R && c < Cc) ? in[r * ldi + c] : T(0.f);
  }
  __syncthreads();
  for (int rr = ty; rr < 32; rr += 8) {
    const long long c = c0 + rr, r = r0 + tx;
    if (c < Cc && r < ldo) out[c * ldo + r] = tile[tx][rr];
  }
}

int transpose_2d(bool bf16, const void* in, void* out, long long R, long long Cc, long long ldi, long long ldo, cudaStream_t stream) {
  PV_REQUIRE(R > 0 && Cc > 0 && ldi >= Cc && ldo >= R, "bad shape R=%lld C=%lld ldi=%lld ldo=%lld", R, Cc, ldi, ldo);
  PV_REQUIRE((ldo + 31) / 32 <= 65535, "too many rows");
  dim3 grid(static_cast<unsigned>((Cc + 31) / 32), static_cast<unsigned>((ldo + 31) / 32));
  if (bf16) transpose2d_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(in), static_cast<__nv_bfloat16*>(out), R, Cc, ldi, ldo);
  else transpose2d_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(in), static_cast<float*>(out), R, Cc, ldi, ldo);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// dW[N,K] = alpha * sum_m G[m,n] X[m,k]   -- SIMT fp32, split over M, deterministic two-pass reduction
// ------------------------------------------------------------------------------------------------
constexpr int WG_MCHUNK = 128;       // rows per block: a block walks them in 16-row steps, so short chunks = many blocks

template <typename T>
__global__ void __launch_bounds__(256)
wgrad_partial_kernel(const T* __restrict__ G, const T* __restrict__ X, float* __restrict__ part, long long M, int N, int K,
                     long long ldg, long long ldx) {
  __shared__ float Gs[16][64 + 4];
  __shared__ float Xs[16][64 + 4];
  const int n0 = blockIdx.y * 64, k0 = blockIdx.x * 64;
  const long long m_begin = static_cast<long long>(blockIdx.z) * WG_MCHUNK;
  const long long m_end = m_begin + WG_MCHUNK < M ? m_begin + WG_MCHUNK : M;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lm = threadIdx.x >> 4;            // 0..15: row of the 16-row step loaded by this thread
  const int lc = (threadIdx.x & 15) * 4;      // first of its 4 columns
  float acc[4][4] = {};
  for (long long m0 = m_begin; m0 < m_end; m0 += 16) {
    const long long m = m0 + lm;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + lc + j, k = k0 + lc + j;
      Gs[lm][lc + j] = (m < m_end && n < N) ? ldf(G + m * ldg + n) : 0.f;
      Xs[lm][lc + j] = (m < m_end && k < K) ? ldf(X + m * ldx + k) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int mm = 0; mm < 16; ++mm) {
      float g[4], x[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) g[i] = Gs[mm][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) x[j] = Xs[mm][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(g[i], x[j], acc[i][j]);
    }
    __syncthreads();
  }
  float* dst = part + static_cast<size_t>(blockIdx.z) * N * K;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int n = n0 + ty * 4 + i;
    if (n >= N) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx * 4 + j;
      if (k < K) dst[static_cast<size_t>(n) * K + k] = acc[i][j];
    }
  }
}

// out[i] = alpha * sum_z part[z][i] (+ beta * out[i])
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const float* __restrict__ part, float* __restrict__ out, long long n, int splits, float alpha, float beta) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int z = 0; z < splits; ++z) s += part[static_cast<size_t>(z) * n + i];
  out[i] = (beta != 0.f) ? fmaf(beta, out[i], alpha * s) : alpha * s;
}

__global__ void __launch_bounds__(256)
scale_copy_kernel(const float* __restrict__ in, float* __restrict__ out, long long n, float alpha, float beta) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (beta != 0.f) ? fmaf(beta, out[i], alpha * in[i]) : alpha * in[i];
}

long long wgrad_ws_bytes(bool bf16, long long M, long long N, long long K) {
  const long long splits = (M + WG_MCHUNK - 1) / WG_MCHUNK;
  const long long simt = splits * N * K * 4;
  const long long Mp = (M + 7) / 8 * 8;
  const long long tens = bf16 ? (N + K) * Mp * 2 + N * K * 4 : 0;
  return simt > tens ? simt : tens;
}

// dW[N,K] (fp32, row stride K) = alpha * G^T X + beta * dW ; G:[M,N] (ldg), X:[M,K] (ldx), both `bf16 ? bf16 : fp32`
int linear_bwd_weight(bool bf16, const void* G, const void* X, float* dW, void* ws, long long M, long long N, long long K,
                      long long ldg, long long ldx, float alpha, float beta, cudaStream_t stream) {
  PV_REQUIRE(M > 0 && N > 0 && K > 0, "empty problem");
  PV_REQUIRE(ws != nullptr, "workspace required (pv_linear_bwd_weight_ws_bytes)");
  const bool tensor = bf16 && M >= 512 && N >= 128 && K >= 128 && N % 8 == 0 && K % 4 == 0;
  if (tensor) {
    // G^T [N, Mp] and X^T [K, Mp] (bf16, zero-padded to a multiple of 8 rows), then one tcgen05 GEMM over K' = M
    const long long Mp = (M + 7) / 8 * 8;
    __nv_bfloat16* Gt = static_cast<__nv_bfloat16*>(ws);
    __nv_bfloat16* Xt = Gt + N * Mp;
    float* tmp = reinterpret_cast<float*>(Xt + K * Mp);
    dim3 g1((N + 31) / 32, (Mp + 31) / 32), g2((K + 31) / 32, (Mp + 31) / 32);
    transpose2d_kernel<__nv_bfloat16><<<g1, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(G), Gt, M, N, ldg, Mp);
    PV_LAUNCHED();
    transpose2d_kernel<__nv_bfloat16><<<g2, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(X), Xt, M, K, ldx, Mp);
    PV_LAUNCHED();
    const bool direct = (alpha == 1.f && beta == 0.f);
    int rc = gemm_bf16(Gt, Xt, nullptr, direct ? dW : tmp, true, N, K, Mp, 1, Mp, Mp, K, 0, 0, 0, 0, stream);
    if (rc) return rc;
    if (!direct) {
      const long long n = N * K;
      scale_copy_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(tmp, dW, n, alpha, beta);
      PV_LAUNCHED();
    }
    return PV_OK;
  }
  const long long splits = (M + WG_MCHUNK - 1) / WG_MCHUNK;
  PV_REQUIRE(splits <= 65535, "M too large");
  dim3 grid(static_cast<unsigned>((K + 63) / 64), static_cast<unsigned>((N + 63) / 64), static_cast<unsigned>(splits));
  float* part = static_cast<float*>(ws);
  if (bf16)
    wgrad_partial_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(G), static_cast<const __nv_bfloat16*>(X),
                                                                 part, M, (int)N, (int)K, ldg, ldx);
  else
    wgrad_partial_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(G), static_cast<const float*>(X), part, M, (int)N,
                                                         (int)K, ldg, ldx);
  PV_LAUNCHED();
  const long long n = N * K;
  reduce_partials_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(part, dW, n, (int)splits, alpha, beta);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// out[n] = sum_m G[m, n]   (bias gradients) -- two-pass
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
colsum_partial_kernel(const T* __restrict__ G, float* __restrict__ part, long long M, int N, long long ldg, int rows_per_block) {
  const int n = blockIdx.x * 256 + threadIdx.x;
  if (n >= N) return;
  const long long m0 = static_cast<long long>(blockIdx.y) * rows_per_block;
  const long long m1 = m0 + rows_per_block < M ? m0 + rows_per_block : M;
  float s = 0.f;
  for (long long m = m0; m < m1; ++m) s += ldf(G + m * ldg + n);
  part[static_cast<size_t>(blockIdx.y) * N + n] = s;
}

long long colsum_ws_bytes(long long M, long long N) { return ((M + 255) / 256) * N * 4; }

int col_sum(bool bf16, const void* G, float* out, void* ws, long long M, long long N, long long ldg, cudaStream_t stream) {
  PV_REQUIRE(M > 0 && N > 0 && ws != nullptr, "bad arguments");
  const int rpb = 256;
  const long long nb = (M + rpb - 1) / rpb;
  PV_REQUIRE(nb <= 65535, "M too large");
  dim3 grid(static_cast<unsigned>((N + 255) / 256), static_cast<unsigned>(nb));
  float* part = static_cast<float*>(ws);
  if (bf16) colsum_partial_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(G), part, M, (int)N, ldg, rpb);
  else colsum_partial_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(G), part, M, (int)N, ldg, rpb);
  PV_LAUNCHED();
  reduce_partials_kernel<<<static_cast<unsigned>((N + 255) / 256), 256, 0, stream>>>(part, out, N, (int)nb, 1.f, 0.f);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// LayerNorm(1024) + LeakyReLU backward (adapters.py:15-16, 18-19).  One warp per row, rows of a block strided.
//   xhat = (x - mean) rstd ; y = xhat g + b ; a = y > 0 ? y : slope y
//   gy = da (y > 0 ? 1 : slope) ; db += gy ; dg += gy xhat ; dxh = gy g
//   dx = rstd (dxh - mean(dxh) - xhat mean(dxh xhat))
// ------------------------------------------------------------------------------------------------
constexpr int LNB_ROWS = 64;     // rows per block

template <int NVEC, typename TD>
__global__ void __launch_bounds__(256)
ln_lrelu_bwd_kernel(const TD* __restrict__ da, const float* __restrict__ x, const float* __restrict__ mean,
                    const float* __restrict__ rstd, const float* __restrict__ gamma, const float* __restrict__ beta,
                    TD* __restrict__ dx, float* __restrict__ part, long long rows_per_group, int cols, float slope) {
  __shared__ float red[8][NVEC * 128];       // per-warp partial of one quantity at a time
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long grp = blockIdx.y;
  const long long r0 = static_cast<long long>(blockIdx.x) * LNB_ROWS;
  const float4* g4 = reinterpret_cast<const float4*>(gamma + grp * cols);
  const float4* b4 = reinterpret_cast<const float4*>(beta + grp * cols);
  float4 gv[NVEC], bv[NVEC], dg[NVEC], db[NVEC];
#pragma unroll
  for (int i = 0; i < NVEC; ++i) {
    gv[i] = g4[i * 32 + lane];
    bv[i] = b4[i * 32 + lane];
    dg[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    db[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int rr = warp; rr < LNB_ROWS; rr += 8) {
    const long long rg = r0 + rr;
    if (rg >= rows_per_group) break;
    const long long row = grp * rows_per_group + rg;
    const float mu = mean[row], rs = rstd[row];
    const float4* xr = reinterpret_cast<const float4*>(x + row * cols);
    float4 xh[NVEC], dh[NVEC];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < NVEC; ++i) {
      const float4 xv = xr[i * 32 + lane];
      float d[4];
      const TD* dap = da + row * cols + (i * 32 + lane) * 4;
#pragma unroll
      for (int k = 0; k < 4; ++k) d[k] = ldf(dap + k);
      const float xa[4] = {(xv.x - mu) * rs, (xv.y - mu) * rs, (xv.z - mu) * rs, (xv.w - mu) * rs};
      const float ga[4] = {gv[i].x, gv[i].y, gv[i].z, gv[i].w};
      const float ba[4] = {bv[i].x, bv[i].y, bv[i].z, bv[i].w};
      float gy[4], dxh[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float y = fmaf(xa[k], ga[k], ba[k]);
        gy[k] = d[k] * (y > 0.f ? 1.f : slope);
        dxh[k] = gy[k] * ga[k];
        s1 += dxh[k];
        s2 = fmaf(dxh[k], xa[k], s2);
      }
      db[i].x += gy[0]; db[i].y += gy[1]; db[i].z += gy[2]; db[i].w += gy[3];
      dg[i].x = fmaf(gy[0], xa[0], dg[i].x); dg[i].y = fmaf(gy[1], xa[1], dg[i].y);
      dg[i].z = fmaf(gy[2], xa[2], dg[i].z); dg[i].w = fmaf(gy[3], xa[3], dg[i].w);
      xh[i] = make_float4(xa[0], xa[1], xa[2], xa[3]);
      dh[i] = make_float4(dxh[0], dxh[1], dxh[2], dxh[3]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1 += __shfl_xor_sync(0xffffffffu, s1, o);
      s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    const float m1 = s1 / static_cast<float>(cols), m2 = s2 / static_cast<float>(cols);
#pragma unroll
    for (int i = 0; i < NVEC; ++i) {
      TD* dxp = dx + row * cols + (i * 32 + lane) * 4;
      stf(dxp + 0, rs * (dh[i].x - m1 - xh[i].x * m2));
      stf(dxp + 1, rs * (dh[i].y - m1 - xh[i].y * m2));
      stf(dxp + 2, rs * (dh[i].z - m1 - xh[i].z * m2));
      stf(dxp + 3, rs * (dh[i].w - m1 - xh[i].w * m2));
    }
  }
  // block reduction of dgamma / dbeta over the 8 warps (fixed order), one partial row per block
  float* pg = part + ((grp * gridDim.x + blockIdx.x) * 2) * cols;
  for (int pass = 0; pass < 2; ++pass) {
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NVEC; ++i) {
      const float4 v = pass == 0 ? dg[i] : db[i];
      *reinterpret_cast<float4*>(&red[warp][(i * 32 + lane) * 4]) = v;
    }
    __syncthreads();
    for (int c = threadIdx.x; c < cols; c += 256) {
      float s = 0.f;
#pragma unroll
      for (int w = 0; w < 8; ++w) s += red[w][c];
      pg[pass * cols + c] = s;
    }
  }
}

// out[grp][q][c] = sum over the blocks of group grp   (q: 0 dgamma, 1 dbeta)
__global__ void __launch_bounds__(256)
ln_reduce_kernel(const float* __restrict__ part, float* __restrict__ dgamma, float* __restrict__ dbeta, int nblk, int cols) {
  const int grp = blockIdx.y;
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= cols) return;
  float sg = 0.f, sb = 0.f;
  for (int b = 0; b < nblk; ++b) {
    const float* p = part + ((static_cast<size_t>(grp) * nblk + b) * 2) * cols;
    sg += p[c];
    sb += p[cols + c];
  }
  dgamma[static_cast<size_t>(grp) * cols + c] = sg;
  dbeta[static_cast<size_t>(grp) * cols + c] = sb;
}

long long ln_bwd_ws_bytes(long long groups, long long rows_per_group, int cols) {
  return groups * ((rows_per_group + LNB_ROWS - 1) / LNB_ROWS) * 2 * cols * 4;
}

int ln_lrelu_bwd(bool bf16, const void* da, const float* x, const float* mean, const float* rstd, const float* gamma,
                 const float* beta, void* dx, float* dgamma, float* dbeta, void* ws, long long groups,
                 long long rows_per_group, int cols, float slope, cudaStream_t stream) {
  PV_REQUIRE(groups > 0 && groups <= 65535 && rows_per_group > 0 && cols == 1024, "ln_lrelu_bwd: cols must be 1024 (adapter width), got %d", cols);
  const int nblk = static_cast<int>((rows_per_group + LNB_ROWS - 1) / LNB_ROWS);
  dim3 grid(nblk, static_cast<unsigned>(groups));
  float* part = static_cast<float*>(ws);
  if (bf16)
    ln_lrelu_bwd_kernel<8, __nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(da), x, mean, rstd, gamma, beta,
                                                                  static_cast<__nv_bfloat16*>(dx), part, rows_per_group, cols, slope);
  else
    ln_lrelu_bwd_kernel<8, float><<<grid, 256, 0, stream>>>(static_cast<const float*>(da), x, mean, rstd, gamma, beta,
                                                          static_cast<float*>(dx), part, rows_per_group, cols, slope);
  PV_LAUNCHED();
  dim3 g2((cols + 255) / 256, static_cast<unsigned>(groups));
  ln_reduce_kernel<<<g2, 256, 0, stream>>>(part, dgamma, dbeta, nblk, cols);
  PV_LAUNCHED();
  return PV_OK;
}

// dx[g, p, :] = dy[g, :] / P
template <typename T>
__global__ void __launch_bounds__(256)
group_mean_bwd_kernel(const T* __restrict__ dy, T* __restrict__ dx, int P, int cols, long long ldy) {
  const long long g = blockIdx.y;
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= cols) return;
  const float v = ldf(dy + g * ldy + c) / static_cast<float>(P);
  T* o = dx + g * P * cols + c;
  for (int r = 0; r < P; ++r) stf(o + static_cast<long long>(r) * cols, v);
}

int group_mean_bwd(bool bf16, const void* dy, void* dx, long long groups, int P, int cols, long long ldy, cudaStream_t stream) {
  PV_REQUIRE(groups > 0 && groups <= 65535 && P > 0 && cols > 0, "bad shape");
  dim3 grid((cols + 255) / 256, static_cast<unsigned>(groups));
  if (bf16) group_mean_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(dy), static_cast<__nv_bfloat16*>(dx), P, cols, ldy);
  else group_mean_bwd_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(dy), static_cast<float*>(dx), P, cols, ldy);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// Dual-branch attention backward core.
//   inputs : dO, Q [B,S,C] (T) ; K/V fp32 projections kv_text [B*Lt, 2C], kv_img [B*Li, 2C] (cols [0,C) = K, [C,2C) = V) ;
//            stats [B,H,S,4] = (m_text, l_text, m_img, l_img) of the scaled (log2) logits, from the forward kernel
//   outputs: dQ [B,S,C] (T) ; part [nchunk][B][H][2][L][d] fp32 partial dK / dV of each query chunk
//   p^ = 2^(s cs - m)/l per segment ; O = sum_seg w_seg sum_k p^_k V_k
//   dp_k = dO.V_k ; delta_seg = sum_{k in seg} p^_k dp_k ; ds_k = w_seg p^_k (dp_k - delta_seg)
//   dQ = scale sum_k ds_k K_k ; dK_k = scale sum_q ds_k Q_q ; dV_k = sum_q w_seg p^_k dO_q
// block = (query chunk, head, sample), 256 threads; dK / dV of the chunk accumulate in registers.
// ------------------------------------------------------------------------------------------------
constexpr int AB_TQ = 32;         // queries per tile
constexpr int AB_CHUNK = 128;     // queries per block (== the row tile of the tensor-core kernel in pv_bwd_mma.cu)
constexpr int AB_LP = PV_KEYS_PAD + 1;

// MASK: the image keys of query row s are weighted w_img * img_row_weight[b, s] (ip_adapter_masks)
template <int D, typename T, bool MASK>
__global__ void __launch_bounds__(256, 1)
attn_bwd_kernel(const T* __restrict__ dO, const T* __restrict__ Q, const float* __restrict__ kv_text,
                const float* __restrict__ kv_img, const float* __restrict__ stats, T* __restrict__ dQ,
                float* __restrict__ part, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                float scale, float scale_log2e, const float* __restrict__ img_row_weight) {
  constexpr int DP = D + 1;
  constexpr int R = (PV_KEYS_PAD * D + 255) / 256;
  extern __shared__ float sm[];
  const int L = Lt + Li;
  float* Ks = sm;                         // [L][DP]
  float* Vs = Ks + PV_KEYS_PAD * DP;      // [L][DP]
  float* qs = Vs + PV_KEYS_PAD * DP;      // [TQ][DP]
  float* dos = qs + AB_TQ * DP;           // [TQ][DP]
  float* ps = dos + AB_TQ * DP;           // [TQ][LP]  w_seg p^
  float* dss = ps + AB_TQ * AB_LP;        // [TQ][LP]  scale * ds
  const int chunk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int C2 = 2 * C;
  for (int i = threadIdx.x; i < L * D; i += 256) {
    const int k = i / D, c = i - k * D;
    const float* src = (k < Lt) ? kv_text + (static_cast<size_t>(b) * Lt + k) * C2 : kv_img + (static_cast<size_t>(b) * Li + (k - Lt)) * C2;
    Ks[k * DP + c] = src[h * D + c];
    Vs[k * DP + c] = src[C + h * D + c];
  }
  float accK[R], accV[R];
#pragma unroll
  for (int r = 0; r < R; ++r) { accK[r] = 0.f; accV[r] = 0.f; }
  const int q_begin = chunk * AB_CHUNK;
  const int q_end = q_begin + AB_CHUNK < S ? q_begin + AB_CHUNK : S;
  for (int q0 = q_begin; q0 < q_end; q0 += AB_TQ) {
    __syncthreads();
    for (int i = threadIdx.x; i < AB_TQ * D; i += 256) {
      const int rr = i / D, c = i - rr * D;
      const int srow = q0 + rr;
      float qv = 0.f, dv = 0.f;
      if (srow < q_end) {
        const size_t off = (static_cast<size_t>(b) * S + srow) * C + h * D + c;
        qv = ldf(Q + off);
        dv = ldf(dO + off);
      }
      qs[rr * DP + c] = qv;
      dos[rr * DP + c] = dv;
    }
    __syncthreads();
    // ---- per query row: p^, dp, delta, ds ----
    for (int rr = warp; rr < AB_TQ; rr += 8) {
      const int srow = q0 + rr;
      float pw[3], dsv[3];
      if (srow < q_end) {
        const float4 st = reinterpret_cast<const float4*>(stats)[(static_cast<size_t>(b) * H + h) * S + srow];
        const float* qr = qs + rr * DP;
        const float* dr = dos + rr * DP;
        float ph[3], dp[3];
        float delt = 0.f, deli = 0.f;
        const float wi = MASK ? w_img * __ldg(img_row_weight + static_cast<size_t>(b) * S + srow) : w_img;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          const int k = lane + 32 * t;
          ph[t] = 0.f; dp[t] = 0.f;
          if (k < L) {
            const float* kr = Ks + k * DP;
            const float* vr = Vs + k * DP;
            float s = 0.f, d = 0.f;
            for (int c = 0; c < D; ++c) { s = fmaf(qr[c], kr[c], s); d = fmaf(dr[c], vr[c], d); }
            const bool is_t = k < Lt;
            ph[t] = exp2f(fmaf(s, scale_log2e, -(is_t ? st.x : st.z))) / (is_t ? st.y : st.w);
            dp[t] = d;
            if (is_t) delt = fmaf(ph[t], d, delt); else deli = fmaf(ph[t], d, deli);
          }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          delt += __shfl_xor_sync(0xffffffffu, delt, o);
          deli += __shfl_xor_sync(0xffffffffu, deli, o);
        }
#pragma unroll
        for (int t = 0; t < 3; ++t) {
          const int k = lane + 32 * t;
          const bool is_t = k < Lt;
          const float w = is_t ? w_text : wi;
          pw[t] = w * ph[t];
          dsv[t] = scale * w * ph[t] * (dp[t] - (is_t ? delt : deli));
        }
      } else {
#pragma unroll
        for (int t = 0; t < 3; ++t) { pw[t] = 0.f; dsv[t] = 0.f; }
      }
#pragma unroll
      for (int t = 0; t < 3; ++t) {
        const int k = lane + 32 * t;
        if (k < PV_KEYS_PAD) { ps[rr * AB_LP + k] = pw[t]; dss[rr * AB_LP + k] = dsv[t]; }
      }
    }
    __syncthreads();
    // ---- dQ tile ----
    for (int i = threadIdx.x; i < AB_TQ * D; i += 256) {
      const int rr = i / D, c = i - rr * D;
      const int srow = q0 + rr;
      if (srow >= q_end) continue;
      const float* dr = dss + rr * AB_LP;
      float a = 0.f;
      for (int k = 0; k < L; ++k) a = fmaf(dr[k], Ks[k * DP + c], a);
      stf(dQ + (static_cast<size_t>(b) * S + srow) * C + h * D + c, a);
    }
    // ---- dK / dV accumulation (registers) ----
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int e = threadIdx.x + 256 * r;
      if (e < L * D) {
        const int k = e / D, c = e - k * D;
        float ak = accK[r], av = accV[r];
#pragma unroll 8
        for (int rr = 0; rr < AB_TQ; ++rr) {
          ak = fmaf(dss[rr * AB_LP + k], qs[rr * DP + c], ak);
          av = fmaf(ps[rr * AB_LP + k], dos[rr * DP + c], av);
        }
        accK[r] = ak; accV[r] = av;
      }
    }
  }
  float* dst = part + ((static_cast<size_t>(chunk) * B + b) * H + h) * 2 * L * D;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int e = threadIdx.x + 256 * r;
    if (e < L * D) { dst[e] = accK[r]; dst[L * D + e] = accV[r]; }
  }
}

int attn_bwd_mma_chunks(int S, int d);
extern int g_opt_bwd_mma;
// Query-row chunks whose dK / dV partials kv_bwd_reduce sums: 128-row blocks of the SIMT kernel, or the (longer) blocks of
// the tensor-core kernel.  The workspace is sized for the finer split.
int attn_bwd_chunks(int S) { return (S + AB_CHUNK - 1) / AB_CHUNK; }
int attn_bwd_chunks_used(bool bf16, int S, int d) {
  return (bf16 && g_opt_bwd_mma != 0) ? attn_bwd_mma_chunks(S, d) : attn_bwd_chunks(S);
}

template <int D, typename T>
static int launch_attn_bwd(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats,
                           void* dQ, float* part, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                           cudaStream_t stream, const float* img_row_weight) {
  auto kern = img_row_weight ? attn_bwd_kernel<D, T, true> : attn_bwd_kernel<D, T, false>;
  const size_t smem = (2 * PV_KEYS_PAD * (D + 1) + 2 * AB_TQ * (D + 1) + 2 * AB_TQ * AB_LP) * sizeof(float);
  PV_CUDA(set_max_smem_once(kern, static_cast<int>(smem)));
  dim3 grid(attn_bwd_chunks(S), H, B);
  const float scale = 1.f / sqrtf(static_cast<float>(D));
  kern<<<grid, 256, smem, stream>>>(static_cast<const T*>(dO), static_cast<const T*>(Q), kv_text, kv_img, stats,
                                    static_cast<T*>(dQ), part, B, S, C, H, Lt, Li, w_text, w_img, scale,
                                    scale * 1.4426950408889634f, img_row_weight);
  PV_LAUNCHED();
  return PV_OK;
}

int dual_attn_bwd_mma(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats, void* dQ,
                      float* part, int nchunk, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                      cudaStream_t stream, const float* img_row_weight);

// img_row_weight: optional [B, S] fp32 factor of each query row's image keys (nullptr: the unmasked kernels)
int dual_attn_bwd(bool bf16, const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats,
                  void* dQ, float* part, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                  cudaStream_t stream, const float* img_row_weight) {
  PV_REQUIRE(B > 0 && S > 0 && H > 0 && C % H == 0 && B <= 65535 && H <= 65535, "bad shape");
  PV_REQUIRE(Lt >= 1 && Li >= 1 && Lt + Li <= PV_KEYS_PAD, "need 1 <= Lt, 1 <= Li, Lt+Li <= %d", PV_KEYS_PAD);
  const int d = C / H;
  if (bf16 && g_opt_bwd_mma != 0)       // tensor-core kernel (pv_bwd_mma.cu); the SIMT kernel below is the fp32 parity path
    return dual_attn_bwd_mma(dO, Q, kv_text, kv_img, stats, dQ, part, attn_bwd_mma_chunks(S, d), B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
#define PV_AB(DD)                                                                                                        \
  return bf16 ? launch_attn_bwd<DD, __nv_bfloat16>(dO, Q, kv_text, kv_img, stats, dQ, part, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight) \
              : launch_attn_bwd<DD, float>(dO, Q, kv_text, kv_img, stats, dQ, part, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight)
  switch (d) {
    case 40: PV_AB(40);
    case 80: PV_AB(80);
    case 160: PV_AB(160);
    default: PV_FAIL(PV_ERR_UNSUPPORTED, "head_dim %d unsupported (40/80/160)", d);
  }
#undef PV_AB
}

// ------------------------------------------------------------------------------------------------
// Reduce the per-chunk dK / dV partials, add the backward of the `to_v_ip_norm` side output
// (d||V|| = V / ||V||, attention_processor.py:397 + models/unet.py:38-47) and scatter into the projection layout:
//   dkv_text [B*Lt, 2C], dkv_img [B*Li, 2C]   (T; columns [0,C) = dK, [C,2C) = dV)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
kv_bwd_reduce_kernel(const float* __restrict__ part, const float* __restrict__ kv_img, const float* __restrict__ v_ip_norm,
                     const float* __restrict__ d_vnorm, T* __restrict__ dkv_text, T* __restrict__ dkv_img, int nchunk,
                     int B, int H, int Lt, int Li, int C, int d) {
  const int L = Lt + Li;
  const int key = blockIdx.x, b = blockIdx.y;
  const int C2 = 2 * C;
  for (int col = threadIdx.x; col < C2; col += 256) {
    const int which = col >= C;                 // 0: dK, 1: dV
    const int cc = col - which * C;
    const int h = cc / d, c = cc - h * d;
    float s = 0.f;
    for (int z = 0; z < nchunk; ++z)
      s += part[(((static_cast<size_t>(z) * B + b) * H + h) * 2 + which) * L * d + static_cast<size_t>(key) * d + c];
    if (key < Lt) {
      stf(dkv_text + (static_cast<size_t>(b) * Lt + key) * C2 + col, s);
    } else {
      const int li = key - Lt;
      if (which == 1 && d_vnorm != nullptr) {
        const size_t ni = (static_cast<size_t>(b) * H + h) * Li + li;
        const float vn = v_ip_norm[ni];
        if (vn > 0.f) s = fmaf(d_vnorm[ni] / vn, kv_img[(static_cast<size_t>(b) * Li + li) * C2 + col], s);
      }
      stf(dkv_img + (static_cast<size_t>(b) * Li + li) * C2 + col, s);
    }
  }
}

int kv_pack_bwd(bool bf16, const float* part, const float* kv_img, const float* v_ip_norm, const float* d_vnorm,
                void* dkv_text, void* dkv_img, int nchunk, int B, int Lt, int Li, int C, int H, cudaStream_t stream) {
  PV_REQUIRE(B > 0 && B <= 65535 && nchunk > 0 && C % H == 0, "bad shape");
  dim3 grid(Lt + Li, B);
  const int d = C / H;
  if (bf16)
    kv_bwd_reduce_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(part, kv_img, v_ip_norm, d_vnorm, static_cast<__nv_bfloat16*>(dkv_text),
                                                                 static_cast<__nv_bfloat16*>(dkv_img), nchunk, B, H, Lt, Li, C, d);
  else
    kv_bwd_reduce_kernel<float><<<grid, 256, 0, stream>>>(part, kv_img, v_ip_norm, d_vnorm, static_cast<float*>(dkv_text),
                                                         static_cast<float*>(dkv_img), nchunk, B, H, Lt, Li, C, d);
  PV_LAUNCHED();
  return PV_OK;
}

}  // namespace pv
