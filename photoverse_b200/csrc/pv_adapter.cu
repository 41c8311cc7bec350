// photoverse_b200 -- adapter MLP epilogues (reference models/adapters.py:15-16, 18-19, 36, 41).
//
//  * ln_lrelu   : y = LeakyReLU(LayerNorm(x) * gamma + beta) -- one warp per row, 16-byte vector loads,
//                 warp-shuffle reductions, two-pass variance in registers (HBM-bound: 4 B in, 2 B out per element)
//                 (16-bit inputs / outputs: bf16 or fp16; a mixed bf16 / fp16 pair is rejected by the C ABI)
//  * group_mean : mean over the 256 patch tokens of each (head, sample) -- commuted in front of the last Linear
#include "pv_common.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int LN_MAX_VEC = 32;   // float4 per lane -> cols <= 4096

// OUT16: 16-bit output of type T16 (__nv_bfloat16 or __half), else fp32
template <int NVEC, bool OUT16, typename T16>
__global__ void __launch_bounds__(256)
ln_lrelu_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                void* __restrict__ y, float* __restrict__ save_mean, float* __restrict__ save_rstd, long long rows,
                int cols, long long ldx, long long ldy, long long rows_per_group, float eps, float slope) {
  const long long row = static_cast<long long>(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const float4* xr = reinterpret_cast<const float4*>(x + row * ldx);
  float4 v[NVEC];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NVEC; ++i) {
    v[i] = xr[i * 32 + lane];
    s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / static_cast<float>(cols);
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < NVEC; ++i) {
    const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
    ss += (a * a + b * b) + (c * c + d * d);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = rsqrtf(ss / static_cast<float>(cols) + eps);
  if (lane == 0) {
    if (save_mean) save_mean[row] = mean;
    if (save_rstd) save_rstd[row] = rstd;
  }
  const long long grp = rows_per_group > 0 ? row / rows_per_group : 0;
  const float4* g4 = reinterpret_cast<const float4*>(gamma + grp * cols);
  const float4* b4 = reinterpret_cast<const float4*>(beta + grp * cols);
#pragma unroll
  for (int i = 0; i < NVEC; ++i) {
    const float4 g = __ldg(g4 + i * 32 + lane), bt = __ldg(b4 + i * 32 + lane);
    float o0 = fmaf((v[i].x - mean) * rstd, g.x, bt.x);
    float o1 = fmaf((v[i].y - mean) * rstd, g.y, bt.y);
    float o2 = fmaf((v[i].z - mean) * rstd, g.z, bt.z);
    float o3 = fmaf((v[i].w - mean) * rstd, g.w, bt.w);
    o0 = o0 > 0.f ? o0 : o0 * slope;
    o1 = o1 > 0.f ? o1 : o1 * slope;
    o2 = o2 > 0.f ? o2 : o2 * slope;
    o3 = o3 > 0.f ? o3 : o3 * slope;
    if constexpr (OUT16) {
      uint2* yr = reinterpret_cast<uint2*>(static_cast<T16*>(y) + row * ldy);
      yr[i * 32 + lane] = make_uint2(pack_x2<T16>(o0, o1), pack_x2<T16>(o2, o3));
    } else {
      float4* yr = reinterpret_cast<float4*>(static_cast<float*>(y) + row * ldy);
      yr[i * 32 + lane] = make_float4(o0, o1, o2, o3);
    }
  }
}

template <int NVEC>
static int launch_ln(pv_dtype out_dt, const float* x, const float* gamma, const float* beta, void* y, float* sm,
                     float* sr, long long rows, int cols, long long ldx, long long ldy, long long rpg, float eps,
                     float slope, cudaStream_t stream) {
  const int blocks = static_cast<int>((rows + 7) / 8);
  auto kern = out_dt == PV_BF16 ? ln_lrelu_kernel<NVEC, true, __nv_bfloat16>
               : out_dt == PV_F16 ? ln_lrelu_kernel<NVEC, true, __half> : ln_lrelu_kernel<NVEC, false, __nv_bfloat16>;
  kern<<<blocks, 256, 0, stream>>>(x, gamma, beta, y, sm, sr, rows, cols, ldx, ldy, rpg, eps, slope);
  PV_LAUNCHED();
  return PV_OK;
}

int ln_lrelu(pv_dtype out_dt, const float* x, const float* gamma, const float* beta, void* y, float* save_mean,
             float* save_rstd, long long rows, int cols, long long ldx, long long ldy, long long rows_per_group,
             float eps, float slope, cudaStream_t stream) {
  PV_REQUIRE(rows > 0 && cols > 0 && cols % 128 == 0 && cols / 128 <= LN_MAX_VEC, "cols=%d must be a multiple of 128, <= 4096", cols);
  PV_REQUIRE(ldx % 4 == 0 && ldy % 4 == 0, "row strides must be multiples of 4 elements");
  PV_REQUIRE((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y) | reinterpret_cast<uintptr_t>(gamma) |
              reinterpret_cast<uintptr_t>(beta)) % 16 == 0, "pointers must be 16-byte aligned");
  switch (cols / 128) {
    case 8: return launch_ln<8>(out_dt, x, gamma, beta, y, save_mean, save_rstd, rows, cols, ldx, ldy, rows_per_group, eps, slope, stream);
    case 6: return launch_ln<6>(out_dt, x, gamma, beta, y, save_mean, save_rstd, rows, cols, ldx, ldy, rows_per_group, eps, slope, stream);
    case 4: return launch_ln<4>(out_dt, x, gamma, beta, y, save_mean, save_rstd, rows, cols, ldx, ldy, rows_per_group, eps, slope, stream);
    case 2: return launch_ln<2>(out_dt, x, gamma, beta, y, save_mean, save_rstd, rows, cols, ldx, ldy, rows_per_group, eps, slope, stream);
    case 1: return launch_ln<1>(out_dt, x, gamma, beta, y, save_mean, save_rstd, rows, cols, ldx, ldy, rows_per_group, eps, slope, stream);
    default: PV_FAIL(PV_ERR_UNSUPPORTED, "cols=%d not instantiated (128/256/512/768/1024)", cols);
  }
}

// x:[groups, P, cols] -> y:[groups, cols].  A block owns 64 adjacent columns of one group: lane = 2 columns (one 4- / 8-byte
// load, 128 / 256 contiguous bytes per warp and row), its 8 warps take the rows w, w + 8, ... with four independent
// accumulator pairs (loads in flight instead of one serial chain of P round trips), and warp 0 adds the 8 slice sums in a
// fixed order.  HBM-bound: x is read once.
// IN16 / OUT16: 16-bit input / output of type T16 (__nv_bfloat16 or __half), else fp32
template <bool IN16, bool OUT16, typename T16>
__global__ void __launch_bounds__(256)
group_mean_kernel(const void* __restrict__ x, void* __restrict__ y, int P, int cols, long long ldy) {
  __shared__ float red[8][64];
  const long long g = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * 64 + lane * 2;
  float a[4][2] = {};
  if (c < cols) {
    auto ld = [&](int r, float& v0, float& v1) {
      if constexpr (IN16 && std::is_same<T16, __half>::value) {
        const float2 f = __half22float2(*reinterpret_cast<const __half2*>(
            static_cast<const __half*>(x) + (g * P + r) * static_cast<long long>(cols) + c));
        v0 = f.x; v1 = f.y;
      } else if constexpr (IN16) {
        const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(
            static_cast<const __nv_bfloat16*>(x) + (g * P + r) * static_cast<long long>(cols) + c));
        v0 = f.x; v1 = f.y;
      } else {
        const float2 f = *reinterpret_cast<const float2*>(static_cast<const float*>(x) + (g * P + r) * static_cast<long long>(cols) + c);
        v0 = f.x; v1 = f.y;
      }
    };
    int r = warp;
    for (; r + 24 < P; r += 32) {
      float v[4][2];
#pragma unroll
      for (int k = 0; k < 4; ++k) ld(r + 8 * k, v[k][0], v[k][1]);
#pragma unroll
      for (int k = 0; k < 4; ++k) { a[k][0] += v[k][0]; a[k][1] += v[k][1]; }
    }
    for (; r < P; r += 8) {
      float v0, v1;
      ld(r, v0, v1);
      a[0][0] += v0; a[0][1] += v1;
    }
  }
  red[warp][2 * lane] = (a[0][0] + a[1][0]) + (a[2][0] + a[3][0]);
  red[warp][2 * lane + 1] = (a[0][1] + a[1][1]) + (a[2][1] + a[3][1]);
  __syncthreads();
  if (warp == 0 && c < cols) {
    float s0 = red[0][2 * lane], s1 = red[0][2 * lane + 1];
#pragma unroll
    for (int w = 1; w < 8; ++w) { s0 += red[w][2 * lane]; s1 += red[w][2 * lane + 1]; }
    const float inv = 1.f / static_cast<float>(P);
    s0 *= inv; s1 *= inv;
    if constexpr (OUT16) {
      *reinterpret_cast<uint32_t*>(static_cast<T16*>(y) + g * ldy + c) = pack_x2<T16>(s0, s1);
    } else {
      *reinterpret_cast<float2*>(static_cast<float*>(y) + g * ldy + c) = make_float2(s0, s1);
    }
  }
}

int group_mean(pv_dtype in_dt, pv_dtype out_dt, const void* x, void* y, long long groups, int P, int cols, long long ldy,
               cudaStream_t stream) {
  PV_REQUIRE(groups > 0 && groups <= 65535 && P > 0 && cols > 0 && cols % 2 == 0 && ldy % 2 == 0, "bad shape");
  dim3 grid((cols + 63) / 64, static_cast<unsigned>(groups));
  const bool in16 = in_dt != PV_F32, out16 = out_dt != PV_F32;
  if (in_dt == PV_F16 || out_dt == PV_F16) {
    if (in16 && out16) group_mean_kernel<true, true, __half><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
    else if (in16) group_mean_kernel<true, false, __half><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
    else group_mean_kernel<false, true, __half><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
  } else if (in16 && out16) group_mean_kernel<true, true, __nv_bfloat16><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
  else if (in16) group_mean_kernel<true, false, __nv_bfloat16><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
  else if (out16) group_mean_kernel<false, true, __nv_bfloat16><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
  else group_mean_kernel<false, false, __nv_bfloat16><<<grid, 256, 0, stream>>>(x, y, P, cols, ldy);
  PV_LAUNCHED();
  return PV_OK;
}

}  // namespace pv
