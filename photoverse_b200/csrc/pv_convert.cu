// photoverse_b200 -- dtype conversion of activations (pv_convert_fwd): float32 <-> bfloat16 / float16.
//
// Under torch.autocast a float32 model hands the processor and the adapters float32 activations while the compute dtype is
// 16-bit (DESIGN.md 4.9); this kernel is the one place where such an activation enters (and its gradient leaves) the 16-bit
// path.  Memory-bound: every thread keeps CV_UNROLL vectors of 8 elements in flight, each a 32-byte fp32 access and a 16-byte
// 16-bit access (LDG/STG .256 and .128).  Rounding is to nearest even (__float2bfloat16_rn / __float2half_rn): bit-identical
// to torch.Tensor.to for every finite input, fp16 overflow becomes +-inf, NaN stays NaN.  Leading elements up to the first
// vector boundary of both pointers and the last n % 8 elements are converted one by one; pointers whose element offsets
// differ modulo 8 take the scalar loop throughout.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int CV_THREADS = 256;
constexpr int CV_UNROLL = 4;

template <typename T> __device__ __forceinline__ T cv_from_f32(float x);
template <> __device__ __forceinline__ __nv_bfloat16 cv_from_f32<__nv_bfloat16>(float x) { return __float2bfloat16_rn(x); }
template <> __device__ __forceinline__ __half cv_from_f32<__half>(float x) { return __float2half_rn(x); }
__device__ __forceinline__ float cv_to_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float cv_to_f32(__half x) { return __half2float(x); }

__device__ __forceinline__ uint32_t cv_pack2(float a, float b, __nv_bfloat16*) {
  const __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&p);
}
__device__ __forceinline__ uint32_t cv_pack2(float a, float b, __half*) {
  const __half2 p = __floats2half2_rn(a, b);
  return *reinterpret_cast<const uint32_t*>(&p);
}
__device__ __forceinline__ float2 cv_unpack2(uint32_t w, __nv_bfloat16*) {
  return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xffff0000u));
}
__device__ __forceinline__ float2 cv_unpack2(uint32_t w, __half*) {
  return __half22float2(*reinterpret_cast<const __half2*>(&w));
}

struct F32x8 { float v[8]; };

__device__ __forceinline__ F32x8 ld_f32x8(const float* p) {
  F32x8 r;
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_f32x8(float* p, const F32x8& r) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]),
               "f"(r.v[3]), "f"(r.v[4]), "f"(r.v[5]), "f"(r.v[6]), "f"(r.v[7])
               : "memory");
}

// fp32 -> 16-bit.  Elements [0, head) and [head + 8 * nvec, n) scalar, the vectors in between vectorised.
template <typename T>
__global__ void __launch_bounds__(CV_THREADS) convert_from_f32_kernel(const float* __restrict__ src, T* __restrict__ dst,
                                                                      long long n, long long head, long long nvec) {
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long nthr = static_cast<long long>(gridDim.x) * blockDim.x;
  const float* vs = src + head;
  uint4* vd = reinterpret_cast<uint4*>(dst + head);
  for (long long base = tid; base < nvec; base += nthr * CV_UNROLL) {
    F32x8 r[CV_UNROLL];
#pragma unroll
    for (int u = 0; u < CV_UNROLL; ++u) {
      const long long i = base + u * nthr;
      if (i < nvec) r[u] = ld_f32x8(vs + 8 * i);
    }
#pragma unroll
    for (int u = 0; u < CV_UNROLL; ++u) {
      const long long i = base + u * nthr;
      if (i < nvec)
        vd[i] = make_uint4(cv_pack2(r[u].v[0], r[u].v[1], (T*)nullptr), cv_pack2(r[u].v[2], r[u].v[3], (T*)nullptr),
                           cv_pack2(r[u].v[4], r[u].v[5], (T*)nullptr), cv_pack2(r[u].v[6], r[u].v[7], (T*)nullptr));
    }
  }
  const long long tail0 = head + 8 * nvec;
  for (long long i = tid; i < head + (n - tail0); i += nthr) {
    const long long j = i < head ? i : tail0 + (i - head);
    dst[j] = cv_from_f32<T>(src[j]);
  }
}

// 16-bit -> fp32 (exact).  Same split as above.
template <typename T>
__global__ void __launch_bounds__(CV_THREADS) convert_to_f32_kernel(const T* __restrict__ src, float* __restrict__ dst,
                                                                    long long n, long long head, long long nvec) {
  const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long long nthr = static_cast<long long>(gridDim.x) * blockDim.x;
  const uint4* vs = reinterpret_cast<const uint4*>(src + head);
  float* vd = dst + head;
  for (long long base = tid; base < nvec; base += nthr * CV_UNROLL) {
    uint4 r[CV_UNROLL];
#pragma unroll
    for (int u = 0; u < CV_UNROLL; ++u) {
      const long long i = base + u * nthr;
      if (i < nvec) r[u] = __ldg(vs + i);
    }
#pragma unroll
    for (int u = 0; u < CV_UNROLL; ++u) {
      const long long i = base + u * nthr;
      if (i < nvec) {
        const uint32_t w[4] = {r[u].x, r[u].y, r[u].z, r[u].w};
        F32x8 o;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 f = cv_unpack2(w[k], (T*)nullptr);
          o.v[2 * k] = f.x;
          o.v[2 * k + 1] = f.y;
        }
        st_f32x8(vd + 8 * i, o);
      }
    }
  }
  const long long tail0 = head + 8 * nvec;
  for (long long i = tid; i < head + (n - tail0); i += nthr) {
    const long long j = i < head ? i : tail0 + (i - head);
    dst[j] = cv_to_f32(src[j]);
  }
}

static const char* dtype_name(pv_dtype dt) {
  switch (dt) {
    case PV_F32: return "PV_F32";
    case PV_BF16: return "PV_BF16";
    case PV_F16: return "PV_F16";
    default: return "an unknown pv_dtype";
  }
}

}  // namespace pv

using namespace pv;

extern "C" int pv_convert_fwd(pv_dtype in_dt, pv_dtype out_dt, const void* src, void* dst, int64_t n, void* stream) {
  const bool from_f32 = in_dt == PV_F32 && (out_dt == PV_BF16 || out_dt == PV_F16);
  const bool to_f32 = out_dt == PV_F32 && (in_dt == PV_BF16 || in_dt == PV_F16);
  if (!from_f32 && !to_f32)
    PV_FAIL(PV_ERR_UNSUPPORTED, "%s -> %s is not supported (supported: PV_F32 -> PV_BF16 | PV_F16 and back)",
            dtype_name(in_dt), dtype_name(out_dt));
  PV_REQUIRE(n >= 0, "n must be >= 0 (got %lld)", static_cast<long long>(n));
  if (n == 0) return PV_OK;
  PV_REQUIRE(src && dst, "null pointer");
  const uintptr_t p32 = reinterpret_cast<uintptr_t>(from_f32 ? src : dst);
  const uintptr_t p16 = reinterpret_cast<uintptr_t>(from_f32 ? dst : src);
  PV_REQUIRE(p32 % 4 == 0 && p16 % 2 == 0, "pointers must be aligned to their element size");
  // vectors start where both pointers sit on a vector boundary (32 bytes of fp32, 16 bytes of 16-bit elements)
  long long head = 0, nvec = 0;
  const long long a32 = static_cast<long long>((p32 / 4) % 8), a16 = static_cast<long long>((p16 / 2) % 8);
  if (a32 == a16) {
    head = (8 - a32) % 8;
    if (head > n) head = n;
    nvec = (n - head) / 8;
  } else {
    head = n;
  }
  const long long work = nvec > 0 ? (nvec + CV_UNROLL - 1) / CV_UNROLL : (n - 8 * nvec);
  long long blocks = (work + CV_THREADS - 1) / CV_THREADS;
  const long long cap = 8ll * sm_count();
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const unsigned g = static_cast<unsigned>(blocks);
  if (from_f32) {
    if (out_dt == PV_BF16)
      convert_from_f32_kernel<<<g, CV_THREADS, 0, s>>>(static_cast<const float*>(src), static_cast<__nv_bfloat16*>(dst), n, head, nvec);
    else
      convert_from_f32_kernel<<<g, CV_THREADS, 0, s>>>(static_cast<const float*>(src), static_cast<__half*>(dst), n, head, nvec);
  } else {
    if (in_dt == PV_BF16)
      convert_to_f32_kernel<<<g, CV_THREADS, 0, s>>>(static_cast<const __nv_bfloat16*>(src), static_cast<float*>(dst), n, head, nvec);
    else
      convert_to_f32_kernel<<<g, CV_THREADS, 0, s>>>(static_cast<const __half*>(src), static_cast<float*>(dst), n, head, nvec);
  }
  PV_LAUNCHED();
  return PV_OK;
}
