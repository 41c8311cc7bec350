// photoverse_b200 -- layout / packing kernels (HBM-bound, vectorised, coalesced).
//
//  * pack_weight      : W_eff = W + scaling * B A  (peft lora.Linear merged form) -> bf16 / fp16 / fp32
//  * kv_pack_bf16     : fp32 K/V projections -> per-(sample, head) bf16 / fp16 UMMA operand images consumed by the fused
//                       attention kernel via 1-D TMA bulk copies, + the `to_v_ip_norm` side output
//                       (attention_processor.py:395-397)
//  * kv_pack_f32      : same gather for the fp32 parity path ([B,H,L,d] fp32)
#include "pv_common.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

// OUT16: 16-bit output of type T16 (__nv_bfloat16 or __half), else fp32
template <bool OUT16, typename T16>
__global__ void __launch_bounds__(256)
pack_weight_kernel(const float* __restrict__ W, const float* __restrict__ A, const float* __restrict__ Bm,
                   float scaling, void* __restrict__ out, int out_f, int in_f, int r) {
  // one thread = 4 consecutive input features of one output row
  const long long idx = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) * 4;
  const long long total = static_cast<long long>(out_f) * in_f;
  if (idx >= total) return;
  const int o = static_cast<int>(idx / in_f);
  const int i = static_cast<int>(idx % in_f);
  float4 w = *reinterpret_cast<const float4*>(W + idx);
  if (r > 0) {
    float dx = 0.f, dy = 0.f, dz = 0.f, dw = 0.f;
    for (int k = 0; k < r; ++k) {
      const float bk = Bm[static_cast<long long>(o) * r + k];
      const float4 a = *reinterpret_cast<const float4*>(A + static_cast<long long>(k) * in_f + i);
      dx = fmaf(bk, a.x, dx); dy = fmaf(bk, a.y, dy); dz = fmaf(bk, a.z, dz); dw = fmaf(bk, a.w, dw);
    }
    w.x = fmaf(scaling, dx, w.x); w.y = fmaf(scaling, dy, w.y);
    w.z = fmaf(scaling, dz, w.z); w.w = fmaf(scaling, dw, w.w);
  }
  if constexpr (OUT16) {
    uint2 pk = make_uint2(pack_x2<T16>(w.x, w.y), pack_x2<T16>(w.z, w.w));
    *reinterpret_cast<uint2*>(static_cast<T16*>(out) + idx) = pk;
  } else {
    *reinterpret_cast<float4*>(static_cast<float*>(out) + idx) = w;
  }
}

int pack_weight(pv_dtype out_dt, const float* W, const float* A, const float* Bm, float scaling, void* out, int out_f,
                int in_f, int r, cudaStream_t stream) {
  PV_REQUIRE(out_f > 0 && in_f > 0 && in_f % 4 == 0 && r >= 0, "bad shape out=%d in=%d r=%d", out_f, in_f, r);
  PV_REQUIRE(r == 0 || (A != nullptr && Bm != nullptr), "LoRA rank %d without A/B", r);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(A)) % 16 == 0,
             "pointers must be 16-byte aligned");
  const long long total4 = static_cast<long long>(out_f) * in_f / 4;
  const int blocks = static_cast<int>((total4 + 255) / 256);
  if (out_dt == PV_BF16) pack_weight_kernel<true, __nv_bfloat16><<<blocks, 256, 0, stream>>>(W, A, Bm, scaling, out, out_f, in_f, r);
  else if (out_dt == PV_F16) pack_weight_kernel<true, __half><<<blocks, 256, 0, stream>>>(W, A, Bm, scaling, out, out_f, in_f, r);
  else pack_weight_kernel<false, __nv_bfloat16><<<blocks, 256, 0, stream>>>(W, A, Bm, scaling, out, out_f, in_f, r);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// kv_text:[B*Lt, 2C] fp32 (cols [0,C)=K, [C,2C)=V), kv_img:[B*Li, 2C] fp32
// Kp[b][h] : K-major core-matrix image of K_h  [96 keys  x d_pad]: chunk kc (8 dims) of key r at (kc*96   + r)*16 B
// Vp[b][h] : K-major core-matrix image of V_h^T [d_pad   x 96   ]: chunk kc (8 keys) of dim n at (kc*d_pad + n)*16 B
// ------------------------------------------------------------------------------------------------
// `img_off`: slot of the first image key (PV_IMG_KEY_OFFSET in the padded bf16 tiles, Lt in the compact fp32 layout)
__device__ __forceinline__ float kv_fetch(const float* __restrict__ kv_text, const float* __restrict__ kv_img, int b,
                                          int key, int col, int Lt, int Li, int C2, int img_off) {
  if (key < Lt) return kv_text[(static_cast<size_t>(b) * Lt + key) * C2 + col];
  if (key >= img_off && key < img_off + Li) return kv_img[(static_cast<size_t>(b) * Li + (key - img_off)) * C2 + col];
  return 0.f;
}

template <typename T>   // __nv_bfloat16 or __half tiles
__global__ void __launch_bounds__(256)
kv_pack_bf16_kernel(const float* __restrict__ kv_text, const float* __restrict__ kv_img, uint8_t* __restrict__ Kp,
                    uint8_t* __restrict__ Vp, float* __restrict__ v_ip_norm, int Lt, int Li, int C, int H, int d,
                    int d_pad) {
  const int h = blockIdx.x, b = blockIdx.y;
  const int C2 = 2 * C;
  const size_t tile_bytes = static_cast<size_t>(PV_KEYS_PAD) * d_pad * 2;
  uint8_t* kt = Kp + (static_cast<size_t>(b) * H + h) * tile_bytes;
  uint8_t* vt = Vp + (static_cast<size_t>(b) * H + h) * tile_bytes;
  const int nkc = d_pad / 8;
  // K tile: nkc * 96 chunks
  for (int idx = threadIdx.x; idx < nkc * PV_KEYS_PAD; idx += blockDim.x) {
    const int kc = idx / PV_KEYS_PAD, key = idx % PV_KEYS_PAD;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int dim = kc * 8 + i;
      v[i] = (dim < d) ? kv_fetch(kv_text, kv_img, b, key, h * d + dim, Lt, Li, C2, PV_IMG_KEY_OFFSET) : 0.f;
    }
    *reinterpret_cast<uint4*>(kt + static_cast<size_t>(idx) * 16) =
        make_uint4(pack_x2<T>(v[0], v[1]), pack_x2<T>(v[2], v[3]), pack_x2<T>(v[4], v[5]), pack_x2<T>(v[6], v[7]));
  }
  // V^T tile: 12 * d_pad chunks
  for (int idx = threadIdx.x; idx < (PV_KEYS_PAD / 8) * d_pad; idx += blockDim.x) {
    const int kc = idx / d_pad, dim = idx % d_pad;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int key = kc * 8 + i;
      v[i] = (dim < d) ? kv_fetch(kv_text, kv_img, b, key, C + h * d + dim, Lt, Li, C2, PV_IMG_KEY_OFFSET) : 0.f;
    }
    *reinterpret_cast<uint4*>(vt + static_cast<size_t>(idx) * 16) =
        make_uint4(pack_x2<T>(v[0], v[1]), pack_x2<T>(v[2], v[3]), pack_x2<T>(v[4], v[5]), pack_x2<T>(v[6], v[7]));
  }
  // ||V_img||_2 over head_dim, from the fp32 projections
  for (int li = threadIdx.x; li < Li; li += blockDim.x) {
    const float* row = kv_img + (static_cast<size_t>(b) * Li + li) * C2 + C + h * d;
    float s = 0.f;
    for (int i = 0; i < d; ++i) s = fmaf(row[i], row[i], s);
    v_ip_norm[(static_cast<size_t>(b) * H + h) * Li + li] = sqrtf(s);
  }
}

__global__ void __launch_bounds__(256)
kv_pack_f32_kernel(const float* __restrict__ kv_text, const float* __restrict__ kv_img, float* __restrict__ Kp,
                   float* __restrict__ Vp, float* __restrict__ v_ip_norm, int Lt, int Li, int C, int H, int d) {
  const int h = blockIdx.x, b = blockIdx.y;
  const int C2 = 2 * C, L = Lt + Li;
  float* kt = Kp + (static_cast<size_t>(b) * H + h) * L * d;
  float* vt = Vp + (static_cast<size_t>(b) * H + h) * L * d;
  for (int idx = threadIdx.x; idx < L * d; idx += blockDim.x) {
    const int key = idx / d, dim = idx % d;
    kt[idx] = kv_fetch(kv_text, kv_img, b, key, h * d + dim, Lt, Li, C2, Lt);
    vt[idx] = kv_fetch(kv_text, kv_img, b, key, C + h * d + dim, Lt, Li, C2, Lt);
  }
  for (int li = threadIdx.x; li < Li; li += blockDim.x) {
    const float* row = kv_img + (static_cast<size_t>(b) * Li + li) * C2 + C + h * d;
    float s = 0.f;
    for (int i = 0; i < d; ++i) s = fmaf(row[i], row[i], s);
    v_ip_norm[(static_cast<size_t>(b) * H + h) * Li + li] = sqrtf(s);
  }
}

int kv_pack(pv_dtype dt, const float* kv_text, const float* kv_img, void* Kp, void* Vp, float* v_ip_norm, int B, int Lt,
            int Li, int C, int H, cudaStream_t stream) {
  const int d = C / H;
  PV_REQUIRE(B <= 65535, "grid too large");
  dim3 grid(H, B);
  if (dt != PV_F32) {
    const int d_pad = (d + 15) / 16 * 16;
    auto kern = dt == PV_F16 ? kv_pack_bf16_kernel<__half> : kv_pack_bf16_kernel<__nv_bfloat16>;
    kern<<<grid, 256, 0, stream>>>(kv_text, kv_img, static_cast<uint8_t*>(Kp), static_cast<uint8_t*>(Vp), v_ip_norm, Lt, Li,
                                   C, H, d, d_pad);
  } else {
    kv_pack_f32_kernel<<<grid, 256, 0, stream>>>(kv_text, kv_img, static_cast<float*>(Kp), static_cast<float*>(Vp),
                                                 v_ip_norm, Lt, Li, C, H, d);
  }
  PV_LAUNCHED();
  return PV_OK;
}

}  // namespace pv

// ------------------------------------------------------------------------------------------------
// Concept-token injection into the CLIP token embeddings (reference models/clip.py:17-24):
//   out[b, l] = in[b, l]                 l <  idx_b
//             = concept[b, l - idx_b]    idx_b <= l < idx_b + T
//             = in[b, l - T + 1]         l >= idx_b + T          (the placeholder token in[b, idx_b] is dropped,
//                                                                 the tail is shifted right and truncated at L)
// and its backward (d_in, d_concept from d_out).  16-byte vectors, one thread per vector.
// ------------------------------------------------------------------------------------------------
namespace pv {

__global__ void __launch_bounds__(256)
inject_concept_fwd_kernel(const uint4* __restrict__ in, const uint4* __restrict__ concept, const int* __restrict__ idx,
                          uint4* __restrict__ out, int L, int T, int vec_per_row) {
  const int b = blockIdx.z, l = blockIdx.y;
  const int v = blockIdx.x * 256 + threadIdx.x;
  if (v >= vec_per_row) return;
  const int i = idx[b];
  uint4 val;
  if (l < i) val = in[(static_cast<size_t>(b) * L + l) * vec_per_row + v];
  else if (l < i + T) val = concept[(static_cast<size_t>(b) * T + (l - i)) * vec_per_row + v];
  else val = in[(static_cast<size_t>(b) * L + (l - T + 1)) * vec_per_row + v];
  out[(static_cast<size_t>(b) * L + l) * vec_per_row + v] = val;
}

template <typename T2>
__global__ void __launch_bounds__(256)
inject_concept_bwd_kernel(const T2* __restrict__ dout, const int* __restrict__ idx, T2* __restrict__ din,
                          T2* __restrict__ dconcept, int L, int T, int cols) {
  // grid.y covers L rows of d_in followed by T rows of d_concept
  const int b = blockIdx.z, r = blockIdx.y;
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= cols) return;
  const int i = idx[b];
  if (r < L) {
    const int l = r;
    float g = 0.f;
    if (l < i) g = static_cast<float>(dout[(static_cast<size_t>(b) * L + l) * cols + c]);
    else if (l > i && l + T - 1 < L) g = static_cast<float>(dout[(static_cast<size_t>(b) * L + (l + T - 1)) * cols + c]);
    din[(static_cast<size_t>(b) * L + l) * cols + c] = static_cast<T2>(g);
  } else {
    const int t = r - L;
    dconcept[(static_cast<size_t>(b) * T + t) * cols + c] = dout[(static_cast<size_t>(b) * L + (i + t)) * cols + c];
  }
}

int inject_concept_fwd(bool bf16, const void* in, const void* concept, const int* idx, void* out, int B, int L, int T,
                       int cols, cudaStream_t stream) {
  const int eb = bf16 ? 2 : 4;
  PV_REQUIRE(B > 0 && B <= 65535 && L > 0 && L <= 65535 && T > 0 && T <= L && cols > 0 && (cols * eb) % 16 == 0,
             "bad shape B=%d L=%d T=%d cols=%d", B, L, T, cols);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(concept) | reinterpret_cast<uintptr_t>(out)) % 16 == 0,
             "pointers must be 16-byte aligned");
  const int vpr = cols * eb / 16;
  dim3 grid((vpr + 255) / 256, L, B);
  inject_concept_fwd_kernel<<<grid, 256, 0, stream>>>(static_cast<const uint4*>(in), static_cast<const uint4*>(concept), idx,
                                                      static_cast<uint4*>(out), L, T, vpr);
  PV_LAUNCHED();
  return PV_OK;
}

int inject_concept_bwd(bool bf16, const void* dout, const int* idx, void* din, void* dconcept, int B, int L, int T, int cols,
                       cudaStream_t stream) {
  PV_REQUIRE(B > 0 && B <= 65535 && L > 0 && T > 0 && L + T <= 65535 && cols > 0, "bad shape");
  dim3 grid((cols + 255) / 256, L + T, B);
  if (bf16)
    inject_concept_bwd_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(static_cast<const __nv_bfloat16*>(dout), idx,
                                                                      static_cast<__nv_bfloat16*>(din),
                                                                      static_cast<__nv_bfloat16*>(dconcept), L, T, cols);
  else
    inject_concept_bwd_kernel<float><<<grid, 256, 0, stream>>>(static_cast<const float*>(dout), idx, static_cast<float*>(din),
                                                              static_cast<float*>(dconcept), L, T, cols);
  PV_LAUNCHED();
  return PV_OK;
}

// ------------------------------------------------------------------------------------------------
// LoRA dropout backward (peft lora.Linear: y = W x + s B A dropout(x); train.py:264-269, 348-354):
//   dst[i] += mask[i] ? alpha * src[i] : 0        alpha = 1 / (1 - p)
// dst is the input gradient that already holds the base-weight term, src = (dY B) A s, mask the keep-mask of the forward
// dropout (1 byte per element).  8 elements per thread.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
dropout_bwd_acc_kernel(T* __restrict__ dst, const T* __restrict__ src, const uint8_t* __restrict__ mask, float alpha,
                       long long n) {
  const long long base = (static_cast<long long>(blockIdx.x) * 256 + threadIdx.x) * 8;
  if (base >= n) return;
  if (base + 8 <= n) {
    const uint2 m = *reinterpret_cast<const uint2*>(mask + base);
    const uint8_t* mb = reinterpret_cast<const uint8_t*>(&m);
    T d[8], v[8];
    if constexpr (sizeof(T) == 2) {
      *reinterpret_cast<uint4*>(d) = *reinterpret_cast<const uint4*>(dst + base);
      *reinterpret_cast<uint4*>(v) = *reinterpret_cast<const uint4*>(src + base);
    } else {
      reinterpret_cast<uint4*>(d)[0] = reinterpret_cast<const uint4*>(dst + base)[0];
      reinterpret_cast<uint4*>(d)[1] = reinterpret_cast<const uint4*>(dst + base)[1];
      reinterpret_cast<uint4*>(v)[0] = reinterpret_cast<const uint4*>(src + base)[0];
      reinterpret_cast<uint4*>(v)[1] = reinterpret_cast<const uint4*>(src + base)[1];
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
      if (mb[j]) d[j] = static_cast<T>(static_cast<float>(d[j]) + alpha * static_cast<float>(v[j]));
    if constexpr (sizeof(T) == 2) {
      *reinterpret_cast<uint4*>(dst + base) = *reinterpret_cast<uint4*>(d);
    } else {
      reinterpret_cast<uint4*>(dst + base)[0] = reinterpret_cast<uint4*>(d)[0];
      reinterpret_cast<uint4*>(dst + base)[1] = reinterpret_cast<uint4*>(d)[1];
    }
  } else {
    for (long long i = base; i < n; ++i)
      if (mask[i]) dst[i] = static_cast<T>(static_cast<float>(dst[i]) + alpha * static_cast<float>(src[i]));
  }
}

int dropout_bwd_acc(bool bf16, void* dst, const void* src, const uint8_t* mask, float alpha, long long n,
                    cudaStream_t stream) {
  PV_REQUIRE(n > 0 && n % 8 == 0, "element count must be a positive multiple of 8 (n=%lld)", n);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) % 16 == 0 &&
                 reinterpret_cast<uintptr_t>(mask) % 8 == 0, "pointers must be 16-byte (mask: 8-byte) aligned");
  const long long blocks = (n / 8 + 255) / 256;
  PV_REQUIRE(blocks <= 0x7fffffffLL, "too many elements");
  if (bf16)
    dropout_bwd_acc_kernel<__nv_bfloat16><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(
        static_cast<__nv_bfloat16*>(dst), static_cast<const __nv_bfloat16*>(src), mask, alpha, n);
  else
    dropout_bwd_acc_kernel<float><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(
        static_cast<float*>(dst), static_cast<const float*>(src), mask, alpha, n);
  PV_LAUNCHED();
  return PV_OK;
}

}  // namespace pv
