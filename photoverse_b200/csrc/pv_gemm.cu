// photoverse_b200 -- tcgen05 projection GEMM for sm_100a:  D[b] = A[b] * W[b]^T + bias
//
// Used for every dense projection on the PhotoVerse hot path that is not fused into the attention
// kernel: the out projection (attention_processor.py:423), the K/V projections (:304-305, :392-393)
// and the adapter MLP layers (adapters.py:14-28).
//
// Structure (one 128 x BN output tile per CTA, 192 threads):
//   warp 0      TMA producer : cp.async.bulk.tensor 3-D loads of the A tile [128 x 64] and W tile [BN x 64]
//                              (bf16, 128-byte swizzle) into a STAGES-deep mbarrier ring
//   warp 1      MMA issuer   : one elected thread issues tcgen05.mma (M=128, N=BN, K=16) x4 per stage,
//                              accumulating fp32 in TMEM; tcgen05.commit frees the smem slot
//   warps 2..5  epilogue     : tcgen05.ld (32 lanes x 32 columns) -> +bias -> bf16/fp32 -> swizzled smem
//                              staging -> per-warp TMA store (TMA clips the ragged M / N edges)
#include "pv_common.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_THREADS = 192;
constexpr int GEMM_A_BYTES = GEMM_BM * GEMM_BK * 2;

// STAGES_ == 0: deep ring, one CTA per SM (long K).  STAGES_ == 2: shallow ring so that TWO CTAs fit per SM
// (<= 113 KB smem, <= 256 TMEM columns each): with short K (the C=320 projections have 5 K-blocks) a tile is
// dominated by its prologue / epilogue, which the second resident CTA overlaps with its own main loop.
template <int BN, int STAGES_>
struct GemmCfg {
  static constexpr int W_BYTES = BN * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = GEMM_A_BYTES + W_BYTES;
  static constexpr int STAGES = STAGES_ > 0 ? STAGES_ : (BN >= 256 ? 4 : (BN >= 160 ? 5 : 6));
  static constexpr int MIN_CTAS = STAGES_ == 2 ? 2 : 1;
  static constexpr int EPI_TILE_BYTES = 32 * 128;          // per warp per buffer (fp32: 32x32x4, bf16 uses half)
  static constexpr int EPI_BYTES = 4 * 2 * EPI_TILE_BYTES;  // 4 warps, double buffered
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + BAR_BYTES + 1024;  // +1024 alignment slack
  static constexpr uint32_t TMEM_COLS = BN <= 32 ? 32 : BN <= 64 ? 64 : BN <= 128 ? 128 : 256;
};

// T: the 16-bit type of A, W and (OUT_F32 == false) D: __nv_bfloat16 or __half
template <int BN, int STAGES_, bool OUT_F32, bool EPI_SWZ, typename T>
__global__ void __launch_bounds__(GEMM_THREADS, (STAGES_ == 2 ? 2 : 1))
gemm_bf16_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                         const __grid_constant__ CUtensorMap tmD, const float* __restrict__ bias,
                         long long strideBias, int N, int K, int w_batched) {
  using Cfg = GemmCfg<BN, STAGES_>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* epi = smem + Cfg::STAGES * Cfg::STAGE_BYTES;
  uint64_t* full = reinterpret_cast<uint64_t*>(epi + Cfg::EPI_BYTES);
  uint64_t* empty = full + Cfg::STAGES;
  uint64_t* accum_full = empty + Cfg::STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(accum_full + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int n0 = blockIdx.x * BN;
  const int m0 = blockIdx.y * GEMM_BM;
  const int batch = blockIdx.z;
  const int kblocks = (K + GEMM_BK - 1) / GEMM_BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmD);
    for (int s = 0; s < Cfg::STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(accum_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_acc = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    for (int kb = 0; kb < kblocks; ++kb) {
      const int s = kb % Cfg::STAGES;
      const uint32_t ph = (kb / Cfg::STAGES) & 1;
      mbar_wait(&empty[s], ph ^ 1);
      if (elect_one()) {
        uint8_t* a_dst = smem + s * Cfg::STAGE_BYTES;
        uint8_t* w_dst = a_dst + GEMM_A_BYTES;
        mbar_expect_tx(&full[s], Cfg::STAGE_BYTES);
        tma_load_3d(a_dst, &tmA, &full[s], kb * GEMM_BK, m0, batch);
        tma_load_3d(w_dst, &tmW, &full[s], kb * GEMM_BK, n0, w_batched ? batch : 0);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = umma_idesc<T>(GEMM_BM, BN);
    for (int kb = 0; kb < kblocks; ++kb) {
      const int s = kb % Cfg::STAGES;
      const uint32_t ph = (kb / Cfg::STAGES) & 1;
      mbar_wait(&full[s], ph);
      tc_fence_after();
      if (elect_one()) {        // elect.sync, not `lane == 0`: lets the compiler issue the UTCHMMAs back to back
        const uint8_t* a_src = smem + s * Cfg::STAGE_BYTES;
        const uint8_t* w_src = a_src + GEMM_A_BYTES;
        const uint64_t da = umma_desc_sw128(a_src);
        const uint64_t dw = umma_desc_sw128(w_src);
#pragma unroll
        for (int k = 0; k < GEMM_BK / 16; ++k) {
          // +32 bytes per K=16 step inside the 128-byte swizzle atom -> +2 in the (addr >> 4) field
          umma_bf16_ss(tmem_acc, da + 2 * k, dw + 2 * k, idesc, (kb | k) != 0);
        }
        umma_commit(&empty[s]);
        if (kb == kblocks - 1) umma_commit(accum_full);
      }
      __syncwarp();
    }
  } else {
    // ===================== epilogue warps =====================
    const int q = warp & 3;                    // TMEM lane quarter this warp may access
    uint8_t* stg = epi + q * 2 * Cfg::EPI_TILE_BYTES;
    const float* bias_b = bias ? bias + strideBias * batch : nullptr;
    mbar_wait(accum_full, 0);
    tc_fence_after();
    const int row = lane;                      // row inside this warp's 32-row slab
#pragma unroll 1
    for (int c = 0; c < BN / 32; ++c) {
      if (n0 + c * 32 >= N) break;             // whole chunk is beyond the matrix edge (warp-uniform)
      uint32_t v[32];
      tmem_ld_x32(tmem_acc + (static_cast<uint32_t>(q * 32) << 16) + c * 32, v);
      tmem_ld_wait();
      uint8_t* buf = stg + (c & 1) * Cfg::EPI_TILE_BYTES;
      if (c >= 2) {                            // the TMA store that last read this buffer must be done
        if (elect_one()) bulk_wait_read<1>();
        __syncwarp();
      }
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        float b = 0.f;
        if (bias_b) {
          const int n = n0 + c * 32 + j;
          b = (n < N) ? __ldg(bias_b + n) : 0.f;
        }
        f[j] = __uint_as_float(v[j]) + b;
      }
      if constexpr (OUT_F32) {
        // 32 rows x 128 B ; SW128: 16-byte chunk index ^= (row & 7)
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) {
          const int pch = EPI_SWZ ? (ch ^ (row & 7)) : ch;
          st_shared_v4(buf + row * 128 + pch * 16, __float_as_uint(f[ch * 4 + 0]), __float_as_uint(f[ch * 4 + 1]),
                       __float_as_uint(f[ch * 4 + 2]), __float_as_uint(f[ch * 4 + 3]));
        }
      } else {
        // 32 rows x 64 B ; SW64: 16-byte chunk index ^= ((row >> 1) & 3)
#pragma unroll
        for (int ch = 0; ch < 4; ++ch) {
          const int pch = EPI_SWZ ? (ch ^ ((row >> 1) & 3)) : ch;
          st_shared_v4(buf + row * 64 + pch * 16, pack_x2<T>(f[ch * 8 + 0], f[ch * 8 + 1]),
                       pack_x2<T>(f[ch * 8 + 2], f[ch * 8 + 3]), pack_x2<T>(f[ch * 8 + 4], f[ch * 8 + 5]),
                       pack_x2<T>(f[ch * 8 + 6], f[ch * 8 + 7]));
        }
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        tma_store_3d(&tmD, buf, n0 + c * 32, m0 + q * 32, batch);
        bulk_commit();
      }
      __syncwarp();
    }
    if (elect_one()) bulk_wait_read<0>();
    __syncwarp();
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 1) tmem_dealloc<Cfg::TMEM_COLS>(tmem_acc);
}

// ------------------------------------------------------------------------------------------------
// host launcher
// ------------------------------------------------------------------------------------------------
extern int g_opt_epi_swizzle;
extern int g_opt_force_bn;

template <int BN, int STAGES_, bool OUT_F32, bool EPI_SWZ, typename T>
static int launch_one(const CUtensorMap& tmA, const CUtensorMap& tmW, const CUtensorMap& tmD, const float* bias,
                      long long strideBias, int M, int N, int K, int batch, int w_batched, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, STAGES_>;
  auto kern = gemm_bf16_tcgen05_kernel<BN, STAGES_, OUT_F32, EPI_SWZ, T>;
  PV_CUDA(set_max_smem_once(kern, Cfg::SMEM_BYTES));
  dim3 grid((N + BN - 1) / BN, (M + GEMM_BM - 1) / GEMM_BM, batch);
  kern<<<grid, GEMM_THREADS, Cfg::SMEM_BYTES, stream>>>(tmA, tmW, tmD, bias, strideBias, N, K, w_batched);
  PV_LAUNCHED();
  return PV_OK;
}

extern int g_opt_gemm_two_cta;
extern int g_opt_gemm_persistent;
int gemm3_bf16(const void* A, const void* W, const float* bias, void* D, long long M, long long N, long long K, long long lda,
               long long ldw, long long ldd, cudaStream_t stream, bool w_static, bool f16);

template <int BN, typename T>
static int launch_bn(bool out_f32, bool swz, const CUtensorMap& tmA, const CUtensorMap& tmW, const CUtensorMap& tmD,
                     const float* bias, long long strideBias, int M, int N, int K, int batch, int w_batched,
                     cudaStream_t stream) {
  // short K (<= 8 K-blocks): shallow ring, two CTAs per SM; the un-swizzled staging variant is kept for the
  // deep-ring bf16-out kernel only (A/B switch `epi_swizzle`, validated identical on B200)
  const bool two = g_opt_gemm_two_cta != 0 && (K + GEMM_BK - 1) / GEMM_BK <= 8;
  if (two) {
    return out_f32 ? launch_one<BN, 2, true, true, T>(tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream)
                   : launch_one<BN, 2, false, true, T>(tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream);
  }
  if (out_f32) return launch_one<BN, 0, true, true, T>(tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream);
  return swz ? launch_one<BN, 0, false, true, T>(tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream)
             : launch_one<BN, 0, false, false, T>(tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream);
}

static int pick_bn(long long M, long long N, long long batch, bool two_cta) {
  if (g_opt_force_bn == 64 || g_opt_force_bn == 128 || g_opt_force_bn == 160 || g_opt_force_bn == 256)
    return g_opt_force_bn;
  const int cands[4] = {256, 160, 128, 64};
  const long long sms = static_cast<long long>(sm_count()) * (two_cta ? 2 : 1);   // resident CTA slots
  long long best_cost = -1;
  int best = 128;
  for (int bn : cands) {
    if (bn == 64 && N > 64) continue;
    const long long tiles = ((M + GEMM_BM - 1) / GEMM_BM) * ((N + bn - 1) / bn) * batch;
    const long long waves = (tiles + sms - 1) / sms;
    const long long cost = waves * (bn + 32);   // per-tile time ~ BN (+ fixed prologue/epilogue share)
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = bn;
    }
  }
  return best;
}

// D[b] = A[b] W[b]^T + bias ; bf16 (f16: fp16) operands, output of the operand type or fp32.
int gemm_bf16(const void* A, const void* W, const float* bias, void* D, bool out_f32, long long M, long long N,
              long long K, long long batch, long long lda, long long ldw, long long ldd, long long strideA,
              long long strideW, long long strideBias, long long strideD, cudaStream_t stream, bool w_static, bool f16) {
  PV_REQUIRE(M > 0 && N > 0 && K > 0 && batch > 0, "empty problem M=%lld N=%lld K=%lld batch=%lld", M, N, K, batch);
  PV_REQUIRE(K % 8 == 0 && lda % 8 == 0 && ldw % 8 == 0, "bf16 rows must be 16-byte multiples (K=%lld lda=%lld ldw=%lld)",
             K, lda, ldw);
  const int oe = out_f32 ? 4 : 2;
  PV_REQUIRE((ldd * oe) % 16 == 0 && (strideD * oe) % 16 == 0, "output rows must be 16-byte multiples (ldd=%lld)", ldd);
  PV_REQUIRE((strideA * 2) % 16 == 0 && (strideW * 2) % 16 == 0, "batch strides must be 16-byte multiples");
  PV_REQUIRE((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(D)) % 16 == 0,
             "pointers must be 16-byte aligned");
  PV_REQUIRE(batch <= 65535 && (M + GEMM_BM - 1) / GEMM_BM <= 65535, "grid too large");
  // persistent CTA-pair kernel (pv_gemm3.cu): the out projection shapes (bf16 out, N % 160 == 0, K % 64 == 0, tall M)
  if (g_opt_gemm_persistent != 0 && g_opt_force_bn == 0 && !out_f32 && batch == 1 && M >= 512 && N % 160 == 0 && K % 64 == 0)
    return gemm3_bf16(A, W, bias, D, M, N, K, lda, ldw, ldd, stream, w_static, f16);
  const bool two_cta = g_opt_gemm_two_cta != 0 && (K + GEMM_BK - 1) / GEMM_BK <= 8;
  const int bn = pick_bn(M, N, batch, two_cta);
  const bool swz = g_opt_epi_swizzle != 0 || out_f32 || two_cta;
  const int w_batched = strideW != 0;
  CUtensorMap tmA, tmW, tmD;
  // batch stride 0 is not encodable: give un-batched operands a dummy stride with extent 1
  if (make_tmap_3d(&tmA, A, 2, K, M, batch, lda * 2, (batch > 1 ? strideA : lda * M) * 2, GEMM_BK, GEMM_BM, 1, Swz::B128, f16))
    return PV_ERR_CUDA;
  if (make_tmap_3d(&tmW, W, 2, K, N, w_batched ? batch : 1, ldw * 2, (w_batched ? strideW : ldw * N) * 2, GEMM_BK, bn, 1,
                   Swz::B128, f16))
    return PV_ERR_CUDA;
  if (make_tmap_3d(&tmD, D, oe, N, M, batch, ldd * oe, (batch > 1 ? strideD : ldd * M) * oe, 32, 32, 1,
                   swz ? (out_f32 ? Swz::B128 : Swz::B64) : Swz::None, f16))
    return PV_ERR_CUDA;
#define PV_GEMM_BN(BN)                                                                                         \
  (f16 ? launch_bn<BN, __half>(out_f32, swz, tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream)        \
       : launch_bn<BN, __nv_bfloat16>(out_f32, swz, tmA, tmW, tmD, bias, strideBias, M, N, K, batch, w_batched, stream))
  switch (bn) {
    case 256: return PV_GEMM_BN(256);
    case 160: return PV_GEMM_BN(160);
    case 128: return PV_GEMM_BN(128);
    default:  return PV_GEMM_BN(64);
  }
#undef PV_GEMM_BN
}

}  // namespace pv
