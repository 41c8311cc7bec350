// photoverse_b200 -- persistent CTA-pair (cta_group::2) projection GEMM for the out projection of the processor
// (reference models/attention_processor.py:423):   D[M, N] = A[M, K] * W[N, K]^T + bias,  bf16 in / bf16 out,
// N % 160 == 0, K % 64 == 0.
//
// It is the projection pipeline of pv_attn4.cu with a plain epilogue instead of the attention: a pair of CTAs walks
// 256-row x 160-column output tiles of ONE column group g (so the pair's W slice never changes),
//   * the W slice [160 x K] is split across the pair (80 rows each) and, for K <= 640, stays RESIDENT in shared memory:
//     only A is streamed (16 KB per K-block per CTA) through a deep TMA ring;  K = 1280 streams 10 KB W halves as well
//   * ONE tcgen05.mma stream of M = 256 issued by the leader into double-buffered TMEM accumulators (2 x 160 columns):
//     the MMAs of tile i+1 run under the epilogue of tile i
//   * epilogue warps (2 x 4 per CTA): TMEM -> +bias -> bf16 (fp16 for fp16 operands) -> per-warp staging tile -> TMA store
// The single-CTA kernel of pv_gemm.cu spends most of a K = 320 tile in its prologue / epilogue (5 K-blocks) and is bound
// by TMA ingest (36 KB per K-block); this one has neither problem.
//
// linear_geglu_bf16 runs the same pipeline with the GEGLU epilogue: the feed-forward projection of a transformer block and
// its `a * gelu(gate)` in one launch, so the [M, 2N] projection never goes through global memory.
#include "pv_common.cuh"
#include "pv_outproj.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int G3_THREADS = 384;          // warp 0 TMA, warp 1 MMA (leader), warps 4..11 epilogue

// The pipeline itself is outproj_phase (pv_outproj.cuh) -- the same code that runs as the second phase of the fused
// processor kernels -- here without row-block counters (every A tile is ready when the kernel starts).
// EPI = OP_EPI_GEGLU: D[M, N / 2] = GEGLU of the packed projection (see pv_outproj.cuh); a pair's tiles are the contiguous
// share [T p / npairs, T (p + 1) / npairs) of the T = G V (group, unit) entries instead of the units of one group.
template <typename Cfg, int EPI, typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(G3_THREADS, 1)
gemm3_pair_persistent_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmW,
                             const __grid_constant__ CUtensorMap tmD, const float* __restrict__ bias, int G, int V, int K,
                             int w_static) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (Cfg::BYTES + 15) / 16 * 16);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + OP_BAR_BYTES / 8 + (EPI == OP_EPI_GEGLU ? 1 : 0));   // after w_free
  const int warp = threadIdx.x >> 5;
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  int g, u0, u1;
  if constexpr (EPI == OP_EPI_GEGLU) {
    const long long T = static_cast<long long>(G) * V;
    u0 = static_cast<int>(T * pair / npairs);
    u1 = static_cast<int>(T * (pair + 1) / npairs);
    g = u0 / V;
  } else {
    g = pair % G;
    const int r_pair = pair / G;
    const int npair_g = (npairs - g + G - 1) / G;
    u0 = static_cast<int>((static_cast<long long>(V) * r_pair) / npair_g);
    u1 = static_cast<int>((static_cast<long long>(V) * (r_pair + 1)) / npair_g);
  }

  if (warp == 0 && (threadIdx.x & 31) == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    tma_prefetch_desc(&tmD);
    op_mbar_init(bars);
    if constexpr (EPI == OP_EPI_GEGLU) mbar_init(bars + OP_W_FREE, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  // Nothing above reads global memory.  `w_static` (set only by the processor's own out-projection call, whose Wo was
  // packed many kernels earlier): the resident W half is requested before the dependency wait, under the predecessor's
  // tail; on the generic pv_linear_fwd route W, bias, A and D are all touched only after the predecessor has completed.
  if constexpr (Cfg::WSTAT) {
    if (w_static && warp == 0 && u0 < u1) {
      if (elect_one()) op_preload_w<Cfg>(smem, bars, &tmW, g, cluster_ctarank());
      __syncwarp();
    }
  }
  pdl_wait();
  pdl_launch_dependents();

  OutProjArgs oa;
  oa.bias = bias;
  oa.sync = nullptr;
  oa.G = G; oa.C = K; oa.V = V;
  oa.MTP = V > 0 ? V : 1;             // one "sample": tile u covers rows [256 u, 256 u + 256) of the flat [M, K] operand
  oa.u0 = u0;
  oa.u1 = u1;
  oa.g = g;
  oa.ready_target = 0;
  oa.w_preloaded = Cfg::WSTAT && w_static && u0 < u1;
  oa.trace = nullptr; oa.trace_cap = 0; oa.trace_block = 0;
  outproj_phase<Cfg, EPI, T>(smem, bars, tmem, &tmA, &tmW, &tmD, oa);

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  if (warp == 2) tmem_dealloc_2sm<512>(tmem);
}

template <int KB_RES, int STAGES, int EPI, typename T>
static int launch_g3(const CUtensorMap& tmA, const CUtensorMap& tmW, const CUtensorMap& tmD, const float* bias, int G, int V,
                     int K, int w_static, cudaStream_t stream) {
  using Cfg = OutProjCfg<KB_RES, STAGES>;
  constexpr int SMEM_BYTES = (Cfg::BYTES + 15) / 16 * 16 + 256 + 1024;
  static_assert(OP_BAR_BYTES + 8 + 8 <= 256 && SMEM_BYTES <= 227 * 1024, "shared memory budget");
  auto kern = gemm3_pair_persistent_kernel<Cfg, EPI, T>;
  PV_CUDA(set_max_smem_once(kern, SMEM_BYTES));
  const long long units = static_cast<long long>(G) * V;
  const long long max_pairs = sm_count() / 2;
  const int npairs = static_cast<int>(units < max_pairs ? units : max_pairs);
  PV_CUDA(launch_pdl(kern, dim3(2 * npairs), dim3(G3_THREADS), SMEM_BYTES, stream, tmA, tmW, tmD, bias, G, V, K, w_static));
  PV_LAUNCHED();
  return PV_OK;
}

// D[M,N] (bf16 or, with f16, fp16; row stride ldd) = A[M,K] (lda) * W[N,K]^T (ldw) + bias ; N % 160 == 0, K % 64 == 0
int gemm3_bf16(const void* A, const void* W, const float* bias, void* D, long long M, long long N, long long K, long long lda,
               long long ldw, long long ldd, cudaStream_t stream, bool w_static, bool f16) {
  PV_REQUIRE(M > 0 && N % OP_BN == 0 && K % OP_BK == 0 && N > 0 && K > 0, "gemm3: need N %% 160 == 0 and K %% 64 == 0 (N=%lld K=%lld)", N, K);
  PV_REQUIRE((lda * 2) % 16 == 0 && (ldw * 2) % 16 == 0 && (ldd * 2) % 16 == 0, "row strides must be 16-byte multiples");
  CUtensorMap tmA, tmW, tmD;
  if (make_tmap_3d(&tmA, A, 2, K, M, 1, lda * 2, lda * M * 2, OP_BK, 128, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmW, W, 2, K, N, 1, ldw * 2, ldw * N * 2, OP_BK, OP_BN / 2, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmD, D, 2, N, M, 1, ldd * 2, ldd * M * 2, 80, 32, 1, Swz::None, f16)) return PV_ERR_CUDA;
  const int G = static_cast<int>(N / OP_BN);
  const long long V = (M + 255) / 256;
  PV_REQUIRE(V * G < (1ll << 30), "too many tiles");
#define PV_G3(KB, ST)                                                                                                    \
  (f16 ? launch_g3<KB, ST, OP_EPI_BIAS, __half>(tmA, tmW, tmD, bias, G, static_cast<int>(V), static_cast<int>(K), w_static, stream) \
       : launch_g3<KB, ST, OP_EPI_BIAS, __nv_bfloat16>(tmA, tmW, tmD, bias, G, static_cast<int>(V), static_cast<int>(K), w_static, stream))
  if (K == 320) return PV_G3(5, 8);
  if (K == 640) return PV_G3(10, 5);
  return PV_G3(0, 7);
#undef PV_G3
}

// y[M, N] (bf16, row stride ldy) = GEGLU of x[M, K] (ldx) * Wp[2N, K]^T + bp, with Wp / bp packed per 80 output columns
// (rows [160 j, 160 j + 80) = value rows [80 j, 80 j + 80) of the nn.Linear(K, 2N), rows [160 j + 80, 160 j + 160) = gate rows
// N + [80 j, 80 j + 80)); N % 80 == 0, K % 64 == 0.  No split-K: a row's result does not depend on M or on its tile.
int linear_geglu_bf16(const void* x, const void* Wp, const float* bp, void* y, long long M, long long N, long long K,
                      long long ldx, long long ldy, cudaStream_t stream) {
  PV_REQUIRE(M > 0 && N > 0 && K > 0 && N % (OP_BN / 2) == 0 && K % OP_BK == 0,
             "linear_geglu: need M > 0, N %% 80 == 0 and K %% 64 == 0 (M=%lld N=%lld K=%lld)", M, N, K);
  PV_REQUIRE(ldx >= K && ldy >= N && ldx % 8 == 0 && ldy % 8 == 0, "linear_geglu: row strides must be >= the row and 16-byte multiples (ldx=%lld ldy=%lld)", ldx, ldy);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(Wp) | reinterpret_cast<uintptr_t>(y)) % 16 == 0,
             "linear_geglu: pointers must be 16-byte aligned");
  const long long G = 2 * N / OP_BN;
  const long long V = (M + 255) / 256;
  PV_REQUIRE(V * G < (1ll << 30), "too many tiles");
  CUtensorMap tmA, tmW, tmD;
  if (make_tmap_3d(&tmA, x, 2, K, M, 1, ldx * 2, ldx * M * 2, OP_BK, 128, 1, Swz::B128)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmW, Wp, 2, K, 2 * N, 1, K * 2, K * 2 * N * 2, OP_BK, OP_BN / 2, 1, Swz::B128)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmD, y, 2, N, M, 1, ldy * 2, ldy * M * 2, 40, 32, 1, Swz::None)) return PV_ERR_CUDA;
  // the packed weight is a cached copy of a parameter, never written by the kernel this launch may overlap (w_static)
  if (K == 320) return launch_g3<5, 8, OP_EPI_GEGLU, __nv_bfloat16>(tmA, tmW, tmD, bp, static_cast<int>(G), static_cast<int>(V), static_cast<int>(K), 1, stream);
  if (K == 640) return launch_g3<10, 5, OP_EPI_GEGLU, __nv_bfloat16>(tmA, tmW, tmD, bp, static_cast<int>(G), static_cast<int>(V), static_cast<int>(K), 1, stream);
  return launch_g3<0, 7, OP_EPI_GEGLU, __nv_bfloat16>(tmA, tmW, tmD, bp, static_cast<int>(G), static_cast<int>(V), static_cast<int>(K), 1, stream);
}

}  // namespace pv
