// photoverse_b200 -- dual-branch attention backward core on tcgen05 (bf16 training path, head_dim 40 / 80).
//
// Same contract as attn_bwd_mma_kernel (pv_bwd_mma.cu) and attn_bwd_kernel (pv_bwd.cu): from dO, Q [B,S,C] (bf16), the fp32
// K / V projections and the forward kernel's per-row statistics, dQ [B,S,C] and per-chunk partial dK / dV (fp32) that
// kv_bwd_reduce_kernel sums.  Reference: the autograd graph of models/attention_processor.py:307-322, 400-420.
//   p^ = 2^(s cs - m)/l per segment ; dp_k = dO.V_k ; delta_seg = sum_{k in seg} p^_k dp_k ; ds_k = w_seg p^_k (dp_k - delta_seg)
//   dQ = scale ds K ; dK = scale ds^T Q ; dV = (w p^)^T dO
// One CTA = T consecutive 128-query-row tiles of one (sample, head); all five contractions are tcgen05.mma (M = 128) with
// fp32 accumulators in TMEM:
//   S  = Q K^T   [rows x 96 keys]   A = Q tile  (TMA, 128-byte swizzle, K-major)       B = K image (K-major)
//   dP = dO V^T  [rows x 96 keys]   A = dO tile                                        B = V image
//   dQ = dS K    [rows x d]         A = dS image (K-major)                             B = K image read MN-major
//   dK += dS^T Q [keys x d]         A = dS image read MN-major (transposed for free)   B = Q tile read MN-major
//   dV += P^T dO [keys x d]         A = P image read MN-major                          B = dO tile read MN-major
// dK / dV stay in TMEM across the CTA's tiles.  The transposes the mma.sync kernel does with ldmatrix.trans are a bit in
// the instruction descriptor here (operand "major-ness"): every operand is stored once.
// Warps: 0 TMA producer (Q / dO, two stages), 1 tcgen05 issuer, 2 TMEM allocator, 4-7 and 8-11 two groups with one thread
// per query row (= TMEM lane) each: softmax / dS of half the key slots, half of the dQ drain, dK resp. dV drain at the end.
#include <type_traits>

#include "pv_common.cuh"
#include "pv_host.h"
#include "pv_softmax.cuh"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int BT_KEYS = PV_KEYS_PAD;          // 96 key slots: keys [0, Lt) text, [Lt, Lt + Li) image, rest zero
constexpr int BT_THREADS = 384;

template <int D>
struct BtCfg {
  static constexpr int DP = (D + 15) / 16 * 16;            // 48 / 80
  static constexpr int NBOX = (DP + 63) / 64;              // 64-column TMA boxes per Q / dO tile
  static constexpr int BOX_BYTES = 128 * 128;              // 128 rows x 128 bytes
  static constexpr int QT_BYTES = NBOX * BOX_BYTES;
  static constexpr int NKC = DP / 8;                       // 16-byte chunks per key row
  static constexpr int KV_BYTES = NKC * BT_KEYS * 16;      // K / V image [d chunk][key][8]
  static constexpr int PS_BYTES = 16 * 128 * 16;           // P / dS image [key chunk (16: M = 128 keys)][row][8 keys]
  static constexpr int OFF_Q = 0;                          // two stages
  static constexpr int OFF_DO = OFF_Q + 2 * QT_BYTES;
  static constexpr int OFF_P = OFF_DO + 2 * QT_BYTES;
  static constexpr int OFF_DS = OFF_P + PS_BYTES;
  static constexpr int OFF_K = OFF_DS + PS_BYTES;
  static constexpr int OFF_V = OFF_K + KV_BYTES;
  static constexpr int OFF_XCH = OFF_V + KV_BYTES;        // partial segment sums exchanged by the two groups
  static constexpr int OFF_BAR = OFF_XCH + 2 * 2 * 128 * 2 * 4;
  static constexpr int SMEM_BYTES = OFF_BAR + 128;
  static constexpr int TM_S = 0, TM_DP = BT_KEYS, TM_DQ = 2 * BT_KEYS, TM_DK = TM_DQ + DP, TM_DV = TM_DK + DP;
  static_assert(TM_DV + DP <= 512, "TMEM columns");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory");
};

struct BtParams {
  const float* kv_text;
  const float* kv_img;
  const float* stats;
  __nv_bfloat16* dQ;
  float* part;
  int B, S, C, H, Lt, Li, T;
  float w_text, w_img, scale, scale_log2e;
  const float* img_row_weight;     // MASK kernels: [B, S] fp32 factor of each query row's image keys (ip_adapter_masks)
};

// LT77: 77 text keys (CLIP) -- the segment of every key slot is known at compile time.  MASK: the image keys of row s are
// weighted w_img * img_row_weight[b, s].
template <int D, bool LT77, bool MASK>
__global__ void __launch_bounds__(BT_THREADS, 1)
attn_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmdO, const BtParams p) {
  using Cfg = BtCfg<D>;
  constexpr int DP = Cfg::DP;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* q_full = bars;          // [2]  Q + dO tile landed
  uint64_t* q_empty = bars + 2;     // [2]  the tile's last MMAs have completed
  uint64_t* s_full = bars + 4;      // S and dP of a tile are in TMEM
  uint64_t* ds_ready = bars + 5;    // P / dS images written (and S / dP read for the last time)
  uint64_t* mma2_done = bars + 6;   // dQ, dK, dV contributions of a tile accumulated
  uint64_t* dq_free = bars + 7;     // the dQ accumulator has been read
  uint64_t* sdp_free = bars + 8;    // S and dP of a tile are in registers: the next tile's may overwrite them
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int L = p.Lt + p.Li, S = p.S;
  const int MT = (S + 127) / 128;
  const int t_begin = chunk * p.T;
  const int nt = min(p.T, MT - t_begin);            // tiles of this CTA (>= 1 by construction of the grid)

  if (threadIdx.x == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(&q_full[s], 1);
      mbar_init(&q_empty[s], 1);
    }
    mbar_init(s_full, 1);
    mbar_init(ds_ready, 8);
    mbar_init(mma2_done, 1);
    mbar_init(dq_free, 8);
    mbar_init(sdp_free, 8);
    fence_barrier_init();
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmdO);
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  // ---- K / V images: fp32 projections -> bf16 (the rounding the forward kernel's tiles have), [d chunk][key][8] ----
  {
    const int C2 = 2 * p.C;
    for (int i = threadIdx.x; i < Cfg::NKC * BT_KEYS; i += BT_THREADS) {
      const int ch = i / BT_KEYS, k = i - ch * BT_KEYS;
      uint4 kq = make_uint4(0, 0, 0, 0), vq = kq;
      if (k < L && ch * 8 < D) {
        const float* src = (k < p.Lt) ? p.kv_text + (static_cast<size_t>(b) * p.Lt + k) * C2
                                      : p.kv_img + (static_cast<size_t>(b) * p.Li + (k - p.Lt)) * C2;
        const float4 k0 = *reinterpret_cast<const float4*>(src + h * D + ch * 8);
        const float4 k1 = *reinterpret_cast<const float4*>(src + h * D + ch * 8 + 4);
        const float4 v0 = *reinterpret_cast<const float4*>(src + p.C + h * D + ch * 8);
        const float4 v1 = *reinterpret_cast<const float4*>(src + p.C + h * D + ch * 8 + 4);
        kq = make_uint4(pack_bf16x2(k0.x, k0.y), pack_bf16x2(k0.z, k0.w), pack_bf16x2(k1.x, k1.y), pack_bf16x2(k1.z, k1.w));
        vq = make_uint4(pack_bf16x2(v0.x, v0.y), pack_bf16x2(v0.z, v0.w), pack_bf16x2(v1.x, v1.y), pack_bf16x2(v1.z, v1.w));
      }
      *reinterpret_cast<uint4*>(smem + Cfg::OFF_K + i * 16) = kq;
      *reinterpret_cast<uint4*>(smem + Cfg::OFF_V + i * 16) = vq;
    }
    // key chunks 12..15 of the P / dS images (M = 128 keys, 96 real slots) only feed accumulator rows that are never
    // read; cleared once so that those rows stay finite
    for (int i = threadIdx.x; i < 4 * 128; i += BT_THREADS) {
      *reinterpret_cast<uint4*>(smem + Cfg::OFF_P + (12 * 128 + i) * 16) = make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4*>(smem + Cfg::OFF_DS + (12 * 128 + i) * 16) = make_uint4(0, 0, 0, 0);
    }
    fence_proxy_async_smem();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  if (warp == 0) {
    // ---------------------------------------------------------------- producer
    if (elect_one()) {
      for (int t = 0; t < nt; ++t) {
        const int s = t & 1;
        if (t >= 2) mbar_wait(&q_empty[s], ((t >> 1) - 1) & 1);
        mbar_expect_tx(&q_full[s], 2 * Cfg::QT_BYTES);
        const int q0 = (t_begin + t) * 128;
#pragma unroll
        for (int bx = 0; bx < Cfg::NBOX; ++bx) {
          tma_load_3d(smem + Cfg::OFF_Q + s * Cfg::QT_BYTES + bx * Cfg::BOX_BYTES, &tmQ, &q_full[s], h * D + bx * 64, q0, b);
          tma_load_3d(smem + Cfg::OFF_DO + s * Cfg::QT_BYTES + bx * Cfg::BOX_BYTES, &tmdO, &q_full[s], h * D + bx * 64, q0, b);
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ---------------------------------------------------------------- tcgen05 issuer
    constexpr uint32_t ID_S = umma_idesc_bf16(128, BT_KEYS);                                  // A, B K-major
    constexpr uint32_t ID_DQ = umma_idesc_bf16(128, DP) | (1u << 16);                         // B MN-major
    constexpr uint32_t ID_DKV = umma_idesc_bf16(128, DP) | (1u << 15) | (1u << 16);           // A and B MN-major
    const uint32_t q_addr = smem_u32(smem + Cfg::OFF_Q), do_addr = smem_u32(smem + Cfg::OFF_DO);
    const uint32_t p_addr = smem_u32(smem + Cfg::OFF_P), ds_addr = smem_u32(smem + Cfg::OFF_DS);
    const uint32_t k_addr = smem_u32(smem + Cfg::OFF_K), v_addr = smem_u32(smem + Cfg::OFF_V);
    // K-major 128-byte-swizzled A operand of k step ks (16 dims = 32 bytes inside the swizzled row; 64 dims per box)
    auto a_sw = [&](uint32_t tile, int ks) {
      return umma_desc(tile + (ks >> 2) * Cfg::BOX_BYTES + (ks & 3) * 32, 16, 1024, UMMA_LAYOUT_SW128);
    };
    auto issue_s_dp = [&](int s) {
      const uint32_t qt = q_addr + s * Cfg::QT_BYTES, ot = do_addr + s * Cfg::QT_BYTES;
      const uint64_t kb = umma_desc(k_addr, BT_KEYS * 16, 128, UMMA_LAYOUT_NONE);    // [key][d]: K-major, chunk stride = LBO
      const uint64_t vb = umma_desc(v_addr, BT_KEYS * 16, 128, UMMA_LAYOUT_NONE);
#pragma unroll
      for (int ks = 0; ks < DP / 16; ++ks)
        umma_bf16_ss(tmem + Cfg::TM_S, a_sw(qt, ks), kb + static_cast<uint64_t>(ks * (2 * BT_KEYS * 16 >> 4)), ID_S, ks > 0);
#pragma unroll
      for (int ks = 0; ks < DP / 16; ++ks)
        umma_bf16_ss(tmem + Cfg::TM_DP, a_sw(ot, ks), vb + static_cast<uint64_t>(ks * (2 * BT_KEYS * 16 >> 4)), ID_S, ks > 0);
      umma_commit(s_full);
    };
    auto issue_grads = [&](int s, bool first) {
      const uint32_t qt = q_addr + s * Cfg::QT_BYTES, ot = do_addr + s * Cfg::QT_BYTES;
      // dQ = dS K: A = dS [row][key] K-major (key chunks 2048 bytes apart); B = K image read MN-major (n = dim, k = key):
      // LBO = 8-key groups (128 bytes), SBO = 8-dim groups (one d chunk = 96 keys x 16 bytes)
      const uint64_t a_ds = umma_desc(ds_addr, 128 * 16, 128, UMMA_LAYOUT_NONE);
      const uint64_t b_k = umma_desc(k_addr, 128, BT_KEYS * 16, UMMA_LAYOUT_NONE);
#pragma unroll
      for (int ks = 0; ks < BT_KEYS / 16; ++ks)
        umma_bf16_ss(tmem + Cfg::TM_DQ, a_ds + static_cast<uint64_t>(ks * (2 * 128 * 16 >> 4)), b_k + static_cast<uint64_t>(ks * (256 >> 4)),
                     ID_DQ, ks > 0);
      // dK += dS^T Q, dV += P^T dO: A = the same images read MN-major (m = key, k = row): SBO = 8-key groups (2048 bytes),
      // LBO = 8-row groups (128 bytes); B = the swizzled Q / dO tile read MN-major (n = dim, k = row): 8-row groups 1024
      // bytes apart (SBO), 64-dim boxes BOX_BYTES apart (LBO); 16 rows per k step
      const uint64_t a_dst = umma_desc(ds_addr, 128, 128 * 16, UMMA_LAYOUT_NONE);
      const uint64_t a_pt = umma_desc(p_addr, 128, 128 * 16, UMMA_LAYOUT_NONE);
      const uint64_t b_q = umma_desc(qt, Cfg::BOX_BYTES, 1024, UMMA_LAYOUT_SW128);
      const uint64_t b_o = umma_desc(ot, Cfg::BOX_BYTES, 1024, UMMA_LAYOUT_SW128);
#pragma unroll
      for (int ks = 0; ks < 128 / 16; ++ks)
        umma_bf16_ss(tmem + Cfg::TM_DK, a_dst + static_cast<uint64_t>(ks * (256 >> 4)), b_q + static_cast<uint64_t>(ks * (2048 >> 4)),
                     ID_DKV, (!first || ks > 0) ? 1u : 0u);
#pragma unroll
      for (int ks = 0; ks < 128 / 16; ++ks)
        umma_bf16_ss(tmem + Cfg::TM_DV, a_pt + static_cast<uint64_t>(ks * (256 >> 4)), b_o + static_cast<uint64_t>(ks * (2048 >> 4)),
                     ID_DKV, (!first || ks > 0) ? 1u : 0u);
      umma_commit(mma2_done);
      umma_commit(&q_empty[s]);
    };
    mbar_wait(&q_full[0], 0);
    tc_fence_after();
    if (elect_one()) issue_s_dp(0);
    __syncwarp();
    for (int t = 0; t < nt; ++t) {
      const int s = t & 1;
      // the next tile's S / dP as soon as this tile's are in registers: they are ready when the groups come back
      if (t + 1 < nt) {
        mbar_wait(&q_full[s ^ 1], ((t + 1) >> 1) & 1);
        mbar_wait(sdp_free, t & 1);
        tc_fence_after();
        if (elect_one()) issue_s_dp(s ^ 1);
        __syncwarp();
      }
      mbar_wait(ds_ready, t & 1);
      if (t > 0) mbar_wait(dq_free, (t - 1) & 1);
      tc_fence_after();
      if (elect_one()) issue_grads(s, t == 0);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ---------------------------------------------------------------- softmax / dS / drains: two groups of 128 threads, one
    // thread per query row (= TMEM lane) in each; group 0 takes key slots [0, 48), group 1 [48, 96) of every row (the dS pass
    // is the longest stage of the pipeline and a serial instruction stream per warp); they exchange their partial
    // segment sums through shared memory, split the dQ drain by columns, and drain dK (group 0) / dV (group 1) at the end.
    const int wg = (warp - 4) >> 2;
    const int wq = warp & 3, row = wq * 32 + lane;
    const uint32_t lane_base = static_cast<uint32_t>(wq * 32) << 16;
    const uint32_t s_t = tmem + lane_base + Cfg::TM_S, dp_t = tmem + lane_base + Cfg::TM_DP;
    const uint32_t p_row = smem_u32(smem + Cfg::OFF_P) + row * 16, ds_row = smem_u32(smem + Cfg::OFF_DS) + row * 16;
    float* xch = reinterpret_cast<float*>(smem + Cfg::OFF_XCH);            // [parity][group][row][2]
    const int Lt = p.Lt;
    auto load_stats = [&](int t) {
      const int r = (t_begin + t) * 128 + row;
      float4 v = make_float4(0.f, 1.f, 0.f, 1.f);
      if (t < nt && r < S) v = __ldg(reinterpret_cast<const float4*>(p.stats) + (static_cast<size_t>(b) * p.H + h) * S + r);
      return v;
    };
    // this group's share of the dQ accumulator of tile t -> global memory
    auto drain_dq = [&](int t) {
      mbar_wait(mma2_done, t & 1);
      tc_fence_after();
      const int grow = (t_begin + t) * 128 + row;
      __nv_bfloat16* dst = p.dQ + (static_cast<size_t>(b) * S + grow) * p.C + h * D;
      constexpr int CSPLIT = D == 40 ? 24 : D / 2;
      const int cb = wg == 0 ? 0 : CSPLIT, ce = wg == 0 ? CSPLIT : D;
#pragma unroll
      for (int c = 0; c < D; c += 8) {
        if (c < cb || c >= ce) continue;                 // (group-uniform)
        uint32_t o[8];
        tmem_ld_x8(tmem + lane_base + Cfg::TM_DQ + c, o);
        tmem_ld_wait();
        if (grow < S)
          st_global_v4(dst + c, pack_bf16x2(__uint_as_float(o[0]), __uint_as_float(o[1])), pack_bf16x2(__uint_as_float(o[2]), __uint_as_float(o[3])),
                       pack_bf16x2(__uint_as_float(o[4]), __uint_as_float(o[5])), pack_bf16x2(__uint_as_float(o[6]), __uint_as_float(o[7])));
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(dq_free);
    };
    auto run = [&](auto k0c) {
      constexpr int K0 = decltype(k0c)::value;            // first key slot of this group; 48 slots
      float4 st_next = load_stats(0);
      for (int t = 0; t < nt; ++t) {
        const int grow = (t_begin + t) * 128 + row;
        const float4 st = st_next;
        st_next = load_stats(t + 1);                      // one tile ahead: the load's latency hides under this tile's work
        const float ilt = grow < S ? 1.f / st.y : 0.f, ili = grow < S ? 1.f / st.w : 0.f;     // rows past S: p^ = 0
        mbar_wait(s_full, t & 1);
        tc_fence_after();
        // ---- pass 1: p^ of my 48 key slots (kept in registers) and my part of the two segment sums of p^ dp
        float e[48];
        uint32_t dp[48];
        {
          uint32_t* eu = reinterpret_cast<uint32_t*>(e);
          tmem_ld32_raw(s_t + K0, eu);
          tmem_ld16_raw(s_t + K0 + 32, eu + 32);
          tmem_ld32_raw(dp_t + K0, dp);
          tmem_ld16_raw(dp_t + K0 + 32, dp + 32);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(sdp_free);
        }
        float dsum_t = 0.f, dsum_i = 0.f;
        if constexpr (LT77) {
          // 77 text keys: the segment of every slot is a compile-time fact; packed fp32x2 arithmetic.  Pairs (k, k+1):
          // k + 1 < 77 text, k >= 78 image (masked by k < L); the pair (76, 77) straddles the boundary (scalar form).
          const uint64_t sc2 = f2_pack(p.scale_log2e, p.scale_log2e);
          const uint64_t nmt2 = f2_pack(-st.x, -st.x), nmi2 = f2_pack(-st.z, -st.z);
          const uint64_t ilt2 = f2_pack(ilt, ilt), ili2 = f2_pack(ili, ili);
          uint64_t dt2 = f2_pack(0.f, 0.f), di2 = dt2;
#pragma unroll
          for (int i = 0; i < 48; i += 2) {
            const int key = K0 + i;
            const uint64_t pd = f2_pack(__uint_as_float(dp[i]), __uint_as_float(dp[i + 1]));
            if (key + 1 < 77) {
              float a, b2;
              f2_unpack(f2_fma(f2_pack(e[i], e[i + 1]), sc2, nmt2), a, b2);
              const uint64_t v2 = f2_mul(f2_pack(fast_exp2(a), fast_exp2(b2)), ilt2);
              f2_unpack(v2, e[i], e[i + 1]);
              dt2 = f2_fma(v2, pd, dt2);
            } else if (key >= 78) {
              float a, b2;
              f2_unpack(f2_fma(f2_pack(e[i], e[i + 1]), sc2, nmi2), a, b2);
              f2_unpack(f2_mul(f2_pack(fast_exp2(a), fast_exp2(b2)), ili2), a, b2);
              e[i] = key < L ? a : 0.f;
              e[i + 1] = key + 1 < L ? b2 : 0.f;
              di2 = f2_fma(f2_pack(e[i], e[i + 1]), pd, di2);
            } else {                                                      // keys 76 (text) and 77 (image, always present)
              e[i] = fast_exp2(fmaf(e[i], p.scale_log2e, -st.x)) * ilt;
              e[i + 1] = fast_exp2(fmaf(e[i + 1], p.scale_log2e, -st.z)) * ili;
              dsum_t = e[i] * __uint_as_float(dp[i]);
              dsum_i = e[i + 1] * __uint_as_float(dp[i + 1]);
            }
          }
          float s0, s1;
          f2_unpack(dt2, s0, s1);
          dsum_t += s0 + s1;
          f2_unpack(di2, s0, s1);
          dsum_i += s0 + s1;
        } else {
#pragma unroll
          for (int i = 0; i < 48; ++i) {
            const int key = K0 + i;
            const bool is_t = key < Lt;
            const float v = fast_exp2(fmaf(e[i], p.scale_log2e, is_t ? -st.x : -st.z)) * (is_t ? ilt : ili);
            e[i] = key < L ? v : 0.f;
            const float pd = e[i] * __uint_as_float(dp[i]);
            if (is_t) dsum_t += pd; else dsum_i += pd;
          }
        }
        // ---- the other group's part of the sums
        {
          float* mine = xch + (((t & 1) * 2 + wg) * 128 + row) * 2;
          const float* theirs = xch + (((t & 1) * 2 + (wg ^ 1)) * 128 + row) * 2;
          mine[0] = dsum_t;
          mine[1] = dsum_i;
          named_bar_sync(1, 256);
          dsum_t += theirs[0];
          dsum_i += theirs[1];
        }
        // ---- the previous tile: its gradient contractions have completed (the P / dS images are free again) -> my share of dQ
        if (t > 0) drain_dq(t - 1);
        // ---- pass 2: w p^ and scale w p^ (dp - delta) as bf16, 8 keys (16 bytes) at a time
        float wi = p.w_img;
        if constexpr (MASK) wi *= grow < S ? __ldg(p.img_row_weight + static_cast<size_t>(b) * S + grow) : 0.f;
        const float swt = p.scale * p.w_text, swi = p.scale * wi;
#pragma unroll
        for (int c = 0; c < 6; ++c) {
          uint32_t pw[4], dw[4];
#pragma unroll
          for (int q2 = 0; q2 < 4; ++q2) {
            const int i = 8 * c + 2 * q2, key = K0 + i;
            float a, b2, c1, d1;
            if (LT77 && (key + 1 < 77 || key >= 78)) {
              const bool txt = key + 1 < 77;
              const uint64_t e2 = f2_pack(e[i], e[i + 1]);
              const uint64_t pd = f2_pack(__uint_as_float(dp[i]), __uint_as_float(dp[i + 1]));
              const float w = txt ? p.w_text : wi, sw = txt ? swt : swi, nd = txt ? -dsum_t : -dsum_i;
              f2_unpack(f2_mul(e2, f2_pack(w, w)), a, b2);
              f2_unpack(f2_mul(f2_mul(e2, f2_pack(sw, sw)), f2_add(pd, f2_pack(nd, nd))), c1, d1);
            } else {
              const bool t0 = LT77 ? true : key < Lt, t1 = LT77 ? false : key + 1 < Lt;
              a = (t0 ? p.w_text : wi) * e[i];
              b2 = (t1 ? p.w_text : wi) * e[i + 1];
              c1 = (t0 ? swt : swi) * e[i] * (__uint_as_float(dp[i]) - (t0 ? dsum_t : dsum_i));
              d1 = (t1 ? swt : swi) * e[i + 1] * (__uint_as_float(dp[i + 1]) - (t1 ? dsum_t : dsum_i));
            }
            pw[q2] = pack_bf16x2(a, b2);
            dw[q2] = pack_bf16x2(c1, d1);
          }
          const int kc = K0 / 8 + c;
          st_shared_v4_a(p_row + kc * 2048, pw[0], pw[1], pw[2], pw[3]);
          st_shared_v4_a(ds_row + kc * 2048, dw[0], dw[1], dw[2], dw[3]);
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(ds_ready);
      }
      drain_dq(nt - 1);
    };
    if (wg == 0) run(std::integral_constant<int, 0>{});
    else run(std::integral_constant<int, 48>{});
    // ---- dK (group 0) / dV (group 1): TMEM lane = key.  (tcgen05.ld is warp-collective: every lane loads, only the lanes
    // of real keys store.)
    {
      const int key = row;
      float* dst = p.part + ((static_cast<size_t>(chunk) * p.B + b) * p.H + h) * 2 * L * D + static_cast<size_t>(wg) * L * D +
                   static_cast<size_t>(key) * D;
      const uint32_t src = tmem + lane_base + (wg == 0 ? Cfg::TM_DK : Cfg::TM_DV);
#pragma unroll
      for (int c = 0; c < D; c += 8) {
        uint32_t kk[8];
        tmem_ld_x8(src + c, kk);
        tmem_ld_wait();
        if (key < L) {
          *reinterpret_cast<uint4*>(dst + c) = make_uint4(kk[0], kk[1], kk[2], kk[3]);
          *reinterpret_cast<uint4*>(dst + c + 4) = make_uint4(kk[4], kk[5], kk[6], kk[7]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

// 128-row tiles per CTA (a function of the layer shape only: kv_bwd_reduce must know the chunk count)
int attn_bwd_tc_tiles(int S, int d) {
  (void)d;
  return S >= 2048 ? 8 : (S >= 512 ? 4 : 2);
}
int attn_bwd_tc_chunks(int S, int d) {
  const int rows = 128 * attn_bwd_tc_tiles(S, d);
  return (S + rows - 1) / rows;
}
bool attn_bwd_tc_supported(int d, int C) { return (d == 40 || d == 80) && C % 8 == 0; }

template <int D>
static int launch_attn_bwd_tc(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats, void* dQ,
                              float* part, int nchunk, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                              cudaStream_t stream, const float* img_row_weight) {
  using Cfg = BtCfg<D>;
  CUtensorMap tmQ, tmdO;
  if (make_tmap_3d(&tmQ, Q, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, 64, 128, 1, Swz::B128)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmdO, dO, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, 64, 128, 1, Swz::B128)) return PV_ERR_CUDA;
  BtParams p;
  p.kv_text = kv_text; p.kv_img = kv_img; p.stats = stats;
  p.dQ = static_cast<__nv_bfloat16*>(dQ); p.part = part;
  p.B = B; p.S = S; p.C = C; p.H = H; p.Lt = Lt; p.Li = Li; p.T = attn_bwd_tc_tiles(S, D);
  p.w_text = w_text; p.w_img = w_img;
  p.scale = 1.f / sqrtf(static_cast<float>(D));
  p.scale_log2e = p.scale * 1.4426950408889634f;
  p.img_row_weight = img_row_weight;
  const bool mask = img_row_weight != nullptr;
  auto kern = Lt == 77 ? (mask ? attn_bwd_tc_kernel<D, true, true> : attn_bwd_tc_kernel<D, true, false>)
                       : (mask ? attn_bwd_tc_kernel<D, false, true> : attn_bwd_tc_kernel<D, false, false>);
  PV_CUDA(set_max_smem_once(kern, Cfg::SMEM_BYTES));
  kern<<<dim3(nchunk, H, B), BT_THREADS, Cfg::SMEM_BYTES, stream>>>(tmQ, tmdO, p);
  PV_LAUNCHED();
  return PV_OK;
}

int dual_attn_bwd_tc(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats, void* dQ,
                     float* part, int nchunk, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                     cudaStream_t stream, const float* img_row_weight) {
  const int d = C / H;
  PV_REQUIRE(nchunk == attn_bwd_tc_chunks(S, d), "chunk count mismatch (%d for S=%d)", nchunk, S);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(dO) | reinterpret_cast<uintptr_t>(Q) | reinterpret_cast<uintptr_t>(dQ)) % 16 == 0,
             "pointers must be 16-byte aligned");
  if (d == 40) return launch_attn_bwd_tc<40>(dO, Q, kv_text, kv_img, stats, dQ, part, nchunk, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
  if (d == 80) return launch_attn_bwd_tc<80>(dO, Q, kv_text, kv_img, stats, dQ, part, nchunk, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
  PV_FAIL(PV_ERR_UNSUPPORTED, "head_dim %d: tcgen05 backward supports 40 / 80", d);
}

}  // namespace pv
