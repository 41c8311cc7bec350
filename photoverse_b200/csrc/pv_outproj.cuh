// photoverse_b200 -- the out projection (reference models/attention_processor.py:423) as a PHASE of the fused processor
// kernels: after a CTA pair has finished its attention units it runs, inside the same launch, the
//   Y[256 rows, 160 cols] = O[256 rows, C] * Wo[160 cols, C]^T + bias
// tiles of its own static (head group, unit range) share.  A tile's 256 rows of O were written (TMA stores) by the G
// pairs that own the row block's head groups; they announce a finished unit on a per-row-block counter in global memory
// and the tile's producer waits for that counter instead of for a kernel boundary.
//
// The pipeline is the persistent CTA-pair GEMM of pv_gemm3.cu (W slice split across the pair and resident for C <= 640,
// deep A ring, M = 256 cta_group::2 MMAs into double-buffered TMEM accumulators, bias / bf16 / TMA-store epilogue under
// the next tile's MMAs) with 3-D (channel, row, sample) coordinates so that tiles coincide with attention units.
//
// The same pipeline with the GEGLU epilogue (OP_EPI_GEGLU, pv_gemm3.cu only) computes a transformer block's feed-forward
// projection y = (x Wa^T + ba) * gelu(x Wg^T + bg) in one launch: the weight is packed so that the 160 rows of column group
// g are the 80 value rows of output columns [80 g, 80 g + 80) followed by their 80 gate rows, and each epilogue warp group
// holds both operands of its 40 outputs.  There a pair's tiles are a contiguous range of the flattened (group, unit)
// list, which may cross into the next column group (the resident W slice is then reloaded).
#pragma once
#include "pv_common.cuh"
#include "pv_softmax.cuh"

namespace pv {

constexpr int OP_BN = 160;
constexpr int OP_BK = 64;
constexpr int OP_A_BYTES = 128 * OP_BK * 2;
constexpr int OP_WH_BYTES = (OP_BN / 2) * OP_BK * 2;
constexpr int OP_MAX_STAGES = 8;
constexpr int OP_BAR_BYTES = (2 * OP_MAX_STAGES + 5) * 8;     // full[8] empty[8] acc_full[2] slot_free[2] w_full
constexpr int OP_W_FREE = 2 * OP_MAX_STAGES + 5;              // GEGLU only: w_free (resident W slice read by the last MMA)

constexpr int OP_EPI_BIAS = 0;     // D = acc + bias                                   (D: 160 columns per group)
constexpr int OP_EPI_GEGLU = 1;    // D = bf16(acc_a + b_a) * bf16(gelu(bf16(acc_g + b_g)))  (D: 80 columns per group)

template <int KB_RES, int NSTAGES>                            // resident K-blocks of the W half (0: streamed)
struct OutProjCfg {
  static constexpr bool WSTAT = KB_RES > 0;
  static constexpr int KB_RESIDENT = KB_RES;
  static constexpr int W_RES_BYTES = KB_RES * OP_WH_BYTES;
  static constexpr int STAGES = NSTAGES;
  static constexpr int STAGE_BYTES = WSTAT ? OP_A_BYTES : OP_A_BYTES + OP_WH_BYTES;
  // the resident W half comes FIRST: the fused kernels load it into the (already drained) X ring of the attention phase
  // while the last attention units are still running (op_preload_w)
  static constexpr int OFF_W = 0;
  static constexpr int OFF_STAGES = W_RES_BYTES;
  static constexpr int OFF_OST = OFF_STAGES + STAGES * STAGE_BYTES;
  static constexpr int OST_WARP_BYTES = 32 * 80 * 2;
  static constexpr int OFF_BIAS = OFF_OST + 8 * OST_WARP_BYTES;
  static constexpr int BYTES = OFF_BIAS + OP_BN * 4;
  static_assert(STAGES <= OP_MAX_STAGES, "barrier array");
};

struct OutProjArgs {
  const float* bias;       // [C] or nullptr
  unsigned int* sync;      // [2 * V] : ready[V] then seen[V]; all zero between launches (self-resetting)
  int G, MTP, C;
  int V;                   // units per column group = B * MTP
  int u0, u1;              // this pair's tiles: units [u0, u1) of column group g
                           // (OP_EPI_GEGLU: entries [u0, u1) of the flattened list, entry f = unit f % V of group f / V)
  int g;
  unsigned int ready_target;   // arrivals that complete a row block: (draining warps per unit) x G
  int w_preloaded;             // the resident W half has already been requested (op_preload_w)
  unsigned long long* trace;   // debug timeline (PV_TRACE builds)
  int trace_cap, trace_block;
};

__device__ __forceinline__ void op_mbar_init(uint64_t* pb) {
  uint64_t* full = pb;
  uint64_t* empty = full + OP_MAX_STAGES;
  uint64_t* acc_full = empty + OP_MAX_STAGES;
  uint64_t* slot_free = acc_full + 2;
  uint64_t* w_full = slot_free + 2;
  for (int s = 0; s < OP_MAX_STAGES; ++s) {
    mbar_init(&full[s], 1);
    mbar_init(&empty[s], 1);
  }
  for (int i = 0; i < 2; ++i) {
    mbar_init(&acc_full[i], 1);
    mbar_init(&slot_free[i], 16);
  }
  mbar_init(w_full, 1);
}

// The resident W half of column group g -> shared memory [0, W_RES_BYTES); completion on the LEADER's w_full barrier.
// One elected lane of the producer warp of BOTH CTAs calls it, either inside outproj_phase or earlier, as soon as that
// shared memory is free in both CTAs.
template <typename Cfg>
__device__ __forceinline__ void op_preload_w(uint8_t* smem, uint64_t* pb, const CUtensorMap* tmW, int g, uint32_t rank) {
  uint64_t* w_full = pb + 2 * OP_MAX_STAGES + 4;
  const uint32_t bar = mapa_u32(smem_u32(w_full), 0);
  const uint64_t pol_w = l2_policy_evict_last();           // every pair of the column group reads the same slice
  if (rank == 0) mbar_expect_tx(w_full, 2 * Cfg::W_RES_BYTES);
  for (int kb = 0; kb < Cfg::KB_RESIDENT; ++kb)
    tma_load_3d_2sm_hint(smem + Cfg::OFF_W + kb * OP_WH_BYTES, tmW, bar, kb * OP_BK, g * OP_BN + static_cast<int>(rank) * (OP_BN / 2), 0,
                         pol_w);
}

// An attention unit's O rows are in global memory: publish.  Called by ONE lane of a warp after
// cp.async.bulk.wait_group (full completion, not .read) has covered the warp's stores of that unit.
__device__ __forceinline__ void op_signal_unit(unsigned int* sync, int u) {
  asm volatile("fence.proxy.async;" ::: "memory");          // async-proxy (TMA) writes -> ordered before the release below
  asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(sync + u) : "memory");
}
// ... the same for units [u0, u0 + n) with one proxy fence and one gpu-scope fence
__device__ __forceinline__ void op_signal_units(unsigned int* sync, int u0, int n) {
  asm volatile("fence.proxy.async;" ::: "memory");
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
  for (int k = 0; k < n; ++k) asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(sync + u0 + k) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait_all() {             // groups complete AND their writes performed
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// The exact (erf) GELU of a bf16 value, in the expression of geglu_kernel (pv_backbone.cu) so that both round alike.
__device__ __forceinline__ float op_gelu_erf(float g) { return 0.5f * g * (1.f + erff(g * 0.70710678118654752f)); }

// The GEGLU epilogue (warps 4..11 of both CTAs).  Warp group w takes the value columns [40 w, 40 w + 40) and the gate
// columns [80 + 40 w, 80 + 40 w + 40) of the accumulator, i.e. output columns [80 g + 40 w, 80 g + 40 w + 40) of its 32
// rows; the staging tile is 32 rows x 80 bytes (16-byte stores of a quarter warp land in 8 distinct bank quads).
// Rounding points of the two-launch path (bf16 projection, then geglu_kernel): h_a and h_g are rounded to bf16 after the
// bias, gelu(h_g) is rounded to bf16, and the product of the two bf16 values is rounded once (fma.rn.bf16x2 with -0).
__device__ __forceinline__ void op_geglu_epilogue(uint8_t* smem_ost, float* sbias, uint64_t* acc_full, uint64_t* slot_free,
                                                  uint32_t tmem, const CUtensorMap* tmD, const OutProjArgs& a) {
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int w = (warp - 4) >> 2;
  const int q = warp & 3;
  const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
  uint8_t* ost = smem_ost + (warp - 4) * (32 * 80 * 2);
  float* gbias = sbias + 80 * w;                             // [0, 40): value bias, [40, 80): gate bias of this group
  const uint32_t bias_a = smem_u32(gbias);
  const uint32_t ost_a = smem_u32(ost);
  auto load_bias = [&](int g) {
    for (int c = q * 32 + lane; c < 80; c += 128)
      gbias[c] = a.bias ? a.bias[g * OP_BN + (c < 40 ? 40 * w + c : 80 + 40 * w + (c - 40))] : 0.f;
  };
  int gb = a.u0 < a.u1 ? a.u0 / a.V : 0;                    // group whose bias is in shared memory
  load_bias(gb);
  named_bar_sync(9 + w, 128);
  int i = 0;
  for (int f = a.u0; f < a.u1; ++f, ++i) {
    const int g = f / a.V;
    const int u = f - g * a.V;
    const int slot = i & 1;
    const int m0 = (2 * u + static_cast<int>(rank)) * 128;
    if (g != gb) {                                          // the range crossed into the next column group
      named_bar_sync(9 + w, 128);
      gb = g;
      load_bias(gb);
      named_bar_sync(9 + w, 128);
    }
    mbar_wait(&acc_full[slot], (i >> 1) & 1);
    tc_fence_after();
    uint32_t v[80];                                          // [0, 40): value accumulators, [40, 80): gate accumulators
    const uint32_t src = tlane + slot * OP_BN + 40 * w;
    tmem_ld32_raw(src, v);
    tmem_ld_x8(src + 32, *reinterpret_cast<uint32_t(*)[8]>(v + 32));
    tmem_ld32_raw(src + 80, v + 40);
    tmem_ld_x8(src + 112, *reinterpret_cast<uint32_t(*)[8]>(v + 72));
    tmem_ld_wait();
    tc_fence_before();
    __syncwarp();
    if (elect_one()) mbar_arrive_cluster(mapa_u32(smem_u32(&slot_free[slot]), 0));   // accumulator is in registers
    if (elect_one()) bulk_wait_read<0>();                // previous TMA store of this warp has read the staging tile
    __syncwarp();
    uint32_t y[20];                                          // word k = output columns 2k, 2k + 1
#pragma unroll
    for (int c = 0; c < 10; ++c) {
      float4 ba, bg;
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(ba.x), "=f"(ba.y), "=f"(ba.z), "=f"(ba.w) : "r"(bias_a + c * 16));
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(bg.x), "=f"(bg.y), "=f"(bg.z), "=f"(bg.w) : "r"(bias_a + 160 + c * 16));
      const float bav[4] = {ba.x, ba.y, ba.z, ba.w};
      const float bgv[4] = {bg.x, bg.y, bg.z, bg.w};
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int j = 4 * c + 2 * k;
        const uint32_t ha = pack_bf16x2(__uint_as_float(v[j]) + bav[2 * k], __uint_as_float(v[j + 1]) + bav[2 * k + 1]);
        const uint32_t hg = pack_bf16x2(__uint_as_float(v[40 + j]) + bgv[2 * k], __uint_as_float(v[41 + j]) + bgv[2 * k + 1]);
        const uint32_t ge = pack_bf16x2(op_gelu_erf(__uint_as_float(hg << 16)), op_gelu_erf(__uint_as_float(hg & 0xffff0000u)));
        uint32_t p;
        asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(p) : "r"(ha), "r"(ge), "r"(0x80008000u));
        y[2 * c + k] = p;
      }
    }
    const uint32_t row_a = ost_a + lane * 80;
#pragma unroll
    for (int c = 0; c < 5; ++c) st_shared_v4_a(row_a + c * 16, y[4 * c], y[4 * c + 1], y[4 * c + 2], y[4 * c + 3]);
    fence_proxy_async_smem();
    __syncwarp();
    if (elect_one()) {
      tma_store_3d(tmD, ost, 80 * g + 40 * w, m0 + q * 32, 0);
      bulk_commit();
    }
    __syncwarp();
  }
  if (elect_one()) bulk_wait_read<0>();
  __syncwarp();
}

// Runs the out-projection tiles of this pair.  Every thread of BOTH CTAs of the pair calls it after a CTA + cluster
// barrier that closed the attention phase (shared memory [0, Cfg::BYTES) and all 512 TMEM columns are free, the barriers
// at `pb` were initialised by op_mbar_init at kernel start and never used).  Roles: warp 0 producer (both CTAs),
// warp 1 MMA issuer (leader), warps 4..11 epilogue (both CTAs); other warps return at once.
// OP_EPI_GEGLU (plain GEMM only, a.sync == nullptr) also needs the w_free barrier at pb[OP_W_FREE], initialised with count 1.
// T: the 16-bit type of A, W and D (__nv_bfloat16 or __half; the GEGLU epilogue is bf16 only).
template <typename Cfg, int EPI = OP_EPI_BIAS, typename T = __nv_bfloat16>
__device__ __forceinline__ void outproj_phase(uint8_t* smem, uint64_t* pb, uint32_t tmem, const CUtensorMap* tmA,
                                              const CUtensorMap* tmW, const CUtensorMap* tmD, const OutProjArgs& a) {
  constexpr bool WSTAT = Cfg::WSTAT;
  constexpr bool GEGLU = EPI == OP_EPI_GEGLU;
  static_assert(!GEGLU || std::is_same<T, __nv_bfloat16>::value, "the GEGLU epilogue rounds like the bf16 geglu_kernel");
  constexpr int nst = Cfg::STAGES;
  uint64_t* full = pb;
  uint64_t* empty = full + OP_MAX_STAGES;
  uint64_t* acc_full = empty + OP_MAX_STAGES;
  uint64_t* slot_free = acc_full + 2;
  uint64_t* w_full = slot_free + 2;
  uint64_t* w_free = pb + OP_W_FREE;
  float* sbias = reinterpret_cast<float*>(smem + Cfg::OFF_BIAS);
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int kblocks = a.C / OP_BK;
  const int n0 = a.g * OP_BN;
  // tile index -> (column group, unit): the identity on a.g for the bias epilogue, the flattened list for GEGLU
  auto group_of = [&](int u) -> int {
    if constexpr (GEGLU) return u / a.V;
    else return a.g;
  };
  auto unit_of = [&](int u) -> int {
    if constexpr (GEGLU) return u - (u / a.V) * a.V;
    else return u;
  };

  if (warp == 0) {
    // ===================== producer (both CTAs): resident W half, then the A (= O) tiles as they become ready ==========
    A3Trace tr = a3_trace_init_raw(a.trace, a.trace_cap, 4, a.trace_block);
    a3_trace(tr, 50, 0);
    uint32_t it = 0;
    const uint64_t pol_a = l2_policy_evict_first();        // the A tiles are read once here
    const bool has_sync = a.sync != nullptr;     // nullptr: plain GEMM, every tile is ready (pv_gemm3.cu)
    const unsigned int target = a.ready_target;
    unsigned int* ready = a.sync;
    unsigned int* seen = a.sync + a.V;
    // Almost every tile's rows were announced long before this pair got here: probe 32 tiles at a time, one per lane
    // (one L2 round trip for all of them); only a tile that is not complete yet is waited for individually.
    auto probe32 = [&](int t0, uint32_t known) -> uint32_t {     // known: tiles of this group of 32 already seen complete
      const int u = a.u0 + t0 + lane;
      bool ok = false;
      if (u < a.u1 && !((known >> lane) & 1u)) {
        unsigned int v;
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ready + u) : "memory");
        ok = v >= target;
      }
      return known | __ballot_sync(0xffffffffu, ok);
    };
    // The proxy fence (generic-proxy acquire -> async-proxy TMA reads) also waits for this thread's TMA loads in flight
    // (~1 us): it is executed only right after an observation, never once per tile.
    uint32_t ready_mask = 0;
    if (has_sync && a.u0 < a.u1) {
      ready_mask = probe32(0, 0u);
      __syncwarp();
      a3_pair_time(a.trace, a.trace_block, 5);     // first probe answered
      asm volatile("fence.proxy.async;" ::: "memory");
    }
    if constexpr (WSTAT) {
      if (!a.w_preloaded && a.u0 < a.u1 && elect_one()) op_preload_w<Cfg>(smem, pb, tmW, a.g, rank);
      __syncwarp();
    }
    [[maybe_unused]] int gw = a.g;                // column group of the resident W slice
    [[maybe_unused]] uint32_t w_loads = 0;
    for (int u = a.u0; u < a.u1; ++u) {
      if constexpr (GEGLU && WSTAT) {
        if (group_of(u) != gw) {
          // the range crossed into the next column group: once the MMAs have read the old slice, load the new one
          mbar_wait(w_free, w_loads & 1);
          ++w_loads;
          gw = group_of(u);
          if (elect_one()) op_preload_w<Cfg>(smem, pb, tmW, gw, rank);
          __syncwarp();
        }
      }
      const int b = unit_of(u) / a.MTP;
      const int mt = 2 * (unit_of(u) - b * a.MTP) + static_cast<int>(rank);
      const int t = u - a.u0;
      if (has_sync) {
        bool observed = false;
        if ((t & 31) == 0 && t > 0) { ready_mask = probe32(t, 0u); observed = true; }
        if (!((ready_mask >> (t & 31)) & 1u)) {
          // not announced at the last look: look at the whole group of 32 again, then wait for this very tile
          ready_mask = probe32(t & ~31, ready_mask);
          observed = true;
          if (!((ready_mask >> (t & 31)) & 1u)) {
            if (lane == 0) {
              unsigned int v;
              uint32_t tries = 0;
              for (;;) {
                asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(ready + u) : "memory");
                if (v >= target) break;
                __nanosleep(32);
                if (++tries > 20000000u) __trap();    // > 1 s: a protocol bug must surface as an error, not hang the GPU
              }
            }
            ready_mask |= 1u << (t & 31);
          }
        }
        a3_trace(tr, 51, t);
        if (t == 0) a3_pair_time(a.trace, a.trace_block, 2);      // first tile ready
        if (u == a.u1 - 1) a3_pair_time(a.trace, a.trace_block, 6);   // last tile ready
        if (observed) {
          __syncwarp();
          asm volatile("fence.proxy.async;" ::: "memory");    // acquires above -> ordered before the TMA (async-proxy) reads
        }
      }
      for (int kb = 0; kb < kblocks; ++kb, ++it) {
        const int s = it % nst;
        const uint32_t ph = (it / nst) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        if (elect_one()) {
          uint8_t* a_dst = smem + Cfg::OFF_STAGES + s * Cfg::STAGE_BYTES;
          const uint32_t bar = mapa_u32(smem_u32(&full[s]), 0);
          if (rank == 0) mbar_expect_tx(&full[s], 2 * Cfg::STAGE_BYTES);
          tma_load_3d_2sm_hint(a_dst, tmA, bar, kb * OP_BK, mt * 128, b, pol_a);
          if constexpr (!WSTAT)
            tma_load_3d_2sm(a_dst + OP_A_BYTES, tmW, bar, kb * OP_BK, group_of(u) * OP_BN + static_cast<int>(rank) * (OP_BN / 2), 0);
        }
        __syncwarp();
      }
      a3_trace(tr, 52, t);
    }
    // 2 G producers (both CTAs of the G pairs that own a row block's column groups) have looked at ready[u]; the last one
    // to say so puts both words back to zero for the next launch.  Off the critical path: every load has been issued.
    if (has_sync) {
      for (int u = a.u0 + lane; u < a.u1; u += 32) {
        unsigned int old;
        asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(seen + u) : "memory");
        if (old == static_cast<unsigned int>(2 * a.G - 1)) {
          asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(ready + u), "r"(0u) : "memory");
          asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(seen + u), "r"(0u) : "memory");
        }
      }
    }
    a3_trace_done_raw(a.trace, tr, 4);
  } else if (warp == 1) {
    if (rank == 0) {
      // ===================== MMA issuer (leader): M = 256, N = 160 for both CTAs =====================
      constexpr uint32_t idesc = umma_idesc<T>(256, OP_BN);
      A3Trace tr = a3_trace_init_raw(a.trace, a.trace_cap, 5, a.trace_block);
      uint32_t it = 0;
      int i = 0;
      if constexpr (WSTAT) {
        if (a.u0 < a.u1) mbar_wait(w_full, 0);
      }
      [[maybe_unused]] int gw = a.g;
      [[maybe_unused]] uint32_t w_loads = 0;
      for (int u = a.u0; u < a.u1; ++u, ++i) {
        const int slot = i & 1;
        if (i >= 2) mbar_wait(&slot_free[slot], ((i >> 1) - 1) & 1);
        if constexpr (GEGLU && WSTAT) {
          if (group_of(u) != gw) {                 // the producer has reloaded the resident W slice for this group
            ++w_loads;
            gw = group_of(u);
            mbar_wait(w_full, w_loads & 1);
          }
        }
        tc_fence_after();
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const int s = it % nst;
          const uint32_t ph = (it / nst) & 1;
          mbar_wait(&full[s], ph);
          tc_fence_after();
          if (kb == 0) a3_trace(tr, 60, i);
          if (elect_one()) {
            const uint8_t* a_src = smem + Cfg::OFF_STAGES + s * Cfg::STAGE_BYTES;
            const uint64_t da = umma_desc_sw128(a_src);
            const uint64_t dw = umma_desc_sw128(WSTAT ? smem + Cfg::OFF_W + kb * OP_WH_BYTES : a_src + OP_A_BYTES);
#pragma unroll
            for (int k = 0; k < OP_BK / 16; ++k) umma_bf16_ss_2sm(tmem + slot * OP_BN, da + 2 * k, dw + 2 * k, idesc, (kb | k) != 0);
            umma_commit_2sm(&empty[s]);
            if (kb == kblocks - 1) umma_commit_2sm(&acc_full[slot]);
            if constexpr (GEGLU && WSTAT) {
              if (kb == kblocks - 1 && u + 1 < a.u1 && group_of(u + 1) != gw) umma_commit_2sm(w_free);
            }
          }
          __syncwarp();
        }
        a3_trace(tr, 61, i);
      }
      a3_trace_done_raw(a.trace, tr, 5);
    }
  } else if (GEGLU && warp >= 4 && warp < 12) {
    op_geglu_epilogue(smem + Cfg::OFF_OST, sbias, acc_full, slot_free, tmem, tmD, a);
  } else if (warp >= 4 && warp < 12) {
    // ===================== epilogue (both CTAs): group w handles columns [80 w, 80 w + 80) =====================
    const int w = (warp - 4) >> 2;
    const int q = warp & 3;
    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    uint8_t* ost = smem + Cfg::OFF_OST + (warp - 4) * Cfg::OST_WARP_BYTES;
    const uint32_t bias_a = smem_u32(sbias + 80 * w);
    const uint32_t ost_a = smem_u32(ost);
    // this group's 80 bias values (the attention phase owned the shared memory until the barrier before this call)
    for (int c = (warp & 3) * 32 + lane; c < 80; c += 128) sbias[80 * w + c] = a.bias ? a.bias[n0 + 80 * w + c] : 0.f;
    named_bar_sync(9 + w, 128);
    A3Trace tr = a3_trace_init_raw(a.trace, a.trace_cap, 6, a.trace_block);
    if (warp != 4) tr.base = nullptr;
    int i = 0;
    for (int u = a.u0; u < a.u1; ++u, ++i) {
      const int slot = i & 1;
      const int b = u / a.MTP;
      const int m0 = (2 * (u - b * a.MTP) + static_cast<int>(rank)) * 128;
      mbar_wait(&acc_full[slot], (i >> 1) & 1);
      tc_fence_after();
      a3_trace(tr, 70, i);
      uint32_t v[80];
      const uint32_t src = tlane + slot * OP_BN + 80 * w;
      tmem_ld32_raw(src, v);
      tmem_ld32_raw(src + 32, v + 32);
      tmem_ld16_raw(src + 64, v + 64);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      a3_trace(tr, 73, i);
      if (elect_one()) mbar_arrive_cluster(mapa_u32(smem_u32(&slot_free[slot]), 0));   // accumulator is in registers
      if (elect_one()) bulk_wait_read<0>();              // previous TMA store of this warp has read the staging tile
      __syncwarp();
      a3_trace(tr, 74, i);
      // + bias -> 16-bit pairs, in place (word 4c + k = columns 8c + 2k, 8c + 2k + 1).  The tensor core's operand reads and
      // the TMA writes leave little shared-memory bandwidth: the bias comes in 16-byte (broadcast) loads ...
#pragma unroll
      for (int c = 0; c < 10; ++c) {
        float4 b0, b1;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b0.x), "=f"(b0.y), "=f"(b0.z), "=f"(b0.w) : "r"(bias_a + c * 32));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b1.x), "=f"(b1.y), "=f"(b1.z), "=f"(b1.w) : "r"(bias_a + c * 32 + 16));
        v[4 * c + 0] = pack_x2<T>(__uint_as_float(v[8 * c + 0]) + b0.x, __uint_as_float(v[8 * c + 1]) + b0.y);
        v[4 * c + 1] = pack_x2<T>(__uint_as_float(v[8 * c + 2]) + b0.z, __uint_as_float(v[8 * c + 3]) + b0.w);
        v[4 * c + 2] = pack_x2<T>(__uint_as_float(v[8 * c + 4]) + b1.x, __uint_as_float(v[8 * c + 5]) + b1.y);
        v[4 * c + 3] = pack_x2<T>(__uint_as_float(v[8 * c + 6]) + b1.z, __uint_as_float(v[8 * c + 7]) + b1.w);
      }
      // ... and the 16-byte staging stores of a quarter warp must not collide: rows are 160 bytes apart (8 l mod 32
      // banks), so lanes 4..7 of every quarter write the NEXT 16-byte chunk of their row in the same instruction
      {
        const bool hi = (lane & 4) != 0;
        const uint32_t row_a = ost_a + lane * 160;
#pragma unroll
        for (int c = 0; c < 10; ++c) {
          const int c2 = (c + 1) % 10;
          const uint32_t w0 = hi ? v[4 * c2 + 0] : v[4 * c + 0];
          const uint32_t w1 = hi ? v[4 * c2 + 1] : v[4 * c + 1];
          const uint32_t w2 = hi ? v[4 * c2 + 2] : v[4 * c + 2];
          const uint32_t w3 = hi ? v[4 * c2 + 3] : v[4 * c + 3];
          st_shared_v4_a(row_a + (hi ? c2 : c) * 16, w0, w1, w2, w3);
        }
      }
      a3_trace(tr, 75, i);
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        tma_store_3d(tmD, ost, n0 + 80 * w, m0 + q * 32, b);
        bulk_commit();
      }
      __syncwarp();
      a3_trace(tr, 71, i);
    }
    if (elect_one()) bulk_wait_read<0>();
    __syncwarp();
    a3_trace(tr, 72, 0);
    a3_trace_done_raw(a.trace, tr, 6);
  }
}

}  // namespace pv
