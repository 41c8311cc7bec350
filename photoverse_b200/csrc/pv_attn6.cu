// photoverse_b200 -- fused Q-projection + dual-branch cross-attention, variant 6: persistent CTA pairs with DECOUPLED
// roles, for head_dim 40 (C = 320: Wq slice resident) and head_dim 80 (X and Wq streamed together).
//
// The device timelines of variants 4 / 5 (tools/attn_trace.py, DESIGN.md 4.1) showed that at C = 320 the kernel is
// bound by the CUDA-core side, not by the tensor pipe or the TMA ingest: a softmax group spent ~2200 cycles on the
// softmax of a head, ~1000 on draining the previous O accumulator, ~400 per unit on converting Q, and idled ~40 % of
// the time on the chain P(n) -> PV(n) -> QK^T(n+2) -> S(n+2), whose every hop costs a few hundred cycles because the
// single issuer warp shares its scheduler and the SM's MIO path (mbarrier probes ~150-300 cycles) with the softmax warps.
// This variant removes every one of those serialisations:
//   * P goes to SHARED memory (12 key chunks x 128 rows x 16 B, canonical K-major no-swizzle layout) instead of over S in
//     tensor memory: an S buffer is free again as soon as its logits are in registers (`s_free`), so QK^T(n+2) is issued
//     while softmax(n) is still running and S(n+2) is waiting when the group comes back.  PV is an SS-form MMA.
//   * TWO issuer warps: warp 2 issues QK^T (waits q_ready / s_free only), warp 3 issues PV (waits p_ready / o_free only).
//     No ordering between the two streams is needed: every hazard is covered by a barrier (see the role comments).
//   * FOUR epilogue warps (one per TMEM lane quarter) convert Q (fp32 accumulator -> packed bf16, in place) and drain
//     the O accumulators (row scale from shared memory, bf16, staging tile, TMA store); they own q_ready / o_free /
//     slot_free.  The eight softmax warps do nothing but softmax.
// Shared-memory operands, TMEM maps, the pair protocol (cta_group::2, leader-side barriers, multicast commits) and the
// softmax arithmetic are those of pv_attn4.cu.
#include <type_traits>

#include "pv_common.cuh"
#include "pv_softmax.cuh"
#include "pv_outproj.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int A6_BM = 128;
constexpr int A6_BN = 160;
constexpr int A6_BK = 64;
constexpr int A6_KEYS = PV_KEYS_PAD;
constexpr int A6_IMG_OFF = PV_IMG_KEY_OFFSET;
constexpr int A6_THREADS = 512;           // 0 TMA, 1 projection MMA, 2 QK^T MMA, 3 PV MMA + K/V relay, 4..11 softmax, 12..15 epilogue
constexpr int A6_STAGES = 4;
constexpr int A6_A_BYTES = A6_BM * A6_BK * 2;                 // one X stage (this CTA's 128 rows)
constexpr int A6_WH_BYTES = (A6_BN / 2) * A6_BK * 2;          // this CTA's half of a Wq K-block
constexpr int A6_P_BYTES = A6_BM * A6_KEYS * 2;               // one group's P tile
static_assert(A6_KEYS == 96 && A6_IMG_OFF == 80, "written for 80 text + 16 image key slots");
constexpr uint32_t A6_TM_SBUF0 = 320;
constexpr uint32_t A6_TM_SBUF1 = 416;

// D = 40 (C = 320): 4 heads per 160-column group, the Wq slice of the group is RESIDENT (5 K-blocks) and only X streams.
// D = 80: 2 heads per group, X and the CTA's half of the Wq K-block stream together (26 KB per stage).
template <int D>
struct Attn6Cfg {
  static_assert(D == 40 || D == 80, "head_dim 40 or 80");
  static constexpr bool WSTAT = (D == 40);
  static constexpr int HPC = A6_BN / D;
  static constexpr int DPAD = (D + 15) / 16 * 16;
  static constexpr int KB_RES = 5;                                  // resident K-blocks (WSTAT: C = 320)
  static constexpr int STAGE_BYTES = WSTAT ? A6_A_BYTES : A6_A_BYTES + A6_WH_BYTES;
  static constexpr int KH_BYTES = (A6_KEYS / 2) * DPAD * 2;         // 48 keys of a K tile
  static constexpr int VH_BYTES = (DPAD / 2) * A6_KEYS * 2;         // DPAD/2 dims of a V^T tile
  static constexpr int KV_HEAD_BYTES = KH_BYTES + VH_BYTES;
  static constexpr int KV_BYTES = HPC * KV_HEAD_BYTES;
  static constexpr int OST_BYTES = 32 * D * 2;                      // one staging slab: 32 rows x D channels
  static constexpr int OFF_W = A6_STAGES * STAGE_BYTES;
  static constexpr int OFF_KV = OFF_W + (WSTAT ? KB_RES * A6_WH_BYTES : 0);
  static constexpr int OFF_OST = OFF_KV + KV_BYTES;                 // [epilogue warp][group] slabs
  static constexpr int OFF_P = OFF_OST + 4 * 2 * OST_BYTES;
  static constexpr int OFF_OSC = OFF_P + 2 * A6_P_BYTES;            // O row scales [group][parity][128] fp32
  // fused out projection (second phase of the same launch): C = 320 keeps its Wo half resident next to an 8-stage ring
  // of O tiles, C = 640 next to a 5-stage ring
  using OP = OutProjCfg<WSTAT ? 5 : 10, WSTAT ? 8 : 5>;
  static constexpr int OFF_BAR_1 = OFF_OSC + 2 * 2 * A6_BM * 4;
  static constexpr int OFF_BAR = ((OFF_BAR_1 > OP::BYTES ? OFF_BAR_1 : OP::BYTES) + 15) / 16 * 16;
  static constexpr int OP_BAR_OFF = 320;                            // phase-2 barriers inside the 512-byte barrier block
  static constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  // TMEM: packed bf16 Q of head j / O accumulator of softmax group w inside a 160-column slot
  __host__ __device__ static constexpr uint32_t q_col(int j) { return D == 40 ? 40 * j + 16 : 80 * j + 40; }
  __host__ __device__ static constexpr uint32_t o_col(int w) { return D == 40 ? 48 * w : 80 * w; }
};

struct Attn6Params {
  const uint8_t* Kp;
  const uint8_t* Vp;
  float* stats;            // optional [B,H,S,4]
  int S, C, H, Lt, Li;
  int G, MTP;              // head groups per sample (C/160), row-tile PAIRS per sample
  int V;                   // units per head group = B * MTP
  float w_text, w_img, scale_log2e;
  unsigned long long* trace;
  int trace_cap;
  int trace_block;         // which (leader) CTA writes the debug timeline
  // fused out projection (FUSE kernels only)
  const float* bias;       // [C] or nullptr
  unsigned int* sync;      // [2 * V] row-block counters, zero between launches (pv_outproj.cuh)
  int prefetch_s;          // softmax warps fetch the next head's S row under the current head's P pack
  int mufu_token;          // d = 40: the two softmax groups take turns on the exponentials
};

template <int D, bool LT77, bool FUSE, typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(A6_THREADS, 1)
dual_attn_fwd_pair_roles_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmWq,
                                const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmOa,
                                const __grid_constant__ CUtensorMap tmWo, const __grid_constant__ CUtensorMap tmY,
                                const Attn6Params p) {
  using Cfg = Attn6Cfg<D>;
  constexpr int A6_HPC = Cfg::HPC;
  constexpr int A6_DPAD = Cfg::DPAD;
  constexpr int A6_D = D;
  constexpr int A6_OFF_W = Cfg::OFF_W, A6_OFF_KV = Cfg::OFF_KV, A6_OFF_OST = Cfg::OFF_OST, A6_OFF_P = Cfg::OFF_P;
  constexpr int A6_OFF_OSC = Cfg::OFF_OSC, A6_OFF_BAR = Cfg::OFF_BAR;
  constexpr int A6_KH_BYTES = Cfg::KH_BYTES, A6_KV_HEAD_BYTES = Cfg::KV_HEAD_BYTES, A6_KV_BYTES = Cfg::KV_BYTES;
  constexpr int A6_OST_BYTES = Cfg::OST_BYTES;
  const int A6_KB = p.C / A6_BK;                  // K-blocks of the projection
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* kv = smem + A6_OFF_KV;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + A6_OFF_BAR);
  uint64_t* full = bars;                        // [STAGES] (leader) both CTAs' X stages landed
  uint64_t* empty = full + A6_STAGES;           // [STAGES] multicast commit
  uint64_t* w_full = empty + A6_STAGES;         // 1  (leader) both halves of the resident Wq slice landed
  uint64_t* kv_full = w_full + 1;               // 1  local: this CTA's K/V halves landed
  uint64_t* kv_both = kv_full + 1;              // 1  (leader) count 2
  uint64_t* kv_free = kv_both + 1;              // 1  multicast commit after the last PV of a sample
  uint64_t* q_full = kv_free + 1;               // [2] multicast commit: Q accumulators of a slot complete
  uint64_t* q_ready = q_full + 2;               // [2][4] (leader) packed bf16 Q of head j of the slot in both CTAs' TMEM: count 8
                                                //        (epilogue warps).  Per HEAD: the first QK^T of a unit does not wait for
                                                //        the conversion of the other heads (~450 cycles each, serial per warp)
  uint64_t* slot_free = q_ready + 8;            // [2] (leader) every O of the unit has left TMEM      count 8 (epilogue warps)
  uint64_t* s_full = slot_free + 2;             // [2] multicast commit, per softmax group
  uint64_t* s_free = s_full + 2;                // [2] (leader) S buffer in registers in both CTAs     count 8 (softmax warps)
  uint64_t* p_ready = s_free + 2;               // [2] (leader) P tile + row scales in shared memory   count 8 (softmax warps)
  uint64_t* o_full = p_ready + 2;               // [2] multicast commit: PV complete
  uint64_t* o_free = o_full + 2;                // [2] (leader) O accumulator in registers             count 8 (epilogue warps)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_free + 2);

  const long long t_entry = clock64();
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  // Static schedule (as pv_attn4.cu): pair c serves head group g = c % G and units [u0, u1) of that group's V = B * MTP
  // (sample, row-tile pair) units; CTA `rank` owns row tile 2 * pair_index + rank.
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  const int g = pair % p.G;
  const int r_pair = pair / p.G;
  const int npair_g = (npairs - g + p.G - 1) / p.G;
  const int u0 = static_cast<int>((static_cast<long long>(p.V) * r_pair) / npair_g);
  const int u1 = static_cast<int>((static_cast<long long>(p.V) * (r_pair + 1)) / npair_g);
  const int nunits = u1 - u0;
  const int nheads = nunits * A6_HPC;
  // K/V of one sample serve MTP consecutive units: first unit (relative to u0) of the second sample this pair touches
  const int first_end = (u0 / p.MTP + 1) * p.MTP - u0;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmWq);
    tma_prefetch_desc(&tmO);
    if constexpr (FUSE) {
      tma_prefetch_desc(&tmOa);
      tma_prefetch_desc(&tmWo);
      tma_prefetch_desc(&tmY);
      op_mbar_init(reinterpret_cast<uint64_t*>(smem + A6_OFF_BAR + Cfg::OP_BAR_OFF));
    }
    for (int s = 0; s < A6_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(w_full, 1);
    mbar_init(kv_full, 1);
    mbar_init(kv_both, 2);
    mbar_init(kv_free, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      for (int j = 0; j < 4; ++j) mbar_init(&q_ready[4 * i + j], 8);
      mbar_init(&slot_free[i], 8);
      mbar_init(&s_full[i], 1);
      mbar_init(&s_free[i], 8);
      mbar_init(&p_ready[i], 8);
      mbar_init(&o_full[i], 1);
      mbar_init(&o_free[i], 8);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                 // the peer's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;
  const long long t_sync = clock64();

  // Nothing above reads what a predecessor kernel may have written; the resident Wq slice (static weights) is requested
  // before the dependency wait as well.
  if constexpr (Cfg::WSTAT) {
    if (warp == 0) {
      if (nunits > 0 && elect_one()) {
        const uint32_t bar = mapa_u32(smem_u32(w_full), 0);
        if (rank == 0) mbar_expect_tx(w_full, 2 * Cfg::KB_RES * A6_WH_BYTES);
        for (int kb = 0; kb < Cfg::KB_RES; ++kb)
          tma_load_3d_2sm(smem + A6_OFF_W + kb * A6_WH_BYTES, &tmWq, bar, kb * A6_BK, g * A6_BN + static_cast<int>(rank) * (A6_BN / 2), 0);
      }
      __syncwarp();
    }
  }
  pdl_wait();
  pdl_launch_dependents();
  const long long t_pdl = clock64();
  a3_pair_time(p.trace, p.trace_block, 0);

  // one elected lane per warp arrives on the LEADER CTA's copy of `bar`
  auto arrive_leader = [&](uint64_t* bar) {
    __syncwarp();
    if (elect_one()) mbar_arrive_cluster(mapa_u32(smem_u32(bar), 0));
    __syncwarp();
  };

  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");   // 128*56 + 256*192 + 128*72 == 512*128 (the launch allocation)
    if (warp == 0) {
      // ===================== TMA producer (both CTAs: own X rows, own halves of K / V^T) =====================
      uint32_t it = 0;
      uint32_t kv_gen = 0;
      int kv_end = 0;
      const uint64_t pol_x = l2_policy_evict_first();      // X is read once
      for (int i = 0; i < nunits; ++i) {
        const int u = u0 + i;
        const int b = u / p.MTP;
        const int mt = 2 * (u - b * p.MTP) + static_cast<int>(rank);
        for (int kb = 0; kb < A6_KB; ++kb, ++it) {
          const int s = it % A6_STAGES;
          const uint32_t ph = (it / A6_STAGES) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          if (elect_one()) {
            const uint32_t bar = mapa_u32(smem_u32(&full[s]), 0);
            if (rank == 0) mbar_expect_tx(&full[s], 2 * Cfg::STAGE_BYTES);
            tma_load_3d_2sm_hint(smem + s * Cfg::STAGE_BYTES, &tmX, bar, kb * A6_BK, mt * A6_BM, b, pol_x);
            if constexpr (!Cfg::WSTAT)
              tma_load_3d_2sm(smem + s * Cfg::STAGE_BYTES + A6_A_BYTES, &tmWq, bar, kb * A6_BK,
                              g * A6_BN + static_cast<int>(rank) * (A6_BN / 2), 0);
          }
          __syncwarp();
        }
        if (i >= kv_end) {
          // this CTA's halves of the K / V^T tiles of (sample b, head group g): keys [48 rank, +48) of K, dims
          // [24 rank, +24) of V^T -- contiguous pieces of the packed UMMA images
          if (kv_gen > 0) mbar_wait(kv_free, (kv_gen - 1) & 1);
          if (elect_one()) {
            mbar_expect_tx(kv_full, A6_KV_BYTES);
            for (int j = 0; j < A6_HPC; ++j) {
              const size_t tile = (static_cast<size_t>(b) * p.H + (g * A6_HPC + j)) * (A6_KEYS * A6_DPAD * 2);
              uint8_t* kd = kv + j * A6_KV_HEAD_BYTES;
              for (int kc = 0; kc < A6_DPAD / 8; ++kc)
                bulk_load_1d(kd + kc * (48 * 16), p.Kp + tile + (static_cast<size_t>(kc) * A6_KEYS + 48 * rank) * 16, 48 * 16, kv_full);
              uint8_t* vd = kd + A6_KH_BYTES;
              for (int kc = 0; kc < A6_KEYS / 8; ++kc)
                bulk_load_1d(vd + kc * ((A6_DPAD / 2) * 16),
                             p.Vp + tile + (static_cast<size_t>(kc) * A6_DPAD + (A6_DPAD / 2) * rank) * 16, (A6_DPAD / 2) * 16, kv_full);
            }
          }
          __syncwarp();
          ++kv_gen;
          kv_end = (kv_end == 0) ? first_end : kv_end + p.MTP;
        }
      }
      if constexpr (FUSE) {
        // The last projection has consumed every X stage (wait for the commit of each stage's last fill): the ring is
        // dead from here on in BOTH CTAs (the leader's MMAs read both), and the resident Wo half of the second phase
        // lives inside it -- request it now, under the remaining attention units.
        static_assert(Cfg::OP::W_RES_BYTES <= A6_STAGES * Cfg::STAGE_BYTES, "resident Wo half must fit the X ring");
        if (nunits > 0) {
          for (int s = 0; s < A6_STAGES; ++s) {
            const uint32_t fills = (it + A6_STAGES - 1 - s) / A6_STAGES;     // loads that went to stage s
            if (fills > 0) mbar_wait(&empty[s], (fills - 1) & 1);
          }
          // the peer's ring must be dead too: its producer runs the same schedule, and the multicast commits that
          // complete my `empty` barriers complete the peer's copies at the same time
          if (elect_one()) op_preload_w<typename Cfg::OP>(smem, reinterpret_cast<uint64_t*>(smem + A6_OFF_BAR + Cfg::OP_BAR_OFF), &tmWo, g, rank);
          __syncwarp();
        }
      }
    } else if (warp == 1) {
      if (rank == 0) {
        // ===================== projection MMA issuer (leader): Q = X Wq^T for BOTH CTAs, M = 256, N = 160 =====================
        constexpr uint32_t idesc_q = umma_idesc<T>(2 * A6_BM, A6_BN);
        A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 0, p.trace_block);
        a3_trace(tr, 1, static_cast<int>(t_sync - t_entry));      // prologue: barrier init, TMEM allocation, cluster sync
        a3_trace(tr, 2, static_cast<int>(t_pdl - t_entry));       // ... + wait for the predecessor grid
        uint32_t it = 0;
        if constexpr (Cfg::WSTAT) {
          if (nunits > 0) mbar_wait(w_full, 0);
        }
        for (int i = 0; i < nunits; ++i) {
          const int slot = i & 1;
          if (i >= 2) mbar_wait(&slot_free[slot], ((i >> 1) - 1) & 1);
          tc_fence_after();
          a3_trace(tr, 10, i);
          for (int kb = 0; kb < A6_KB; ++kb, ++it) {
            const int s = it % A6_STAGES;
            const uint32_t ph = (it / A6_STAGES) & 1;
            mbar_wait(&full[s], ph);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t da = umma_desc_sw128(smem + s * Cfg::STAGE_BYTES);
              const uint64_t dw = umma_desc_sw128(Cfg::WSTAT ? smem + A6_OFF_W + kb * A6_WH_BYTES
                                                             : smem + s * Cfg::STAGE_BYTES + A6_A_BYTES);
#pragma unroll
              for (int k = 0; k < A6_BK / 16; ++k)
                umma_bf16_ss_2sm(tmem + slot * A6_BN, da + 2 * k, dw + 2 * k, idesc_q, (kb | k) != 0);
              umma_commit_2sm(&empty[s]);
              if (kb == A6_KB - 1) umma_commit_2sm(&q_full[slot]);
            }
            __syncwarp();
          }
          a3_trace(tr, 11, i);
        }
        a3_trace_done_raw(p.trace, tr, 0);
      }
    } else if (warp == 2) {
      if (rank == 0) {
        // ===================== QK^T issuer (leader): S(nn) = Q_head K_head^T, one head ahead of each softmax group ============
        // Needs: packed bf16 Q of the unit (q_ready), the sample's K/V (kv_both), S buffer nn & 1 read out (s_free).
        constexpr uint32_t idesc_s = umma_idesc<T>(2 * A6_BM, A6_KEYS);
        A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 1, p.trace_block);
        const uint64_t kdesc0 = umma_desc(smem_u32(kv), 48 * 16, 128, UMMA_LAYOUT_NONE);
        uint32_t kv_gen = 0;
        int kv_end = 0;
#pragma unroll 1
        for (int i = 0; i < nunits; ++i) {
          if (i >= kv_end) {
            mbar_wait(kv_both, kv_gen & 1);
            ++kv_gen;
            kv_end = (kv_end == 0) ? first_end : kv_end + p.MTP;
          }
          const uint32_t tslot = tmem + (i & 1) * A6_BN;
#pragma unroll 1
          for (int j = 0; j < A6_HPC; ++j) {
            const int nn = i * A6_HPC + j;
            mbar_wait(&q_ready[4 * (i & 1) + j], (i >> 1) & 1);
            if (nn >= 2) mbar_wait(&s_free[j & 1], ((nn - 2) >> 1) & 1);
            tc_fence_after();
            if (elect_one()) {
              const uint64_t kd = kdesc0 + static_cast<uint32_t>(j * (A6_KV_HEAD_BYTES >> 4));
#pragma unroll
              for (int k = 0; k < A6_DPAD / 16; ++k)
                umma_bf16_ts_2sm(tmem + ((j & 1) ? A6_TM_SBUF1 : A6_TM_SBUF0), tslot + Cfg::q_col(j) + k * 8,
                                 kd + k * ((2 * 48 * 16) >> 4), idesc_s, k != 0);
              umma_commit_2sm(&s_full[j & 1]);
            }
            __syncwarp();
            a3_trace(tr, 20, nn);
          }
        }
        a3_trace_done_raw(p.trace, tr, 1);
      }
    } else {
      // ===================== K/V relay (both CTAs) + PV issuer (leader): O(nn) = P(nn) V_head =====================
      // Needs: P tile + row scales in shared memory (p_ready), the group's O accumulator drained (o_free).  PV(nn)
      // overwrites TMEM columns that held the packed Q of heads 0 / 1 of the slot: their QK^T completed before the
      // softmax group could read S, i.e. before p_ready.
      constexpr uint32_t idesc_o = umma_idesc<T>(2 * A6_BM, A6_DPAD);
      const uint64_t vdesc0 = umma_desc(smem_u32(kv + A6_KH_BYTES), (A6_DPAD / 2) * 16, 128, UMMA_LAYOUT_NONE);
      const uint64_t pdesc0 = umma_desc(smem_u32(smem + A6_OFF_P), A6_BM * 16, 128, UMMA_LAYOUT_NONE);
      A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 6, p.trace_block);   // (role 6 belongs to phase 2 in the fused kernels)
      if (FUSE || rank != 0) tr.base = nullptr;
      uint32_t kv_gen = 0;
      int kv_end = 0;
#pragma unroll 1
      for (int i = 0; i < nunits; ++i) {
        if (i >= kv_end) {
          mbar_wait(kv_full, kv_gen & 1);                       // my halves of the sample's K / V^T have landed
          if (elect_one()) mbar_arrive_cluster(mapa_u32(smem_u32(kv_both), 0));
          __syncwarp();
          ++kv_gen;
          kv_end = (kv_end == 0) ? first_end : kv_end + p.MTP;
        }
        if (rank != 0) continue;
        const uint32_t tslot = tmem + (i & 1) * A6_BN;
        // d = 40: the O accumulators [48 w, +48) reach into the fp32 Q columns of the NEXT head (head 1: [40, 80), head 2:
        // [80, 120)), which the epilogue warps must have converted; they convert in head order, so the last head's
        // barrier covers all (long complete by the time a softmax has finished).
        mbar_wait(&q_ready[4 * (i & 1) + A6_HPC - 1], (i >> 1) & 1);
#pragma unroll 1
        for (int j = 0; j < A6_HPC; ++j) {
          const int nn = i * A6_HPC + j;
          const uint32_t w = j & 1;
          mbar_wait(&p_ready[w], (nn >> 1) & 1);
          if (nn >= 2) mbar_wait(&o_free[w], ((nn - 2) >> 1) & 1);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t pd = pdesc0 + static_cast<uint32_t>(w * (A6_P_BYTES >> 4));
            const uint64_t vd = vdesc0 + static_cast<uint32_t>(j * (A6_KV_HEAD_BYTES >> 4));
#pragma unroll
            for (int k = 0; k < A6_KEYS / 16; ++k)
              umma_bf16_ss_2sm(tslot + Cfg::o_col(w), pd + k * ((2 * A6_BM * 16) >> 4), vd + k * ((2 * (A6_DPAD / 2) * 16) >> 4), idesc_o, k != 0);
            umma_commit_2sm(&o_full[w]);
            // the next unit belongs to another sample: its K/V tiles may replace these once this PV has read them
            if (j == A6_HPC - 1 && i + 1 < nunits && i + 1 == kv_end) umma_commit_2sm(kv_free);
          }
          __syncwarp();
          a3_trace(tr, 21, nn);
        }
      }
      a3_trace_done_raw(p.trace, tr, 6);
    }
    // the second phase runs every warp on the launch allocation again (blocks until the softmax warps have released theirs)
    if constexpr (FUSE) { __syncwarp(); asm volatile("setmaxnreg.inc.sync.aligned.u32 128;"); }
  } else if (warp < 12) {
    // ===================== softmax groups (warps 4..7 and 8..11) of BOTH CTAs: one thread per query row =====================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 192;");
    const int wg = (warp - 4) >> 2;
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t sbuf = tlane + (wg ? A6_TM_SBUF1 : A6_TM_SBUF0);
    // 32-bit shared addresses kept in registers: barrier / tile addresses are used several times per head
    const uint32_t ptile_a = smem_u32(smem + A6_OFF_P + wg * A6_P_BYTES + row * 16);
    const uint32_t osc_a = smem_u32(smem + A6_OFF_OSC) + (wg * 2 * A6_BM + row) * 4;
    const uint32_t s_full_a = smem_u32(&s_full[wg]), o_full_a = smem_u32(&o_full[wg]);
    const uint32_t s_free_l = mapa_u32(smem_u32(&s_free[wg]), 0), p_ready_l = mapa_u32(smem_u32(&p_ready[wg]), 0);
    const bool text_on = (p.w_text != 0.f);        // image-only fusion branch: the text part of P is zero
    const int Lt = p.Lt;
    const int Li = p.Li;
    const float cs = p.scale_log2e;
    A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 2 + wg, p.trace_block);
    if (q != 0) tr.base = nullptr;
    int kv_end = 0;                                  // only to track the sample index of a unit without dividing per head
    int b = u0 / p.MTP - 1;

    // The S row of the group's NEXT head is fetched from tensor memory while the current head's P is packed (the
    // registers of a packed key chunk are dead): the TMEM round trip (~400 cycles) leaves the per-head chain
    // load -> max -> exponentials -> pack, which is what bounds the kernel at head_dim 40 (DESIGN.md 4.1).
    uint32_t sr[A6_KEYS];                            // S row (fp32 bits), later the exponentials
    const int gheads = nunits * (A6_HPC / 2);        // heads this group serves: nn = wg + 2 k, barrier parity k & 1
    const bool prefetch_s = p.prefetch_s != 0;
    const bool mufu_token = p.mufu_token != 0;
    auto release_s = [&]() {                         // the row is in registers: QK^T(nn + 2) may overwrite the S buffer
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (elect_one()) mbar_arrive_cluster(s_free_l);
    };
    if (gheads > 0) {
      mbar_wait_a(s_full_a, 0);
      tc_fence_after();
      tmem_ld32_raw(sbuf, sr);
      tmem_ld32_raw(sbuf + 32, sr + 32);
      tmem_ld32_raw(sbuf + 64, sr + 64);
      release_s();
    }

#pragma unroll 1
    for (int i = 0; i < nunits; ++i) {
      if (i >= kv_end) {
        ++b;
        kv_end = (kv_end == 0) ? first_end : kv_end + p.MTP;
      }
      const int mt = 2 * (u0 + i - b * p.MTP) + static_cast<int>(rank);
      const int m0 = mt * A6_BM;
      const bool row_ok = (m0 + row) < p.S;
#pragma unroll 1
      for (int jj = 0; jj < A6_HPC / 2; ++jj) {
        const int j = wg + 2 * jj;                   // this group's heads of the unit
        const int nn = i * A6_HPC + j;
        const uint32_t par = (nn >> 1) & 1;
        const bool has_next = (nn >> 1) + 1 < gheads;
        a3_trace(tr, 33 + 10 * wg, nn);
        float fi = 1.f, oscale = 1.f;
        {
          auto tvalid = [&](int c) -> bool { if constexpr (LT77) return c < 77; else return c < Lt; };
          float mt2[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
          for (int c = 0; c < A6_IMG_OFF; ++c) {
            if (LT77 && c >= 77) continue;
            const float v = __uint_as_float(sr[c]);
            mt2[c & 3] = fmaxf(mt2[c & 3], LT77 ? v : (tvalid(c) ? v : -INFINITY));
          }
          float mi2[2] = {-INFINITY, -INFINITY};
          if (Li <= 2) {
            mi2[0] = __uint_as_float(sr[A6_IMG_OFF]);
            if (Li > 1) mi2[1] = __uint_as_float(sr[A6_IMG_OFF + 1]);
          } else {
#pragma unroll
            for (int c = 0; c < A6_KEYS - A6_IMG_OFF; ++c)
              mi2[c & 1] = fmaxf(mi2[c & 1], (c < Li) ? __uint_as_float(sr[A6_IMG_OFF + c]) : -INFINITY);
          }
          const float mts = fmaxf(fmaxf(mt2[0], mt2[1]), fmaxf(mt2[2], mt2[3])) * cs, mis = fmaxf(mi2[0], mi2[1]) * cs;
          const uint64_t cs2 = f2_pack(cs, cs);
          const uint64_t nmt2 = f2_pack(-mts, -mts), nmi2 = f2_pack(-mis, -mis);
          uint64_t lacc[2] = {f2_pack(0.f, 0.f), f2_pack(0.f, 0.f)};
          uint64_t iacc = f2_pack(0.f, 0.f);
          // The exponentials are MUFU-bound (8 cycles per warp instruction) and the two groups' warps of a lane quarter
          // share one scheduler: a token (two producer/consumer named barriers) makes them take turns, so that one
          // warp's exponentials overlap the other's TMEM loads, max pass, packing and stores instead of its exponentials.
          // (d = 80 has one head per group and unit: there the unit's latency matters, not the MUFU throughput.)
          a3_trace(tr, 38 + 10 * wg, nn);
          if (D == 40 && mufu_token) {
            if (wg == 0) { if (nn >= 2) named_bar_sync(5 + q, 64); }
            else         { named_bar_sync(1 + q, 64); }
          }
          a3_trace(tr, 32 + 10 * wg, nn);
#pragma unroll
          for (int k = 0; k < A6_IMG_OFF / 2; ++k) {
            const int c = 2 * k;
            if (LT77 && c >= 77) { sr[c] = 0u; sr[c + 1] = 0u; continue; }
            float a, b2;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmt2), a, b2);
            a = fast_exp2(a);
            b2 = fast_exp2(b2);
            if constexpr (LT77) {
              if (c + 1 >= 77) b2 = 0.f;
            } else {
              a = tvalid(c) ? a : 0.f;
              b2 = tvalid(c + 1) ? b2 : 0.f;
            }
            sr[c] = __float_as_uint(a);
            sr[c + 1] = __float_as_uint(b2);
          }
          if (Li > 8) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
              const int c = A6_IMG_OFF + 2 * k;
              float a, b2;
              f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmi2), a, b2);
              a = (2 * k < Li) ? fast_exp2(a) : 0.f;
              b2 = (2 * k + 1 < Li) ? fast_exp2(b2) : 0.f;
              sr[c] = __float_as_uint(a);
              sr[c + 1] = __float_as_uint(b2);
            }
          } else if (Li <= 2) {                      // one image token (`token_index` given, the generate.py default) or two
            const int c = A6_IMG_OFF;
            float a, b2;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmi2), a, b2);
            a = fast_exp2(a);
            b2 = (Li > 1) ? fast_exp2(b2) : 0.f;
            sr[c] = __float_as_uint(a);
            sr[c + 1] = __float_as_uint(b2);
#pragma unroll
            for (int cc = A6_IMG_OFF + 2; cc < A6_KEYS; ++cc) sr[cc] = 0u;
          } else {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int c = A6_IMG_OFF + 2 * k;
              float a, b2;
              f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmi2), a, b2);
              a = (2 * k < Li) ? fast_exp2(a) : 0.f;
              b2 = (2 * k + 1 < Li) ? fast_exp2(b2) : 0.f;
              sr[c] = __float_as_uint(a);
              sr[c + 1] = __float_as_uint(b2);
            }
#pragma unroll
            for (int c = A6_IMG_OFF + 8; c < A6_KEYS; ++c) sr[c] = 0u;
          }
          if (D == 40 && mufu_token) {
            if (wg == 0) { named_bar_arrive(1 + q, 64); }
            else         { if (nn + 2 < nheads) named_bar_arrive(5 + q, 64); }
          }
          // Row sums AFTER the token has been handed on: inside the exponent loop every add waited for its two MUFU
          // results (in-order issue: ~15 cycles of XU bubble per pair, the phase took ~1150 cycles for 640 of MUFU work);
          // here they are FMA-pipe work that overlaps the other group's exponentials.  Masked slots hold zeros.
#pragma unroll
          for (int k = 0; k < A6_IMG_OFF / 2; ++k) {
            if (LT77 && 2 * k >= 77) continue;
            lacc[k & 1] = f2_add_v(lacc[k & 1], f2_pack(__uint_as_float(sr[2 * k]), __uint_as_float(sr[2 * k + 1])));
          }
          if (Li <= 2) {
            iacc = f2_pack(__uint_as_float(sr[A6_IMG_OFF]), __uint_as_float(sr[A6_IMG_OFF + 1]));
          } else {
#pragma unroll
            for (int k = 0; k < (A6_KEYS - A6_IMG_OFF) / 2; ++k)
              iacc = f2_add_v(iacc, f2_pack(__uint_as_float(sr[A6_IMG_OFF + 2 * k]), __uint_as_float(sr[A6_IMG_OFF + 2 * k + 1])));
          }
          float l0, l1, l2, l3, li0, li1;
          f2_unpack(lacc[0], l0, l1);
          f2_unpack(lacc[1], l2, l3);
          f2_unpack(iacc, li0, li1);
          const float lt = (l0 + l1) + (l2 + l3);
          const float li = li0 + li1;
          const float at = __fdividef(p.w_text, lt);      // l >= 1 (the max term), far from the ranges where the fast
          const float ai = __fdividef(p.w_img, li);       // division loses accuracy
          if (p.stats != nullptr && row_ok) {
            const size_t idx = ((static_cast<size_t>(b) * p.H + (g * A6_HPC + j)) * p.S + (m0 + row));
            reinterpret_cast<float4*>(p.stats)[idx] = make_float4(mts, lt, mis, li);
          }
          // P = [e_text | e_img * fi], O row scaled by `oscale` when it is drained: the text segment stays unscaled.
          // w_text == 0 (image-only fusion branch) flips the roles.
          if (text_on) { fi = __fdividef(ai, at); oscale = at; }
          else         { fi = 1.f; oscale = ai; }
        }
        a3_trace(tr, 36 + 10 * wg, nn);
        // the P tile and the row-scale slot of this parity are re-used: PV(nn - 2) has read the tile once o_full(nn - 2)
        // completed, and the epilogue has read the scales of head nn - 4 long before (it drained O(nn - 2) since).
        if (nn >= 2) mbar_wait_a(o_full_a, par ^ 1);
        st_shared_f32_a(osc_a + par * (A6_BM * 4), oscale);
        // key chunks [c0, c1) of this row (8 keys = 16 bytes each): text chunks unscaled, image chunks * fi
        const uint64_t fi2 = f2_pack(fi, fi);
        auto pack_chunks = [&](auto text_, auto c0_, auto c1_) {
          constexpr bool text = decltype(text_)::value;
          constexpr int c0 = decltype(c0_)::value, c1 = decltype(c1_)::value;
#pragma unroll
          for (int c = c0; c < c1; ++c) {
            uint32_t pk[4];
            if (c < A6_IMG_OFF / 8) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                pk[k] = text ? pack_x2<T>(__uint_as_float(sr[8 * c + 2 * k]), __uint_as_float(sr[8 * c + 2 * k + 1])) : 0u;
            } else {
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                float a, b2;
                f2_unpack(f2_mul(f2_pack(__uint_as_float(sr[8 * c + 2 * k]), __uint_as_float(sr[8 * c + 2 * k + 1])), fi2), a, b2);
                pk[k] = pack_x2<T>(a, b2);
              }
            }
            st_shared_v4_a(ptile_a + c * (A6_BM * 16), pk[0], pk[1], pk[2], pk[3]);
          }
        };
        using std::integral_constant;
        using std::true_type;
        using std::false_type;
        // S(nn + 2) was issued when this head's row reached the registers, ~2000 cycles ago: normally it is there.  If it
        // is not (pipeline fill, a late projection), P is not held back for it.  (The image-only fusion branch, a
        // training-time event, takes the plain path.)
        const bool pre = prefetch_s && has_next && text_on && __all_sync(0xffffffffu, mbar_test_wait_a(s_full_a, par ^ 1));
        a3_trace(tr, 37 + 10 * wg, pre ? 1 : 0);
        if (pre) {
          tc_fence_after();
          pack_chunks(true_type{}, integral_constant<int, 0>{}, integral_constant<int, 4>{});
          tmem_ld32_raw(sbuf, sr);                   // keys 0..31 are packed: their registers take the next row
          pack_chunks(true_type{}, integral_constant<int, 4>{}, integral_constant<int, 8>{});
          tmem_ld32_raw(sbuf + 32, sr + 32);
          pack_chunks(true_type{}, integral_constant<int, 8>{}, integral_constant<int, A6_KEYS / 8>{});
          tmem_ld32_raw(sbuf + 64, sr + 64);
        } else if (text_on) {
          pack_chunks(true_type{}, integral_constant<int, 0>{}, integral_constant<int, A6_KEYS / 8>{});
        } else {
          pack_chunks(false_type{}, integral_constant<int, 0>{}, integral_constant<int, A6_KEYS / 8>{});
        }
        fence_proxy_async_smem();                    // generic-proxy stores -> visible to the tensor core's operand reads
        __syncwarp();
        if (elect_one()) mbar_arrive_cluster(p_ready_l);
        a3_trace(tr, 34 + 10 * wg, nn);
        if (has_next) {
          if (!pre) {
            mbar_wait_a(s_full_a, par ^ 1);
            tc_fence_after();
            tmem_ld32_raw(sbuf, sr);
            tmem_ld32_raw(sbuf + 32, sr + 32);
            tmem_ld32_raw(sbuf + 64, sr + 64);
          }
          release_s();
          a3_trace(tr, 35 + 10 * wg, nn + 2);
        }
      }
    }
    a3_trace_done_raw(p.trace, tr, 2 + wg);
    if constexpr (FUSE) { __syncwarp(); asm volatile("setmaxnreg.dec.sync.aligned.u32 128;"); }
  } else {
    // ===================== epilogue warps 12..15 of BOTH CTAs: Q conversion + O drain for lane quarter q =====================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 72;");
    const int q = warp & 3;
    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    uint8_t* ost = smem + A6_OFF_OST + q * (2 * A6_OST_BYTES);
    const uint32_t osc_a = smem_u32(smem + A6_OFF_OSC) + (q * 32 + lane) * 4;
    int converted = 0, drained = 0;
    const uint64_t pol_o = l2_policy_evict_last();     // O is read back by the out projection: keep it in L2
    A3Trace etr = a3_trace_init_raw(p.trace, p.trace_cap, 7, p.trace_block);   // (role 7: phase 2 in the fused kernels)
    if (FUSE || q != 0) etr.base = nullptr;
    int kv_end_d = 0;                                // sample tracking for the drain stream
    int b_d = u0 / p.MTP - 1;
    int m0_d = 0;

    // Q of unit iu, fp32 accumulator -> packed bf16 in place.  d = 40: [40 j, +40) -> [40 j + 16, 40 j + 40), dims 40..47
    // zero (K = 48 contraction).  d = 80: [80 j, +80) -> [80 j + 40, 80 j + 80), upper half first so that every store
    // lands on columns whose fp32 source is already in registers.
    auto convert_unit = [&](int iu) {
      const uint32_t tslot = tlane + (iu & 1) * A6_BN;
      tc_fence_after();
      a3_trace(etr, 30, iu);
#pragma unroll
      for (int j = 0; j < A6_HPC; ++j) {
        if constexpr (D == 40) {
          uint32_t a[32], c8[8], o[24];
          tmem_ld_x32(tslot + 40 * j, a);
          tmem_ld_x8(tslot + 40 * j + 32, c8);
          tmem_ld_wait();
          pack_pairs3<32, T>(a, o);
          pack_pairs3<8, T>(c8, o + 16);
          o[20] = o[21] = o[22] = o[23] = 0u;
          tmem_st_x16(tslot + 40 * j + 16, o);
          tmem_st_x8(tslot + 40 * j + 32, o + 16);
        } else {
#pragma unroll
          for (int hh = 1; hh >= 0; --hh) {
            uint32_t a[32], c8[8], o[20];
            tmem_ld_x32(tslot + 80 * j + 40 * hh, a);
            tmem_ld_x8(tslot + 80 * j + 40 * hh + 32, c8);
            tmem_ld_wait();
            pack_pairs3<32, T>(a, o);
            pack_pairs3<8, T>(c8, o + 16);
            tmem_st_x16(tslot + 80 * j + 40 + 20 * hh, o);
            tmem_st_x4(tslot + 80 * j + 40 + 20 * hh + 16, o + 16);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        arrive_leader(&q_ready[4 * (iu & 1) + j]);
      }
      a3_trace(etr, 31, iu);
    };
    // O(nn): TMEM -> registers (accumulator released at once) -> * row scale -> bf16 -> staging slab -> TMA store
    auto drain_head = [&](int nn) {
      const int i = nn / A6_HPC, j = nn % A6_HPC;
      const uint32_t w = j & 1;
      const uint32_t par = (nn >> 1) & 1;
      if (j == 0) {                                  // first head of a unit: where its rows live
        if (i >= kv_end_d) {
          ++b_d;
          kv_end_d = (kv_end_d == 0) ? first_end : kv_end_d + p.MTP;
        }
        m0_d = (2 * (u0 + i - b_d * p.MTP) + static_cast<int>(rank)) * A6_BM;
      }
      tc_fence_after();
      a3_trace(etr, 80, nn);
      const uint32_t taddr = tlane + (i & 1) * A6_BN + Cfg::o_col(w);
      const float oscale = ld_shared_f32_a(osc_a + (w * 2 + par) * (A6_BM * 4));   // read before the release below: the slot is rewritten two heads on
      uint8_t* slab = ost + w * A6_OST_BYTES;
      if (elect_one()) bulk_wait_read<1>();          // the store that last read this slab (two drains ago) has finished
      __syncwarp();
      const uint64_t sc2 = f2_pack(oscale, oscale);
      auto stage = [&](const uint32_t* v, int col0, int ncols) {
#pragma unroll
        for (int c = 0; c < ncols / 8; ++c) {
          uint32_t w4[4];
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            float x0, x1;
            f2_unpack(f2_mul(f2_pack(__uint_as_float(v[c * 8 + 2 * k]), __uint_as_float(v[c * 8 + 2 * k + 1])), sc2), x0, x1);
            w4[k] = pack_x2<T>(x0, x1);
          }
          st_shared_v4(slab + lane * (A6_D * 2) + (col0 + c * 8) * 2, w4[0], w4[1], w4[2], w4[3]);
        }
      };
      auto release = [&]() {
        tc_fence_before();
        arrive_leader(&o_free[w]);                   // PV(nn + 2) may overwrite the accumulator
        if (j == A6_HPC - 1) arrive_leader(&slot_free[i & 1]);   // ... and the projection of unit i + 2 the whole slot
      };
#pragma unroll
      for (int ch = 0; ch < D / 40; ++ch) {          // 40 accumulator columns at a time
        uint32_t a[32], c8[8];
        tmem_ld_x32(taddr + 40 * ch, a);
        tmem_ld_x8(taddr + 40 * ch + 32, c8);
        tmem_ld_wait();
        if (ch == D / 40 - 1) release();
        stage(a, 40 * ch, 32);
        stage(c8, 40 * ch + 32, 8);
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        tma_store_3d_hint(&tmO, slab, g * A6_BN + j * A6_D, m0_d + q * 32, b_d, pol_o);
        bulk_commit();
      }
      __syncwarp();
      a3_trace(etr, 81, nn);
    };

    while (drained < nheads) {
      const int du = drained / A6_HPC;                   // unit of the next head to drain
      if (converted <= du) {                         // its Q is not even converted yet: nothing else can make progress
        mbar_wait(&q_full[converted & 1], (converted >> 1) & 1);
        convert_unit(converted);
        ++converted;
        continue;
      }
      if (converted < nunits && mbar_test_wait(&q_full[converted & 1], (converted >> 1) & 1)) {
        convert_unit(converted);                     // the next unit's projection has finished: convert ahead
        ++converted;
        continue;
      }
      const uint32_t w = drained & 1;
      if (mbar_try_wait_hint(&o_full[w], (drained >> 1) & 1, 64u)) {
        drain_head(drained);
        ++drained;
      }
    }
    if (elect_one()) bulk_wait_read<0>();             // the staging slabs are free (the stores may still be in flight)
    __syncwarp();
    a3_trace_done_raw(p.trace, etr, 7);
    if constexpr (FUSE) asm volatile("setmaxnreg.inc.sync.aligned.u32 128;");
  }

  if constexpr (FUSE) {
    // ===================== second phase: the out-projection tiles of this pair's (head group, unit range) =====================
    // Every MMA of the attention phase has completed (the epilogue warps drained the last accumulator), every TMA store
    // has read its staging slab: shared memory and tensor memory are free in both CTAs after this barrier.
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    a3_pair_time(p.trace, p.trace_block, 1);
    if (warp >= 12) {
      // The epilogue warps have nothing to do in the second phase: they wait for their O stores to COMPLETE and announce
      // this pair's units on the row-block counters.  Announcing per unit inside the attention loop costs ~2000 cycles
      // per unit on the warps that own q_ready / o_free (the writer-side proxy fence drains the stores in flight), and
      // the pairs that share a row block run in lockstep anyway.
      A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 7, p.trace_block);
      if ((warp & 3) != 0) tr.base = nullptr;
      a3_trace(tr, 84, 0);
      if (elect_one()) {
        bulk_wait_all<0>();
        op_signal_units(p.sync, u0, nunits);
      }
      __syncwarp();
      a3_trace(tr, 85, 0);
      a3_trace_done_raw(p.trace, tr, 7);
    }
    OutProjArgs oa;
    oa.bias = p.bias;
    oa.sync = p.sync;
    oa.G = p.G; oa.MTP = p.MTP; oa.C = p.C; oa.V = p.V;
    oa.u0 = u0; oa.u1 = u1; oa.g = g;
    oa.w_preloaded = 1;
    oa.ready_target = static_cast<unsigned int>(8 * p.G);        // 4 epilogue warps x 2 CTAs announce every unit
    oa.trace = p.trace; oa.trace_cap = p.trace_cap; oa.trace_block = p.trace_block;
    outproj_phase<typename Cfg::OP, OP_EPI_BIAS, T>(smem, reinterpret_cast<uint64_t*>(smem + A6_OFF_BAR + Cfg::OP_BAR_OFF), tmem, &tmOa, &tmWo,
                                    &tmY, oa);
    a3_pair_time(p.trace, p.trace_block, 3);     // the producer (thread 0's warp) has issued its last load
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                 // neither CTA frees TMEM / exits while pair-wide MMAs or remote signals are in flight
  tc_fence_after();
  a3_pair_time(p.trace, p.trace_block, 4);
  if (warp == 2) tmem_dealloc_2sm<512>(tmem);
}

extern unsigned long long* g_attn3_trace;
extern int g_attn3_trace_cap;
extern int g_opt_trace_block;
extern int g_opt_attn6_prefetch;
extern int g_opt_attn6_token;

template <int D, bool LT77, bool FUSE, typename T>
static int launch_attn6(const CUtensorMap& tmX, const CUtensorMap& tmWq, const CUtensorMap& tmO, const CUtensorMap& tmOa,
                        const CUtensorMap& tmWo, const CUtensorMap& tmY, const Attn6Params& p, long long unit_pairs,
                        cudaStream_t stream) {
  auto kern = dual_attn_fwd_pair_roles_kernel<D, LT77, FUSE, T>;
  PV_CUDA(set_max_smem_once(kern, Attn6Cfg<D>::SMEM_BYTES));
  const long long max_pairs = sm_count() / 2;
  const int npairs = static_cast<int>(unit_pairs < max_pairs ? unit_pairs : max_pairs);
  PV_CUDA(launch_pdl(kern, dim3(2 * npairs), dim3(A6_THREADS), Attn6Cfg<D>::SMEM_BYTES, stream, tmX, tmWq, tmO, tmOa, tmWo,
                     tmY, p));
  PV_LAUNCHED();
  return PV_OK;
}

// Same contract as dual_attn_core_bf16_pair (pv_attn4.cu), for head_dim 40 with C = 320 (resident Wq slice) and for
// head_dim 80, with at least two row tiles per sample.
bool dual_attn_pair_roles_supported(int S, int C, int H) {
  if (H <= 0 || C % H != 0 || S <= A6_BM || C % A6_BN != 0 || C % A6_BK != 0) return false;
  const int d = C / H;
  return (d == 40 && C == Attn6Cfg<40>::KB_RES * A6_BK) || d == 80;
}
// ... and the out projection as a second phase of the same launch (pv_outproj.cuh): C = 320 / 640 (resident Wo halves)
bool dual_attn_pair_roles_fused_supported(int S, int C, int H) {
  return dual_attn_pair_roles_supported(S, C, H) && (C == 320 || C == 640);
}

// Wo == nullptr: attention only, O = result.  Otherwise the whole processor call in ONE launch:
// Y = O Wo^T + bo, with O also left in global memory (saved for the backward pass) and `sync` = 2 * B * ceil(S / 256)
// zero-initialised counters that the kernel leaves zeroed.
int dual_attn_core_bf16_pair_roles(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats,
                                   int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                                   cudaStream_t stream, const void* Wo, const float* bo, void* Y, unsigned int* sync,
                                   bool f16) {
  PV_REQUIRE(B > 0 && dual_attn_pair_roles_supported(S, C, H), "needs head_dim 40 with C=320 or head_dim 80, S>128 (B=%d S=%d C=%d H=%d)",
             B, S, C, H);
  const bool fuse = Wo != nullptr;
  PV_REQUIRE(!fuse || (dual_attn_pair_roles_fused_supported(S, C, H) && Y != nullptr && sync != nullptr),
             "fused out projection needs C = 320 or 640, Y and the sync workspace");
  const int d = C / H;
  PV_REQUIRE(Lt >= 1 && Lt <= A6_IMG_OFF && Li >= 1 && Li <= A6_KEYS - A6_IMG_OFF,
             "need 1 <= Lt <= %d and 1 <= Li <= %d (Lt=%d Li=%d)", A6_IMG_OFF, A6_KEYS - A6_IMG_OFF, Lt, Li);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(Wq) | reinterpret_cast<uintptr_t>(Kp) |
              reinterpret_cast<uintptr_t>(Vp) | reinterpret_cast<uintptr_t>(O) | reinterpret_cast<uintptr_t>(Wo) |
              reinterpret_cast<uintptr_t>(Y)) % 16 == 0, "pointers must be 16-byte aligned");
  CUtensorMap tmX, tmWq, tmO, tmOa, tmWo, tmY;
  if (make_tmap_3d(&tmX, X, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, A6_BK, A6_BM, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmWq, Wq, 2, C, C, 1, C * 2ull, static_cast<uint64_t>(C) * C * 2, A6_BK, A6_BN / 2, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmO, O, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, d, 32, 1, Swz::None, f16)) return PV_ERR_CUDA;
  if (fuse) {
    if (make_tmap_3d(&tmOa, O, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, OP_BK, 128, 1, Swz::B128, f16)) return PV_ERR_CUDA;
    if (make_tmap_3d(&tmWo, Wo, 2, C, C, 1, C * 2ull, static_cast<uint64_t>(C) * C * 2, OP_BK, OP_BN / 2, 1, Swz::B128, f16)) return PV_ERR_CUDA;
    if (make_tmap_3d(&tmY, Y, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, 80, 32, 1, Swz::None, f16)) return PV_ERR_CUDA;
  } else {
    tmOa = tmO; tmWo = tmO; tmY = tmO;
  }
  Attn6Params p;
  p.Kp = static_cast<const uint8_t*>(Kp);
  p.Vp = static_cast<const uint8_t*>(Vp);
  p.stats = stats;
  p.S = S; p.C = C; p.H = H; p.Lt = Lt; p.Li = Li;
  p.G = C / A6_BN;
  const int MT = (S + A6_BM - 1) / A6_BM;
  p.MTP = (MT + 1) / 2;
  p.V = B * p.MTP;
  const long long unit_pairs = static_cast<long long>(p.V) * p.G;
  PV_REQUIRE(unit_pairs < (1ll << 28), "too many work units");
  p.w_text = w_text; p.w_img = w_img;
  p.trace = g_attn3_trace;
  p.trace_cap = g_attn3_trace_cap;
  p.trace_block = g_opt_trace_block;
  p.scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(d));
  p.bias = bo;
  p.sync = sync;
  p.prefetch_s = g_opt_attn6_prefetch;
  p.mufu_token = g_opt_attn6_token;
#define PV_A6_LAUNCH(DD, LT, FU)                                                                         \
  (f16 ? launch_attn6<DD, LT, FU, __half>(tmX, tmWq, tmO, tmOa, tmWo, tmY, p, unit_pairs, stream)        \
       : launch_attn6<DD, LT, FU, __nv_bfloat16>(tmX, tmWq, tmO, tmOa, tmWo, tmY, p, unit_pairs, stream))
  if (d == 40) {
    if (fuse) return Lt == 77 ? PV_A6_LAUNCH(40, true, true) : PV_A6_LAUNCH(40, false, true);
    return Lt == 77 ? PV_A6_LAUNCH(40, true, false) : PV_A6_LAUNCH(40, false, false);
  }
  if (fuse) return Lt == 77 ? PV_A6_LAUNCH(80, true, true) : PV_A6_LAUNCH(80, false, true);
  return Lt == 77 ? PV_A6_LAUNCH(80, true, false) : PV_A6_LAUNCH(80, false, false);
#undef PV_A6_LAUNCH
}

}  // namespace pv
