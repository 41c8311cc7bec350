// photoverse_b200 -- fused Q-projection + dual-branch cross-attention, variant 4: persistent CTA PAIRS (cta_group::2).
//
// Same math, warp roles, TMEM maps and softmax code as pv_attn3.cu, but two CTAs of a cluster (two SMs) work on two
// consecutive 128-row tiles of the same (sample, head group) and drive ONE tcgen05.mma stream of M = 256, issued by the
// leader CTA.  Every B operand (Wq K-block, K tile, V^T tile) is split across the pair along N, so per CTA
//   * the Wq slice of the head group is 50 KB instead of 100 KB  -> for C = 320 it stays RESIDENT in shared memory next
//     to the K/V halves, and the freed space becomes a 7-stage X ring (the single-CTA W-stationary variant had room for
//     2 stages and was TMA-latency bound);  for C >= 640 the streamed W half costs 10 KB instead of 20 KB per K-block
//   * TMA ingest per K-block drops from 36 KB to 16 KB (C = 320) / 26 KB: the knock-out experiments of DESIGN.md 4.1
//     show per-SM TMA ingest (~44 B/clk), not the tensor pipe, bounds this kernel.
// Cross-CTA protocol: TMA loads of both CTAs complete on the LEADER's `full` / `w_full` barriers (.cta_group::2 form);
// bulk K/V copies complete locally and warp 3 relays "landed" to the leader; MMA completion is multicast to both CTAs
// (tcgen05.commit ... multicast::cluster); the softmax warps of both CTAs arrive (one elected lane per warp, remote
// mbarrier.arrive) on the leader's q_ready / p_ready / slot_free barriers.
#include "pv_common.cuh"
#include "pv_softmax.cuh"
#include "pv_outproj.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int A4_BM = 128;
constexpr int A4_BN = 160;
constexpr int A4_BK = 64;
constexpr int A4_KEYS = PV_KEYS_PAD;
constexpr int A4_IMG_OFF = PV_IMG_KEY_OFFSET;
constexpr int A4_THREADS = 384;      // 0 TMA, 1 projection MMA (leader), 2 attention MMA (leader), 3 K/V relay, 4..11 softmax
constexpr int A4_A_BYTES = A4_BM * A4_BK * 2;
constexpr int A4_WH_BYTES = (A4_BN / 2) * A4_BK * 2;     // this CTA's half of a Wq K-block
constexpr int A4_KB_WSTAT = 5;
constexpr int A4_MAX_STAGES = 8;

template <int D, bool WSTAT>
struct Attn4Cfg {
  static constexpr int HPC = A4_BN / D;
  static constexpr int D_PAD = (D + 15) / 16 * 16;
  static constexpr int NB = (D == 160) ? 80 : D_PAD;              // N of one PV MMA (pair-wide)
  static constexpr int NBLK = (D == 160) ? 2 : 1;
  static constexpr int KH_BYTES = (A4_KEYS / 2) * D_PAD * 2;       // 48 keys of a K tile
  static constexpr int VBLK_BYTES = (NB / 2) * A4_KEYS * 2;        // NB/2 dims of a V^T tile
  static constexpr int VH_BYTES = NBLK * VBLK_BYTES;
  static constexpr int KV_HEAD_BYTES = KH_BYTES + VH_BYTES;
  static constexpr int KV_BYTES = HPC * KV_HEAD_BYTES;
  static constexpr int STAGE_BYTES = WSTAT ? A4_A_BYTES : A4_A_BYTES + A4_WH_BYTES;
  static constexpr int STAGES = WSTAT ? 7 : (D == 40 ? 6 : 5);
  static constexpr int OFF_W = STAGES * STAGE_BYTES;
  static constexpr int W_RES_BYTES = WSTAT ? A4_KB_WSTAT * A4_WH_BYTES : 0;
  static constexpr int OFF_KV = OFF_W + W_RES_BYTES;
  static constexpr int OW = (D == 160) ? 80 : D;
  static constexpr int OST_WARP_BYTES = 32 * OW * 2;
  static constexpr int OFF_OST = OFF_KV + KV_BYTES;
  // fused out projection (second phase of the same launch, pv_outproj.cuh): Wo streamed with the O tiles, 7-stage ring
  using OP = OutProjCfg<0, 7>;
  static constexpr int OFF_BAR_1 = OFF_OST + 8 * OST_WARP_BYTES;
  static constexpr int OFF_BAR = ((OFF_BAR_1 > OP::BYTES ? OFF_BAR_1 : OP::BYTES) + 15) / 16 * 16;
  static constexpr int OP_BAR_OFF = 320;                           // phase-2 barriers inside the 512-byte barrier block
  static constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  static_assert(STAGES <= A4_MAX_STAGES, "barrier array");
  static constexpr uint32_t TM_SBUF0 = 320;
  static constexpr uint32_t TM_SBUF1 = 416;
  __host__ __device__ static constexpr uint32_t q_col(int j) { return D == 40 ? 40 * j + 16 : D == 80 ? 80 * j + 40 : 40; }
  __host__ __device__ static constexpr uint32_t o_col(int w) { return D == 40 ? 48 * w : D == 80 ? 80 * w : 0; }
};

struct Attn4Params {
  const uint8_t* Kp;
  const uint8_t* Vp;
  float* stats;            // optional [B,H,S,4]
  int S, C, H, Lt, Li;
  int G, MTP;              // head groups per sample (C/160), row-tile PAIRS per sample
  int V;                   // units per head group = B * MTP
  float w_text, w_img, scale_log2e;
  unsigned long long* trace;   // debug timeline (leader CTA 0 only)
  int trace_cap;
  // fused out projection (FUSE kernels only)
  const float* bias;           // [C] or nullptr
  unsigned int* sync;          // [2 * V] row-block counters, zero between launches (pv_outproj.cuh)
};

template <int D, bool LT77, bool WSTAT, bool FUSE, typename T>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(A4_THREADS, 1)
dual_attn_fwd_pair_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmWq,
                          const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmOa,
                          const __grid_constant__ CUtensorMap tmWo, const __grid_constant__ CUtensorMap tmY,
                          const Attn4Params p) {
  using Cfg = Attn4Cfg<D, WSTAT>;
  constexpr int HPC = Cfg::HPC;
  constexpr int D_PAD = Cfg::D_PAD;
  constexpr int nst = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* kv = smem + Cfg::OFF_KV;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* full = bars;                        // [STAGES]  (leader) both CTAs' X (+W half) stages landed
  uint64_t* empty = full + A4_MAX_STAGES;       // [STAGES]  multicast commit
  uint64_t* kv_full = empty + A4_MAX_STAGES;    // 1  local: this CTA's K/V halves landed
  uint64_t* kv_both = kv_full + 1;              // 1  (leader) both CTAs' K/V halves landed            count 2
  uint64_t* kv_free = kv_both + 1;              // 1  multicast commit
  uint64_t* q_full = kv_free + 1;               // [2] multicast commit: Q accumulators of a slot complete
  uint64_t* q_ready = q_full + 2;               // [2] (leader) packed bf16 Q in both CTAs' TMEM         count 16
  uint64_t* slot_free = q_ready + 2;            // [2] (leader) slot consumed in both CTAs               count 16
  uint64_t* s_full = slot_free + 2;             // [2] multicast commit, per softmax group
  uint64_t* p_ready = s_full + 2;               // [2] (leader)                                          count 8
  uint64_t* o_full = p_ready + 2;               // [2] multicast commit
  uint64_t* w_full = o_full + 2;                // 1  (leader) both halves of the resident Wq slice landed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int kblocks = p.C / A4_BK;
  // Static schedule: pair c serves head group g = c % G and a contiguous range [u0, u1) of that group's V = B * MTP
  // (sample, row-tile pair) units; CTA `rank` of the pair owns row tile 2 * pair + rank.
  const int pair = blockIdx.x >> 1;
  const int npairs = gridDim.x >> 1;
  const int g = pair % p.G;
  const int r_pair = pair / p.G;
  const int npair_g = (npairs - g + p.G - 1) / p.G;
  const int u0 = static_cast<int>((static_cast<long long>(p.V) * r_pair) / npair_g);
  const int u1 = static_cast<int>((static_cast<long long>(p.V) * (r_pair + 1)) / npair_g);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmWq);
    tma_prefetch_desc(&tmO);
    if constexpr (FUSE) {
      tma_prefetch_desc(&tmOa);
      tma_prefetch_desc(&tmWo);
      tma_prefetch_desc(&tmY);
      op_mbar_init(reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR + Cfg::OP_BAR_OFF));
    }
    for (int s = 0; s < A4_MAX_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(kv_full, 1);
    mbar_init(kv_both, 2);
    mbar_init(kv_free, 1);
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_ready[i], 16);
      mbar_init(&slot_free[i], 16);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 8);
      mbar_init(&o_full[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_2sm<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                 // the peer's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  // Everything above reads nothing a predecessor kernel may have written; the resident Wq slice (static weights) is
  // requested before the wait as well, so launch latency, TMEM allocation and that load overlap the previous kernel's tail.
  if constexpr (WSTAT) {
    if (warp == 0) {
      if (u0 < u1 && elect_one()) {
        const uint32_t bar = mapa_u32(smem_u32(w_full), 0);
        if (rank == 0) mbar_expect_tx(w_full, 2 * Cfg::W_RES_BYTES);
        for (int kb = 0; kb < A4_KB_WSTAT; ++kb)
          tma_load_3d_2sm(smem + Cfg::OFF_W + kb * A4_WH_BYTES, &tmWq, bar, kb * A4_BK, g * A4_BN + static_cast<int>(rank) * (A4_BN / 2), 0);
      }
      __syncwarp();
    }
  }
  pdl_wait();
  pdl_launch_dependents();

  // one elected lane per warp arrives on the LEADER CTA's copy of `bar` (after every lane's TMEM traffic is fenced)
  auto arrive_leader = [&](uint64_t* bar) {
    __syncwarp();
    if (elect_one()) mbar_arrive_cluster(mapa_u32(smem_u32(bar), 0));
    __syncwarp();
  };

  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");   // 128*88 + 256*208 == 384*168 (the launch allocation)
  if (warp == 0) {
    // ===================== TMA producer (both CTAs: own X rows, own halves of Wq / K / V^T) =====================
    uint32_t it = 0;
    int prev_b = -1;
    uint32_t kv_gen = 0;
    const uint64_t pol_x = l2_policy_evict_first();        // X is read once
    for (int u = u0; u < u1; ++u) {
      const int b = u / p.MTP;
      const int mt = 2 * (u - b * p.MTP) + static_cast<int>(rank);
      for (int kb = 0; kb < kblocks; ++kb, ++it) {
        const int s = it % nst;
        const uint32_t ph = (it / nst) & 1;
        mbar_wait(&empty[s], ph ^ 1);
        if (elect_one()) {
          uint8_t* a_dst = smem + s * Cfg::STAGE_BYTES;
          const uint32_t bar = mapa_u32(smem_u32(&full[s]), 0);
          if (rank == 0) mbar_expect_tx(&full[s], 2 * Cfg::STAGE_BYTES);
          tma_load_3d_2sm_hint(a_dst, &tmX, bar, kb * A4_BK, mt * A4_BM, b, pol_x);
          if constexpr (!WSTAT)
            tma_load_3d_2sm(a_dst + A4_A_BYTES, &tmWq, bar, kb * A4_BK, g * A4_BN + static_cast<int>(rank) * (A4_BN / 2), 0);
        }
        __syncwarp();
      }
      if (b != prev_b) {
        // this CTA's halves of the K / V^T tiles of (sample b, head group g): keys [48 rank, 48 rank + 48) of K,
        // dims [NB/2 rank, NB/2 rank + NB/2) of every N-block of V^T -- contiguous pieces of the packed UMMA images
        if (kv_gen > 0) mbar_wait(kv_free, (kv_gen - 1) & 1);
        if (elect_one()) {
          mbar_expect_tx(kv_full, Cfg::KV_BYTES);
          for (int j = 0; j < HPC; ++j) {
            const size_t tile = (static_cast<size_t>(b) * p.H + (g * HPC + j)) * (A4_KEYS * D_PAD * 2);
            uint8_t* kd = kv + j * Cfg::KV_HEAD_BYTES;
            for (int kc = 0; kc < D_PAD / 8; ++kc)
              bulk_load_1d(kd + kc * (48 * 16), p.Kp + tile + (static_cast<size_t>(kc) * A4_KEYS + 48 * rank) * 16, 48 * 16, kv_full);
            uint8_t* vd = kd + Cfg::KH_BYTES;
            for (int blk = 0; blk < Cfg::NBLK; ++blk)
              for (int kc = 0; kc < A4_KEYS / 8; ++kc)
                bulk_load_1d(vd + blk * Cfg::VBLK_BYTES + kc * ((Cfg::NB / 2) * 16),
                             p.Vp + tile + (static_cast<size_t>(kc) * D_PAD + blk * Cfg::NB + (Cfg::NB / 2) * rank) * 16,
                             (Cfg::NB / 2) * 16, kv_full);
          }
        }
        __syncwarp();
        ++kv_gen;
        prev_b = b;
      }
    }
  } else if (warp == 3) {
    // ===================== K/V relay: "my halves have landed" -> leader's kv_both =====================
    int prev_b = -1;
    uint32_t kv_gen = 0;
    for (int u = u0; u < u1; ++u) {
      const int b = u / p.MTP;
      if (b != prev_b) {
        mbar_wait(kv_full, kv_gen & 1);
        if (elect_one()) mbar_arrive_cluster(mapa_u32(smem_u32(kv_both), 0));
        __syncwarp();
        ++kv_gen;
        prev_b = b;
      }
    }
  } else if (warp == 1 && rank == 0) {
    // ===================== projection MMA issuer (leader): Q = X Wq^T for BOTH CTAs, M = 256, N = 160 =====================
    constexpr uint32_t idesc_q = umma_idesc<T>(2 * A4_BM, A4_BN);
    A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 0);
    uint32_t it = 0;
    int i = 0;
    if constexpr (WSTAT) {
      if (u0 < u1) mbar_wait(w_full, 0);
    }
    for (int u = u0; u < u1; ++u, ++i) {
      const int slot = i & 1;
      if (i >= 2) mbar_wait(&slot_free[slot], ((i >> 1) - 1) & 1);
      tc_fence_after();
      a3_trace(tr, 10, i);
      for (int kb = 0; kb < kblocks; ++kb, ++it) {
        const int s = it % nst;
        const uint32_t ph = (it / nst) & 1;
        mbar_wait(&full[s], ph);
        tc_fence_after();
        a3_trace(tr, 12, kb);
        if (elect_one()) {
          const uint8_t* a_src = smem + s * Cfg::STAGE_BYTES;
          const uint64_t da = umma_desc_sw128(a_src);
          const uint64_t dw = umma_desc_sw128(WSTAT ? smem + Cfg::OFF_W + kb * A4_WH_BYTES : a_src + A4_A_BYTES);
#pragma unroll
          for (int k = 0; k < A4_BK / 16; ++k)
            umma_bf16_ss_2sm(tmem + slot * A4_BN, da + 2 * k, dw + 2 * k, idesc_q, (kb | k) != 0);
          umma_commit_2sm(&empty[s]);
          if (kb == kblocks - 1) umma_commit_2sm(&q_full[slot]);
        }
        __syncwarp();
      }
      a3_trace(tr, 11, i);
    }
    a3_trace_done_raw(p.trace, tr, 0);
  } else if (warp == 2 && rank == 0) {
    // ===================== attention MMA issuer (leader), flat loop over the heads (see pv_attn3.cu) =====================
    constexpr uint32_t idesc_s = umma_idesc<T>(2 * A4_BM, A4_KEYS);
    constexpr uint32_t idesc_o = umma_idesc<T>(2 * A4_BM, Cfg::NB);
    A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 1);
    const int nheads = (u1 - u0) * HPC;
    int issued_qk = 0;
    uint32_t kv_gen = 0;
    int kv_b = -1;
    int q_units_ready = 0;
    auto unit_of = [&](int nn) { return nn / HPC; };
    auto issue_qk = [&](int nn) {
      const int i = unit_of(nn), j = nn - i * HPC;
      const uint32_t tslot = tmem + (i & 1) * A4_BN;
      const uint32_t sbuf = tmem + ((nn & 1) ? Cfg::TM_SBUF1 : Cfg::TM_SBUF0);
      const uint32_t k_half = smem_u32(kv + j * Cfg::KV_HEAD_BYTES);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < D_PAD / 16; ++k) {
          const uint64_t db = umma_desc(k_half + k * 2 * (48 * 16), 48 * 16, 128, UMMA_LAYOUT_NONE);
          umma_bf16_ts_2sm(sbuf, tslot + Cfg::q_col(j) + k * 8, db, idesc_s, k != 0);
        }
        umma_commit_2sm(&s_full[nn & 1]);
      }
      __syncwarp();
      a3_trace(tr, 20, nn);
    };
#pragma unroll 1
    for (int nn = 0; nn < nheads; ++nn) {
      const int i = unit_of(nn), j = nn - i * HPC;
      const int b = (u0 + i) / p.MTP;
      if (issued_qk <= nn) {
        if (q_units_ready <= i) { mbar_wait(&q_ready[i & 1], (i >> 1) & 1); q_units_ready = i + 1; }
        if (b != kv_b) { mbar_wait(kv_both, kv_gen & 1); ++kv_gen; kv_b = b; }
        tc_fence_after();
        issue_qk(nn);
        issued_qk = nn + 1;
      }
      if (nn + 1 < nheads && issued_qk == nn + 1) {
        const int i2 = unit_of(nn + 1);
        bool ok = (i2 == i);
        if (!ok && (u0 + i2) / p.MTP == kv_b) {
          if (q_units_ready > i2) ok = true;
          else if (mbar_test_wait(&q_ready[i2 & 1], (i2 >> 1) & 1)) { ok = true; q_units_ready = i2 + 1; }
        }
        if (ok) {
          tc_fence_after();
          issue_qk(nn + 1);
          issued_qk = nn + 2;
        }
      }
      const uint32_t w = nn & 1;
      a3_trace(tr, 25, nn);
      mbar_wait(&p_ready[w], (nn >> 1) & 1);
      tc_fence_after();
      a3_trace(tr, 26, nn);
      if (elect_one()) {
        const uint32_t tslot = tmem + (i & 1) * A4_BN;
        const uint32_t sbuf = tmem + (w ? Cfg::TM_SBUF1 : Cfg::TM_SBUF0);
        const uint32_t v_half = smem_u32(kv + j * Cfg::KV_HEAD_BYTES + Cfg::KH_BYTES);
#pragma unroll
        for (int blk = 0; blk < Cfg::NBLK; ++blk) {
#pragma unroll
          for (int k = 0; k < A4_KEYS / 16; ++k) {
            const uint64_t db = umma_desc(v_half + blk * Cfg::VBLK_BYTES + k * 2 * ((Cfg::NB / 2) * 16), (Cfg::NB / 2) * 16, 128,
                                          UMMA_LAYOUT_NONE);
            umma_bf16_ts_2sm(tslot + Cfg::o_col(w) + blk * Cfg::NB, sbuf + k * 8, db, idesc_o, k != 0);
          }
        }
        umma_commit_2sm(&o_full[w]);
        if (j == HPC - 1 && nn + 1 < nheads && (u0 + i + 1) / p.MTP != b) umma_commit_2sm(kv_free);
      }
      __syncwarp();
      a3_trace(tr, 21, nn);
    }
    a3_trace_done_raw(p.trace, tr, 1);
  }
  // the second phase runs every warp on the launch allocation again (blocks until the softmax warps have released theirs)
  if constexpr (FUSE) { __syncwarp(); asm volatile("setmaxnreg.inc.sync.aligned.u32 168;"); }
  } else {
    // ===================== softmax groups (warps 4..7 and 8..11) of BOTH CTAs: one thread per query row =====================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 208;");
    const int wg = (warp - 4) >> 2;
    const int q = warp & 3;                         // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;
    const uint32_t tlane = tmem + (static_cast<uint32_t>(q * 32) << 16);
    const uint32_t sbuf = tlane + (wg ? Cfg::TM_SBUF1 : Cfg::TM_SBUF0);
    const int Lt = p.Lt;
    const int Li = p.Li;
    const float cs = p.scale_log2e;
    A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 2 + wg);
    if (q != 0) tr.base = nullptr;
    PendingO pend;
    pend.valid = false;
    const uint64_t pol_o = l2_policy_evict_last();         // O is read back by the out projection: keep it in L2

    // O accumulator -> registers -> * row scale -> bf16 -> this warp's staging tile -> TMA store (clips rows >= S)
    uint8_t* ost = smem + Cfg::OFF_OST + ((warp - 4) * Cfg::OST_WARP_BYTES);
    auto stage_store = [&](const uint32_t* v, float oscale, int col0, int ncols) {
      const uint64_t sc2 = f2_pack(oscale, oscale);
#pragma unroll
      for (int c = 0; c < ncols / 8; ++c) {
        uint32_t w4[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float a, b2;
          f2_unpack(f2_mul(f2_pack(__uint_as_float(v[c * 8 + 2 * k]), __uint_as_float(v[c * 8 + 2 * k + 1])), sc2), a, b2);
          w4[k] = pack_x2<T>(a, b2);
        }
        st_shared_v4(ost + lane * (Cfg::OW * 2) + (col0 + c * 8) * 2, w4[0], w4[1], w4[2], w4[3]);
      }
    };
    auto drain = [&](const PendingO& po) {
      mbar_wait(&o_full[wg], po.parity);
      tc_fence_after();
#pragma unroll
      for (int h = 0; h < (D == 160 ? 2 : 1); ++h) {
        if (elect_one()) bulk_wait_read<0>();          // the previous TMA store of this warp has read the tile
        __syncwarp();
        if constexpr (D == 40) {
          uint32_t a[32], c8[8];
          tmem_ld_x32(po.taddr, a);
          tmem_ld_x8(po.taddr + 32, c8);
          tmem_ld_wait();
          stage_store(a, po.oscale, 0, 32);
          stage_store(c8, po.oscale, 32, 8);
        } else {
          uint32_t a[32], b2[32], c16[16];
          tmem_ld_x32(po.taddr + h * 80, a);
          tmem_ld_x32(po.taddr + h * 80 + 32, b2);
          tmem_ld_x16(po.taddr + h * 80 + 64, c16);
          tmem_ld_wait();
          stage_store(a, po.oscale, 0, 32);
          stage_store(b2, po.oscale, 32, 32);
          stage_store(c16, po.oscale, 64, 16);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (elect_one()) {
          tma_store_3d_hint(&tmO, ost, po.c0 + h * 80, po.r0, po.b, pol_o);
          bulk_commit();
        }
        __syncwarp();
      }
    };

    // Q of unit iu: fp32 accumulator -> packed bf16, written inside the columns this group has just read
    auto convert_unit = [&](int iu) {
      const int slot = iu & 1;
      const uint32_t tslot = tlane + slot * A4_BN;
      tc_fence_after();
      if constexpr (D == 40) {
        // group wg converts heads wg and wg + 2 : fp32 [40 j, 40 j + 40) -> bf16 [40 j + 16, 40 j + 40)
#pragma unroll
        for (int jj = 0; jj < 2; ++jj) {
          const int j = wg + 2 * jj;
          uint32_t a[32], c8[8], o[24];
          tmem_ld_x32(tslot + 40 * j, a);
          tmem_ld_x8(tslot + 40 * j + 32, c8);
          tmem_ld_wait();
          pack_pairs3<32, T>(a, o);
          pack_pairs3<8, T>(c8, o + 16);
          o[20] = o[21] = o[22] = o[23] = 0u;          // dims 40..47 pad the K = 48 contraction
          tmem_st_x16(tslot + 40 * j + 16, o);
          tmem_st_x8(tslot + 40 * j + 32, o + 16);
        }
      } else {
        // d=80: group wg converts head wg; d=160: dims [80 wg, 80 wg + 80) of the single head.
        // fp32 [80 wg, 80 wg + 80) -> bf16 [80 wg + 40, 80 wg + 80) (d=80) / [40 + 40 wg, 80 + 40 wg) (d=160)
        uint32_t a[32], b2[32], c16[16], o[40];
        tmem_ld_x32(tslot + wg * 80, a);
        tmem_ld_x32(tslot + wg * 80 + 32, b2);
        tmem_ld_x16(tslot + wg * 80 + 64, c16);
        tmem_ld_wait();
        pack_pairs3<32, T>(a, o);
        pack_pairs3<32, T>(b2, o + 16);
        pack_pairs3<16, T>(c16, o + 32);
        const uint32_t dstc = tslot + ((D == 80) ? (wg * 80 + 40) : (40 + wg * 40));
        tmem_st_x16(dstc, o);
        tmem_st_x16(dstc + 16, o + 16);
        tmem_st_x8(dstc + 32, o + 32);
      }
      tmem_st_wait();
      tc_fence_before();
      arrive_leader(&q_ready[slot]);
    };
    int converted = 0;              // units [0, converted) of this CTA have had their Q converted by this group

    int i = 0;
#pragma unroll 1
    for (int u = u0; u < u1; ++u, ++i) {
      const int slot = i & 1;
      const uint32_t tslot = tlane + slot * A4_BN;
      const int b = u / p.MTP;
      const int mt = 2 * (u - b * p.MTP) + static_cast<int>(rank);
      const int m0 = mt * A4_BM;

      if (converted <= i) {            // not converted ahead of time (see below): wait for the projection now
        mbar_wait(&q_full[slot], (i >> 1) & 1);
        a3_trace(tr, 30 + 10 * wg, i);
        convert_unit(i);
        converted = i + 1;
        a3_trace(tr, 31 + 10 * wg, i);
      }
      // this group's last head of the previous unit: its PV ran during the conversion above; draining it now (rather
      // than after the next softmax) returns the previous slot to the projection pipeline as early as possible
      if (pend.valid) {
        drain(pend);
        tc_fence_before();
        arrive_leader(&slot_free[pend.slot]);
        pend.valid = false;
        a3_trace(tr, 32 + 10 * wg, i);
      }

      const bool row_ok = (m0 + row) < p.S;
      bool had_head = false;

#pragma unroll 1
      for (int j = 0; j < HPC; ++j) {
        const int nn = i * HPC + j;
        if ((nn & 1) != wg) continue;
        had_head = true;
        const uint32_t par = (nn >> 1) & 1;
        mbar_wait(&s_full[wg], par);
        tc_fence_after();
        a3_trace(tr, 33 + 10 * wg, nn);
        uint32_t sr[A4_KEYS];                    // S row (fp32 bits), later the exponentials
        tmem_ld32_raw(sbuf, sr);
        tmem_ld32_raw(sbuf + 32, sr + 32);
        tmem_ld32_raw(sbuf + 64, sr + 64);
        tmem_ld_wait();
        float fi = 1.f, oscale = 1.f;
        bool text_on = true;
        {
        // Key-slot validity.  LT77 (the CLIP context length, every PhotoVerse caller): the text mask is a compile-time
        // constant, so padding slots 77..79 cost nothing; otherwise it is a per-slot runtime select.  The 16 image
        // slots are always masked at run time (Li = 1..16).
        auto tvalid = [&](int c) -> bool { if constexpr (LT77) return c < 77; else return c < Lt; };
        float mt2[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
        for (int c = 0; c < A4_IMG_OFF; ++c) {
          if (LT77 && c >= 77) continue;
          const float v = __uint_as_float(sr[c]);
          mt2[c & 3] = fmaxf(mt2[c & 3], LT77 ? v : (tvalid(c) ? v : -INFINITY));
        }
        float mi2[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int c = 0; c < A4_KEYS - A4_IMG_OFF; ++c)
          mi2[c & 1] = fmaxf(mi2[c & 1], (c < Li) ? __uint_as_float(sr[A4_IMG_OFF + c]) : -INFINITY);
        const float mts = fmaxf(fmaxf(mt2[0], mt2[1]), fmaxf(mt2[2], mt2[3])) * cs, mis = fmaxf(mi2[0], mi2[1]) * cs;
        // exponentials: e = 2^(s * cs - m) -- one FFMA2 per two keys, one MUFU.EX2 per key, one FADD2 per two keys
        const uint64_t cs2 = f2_pack(cs, cs);
        const uint64_t nmt2 = f2_pack(-mts, -mts), nmi2 = f2_pack(-mis, -mis);
        uint64_t lacc[2] = {f2_pack(0.f, 0.f), f2_pack(0.f, 0.f)};
        uint64_t iacc = f2_pack(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < A4_IMG_OFF / 2; ++k) {
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
          lacc[k & 1] = f2_add(lacc[k & 1], f2_pack(a, b2));
          sr[c] = __float_as_uint(a);
          sr[c + 1] = __float_as_uint(b2);
        }
        if (Li > 8) {
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const int c = A4_IMG_OFF + 2 * k;
            float a, b2;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmi2), a, b2);
            a = (2 * k < Li) ? fast_exp2(a) : 0.f;
            b2 = (2 * k + 1 < Li) ? fast_exp2(b2) : 0.f;
            iacc = f2_add(iacc, f2_pack(a, b2));
            sr[c] = __float_as_uint(a);
            sr[c + 1] = __float_as_uint(b2);
          }
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int c = A4_IMG_OFF + 2 * k;
            float a, b2;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmi2), a, b2);
            a = (2 * k < Li) ? fast_exp2(a) : 0.f;
            b2 = (2 * k + 1 < Li) ? fast_exp2(b2) : 0.f;
            iacc = f2_add(iacc, f2_pack(a, b2));
            sr[c] = __float_as_uint(a);
            sr[c + 1] = __float_as_uint(b2);
          }
#pragma unroll
          for (int c = A4_IMG_OFF + 8; c < A4_KEYS; ++c) sr[c] = 0u;
        }
        float l0, l1, l2, l3, li0, li1;
        f2_unpack(lacc[0], l0, l1);
        f2_unpack(lacc[1], l2, l3);
        f2_unpack(iacc, li0, li1);
        const float lt = (l0 + l1) + (l2 + l3);
        const float li = li0 + li1;
        const float at = p.w_text / lt;
        const float ai = p.w_img / li;
        if (p.stats != nullptr && row_ok) {
          const size_t idx = ((static_cast<size_t>(b) * p.H + (g * HPC + j)) * p.S + (m0 + row));
          reinterpret_cast<float4*>(p.stats)[idx] = make_float4(mts, lt, mis, li);
        }
        // P = [e_text | e_img * fi], O row scaled by `oscale` afterwards: the text segment stays unscaled.
        // w_text == 0 (image-only fusion branch) flips the roles.
        if (p.w_text != 0.f) { fi = ai / at; oscale = at; }
        else                 { text_on = false; fi = 1.f; oscale = ai; }
        }
        // the previous head of this group: its PV ran while the softmax above was computed.  It must leave TMEM
        // before P(nn) is published, because PV(nn) overwrites the group's O columns.
        if (pend.valid) {          // only heads of this same unit reach here (d = 40: the group's first head)
          drain(pend);
          pend.valid = false;
        }
        // P (bf16 pairs) over the first 48 columns of the S buffer, packed and stored 32 keys at a time
        {
          const uint64_t fi2 = f2_pack(fi, fi);
#pragma unroll
          for (int c = 0; c < A4_KEYS / 32; ++c) {
            uint32_t pk[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const int e = 32 * c + 2 * k;
              if (e < A4_IMG_OFF) {
                pk[k] = text_on ? pack_x2<T>(__uint_as_float(sr[e]), __uint_as_float(sr[e + 1])) : 0u;
              } else {
                float a, b2;
                f2_unpack(f2_mul(f2_pack(__uint_as_float(sr[e]), __uint_as_float(sr[e + 1])), fi2), a, b2);
                pk[k] = pack_x2<T>(a, b2);
              }
            }
            tmem_st_x16(sbuf + 16 * c, pk);
          }
        }
        tmem_st_wait();
        tc_fence_before();
        arrive_leader(&p_ready[wg]);
        a3_trace(tr, 34 + 10 * wg, nn);
        // While the PV MMA of this head and the QK^T of the next one run: convert the NEXT unit's Q if its projection
        // has already completed (the pair's projection pipeline runs well ahead), so that the attention issuer can
        // look ahead across the unit boundary and this group does not idle on s_full.
        if (converted == i + 1 && u + 1 < u1 && mbar_test_wait(&q_full[(i + 1) & 1], ((i + 1) >> 1) & 1)) {
          convert_unit(i + 1);
          converted = i + 2;
        }

        pend.valid = true;
        pend.c0 = g * A4_BN + j * D;
        pend.r0 = m0 + q * 32;
        pend.b = b;
        pend.taddr = tslot + Cfg::o_col(wg);
        pend.oscale = oscale;
        pend.parity = par;
        pend.slot = slot;
      }
      if (!had_head) {                                         // d = 160: the other group owns this unit's head
        arrive_leader(&slot_free[slot]);
        if (converted == i + 1 && u + 1 < u1 && mbar_test_wait(&q_full[(i + 1) & 1], ((i + 1) >> 1) & 1)) {
          convert_unit(i + 1);
          converted = i + 2;
        }
      }
    }
    if (pend.valid) drain(pend);
    if (elect_one()) bulk_wait_read<0>();            // the staging tiles are free (the stores may still be in flight)
    __syncwarp();
    a3_trace_done_raw(p.trace, tr, 2 + wg);
    if constexpr (FUSE) asm volatile("setmaxnreg.dec.sync.aligned.u32 168;");
  }

  if constexpr (FUSE) {
    // ===================== second phase: the out-projection tiles of this pair's (head group, unit range) =====================
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();
    tc_fence_after();
    if (warp >= 4) {
      // Every draining warp announces this pair's units once its O stores have COMPLETED (per-unit announcements inside
      // the attention loop stall the warps on the writer-side proxy fence); the first out-projection tile's loads and
      // MMAs run meanwhile.  A warp announces every unit, also those whose head its group did not drain: the counter
      // target is (all softmax warps of the pair) x G.
      if (elect_one()) {
        bulk_wait_all<0>();
        op_signal_units(p.sync, u0, u1 - u0);
      }
      __syncwarp();
    }
    OutProjArgs oa;
    oa.bias = p.bias;
    oa.sync = p.sync;
    oa.G = p.G; oa.MTP = p.MTP; oa.C = p.C; oa.V = p.V;
    oa.u0 = u0; oa.u1 = u1; oa.g = g;
    oa.w_preloaded = 0;
    oa.ready_target = static_cast<unsigned int>(16 * p.G);       // 8 softmax warps x 2 CTAs announce every unit
    oa.trace = p.trace; oa.trace_cap = p.trace_cap; oa.trace_block = 0;
    outproj_phase<typename Cfg::OP, OP_EPI_BIAS, T>(smem, reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR + Cfg::OP_BAR_OFF), tmem, &tmOa, &tmWo,
                                    &tmY, oa);
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();                 // neither CTA frees TMEM / exits while pair-wide MMAs or remote signals are in flight
  tc_fence_after();
  if (warp == 2) tmem_dealloc_2sm<512>(tmem);
}

extern unsigned long long* g_attn3_trace;
extern int g_attn3_trace_cap;

template <int D, bool LT77, bool WSTAT, bool FUSE, typename T>
static int launch_attn4(const CUtensorMap& tmX, const CUtensorMap& tmWq, const CUtensorMap& tmO, const CUtensorMap& tmOa,
                        const CUtensorMap& tmWo, const CUtensorMap& tmY, const Attn4Params& p, long long unit_pairs,
                        cudaStream_t stream) {
  using Cfg = Attn4Cfg<D, WSTAT>;
  auto kern = dual_attn_fwd_pair_kernel<D, LT77, WSTAT, FUSE, T>;
  PV_CUDA(set_max_smem_once(kern, Cfg::SMEM_BYTES));
  const long long max_pairs = sm_count() / 2;
  const int npairs = static_cast<int>(unit_pairs < max_pairs ? unit_pairs : max_pairs);
  PV_CUDA(launch_pdl(kern, dim3(2 * npairs), dim3(A4_THREADS), Cfg::SMEM_BYTES, stream, tmX, tmWq, tmO, tmOa, tmWo, tmY, p));
  PV_LAUNCHED();
  return PV_OK;
}

// Fused Q projection + dual-branch attention on CTA pairs; requires at least two row tiles per sample (S > 128).
// Wo == nullptr: attention only.  Otherwise the whole processor call in ONE launch: Y = O Wo^T + bo as a second phase
// (pv_outproj.cuh), O also left in global memory, `sync` = 2 * B * ceil(S / 256) zeroed counters (left zeroed).
int dual_attn_core_bf16_pair(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats, int B,
                             int S, int C, int H, int Lt, int Li, float w_text, float w_img, cudaStream_t stream,
                             const void* Wo, const float* bo, void* Y, unsigned int* sync, bool f16) {
  PV_REQUIRE(B > 0 && S > 0 && H > 0 && C % H == 0, "bad shape B=%d S=%d C=%d H=%d", B, S, C, H);
  const int d = C / H;
  PV_REQUIRE(d == 40 || d == 80 || d == 160, "head_dim %d unsupported (40/80/160)", d);
  PV_REQUIRE(C % A4_BN == 0 && C % A4_BK == 0, "C=%d must be a multiple of 320", C);
  PV_REQUIRE(Lt >= 1 && Lt <= A4_IMG_OFF && Li >= 1 && Li <= A4_KEYS - A4_IMG_OFF,
             "need 1 <= Lt <= %d and 1 <= Li <= %d (Lt=%d Li=%d)", A4_IMG_OFF, A4_KEYS - A4_IMG_OFF, Lt, Li);
  const bool fuse = Wo != nullptr;
  PV_REQUIRE(!fuse || (Y != nullptr && sync != nullptr), "fused out projection needs Y and the sync workspace");
  PV_REQUIRE((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(Wq) | reinterpret_cast<uintptr_t>(Kp) |
              reinterpret_cast<uintptr_t>(Vp) | reinterpret_cast<uintptr_t>(O) | reinterpret_cast<uintptr_t>(Wo) |
              reinterpret_cast<uintptr_t>(Y)) % 16 == 0, "pointers must be 16-byte aligned");
  CUtensorMap tmX, tmWq, tmO, tmOa, tmWo, tmY;
  if (make_tmap_3d(&tmX, X, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, A4_BK, A4_BM, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmWq, Wq, 2, C, C, 1, C * 2ull, static_cast<uint64_t>(C) * C * 2, A4_BK, A4_BN / 2, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmO, O, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, d == 160 ? 80 : d, 32, 1, Swz::None, f16)) return PV_ERR_CUDA;
  if (fuse) {
    if (make_tmap_3d(&tmOa, O, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, OP_BK, 128, 1, Swz::B128, f16)) return PV_ERR_CUDA;
    if (make_tmap_3d(&tmWo, Wo, 2, C, C, 1, C * 2ull, static_cast<uint64_t>(C) * C * 2, OP_BK, OP_BN / 2, 1, Swz::B128, f16)) return PV_ERR_CUDA;
    if (make_tmap_3d(&tmY, Y, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, 80, 32, 1, Swz::None, f16)) return PV_ERR_CUDA;
  } else {
    tmOa = tmO; tmWo = tmO; tmY = tmO;
  }
  Attn4Params p;
  p.Kp = static_cast<const uint8_t*>(Kp);
  p.Vp = static_cast<const uint8_t*>(Vp);
  p.stats = stats;
  p.S = S; p.C = C; p.H = H; p.Lt = Lt; p.Li = Li;
  p.G = C / A4_BN;
  const int MT = (S + A4_BM - 1) / A4_BM;
  p.MTP = (MT + 1) / 2;
  p.V = B * p.MTP;
  const long long unit_pairs = static_cast<long long>(p.V) * p.G;
  PV_REQUIRE(unit_pairs < (1ll << 30), "too many work units");
  p.w_text = w_text; p.w_img = w_img;
  p.trace = g_attn3_trace;
  p.trace_cap = g_attn3_trace_cap;
  p.scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(d));
  p.bias = bo;
  p.sync = sync;
#define PV_A4_LAUNCH(DD, LT, WS, FU)                                                                          \
  (f16 ? launch_attn4<DD, LT, WS, FU, __half>(tmX, tmWq, tmO, tmOa, tmWo, tmY, p, unit_pairs, stream)         \
       : launch_attn4<DD, LT, WS, FU, __nv_bfloat16>(tmX, tmWq, tmO, tmOa, tmWo, tmY, p, unit_pairs, stream))
#define PV_A4_LT(DD, WS, FU) (Lt == 77 ? PV_A4_LAUNCH(DD, true, WS, FU) : PV_A4_LAUNCH(DD, false, WS, FU))
  switch (d) {
    case 40:
      if (C == A4_KB_WSTAT * A4_BK) return fuse ? PV_A4_LT(40, true, true) : PV_A4_LT(40, true, false);
      return fuse ? PV_A4_LT(40, false, true) : PV_A4_LT(40, false, false);
    case 80:
      return fuse ? PV_A4_LT(80, false, true) : PV_A4_LT(80, false, false);
    default:
      return fuse ? PV_A4_LT(160, false, true) : PV_A4_LT(160, false, false);
  }
#undef PV_A4_LT
#undef PV_A4_LAUNCH
}

}  // namespace pv
