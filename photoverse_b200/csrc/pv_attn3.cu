// photoverse_b200 -- fused Q-projection + dual-branch cross-attention, variant 3: PERSISTENT, software-pipelined.
//
// Same math as pv_attn.cu / pv_attn2.cu (reference models/attention_processor.py:297, 307-322, 400-407, 411-420):
//   O[b, rows, g*160:(g+1)*160] = sum over the heads h of group g of  P_h V_h,   Q = X Wq^T on the fly,
//   P_h = [ w_text * softmax(Q_h K_text,h^T / sqrt(d)) | w_img * softmax(Q_h K_img,h^T / sqrt(d)) ]
//
// What is different: one CTA per SM walks a contiguous range of work units (unit = 128 query rows x 160 channels =
// 4 / 2 / 1 heads of d = 40 / 80 / 160) and keeps THREE pipelines running against each other:
//
//   warp 0        TMA producer      X [128x64] + Wq [160x64] K-blocks into a 4-stage ring (runs units ahead);
//                                   packed K / V^T tiles of the unit's heads, re-loaded only when (sample, head group)
//                                   changes -- consecutive units of a CTA are row tiles of the same (b, g)
//   warp 1        projection MMA    Q(unit i+1) = X Wq^T into TMEM slot (i+1)&1   ... while ...
//   warp 2        attention MMA     S = Q_h K_h^T and O = P_h V_h of unit i (A operands Q / P live in TMEM)
//   warps 4..7    softmax group 0   even heads: segment softmax straight out of TMEM, P written back in place,
//   warps 8..11   softmax group 1   odd heads : O drained -> scaled -> bf16 -> HBM; both groups convert Q to bf16
//
// TMEM (512 columns): two 160-column slots (Q accumulator of unit i, i+1; after conversion the slot holds the packed
// bf16 Q and, once the QK^T MMAs have consumed it, the O accumulators -- column maps in Attn3Cfg) + two 96-column
// S/P buffers at [320,416) and [416,512), one per softmax group.  Each group drains its O accumulator only after
// computing its NEXT softmax, so the PV MMA latency is hidden.
#include "pv_common.cuh"
#include "pv_softmax.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int A3_BM = 128;
constexpr int A3_BN = 160;
constexpr int A3_BK = 64;
constexpr int A3_KEYS = PV_KEYS_PAD;
constexpr int A3_IMG_OFF = PV_IMG_KEY_OFFSET;
constexpr int A3_WARPS = 12;       // 0 TMA, 1 projection MMA, 2 attention MMA, 3 spare, 4..7 / 8..11 softmax groups
constexpr int A3_THREADS = A3_WARPS * 32;
constexpr int A3_A_BYTES = A3_BM * A3_BK * 2;
constexpr int A3_W_BYTES = A3_BN * A3_BK * 2;
constexpr int A3_STAGE_BYTES = A3_A_BYTES + A3_W_BYTES;
constexpr int A3_MAX_STAGES = 4;
constexpr int A3_KB_WSTAT = 5;      // K-blocks of the resident Wq slice (C = 320)

// WSTAT (C = 320 only): the CTA's Wq slice [160 x 320] stays resident in shared memory for all of its units and only X
// is streamed -- 16 KB instead of 36 KB of TMA ingest per K-block.  Measured on B200 (tools/attn_dbg.py, dbg 7): the
// kernel is bound by per-SM TMA ingest (~44 B/clk), not by the tensor pipe or the softmax warps.
template <int D, bool WSTAT>
struct Attn3Cfg {
  static constexpr int HPC = A3_BN / D;
  static constexpr int D_PAD = (D + 15) / 16 * 16;
  static constexpr int QB_COLS = D_PAD / 2;
  static constexpr int KV_TILE_BYTES = A3_KEYS * D_PAD * 2;
  static constexpr int KV_BYTES = HPC * 2 * KV_TILE_BYTES;
  static constexpr int STAGES = WSTAT ? 2 : 3;      // measured: 3, 4, 5 stages give the same projection-pipeline rate
  static constexpr int STAGE_BYTES = WSTAT ? A3_A_BYTES : A3_STAGE_BYTES;
  static constexpr int OFF_W = STAGES * STAGE_BYTES;
  static constexpr int W_RES_BYTES = WSTAT ? A3_KB_WSTAT * A3_W_BYTES : 0;
  static constexpr int OFF_KV = OFF_W + W_RES_BYTES;
  static constexpr int OW = (D == 160) ? 80 : D;                 // channels per O staging tile / TMA store
  static constexpr int OST_WARP_BYTES = 32 * OW * 2;             // one [32 rows x OW] bf16 tile per softmax warp
  static constexpr int OFF_OST = OFF_KV + KV_BYTES;
  static constexpr int OFF_BAR = OFF_OST + 8 * OST_WARP_BYTES;
  static constexpr int SMEM_BYTES = OFF_BAR + 512 + 1024;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  static constexpr uint32_t TM_SBUF0 = 320;
  static constexpr uint32_t TM_SBUF1 = 416;
  // Column maps inside a 160-column slot.  The packed bf16 Q of head j is written INSIDE the fp32 columns the
  // converting softmax group has just read (no cross-group hazard); the O accumulator of group w re-uses columns
  // whose Q has already been consumed by the (in-order) QK^T MMAs issued before the first PV of the unit.
  //   d=40 : fp32 Q_j [40j,40j+40)  -> bf16 Q_j [40j+16,40j+40)   O(w) = [48w, 48w+48)
  //   d=80 : fp32 Q_j [80j,80j+80)  -> bf16 Q_j [80j+40,80j+80)   O(w) = [80w, 80w+80)
  //   d=160: fp32 Q   [0,160)       -> bf16 Q   [40,120)          O    = [0,160) (two N=80 halves)
  __host__ __device__ static constexpr uint32_t q_col(int j) { return D == 40 ? 40 * j + 16 : D == 80 ? 80 * j + 40 : 40; }
  __host__ __device__ static constexpr uint32_t o_col(int w) { return D == 40 ? 48 * w : D == 80 ? 80 * w : 0; }
};

struct Attn3Params {
  const uint8_t* Kp;
  const uint8_t* Vp;
  void* O;                 // [B,S,C]
  float* stats;            // optional [B,H,S,4]
  int S, C, H, Lt, Li;
  int G, MT;               // head groups per sample (C/160), row tiles per sample
  int V;                   // units per head group = B * MT
  long long units;         // B * G * MT
  float w_text, w_img, scale_log2e;
  unsigned long long* trace;   // optional [1 + 3*n] event buffer (CTA 0 only): count, then (event, index, clock) triples
  int trace_cap;
  const float* img_row_weight; // MASK kernels: [B, S] fp32 factor of each query row's image segment (ip_adapter_masks)
};

template <int D, bool LT77, bool WSTAT, typename T, bool MASK>
__global__ void __launch_bounds__(A3_THREADS, 1)
dual_attn_fwd_persistent_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmWq,
                                const __grid_constant__ CUtensorMap tmO, const Attn3Params p) {
  using Cfg = Attn3Cfg<D, WSTAT>;
  constexpr int HPC = Cfg::HPC;
  constexpr int D_PAD = Cfg::D_PAD;
  constexpr int nst = Cfg::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* kv = smem + Cfg::OFF_KV;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::OFF_BAR);
  uint64_t* full = bars;                        // [STAGES]  TMA -> projection MMA
  uint64_t* empty = full + A3_MAX_STAGES;       // [STAGES]
  uint64_t* kv_full = empty + A3_MAX_STAGES;    // 1
  uint64_t* kv_free = kv_full + 1;              // 1
  uint64_t* q_full = kv_free + 1;               // [2] projection MMA -> softmax groups (Q accumulator complete)
  uint64_t* q_ready = q_full + 2;               // [2] softmax groups -> attention MMA (packed bf16 Q in TMEM)
  uint64_t* slot_free = q_ready + 2;            // [2] softmax groups -> projection MMA (slot fully consumed)
  uint64_t* s_full = slot_free + 2;             // [2] per softmax group
  uint64_t* p_ready = s_full + 2;               // [2]
  uint64_t* o_full = p_ready + 2;               // [2]
  uint64_t* w_full = o_full + 2;                // 1  resident Wq slice loaded (WSTAT)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(w_full + 1);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int kblocks = p.C / A3_BK;
  // Static schedule: CTA c serves head group g = c % G (so its Wq slice and, mostly, its K/V tiles never change) and a
  // contiguous range [u0, u1) of that group's V = B * MT (sample, row tile) units.
  const int g = blockIdx.x % p.G;
  const int r_cta = blockIdx.x / p.G;
  const int ncta_g = (gridDim.x - g + p.G - 1) / p.G;
  const int u0 = static_cast<int>((static_cast<long long>(p.V) * r_cta) / ncta_g);
  const int u1 = static_cast<int>((static_cast<long long>(p.V) * (r_cta + 1)) / ncta_g);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmWq);
    tma_prefetch_desc(&tmO);
    for (int s = 0; s < A3_MAX_STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(kv_full, 1);
    mbar_init(kv_free, 1);
    mbar_init(w_full, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_ready[i], 256);
      mbar_init(&slot_free[i], 256);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_ready[i], 128);
      mbar_init(&o_full[i], 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<512>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = *tmem_slot;

  pdl_wait();                 // nothing above touches data a predecessor kernel may have written
  pdl_launch_dependents();

  // register re-distribution (warpgroup granular): the producer / issuer warps need few, the row threads many
  if (warp < 4) {
  asm volatile("setmaxnreg.dec.sync.aligned.u32 88;");   // 128*88 + 256*208 == 384*168 (the launch allocation)
  if (warp == 0) {
    // ===================== TMA producer =====================
    {
      uint32_t it = 0;
      int prev_b = -1;
      uint32_t kv_gen = 0;
      if constexpr (WSTAT) {
        if (u0 < u1 && elect_one()) {
          mbar_expect_tx(w_full, Cfg::W_RES_BYTES);
          for (int kb = 0; kb < A3_KB_WSTAT; ++kb)
            tma_load_3d(smem + Cfg::OFF_W + kb * A3_W_BYTES, &tmWq, w_full, kb * A3_BK, g * A3_BN, 0);
        }
        __syncwarp();
      }
      for (int u = u0; u < u1; ++u) {
        const int b = u / p.MT;
        const int mt = u - b * p.MT;
        for (int kb = 0; kb < kblocks; ++kb, ++it) {
          const int s = it % nst;
          const uint32_t ph = (it / nst) & 1;
          mbar_wait(&empty[s], ph ^ 1);
          if (elect_one()) {
            uint8_t* a_dst = smem + s * Cfg::STAGE_BYTES;
            mbar_expect_tx(&full[s], Cfg::STAGE_BYTES);
            tma_load_3d(a_dst, &tmX, &full[s], kb * A3_BK, mt * A3_BM, b);
            if constexpr (!WSTAT) tma_load_3d(a_dst + A3_A_BYTES, &tmWq, &full[s], kb * A3_BK, g * A3_BN, 0);
          }
          __syncwarp();
        }
        if (b != prev_b) {
          // K / V^T tiles of this (sample, head group): needed only once the projection above has completed
          if (kv_gen > 0) mbar_wait(kv_free, (kv_gen - 1) & 1);
          if (elect_one()) {
            mbar_expect_tx(kv_full, Cfg::KV_BYTES);
            for (int j = 0; j < HPC; ++j) {
              const size_t tile = (static_cast<size_t>(b) * p.H + (g * HPC + j)) * Cfg::KV_TILE_BYTES;
              bulk_load_1d(kv + (2 * j) * Cfg::KV_TILE_BYTES, p.Kp + tile, Cfg::KV_TILE_BYTES, kv_full);
              bulk_load_1d(kv + (2 * j + 1) * Cfg::KV_TILE_BYTES, p.Vp + tile, Cfg::KV_TILE_BYTES, kv_full);
            }
          }
          __syncwarp();
          ++kv_gen;
          prev_b = b;
        }
      }
    }
  } else if (warp == 1) {
    // ===================== projection MMA issuer: Q(unit) = X Wq^T  (M=128, N=160, K=C) =====================
    constexpr uint32_t idesc_q = umma_idesc<T>(A3_BM, A3_BN);
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
          const uint64_t dw = umma_desc_sw128(WSTAT ? smem + Cfg::OFF_W + kb * A3_W_BYTES : a_src + A3_A_BYTES);
#pragma unroll
          for (int k = 0; k < A3_BK / 16; ++k)
            umma_bf16_ss(tmem + slot * A3_BN, da + 2 * k, dw + 2 * k, idesc_q, (kb | k) != 0);
          umma_commit(&empty[s]);
          if (kb == kblocks - 1) umma_commit(&q_full[slot]);
        }
        __syncwarp();
        a3_trace(tr, 13, kb);
      }
      a3_trace(tr, 11, i);
    }
    a3_trace_done_raw(p.trace, tr, 0);
  } else if (warp == 2) {
    // ===================== attention MMA issuer =====================
    // Flat loop over the heads of all units of this CTA (head nn belongs to softmax group nn & 1 and uses that
    // group's S/P buffer).  Issue order  QK(nn+1) ; [wait P(nn)] ; PV(nn)  keeps one QK^T ahead of the softmax.
    // The tensor pipe executes the MMAs of this thread in order, which is what makes the TMEM re-use legal:
    //   S/P buffer of nn+2 <- overwritten only after PV(nn) has read P(nn);   O(w) columns <- overwritten only after
    //   the QK^T MMAs that read the packed Q living there.
    constexpr uint32_t idesc_s = umma_idesc<T>(A3_BM, A3_KEYS);
    constexpr uint32_t idesc_o = umma_idesc<T>(A3_BM, (D == 160) ? 80 : D_PAD);
    A3Trace tr = a3_trace_init_raw(p.trace, p.trace_cap, 1);
    const int nheads = (u1 - u0) * HPC;
    int issued_qk = 0;
    uint32_t kv_gen = 0;
    int kv_b = -1;                  // sample whose K/V tiles (of this CTA's head group) are resident
    int q_units_ready = 0;          // units [0, q_units_ready) have had their q_ready observed
    auto unit_of = [&](int nn) { return nn / HPC; };
    auto issue_qk = [&](int nn) {
      const int i = unit_of(nn), j = nn - i * HPC;
      const uint32_t tslot = tmem + (i & 1) * A3_BN;
      const uint32_t sbuf = tmem + ((nn & 1) ? Cfg::TM_SBUF1 : Cfg::TM_SBUF0);
      const uint32_t k_tile = smem_u32(kv + (2 * j) * Cfg::KV_TILE_BYTES);
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < D_PAD / 16; ++k) {
          const uint64_t db = umma_desc(k_tile + k * 2 * (A3_KEYS * 16), A3_KEYS * 16, 128, UMMA_LAYOUT_NONE);
          umma_bf16_ts(sbuf, tslot + Cfg::q_col(j) + k * 8, db, idesc_s, k != 0);
        }
        umma_commit(&s_full[nn & 1]);
      }
      __syncwarp();
      a3_trace(tr, 20, nn);
    };
#pragma unroll 1
    for (int nn = 0; nn < nheads; ++nn) {
      const int i = unit_of(nn), j = nn - i * HPC;
      const int b = (u0 + i) / p.MT;
      if (issued_qk <= nn) {
        // first head of a unit whose Q was not ready for look-ahead (or new K/V tiles): blocking
        if (q_units_ready <= i) { mbar_wait(&q_ready[i & 1], (i >> 1) & 1); q_units_ready = i + 1; }
        if (b != kv_b) { mbar_wait(kv_full, kv_gen & 1); ++kv_gen; kv_b = b; }
        tc_fence_after();
        issue_qk(nn);
        issued_qk = nn + 1;
      }
      if (nn + 1 < nheads && issued_qk == nn + 1) {
        const int i2 = unit_of(nn + 1);
        bool ok = (i2 == i);
        if (!ok && (u0 + i2) / p.MT == kv_b) {             // next unit, same K/V: look ahead only if Q is ready
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
        const uint32_t tslot = tmem + (i & 1) * A3_BN;
        const uint32_t sbuf = tmem + (w ? Cfg::TM_SBUF1 : Cfg::TM_SBUF0);
        const uint32_t v_tile = smem_u32(kv + (2 * j + 1) * Cfg::KV_TILE_BYTES);
#pragma unroll
        for (int k = 0; k < A3_KEYS / 16; ++k) {
          const uint64_t db = umma_desc(v_tile + k * 2 * (D_PAD * 16), D_PAD * 16, 128, UMMA_LAYOUT_NONE);
          umma_bf16_ts(tslot + Cfg::o_col(w), sbuf + k * 8, db, idesc_o, k != 0);
        }
        if constexpr (D == 160) {
#pragma unroll
          for (int k = 0; k < A3_KEYS / 16; ++k) {
            const uint64_t db = umma_desc(v_tile + 80 * 16 + k * 2 * (D_PAD * 16), D_PAD * 16, 128, UMMA_LAYOUT_NONE);
            umma_bf16_ts(tslot + 80, sbuf + k * 8, db, idesc_o, k != 0);
          }
        }
        umma_commit(&o_full[w]);
        // last head of the last unit that uses the resident K/V tiles -> the producer may overwrite them
        if (j == HPC - 1 && nn + 1 < nheads && (u0 + i + 1) / p.MT != b) umma_commit(kv_free);
      }
      __syncwarp();
      a3_trace(tr, 21, nn);
    }
    a3_trace_done_raw(p.trace, tr, 1);
  }
  } else {
    // ===================== softmax groups (warps 4..7 and 8..11): one thread per query row =====================
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
          tma_store_3d(&tmO, ost, po.c0 + h * 80, po.r0, po.b);
          bulk_commit();
        }
        __syncwarp();
      }
    };

    int i = 0;
#pragma unroll 1
    for (int u = u0; u < u1; ++u, ++i) {
      const int slot = i & 1;
      const uint32_t tslot = tlane + slot * A3_BN;
      const int b = u / p.MT;
      const int mt = u - b * p.MT;
      const int m0 = mt * A3_BM;

      // ---- Q: fp32 accumulator -> packed bf16, written inside the columns this group has just read ----
      mbar_wait(&q_full[slot], (i >> 1) & 1);
      tc_fence_after();
      a3_trace(tr, 30 + 10 * wg, i);
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
      mbar_arrive(&q_ready[slot]);
      a3_trace(tr, 31 + 10 * wg, i);
      // this group's last head of the previous unit: its PV ran during the conversion above; draining it now (rather
      // than after the next softmax) returns the previous slot to the projection pipeline as early as possible
      if (pend.valid) {
        drain(pend);
        tc_fence_before();
        mbar_arrive(&slot_free[pend.slot]);
        pend.valid = false;
        a3_trace(tr, 32 + 10 * wg, i);
      }

      const bool row_ok = (m0 + row) < p.S;
      bool had_head = false;
      // image segment weight of this row: w_img, times the row's mask weight in the MASK kernels (w_img * 1 is exact)
      float wi = p.w_img;
      if constexpr (MASK) wi *= row_ok ? __ldg(p.img_row_weight + static_cast<size_t>(b) * p.S + m0 + row) : 0.f;

#pragma unroll 1
      for (int j = 0; j < HPC; ++j) {
        const int nn = i * HPC + j;
        if ((nn & 1) != wg) continue;
        had_head = true;
        const uint32_t par = (nn >> 1) & 1;
        mbar_wait(&s_full[wg], par);
        tc_fence_after();
        a3_trace(tr, 33 + 10 * wg, nn);
        uint32_t sr[A3_KEYS];                    // S row (fp32 bits), later the exponentials
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
        for (int c = 0; c < A3_IMG_OFF; ++c) {
          if (LT77 && c >= 77) continue;
          const float v = __uint_as_float(sr[c]);
          mt2[c & 3] = fmaxf(mt2[c & 3], LT77 ? v : (tvalid(c) ? v : -INFINITY));
        }
        float mi2[2] = {-INFINITY, -INFINITY};
#pragma unroll
        for (int c = 0; c < A3_KEYS - A3_IMG_OFF; ++c)
          mi2[c & 1] = fmaxf(mi2[c & 1], (c < Li) ? __uint_as_float(sr[A3_IMG_OFF + c]) : -INFINITY);
        const float mts = fmaxf(fmaxf(mt2[0], mt2[1]), fmaxf(mt2[2], mt2[3])) * cs, mis = fmaxf(mi2[0], mi2[1]) * cs;
        // exponentials: e = 2^(s * cs - m) -- one FFMA2 per two keys, one MUFU.EX2 per key, one FADD2 per two keys
        const uint64_t cs2 = f2_pack(cs, cs);
        const uint64_t nmt2 = f2_pack(-mts, -mts), nmi2 = f2_pack(-mis, -mis);
        uint64_t lacc[2] = {f2_pack(0.f, 0.f), f2_pack(0.f, 0.f)};
        uint64_t iacc = f2_pack(0.f, 0.f);
#pragma unroll
        for (int k = 0; k < A3_IMG_OFF / 2; ++k) {
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
            const int c = A3_IMG_OFF + 2 * k;
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
            const int c = A3_IMG_OFF + 2 * k;
            float a, b2;
            f2_unpack(f2_fma(f2_pack(__uint_as_float(sr[c]), __uint_as_float(sr[c + 1])), cs2, nmi2), a, b2);
            a = (2 * k < Li) ? fast_exp2(a) : 0.f;
            b2 = (2 * k + 1 < Li) ? fast_exp2(b2) : 0.f;
            iacc = f2_add(iacc, f2_pack(a, b2));
            sr[c] = __float_as_uint(a);
            sr[c + 1] = __float_as_uint(b2);
          }
#pragma unroll
          for (int c = A3_IMG_OFF + 8; c < A3_KEYS; ++c) sr[c] = 0u;
        }
        float l0, l1, l2, l3, li0, li1;
        f2_unpack(lacc[0], l0, l1);
        f2_unpack(lacc[1], l2, l3);
        f2_unpack(iacc, li0, li1);
        const float lt = (l0 + l1) + (l2 + l3);
        const float li = li0 + li1;
        const float at = p.w_text / lt;
        const float ai = wi / li;
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
          for (int c = 0; c < A3_KEYS / 32; ++c) {
            uint32_t pk[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) {
              const int e = 32 * c + 2 * k;
              if (e < A3_IMG_OFF) {
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
        mbar_arrive(&p_ready[wg]);
        a3_trace(tr, 34 + 10 * wg, nn);

        pend.valid = true;
        pend.c0 = g * A3_BN + j * D;
        pend.r0 = m0 + q * 32;
        pend.b = b;
        pend.taddr = tslot + Cfg::o_col(wg);
        pend.oscale = oscale;
        pend.parity = par;
        pend.slot = slot;
      }
      if (!had_head) mbar_arrive(&slot_free[slot]);      // d = 160: the other group owns this unit's head
    }
    if (pend.valid) drain(pend);
    if (elect_one()) bulk_wait_read<0>();
    __syncwarp();
    a3_trace_done_raw(p.trace, tr, 2 + wg);
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == 2) tmem_dealloc<512>(tmem);
}

extern unsigned long long* g_attn3_trace;
extern int g_attn3_trace_cap;

template <int D, bool LT77, bool WSTAT, typename T, bool MASK>
static int launch_attn3(const CUtensorMap& tmX, const CUtensorMap& tmWq, const CUtensorMap& tmO, const Attn3Params& p,
                        cudaStream_t stream) {
  using Cfg = Attn3Cfg<D, WSTAT>;
  auto kern = dual_attn_fwd_persistent_kernel<D, LT77, WSTAT, T, MASK>;
  PV_CUDA(set_max_smem_once(kern, Cfg::SMEM_BYTES));
  const long long sms = sm_count();
  const int grid = static_cast<int>(p.units < sms ? p.units : sms);
  PV_CUDA(launch_pdl(kern, dim3(grid), dim3(A3_THREADS), Cfg::SMEM_BYTES, stream, tmX, tmWq, tmO, p));
  PV_LAUNCHED();
  return PV_OK;
}

int dual_attn_core_bf16_persistent(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats,
                                   int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                                   cudaStream_t stream, bool f16, const float* img_row_weight) {
  PV_REQUIRE(B > 0 && S > 0 && H > 0 && C % H == 0, "bad shape B=%d S=%d C=%d H=%d", B, S, C, H);
  const int d = C / H;
  PV_REQUIRE(d == 40 || d == 80 || d == 160, "head_dim %d unsupported (40/80/160)", d);
  PV_REQUIRE(C % A3_BN == 0 && C % A3_BK == 0, "C=%d must be a multiple of 320", C);
  PV_REQUIRE(Lt >= 1 && Lt <= A3_IMG_OFF && Li >= 1 && Li <= A3_KEYS - A3_IMG_OFF,
             "need 1 <= Lt <= %d and 1 <= Li <= %d (Lt=%d Li=%d)", A3_IMG_OFF, A3_KEYS - A3_IMG_OFF, Lt, Li);
  PV_REQUIRE((reinterpret_cast<uintptr_t>(X) | reinterpret_cast<uintptr_t>(Wq) | reinterpret_cast<uintptr_t>(Kp) |
              reinterpret_cast<uintptr_t>(Vp) | reinterpret_cast<uintptr_t>(O)) % 16 == 0, "pointers must be 16-byte aligned");
  CUtensorMap tmX, tmWq, tmO;
  if (make_tmap_3d(&tmX, X, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, A3_BK, A3_BM, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmWq, Wq, 2, C, C, 1, C * 2ull, static_cast<uint64_t>(C) * C * 2, A3_BK, A3_BN, 1, Swz::B128, f16)) return PV_ERR_CUDA;
  if (make_tmap_3d(&tmO, O, 2, C, S, B, C * 2ull, static_cast<uint64_t>(S) * C * 2, d == 160 ? 80 : d, 32, 1, Swz::None, f16)) return PV_ERR_CUDA;
  Attn3Params p;
  p.Kp = static_cast<const uint8_t*>(Kp);
  p.Vp = static_cast<const uint8_t*>(Vp);
  p.O = O;
  p.stats = stats;
  p.S = S; p.C = C; p.H = H; p.Lt = Lt; p.Li = Li;
  p.G = C / A3_BN;
  p.MT = (S + A3_BM - 1) / A3_BM;
  p.V = B * p.MT;
  p.units = static_cast<long long>(B) * p.G * p.MT;
  PV_REQUIRE(p.units < (1ll << 30), "too many work units");
  p.w_text = w_text; p.w_img = w_img;
  p.trace = g_attn3_trace;
  p.trace_cap = g_attn3_trace_cap;
  p.scale_log2e = 1.4426950408889634f / sqrtf(static_cast<float>(d));
  p.img_row_weight = img_row_weight;
#define PV_A3_LAUNCH_M(DD, LT, WS, M)                                                             \
  (f16 ? launch_attn3<DD, LT, WS, __half, M>(tmX, tmWq, tmO, p, stream)                           \
       : launch_attn3<DD, LT, WS, __nv_bfloat16, M>(tmX, tmWq, tmO, p, stream))
#define PV_A3_LAUNCH(DD, LT, WS) \
  (img_row_weight ? PV_A3_LAUNCH_M(DD, LT, WS, true) : PV_A3_LAUNCH_M(DD, LT, WS, false))
  switch (d) {
    case 40:
      if (C == A3_KB_WSTAT * A3_BK) return Lt == 77 ? PV_A3_LAUNCH(40, true, true) : PV_A3_LAUNCH(40, false, true);
      return Lt == 77 ? PV_A3_LAUNCH(40, true, false) : PV_A3_LAUNCH(40, false, false);
    case 80: return Lt == 77 ? PV_A3_LAUNCH(80, true, false) : PV_A3_LAUNCH(80, false, false);
    default: return Lt == 77 ? PV_A3_LAUNCH(160, true, false) : PV_A3_LAUNCH(160, false, false);
  }
#undef PV_A3_LAUNCH
#undef PV_A3_LAUNCH_M
}

}  // namespace pv
