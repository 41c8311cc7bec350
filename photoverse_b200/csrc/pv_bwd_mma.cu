// photoverse_b200 -- dual-branch attention backward core on the tensor cores (bf16 training path).
//
// Same contract as attn_bwd_kernel (pv_bwd.cu): from dO, Q [B,S,C] (bf16), the fp32 K/V projections and the forward
// kernel's per-row statistics it produces dQ [B,S,C] and the per-chunk partial dK / dV that kv_bwd_reduce_kernel sums.
//   p^ = 2^(s cs - m)/l per segment ; dp_k = dO.V_k ; delta_seg = sum_{k in seg} p^_k dp_k ; ds_k = w_seg p^_k (dp_k - delta_seg)
//   dQ = scale ds K ; dK = scale ds^T Q ; dV = (w p^)^T dO
// One block = up to T consecutive 128-query-row tiles of one (sample, head) (T = 4 for head_dim 40 / 80 at S >= 2048, else
// 2 / 1: attn_bwd_mma_tiles): K / V are staged once per block and dK / dV accumulate in registers across the tiles, so
// the fp32 partials (82 x head_dim x 2 per block) cost T times less traffic than one block per tile; dQ leaves through
// shared memory as 16-byte row segments.  8 warps x 16 rows per tile.  All five contractions are warp-level
// mma.sync.m16n8k16 (bf16 in, fp32 accumulate) -- with 96 key slots the tiles are far too small for tcgen05 / TMEM to pay:
//   phase 1 (warp = 16 query rows): S = Q K^T and dP = dO V^T (B operands straight from the [key][dim] tiles), softmax
//            from the saved statistics, dS, dQ = dS K (dS re-used from its accumulator registers as the A operand, K via
//            ldmatrix.trans); w p^ and dS go to shared memory as bf16
//   phase 2 (warp = a set of 16x8 output tiles): dK^T-free form dK = dS^T Q, dV = P^T dO with A = transposed loads of the
//            [row][key] tiles and B = transposed loads of the [row][dim] tiles, k-loop over the block's 128 rows.
// The SIMT kernel in pv_bwd.cu remains the fp32 parity path (and the A/B reference: pv_set_option("bwd_mma", 0)).
#include "pv_common.cuh"
#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

constexpr int BM_ROWS = 128;                 // query rows per block == attn_bwd_chunks() granularity
constexpr int BM_KEYS = PV_KEYS_PAD;         // 96 key slots (keys [0, Lt) text, [Lt, Lt + Li) image, rest zero)
constexpr int BM_PKEY = BM_KEYS + 8;         // pitch (elements) of the [row][key] tiles

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t addr, uint32_t& r0, uint32_t& r1) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];" : "=r"(r0), "=r"(r1) : "r"(addr));
}
// D (16x8, fp32) += A (16x16, bf16, row) * B (16x8, bf16, col)
__device__ __forceinline__ void mma_bf16(float (&d)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

template <int D>
struct BwdMmaCfg {
  static constexpr int DP = (D + 15) / 16 * 16;        // head_dim padded to the MMA k step
  static constexpr int PD = DP + 8;                    // pitch (elements) of the [.][dim] tiles: odd multiple of 16 B
  static constexpr int NT_D = DP / 8;                  // 8-wide n tiles over the head dim
  static constexpr int TILES = (BM_KEYS / 16) * NT_D;  // 16x8 output tiles of dK (and of dV)
  static constexpr int TPW = (TILES + 7) / 8;          // tiles per warp in phase 2
  static constexpr int OFF_K = 0;
  static constexpr int OFF_V = OFF_K + BM_KEYS * PD * 2;
  static constexpr int OFF_Q = OFF_V + BM_KEYS * PD * 2;
  static constexpr int OFF_DO = OFF_Q + BM_ROWS * PD * 2;
  static constexpr int OFF_P = OFF_DO + BM_ROWS * PD * 2;
  static constexpr int OFF_DS = OFF_P + BM_ROWS * BM_PKEY * 2;
  static constexpr int SMEM_BYTES = OFF_DS + BM_ROWS * BM_PKEY * 2;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};

// MASK: the image keys of query row s are weighted w_img * img_row_weight[b, s] (ip_adapter_masks)
template <int D, bool MASK>
__global__ void __launch_bounds__(256, 1)
attn_bwd_mma_kernel(const __nv_bfloat16* __restrict__ dO, const __nv_bfloat16* __restrict__ Q,
                    const float* __restrict__ kv_text, const float* __restrict__ kv_img, const float* __restrict__ stats,
                    __nv_bfloat16* __restrict__ dQ, float* __restrict__ part, int B, int S, int C, int H, int Lt, int Li,
                    float w_text, float w_img, float scale, float scale_log2e, int tiles_per_block,
                    const float* __restrict__ img_row_weight) {
  using Cfg = BwdMmaCfg<D>;
  constexpr int DP = Cfg::DP, PD = Cfg::PD, NT_D = Cfg::NT_D;
  extern __shared__ __align__(16) uint8_t smem_b[];
  __nv_bfloat16* Ks = reinterpret_cast<__nv_bfloat16*>(smem_b + Cfg::OFF_K);     // [96][PD]   key-major
  __nv_bfloat16* Vs = reinterpret_cast<__nv_bfloat16*>(smem_b + Cfg::OFF_V);     // [96][PD]
  __nv_bfloat16* Qs = reinterpret_cast<__nv_bfloat16*>(smem_b + Cfg::OFF_Q);     // [128][PD]  row-major
  __nv_bfloat16* Os = reinterpret_cast<__nv_bfloat16*>(smem_b + Cfg::OFF_DO);    // [128][PD]  dO
  __nv_bfloat16* Ps = reinterpret_cast<__nv_bfloat16*>(smem_b + Cfg::OFF_P);     // [128][104] w_seg p^
  __nv_bfloat16* Ds = reinterpret_cast<__nv_bfloat16*>(smem_b + Cfg::OFF_DS);    // [128][104] scale * ds
  const int chunk = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int L = Lt + Li;
  const int C2 = 2 * C;
  // dK / dV tiles of this warp, accumulated over the block's row tiles
  float ak[Cfg::TPW][4], av[Cfg::TPW][4];
#pragma unroll
  for (int i = 0; i < Cfg::TPW; ++i)
#pragma unroll
    for (int e = 0; e < 4; ++e) { ak[i][e] = 0.f; av[i][e] = 0.f; }

  // ---- stage K, V (fp32 projections -> bf16, the rounding the forward kernel's tiles have) once per block ----
  for (int i = threadIdx.x; i < BM_KEYS * (DP / 2); i += 256) {
    const int k = i / (DP / 2), c = (i - k * (DP / 2)) * 2;
    float k0 = 0.f, k1 = 0.f, v0 = 0.f, v1 = 0.f;
    if (k < L && c < D) {
      const float* src = (k < Lt) ? kv_text + (static_cast<size_t>(b) * Lt + k) * C2 : kv_img + (static_cast<size_t>(b) * Li + (k - Lt)) * C2;
      const float2 kk = *reinterpret_cast<const float2*>(src + h * D + c);
      const float2 vv = *reinterpret_cast<const float2*>(src + C + h * D + c);
      k0 = kk.x; k1 = kk.y; v0 = vv.x; v1 = vv.y;
    }
    *reinterpret_cast<uint32_t*>(Ks + k * PD + c) = pack_bf16x2(k0, k1);
    *reinterpret_cast<uint32_t*>(Vs + k * PD + c) = pack_bf16x2(v0, v1);
  }
#pragma unroll 1
  for (int tile_i = 0; tile_i < tiles_per_block; ++tile_i) {
  const int q0 = (chunk * tiles_per_block + tile_i) * BM_ROWS;
  if (q0 >= S) break;
  if (tile_i > 0) __syncthreads();           // the previous tile's dQ copy-out still reads Qs
  // ---- this tile's Q, dO ----
  for (int i = threadIdx.x; i < BM_ROWS * (DP / 8); i += 256) {
    const int r = i / (DP / 8), c = (i - r * (DP / 8)) * 8;
    uint4 qv = make_uint4(0u, 0u, 0u, 0u), ov = qv;
    if (q0 + r < S && c < D) {
      const size_t off = (static_cast<size_t>(b) * S + q0 + r) * C + h * D + c;
      qv = *reinterpret_cast<const uint4*>(Q + off);
      ov = *reinterpret_cast<const uint4*>(dO + off);
    }
    *reinterpret_cast<uint4*>(Qs + r * PD + c) = qv;
    *reinterpret_cast<uint4*>(Os + r * PD + c) = ov;
  }
  __syncthreads();

  // =============================== phase 1: this warp's 16 query rows ===============================
  uint32_t dqr[NT_D / 2][4];                 // this thread's dQ fragments: [dim tile pair][row g | g + 8, dims 8 half + 2 t]
  {
    const int r0 = warp * 16;
    const int g = lane >> 2, t = lane & 3;
    float sacc[BM_KEYS / 8][4], pacc[BM_KEYS / 8][4];
#pragma unroll
    for (int n = 0; n < BM_KEYS / 8; ++n)
#pragma unroll
      for (int e = 0; e < 4; ++e) { sacc[n][e] = 0.f; pacc[n][e] = 0.f; }
    // A operands: rows r0 + (lane & 7) + 8 * ((lane >> 3) & 1), k columns 8 * (lane >> 4)
    const uint32_t a_row = r0 + (lane & 7) + ((lane >> 3) & 1) * 8;
    const uint32_t qa = smem_u32(Qs + a_row * PD + (lane >> 4) * 8);
    const uint32_t oa = smem_u32(Os + a_row * PD + (lane >> 4) * 8);
    // B operands of S / dP: tiles stored [key][dim] = [n][k]: two key tiles per x4 load
    const uint32_t b_key = (lane & 7) + (lane >> 4) * 8;
    const uint32_t kb = smem_u32(Ks + b_key * PD + ((lane >> 3) & 1) * 8);
    const uint32_t vb = smem_u32(Vs + b_key * PD + ((lane >> 3) & 1) * 8);
#pragma unroll
    for (int kk = 0; kk < DP / 16; ++kk) {
      uint32_t q0r, q1r, q2r, q3r, o0r, o1r, o2r, o3r;
      ldsm_x4(qa + kk * 32, q0r, q1r, q2r, q3r);
      ldsm_x4(oa + kk * 32, o0r, o1r, o2r, o3r);
#pragma unroll
      for (int n2 = 0; n2 < BM_KEYS / 16; ++n2) {
        uint32_t k0r, k1r, k2r, k3r, v0r, v1r, v2r, v3r;
        ldsm_x4(kb + (n2 * 16 * PD + kk * 16) * 2, k0r, k1r, k2r, k3r);
        ldsm_x4(vb + (n2 * 16 * PD + kk * 16) * 2, v0r, v1r, v2r, v3r);
        mma_bf16(sacc[2 * n2], q0r, q1r, q2r, q3r, k0r, k1r);
        mma_bf16(sacc[2 * n2 + 1], q0r, q1r, q2r, q3r, k2r, k3r);
        mma_bf16(pacc[2 * n2], o0r, o1r, o2r, o3r, v0r, v1r);
        mma_bf16(pacc[2 * n2 + 1], o0r, o1r, o2r, o3r, v2r, v3r);
      }
    }
    // softmax from the saved statistics; this thread holds rows g and g + 8, keys 8 n + 2 t + {0, 1}
    const int row_a = q0 + r0 + g, row_b = row_a + 8;
    float4 st_a = make_float4(0.f, 1.f, 0.f, 1.f), st_b = st_a;
    if (row_a < S) st_a = reinterpret_cast<const float4*>(stats)[(static_cast<size_t>(b) * H + h) * S + row_a];
    if (row_b < S) st_b = reinterpret_cast<const float4*>(stats)[(static_cast<size_t>(b) * H + h) * S + row_b];
    const float ilt_a = 1.f / st_a.y, ili_a = 1.f / st_a.w, ilt_b = 1.f / st_b.y, ili_b = 1.f / st_b.w;
    float dt_a = 0.f, di_a = 0.f, dt_b = 0.f, di_b = 0.f;
#pragma unroll
    for (int n = 0; n < BM_KEYS / 8; ++n) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = 8 * n + 2 * t + (e & 1);
        const bool lo = e < 2;                     // row g (else g + 8)
        const bool is_t = key < Lt;
        const bool valid = key < L && (lo ? row_a : row_b) < S;
        const float m = lo ? (is_t ? st_a.x : st_a.z) : (is_t ? st_b.x : st_b.z);
        const float il = lo ? (is_t ? ilt_a : ili_a) : (is_t ? ilt_b : ili_b);
        const float ph = valid ? exp2f(fmaf(sacc[n][e], scale_log2e, -m)) * il : 0.f;
        sacc[n][e] = ph;                           // p^
        const float pd = ph * pacc[n][e];
        if (is_t) { if (lo) dt_a += pd; else dt_b += pd; }
        else      { if (lo) di_a += pd; else di_b += pd; }
      }
    }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      dt_a += __shfl_xor_sync(0xffffffffu, dt_a, o);
      di_a += __shfl_xor_sync(0xffffffffu, di_a, o);
      dt_b += __shfl_xor_sync(0xffffffffu, dt_b, o);
      di_b += __shfl_xor_sync(0xffffffffu, di_b, o);
    }
    // w p^ and scale * ds, packed to bf16: A operands of dQ (from registers) and of phase 2 (through shared memory)
    uint32_t pw[BM_KEYS / 8][2], dsr[BM_KEYS / 8][2];
    float wi_a = w_img, wi_b = w_img;
    if constexpr (MASK) {
      if (row_a < S) wi_a *= __ldg(img_row_weight + static_cast<size_t>(b) * S + row_a);
      if (row_b < S) wi_b *= __ldg(img_row_weight + static_cast<size_t>(b) * S + row_b);
    }
#pragma unroll
    for (int n = 0; n < BM_KEYS / 8; ++n) {
      float pv[4], dv[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int key = 8 * n + 2 * t + (e & 1);
        const bool lo = e < 2;
        const bool is_t = key < Lt;
        const float w = is_t ? w_text : (lo ? wi_a : wi_b);
        const float delta = lo ? (is_t ? dt_a : di_a) : (is_t ? dt_b : di_b);
        pv[e] = w * sacc[n][e];
        dv[e] = scale * w * sacc[n][e] * (pacc[n][e] - delta);
      }
      pw[n][0] = pack_bf16x2(pv[0], pv[1]);
      pw[n][1] = pack_bf16x2(pv[2], pv[3]);
      dsr[n][0] = pack_bf16x2(dv[0], dv[1]);
      dsr[n][1] = pack_bf16x2(dv[2], dv[3]);
      *reinterpret_cast<uint32_t*>(Ps + (r0 + g) * BM_PKEY + 8 * n + 2 * t) = pw[n][0];
      *reinterpret_cast<uint32_t*>(Ps + (r0 + g + 8) * BM_PKEY + 8 * n + 2 * t) = pw[n][1];
      *reinterpret_cast<uint32_t*>(Ds + (r0 + g) * BM_PKEY + 8 * n + 2 * t) = dsr[n][0];
      *reinterpret_cast<uint32_t*>(Ds + (r0 + g + 8) * BM_PKEY + 8 * n + 2 * t) = dsr[n][1];
    }
    // dQ = (scale ds) K : A = ds fragments (accumulator layout == A layout over pairs of key tiles), B = K^T via ldmatrix.trans
    // of the [key][dim] tile: matrix rows = keys 16 j + (lane & 7) + 8 ((lane >> 3) & 1), columns = dims 8 n + 8 (lane >> 4)
    const uint32_t kt = smem_u32(Ks + ((lane & 7) + ((lane >> 3) & 1) * 8) * PD + (lane >> 4) * 8);
#pragma unroll
    for (int n2 = 0; n2 < NT_D / 2; ++n2) {        // two 8-wide dim tiles per x4 load
      float acc0[4] = {0.f, 0.f, 0.f, 0.f}, acc1[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int j = 0; j < BM_KEYS / 16; ++j) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(kt + (j * 16 * PD + n2 * 16) * 2, b0, b1, b2, b3);
        mma_bf16(acc0, dsr[2 * j][0], dsr[2 * j][1], dsr[2 * j + 1][0], dsr[2 * j + 1][1], b0, b1);
        mma_bf16(acc1, dsr[2 * j][0], dsr[2 * j][1], dsr[2 * j + 1][0], dsr[2 * j + 1][1], b2, b3);
      }
      // bf16 pairs, kept in registers until phase 2 has read Q: the tile then leaves through Qs as 16-byte segments
      dqr[n2][0] = pack_bf16x2(acc0[0], acc0[1]);
      dqr[n2][1] = pack_bf16x2(acc0[2], acc0[3]);
      dqr[n2][2] = pack_bf16x2(acc1[0], acc1[1]);
      dqr[n2][3] = pack_bf16x2(acc1[2], acc1[3]);
    }
  }
  __syncthreads();

  // =============================== phase 2: dK = (scale ds)^T Q, dV = (w p^)^T dO ===============================
  {
    const int g = lane >> 2, t = lane & 3;
    // A (16 keys x 16 rows) = transposed load of the [row][key] tiles: matrix rows = rows 16 k + (lane & 7) + 8 (lane >> 4),
    // columns = keys 16 mt + 8 ((lane >> 3) & 1)
    const uint32_t a_off = ((lane & 7) + (lane >> 4) * 8) * BM_PKEY + ((lane >> 3) & 1) * 8;
    // B (16 rows x 8 dims) = transposed load of the [row][dim] tiles: matrix rows = rows 16 k + (lane & 7) + 8 ((lane >> 3) & 1)
    const uint32_t b_off = ((lane & 7) + ((lane >> 3) & 1) * 8) * PD;
#pragma unroll
    for (int i = 0; i < Cfg::TPW; ++i) {
      const int tile = warp + 8 * i;
      if (tile < Cfg::TILES) {
        const int mt = tile / NT_D, nt = tile - mt * NT_D;
        const uint32_t da = smem_u32(Ds + a_off + mt * 16), pa = smem_u32(Ps + a_off + mt * 16);
        const uint32_t qb = smem_u32(Qs + b_off + nt * 8), ob = smem_u32(Os + b_off + nt * 8);
#pragma unroll
        for (int k = 0; k < BM_ROWS / 16; ++k) {
          uint32_t a0, a1, a2, a3, p0, p1, p2, p3, bq0, bq1, bo0, bo1;
          ldsm_x4_t(da + (k * 16 * BM_PKEY) * 2, a0, a1, a2, a3);
          ldsm_x4_t(pa + (k * 16 * BM_PKEY) * 2, p0, p1, p2, p3);
          ldsm_x2_t(qb + (k * 16 * PD) * 2, bq0, bq1);
          ldsm_x2_t(ob + (k * 16 * PD) * 2, bo0, bo1);
          mma_bf16(ak[i], a0, a1, a2, a3, bq0, bq1);
          mma_bf16(av[i], p0, p1, p2, p3, bo0, bo1);
        }
      }
    }
  }
  __syncthreads();                            // phase 2 has read Qs: stage the dQ tile there
  {
    const int r0 = warp * 16;
    const int g = lane >> 2, t = lane & 3;
#pragma unroll
    for (int n2 = 0; n2 < NT_D / 2; ++n2) {
#pragma unroll
      for (int half = 0; half < 2; ++half) {
        const int dim = n2 * 16 + half * 8 + 2 * t;
        *reinterpret_cast<uint32_t*>(Qs + (r0 + g) * PD + dim) = dqr[n2][2 * half];
        *reinterpret_cast<uint32_t*>(Qs + (r0 + g + 8) * PD + dim) = dqr[n2][2 * half + 1];
      }
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < BM_ROWS * (D / 8); i += 256) {
    const int r = i / (D / 8), c = (i - r * (D / 8)) * 8;
    if (q0 + r < S)
      *reinterpret_cast<uint4*>(dQ + (static_cast<size_t>(b) * S + q0 + r) * C + h * D + c) = *reinterpret_cast<const uint4*>(Qs + r * PD + c);
  }
  }   // row tiles of this block

  // ---- this block's dK / dV partials ----
  {
    const int g = lane >> 2, t = lane & 3;
    float* dstK = part + ((static_cast<size_t>(chunk) * B + b) * H + h) * 2 * L * D;
    float* dstV = dstK + static_cast<size_t>(L) * D;
#pragma unroll
    for (int i = 0; i < Cfg::TPW; ++i) {
      const int tile = warp + 8 * i;
      if (tile < Cfg::TILES) {
        const int mt = tile / NT_D, nt = tile - mt * NT_D;
        const int key_a = mt * 16 + g, key_b = key_a + 8;
        const int dim = nt * 8 + 2 * t;
        if (dim < D) {
          if (key_a < L) {
            *reinterpret_cast<float2*>(dstK + static_cast<size_t>(key_a) * D + dim) = make_float2(ak[i][0], ak[i][1]);
            *reinterpret_cast<float2*>(dstV + static_cast<size_t>(key_a) * D + dim) = make_float2(av[i][0], av[i][1]);
          }
          if (key_b < L) {
            *reinterpret_cast<float2*>(dstK + static_cast<size_t>(key_b) * D + dim) = make_float2(ak[i][2], ak[i][3]);
            *reinterpret_cast<float2*>(dstV + static_cast<size_t>(key_b) * D + dim) = make_float2(av[i][2], av[i][3]);
          }
        }
      }
    }
  }
}

// 128-row tiles per block: the dK / dV accumulators of head_dim 160 (120 registers per thread) leave no room to carry them
// next to phase 1's S / dP fragments, and its layers have S <= 576 anyway.
int attn_bwd_mma_tiles(int S, int d) {
  if (d > 80) return 1;
  return S >= 2048 ? 4 : (S >= 512 ? 2 : 1);
}
// pv_bwd_tc.cu: the tcgen05 kernel (head_dim 40 / 80); this file's mma.sync kernel serves head_dim 160 and the A/B option
int attn_bwd_tc_chunks(int S, int d);
bool attn_bwd_tc_supported(int d, int C);
int dual_attn_bwd_tc(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats, void* dQ,
                     float* part, int nchunk, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                     cudaStream_t stream, const float* img_row_weight);
extern int g_opt_bwd_tc;

int attn_bwd_mma_chunks(int S, int d) {
  if (g_opt_bwd_tc != 0 && attn_bwd_tc_supported(d, d * 8)) return attn_bwd_tc_chunks(S, d);
  const int rows = BM_ROWS * attn_bwd_mma_tiles(S, d);
  return (S + rows - 1) / rows;
}

template <int D>
static int launch_attn_bwd_mma(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats,
                               void* dQ, float* part, int nchunk, int B, int S, int C, int H, int Lt, int Li, float w_text,
                               float w_img, cudaStream_t stream, const float* img_row_weight) {
  auto kern = img_row_weight ? attn_bwd_mma_kernel<D, true> : attn_bwd_mma_kernel<D, false>;
  PV_CUDA(set_max_smem_once(kern, BwdMmaCfg<D>::SMEM_BYTES));
  dim3 grid(nchunk, H, B);
  const float scale = 1.f / sqrtf(static_cast<float>(D));
  kern<<<grid, 256, BwdMmaCfg<D>::SMEM_BYTES, stream>>>(static_cast<const __nv_bfloat16*>(dO), static_cast<const __nv_bfloat16*>(Q),
                                                       kv_text, kv_img, stats, static_cast<__nv_bfloat16*>(dQ), part, B, S, C, H,
                                                       Lt, Li, w_text, w_img, scale, scale * 1.4426950408889634f,
                                                       attn_bwd_mma_tiles(S, C / H), img_row_weight);
  PV_LAUNCHED();
  return PV_OK;
}

// bf16 only; nchunk must be attn_bwd_mma_chunks(S, head_dim).  Needs 16-byte aligned Q / dO rows per head (C, head_dim % 8 == 0).
int dual_attn_bwd_mma(const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats, void* dQ,
                      float* part, int nchunk, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                      cudaStream_t stream, const float* img_row_weight) {
  const int d = C / H;
  PV_REQUIRE(nchunk == attn_bwd_mma_chunks(S, d), "chunk count mismatch (%d for S=%d)", nchunk, S);
  if (g_opt_bwd_tc != 0 && attn_bwd_tc_supported(d, d * 8))
    return dual_attn_bwd_tc(dO, Q, kv_text, kv_img, stats, dQ, part, nchunk, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
  switch (d) {
    case 40: return launch_attn_bwd_mma<40>(dO, Q, kv_text, kv_img, stats, dQ, part, nchunk, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
    case 80: return launch_attn_bwd_mma<80>(dO, Q, kv_text, kv_img, stats, dQ, part, nchunk, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
    case 160: return launch_attn_bwd_mma<160>(dO, Q, kv_text, kv_img, stats, dQ, part, nchunk, B, S, C, H, Lt, Li, w_text, w_img, stream, img_row_weight);
    default: PV_FAIL(PV_ERR_UNSUPPORTED, "head_dim %d unsupported (40/80/160)", d);
  }
}

}  // namespace pv
