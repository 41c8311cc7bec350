// photoverse_b200 -- sm_100a device primitives (mbarrier, TMA, tcgen05/TMEM) as thin inline-PTX wrappers.
// Hand-written for Blackwell B200; nothing here compiles for any other architecture on purpose.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <type_traits>

namespace pv {

// ------------------------------------------------------------------------------------------------
// misc
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);   // .x = lo -> low 16 bits -> lower address
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);               // round to nearest even, like pack_bf16x2
  return *reinterpret_cast<uint32_t*>(&v);
}
// The 16-bit operand type T of the tcgen05 kind::f16 kernels: __nv_bfloat16 (PV_BF16) or __half (PV_F16).  pack_x2<T> is
// the one fp32 -> 16-bit conversion of those kernels (two values, lo at the lower address).
template <typename T>
__device__ __forceinline__ uint32_t pack_x2(float lo, float hi) {
  static_assert(std::is_same<T, __nv_bfloat16>::value || std::is_same<T, __half>::value, "bf16 or fp16");
  if constexpr (std::is_same<T, __half>::value) return pack_f16x2(lo, hi);
  else return pack_bf16x2(lo, hi);
}
__device__ __forceinline__ void st_shared_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(smem_u32(p)), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}
__device__ __forceinline__ float fast_exp2(float x) {   // MUFU.EX2, 2 ulp, flushes denormals; exp2(-inf) = 0
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// One lane of the (converged) warp.  tcgen05.mma / commit and the TMA instructions are warp-uniform in SASS (UTCHMMA,
// UTCBAR, UTMALDG take uniform registers): guarded by elect.sync the compiler emits them back to back, whereas an
// `if (lane == 0)` guard makes it wrap EVERY such instruction in an ELECT/BRA.U.ANY uniformisation loop (~95 cycles
// per MMA issue, measured on B200 with the kernel's debug trace).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P1;\n\telect.sync _|P1, 0xffffffff;\n\tselp.u32 %0, 1, 0, P1;\n\t}" : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void named_bar_sync(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(uint32_t id, uint32_t nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Programmatic dependent launch: a kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization may start
// (barrier init, TMEM allocation, loads of static weights) while its predecessor in the stream is still running;
// pdl_wait() blocks until the predecessor grid has completed and its writes are visible.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking probe (mbarrier.try_wait may suspend the thread for a system-dependent time before returning false).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// try_wait with a suspend-time hint: the thread sleeps in hardware until the phase completes (or `ns` elapse) instead of
// spinning -- a spinning waiter costs issue slots that the working warps of the same scheduler need.
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity), "r"(ns)
      : "memory");
  return ok != 0;
}
#ifndef PV_MBAR_HINT_NS
#define PV_MBAR_HINT_NS 20000u
#endif
// Bounded wait: a protocol bug must trap (and surface as a CUDA error) instead of hanging the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  uint32_t tries = 0;
  while (!mbar_try_wait_hint(bar, parity, PV_MBAR_HINT_NS)) {
    if (++tries > 4000000u) {                  // >= 0.1 s even if every probe returned at once: no wait here exceeds microseconds
#ifdef PV_MBAR_DEBUG   // the printf costs registers and a stack frame in every waiting role: debug builds only
      printf("photoverse_b200: mbarrier wait timed out (block %d,%d,%d thread %d bar %u parity %u)\n",
             blockIdx.x, blockIdx.y, blockIdx.z, threadIdx.x, smem_u32(bar), parity);
#endif
      __trap();
    }
  }
}

// Non-blocking probe on a precomputed 32-bit shared address.
__device__ __forceinline__ bool mbar_test_wait_a(uint32_t bar_addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar_addr), "r"(parity) : "memory");
  return ok != 0;
}

// The same wait on a precomputed 32-bit shared address: hot loops keep their barrier addresses in registers instead of
// re-deriving them (generic -> shared conversion of a pointer costs ~8 uniform-datapath instructions per use).
__device__ __forceinline__ void mbar_wait_a(uint32_t bar_addr, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(bar_addr), "r"(parity) : "memory");
  if (ok) return;
  uint32_t tries = 0;
  for (;;) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok) : "r"(bar_addr), "r"(parity), "r"(PV_MBAR_HINT_NS) : "memory");
    if (ok) return;
    if (++tries > 4000000u) __trap();
  }
}
__device__ __forceinline__ void st_shared_v4_a(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ void st_shared_f32_a(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}
__device__ __forceinline__ float ld_shared_f32_a(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr) : "memory");
  return v;
}

// ------------------------------------------------------------------------------------------------
// proxy / tcgen05 fences
// ------------------------------------------------------------------------------------------------
// generic-proxy smem writes -> visible to the async proxy (TMA store, tcgen05.mma operand fetch)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------
// TMA (cp.async.bulk[.tensor])
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                            int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// L2 prefetch of a tile (no shared-memory destination): hides HBM latency behind L2 capacity instead of smem stages
__device__ __forceinline__ void tma_prefetch_3d(const CUtensorMap* m, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(reinterpret_cast<uint64_t>(m)),
               "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
// contiguous global -> shared bulk copy (bytes % 16 == 0, both addresses 16-byte aligned)
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

// ------------------------------------------------------------------------------------------------
// TMEM allocation
// ------------------------------------------------------------------------------------------------
template <uint32_t COLS>   // power of two in [32, 512]; executed by one full warp
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot) {
  static_assert(COLS >= 32 && COLS <= 512 && (COLS & (COLS - 1)) == 0, "TMEM columns: power of 2 in [32,512]");
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
               "r"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(COLS) : "memory");
}

// ------------------------------------------------------------------------------------------------
// UMMA descriptors
// ------------------------------------------------------------------------------------------------
enum : uint32_t { UMMA_LAYOUT_NONE = 0, UMMA_LAYOUT_SW128 = 2, UMMA_LAYOUT_SW64 = 4, UMMA_LAYOUT_SW32 = 6 };

// Shared-memory matrix descriptor (sm_100 format: version field = 1).
//   bits [0,14)  start address >> 4        bits [16,30) leading-dim byte offset >> 4
//   bits [32,46) stride-dim byte offset >> 4   bits [46,48) version=1   bits [61,64) layout type
// K-major canonical layouts (16-byte units):
//   SW128 : rows of 128 B, 8-row groups SBO apart (1024 B when dense), XOR-swizzled 16 B chunks; LBO unused(=1)
//   NONE  : 8x16B core matrices; LBO = byte distance between the two 16 B K-chunks of one K=16 step,
//           SBO = byte distance between consecutive 8-row groups
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr >> 4) & 0x3FFF);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout) << 61;
  return d;
}
__device__ __forceinline__ uint64_t umma_desc_sw128(const void* tile_1024_aligned_plus_koffset) {
  return umma_desc(smem_u32(tile_1024_aligned_plus_koffset), 16, 1024, UMMA_LAYOUT_SW128);
}

// Instruction descriptor, kind::f16, A=B=bf16, D=f32, both operands K-major, dense.
//   [4,6) c_format=1(F32)  [7,10) a_format=1(BF16)  [10,13) b_format=1(BF16)  [15] a_major=0  [16] b_major=0
//   [17,23) N>>3  [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
// The same with A=B=fp16: a_format = b_format = 0 (F16); nothing else of the instruction changes.
__host__ __device__ constexpr uint32_t umma_idesc_f16(uint32_t M, uint32_t N) {
  return (1u << 4) | ((N >> 3) << 17) | ((M >> 4) << 24);
}
template <typename T>
__host__ __device__ constexpr uint32_t umma_idesc(uint32_t M, uint32_t N) {
  return std::is_same<T, __half>::value ? umma_idesc_f16(M, N) : umma_idesc_bf16(M, N);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread
__device__ __forceinline__ void umma_bf16_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T : A = [128 lanes x K] bf16 packed two per 32-bit column (8 columns per K=16)
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued tcgen05.mma of this thread complete -> arrive(1) on the mbarrier
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// ------------------------------------------------------------------------------------------------
// TMEM -> registers.  32x32b: thread t of the warp reads lane (base_lane + t), N consecutive columns.
// A warp may only touch the 32-lane quarter  (warp_id % 4) * 32 .. +31.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x8(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// registers -> TMEM (same lane/column mapping as the loads)
__device__ __forceinline__ void tmem_st_x8(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void st_global_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.global.v4.b32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

}  // namespace pv

// ------------------------------------------------------------------------------------------------
// CTA-pair (cta_group::2) primitives: two CTAs of a cluster drive ONE tcgen05.mma of M = 256; each CTA holds its own
// 128 rows of A and HALF of the N rows of B, so the B operand costs half the TMA ingest and half the smem reads per CTA.
// ------------------------------------------------------------------------------------------------
namespace pv {

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `local_smem_addr` (a shared::cta address) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_smem_addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_smem_addr), "r"(rank));
  return r;
}
// arrive on an mbarrier of another CTA of the cluster (address from mapa_u32).  Default (.release.cta) semantics on
// purpose: what is handed over lives in TMEM and is ordered by the tcgen05 fences; a .release.cluster arrive makes ptxas
// emit a cluster-scope fence (L1 invalidate) that costs ~1000 cycles per hand-off (measured with the device trace).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// TMA load into THIS CTA's shared memory whose completion is signalled on an mbarrier given as a shared::cluster address
// (the leader CTA's barrier): the .cta_group::2 form allows the barrier to live in the peer CTA.
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// L2 eviction-priority hints.  The path streams X in and Y out once, but O is written by the attention phase and read back
// by the out projection a few microseconds later: X loads are marked evict-first and O stores evict-last so that O is
// still in L2 (126 MB, two partitions) when it is needed again.
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ void tma_load_3d_2sm_hint(void* smem_dst, const CUtensorMap* m, uint32_t bar_cluster_addr, int c0,
                                                     int c1, int c2, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(bar_cluster_addr), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d_hint(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2, uint64_t policy) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;" ::"l"(
                   reinterpret_cast<uint64_t>(m)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "l"(policy)
               : "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* smem_slot) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(COLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t COLS>
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(COLS) : "memory");
}
// D[tmem of both CTAs] (+)= A[smem, 128 rows per CTA] * B[smem, N/2 rows per CTA]^T ; issued by ONE thread of the leader CTA
__device__ __forceinline__ void umma_bf16_ss_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_2sm(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread complete -> arrive(1) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(static_cast<uint16_t>(3))
               : "memory");
}

}  // namespace pv
