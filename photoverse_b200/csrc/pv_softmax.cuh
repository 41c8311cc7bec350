// photoverse_b200 -- helpers shared by the persistent attention kernels (pv_attn3.cu, pv_attn4.cu).
#pragma once
#include "pv_common.cuh"

namespace pv {

template <int N, typename T = __nv_bfloat16>
__device__ __forceinline__ void pack_pairs3(const uint32_t* v, uint32_t* out) {
#pragma unroll
  for (int i = 0; i < N / 2; ++i) out[i] = pack_x2<T>(__uint_as_float(v[2 * i]), __uint_as_float(v[2 * i + 1]));
}

// A drained-later O accumulator of one softmax group (the PV MMA runs while the group computes its next softmax).
struct PendingO {
  uint32_t taddr;          // TMEM address (lane quarter included) of the O accumulator
  float oscale;
  uint32_t parity;         // phase parity of o_full[wg]
  int c0, r0, b;           // TMA store coordinates: first channel, first row of this warp's 32-row slab, sample
  int slot;
  bool valid;
};


// packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2 -- half the issue slots of the scalar forms)
__device__ __forceinline__ uint64_t f2_pack(float a, float b) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& a, float& b) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// the same add as a volatile statement: keeps its place relative to barriers / other volatile statements
__device__ __forceinline__ uint64_t f2_add_v(uint64_t a, uint64_t b) {
  uint64_t d;
  asm volatile("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// 32 consecutive TMEM columns of this thread's lane into r[0..31] (no wait)
__device__ __forceinline__ void tmem_ld32_raw(uint32_t taddr, uint32_t* r) {
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

__device__ __forceinline__ void tmem_ld16_raw(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_x4(uint32_t taddr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1, %2, %3, %4};" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]),
               "r"(r[3])
               : "memory");
}

// Debug timeline (-DPV_TRACE builds only): lane 0 of a role warp of one CTA appends (event, index, SM clock) to the
// role's private region of the trace buffer (no atomics: the stores are fire-and-forget).  Release builds compile the
// calls away.
struct A3Trace {
  unsigned long long* base;
  int n, cap;
};
#ifdef PV_TRACE
__device__ __forceinline__ A3Trace a3_trace_init_raw(unsigned long long* trace, int trace_cap, int role, int block = 0) {
  A3Trace t;
  const int per = trace_cap / 8;                  // 8 role regions after an 8-word header of event counts
  t.base = (trace != nullptr && static_cast<int>(blockIdx.x) == block && (threadIdx.x & 31) == 0) ? trace + 8 + static_cast<size_t>(role) * per * 3 : nullptr;
  t.n = 0;
  t.cap = per;
  return t;
}
__device__ __forceinline__ void a3_trace(A3Trace& t, int ev, int idx) {
  if (t.base != nullptr && t.n < t.cap) {
    t.base[3 * t.n] = static_cast<unsigned long long>(ev);
    t.base[3 * t.n + 1] = static_cast<unsigned long long>(idx);
    t.base[3 * t.n + 2] = static_cast<unsigned long long>(clock64());
    ++t.n;
  }
}
__device__ __forceinline__ void a3_trace_done_raw(unsigned long long* trace, const A3Trace& t, int role) {
  if (t.base != nullptr) trace[role] = static_cast<unsigned long long>(t.n);
}
// trace_block == -1: instead of one CTA's event list, every leader CTA records the global timer at a few points of its
// life (slot k of pair `pair`): the load balance of a launch at a glance (tools/pair_times.py).
__device__ __forceinline__ void a3_pair_time(unsigned long long* trace, int trace_block, int k) {
  if (trace != nullptr && trace_block == -1 && threadIdx.x == 0 && (blockIdx.x & 1) == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    trace[8 + (blockIdx.x >> 1) * 8 + k] = t;
  }
}
#else
__device__ __forceinline__ void a3_pair_time(unsigned long long*, int, int) {}
__device__ __forceinline__ A3Trace a3_trace_init_raw(unsigned long long*, int, int, int = 0) { return A3Trace{nullptr, 0, 0}; }
__device__ __forceinline__ void a3_trace(A3Trace&, int, int) {}
__device__ __forceinline__ void a3_trace_done_raw(unsigned long long*, const A3Trace&, int) {}
#endif

}  // namespace pv
