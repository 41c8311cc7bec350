// photoverse_b200 -- host-side helpers shared by the C-ABI translation units.
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>
#include <string>

namespace pv {

// ---- error plumbing: nothing throws across the C ABI -------------------------------------------
void set_error(const std::string& msg);
const char* last_error_cstr();
extern std::atomic<unsigned long long> g_launches;   // kernels launched by this library

#define PV_FAIL(code, ...)                                  \
  do {                                                      \
    char _b[512];                                           \
    snprintf(_b, sizeof(_b), __VA_ARGS__);                  \
    ::pv::set_error(std::string(__func__) + ": " + _b);     \
    return (code);                                          \
  } while (0)

#define PV_REQUIRE(cond, ...)                               \
  do {                                                      \
    if (!(cond)) PV_FAIL(PV_ERR_INVALID, __VA_ARGS__);      \
  } while (0)

#define PV_CUDA(expr)                                                                  \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) PV_FAIL(PV_ERR_CUDA, "%s -> %s", #expr, cudaGetErrorString(_e)); \
  } while (0)

#define PV_LAUNCHED()                                                                  \
  do {                                                                                 \
    ::pv::g_launches.fetch_add(1, std::memory_order_relaxed);                          \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess) PV_FAIL(PV_ERR_CUDA, "kernel launch -> %s", cudaGetErrorString(_e)); \
  } while (0)

// ---- TMA tensor maps ------------------------------------------------------------------------------
enum class Swz { None, B64, B128 };

// Encode a rank-3 tiled tensor map over a (possibly strided) row-major tensor:
//   dims    = {d0 (innermost, contiguous), d1, d2}           in elements
//   strides = {stride of d1, stride of d2}                   in BYTES (multiples of 16)
//   box     = {b0, b1, b2}                                   in elements (b0*elem_bytes <= swizzle span)
// Out-of-bounds box elements read as zero and are skipped on store.
// 2-byte elements are bf16, or fp16 with f16 = true.
// Returns 0 on success; on failure sets the error string.
int make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
                 uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2, Swz swz,
                 bool f16 = false);

int sm_count();                       // SM count of the CURRENT device (cached per device)
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device function attribute: set once per (kernel, device)
cudaError_t set_max_smem_once_impl(const void* kern, int bytes, bool max_carveout);
template <typename K>
cudaError_t set_max_smem_once(K kern, int bytes, bool max_carveout = false) {
  return set_max_smem_once_impl(reinterpret_cast<const void*>(kern), bytes, max_carveout);
}

extern int g_opt_pdl;
// Launch with programmatic stream serialisation (PDL) when enabled: the kernel must call pdl_wait() before touching any
// data a predecessor may have written.
template <typename... KArgs, typename... Args>
cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_opt_pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

}  // namespace pv
