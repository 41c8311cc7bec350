// photoverse_b200 -- the C ABI (include/photoverse_b200.h): argument checking, TMA descriptor encoding,
// dispatch between the bf16 tcgen05 path and the fp32 parity path.  No CPU fallback anywhere.
#include <string.h>

#include <mutex>
#include <unordered_map>

#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

// ---- forward declarations of the launchers -------------------------------------------------------
int gemm_bf16(const void* A, const void* W, const float* bias, void* D, bool out_f32, long long M, long long N,
              long long K, long long batch, long long lda, long long ldw, long long ldd, long long strideA,
              long long strideW, long long strideBias, long long strideD, cudaStream_t stream, bool w_static = false,
              bool f16 = false);
int gemm_f32(const float* A, const float* W, const float* bias, float* D, long long M, long long N, long long K,
             long long batch, long long lda, long long ldw, long long ldd, long long strideA, long long strideW,
             long long strideBias, long long strideD, cudaStream_t stream);
// The tcgen05 launchers below take bf16 operands, or fp16 ones with f16 = true.
int dual_attn_core_bf16_persistent(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats,
                                   int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                                   cudaStream_t stream, bool f16);
bool dual_attn_pair_roles_supported(int S, int C, int H);
bool dual_attn_pair_roles_fused_supported(int S, int C, int H);
int dual_attn_core_bf16_pair_roles(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats,
                                   int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                                   cudaStream_t stream, const void* Wo, const float* bo, void* Y, unsigned int* sync,
                                   bool f16);
int dual_attn_core_bf16_pair(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats, int B,
                             int S, int C, int H, int Lt, int Li, float w_text, float w_img, cudaStream_t stream,
                             const void* Wo, const float* bo, void* Y, unsigned int* sync, bool f16);
int dual_attn_core_f32(const float* Q, const float* Kp, const float* Vp, float* O, float* stats, int B, int S, int C,
                       int H, int Lt, int Li, float w_text, float w_img, cudaStream_t stream);
static int64_t attn_kv_tile_bytes(int d) { return static_cast<int64_t>(PV_KEYS_PAD) * ((d + 15) / 16 * 16) * 2; }
int pack_weight(pv_dtype out_dt, const float* W, const float* A, const float* Bm, float scaling, void* out, int out_f,
                int in_f, int r, cudaStream_t stream);
int kv_pack(pv_dtype dt, const float* kv_text, const float* kv_img, void* Kp, void* Vp, float* v_ip_norm, int B, int Lt,
            int Li, int C, int H, cudaStream_t stream);
int ln_lrelu(pv_dtype out_dt, const float* x, const float* gamma, const float* beta, void* y, float* save_mean,
             float* save_rstd, long long rows, int cols, long long ldx, long long ldy, long long rows_per_group,
             float eps, float slope, cudaStream_t stream);
int group_mean(pv_dtype in_dt, pv_dtype out_dt, const void* x, void* y, long long groups, int P, int cols, long long ldy,
               cudaStream_t stream);

int pack_weight_t(bool out_bf16, const float* W, const float* A, const float* Bm, float scaling, void* out, int out_f,
                  int in_f, int r, cudaStream_t stream);
int transpose_2d(bool bf16, const void* in, void* out, long long R, long long Cc, long long ldi, long long ldo, cudaStream_t stream);
long long wgrad_ws_bytes(bool bf16, long long M, long long N, long long K);
int linear_bwd_weight(bool bf16, const void* G, const void* X, float* dW, void* ws, long long M, long long N, long long K,
                      long long ldg, long long ldx, float alpha, float beta, cudaStream_t stream);
long long colsum_ws_bytes(long long M, long long N);
int col_sum(bool bf16, const void* G, float* out, void* ws, long long M, long long N, long long ldg, cudaStream_t stream);
long long ln_bwd_ws_bytes(long long groups, long long rows_per_group, int cols);
int ln_lrelu_bwd(bool bf16, const void* da, const float* x, const float* mean, const float* rstd, const float* gamma,
                 const float* beta, void* dx, float* dgamma, float* dbeta, void* ws, long long groups,
                 long long rows_per_group, int cols, float slope, cudaStream_t stream);
int group_mean_bwd(bool bf16, const void* dy, void* dx, long long groups, int P, int cols, long long ldy, cudaStream_t stream);
int attn_bwd_chunks(int S);
long long self_attn_ws_bytes(int B, int S, int C, int H);
int self_attn_fwd_bf16(const void* q, const void* k, const void* v, long long ld, void* out, void* ws, int B, int S, int C, int H,
                       cudaStream_t stream);
long long train_loss_ws_bytes();
int train_loss_fwd(bool bf16, const void* pred, const void* target, long long n, const void* concept, long long m, const void* vnorm,
                   long long k, float w_text, float w_vis, float* out4, void* ws, cudaStream_t stream);
int train_loss_bwd(bool bf16, const void* pred, const void* target, long long n, const void* concept, long long m, long long k,
                   float w_text, float w_vis, const float* gloss, void* d_pred, void* d_concept, void* d_vnorm, cudaStream_t stream);
bool lora_bwd_supported(int in_f, int out_f, int r);
long long lora_bwd_ws_bytes(long long M, int in_f, int out_f, int r);
int lora_bwd(bool bf16, const void* X, const void* G, const float* A, const float* Bm, float scaling, float* dAB, void* ws,
             long long M, int in_f, int out_f, int r, long long ldx, long long ldg, cudaStream_t stream);
int attn_bwd_chunks_used(bool bf16, int S, int d);
int dual_attn_bwd(bool bf16, const void* dO, const void* Q, const float* kv_text, const float* kv_img, const float* stats,
                  void* dQ, float* part, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                  cudaStream_t stream);
int kv_pack_bwd(bool bf16, const float* part, const float* kv_img, const float* v_ip_norm, const float* d_vnorm,
                void* dkv_text, void* dkv_img, int nchunk, int B, int Lt, int Li, int C, int H, cudaStream_t stream);

int inject_concept_fwd(bool bf16, const void* in, const void* concept, const int* idx, void* out, int B, int L, int T,
                       int cols, cudaStream_t stream);
int inject_concept_bwd(bool bf16, const void* dout, const int* idx, void* din, void* dconcept, int B, int L, int T, int cols,
                       cudaStream_t stream);
long long group_norm_nhwc_ws_bytes(long long B, long long HW, int C, int G);
int group_norm_nhwc(const void* x, const float* add_bc, const float* gamma, const float* beta, void* y, float* save_stats,
                    void* ws, long long B, long long HW, int C, int G, float eps, bool silu, cudaStream_t stream);
int group_norm_nhwc_bwd(const void* x, const float* add_bc, const void* dy, const float* stats, const float* gamma,
                        const float* beta, void* dx, void* ws, long long B, long long HW, int C, int G, bool silu,
                        cudaStream_t stream);
int add_bias_nhwc(const void* a, const void* b, const float* bias, void* out, long long rows, int C, cudaStream_t stream);
int layer_norm_bf16(const void* x, const void* res, void* sum_out, const float* gamma, const float* beta, void* y, long long rows,
                    int C, float eps, cudaStream_t stream);
int layer_norm_bwd_bf16(const void* x, const void* dy, const float* gamma, void* dx, long long rows, int C, float eps,
                        cudaStream_t stream);
int geglu(const void* h, void* y, long long M, int N, long long ldh, cudaStream_t stream);
int linear_geglu_bf16(const void* x, const void* Wp, const float* bp, void* y, long long M, long long N, long long K,
                      long long ldx, long long ldy, cudaStream_t stream);
int geglu_bwd(const void* h, const void* dy, void* dh, long long M, int N, long long ldh, cudaStream_t stream);
int dropout_bwd_acc(bool bf16, void* dst, const void* src, const uint8_t* mask, float alpha, long long n,
                    cudaStream_t stream);

// ---- globals ---------------------------------------------------------------------------------------
std::atomic<unsigned long long> g_launches{0};
// Test / A-B switches (pv_set_option; process-wide, NOT thread-safe, never needed in production): every value selects
// among correct kernels -- none changes results.
int g_opt_epi_swizzle = 1;       // pv_gemm.cu: swizzled epilogue staging tile
int g_opt_force_bn = 0;          // pv_gemm.cu: force the N tile (64/128/160/256) instead of the wave-count pick
int g_opt_gemm_two_cta = 1;      // pv_gemm.cu: two resident CTAs per SM for short K
int g_opt_pdl = 1;               // programmatic dependent launch for the persistent kernels
int g_opt_gemm_persistent = 1;   // persistent CTA-pair GEMM (pv_gemm3.cu) for the out projection shapes
int g_opt_fuse_out = 1;          // out projection as the second phase of the attention launch: 1 = where it is at least as
                                 // fast as two launches (C <= 320, measured: DESIGN.md 4.2), 2 = every S > 128 shape, 0 = never
int g_opt_bwd_mma = 1;           // bf16 attention backward on tensor cores (0: fp32-accurate SIMT kernel)
unsigned long long* g_attn3_trace = nullptr;   // debug timeline buffer (pv_debug_trace; kernels record only in -DPV_TRACE builds)
int g_attn3_trace_cap = 0;
int g_opt_bwd_tc = 1;            // tcgen05 attention backward for head_dim 40 / 80 (0: the mma.sync kernel)
int g_opt_sattn_poly = 2;        // pv_sattn.cu: exponentials per 8 pairs computed on the FMA pipe instead of MUFU (0 | 2 | 4)
int g_opt_attn6_prefetch = 1;    // pv_attn6.cu: softmax warps fetch the next head's S row under the current head's P pack
int g_opt_attn6_token = 1;       // pv_attn6.cu, head_dim 40: the two softmax groups take turns on the exponentials (MUFU token)
int g_opt_trace_block = 0;       // which leader CTA writes the debug timeline
static thread_local std::string t_error;

void set_error(const std::string& msg) { t_error = msg; }
const char* last_error_cstr() { return t_error.c_str(); }

int sm_count() {
  static std::atomic<int> cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  int n = cache[dev].load(std::memory_order_relaxed);
  if (n == 0) {
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cache[dev].store(n, std::memory_order_relaxed);
  }
  return n;
}

cudaError_t set_max_smem_once_impl(const void* kern, int bytes, bool max_carveout) {
  static std::mutex mu;
  static std::unordered_map<uint64_t, int> done;       // (kernel, device) -> bytes already granted
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const uint64_t key = reinterpret_cast<uint64_t>(kern) * 131u + static_cast<uint64_t>(dev);
  std::lock_guard<std::mutex> lk(mu);
  auto it = done.find(key);
  if (it != done.end() && it->second >= bytes) return cudaSuccess;
  e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  // several CTAs of this kernel are meant to share an SM: ask for the largest shared-memory carve-out
  if (e == cudaSuccess && max_carveout)
    e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  if (e == cudaSuccess) done[key] = bytes;
  return e;
}

// ---- TMA descriptor encoding (driver entry point fetched through the runtime: no link against libcuda) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  });
  return fn;
}

struct TmapKey {
  uint64_t v[12];
  bool operator==(const TmapKey& o) const { return memcmp(v, o.v, sizeof(v)) == 0; }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = 1469598103934665603ull;
    for (uint64_t x : k.v) { h ^= x; h *= 1099511628211ull; }
    return static_cast<size_t>(h);
  }
};

int make_tmap_3d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t d0, uint64_t d1, uint64_t d2,
                 uint64_t stride1_bytes, uint64_t stride2_bytes, uint32_t b0, uint32_t b1, uint32_t b2, Swz swz, bool f16) {
  static std::mutex mu;
  static std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> cache;
  TmapKey key = {{reinterpret_cast<uint64_t>(base), static_cast<uint64_t>(elem_bytes), d0, d1, d2, stride1_bytes,
                  stride2_bytes, b0, b1, b2, static_cast<uint64_t>(swz), static_cast<uint64_t>(f16)}};
  {
    std::lock_guard<std::mutex> lk(mu);
    auto it = cache.find(key);
    if (it != cache.end()) { *out = it->second; return 0; }
  }
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver / device)"); return 1; }
  CUtensorMapDataType dt = elem_bytes != 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                           : f16       ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {stride1_bytes, stride2_bytes};
  cuuint32_t box[3] = {b0, b1, b2};
  cuuint32_t estr[3] = {1, 1, 1};
  CUtensorMapSwizzle sw = swz == Swz::B128 ? CU_TENSOR_MAP_SWIZZLE_128B
                          : swz == Swz::B64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = fn(out, dt, 3, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char buf[384];
    snprintf(buf, sizeof(buf),
             "cuTensorMapEncodeTiled failed (%d): base=%p elem=%d dims=(%llu,%llu,%llu) strides=(%llu,%llu) box=(%u,%u,%u) swz=%d",
             (int)r, base, elem_bytes, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)d2,
             (unsigned long long)stride1_bytes, (unsigned long long)stride2_bytes, b0, b1, b2, (int)swz);
    set_error(buf);
    return 1;
  }
  {
    std::lock_guard<std::mutex> lk(mu);
    if (cache.size() > 8192) cache.clear();
    cache.emplace(key, *out);
  }
  return 0;
}

static inline cudaStream_t as_stream(void* s) { return static_cast<cudaStream_t>(s); }
static inline bool is_16bit(pv_dtype dt) { return dt == PV_BF16 || dt == PV_F16; }
// PV_F16 is an inference dtype: entry points outside the no-grad processor / adapter path reject it by name.
#define PV_NO_F16(dt)                                                                                             \
  do {                                                                                                            \
    if ((dt) == PV_F16) PV_FAIL(PV_ERR_UNSUPPORTED, "PV_F16 is not supported (fp16 runs the inference path only)"); \
  } while (0)

// Fused Q projection + dual-branch attention (+ out projection when Wo is given and the shape family supports the
// single-launch form).  Shape families: S > 128: CTA-pair kernels (pv_attn6.cu for head_dim 40 at C = 320 and head_dim 80,
// pv_attn4.cu otherwise); S <= 128 (a single 128-row tile per sample): the single-CTA persistent kernel of pv_attn3.cu.
// Returns through *fused whether Y has been produced.
// f16: fp16 operands instead of bf16 (same kernels, same launch policy).
static int attn_core_bf16(const void* X, const void* Wq, const void* Kp, const void* Vp, void* O, float* stats, int B,
                          int S, int C, int H, int Lt, int Li, float w_text, float w_img, cudaStream_t st, bool f16,
                          const void* Wo = nullptr, const float* bo = nullptr, void* Y = nullptr, unsigned int* sync = nullptr,
                          bool* fused = nullptr) {
  if (fused) *fused = false;
  if (S > 128) {
    // Single launch where it pays: with G = C / 160 <= 2 column groups the pairs that share a row block run in lockstep and
    // the second phase starts at once; with more groups the wait for the slowest of G pairs (plus the announcement
    // round trip) costs ~1 us more than the launch boundary it replaces (tools/attn_bench.py, DESIGN.md 4.2).
    const bool want = Wo != nullptr && sync != nullptr && (g_opt_fuse_out >= 2 || (g_opt_fuse_out == 1 && C <= 320));
    if (dual_attn_pair_roles_supported(S, C, H)) {
      const bool f = want && dual_attn_pair_roles_fused_supported(S, C, H);
      if (fused) *fused = f;
      return dual_attn_core_bf16_pair_roles(X, Wq, Kp, Vp, O, stats, B, S, C, H, Lt, Li, w_text, w_img, st,
                                            f ? Wo : nullptr, bo, f ? Y : nullptr, f ? sync : nullptr, f16);
    }
    if (fused) *fused = want;
    return dual_attn_core_bf16_pair(X, Wq, Kp, Vp, O, stats, B, S, C, H, Lt, Li, w_text, w_img, st, want ? Wo : nullptr, bo,
                                    want ? Y : nullptr, want ? sync : nullptr, f16);
  }
  return dual_attn_core_bf16_persistent(X, Wq, Kp, Vp, O, stats, B, S, C, H, Lt, Li, w_text, w_img, st, f16);
}

}  // namespace pv

using namespace pv;

extern "C" {

int pv_version(void) { return PV_ABI_VERSION; }
const char* pv_last_error(void) { return last_error_cstr(); }
unsigned long long pv_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int pv_set_option(const char* name, int value) {
  if (!name) PV_FAIL(PV_ERR_INVALID, "null option name");
  if (!strcmp(name, "epi_swizzle")) { g_opt_epi_swizzle = value; return PV_OK; }
  if (!strcmp(name, "force_bn")) { g_opt_force_bn = value; return PV_OK; }
  if (!strcmp(name, "gemm_two_cta")) { g_opt_gemm_two_cta = value; return PV_OK; }
  if (!strcmp(name, "gemm_persistent")) { g_opt_gemm_persistent = value; return PV_OK; }
  if (!strcmp(name, "fuse_out")) { g_opt_fuse_out = value; return PV_OK; }
  if (!strcmp(name, "pdl")) { g_opt_pdl = value; return PV_OK; }
  if (!strcmp(name, "bwd_mma")) { g_opt_bwd_mma = value; return PV_OK; }
  if (!strcmp(name, "bwd_tc")) { g_opt_bwd_tc = value; return PV_OK; }
  if (!strcmp(name, "sattn_poly")) { g_opt_sattn_poly = value; return PV_OK; }
  if (!strcmp(name, "attn6_prefetch")) { g_opt_attn6_prefetch = value; return PV_OK; }
  if (!strcmp(name, "attn6_token")) { g_opt_attn6_token = value; return PV_OK; }
  if (!strcmp(name, "trace_block")) { g_opt_trace_block = value; return PV_OK; }
  PV_FAIL(PV_ERR_INVALID, "unknown option '%s'", name);
}

int pv_debug_trace(void* buf, int capacity_events) {
#ifdef PV_TRACE
  g_attn3_trace = static_cast<unsigned long long*>(buf);
  g_attn3_trace_cap = buf ? capacity_events : 0;
  return PV_OK;
#else
  (void)capacity_events;
  if (buf == nullptr) return PV_OK;
  PV_FAIL(PV_ERR_INVALID, "this build records no device timeline (rebuild with PV_TRACE=1 python -m photoverse_b200.build --force)");
#endif
}

int pv_pack_weight(pv_dtype out_dt, const float* W, const float* lora_A, const float* lora_B, float scaling,
                   void* W_eff, int out_features, int in_features, int r, void* stream) {
  PV_REQUIRE(W && W_eff, "null pointer");
  PV_REQUIRE(out_dt == PV_F32 || is_16bit(out_dt), "unknown dtype %d", (int)out_dt);
  return pack_weight(out_dt, W, lora_A, lora_B, scaling, W_eff, out_features, in_features, r, as_stream(stream));
}

int pv_linear_fwd(pv_dtype dt, pv_dtype out_dt, const void* A, const void* W, const float* bias, void* D, int64_t M,
                  int64_t N, int64_t K, int64_t batch, int64_t lda, int64_t ldw, int64_t ldd, int64_t strideA,
                  int64_t strideW, int64_t strideBias, int64_t strideD, void* stream) {
  PV_REQUIRE(A && W && D, "null pointer");
  if (is_16bit(dt)) {
    PV_REQUIRE(out_dt == dt || out_dt == PV_F32, "%s inputs produce %s or fp32 outputs", dt == PV_F16 ? "PV_F16" : "PV_BF16",
               dt == PV_F16 ? "PV_F16" : "PV_BF16");
    return gemm_bf16(A, W, bias, D, out_dt == PV_F32, M, N, K, batch, lda, ldw, ldd, strideA, strideW, strideBias,
                     strideD, as_stream(stream), /*w_static=*/false, dt == PV_F16);
  }
  PV_REQUIRE(out_dt == PV_F32, "fp32 inputs produce fp32 outputs");
  return gemm_f32(static_cast<const float*>(A), static_cast<const float*>(W), bias, static_cast<float*>(D), M, N, K,
                  batch, lda, ldw, ldd, strideA, strideW, strideBias, strideD, as_stream(stream));
}

int64_t pv_kv_tile_bytes(pv_dtype dt, int C, int H, int Lt, int Li) {
  if (H <= 0 || C % H != 0) return -1;
  const int d = C / H;
  if (is_16bit(dt)) return attn_kv_tile_bytes(d);
  return static_cast<int64_t>(Lt + Li) * d * 4;
}

int pv_kv_pack_fwd(pv_dtype dt, const void* text, const void* img, const void* Wkv_text, const void* Wkv_img,
                   float* kv_text_ws, float* kv_img_ws, void* Kp, void* Vp, float* v_ip_norm, int B, int Lt, int Li,
                   int Dc, int C, int H, void* stream) {
  PV_REQUIRE(text && img && Wkv_text && Wkv_img && kv_text_ws && kv_img_ws && Kp && Vp && v_ip_norm, "null pointer");
  PV_REQUIRE(B > 0 && Lt >= 1 && Li >= 1 && Lt + Li <= PV_KEYS_PAD && C > 0 && H > 0 && C % H == 0 && Dc > 0,
             "bad shape B=%d Lt=%d Li=%d Dc=%d C=%d H=%d", B, Lt, Li, Dc, C, H);
  PV_REQUIRE(dt == PV_F32 || is_16bit(dt), "unknown dtype %d", (int)dt);
  PV_REQUIRE(!is_16bit(dt) || (Lt <= PV_IMG_KEY_OFFSET && Li <= PV_KEYS_PAD - PV_IMG_KEY_OFFSET),
             "PV_BF16 / PV_F16 tiles hold at most %d text and %d image keys (Lt=%d Li=%d)", PV_IMG_KEY_OFFSET,
             PV_KEYS_PAD - PV_IMG_KEY_OFFSET, Lt, Li);
  cudaStream_t st = as_stream(stream);
  int rc;
  if (is_16bit(dt)) {
    const bool f16 = dt == PV_F16;
    rc = gemm_bf16(text, Wkv_text, nullptr, kv_text_ws, true, (long long)B * Lt, 2 * C, Dc, 1, Dc, Dc, 2 * C, 0, 0, 0, 0, st,
                   false, f16);
    if (rc) return rc;
    rc = gemm_bf16(img, Wkv_img, nullptr, kv_img_ws, true, (long long)B * Li, 2 * C, Dc, 1, Dc, Dc, 2 * C, 0, 0, 0, 0, st,
                   false, f16);
    if (rc) return rc;
  } else {
    rc = gemm_f32(static_cast<const float*>(text), static_cast<const float*>(Wkv_text), nullptr, kv_text_ws,
                  (long long)B * Lt, 2 * C, Dc, 1, Dc, Dc, 2 * C, 0, 0, 0, 0, st);
    if (rc) return rc;
    rc = gemm_f32(static_cast<const float*>(img), static_cast<const float*>(Wkv_img), nullptr, kv_img_ws,
                  (long long)B * Li, 2 * C, Dc, 1, Dc, Dc, 2 * C, 0, 0, 0, 0, st);
    if (rc) return rc;
  }
  return kv_pack(dt, kv_text_ws, kv_img_ws, Kp, Vp, v_ip_norm, B, Lt, Li, C, H, st);
}

int64_t pv_dual_attn_sync_words(int B, int S) {
  if (B <= 0 || S <= 0) return -1;
  return 2ll * B * ((S + 255) / 256);
}

int pv_dual_attn_fwd(pv_dtype dt, const void* X, const void* Wq, const void* Kp, const void* Vp, const void* Wo,
                     const float* bo, void* Y, float* ws_q, void* ws_o, float* stats, unsigned int* ws_sync, int B, int S,
                     int C, int H, int Lt, int Li, float w_text, float w_img, void* stream) {
  PV_REQUIRE(X && Wq && Kp && Vp && Wo && Y && ws_o, "null pointer");
  cudaStream_t st = as_stream(stream);
  int rc;
  if (is_16bit(dt)) {
    const bool f16 = dt == PV_F16;
    bool fused = false;
    rc = attn_core_bf16(X, Wq, Kp, Vp, ws_o, stats, B, S, C, H, Lt, Li, w_text, w_img, st, f16, Wo, bo, Y, ws_sync, &fused);
    if (rc || fused) return rc;
    return gemm_bf16(ws_o, Wo, bo, Y, false, (long long)B * S, C, C, 1, C, C, C, 0, 0, 0, 0, st, /*w_static=*/true, f16);
  }
  PV_REQUIRE(dt == PV_F32, "unknown dtype %d", (int)dt);
  PV_REQUIRE(ws_q != nullptr, "PV_F32 needs the ws_q scratch");
  rc = gemm_f32(static_cast<const float*>(X), static_cast<const float*>(Wq), nullptr, ws_q, (long long)B * S, C, C, 1, C,
                C, C, 0, 0, 0, 0, st);
  if (rc) return rc;
  rc = dual_attn_core_f32(ws_q, static_cast<const float*>(Kp), static_cast<const float*>(Vp),
                          static_cast<float*>(ws_o), stats, B, S, C, H, Lt, Li, w_text, w_img, st);
  if (rc) return rc;
  return gemm_f32(static_cast<const float*>(ws_o), static_cast<const float*>(Wo), bo, static_cast<float*>(Y),
                  (long long)B * S, C, C, 1, C, C, C, 0, 0, 0, 0, st);
}

int pv_dual_attn_core_fwd(pv_dtype dt, const void* XorQ, const void* Wq, const void* Kp, const void* Vp, void* O,
                          float* stats, int B, int S, int C, int H, int Lt, int Li, float w_text, float w_img,
                          void* stream) {
  PV_REQUIRE(XorQ && Kp && Vp && O, "null pointer");
  if (is_16bit(dt)) {
    PV_REQUIRE(Wq != nullptr, "PV_BF16 / PV_F16 fuse the Q projection: Wq required");
    return attn_core_bf16(XorQ, Wq, Kp, Vp, O, stats, B, S, C, H, Lt, Li, w_text, w_img, as_stream(stream), dt == PV_F16);
  }
  PV_REQUIRE(dt == PV_F32, "unknown dtype %d", (int)dt);
  return dual_attn_core_f32(static_cast<const float*>(XorQ), static_cast<const float*>(Kp),
                            static_cast<const float*>(Vp), static_cast<float*>(O), stats, B, S, C, H, Lt, Li, w_text,
                            w_img, as_stream(stream));
}

int pv_ln_lrelu_fwd(pv_dtype out_dt, const float* x, const float* gamma, const float* beta, void* y, float* save_mean,
                    float* save_rstd, int64_t rows, int cols, int64_t ldx, int64_t ldy, int64_t rows_per_group,
                    float eps, float slope, void* stream) {
  PV_REQUIRE(x && gamma && beta && y, "null pointer");
  PV_REQUIRE(out_dt == PV_F32 || is_16bit(out_dt), "unknown dtype %d", (int)out_dt);
  return ln_lrelu(out_dt, x, gamma, beta, y, save_mean, save_rstd, rows, cols, ldx, ldy, rows_per_group, eps,
                  slope, as_stream(stream));
}

int pv_group_mean_fwd(pv_dtype in_dt, pv_dtype out_dt, const void* x, void* y, int64_t groups, int P, int cols,
                      int64_t ldy, void* stream) {
  PV_REQUIRE(x && y, "null pointer");
  PV_REQUIRE((in_dt == PV_F32 || is_16bit(in_dt)) && (out_dt == PV_F32 || is_16bit(out_dt)), "unknown dtype");
  PV_REQUIRE(!(is_16bit(in_dt) && is_16bit(out_dt) && in_dt != out_dt), "16-bit input and output must have one type");
  return group_mean(in_dt, out_dt, x, y, groups, P, cols, ldy, as_stream(stream));
}

// ---------------------------------------------------------------------------------------------------------
// backward entry points
// ---------------------------------------------------------------------------------------------------------
int pv_pack_weight_t(pv_dtype out_dt, const float* W, const float* lora_A, const float* lora_B, float scaling,
                     void* W_eff_t, int out_features, int in_features, int r, void* stream) {
  PV_NO_F16(out_dt);
  PV_REQUIRE(W && W_eff_t, "null pointer");
  return pack_weight_t(out_dt == PV_BF16, W, lora_A, lora_B, scaling, W_eff_t, out_features, in_features, r, as_stream(stream));
}

int pv_transpose_2d(pv_dtype dt, const void* in, void* out, int64_t rows, int64_t cols, int64_t ldi, int64_t ldo, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(in && out, "null pointer");
  return transpose_2d(dt == PV_BF16, in, out, rows, cols, ldi, ldo, as_stream(stream));
}

int64_t pv_linear_bwd_weight_ws_bytes(pv_dtype dt, int64_t M, int64_t N, int64_t K) {
  if (dt == PV_F16) { set_error("pv_linear_bwd_weight_ws_bytes: PV_F16 is not supported (fp16 runs the inference path only)"); return -1; }
  return wgrad_ws_bytes(dt == PV_BF16, M, N, K);
}

int pv_linear_bwd_weight(pv_dtype dt, const void* G, const void* X, float* dW, void* ws, int64_t M, int64_t N, int64_t K,
                         int64_t ldg, int64_t ldx, float alpha, float beta, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(G && X && dW, "null pointer");
  return linear_bwd_weight(dt == PV_BF16, G, X, dW, ws, M, N, K, ldg, ldx, alpha, beta, as_stream(stream));
}

int64_t pv_lora_bwd_ws_bytes(int64_t M, int in_features, int out_features, int r) {
  if (M <= 0 || !lora_bwd_supported(in_features, out_features, r)) return -1;       // -1: use the GEMM route
  return lora_bwd_ws_bytes(M, in_features, out_features, r);
}

int pv_lora_bwd(pv_dtype dt, const void* X, const void* G, const float* lora_A, const float* lora_B, float scaling, float* dAB,
                void* ws, int64_t M, int in_features, int out_features, int r, int64_t ldx, int64_t ldg, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(X && G && lora_A && lora_B && dAB, "null pointer");
  return lora_bwd(dt == PV_BF16, X, G, lora_A, lora_B, scaling, dAB, ws, M, in_features, out_features, r, ldx, ldg, as_stream(stream));
}

int64_t pv_col_sum_ws_bytes(int64_t M, int64_t N) { return colsum_ws_bytes(M, N); }

int pv_col_sum(pv_dtype dt, const void* G, float* out, void* ws, int64_t M, int64_t N, int64_t ldg, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(G && out, "null pointer");
  return col_sum(dt == PV_BF16, G, out, ws, M, N, ldg, as_stream(stream));
}

int64_t pv_ln_lrelu_bwd_ws_bytes(int64_t groups, int64_t rows_per_group, int cols) {
  return ln_bwd_ws_bytes(groups, rows_per_group, cols);
}

int pv_ln_lrelu_bwd(pv_dtype dt, const void* da, const float* x, const float* mean, const float* rstd, const float* gamma,
                    const float* beta, void* dx, float* dgamma, float* dbeta, void* ws, int64_t groups,
                    int64_t rows_per_group, int cols, float slope, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(da && x && mean && rstd && gamma && beta && dx && dgamma && dbeta && ws, "null pointer");
  return ln_lrelu_bwd(dt == PV_BF16, da, x, mean, rstd, gamma, beta, dx, dgamma, dbeta, ws, groups, rows_per_group, cols,
                      slope, as_stream(stream));
}

int pv_group_mean_bwd(pv_dtype dt, const void* dy, void* dx, int64_t groups, int P, int cols, int64_t ldy, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(dy && dx, "null pointer");
  return group_mean_bwd(dt == PV_BF16, dy, dx, groups, P, cols, ldy, as_stream(stream));
}

int64_t pv_dual_attn_bwd_ws_bytes(int B, int S, int C, int H, int Lt, int Li) {
  if (H <= 0 || C % H != 0) return -1;
  return static_cast<int64_t>(attn_bwd_chunks(S)) * B * H * 2 * (Lt + Li) * (C / H) * 4;
}

int pv_dual_attn_bwd(pv_dtype dt, const void* dO, const void* Q, const float* kv_text, const float* kv_img,
                     const float* stats, void* dQ, void* ws, int B, int S, int C, int H, int Lt, int Li, float w_text,
                     float w_img, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(dO && Q && kv_text && kv_img && stats && dQ && ws, "null pointer");
  return dual_attn_bwd(dt == PV_BF16, dO, Q, kv_text, kv_img, stats, dQ, static_cast<float*>(ws), B, S, C, H, Lt, Li, w_text,
                       w_img, as_stream(stream));
}

int pv_kv_pack_bwd(pv_dtype dt, const void* ws, const float* kv_img, const float* v_ip_norm, const float* d_v_ip_norm,
                   void* dkv_text, void* dkv_img, int B, int S, int Lt, int Li, int C, int H, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(ws && kv_img && v_ip_norm && dkv_text && dkv_img, "null pointer");
  return kv_pack_bwd(dt == PV_BF16, static_cast<const float*>(ws), kv_img, v_ip_norm, d_v_ip_norm, dkv_text, dkv_img,
                     attn_bwd_chunks_used(dt == PV_BF16, S, H > 0 ? C / H : 0), B, Lt, Li, C, H, as_stream(stream));
}

int pv_inject_concept_fwd(pv_dtype dt, const void* inputs_embeds, const void* concept, const int* placeholder_idx,
                          void* out, int B, int L, int T, int cols, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(inputs_embeds && concept && placeholder_idx && out, "null pointer");
  return inject_concept_fwd(dt == PV_BF16, inputs_embeds, concept, placeholder_idx, out, B, L, T, cols, as_stream(stream));
}

int pv_inject_concept_bwd(pv_dtype dt, const void* d_out, const int* placeholder_idx, void* d_inputs_embeds,
                          void* d_concept, int B, int L, int T, int cols, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(d_out && placeholder_idx && d_inputs_embeds && d_concept, "null pointer");
  return inject_concept_bwd(dt == PV_BF16, d_out, placeholder_idx, d_inputs_embeds, d_concept, B, L, T, cols, as_stream(stream));
}

int64_t pv_train_loss_ws_bytes(void) { return train_loss_ws_bytes(); }

int pv_train_loss_fwd(pv_dtype dt, const void* noise_pred, const void* noise, int64_t n, const void* concept, int64_t m,
                      const void* v_ip_norms, int64_t k, float w_text, float w_vis, float* out4, void* ws, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(noise_pred && noise && out4 && (m == 0 || concept) && (k == 0 || v_ip_norms), "null pointer");
  return train_loss_fwd(dt == PV_BF16, noise_pred, noise, n, concept, m, v_ip_norms, k, w_text, w_vis, out4, ws, as_stream(stream));
}

int pv_train_loss_bwd(pv_dtype dt, const void* noise_pred, const void* noise, int64_t n, const void* concept, int64_t m, int64_t k,
                      float w_text, float w_vis, const float* d_loss, void* d_noise_pred, void* d_concept, void* d_v_ip_norms,
                      void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(noise_pred && noise && d_loss && d_noise_pred && (m == 0 || (concept && d_concept)) && (k == 0 || d_v_ip_norms), "null pointer");
  return train_loss_bwd(dt == PV_BF16, noise_pred, noise, n, concept, m, k, w_text, w_vis, d_loss, d_noise_pred, d_concept,
                        d_v_ip_norms, as_stream(stream));
}

int64_t pv_self_attn_ws_bytes(int B, int S, int C, int heads) { return self_attn_ws_bytes(B, S, C, heads); }

int pv_self_attn_fwd(const void* q, const void* k, const void* v, int64_t ld, void* out, void* ws, int B, int S, int C,
                     int heads, void* stream) {
  PV_REQUIRE(q && k && v && out && ws, "null pointer");
  return self_attn_fwd_bf16(q, k, v, ld, out, ws, B, S, C, heads, as_stream(stream));
}

int pv_dropout_bwd_acc(pv_dtype dt, void* dst, const void* src, const uint8_t* keep_mask, float alpha, int64_t n,
                       void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(dst && src && keep_mask, "null pointer");
  return dropout_bwd_acc(dt == PV_BF16, dst, src, keep_mask, alpha, n, as_stream(stream));
}

int64_t pv_group_norm_nhwc_ws_bytes(int64_t B, int64_t HW, int C, int groups) { return group_norm_nhwc_ws_bytes(B, HW, C, groups); }

int pv_group_norm_nhwc_fwd(pv_dtype dt, const void* x, const float* add_bc, const float* gamma, const float* beta, void* y,
                           float* save_stats, void* ws, int64_t B, int64_t HW, int C, int groups, float eps, int silu,
                           void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(x && gamma && beta && y && ws, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only (the fp32 parity mode keeps the stock GroupNorm)");
  return group_norm_nhwc(x, add_bc, gamma, beta, y, save_stats, ws, B, HW, C, groups, eps, silu != 0, as_stream(stream));
}

int pv_group_norm_nhwc_bwd(pv_dtype dt, const void* x, const float* add_bc, const void* dy, const float* stats,
                           const float* gamma, const float* beta, void* dx, void* ws, int64_t B, int64_t HW, int C, int groups,
                           int silu, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(x && dy && stats && gamma && beta && dx && ws, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return group_norm_nhwc_bwd(x, add_bc, dy, stats, gamma, beta, dx, ws, B, HW, C, groups, silu != 0, as_stream(stream));
}

int pv_add_bias_nhwc_fwd(pv_dtype dt, const void* a, const void* b, const float* bias, void* out, int64_t rows, int C,
                         void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(a && b && bias && out, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return add_bias_nhwc(a, b, bias, out, rows, C, as_stream(stream));
}

int pv_layer_norm_fwd(pv_dtype dt, const void* x, const void* residual, void* sum_out, const float* gamma, const float* beta,
                      void* y, int64_t rows, int C, float eps, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(x && gamma && beta && y, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return layer_norm_bf16(x, residual, sum_out, gamma, beta, y, rows, C, eps, as_stream(stream));
}

int pv_layer_norm_bwd(pv_dtype dt, const void* x, const void* dy, const float* gamma, void* dx, int64_t rows, int C, float eps,
                      void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(x && dy && gamma && dx, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return layer_norm_bwd_bf16(x, dy, gamma, dx, rows, C, eps, as_stream(stream));
}

int pv_geglu_fwd(pv_dtype dt, const void* h, void* y, int64_t M, int N, int64_t ldh, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(h && y, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return geglu(h, y, M, N, ldh, as_stream(stream));
}

int pv_geglu_bwd(pv_dtype dt, const void* h, const void* dy, void* dh, int64_t M, int N, int64_t ldh, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(h && dy && dh, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return geglu_bwd(h, dy, dh, M, N, ldh, as_stream(stream));
}

int pv_linear_geglu_fwd(pv_dtype dt, const void* x, const void* w_packed, const float* b_packed, void* y, int64_t M, int64_t N,
                        int64_t K, int64_t ldx, int64_t ldy, void* stream) {
  PV_NO_F16(dt);
  PV_REQUIRE(x && w_packed && y, "null pointer");
  PV_REQUIRE(dt == PV_BF16, "bf16 activations only");
  return linear_geglu_bf16(x, w_packed, b_packed, y, M, N, K, ldx, ldy, as_stream(stream));
}

}  // extern "C"
