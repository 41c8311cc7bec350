// photoverse_b200 -- regional identity masks (pv_ip_mask_downsample): the [1|B, H_m, W_m] mask of a diffusers caller
// (`cross_attention_kwargs={"ip_adapter_masks": [...]}`) -> the fp32 [B, S] row weights the masked attention kernels
// multiply into the image segment of each query row.
//
// The rule is diffusers 0.27.2 IPAdapterMaskProcessor.downsample(mask, batch_size, num_queries, value_embed_dim):
//   ratio = W_m / H_m, mask_h = int(sqrt(S / ratio)), + 1 when S % mask_h != 0, mask_w = S // mask_h;
//   F.interpolate(size=(mask_h, mask_w), mode="bicubic", align_corners=False), no antialias;
//   repeated to the batch when the mask has one; flattened row-major, zero-padded (or truncated) to S.
// One thread per output weight.  Source coordinates, cubic coefficients (A = -0.75) and the 16-tap sum are fp64, as
// PyTorch computes them for a float64 tensor; taps outside the mask are clamped to its border.  The kernel runs once per
// (mask, S) -- four query grids per generation -- and its result is cached by the caller.
#include <math.h>

#include "pv_host.h"
#include "../../include/photoverse_b200.h"

namespace pv {

__device__ __forceinline__ double ipm_cubic1(double x, double A) { return ((A + 2.0) * x - (A + 3.0)) * x * x + 1.0; }
__device__ __forceinline__ double ipm_cubic2(double x, double A) { return ((A * x - 5.0 * A) * x + 8.0 * A) * x - 4.0 * A; }

// floor of the source coordinate and the cubic weights of its four taps (PyTorch upsample_bicubic2d, align_corners=False)
__device__ __forceinline__ int ipm_taps(int dst, int in, int out, double w[4]) {
  const double real = (static_cast<double>(in) / out) * (dst + 0.5) - 0.5;
  const double fl = floor(real);
  const double t = real - fl;
  constexpr double A = -0.75;
  w[0] = ipm_cubic2(t + 1.0, A);
  w[1] = ipm_cubic1(t, A);
  w[2] = ipm_cubic1(1.0 - t, A);
  w[3] = ipm_cubic2(2.0 - t, A);
  return static_cast<int>(fl);
}

__global__ void __launch_bounds__(256) ip_mask_downsample_kernel(const float* __restrict__ mask, float* __restrict__ rw,
                                                                 int mask_batch, int Hm, int Wm, int B, int S, int mh,
                                                                 int mw) {
  const long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= static_cast<long long>(B) * S) return;
  const int b = static_cast<int>(i / S), s = static_cast<int>(i - static_cast<long long>(b) * S);
  if (s >= mh * mw) {                     // the grid covers fewer than S rows: diffusers zero-pads
    rw[i] = 0.f;
    return;
  }
  const int oy = s / mw, ox = s - oy * mw;
  double wy[4], wx[4];
  const int y0 = ipm_taps(oy, Hm, mh, wy), x0 = ipm_taps(ox, Wm, mw, wx);
  const float* m = mask + static_cast<size_t>(mask_batch == 1 ? 0 : b) * Hm * Wm;
  double acc = 0.0;
#pragma unroll
  for (int ky = 0; ky < 4; ++ky) {
    const int y = min(max(y0 - 1 + ky, 0), Hm - 1);
    double row = 0.0;
#pragma unroll
    for (int kx = 0; kx < 4; ++kx) {
      const int x = min(max(x0 - 1 + kx, 0), Wm - 1);
      row += wx[kx] * static_cast<double>(__ldg(m + static_cast<size_t>(y) * Wm + x));
    }
    acc += wy[ky] * row;
  }
  rw[i] = static_cast<float>(acc);
}

// diffusers' query grid of a mask: mask_h * mask_w rows, mask_h * mask_w <= S (0 when the mask is too wide or too tall
// for S: diffusers divides by zero there or interpolates to an empty grid)
static bool ip_mask_grid(int S, int Hm, int Wm, int* mh, int* mw) {
  const double ratio = static_cast<double>(Wm) / Hm;
  int h = static_cast<int>(sqrt(static_cast<double>(S) / ratio));
  if (h <= 0) return false;
  h += (S % h) != 0;
  const int w = S / h;
  if (w <= 0) return false;
  *mh = h;
  *mw = w;
  return true;
}

}  // namespace pv

using namespace pv;

extern "C" int pv_ip_mask_downsample(const float* mask, int mask_batch, int mask_h, int mask_w, float* row_weight, int B,
                                     int S, void* stream) {
  PV_REQUIRE(mask && row_weight, "null pointer");
  PV_REQUIRE(B > 0 && S > 0 && mask_h > 0 && mask_w > 0, "bad shape B=%d S=%d mask %dx%d", B, S, mask_h, mask_w);
  PV_REQUIRE(mask_batch == 1 || mask_batch == B, "the mask batch must be 1 or B (mask_batch=%d B=%d)", mask_batch, B);
  int mh = 0, mw = 0;
  PV_REQUIRE(ip_mask_grid(S, mask_h, mask_w, &mh, &mw), "a %dx%d mask has no query grid for S=%d", mask_h, mask_w, S);
  const long long n = static_cast<long long>(B) * S;
  const unsigned blocks = static_cast<unsigned>((n + 255) / 256);
  ip_mask_downsample_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(mask, row_weight, mask_batch, mask_h,
                                                                                  mask_w, B, S, mh, mw);
  PV_LAUNCHED();
  return PV_OK;
}
