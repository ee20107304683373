// Validation metric of the reference (src/train.py:263-294 compute_score through src/utils.py:141-151): per-image PSNR and
// SSIM of an SR / HR batch in one pass over both images.
//
// PSNR = skimage peak_signal_noise_ratio(a, b, data_range=1) = 10 log10(1 / mean((a - b)^2)) over all 3 H W elements.
// SSIM = skimage structural_similarity(a, b, win_size=3) on the 3 x H x W array as a 3-D volume (the reference's
// `multichannel=True` is swallowed by **kwargs, channel_axis stays None): a 3x3x3 uniform window (27 points, sample
// covariance 27/26), C1 = 1e-4, C2 = 9e-4, the map cropped by 1 on every axis.  The crop keeps channel 1, rows 1..H-2,
// columns 1..W-2 only, and each of those windows spans channels 0-2, rows h-1..h+1, columns w-1..w+1 in full.
//
// Work split (depends on H and W only, so an image's result does not depend on its batch): one warp per (image, band of
// kBandRows rows, chunk of kChunkCols columns).  A lane owns 4 adjacent columns (one float4 per channel and image when the
// rows are 16-byte aligned) and walks the band plus one halo row above and below.  Per row and column it forms the channel
// sums of x, y, x^2, y^2, xy; the window sums add exactly three such rows (no running sum down the image) and then three
// columns, the outer two from the neighbouring lanes.  A warp loads 128 columns and owns 124 of them (stride 124 keeps the
// float4 alignment); its first column has no left neighbour and belongs to the warp before.
//
// Precision: the window moments are fp64 (products of fp32 inputs are exact in fp64).  vx = (sum x^2 / 27 - ux^2) 27/26
// cancels catastrophically in fp32 on flat bright areas: at 0.99 + 1e-3 noise an all-fp32 evaluation is off by up to 3e-5
// in an image's mean SSIM.  S itself is evaluated in fp32 from the fp64 moments; every partial sum is fp64 and goes to its
// own scratch slot, which a second kernel adds per image in a fixed order (run-to-run and batch-position deterministic).
#include "metrics.cuh"

#include <math.h>
#include <stdint.h>

#include "conv_gemm.cuh"

namespace srg {

namespace {

constexpr int kBandRows = 16;
constexpr int kChunkCols = 124;           // owned columns per warp; it loads 32 lanes x 4 = 128
constexpr int kWarps = 4;                 // warps (independent items) per block
constexpr int kFinalThreads = 256;

inline int bands_of(int H) { return (H + kBandRows - 1) / kBandRows; }
inline int chunks_of(int W) { return (W + kChunkCols - 1) / kChunkCols; }

// one row of a lane's 4 columns, all 3 channels of both images; zeros outside the image
template <bool VEC>
__device__ __forceinline__ void load_row(const float* __restrict__ a, const float* __restrict__ b, size_t plane, int r, int H,
                                         int W, int c0, float (&x)[3][4], float (&y)[3][4]) {
#pragma unroll
  for (int ch = 0; ch < 3; ++ch)
#pragma unroll
    for (int i = 0; i < 4; ++i) x[ch][i] = y[ch][i] = 0.f;
  if (r < 0 || r >= H) return;
  const size_t o = size_t(r) * W + c0;
#pragma unroll
  for (int ch = 0; ch < 3; ++ch) {
    const float* pa = a + ch * plane + o;
    const float* pb = b + ch * plane + o;
    if (VEC) {
      if (c0 < W) {                        // W % 4 == 0: the float4 lies inside the row
        const float4 u = __ldg(reinterpret_cast<const float4*>(pa)), v = __ldg(reinterpret_cast<const float4*>(pb));
        x[ch][0] = u.x; x[ch][1] = u.y; x[ch][2] = u.z; x[ch][3] = u.w;
        y[ch][0] = v.x; y[ch][1] = v.y; y[ch][2] = v.z; y[ch][3] = v.w;
      }
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (c0 + i < W) { x[ch][i] = __ldg(pa + i); y[ch][i] = __ldg(pb + i); }
    }
  }
}

// channel sums of one row: sx, sy, sxx, syy, sxy per column (fp64; the products are exact)
struct Moments {
  double v[5][4];
};
__device__ __forceinline__ void row_moments(const float (&x)[3][4], const float (&y)[3][4], Moments& m) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const double a0 = x[0][i], a1 = x[1][i], a2 = x[2][i];
    const double b0 = y[0][i], b1 = y[1][i], b2 = y[2][i];
    m.v[0][i] = (a0 + a1) + a2;
    m.v[1][i] = (b0 + b1) + b2;
    m.v[2][i] = fma(a2, a2, fma(a1, a1, a0 * a0));
    m.v[3][i] = fma(b2, b2, fma(b1, b1, b0 * b0));
    m.v[4][i] = fma(a2, b2, fma(a1, b1, a0 * b0));
  }
}

// sum over the lane's owned output columns of S(h, w) for the output row between rows p (above), q and r (below)
__device__ __forceinline__ float ssim_row(const Moments& p, const Moments& q, const Moments& r, int lane, int c0, int W) {
  double win[5][4];
#pragma unroll
  for (int k = 0; k < 5; ++k) {
    double v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = (p.v[k][i] + q.v[k][i]) + r.v[k][i];
    const double left = __shfl_up_sync(0xffffffffu, v[3], 1);
    const double right = __shfl_down_sync(0xffffffffu, v[0], 1);
    win[k][0] = (left + v[0]) + v[1];
    win[k][1] = (v[0] + v[1]) + v[2];
    win[k][2] = (v[1] + v[2]) + v[3];
    win[k][3] = (v[2] + v[3]) + right;
  }
  // with sums over the 27 points: ux = Sx / 27, vx = (27 Sxx - Sx^2) / 702, vxy = (27 Sxy - Sx Sy) / 702, so
  // S = (2 Sx Sy + 729 C1)(2 Dxy + 702 C2) / ((Sx^2 + Sy^2 + 729 C1)(Dxx + Dyy + 702 C2)), D.. = 27 S.. - products
  constexpr float kC1 = 729.f * 1e-4f, kC2 = 702.f * 9e-4f;
  float acc = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int lc = 4 * lane + i, c = c0 + i;
    if (lc >= 1 && lc <= kChunkCols && c >= 1 && c <= W - 2) {
      const double sx = win[0][i], sy = win[1][i];
      const float dxx = float(fma(27.0, win[2][i], -(sx * sx)));
      const float dyy = float(fma(27.0, win[3][i], -(sy * sy)));
      const float dxy = float(fma(27.0, win[4][i], -(sx * sy)));
      const float fx = float(sx), fy = float(sy);
      const float num = (2.f * fx * fy + kC1) * (2.f * dxy + kC2);
      const float den = (fx * fx + fy * fy + kC1) * (dxx + dyy + kC2);
      acc += num / den;
    }
  }
  return acc;
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// scratch[item] = sum (sr - hr)^2 over the item's own rows / columns, scratch[items + item] = sum of its S values
template <bool VEC>
__global__ void __launch_bounds__(kWarps * 32) image_metrics_kernel(const float* __restrict__ sr, const float* __restrict__ hr,
                                                                    int H, int W, int chunks, int per_image, int items,
                                                                    double* __restrict__ scratch) {
  const int item = blockIdx.x * kWarps + int(threadIdx.x >> 5);
  if (item >= items) return;              // whole warps only
  const int lane = threadIdx.x & 31;
  const int n = item / per_image, rem = item - n * per_image;
  const int band = rem / chunks, chunk = rem - band * chunks;
  const size_t plane = size_t(H) * W;
  const float* a = sr + size_t(n) * 3 * plane;
  const float* b = hr + size_t(n) * 3 * plane;
  const int h0 = band * kBandRows;
  const int c0 = chunk * kChunkCols + 4 * lane;
  const bool owns = lane < 31;            // lane 31's columns are the next chunk's first four (PSNR ownership)
  double acc_se = 0.0, acc_s = 0.0;
  Moments m[3];
#pragma unroll
  for (int i = 0; i < kBandRows + 2; ++i) {
    const int r = h0 - 1 + i;             // halo row h0 - 1, band rows, halo row h0 + kBandRows
    if (r >= H) break;                    // rows below the image feed no output row
    float x[3][4], y[3][4];
    load_row<VEC>(a, b, plane, r, H, W, c0, x, y);
    if (owns && r >= h0 && r < h0 + kBandRows && r < H) {
      float se = 0.f;
#pragma unroll
      for (int ch = 0; ch < 3; ++ch)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float d = x[ch][k] - y[ch][k];
          se = fmaf(d, d, se);
        }
      acc_se += double(se);
    }
    row_moments(x, y, m[i % 3]);
    if (i >= 2 && r - 1 >= 1 && r - 1 <= H - 2)
      acc_s += double(ssim_row(m[(i + 1) % 3], m[(i + 2) % 3], m[i % 3], lane, c0, W));
  }
  acc_se = warp_sum(acc_se);
  acc_s = warp_sum(acc_s);
  if (lane == 0) {
    scratch[item] = acc_se;
    scratch[size_t(items) + item] = acc_s;
  }
}

// one block per image: its slots in a fixed order -> psnr[n], ssim[n]
__global__ void __launch_bounds__(kFinalThreads) image_metrics_final_kernel(const double* __restrict__ scratch, int per_image,
                                                                            int items, double n_elems, double n_windows,
                                                                            double* __restrict__ psnr, double* __restrict__ ssim) {
  __shared__ double sh[2][kFinalThreads / 32];
  const int n = blockIdx.x;
  const double* se = scratch + size_t(n) * per_image;
  const double* ss = scratch + size_t(items) + size_t(n) * per_image;
  double a = 0.0, b = 0.0;
  for (int j = threadIdx.x; j < per_image; j += kFinalThreads) { a += se[j]; b += ss[j]; }
  a = warp_sum(a);
  b = warp_sum(b);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][warp] = a; sh[1][warp] = b; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double ta = 0.0, tb = 0.0;
    for (int w = 0; w < kFinalThreads / 32; ++w) { ta += sh[0][w]; tb += sh[1][w]; }
    const double mse = ta / n_elems;
    psnr[n] = mse == 0.0 ? double(INFINITY) : 10.0 * log10(1.0 / mse);
    ssim[n] = tb / n_windows;
  }
}

}  // namespace

size_t image_metrics_scratch_bytes(int N, int H, int W) {
  if (N < 1 || H < 3 || W < 3) return 0;
  return size_t(N) * bands_of(H) * chunks_of(W) * 2 * sizeof(double);
}

int launch_image_metrics(const float* sr, const float* hr, int N, int H, int W, double* scratch, double* psnr, double* ssim,
                         cudaStream_t st) {
  const int chunks = chunks_of(W);
  const long long per_image = (long long)bands_of(H) * chunks;
  const long long items = per_image * N;
  if (items > 0x7fffffffll - kWarps) { set_error("image_metrics: batch too large"); return -101; }
  const bool vec = (W & 3) == 0 && (reinterpret_cast<uintptr_t>(sr) & 15) == 0 && (reinterpret_cast<uintptr_t>(hr) & 15) == 0;
  const int blocks = int((items + kWarps - 1) / kWarps);
  if (vec)
    image_metrics_kernel<true><<<blocks, kWarps * 32, 0, st>>>(sr, hr, H, W, chunks, int(per_image), int(items), scratch);
  else
    image_metrics_kernel<false><<<blocks, kWarps * 32, 0, st>>>(sr, hr, H, W, chunks, int(per_image), int(items), scratch);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("image_metrics launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  image_metrics_final_kernel<<<N, kFinalThreads, 0, st>>>(scratch, int(per_image), int(items), 3.0 * H * W,
                                                          double(H - 2) * double(W - 2), psnr, ssim);
  e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("image_metrics_final launch: %s", cudaGetErrorString(e)); return int(e); }
  count_launch();
  return 0;
}

}  // namespace srg
