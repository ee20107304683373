// Per-image PSNR and SSIM of an SR / HR batch (the reference's validation metric, src/utils.py:141-151); see metrics.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>

namespace srg {

// fp64 scratch slots of one srg_image_metrics call: 2 per (image, band, column chunk); depends on N, H, W only
size_t image_metrics_scratch_bytes(int N, int H, int W);
// sr, hr: fp32 [N][3][H][W]; psnr[n], ssim[n]: DEVICE doubles.  Two launches, no allocation, copy or host sync.
int launch_image_metrics(const float* sr, const float* hr, int N, int H, int W, double* scratch, double* psnr, double* ssim,
                         cudaStream_t st);

}  // namespace srg
