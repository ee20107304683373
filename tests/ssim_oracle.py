"""fp64 CPU restatement of the reference's SSIM metric (src/utils.py:148-151).  TEST INFRASTRUCTURE ONLY: imported by
tests/test_metrics_*.py and tools/time_metrics.py as the checker of srg_image_metrics, never by the product package.
PSNR, the other half of the metric, is oracle.srgan_oracle.psnr."""
from __future__ import annotations

import torch
import torch.nn.functional as F

Tensor = torch.Tensor


def ssim(a: Tensor, b: Tensor) -> float:
    """structural_similarity(a, b, win_size=3, multichannel=True) on 3 x H x W arrays.  Under scikit-image 0.25
    ``multichannel`` lands in ``**kwargs``, so the array is one 3-D volume: 3x3x3 uniform window, sample covariance
    (27/26), C1 = (0.01)^2, C2 = (0.03)^2 with data_range 1, the SSIM map cropped by 1 on every axis and averaged.
    avg_pool3d without padding yields exactly the cropped windows (channel 1, rows 1..H-2, columns 1..W-2).  fp64."""
    if a.shape != b.shape or a.dim() != 3 or a.shape[0] != 3 or a.shape[1] < 3 or a.shape[2] < 3:
        raise ValueError(f"ssim: two 3 x H x W arrays with H, W >= 3, got {tuple(a.shape)} and {tuple(b.shape)}")
    x, y = a.double(), b.double()

    def box(t: Tensor) -> Tensor:
        return F.avg_pool3d(t[None, None], 3, stride=1)[0, 0]

    ux, uy = box(x), box(y)
    cov_norm = 27.0 / 26.0
    vx = cov_norm * (box(x * x) - ux * ux)
    vy = cov_norm * (box(y * y) - uy * uy)
    vxy = cov_norm * (box(x * y) - ux * uy)
    c1, c2 = 0.01 ** 2, 0.03 ** 2
    s = ((2 * ux * uy + c1) * (2 * vxy + c2)) / ((ux * ux + uy * uy + c1) * (vx + vy + c2))
    return float(s.mean())
