"""CPU tests of the validation metric (src/utils.py:141-151, src/train.py:263-294): the fp64 SSIM oracle against a
brute-force 27-point loop and a scipy restatement of scikit-image's structural_similarity, the metric's fixed points, and
the argument checks of srg_image_metrics / image_metrics / calculate_ssim, none of which needs a device."""
import itertools
import math
import os
import sys
from ctypes import c_void_p

import numpy as np
import pytest
import torch

import srgan_b200 as S
from oracle import srgan_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ssim_oracle  # noqa: E402  (tests/ssim_oracle.py)


def _brute_ssim(a: np.ndarray, b: np.ndarray) -> float:
    """The definition written out: channel 1, rows 1..H-2, columns 1..W-2, each with its full 3x3x3 window."""
    _, H, W = a.shape
    C1, C2 = 1e-4, 9e-4
    total = 0.0
    for h, w in itertools.product(range(1, H - 1), range(1, W - 1)):
        x = a[:, h - 1:h + 2, w - 1:w + 2].astype(np.float64).ravel()
        y = b[:, h - 1:h + 2, w - 1:w + 2].astype(np.float64).ravel()
        ux, uy = x.sum() / 27, y.sum() / 27
        vx = ((x * x).sum() / 27 - ux * ux) * 27 / 26
        vy = ((y * y).sum() / 27 - uy * uy) * 27 / 26
        vxy = ((x * y).sum() / 27 - ux * uy) * 27 / 26
        total += ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux * ux + uy * uy + C1) * (vx + vy + C2))
    return total / ((H - 2) * (W - 2))


def _skimage_style_ssim(a: np.ndarray, b: np.ndarray) -> float:
    """scikit-image 0.25 structural_similarity(a, b, win_size=3, data_range=1) with channel_axis=None (a 3-D volume):
    uniform_filter on every axis, sample covariance, crop by (win_size - 1) // 2 = 1 on every axis.  fp64."""
    nd = pytest.importorskip("scipy.ndimage")
    x, y = a.astype(np.float64), b.astype(np.float64)
    f = lambda t: nd.uniform_filter(t, size=3)       # noqa: E731
    ux, uy, uxx, uyy, uxy = f(x), f(y), f(x * x), f(y * y), f(x * y)
    cov_norm = 27 / 26
    vx, vy, vxy = cov_norm * (uxx - ux * ux), cov_norm * (uyy - uy * uy), cov_norm * (uxy - ux * uy)
    C1, C2 = 1e-4, 9e-4
    s = ((2 * ux * uy + C1) * (2 * vxy + C2)) / ((ux ** 2 + uy ** 2 + C1) * (vx + vy + C2))
    return float(s[1:-1, 1:-1, 1:-1].mean())


def _pairs():
    g = torch.Generator().manual_seed(3)
    for shape in [(3, 3, 3), (3, 5, 7), (3, 7, 9), (3, 16, 23)]:
        hr = torch.rand(shape, generator=g)
        yield hr + 0.05 * torch.randn(shape, generator=g), hr                        # SR = HR + noise, unclamped
        flat = 0.99 + 1e-3 * torch.randn(shape, generator=g)
        yield flat, 0.99 + 1e-3 * torch.randn(shape, generator=g)                    # near-flat bright pair


def test_oracle_matches_brute_force_window_loop():
    for a, b in _pairs():
        assert abs(ssim_oracle.ssim(a, b) - _brute_ssim(a.numpy(), b.numpy())) < 1e-12, tuple(a.shape)


def test_oracle_matches_skimage_restatement():
    for a, b in _pairs():
        assert abs(ssim_oracle.ssim(a, b) - _skimage_style_ssim(a.numpy(), b.numpy())) < 1e-12, tuple(a.shape)


def test_fixed_points_and_symmetry():
    g = torch.Generator().manual_seed(4)
    a, b = torch.rand(3, 9, 11, generator=g), torch.rand(3, 9, 11, generator=g)
    assert ssim_oracle.ssim(a, a) == pytest.approx(1.0, abs=1e-15)
    assert O.psnr(a, a) == math.inf
    c = torch.full((3, 6, 6), 0.25)
    assert ssim_oracle.ssim(c, c) == pytest.approx(1.0, abs=1e-15)
    assert ssim_oracle.ssim(a, b) == ssim_oracle.ssim(b, a)
    assert O.psnr(a, b) == O.psnr(b, a)
    for bad in [(1, 5, 5), (3, 2, 5), (3, 5, 2)]:
        with pytest.raises(ValueError):
            ssim_oracle.ssim(torch.zeros(bad), torch.zeros(bad))


def _call(L, N=2, C=3, H=8, W=8, sr=16, hr=16, scratch=16, nbytes=None, psnr=16, ssim=16):
    if nbytes is None:
        nbytes = int(L.srg_image_metrics_scratch_bytes(N, H, W))
    ptr = lambda v: c_void_p(v) if v else None       # noqa: E731  (never dereferenced: the checks come first)
    return L.srg_image_metrics(ptr(sr), ptr(hr), N, C, H, W, ptr(scratch), nbytes, ptr(psnr), ptr(ssim), None)


def test_abi_rejects_bad_arguments_without_a_device():
    L = S.lib()
    assert L.srg_image_metrics_scratch_bytes(12, 512, 1024) >= 12 * 2 * 8
    assert L.srg_image_metrics_scratch_bytes(0, 8, 8) == 0 and L.srg_image_metrics_scratch_bytes(1, 2, 8) == 0
    # the slot count depends on (H, W) only: linear in N
    assert L.srg_image_metrics_scratch_bytes(5, 37, 131) == 5 * L.srg_image_metrics_scratch_bytes(1, 37, 131)
    cases = [dict(C=1), dict(C=4), dict(H=2), dict(W=2), dict(N=0), dict(N=-1), dict(sr=0), dict(hr=0), dict(scratch=0),
             dict(psnr=0), dict(ssim=0), dict(nbytes=int(L.srg_image_metrics_scratch_bytes(2, 8, 8)) - 1), dict(nbytes=0)]
    for kw in cases:
        assert _call(L, **kw) != 0, kw
        msg = L.srg_last_error().decode()
        assert msg.startswith("image_metrics:"), (kw, msg)
    _call(L, C=1)
    assert "C=1" in L.srg_last_error().decode()
    _call(L, nbytes=8)
    assert "scratch too small" in L.srg_last_error().decode()


def test_python_wrappers_reject_cpu_tensors_and_mismatched_shapes():
    a = torch.rand(2, 3, 8, 8)
    with pytest.raises(RuntimeError, match="CUDA"):
        S.image_metrics(a, a)
    with pytest.raises(RuntimeError, match="same shape"):
        S.image_metrics(a, torch.rand(2, 3, 8, 9))
    with pytest.raises(RuntimeError, match="same shape"):
        S.image_metrics(a[0], a[0])                     # one image: not a batch
    with pytest.raises(RuntimeError, match="CUDA"):
        S.calculate_ssim(a[0], a[0])
    with pytest.raises(RuntimeError, match="same shape"):
        S.calculate_ssim(a[0], a[1, :, :7])
