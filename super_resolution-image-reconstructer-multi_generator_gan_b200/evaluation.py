"""Evaluation-side pieces of the reference (SURVEY 8f-1 / f-2): checkpoint interop, ImageEnhancer, PSNR.

* ``load_reference_checkpoint``: the reference saves ``state_dict()`` of DDP-wrapped modules (keys prefixed with
  ``module.``, src/train.py:123-125) and strips the prefix when evaluating (src/evaluation.py:24-31); both spellings
  load here, into SRResNet or Discriminator.
* ``resume_learning_rates``: the ``continue_training`` protocol (src/train.py:51-59) divides both learning rates by 5.
* ``ImageEnhancer``: src/models.py:28-41 (Laplacian sharpening + clamp), one fused kernel.
* ``calculate_psnr``: src/utils.py:141-144 (skimage PSNR with data_range=1 over the whole tensor) on the device.
* ``calculate_ssim``: src/utils.py:148-151 (skimage SSIM, win_size=3, the 3 x H x W array as one 3-D volume).
* ``image_metrics``: both per image for a whole batch in one pass, without a host sync (train.compute_score).
"""
from __future__ import annotations

import math
from collections import OrderedDict
from ctypes import c_void_p
from typing import Mapping, Tuple

import torch

from . import _lib
from ._lib import check, stream_ptr


def strip_module_prefix(state_dict: Mapping[str, torch.Tensor]) -> "OrderedDict[str, torch.Tensor]":
    out = OrderedDict()
    for k, v in state_dict.items():
        out[k[7:] if k.startswith("module.") else k] = v       # src/evaluation.py:26-29
    return out


def load_reference_checkpoint(module, checkpoint, strict: bool = True):
    """``checkpoint``: a path written by the reference's ``torch.save(model.state_dict(), ...)`` or a state dict."""
    if not isinstance(checkpoint, Mapping):
        checkpoint = torch.load(checkpoint, map_location="cpu", weights_only=True)
    return module.load_state_dict(strip_module_prefix(checkpoint), strict=strict)


def save_reference_checkpoint(module, path: str, ddp_prefix: bool = True) -> None:
    """Writes what the reference's training run writes (src/train.py:123-125): the state dict of the DDP wrapper."""
    sd = module.state_dict()
    if ddp_prefix:
        sd = OrderedDict(("module." + k, v.detach().cpu().clone()) for k, v in sd.items())
    torch.save(sd, path)


def resume_learning_rates(lr_generator: float, lr_discriminator: float) -> Tuple[float, float]:
    """continue_training=True (src/train.py:51-59): both learning rates / 5 for the "Post-Training" (GAN fine-tune) run."""
    return lr_generator / 5, lr_discriminator / 5


class ImageEnhancer:
    """Drop-in for the reference's ImageEnhancer (src/models.py:28-41): ``x + factor * Laplacian3x3(x)``, clamp [0, 1]."""

    def __init__(self, factor: float = 1):
        self.factor = factor

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        if not x.is_cuda or x.dim() != 4:
            raise RuntimeError("ImageEnhancer (libsrgan_b200): N x C x H x W CUDA tensors only")
        x = x.contiguous().float()
        out = torch.empty_like(x)
        N, C, H, W = x.shape
        check(_lib.lib().srg_image_enhance(c_void_p(x.data_ptr()), N, C, H, W, float(self.factor), c_void_p(out.data_ptr()),
                                           stream_ptr()), "srg_image_enhance")
        return out

    __call__ = forward


def calculate_psnr(img1: torch.Tensor, img2: torch.Tensor) -> float:
    """skimage.metrics.peak_signal_noise_ratio(img1, img2, data_range=1) as used at src/utils.py:141-144."""
    if img1.shape != img2.shape or not img1.is_cuda:
        raise RuntimeError("calculate_psnr: two CUDA tensors of the same shape")
    a, b = img1.contiguous().float(), img2.contiguous().float()
    L = _lib.lib()
    scratch = torch.empty(int(L.srg_recon_loss_scratch_bytes()), dtype=torch.uint8, device=a.device)
    out = torch.empty(1, dtype=torch.float64, device=a.device)
    check(L.srg_mse(c_void_p(a.data_ptr()), c_void_p(b.data_ptr()), a.numel(), c_void_p(scratch.data_ptr()), scratch.numel(),
                    c_void_p(out.data_ptr()), stream_ptr()), "srg_mse")
    mse = float(out.item())
    return float("inf") if mse == 0 else 10.0 * math.log10(1.0 / mse)


_METRICS_SCRATCH = {}


def image_metrics(sr: torch.Tensor, hr: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """Per-image ``(psnr, ssim)`` of an N x 3 x H x W batch pair as two float64 CUDA tensors of shape [N], without a host
    sync (capturable into a CUDA graph once warmed up).  ``psnr[n]`` equals ``calculate_psnr(sr[n], hr[n])`` (+inf for
    identical images) and ``ssim[n]`` equals ``calculate_ssim(sr[n], hr[n])``; an image's values do not depend on the
    rest of the batch.  The fp64 scratch of the reduction is cached per device, stream and (N, H, W)."""
    if sr.shape != hr.shape or sr.dim() != 4:
        raise RuntimeError(f"image_metrics: two N x 3 x H x W tensors of the same shape, got {tuple(sr.shape)} and {tuple(hr.shape)}")
    if not sr.is_cuda or not hr.is_cuda or sr.device != hr.device:
        raise RuntimeError("image_metrics: CUDA tensors on one device only (libsrgan_b200 has no CPU path)")
    a, b = sr.contiguous().float(), hr.contiguous().float()
    N, C, H, W = a.shape
    L = _lib.lib()
    key = (a.device, torch.cuda.current_stream(a.device).cuda_stream, N, H, W)    # stream-ordered reuse only
    scratch = _METRICS_SCRATCH.get(key)
    if scratch is None:
        scratch = torch.empty(max(int(L.srg_image_metrics_scratch_bytes(N, H, W)), 8), dtype=torch.uint8, device=a.device)
        _METRICS_SCRATCH[key] = scratch
    out = torch.empty(2, N, dtype=torch.float64, device=a.device)
    check(L.srg_image_metrics(c_void_p(a.data_ptr()), c_void_p(b.data_ptr()), N, C, H, W, c_void_p(scratch.data_ptr()),
                              scratch.numel(), c_void_p(out[0].data_ptr()), c_void_p(out[1].data_ptr()), stream_ptr()),
          "srg_image_metrics")
    return out[0], out[1]


def calculate_ssim(img1: torch.Tensor, img2: torch.Tensor) -> float:
    """skimage.metrics.structural_similarity(img1, img2, win_size=3, multichannel=True) as called at src/utils.py:148-151
    on one 3 x H x W image pair: under scikit-image 0.25 ``multichannel`` is swallowed by ``**kwargs``, so the array is
    one 3-D volume (3x3x3 window over channels, rows and columns; data_range 1)."""
    if img1.shape != img2.shape or not img1.is_cuda:
        raise RuntimeError("calculate_ssim: two CUDA tensors of the same shape")
    if img1.dim() != 3:
        raise RuntimeError(f"calculate_ssim: one 3 x H x W image pair, got {tuple(img1.shape)}")
    return float(image_metrics(img1[None], img2[None])[1].item())
