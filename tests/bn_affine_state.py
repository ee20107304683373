"""Trained-like BatchNorm state for the generator, and the per-layer BatchNorm references the tests compare the engine with.
TEST INFRASTRUCTURE ONLY: imported by tests/test_bn_affine_*.py, never by the product package.

A freshly initialised SRResNet has gamma = 1 and beta = 0 in every BatchNorm layer and running statistics (0, 1).  With
those values a table that hands a layer another layer's gamma, a channel permutation, a missing gamma factor or a dropped
beta computes exactly what the correct code computes.  ``bn_affine_state`` gives every layer, channel and generator its
own gamma (with negative entries, in front of the ReLU too), beta and running statistics, scaled so that activations stay
O(1) through 16 residual blocks in both modes.
"""
from __future__ import annotations

from typing import Dict, List, Optional, Tuple

import torch
import torch.nn.functional as F

from oracle import srgan_oracle as O

Tensor = torch.Tensor

# Bounds the GPU tests use (the measures of tests/test_generator_gpu.py); the CPU tests show that every bug class moves the
# checked quantity by at least 10x its bound.
TOL_LAYER = 1e-2        # bf16 tensors, max error relative to the reference tensor's largest magnitude
TOL_WGRAD = 5e-3        # weight / gamma / beta / bias gradients (fp32 from identical bf16 inputs)
TOL_RUNNING = 1e-5      # running statistics against the update formula evaluated on the engine's own y
# Eval forward, 16 residual blocks, end to end against the fp32 oracle.  Calibrated from the bf16-storage model of the
# folded eval forward (``eval_forward_bf16_storage``) on the DEEP_EVAL case: max-rel 1.42e-2, PSNR 51.4 dB (psnr_rel).  The
# bound is about twice the model's error, the floor 6 dB below its PSNR.
TOL_EVAL_DEEP = 3e-2
PSNR_EVAL_DEEP = 45.0
# Eval forward, 1 or 2 residual blocks, end to end.  With trained-like BatchNorm, bf16 storage alone costs 0.77e-2 .. 0.98e-2
# end to end (53.1 .. 57.0 dB, the four shallow cases of test_bn_affine_cpu), so 1e-2 there would test rounding luck; the
# 1e-2 bound is kept for each segment the eval engine stores (the BatchNorm-folded trunk of 1 or 2 blocks, each up-sampling
# stage, the output conv), each fed the engine's own input.
TOL_EVAL_SHALLOW = 2e-2
PSNR_EVAL_SHALLOW = 47.0
DEEP_EVAL = dict(seed=61, shape=(4, 3, 64, 64), num_residuals=16)

EPS = O.BN_EPS
MOMENTUM = O.BN_MOMENTUM


def maxrel(a: Tensor, b: Tensor) -> float:
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def psnr_rel(a: Tensor, ref: Tensor) -> float:
    """PSNR of ``a`` against ``ref`` with the reference's largest magnitude as the peak (dB)."""
    a, ref = a.double().cpu(), ref.double().cpu()
    mse = float(((a - ref) ** 2).mean())
    peak = float(ref.abs().max()) ** 2
    return float("inf") if mse == 0 else 10.0 * float(torch.log10(torch.tensor(peak / mse)))


def num_blocks(sd: Dict[str, Tensor]) -> int:
    return len({k.split(".")[1] for k in sd if k.startswith("residual_blocks.") and k.endswith("conv1.weight")})


def bn_layers(sd: Dict[str, Tensor]) -> List[str]:
    """Prefixes of every BatchNorm layer in forward order: residual_blocks.0.bn1, residual_blocks.0.bn2, ..."""
    return [f"residual_blocks.{b}.bn{k}" for b in range(num_blocks(sd)) for k in (1, 2)]


def bn_affine_state(sd: Dict[str, Tensor], seed: int, k: int = 0, calib: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """A copy of ``sd`` (from ``init_srresnet_state`` or ``SRResNet().state_dict()``) with trained-like BatchNorm tensors.

    - gamma: magnitude U(0.3, 2.0), exactly 8 of the 64 channels negative, in bn1 and bn2 alike;
    - beta ~ N(0, 0.3);
    - running statistics: the batch statistics of a float64 oracle training forward (with the new gamma / beta) on a
      calibration batch, perturbed to mean + 0.25 std N(0, 1) and var U(0.5, 2); num_batches_tracked > 0.
    Every value is drawn from a generator seeded by (seed, k), so generators k = 0, 1, ... of one seed all differ.  Conv
    weights and biases are left as they are."""
    st = {key: v.detach().clone() for key, v in sd.items()}
    gen = torch.Generator().manual_seed(1_000_003 * int(seed) + 7_919 * int(k) + 17)
    for p in bn_layers(st):
        c = st[p + ".weight"].numel()
        gamma = torch.empty(c, dtype=torch.float64).uniform_(0.3, 2.0, generator=gen)
        gamma[torch.randperm(c, generator=gen)[: c // 8]] *= -1.0
        st[p + ".weight"] = gamma.float()
        st[p + ".bias"] = (0.3 * torch.randn(c, generator=gen, dtype=torch.float64)).float()
    if calib is None:
        calib = torch.rand(4, 3, 24, 24, generator=gen, dtype=torch.float64)
    taps: Dict[str, Tensor] = {}
    with torch.no_grad():
        O.srresnet_forward(to_double(st), calib.double(), training=True, update_running=False, taps=taps)
    for b in range(num_blocks(st)):
        for j in (1, 2):
            p = f"residual_blocks.{b}.bn{j}"
            y = taps[f"residual_blocks.{b}.conv{j}"]
            mean, var = y.mean(dim=(0, 2, 3)), y.var(dim=(0, 2, 3), unbiased=False)
            c = mean.numel()
            st[p + ".running_mean"] = (mean + 0.25 * var.sqrt() * torch.randn(c, generator=gen, dtype=torch.float64)).float()
            st[p + ".running_var"] = (var * torch.empty(c, dtype=torch.float64).uniform_(0.5, 2.0, generator=gen)).float()
            st[p + ".num_batches_tracked"] = torch.tensor(100 + 10 * k + b, dtype=torch.long)
    return st


def to_double(sd: Dict[str, Tensor]) -> Dict[str, Tensor]:
    return {key: v.double() if v.dtype.is_floating_point else v.clone() for key, v in sd.items()}


def deep_eval_case() -> Tuple[Dict[str, Tensor], Tensor]:
    """The 16-block eval case whose bf16-storage error calibrates TOL_EVAL_DEEP / PSNR_EVAL_DEEP: (state, input)."""
    c = DEEP_EVAL
    sd = bn_affine_state(O.init_srresnet_state(c["seed"], num_residuals=c["num_residuals"]), c["seed"])
    x = torch.rand(*c["shape"], generator=torch.Generator().manual_seed(c["seed"] + 1))
    return sd, x


# ------------------------------------------------------------------------------------------------ per-layer references
def bn_train(y: Tensor, gamma: Tensor, beta: Tensor) -> Tensor:
    return F.batch_norm(y, None, None, gamma.to(y.dtype), beta.to(y.dtype), training=True, momentum=MOMENTUM, eps=EPS)


def bn_train_bwd(y: Tensor, gamma: Tensor, beta: Tensor, dz: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """training-mode BatchNorm backward: (d y, d gamma, d beta)"""
    y = y.detach().clone().requires_grad_(True)
    gamma = gamma.to(y.dtype).clone().requires_grad_(True)
    beta = beta.to(y.dtype).clone().requires_grad_(True)
    return torch.autograd.grad(bn_train(y, gamma, beta), [y, gamma, beta], grad_outputs=dz.to(y.dtype))


def bn_eval_bwd(y: Tensor, sd: Dict[str, Tensor], p: str, dz: Tensor) -> Tuple[Tensor, Tensor, Tensor]:
    """eval-mode (running statistics) BatchNorm backward: (d y, d gamma, d beta); the preceding conv's bias gradient is
    d y summed over (N, H, W)"""
    y = y.detach().clone().requires_grad_(True)
    gamma = sd[p + ".weight"].to(y.dtype).clone().requires_grad_(True)
    beta = sd[p + ".bias"].to(y.dtype).clone().requires_grad_(True)
    out = F.batch_norm(y, sd[p + ".running_mean"].to(y.dtype), sd[p + ".running_var"].to(y.dtype), gamma, beta,
                       training=False, eps=EPS)
    return torch.autograd.grad(out, (y, gamma, beta), grad_outputs=dz.to(y.dtype))


def running_update(rm: Tensor, rv: Tensor, y: Tensor) -> Tuple[Tensor, Tensor]:
    """nn.BatchNorm2d's running update from (rm, rv) with the batch statistics of y (unbiased variance), in float64"""
    y = y.double()
    n = y.numel() // y.shape[1]
    mean = y.mean(dim=(0, 2, 3))
    var = y.var(dim=(0, 2, 3), unbiased=False) * (n / max(n - 1, 1))
    return (1 - MOMENTUM) * rm.double() + MOMENTUM * mean, (1 - MOMENTUM) * rv.double() + MOMENTUM * var


def conv3(x: Tensor, sd: Dict[str, Tensor], name: str) -> Tensor:
    return F.conv2d(x, sd[name + ".weight"].to(x.dtype), sd[name + ".bias"].to(x.dtype), padding=1)


def conv3_dgrad(x: Tensor, sd: Dict[str, Tensor], name: str, dy: Tensor) -> Tensor:
    return torch.nn.grad.conv2d_input(x.shape, sd[name + ".weight"].to(dy.dtype), dy, padding=1)


# ------------------------------------------------------------------------------------------------ bf16-storage eval model
def _r(x: Tensor) -> Tensor:
    return x.to(torch.bfloat16).to(x.dtype)


def eval_forward_bf16_storage(sd: Dict[str, Tensor], x: Tensor) -> Tensor:
    """The folded eval forward with bf16 rounding where the engine stores: bf16 input, bf16 weights, higher-precision
    accumulation, BatchNorm as scale / shift (the shift absorbs the conv bias) in the conv epilogue, every activation
    stored in bf16, the output conv's result kept.  Computed in x's dtype.  Calibrates the end-to-end bound of the deep
    eval forward: what bf16 storage alone costs against the exact oracle."""
    dt = x.dtype

    def conv(t, name, pad, bias=True):
        return F.conv2d(t, _r(sd[name + ".weight"].to(dt)), sd[name + ".bias"].to(dt) if bias else None, padding=pad)

    def fold(p, conv_name):
        sc = sd[p + ".weight"].to(dt) * torch.rsqrt(sd[p + ".running_var"].to(dt) + EPS)
        sh = sd[p + ".bias"].to(dt) + (sd[conv_name + ".bias"].to(dt) - sd[p + ".running_mean"].to(dt)) * sc
        return sc[None, :, None, None], sh[None, :, None, None]

    out1 = _r(F.leaky_relu(conv(_r(x), "conv1", 4), 0.2))
    out = out1
    for b in range(num_blocks(sd)):
        p = f"residual_blocks.{b}"
        sc, sh = fold(p + ".bn1", p + ".conv1")
        z1 = _r(F.relu(conv(out, p + ".conv1", 1, bias=False) * sc + sh))
        sc, sh = fold(p + ".bn2", p + ".conv2")
        out = _r(conv(z1, p + ".conv2", 1, bias=False) * sc + sh + out)
    out = _r(conv(out, "conv2", 1) + out1)
    for j in O.upsample_stage_indices(sd):
        out = _r(F.relu(F.pixel_shuffle(conv(out, f"upsample.{j}", 1), 2)))
    return conv(out, "conv3", 4)
