"""Float64 per-stage reference of the discriminator (src/models.py:90-120).  TEST INFRASTRUCTURE ONLY.

Stage l of D is: strided conv (8x8 / s2 / p2 for l = 0, 4x4 / s2 / p1 after), MaxPool2d(3, 2), InstanceNorm2d (no
affine, biased variance, eps 1e-5), then LeakyReLU(0.2), or Sigmoid for l = 3.  The functions here evaluate one stage,
forward or backward, in float64 on whatever device their inputs live on.  A caller that judges the CUDA engine feeds
them the operands the kernels read (bf16-rounded activations and weights, the fp32 bias, the engine's own fp32 conv
output for the pool / InstanceNorm backward), so that the only difference left is kernel arithmetic.

The helpers at the end translate between NCHW and the engine's operand layouts (space-to-depth ``x1..x3`` and the
stage-0 unfold ``x0``, csrc/discriminator.cu) so that engine tensors can be read back as the maps they stand for.
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
EPS = 1e-5
SLOPE = 0.2
KEYS = ("model.0", "model.4", "model.8", "model.12")
CHANNELS = (3, 64, 128, 256, 512)


def pad_of(l: int) -> int:
    return 2 if l == 0 else 1


def bf16(t: Tensor) -> Tensor:
    """The value a kernel reads from a bf16 operand (round to nearest even), as float64."""
    return t.to(torch.bfloat16).double()


def stage_params(sd: Dict[str, Tensor], l: int, device=None) -> Tuple[Tensor, Tensor]:
    """Stage l's conv weight as the engine's packed bf16 GEMM operand and its fp32 bias, both as float64."""
    w, b = sd[KEYS[l] + ".weight"], sd[KEYS[l] + ".bias"]
    return bf16(w.to(device)), b.to(device).double()


def conv(z: Tensor, w: Tensor, b: Optional[Tensor], l: int) -> Tensor:
    return F.conv2d(z, w, b, stride=2, padding=pad_of(l))


def instance_norm(p: Tensor) -> Tensor:
    """Two-pass InstanceNorm over each (sample, channel) map: (p - mean) / sqrt(biased var + eps)."""
    mean = p.mean(dim=(2, 3), keepdim=True)
    var = (p - mean).square().mean(dim=(2, 3), keepdim=True)
    return (p - mean) / torch.sqrt(var + EPS)


def activation(xhat: Tensor, l: int, positive: Optional[Tensor] = None) -> Tensor:
    """LeakyReLU(0.2) for l < 3, Sigmoid for l = 3.  ``positive`` (bool, xhat's shape) overrides which LeakyReLU
    branch each element takes; it only matters where xhat is within rounding of 0."""
    if l == 3:
        return torch.sigmoid(xhat)
    if positive is None:
        positive = xhat > 0
    return torch.where(positive, xhat, SLOPE * xhat)


def stage_forward(z: Tensor, w: Tensor, b: Tensor, l: int) -> Dict[str, Tensor]:
    """conv output y, pooled p and the stage's output (the next stage's input, or D's output for l = 3)."""
    y = conv(z, w, b, l)
    p = F.max_pool2d(y, 3, 2)
    return dict(y=y, p=p, out=activation(instance_norm(p), l))


def post_forward(y: Tensor, l: int, positive: Optional[Tensor] = None) -> Tensor:
    """MaxPool, InstanceNorm and activation of a given conv output y."""
    return activation(instance_norm(F.max_pool2d(y, 3, 2)), l, positive)


def post_backward(y: Tensor, dout: Tensor, l: int, positive: Optional[Tensor] = None) -> Tensor:
    """d(conv output) from d(stage output): the MaxPool + InstanceNorm + activation backward evaluated at y.  MaxPool
    routes each window's gradient to its first maximum in scan order, the rule the engine's kernels follow, so fed the
    engine's own y both sides route identically."""
    yv = y.detach().double().requires_grad_(True)
    out = post_forward(yv, l, positive)
    (dy,) = torch.autograd.grad(out, yv, dout.double())
    return dy


def conv_backward(z: Tensor, w: Tensor, dy: Tensor, l: int, need_input: bool = True):
    """(dz, dw, db) of stage l's conv for the upstream gradient dy.  dz is None when not needed."""
    zv = z.detach().double().requires_grad_(need_input)
    wv = w.detach().double().requires_grad_(True)
    bv = torch.zeros(w.shape[0], dtype=torch.float64, device=w.device, requires_grad=True)
    outs = [wv, bv] + ([zv] if need_input else [])
    g = torch.autograd.grad(conv(zv, wv, bv, l), outs, dy.double())
    return (g[2] if need_input else None), g[0], g[1]


def forward(sd: Dict[str, Tensor], x: Tensor) -> Tuple[Tensor, list]:
    """The four stages composed: D(x) and the list of stage records (no rounding of operands here)."""
    recs, z = [], x
    for l in range(4):
        r = stage_forward(z, sd[KEYS[l] + ".weight"], sd[KEYS[l] + ".bias"], l)
        r["z"] = z
        recs.append(r)
        z = r["out"]
    return z, recs


def backward(sd: Dict[str, Tensor], recs: list, dout: Tensor) -> Tuple[Tensor, Dict[str, Tensor]]:
    """The stage backwards composed from the records of ``forward``: d(input) and every parameter gradient."""
    grads, dz = {}, dout
    for l in range(3, -1, -1):
        r = recs[l]
        dy = post_backward(r["y"], dz, l)
        dz, grads[KEYS[l] + ".weight"], grads[KEYS[l] + ".bias"] = conv_backward(r["z"], sd[KEYS[l] + ".weight"], dy, l)
    return dz, grads


# ---------------------------------------------------------------------------------------------- engine layouts
def uns2d(xs: Tensor, Hp: int, Wp: int) -> Tuple[Tensor, Tensor]:
    """Engine space-to-depth operand XS[n][h'][w'][(a, b, c)] = z[2h'+a-1][2w'+b-1][c] -> (z as NCHW, the cells
    outside z as an NCHW map over the padded grid, which a forward operand must hold as zeros)."""
    n, Hs, Ws, C4 = xs.shape
    C = C4 // 4
    full = xs.view(n, Hs, Ws, 2, 2, C).permute(0, 5, 1, 3, 2, 4).reshape(n, C, 2 * Hs, 2 * Ws)
    assert 2 * Hs >= Hp + 1 and 2 * Ws >= Wp + 1
    inside = torch.zeros(2 * Hs, 2 * Ws, dtype=torch.bool, device=xs.device)
    inside[1:1 + Hp, 1:1 + Wp] = True
    return full[:, :, 1:1 + Hp, 1:1 + Wp], full[:, :, ~inside]


def s2d(z: Tensor, Hs: int, Ws: int) -> Tensor:
    """Inverse of ``uns2d``: NCHW z -> XS with zero padding cells."""
    n, C, Hp, Wp = z.shape
    full = torch.zeros(n, C, 2 * Hs, 2 * Ws, dtype=z.dtype, device=z.device)
    full[:, :, 1:1 + Hp, 1:1 + Wp] = z
    return full.view(n, C, Hs, 2, Ws, 2).permute(0, 2, 4, 3, 5, 1).reshape(n, Hs, Ws, 4 * C)


def unfold0(x: Tensor, Hs: int, Ws: int) -> Tensor:
    """Stage-0 operand U0[n][h'][w'][ch], ch = ((v*2+a)*2+b)*3+c  <-  x[n][c][2h'+a-2][2(w'+v)+b-2] (zero outside the
    image and for ch >= 48), in x's dtype."""
    n, C, H, W = x.shape
    xp = torch.zeros(n, C, 2 * Hs, 2 * (Ws + 3), dtype=x.dtype, device=x.device)
    h, w = min(H, 2 * Hs - 2), min(W, 2 * (Ws + 3) - 2)
    xp[:, :, 2:2 + h, 2:2 + w] = x[:, :, :h, :w]
    t = xp.view(n, C, Hs, 2, Ws + 3, 2)                                  # [n][c][h'][a][j][b]
    u = torch.stack([t[:, :, :, :, v:v + Ws, :] for v in range(4)])      # [v][n][c][h'][a][w'][b]
    u = u.permute(1, 3, 5, 0, 4, 6, 2).reshape(n, Hs, Ws, 48)
    return torch.cat([u, torch.zeros(n, Hs, Ws, 16, dtype=x.dtype, device=x.device)], dim=3)
