"""Spatially tiled eval forward: window planning for frames whose whole-frame eval workspace exceeds a memory budget.

In eval mode BatchNorm is folded into the conv epilogues, so every layer of SRResNet is local and an output pixel depends
on the input pixels at most ``tile_halo(num_residuals, num_upsample_stages)`` LR pixels away (40 for the default 16
blocks and x4).  A frame is cut into equal-size windows whose crops partition it; each window is run through the
ordinary eval launch sequence (``srg_generator_forward_tiles``) and only its crop is written back.  Windows are
*shifted*, not clipped: the last window on an axis is moved inward so that it stays inside the frame.  Every window
border is then either a frame border, where the engine's zero padding is exactly what the whole-frame forward sees, or
lies at least ``halo`` pixels from the window's crop, so every cropped output pixel is computed from exactly the inputs
the whole-frame forward uses.

Window origins are aligned to even rows (``ROW_ALIGN``).  ``conv3_il_kernel`` (the 3x3 trunk and up-conv kernel) keeps
even and odd image rows of a tile in two accumulator blocks that receive the three row taps in different orders
(even: kh2, kh0, kh1; odd: kh1, kh0, kh2), so an output row's fp32 sum depends on the parity of its row inside the
launch.  With an even window origin every pixel keeps its whole-frame parity at LR (and at x2, x4 the origins are even
anyway), which makes the tiled output bit-identical.  Columns need no alignment.
"""
from __future__ import annotations

import ctypes
from typing import Callable, List, Optional, Tuple

from . import _lib

ROW_ALIGN = 2
MAX_TILES = 64          # SRG_MAX_TILES

Tile = Tuple[int, int, int, int, int, int, int]   # frame, y0, x0, crop_y0, crop_x0, crop_h, crop_w (LR pixels)


class SrgTile(ctypes.Structure):
    """srg_tile_t (include/srgan_b200.h)."""
    _fields_ = [(name, ctypes.c_int32) for name in ("frame", "y0", "x0", "crop_y0", "crop_x0", "crop_h", "crop_w")]


def tile_halo(num_residuals: int, num_upsample_stages: int) -> int:
    """Receptive radius of SRResNet in LR pixels.

    Take the HR pixels of LR pixel y = 0 at scale 2^s.  conv3 (9x9) reaches rows -4 .. 2^s + 3 of its input.  Each
    upsample stage, walked backwards, maps rows [lo, hi] at scale 2^(j+1) to [floor(lo / 2) - 1, floor(hi / 2) + 1] at
    scale 2^j: PixelShuffle halves the index, the stage's 3x3 conv adds one row on each side.  At LR the trunk adds one
    pixel per 3x3 conv (2 per residual block plus conv2) and conv1 (9x9) adds 4.  For (16, 2): -4 .. 7 at x4,
    -3 .. 4 at x2, -3 .. 3 at LR, then 33 + 4 more: 40.
    """
    if num_residuals < 0 or num_upsample_stages < 0:
        raise ValueError("num_residuals and num_upsample_stages must be >= 0")
    lo, hi = -4, (1 << num_upsample_stages) + 3
    for _ in range(num_upsample_stages):
        lo, hi = lo // 2 - 1, hi // 2 + 1
    return max(-lo, hi) + (2 * num_residuals + 1) + 4


# ---- one axis ---------------------------------------------------------------------------------------------------
def _axis_count(L: int, win: int, halo: int, align: int) -> Optional[int]:
    """Windows of size ``win`` that cover an axis of length L (None: no valid tiling with this size)."""
    if win >= L:
        return 1
    edge = win - halo                          # crop of the first / last window (one side is the frame border)
    mid = win - 2 * halo - (align - 1)         # crop of an inner window (origin rounded down by up to align - 1)
    if edge < 1 or (L - win) % align:
        return None
    rest = L - 2 * edge
    if rest <= 0:
        return 2
    if mid < 1:
        return None
    return 2 + -(-rest // mid)


def axis_tiles(L: int, win: int, halo: int, align: int) -> List[Tuple[int, int, int]]:
    """(window origin, crop start relative to the window, crop length) of every window along one axis."""
    if win >= L:
        return [(0, 0, L)]
    edge = win - halo
    mid = win - 2 * halo - (align - 1)
    bounds = [0, edge]
    while L - bounds[-1] > edge:
        bounds.append(bounds[-1] + mid)
    bounds.append(L)
    out = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        o = min(max(lo - halo, 0), L - win)
        o -= o % align
        out.append((o, lo - o, hi - lo))
    return out


def _min_window(L: int, halo: int, align: int) -> int:
    """Smallest window size with a valid tiling of the axis: 2 * halo + 1 (rounded up for the alignment), or L."""
    return _next_valid(L, 2 * halo + 1, halo, align)


def _next_valid(L: int, w: int, halo: int, align: int) -> int:
    while w < L and _axis_count(L, w, halo, align) is None:
        w += 1
    return min(w, L)


def _smallest_window_for(L: int, count: int, halo: int, align: int, lo: int) -> int:
    """Smallest valid window size >= lo (itself valid) that needs at most ``count`` windows.  Over valid sizes the count
    falls as the window grows; sizes that break the row alignment are skipped."""
    a, b = lo, L
    while a < b:
        m = (a + b) // 2
        v = _next_valid(L, m, halo, align)
        if _axis_count(L, v, halo, align) <= count:
            b = m
        else:
            a = m + 1
    return _next_valid(L, a, halo, align)


# ---- planner ----------------------------------------------------------------------------------------------------
def plan_tiles(F: int, H: int, W: int, halo: int, window_bytes_fn: Callable[[int, int], int],
               budget: int) -> Tuple[int, int, int, List[Tile]]:
    """Windows for F frames of H x W LR pixels such that ``tiles_per_call`` windows fit ``budget`` bytes.

    ``window_bytes_fn(h, w)`` is the eval workspace of a one-window engine of h x w (a probe engine's
    ``srg_generator_workspace_bytes``).  Returns ``(window_h, window_w, tiles_per_call, tiles)``: all windows have one
    size (window_h, window_w) <= (H, W) (an axis shorter than the window is not tiled), window origins are on even rows,
    the crops partition every frame, every crop edge that is not a frame edge lies at least ``halo`` pixels inside its
    window, ``tiles_per_call * window_bytes_fn(window_h, window_w) <= budget`` and ``tiles_per_call <= 64``.  Tiles are
    listed frame by frame, row by row.  Among the window sizes that fit, the one that computes the fewest window pixels per
    frame wins (at 1080p that is usually full-height strips: no vertical halo).  Raises RuntimeError if not even the
    smallest window (2 * halo + 1 on each tiled axis) fits.
    """
    if F < 1 or H < 1 or W < 1:
        raise ValueError("F, H and W must be >= 1")
    cache = {}

    def nbytes(h: int, w: int) -> int:
        if (h, w) not in cache:
            cache[(h, w)] = int(window_bytes_fn(h, w))
        return cache[(h, w)]

    min_h, min_w = _min_window(H, halo, ROW_ALIGN), _min_window(W, halo, 1)
    need = nbytes(min_h, min_w)
    if need > budget:
        raise RuntimeError(f"tile budget of {budget} bytes is too small: the smallest window ({min_h} x {min_w} LR pixels, "
                           f"2 * halo + 1 = {2 * halo + 1} with halo {halo}) needs {need} bytes of eval workspace")

    def widest_fit(h: int) -> int:
        """largest valid window width that fits the budget next to window height h (min_w fits: checked by caller)"""
        a, b = min_w, W
        while a < b:
            m = (a + b + 1) // 2
            if nbytes(h, m) <= budget:
                a = m
            else:
                b = m - 1
        while _axis_count(W, a, halo, 1) is None:
            a -= 1
        return a

    best = None                                   # (window pixels per frame, h, w)
    count_h = 1
    while True:
        h = _smallest_window_for(H, count_h, halo, ROW_ALIGN, min_h)
        n_h = _axis_count(H, h, halo, ROW_ALIGN)
        if best is not None and n_h * h * W >= best[0]:
            break                                 # even one full-width column of windows cannot beat the best
        if nbytes(h, min_w) <= budget:
            n_w = _axis_count(W, widest_fit(h), halo, 1)
            w = _smallest_window_for(W, n_w, halo, 1, min_w)
            cost = n_h * h * n_w * w
            if best is None or cost < best[0]:
                best = (cost, h, w)
        if h == min_h:
            break
        count_h = max(count_h, n_h) + 1
    _, win_h, win_w = best
    per_call = max(1, min(MAX_TILES, budget // nbytes(win_h, win_w)))
    rows, cols = axis_tiles(H, win_h, halo, ROW_ALIGN), axis_tiles(W, win_w, halo, 1)
    tiles = [(f, y0, x0, cy, cx, ch, cw) for f in range(F) for (y0, cy, ch) in rows for (x0, cx, cw) in cols]
    return win_h, win_w, per_call, tiles


def forward_tiles(handle, frames, tiles: List[Tile], out, stream) -> None:
    """One ``srg_generator_forward_tiles`` call: ``frames`` F x 3 x H x W and ``out`` F x 3 x (H << s) x (W << s) are
    contiguous fp32 CUDA tensors, ``handle`` an engine bound to an eval workspace whose N >= len(tiles)."""
    arr = (SrgTile * len(tiles))(*[SrgTile(*t) for t in tiles])
    F, _, H, W = frames.shape
    _lib.check(_lib.lib().srg_generator_forward_tiles(handle, ctypes.c_void_p(frames.data_ptr()), F, H, W, arr, len(tiles),
                                                      ctypes.c_void_p(out.data_ptr()), stream),
               "srg_generator_forward_tiles")


def forward_tiles_u8(handle, frames, tiles: List[Tile], out, stream) -> None:
    """One ``srg_generator_forward_tiles_u8`` call: as ``forward_tiles`` on uint8 frames F x H x W x 3 into a uint8
    ``out`` F x (H << s) x (W << s) x 3 (contiguous CUDA tensors), quantised as ``SRResNet.upscale_u8`` documents."""
    arr = (SrgTile * len(tiles))(*[SrgTile(*t) for t in tiles])
    F, H, W, _ = frames.shape
    _lib.check(_lib.lib().srg_generator_forward_tiles_u8(handle, ctypes.c_void_p(frames.data_ptr()), F, H, W, arr,
                                                         len(tiles), ctypes.c_void_p(out.data_ptr()), stream),
               "srg_generator_forward_tiles_u8")


def forward_frozen_tiles(handle, frames, tiles: List[Tile], out, stream) -> None:
    """One ``srg_generator_forward_frozen_tiles`` call: as ``forward_tiles`` on an engine bound to a training workspace,
    keeping the activations for ``backward_tiles``.  ``out`` may be None (a recompute for the backward: no output)."""
    arr = (SrgTile * len(tiles))(*[SrgTile(*t) for t in tiles])
    F, _, H, W = frames.shape
    _lib.check(_lib.lib().srg_generator_forward_frozen_tiles(
        handle, ctypes.c_void_p(frames.data_ptr()), F, H, W, arr, len(tiles),
        ctypes.c_void_p(out.data_ptr()) if out is not None else None, stream), "srg_generator_forward_frozen_tiles")


def backward_tiles(handle, dsr, param_grads: bool, dlr, stream) -> None:
    """One ``srg_generator_backward_tiles`` call for the windows of the last ``forward_frozen_tiles``: the bound flat
    gradient buffer receives their parameter gradients (``param_grads``), ``dlr`` (None: not computed) their input
    gradients, added in window order."""
    _lib.check(_lib.lib().srg_generator_backward_tiles(
        handle, ctypes.c_void_p(dsr.data_ptr()), 1 if param_grads else 0,
        ctypes.c_void_p(dlr.data_ptr()) if dlr is not None else None, stream), "srg_generator_backward_tiles")
