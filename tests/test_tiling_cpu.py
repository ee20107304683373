"""CPU checks of the spatially tiled eval forward: the exported entry points and their argument checks (before any CUDA
call, so no device is needed), the receptive radius against the float64 oracle, and properties of the window planner."""
import ctypes
import random
from ctypes import byref, c_void_p

import numpy as np
import pytest
import torch

import srgan_b200 as S
from srgan_b200 import tiling as T


@pytest.fixture(scope="module")
def L():
    return S.lib()


@pytest.fixture
def engine(L):
    h = c_void_p()
    assert L.srg_generator_create(byref(h), 2, 16, 24, 2, 2) == 0     # N = 2 windows of 16 x 24; create() needs no device
    yield h
    L.srg_generator_destroy(h)


def _err(L) -> str:
    return L.srg_last_error().decode()


def test_library_exports_both_symbols():
    so = ctypes.CDLL(S._lib.SO_PATH)
    for name in ("srg_generator_tile_halo", "srg_generator_forward_tiles"):
        assert hasattr(so, name), name
        assert name in S._lib.EXPORTS, name


@pytest.mark.parametrize("n_res", [0, 1, 2, 16])
@pytest.mark.parametrize("n_up", [0, 1, 2, 4])
def test_library_halo_equals_python_halo(L, n_res, n_up):
    assert L.srg_generator_tile_halo(n_res, n_up) == T.tile_halo(n_res, n_up)


def test_halo_values():
    assert T.tile_halo(16, 2) == 40           # the derivation in tile_halo's docstring
    assert T.tile_halo(16, 1) == 3 + 33 + 4
    assert T.tile_halo(16, 4) == 3 + 33 + 4
    assert T.tile_halo(0, 2) == 3 + 1 + 4
    assert T.tile_halo(16, 0) == 4 + 33 + 4   # no upsample stage: conv3's own 4


def _call(L, g, frames=b"x", F=1, H=40, W=48, tiles=None, n=1, sr=b"x"):
    if tiles is None:
        tiles = [(0, 0, 0, 0, 0, 16, 24)]
    arr = (T.SrgTile * max(len(tiles), 1))(*[T.SrgTile(*t) for t in tiles])
    fb = ctypes.create_string_buffer(16) if frames is not None else None
    sb = ctypes.create_string_buffer(16) if sr is not None else None
    return L.srg_generator_forward_tiles(g, fb, F, H, W, arr if tiles else None, n, sb, None)


def test_null_engine(L):
    assert _call(L, None) != 0
    assert "null engine" in _err(L)


def test_null_pointers(L, engine):
    assert _call(L, engine, frames=None) != 0
    assert "null pointer" in _err(L)
    assert _call(L, engine, sr=None) != 0
    assert "null pointer" in _err(L)
    assert _call(L, engine, tiles=[]) != 0
    assert "null pointer" in _err(L)


@pytest.mark.parametrize("F,H,W", [(0, 40, 48), (1, 0, 48), (1, 40, 0)])
def test_frame_extents(L, engine, F, H, W):
    assert _call(L, engine, F=F, H=H, W=W) != 0
    assert "F, H and W must be >= 1" in _err(L)


@pytest.mark.parametrize("n", [0, 3])
def test_tile_count(L, engine, n):
    tiles = [(0, 0, 0, 0, 0, 16, 24)] * 3
    assert _call(L, engine, tiles=tiles, n=n) != 0
    assert "tile count" in _err(L)


def test_tile_count_is_capped_at_srg_max_tiles(L):
    h = c_void_p()
    assert L.srg_generator_create(byref(h), 65, 16, 24, 2, 2) == 0
    try:
        assert _call(L, h, tiles=[(0, 0, 0, 0, 0, 16, 24)] * 65, n=65) != 0
        assert "tile count 65 outside 1..64" in _err(L)
    finally:
        L.srg_generator_destroy(h)


@pytest.mark.parametrize("frame", [-1, 2])
def test_frame_index(L, engine, frame):
    assert _call(L, engine, F=2, tiles=[(frame, 0, 0, 0, 0, 16, 24)]) != 0
    assert "frame index" in _err(L)


@pytest.mark.parametrize("y0,x0", [(-2, 0), (0, -1), (26, 0), (0, 25)])
def test_window_inside_frame(L, engine, y0, x0):
    assert _call(L, engine, tiles=[(0, y0, x0, 0, 0, 16, 24)]) != 0     # frame 40 x 48, window 16 x 24
    assert "is not inside the 40 x 48 frame" in _err(L)


@pytest.mark.parametrize("ch,cw", [(0, 24), (16, 0)])
def test_empty_crop(L, engine, ch, cw):
    assert _call(L, engine, tiles=[(0, 0, 0, 0, 0, ch, cw)]) != 0
    assert "crop is empty" in _err(L)


@pytest.mark.parametrize("crop", [(-1, 0, 16, 24), (0, -1, 16, 24), (1, 0, 16, 24), (0, 4, 16, 21)])
def test_crop_inside_window(L, engine, crop):
    assert _call(L, engine, tiles=[(0, 0, 0) + crop]) != 0
    assert "crop is not inside its window" in _err(L)


def test_unbound_engine(L, engine):
    assert _call(L, engine, tiles=[(0, 24, 24, 2, 3, 10, 20)]) != 0    # every other argument valid
    assert "no workspace bound" in _err(L)


# ------------------------------------------------------------------------------------------------ halo vs the oracle
@pytest.mark.parametrize("n_res,n_up", [(16, 2), (2, 1), (0, 2)])
def test_halo_against_oracle(n_res, n_up):
    """Perturb one LR pixel in the middle of a small image (float64, eval mode): no HR pixel further than tile_halo LR
    pixels away changes, and the farthest change is at least tile_halo - 1 (a ReLU may hide the outermost ring)."""
    from oracle import srgan_oracle as O
    halo = T.tile_halo(n_res, n_up)
    sd = {k: (v.double() if v.is_floating_point() else v)
          for k, v in O.init_srresnet_state(3, num_residuals=n_res, upscale_factor=2 ** n_up if n_up > 1 else 2).items()}
    gen = torch.Generator().manual_seed(4)
    for k in sd:                              # non-trivial running statistics
        if k.endswith("running_mean"):
            sd[k] = torch.randn(sd[k].shape, generator=gen, dtype=torch.float64) * 0.1
        elif k.endswith("running_var"):
            sd[k] = torch.rand(sd[k].shape, generator=gen, dtype=torch.float64) + 0.5
    long_, short = 2 * halo + 11, 7
    for (H, W, axis) in ((long_, short, 0), (short, long_, 1)):
        x = torch.rand(1, 3, H, W, generator=gen, dtype=torch.float64)
        py, px = H // 2, W // 2
        x2 = x.clone()
        x2[0, :, py, px] += 1.0
        with torch.no_grad():
            d = (O.srresnet_forward(sd, x2, training=False) - O.srresnet_forward(sd, x, training=False)).abs()
        changed = d.sum(dim=(0, 1)) > 0                                 # [H << s, W << s]
        idx = torch.nonzero(changed)[:, axis] >> n_up
        dist = int((idx - (py if axis == 0 else px)).abs().max())
        assert halo - 1 <= dist <= halo, (axis, dist, halo)


# ------------------------------------------------------------------------------------------------ planner properties
def _bytes(h, w):
    return 6_000_000 + 3_600 * h * w + 128 * w        # the shape of the eval layout: fixed part + per-pixel buffers


def _check_plan(F, H, W, halo, budget):
    win_h, win_w, per_call, tiles = T.plan_tiles(F, H, W, halo, _bytes, budget)
    assert 1 <= win_h <= H and 1 <= win_w <= W
    assert 1 <= per_call <= 64 and per_call * _bytes(win_h, win_w) <= budget
    cover = np.zeros((F, H, W), dtype=np.int32)
    for (f, y0, x0, cy, cx, ch, cw) in tiles:
        assert 0 <= f < F
        assert 0 <= y0 and y0 + win_h <= H and 0 <= x0 and x0 + win_w <= W        # window inside the frame
        assert y0 % T.ROW_ALIGN == 0                                               # even window rows
        assert ch >= 1 and cw >= 1 and 0 <= cy and cy + ch <= win_h and 0 <= cx and cx + cw <= win_w
        if y0 + cy > 0:
            assert cy >= halo
        if y0 + cy + ch < H:
            assert win_h - (cy + ch) >= halo
        if x0 + cx > 0:
            assert cx >= halo
        if x0 + cx + cw < W:
            assert win_w - (cx + cw) >= halo
        cover[f, y0 + cy:y0 + cy + ch, x0 + cx:x0 + cx + cw] += 1
    assert (cover == 1).all()                                                       # the crops partition every frame
    if win_h == H:
        assert all(t[1] == 0 for t in tiles)
    if win_w == W:
        assert all(t[2] == 0 for t in tiles)
    return win_h, win_w, per_call, tiles


def test_planner_properties():
    rng = random.Random(7)
    for _ in range(300):
        halo = rng.choice([4, 8, 12, 40])
        F = rng.randint(1, 3)
        H, W = rng.randint(1, 420), rng.randint(1, 420)
        lo = _bytes(T._min_window(H, halo, T.ROW_ALIGN), T._min_window(W, halo, 1))
        budget = rng.randint(lo, max(lo, _bytes(H, W) * 2))
        _check_plan(F, H, W, halo, budget)


def test_planner_rows_stay_even_with_odd_frames():
    for H in (203, 205, 1081):
        for budget in (_bytes(100, 100), _bytes(150, 317), _bytes(90, 90)):
            _check_plan(2, H, 317, 40, budget)


def test_planner_prefers_full_height_strips_at_1080p():
    win_h, win_w, _, tiles = _check_plan(1, 1080, 1920, 40, 4 << 30)
    assert win_h == 1080 and len(tiles) == 2
    win_h, win_w, _, tiles = _check_plan(1, 1080, 1920, 40, 2 << 30)
    assert len(tiles) * win_h * win_w < 1.2 * 1080 * 1920


def test_planner_too_small_budget_names_the_minimum():
    need = _bytes(83, 81)                      # 2 * halo + 1 = 81; rows: the next size that keeps the row alignment
    with pytest.raises(RuntimeError, match=f"needs {need} bytes"):
        T.plan_tiles(1, 203, 317, 40, _bytes, need - 1)
    T.plan_tiles(1, 203, 317, 40, _bytes, need)
    small = _bytes(30, 50)                     # frames smaller than a minimum window: the whole frame is the minimum
    with pytest.raises(RuntimeError, match=f"needs {small} bytes"):
        T.plan_tiles(1, 30, 50, 40, _bytes, small - 1)
