"""CPU checks of eval-mode autograd within a memory budget (SRResNet.grad_budget_bytes, srg_generator_forward_frozen_tiles,
srg_generator_backward_tiles): the exported entry points and the argument checks that run before any CUDA call, the
workspace sizes the budgeted path must leave unchanged, the engine size it builds at 1080p, and the decomposition it
relies on (whole-frame gradients = sums of window-local gradients) on the float64 oracle."""
import ctypes
import os
import sys
from ctypes import byref, c_void_p

import pytest
import torch

import srgan_b200 as S
from srgan_b200 import tiling as T
from oracle import srgan_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bn_affine_state as B  # noqa: E402  (tests/bn_affine_state.py)

NEW = ("srg_generator_forward_frozen_tiles", "srg_generator_backward_tiles")


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
    for name in NEW:
        assert hasattr(so, name), name
        assert name in S._lib.EXPORTS, name


# ------------------------------------------------------------------------------------------------ argument checks
def _fwd(L, g, frames=b"x", F=1, H=40, W=48, tiles=None, n=1, sr=b"x"):
    if tiles is None:
        tiles = [(0, 0, 0, 0, 0, 16, 24)]
    arr = (T.SrgTile * max(len(tiles), 1))(*[T.SrgTile(*t) for t in tiles])
    fb = ctypes.create_string_buffer(16) if frames is not None else None
    sb = ctypes.create_string_buffer(16) if sr is not None else None
    return L.srg_generator_forward_frozen_tiles(g, fb, F, H, W, arr if tiles else None, n, sb, None)


def _bwd(L, g, dsr=b"x", param_grads=1, dlr=b"x"):
    db = ctypes.create_string_buffer(16) if dsr is not None else None
    lb = ctypes.create_string_buffer(16) if dlr is not None else None
    return L.srg_generator_backward_tiles(g, db, param_grads, lb, None)


def test_null_engine(L):
    assert _fwd(L, None) != 0
    assert "srg_generator_forward_frozen_tiles: null engine" in _err(L)
    assert _bwd(L, None) != 0
    assert "srg_generator_backward_tiles: null engine" in _err(L)


def test_null_pointers(L, engine):
    assert _fwd(L, engine, frames=None) != 0
    assert "null pointer" in _err(L)
    assert _fwd(L, engine, tiles=[]) != 0
    assert "null pointer" in _err(L)
    assert _fwd(L, engine, sr=None) != 0                  # no output is allowed (a recompute): the next check fails
    assert "no workspace bound" in _err(L)


@pytest.mark.parametrize("F,H,W", [(0, 40, 48), (1, 0, 48), (1, 40, 0)])
def test_frame_extents(L, engine, F, H, W):
    assert _fwd(L, engine, F=F, H=H, W=W) != 0
    assert "F, H and W must be >= 1" in _err(L)


@pytest.mark.parametrize("n", [0, 3])
def test_tile_count(L, engine, n):
    assert _fwd(L, engine, tiles=[(0, 0, 0, 0, 0, 16, 24)] * 3, n=n) != 0
    assert "tile count" in _err(L)


def test_tile_count_is_capped_at_srg_max_tiles(L):
    h = c_void_p()
    assert L.srg_generator_create(byref(h), 65, 16, 24, 2, 2) == 0
    try:
        assert _fwd(L, h, tiles=[(0, 0, 0, 0, 0, 16, 24)] * 65, n=65) != 0
        assert "tile count 65 outside 1..64" in _err(L)
    finally:
        L.srg_generator_destroy(h)


@pytest.mark.parametrize("frame", [-1, 2])
def test_frame_index(L, engine, frame):
    assert _fwd(L, engine, F=2, tiles=[(frame, 0, 0, 0, 0, 16, 24)]) != 0
    assert "frame index" in _err(L)


@pytest.mark.parametrize("y0,x0", [(-2, 0), (0, -1), (26, 0), (0, 25)])
def test_window_inside_frame(L, engine, y0, x0):
    assert _fwd(L, engine, tiles=[(0, y0, x0, 0, 0, 16, 24)]) != 0
    assert "is not inside the 40 x 48 frame" in _err(L)


@pytest.mark.parametrize("ch,cw", [(0, 24), (16, 0)])
def test_empty_crop(L, engine, ch, cw):
    assert _fwd(L, engine, tiles=[(0, 0, 0, 0, 0, ch, cw)]) != 0
    assert "crop is empty" in _err(L)


@pytest.mark.parametrize("crop", [(-1, 0, 16, 24), (0, -1, 16, 24), (1, 0, 16, 24), (0, 4, 16, 21)])
def test_crop_inside_window(L, engine, crop):
    assert _fwd(L, engine, tiles=[(0, 0, 0) + crop]) != 0
    assert "crop is not inside its window" in _err(L)


def test_unbound_engine(L, engine):
    assert _fwd(L, engine, tiles=[(0, 24, 24, 2, 3, 10, 20)]) != 0
    assert "srg_generator_forward_frozen_tiles: no workspace bound" in _err(L)


def test_backward_checks(L, engine):
    assert _bwd(L, engine, dsr=None) != 0
    assert "null d(sr)" in _err(L)
    assert _bwd(L, engine, param_grads=0, dlr=None) != 0
    assert "nothing to compute" in _err(L)
    assert _bwd(L, engine) != 0
    assert "srg_generator_backward_tiles: needs a training-sized bound workspace" in _err(L)
    assert _bwd(L, engine, param_grads=0) != 0                 # input gradient only: valid up to the workspace check
    assert "needs a training-sized bound workspace" in _err(L)


# ------------------------------------------------------------------------------------------------ workspace sizes
WORKSPACE = [
    # (N, H, W, n_res, n_up), eval bytes, train bytes: the sizes before the budgeted path existed
    ((16, 96, 96, 16, 2), 535043072, 3065029632),
    ((2, 16, 24, 16, 2), 9120768, 65868800),
    ((1, 1080, 1920, 16, 2), 7438422016, 42265253888),
    ((3, 21, 123, 2, 1), 13562880, 75320320),
    ((1, 64, 64, 16, 4), 190004224, 601588736),
    ((1, 40, 56, 2, 0), 3320832, 47325184),
]


@pytest.mark.parametrize("geom,eval_bytes,train_bytes", WORKSPACE)
def test_workspace_bytes_unchanged(L, geom, eval_bytes, train_bytes):
    h = c_void_p()
    assert L.srg_generator_create(byref(h), *geom) == 0
    try:
        assert L.srg_generator_workspace_bytes(h, 0) == eval_bytes
        assert L.srg_generator_workspace_bytes(h, 1) == train_bytes
    finally:
        L.srg_generator_destroy(h)


# ------------------------------------------------------------------------------------------------ the engine at 1080p
@pytest.mark.parametrize("F,gib", [(1, 4), (1, 8), (1, 12), (1, 24), (2, 48), (8, 48)])
def test_1080p_engine_fits_the_budget(F, gib):
    g = S.SRResNet()
    g.grad_budget_bytes = gib << 30
    dev = torch.device("cpu")                          # probe engines only: no device memory is touched
    assert g._train_ws_bytes(F, 1080, 1920, dev) > g.grad_budget_bytes          # the budgeted path applies
    win_h, win_w, n, tiles = g._frozen_tiles_plan(F, 1080, 1920, dev)
    assert 1 <= n <= len(tiles)
    assert g._train_ws_bytes(n, win_h, win_w, dev) <= g.grad_budget_bytes
    covered = sum(ch * cw for (_, _, _, _, _, ch, cw) in tiles)
    assert covered == F * 1080 * 1920


def test_plans_at_1080p_and_4k():
    g = S.SRResNet()
    dev = torch.device("cpu")

    def plan(F, H, W, gib):
        g.grad_budget_bytes = gib << 30
        win_h, win_w, n, tiles = g._frozen_tiles_plan(F, H, W, dev)
        return win_h, win_w, n, len(tiles)

    assert plan(1, 1080, 1920, 4) == (414, 448, 1, 15)
    assert plan(1, 1080, 1920, 12) == (580, 1000, 1, 4)
    assert plan(1, 1080, 1920, 24) == (1080, 1000, 1, 2)
    assert plan(8, 1080, 1920, 48) == (1080, 1920, 1, 8)          # whole frames, one per call
    assert plan(1, 2160, 3840, 12) == (602, 1020, 1, 16)


# ------------------------------------------------------------------------------------------------ decomposition (float64)
def _state(seed, n_res, n_up):
    sd = O.init_srresnet_state(seed, num_residuals=n_res, upscale_factor=1 << n_up)    # int(factor // 2) stages
    return B.to_double(B.bn_affine_state(sd, seed))


def _grads(sd, x, dsr):
    work = O._with_grad(sd)
    xr = x.clone().requires_grad_()
    y = O.srresnet_forward(work, xr, training=False)
    keys = O.trainable_keys(work)
    return torch.autograd.grad(y, [xr] + [work[k] for k in keys], grad_outputs=dsr)


def _window_sum(sd, x, dsr, n_up, win_h, win_w, tiles):
    """every window cropped into one batch (eval mode: items are independent), d(SR) inside its crop and zero elsewhere;
    window input gradients added into x.grad over the whole window, parameter gradients summed by autograd"""
    s = n_up
    xs = torch.stack([x[f, :, y0:y0 + win_h, x0:x0 + win_w] for (f, y0, x0, *_) in tiles])
    ds = torch.zeros(len(tiles), 3, win_h << s, win_w << s, dtype=x.dtype)
    for i, (f, y0, x0, cy, cx, ch, cw) in enumerate(tiles):
        ds[i, :, cy << s:(cy + ch) << s, cx << s:(cx + cw) << s] = \
            dsr[f, :, (y0 + cy) << s:(y0 + cy + ch) << s, (x0 + cx) << s:(x0 + cx + cw) << s]
    g = _grads(sd, xs, ds)
    dx = torch.zeros_like(x)
    for i, (f, y0, x0, *_) in enumerate(tiles):
        dx[f, :, y0:y0 + win_h, x0:x0 + win_w] += g[0][i]
    return (dx,) + tuple(g[1:])


def _worst(a, b) -> float:
    return max(float((u - v).abs().max() / v.abs().max()) for u, v in zip(a, b) if float(v.abs().max()) > 0)


CASES = [
    # (n_res, n_up), (F, H, W), window pixel budget of the planner (pixel count as the window cost)
    pytest.param((2, 1), (2, 44, 46), 30 * 30, id="2-blocks-x2"),
    pytest.param((2, 0), (1, 40, 46), 32 * 32, id="2-blocks-x1"),
    pytest.param((16, 2), (1, 84, 84), 82 * 82, id="16-blocks-x4"),
]


@pytest.mark.parametrize("cfg,shape,budget", CASES)
def test_window_gradients_sum_to_whole_frame_gradients(cfg, shape, budget):
    n_res, n_up = cfg
    sd = _state(31 + n_res + n_up, n_res, n_up)
    gen = torch.Generator().manual_seed(32)
    F, H, W = shape
    x = torch.rand(F, 3, H, W, generator=gen, dtype=torch.float64)
    dsr = torch.randn(F, 3, H << n_up, W << n_up, generator=gen, dtype=torch.float64)
    halo = T.tile_halo(n_res, n_up)
    win_h, win_w, _, tiles = T.plan_tiles(F, H, W, halo, lambda h, w: h * w, budget)
    assert win_h < H and win_w < W                                   # a 2-D grid of windows
    whole = _grads(sd, x, dsr)
    err = _worst(_window_sum(sd, x, dsr, n_up, win_h, win_w, tiles), whole)
    assert err < 1e-9, err
    if n_res == 16:
        return                                                       # the halo's sensitivity: the two cheap cases below
    # negative control: windows planned with halo - 1 leave a crop edge one pixel too close to its window border
    win_h, win_w, _, tiles = T.plan_tiles(F, H, W, halo - 1, lambda h, w: h * w, budget)
    err = _worst(_window_sum(sd, x, dsr, n_up, win_h, win_w, tiles), whole)
    assert err >= 1e-6, err
