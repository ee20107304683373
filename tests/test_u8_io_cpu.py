"""CPU checks of the 8-bit frame I/O of the eval forward (SRResNet.upscale_u8, srg_generator_forward_u8,
srg_generator_forward_tiles_u8): the exported entry points, every argument check that runs before any CUDA call (each with
its own message), the Python-level errors, and the eval and training workspace sizes, which the 8-bit path leaves as they
were."""
import ctypes
from ctypes import byref, c_void_p

import pytest
import torch

import srgan_b200 as S
from srgan_b200 import tiling as T

NEW = ("srg_generator_forward_u8", "srg_generator_forward_tiles_u8")


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


def test_declarations():
    P, I = ctypes.c_void_p, ctypes.c_int
    assert S._lib.EXPORTS["srg_generator_forward_u8"] == (I, [P, P, P, P])
    assert S._lib.EXPORTS["srg_generator_forward_tiles_u8"] == (I, [P, P, I, I, I, P, I, P, P])
    assert hasattr(S.SRResNet, "upscale_u8")
    assert callable(T.forward_tiles_u8)


# ------------------------------------------------------------------------------------------------ argument checks
def _whole(L, g, lr=b"x", sr=b"x"):
    lb = ctypes.create_string_buffer(16) if lr is not None else None
    sb = ctypes.create_string_buffer(16) if sr is not None else None
    return L.srg_generator_forward_u8(g, lb, sb, None)


def _tiles(L, g, frames=b"x", F=1, H=40, W=48, tiles=None, n=1, sr=b"x"):
    if tiles is None:
        tiles = [(0, 0, 0, 0, 0, 16, 24)]
    arr = (T.SrgTile * max(len(tiles), 1))(*[T.SrgTile(*t) for t in tiles])
    fb = ctypes.create_string_buffer(16) if frames is not None else None
    sb = ctypes.create_string_buffer(16) if sr is not None else None
    return L.srg_generator_forward_tiles_u8(g, fb, F, H, W, arr if tiles else None, n, sb, None)


def test_null_engine(L):
    assert _whole(L, None) != 0
    assert _err(L) == "srg_generator_forward_u8: null engine"
    assert _tiles(L, None) != 0
    assert _err(L) == "srg_generator_forward_tiles_u8: null engine"


def test_whole_frame_checks(L, engine):
    assert _whole(L, engine, lr=None) != 0
    assert _err(L) == "srg_generator_forward_u8: null pointer (input frames)"
    assert _whole(L, engine, sr=None) != 0
    assert _err(L) == "srg_generator_forward_u8: null pointer (output)"
    assert _whole(L, engine) != 0                                     # every argument valid
    assert _err(L) == "srg_generator_forward_u8: no workspace bound"


def test_tiles_null_pointers(L, engine):
    assert _tiles(L, engine, frames=None) != 0
    assert _err(L) == "srg_generator_forward_tiles_u8: null pointer (frames)"
    assert _tiles(L, engine, tiles=[]) != 0
    assert _err(L) == "srg_generator_forward_tiles_u8: null pointer (tiles)"
    assert _tiles(L, engine, sr=None) != 0
    assert _err(L) == "srg_generator_forward_tiles_u8: null pointer (output)"


@pytest.mark.parametrize("F,H,W", [(0, 40, 48), (1, 0, 48), (1, 40, 0)])
def test_frame_extents(L, engine, F, H, W):
    assert _tiles(L, engine, F=F, H=H, W=W) != 0
    assert "srg_generator_forward_tiles_u8: F, H and W must be >= 1" in _err(L)


@pytest.mark.parametrize("n", [0, 3])
def test_tile_count(L, engine, n):
    assert _tiles(L, engine, tiles=[(0, 0, 0, 0, 0, 16, 24)] * 3, n=n) != 0
    assert f"srg_generator_forward_tiles_u8: tile count {n} outside 1..2" in _err(L)


def test_tile_count_is_capped_at_srg_max_tiles(L):
    h = c_void_p()
    assert L.srg_generator_create(byref(h), 65, 16, 24, 2, 2) == 0
    try:
        assert _tiles(L, h, tiles=[(0, 0, 0, 0, 0, 16, 24)] * 65, n=65) != 0
        assert "tile count 65 outside 1..64" in _err(L)
    finally:
        L.srg_generator_destroy(h)


@pytest.mark.parametrize("frame", [-1, 2])
def test_frame_index(L, engine, frame):
    assert _tiles(L, engine, F=2, tiles=[(frame, 0, 0, 0, 0, 16, 24)]) != 0
    assert f"tile 0 frame index {frame} outside 0..1" in _err(L)


@pytest.mark.parametrize("y0,x0", [(-2, 0), (0, -1), (26, 0), (0, 25)])
def test_window_inside_frame(L, engine, y0, x0):
    assert _tiles(L, engine, tiles=[(0, y0, x0, 0, 0, 16, 24)]) != 0     # frame 40 x 48, window 16 x 24
    assert "is not inside the 40 x 48 frame" in _err(L)


@pytest.mark.parametrize("ch,cw", [(0, 24), (16, 0)])
def test_empty_crop(L, engine, ch, cw):
    assert _tiles(L, engine, tiles=[(0, 0, 0, 0, 0, ch, cw)]) != 0
    assert "crop is empty" in _err(L)


@pytest.mark.parametrize("crop", [(-1, 0, 16, 24), (0, -1, 16, 24), (1, 0, 16, 24), (0, 4, 16, 21)])
def test_crop_inside_window(L, engine, crop):
    assert _tiles(L, engine, tiles=[(0, 0, 0) + crop]) != 0
    assert "srg_generator_forward_tiles_u8: tile 0 crop is not inside its window" in _err(L)


def test_second_tile_is_checked(L, engine):
    assert _tiles(L, engine, F=2, tiles=[(0, 0, 0, 0, 0, 16, 24), (1, 0, 0, 0, 0, 17, 24)], n=2) != 0
    assert "tile 1 crop is not inside its window" in _err(L)


def test_unbound_engine(L, engine):
    assert _tiles(L, engine, tiles=[(0, 24, 24, 2, 3, 10, 20)]) != 0    # every other argument valid
    assert _err(L) == "srg_generator_forward_tiles_u8: no workspace bound"


# ------------------------------------------------------------------------------------------------ Python-level errors
def test_train_mode_raises():
    g = S.SRResNet(num_residuals=1)
    assert g.training
    with pytest.raises(RuntimeError, match=r"call \.eval\(\)"):
        g.upscale_u8(torch.zeros(1, 8, 8, 3, dtype=torch.uint8))


@pytest.mark.parametrize("dtype", [torch.float32, torch.int32, torch.int8])
def test_dtype_raises(dtype):
    g = S.SRResNet(num_residuals=1).eval()
    with pytest.raises(RuntimeError, match="takes uint8 frames"):
        g.upscale_u8(torch.zeros(1, 8, 8, 3, dtype=dtype))


@pytest.mark.parametrize("shape", [(8, 8, 3), (1, 3, 8, 8), (1, 8, 8, 4), (1, 1, 8, 8, 3), (0, 8, 8, 3), (1, 0, 8, 3)])
def test_shape_raises(shape):
    g = S.SRResNet(num_residuals=1).eval()
    with pytest.raises(RuntimeError, match=r"expects an N x H x W x 3 batch"):
        g.upscale_u8(torch.zeros(*shape, dtype=torch.uint8))


def test_cpu_tensor_raises():
    g = S.SRResNet(num_residuals=1).eval()
    with pytest.raises(RuntimeError, match="takes a CUDA tensor"):
        g.upscale_u8(torch.zeros(1, 8, 8, 3, dtype=torch.uint8))


# ------------------------------------------------------------------------------------------------ workspace sizes
WORKSPACE = [
    # (N, H, W, n_res, n_up), eval bytes, train bytes: the sizes before the 8-bit path existed
    ((2, 203, 317, 16, 2), 467715072, 2680482816),
    ((2, 203, 317, 2, 2), 463553536, 1285417984),
    ((2, 203, 317, 16, 1), 203542528, 1954464768),
    ((8, 1080, 1920, 16, 2), 59462848512, 337702918144),
    ((1, 4320, 7680, 16, 2), 118916381696, 675304670208),
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
