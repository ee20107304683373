"""GPU tests of the spatially tiled eval forward (SRResNet.tile_budget_bytes, srg_generator_forward_tiles): bitwise equality
with the whole-frame eval forward, and with a pure-Python reference (crop window -> srg_generator_forward -> paste crop)
that does not rely on the kernels' position invariance."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def S():
    import srgan_b200
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return srgan_b200


@pytest.fixture
def variant(S, request):
    old = S.lib().srg_set_conv_variant(request.param)
    yield request.param
    S.lib().srg_set_conv_variant(old)


def _generator(S, seed=3, **kw):
    torch.manual_seed(seed)
    g = S.SRResNet(**kw).cuda()
    g.train()                                  # non-trivial running statistics, as a trained generator has
    gen = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for _ in range(2):
            g(torch.rand(2, 3, 24, 32, generator=gen).cuda())
    return g.eval()


def _whole(g, x):
    g.tile_budget_bytes = None
    g.stream_budget_bytes = None
    with torch.no_grad():
        return g(x).clone()


def _tiled(g, x, budget):
    g.tile_budget_bytes = budget
    try:
        with torch.no_grad():
            out = g(x).clone()
        key = ("tiles",) + tuple(x.shape[:1]) + tuple(x.shape[2:]) + (budget,)
        return out, g._rt[key]
    finally:
        g.tile_budget_bytes = None


def _ws(g, h, w):
    return g._eval_ws_bytes(h, w, torch.device("cuda"))


def _python_reference(S, g, x, win_h, win_w, tiles):
    """crop each window into its own tensor, run the ordinary whole-frame forward on it, paste its crop"""
    s = g.num_upsample_stages
    out = torch.full((x.shape[0], 3, x.shape[2] << s, x.shape[3] << s), float("nan"), device=x.device)
    g.tile_budget_bytes = None
    with torch.no_grad():
        for (f, y0, x0, cy, cx, ch, cw) in tiles:
            y = g(x[f:f + 1, :, y0:y0 + win_h, x0:x0 + win_w].contiguous())
            out[f, :, (y0 + cy) << s:(y0 + cy + ch) << s, (x0 + cx) << s:(x0 + cx + cw) << s] = \
                y[0, :, cy << s:(cy + ch) << s, cx << s:(cx + cw) << s]
    return out


CASES = [
    # (constructor kwargs, x shape, (h, w) of the one-window workspace the tile budget is set to)
    pytest.param({}, (1, 3, 203, 317), (120, 160), id="2d-grid"),
    pytest.param({}, (1, 3, 203, 317), (203, 180), id="strips"),
    pytest.param({}, (3, 3, 96, 700), (96, 300), id="strips-3-frames"),
    pytest.param({"upscale_factor": 2}, (2, 3, 203, 317), (110, 150), id="x2"),
    pytest.param({"num_residuals": 2}, (2, 3, 203, 317), (110, 150), id="2-blocks"),
]


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
@pytest.mark.parametrize("kw,shape,win", CASES)
def test_tiled_equals_whole_frame(S, variant, kw, shape, win):
    g = _generator(S, **kw)
    x = torch.rand(*shape, device="cuda")
    full = _whole(g, x)
    out, (win_h, win_w, per_call, tiles) = _tiled(g, x, _ws(g, *win))
    assert win_h < shape[2] or win_w < shape[3]
    if win[0] < shape[2]:
        assert win_h < shape[2] and win_w < shape[3]        # a 2-D grid of windows
    else:
        assert win_h == shape[2] and win_w < shape[3]       # full-height strips
    assert torch.equal(out, full)
    ref = _python_reference(S, g, x, win_h, win_w, tiles)
    assert torch.equal(out, ref)


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
def test_several_windows_of_different_frames_per_call(S, variant):
    """Engine with N = 4 windows; 3 frames x 3 windows = 9 windows in calls of 4, 4, 1: calls mix frames and the last is
    ragged.  Output equals the whole-frame forward and the Python crop reference bitwise."""
    from srgan_b200 import tiling as T
    g = _generator(S)
    x = torch.rand(3, 3, 96, 301, device="cuda")
    full = _whole(g, x)
    halo = T.tile_halo(g.num_residuals, g.num_upsample_stages)
    win_w = 180
    cols = T.axis_tiles(301, win_w, halo, 1)
    assert len(cols) == 3
    tiles = [(f, 0, x0, 0, cx, 96, cw) for f in range(3) for (x0, cx, cw) in cols]
    eng = g._engine(4, 96, win_w, False, x.device, False)
    eng.bind(g._rt["flat"], None, g._rt["flat_buf"])
    S.check(S.lib().srg_generator_pack(eng.handle, S._lib.stream_ptr()))
    out = torch.full_like(full, float("nan"))
    for i in range(0, len(tiles), 4):
        T.forward_tiles(eng.handle, x, tiles[i:i + 4], out, S._lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(out, full)
    assert torch.equal(out, _python_reference(S, g, x, 96, win_w, tiles))


def test_1080p_frame_at_2gb_stays_within_budget(S):
    torch.manual_seed(9)
    g = S.SRResNet().cuda().eval()                 # fresh module: no engine yet
    x = torch.rand(1, 3, 1080, 1920, device="cuda")
    budget = 2 << 30
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    g.tile_budget_bytes = budget
    with torch.no_grad():
        out = g(x)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - before
    assert rise <= budget + out.numel() * 4 + (64 << 20), rise
    assert g.last_engine().H < 1080 or g.last_engine().W < 1920
    assert torch.equal(out, _whole(g, x))


def test_forward_tiles_captures_into_a_cuda_graph(S):
    from srgan_b200 import tiling as T
    g = _generator(S)
    x = torch.rand(2, 3, 203, 317, device="cuda")
    _, (win_h, win_w, _, tiles) = _tiled(g, x, _ws(g, 120, 160))
    eng = g._engine(3, win_h, win_w, False, x.device, False)
    eng.bind(g._rt["flat"], None, g._rt["flat_buf"])
    S.check(S.lib().srg_generator_pack(eng.handle, S._lib.stream_ptr()))
    call = [tiles[0], tiles[len(tiles) // 2 + 1], tiles[-1]]          # windows of both frames
    eager = torch.zeros(2, 3, 203 * 4, 317 * 4, device="cuda")
    T.forward_tiles(eng.handle, x, call, eager, S._lib.stream_ptr())
    replay = torch.zeros_like(eager)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        T.forward_tiles(eng.handle, x, call, replay, S._lib.stream_ptr())     # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    replay.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        T.forward_tiles(eng.handle, x, call, replay, S._lib.stream_ptr())
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(replay, eager)
    assert eager.abs().sum() > 0


def test_no_budget_leaves_engines_and_outputs_unchanged(S):
    """tile_budget_bytes None (the default), and a tile budget every frame fits: the batch is streamed in chunks of frames
    through the same engine as without the tiling feature, with the same output bits."""
    g = _generator(S)
    x = torch.rand(6, 3, 40, 24, device="cuda")
    full = _whole(g, x)
    g.stream_budget_bytes = int(_ws(g, 40, 24) * 2.6)          # chunks of 2 frames: 2 + 2 + 2
    try:
        with torch.no_grad():
            assert g.tile_budget_bytes is None
            a = g(x).clone()
            n_default = g.last_engine().N
            assert n_default == g._stream_chunk(6, 40, 24, x.device) == 2
            g.tile_budget_bytes = _ws(g, 40, 24)                # every frame fits: the frame streaming path as before
            b = g(x).clone()
            assert g.last_engine().N == n_default
            assert g.last_engine().H == 40 and g.last_engine().W == 24
    finally:
        g.tile_budget_bytes = None
        g.stream_budget_bytes = 6 << 30
    assert torch.equal(a, full) and torch.equal(b, full)
