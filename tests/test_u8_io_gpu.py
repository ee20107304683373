"""GPU tests of the 8-bit frame I/O of the eval forward (SRResNet.upscale_u8, srg_generator_forward_u8,
srg_generator_forward_tiles_u8).  The contract is bitwise:

    G.upscale_u8(frames) == q(G(transformers.to_tensor(frames)))
    q(sr) = (sr.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()

for every routing (whole frames, frame streaming, spatial windows) under both conv3 kernel families."""
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


def _frames(*shape, seed=11):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(0, 256, shape, dtype=torch.uint8, device="cuda", generator=gen)


def _q(sr):
    return (sr.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()


def _contract(S, g, frames):
    with torch.no_grad():
        return _q(g(S.transformers.to_tensor(frames)))


def _ws(g, h, w):
    return g._eval_ws_bytes(h, w, torch.device("cuda"))


def _spread_output(g, x):
    """rescale conv3 so that the fp32 SR spans about [-1.5, 2.5]: both clamp bounds and the interior are exercised"""
    with torch.no_grad():
        d = g(x) - g.conv3.bias.detach().view(1, 3, 1, 1)       # conv3's output without its bias
        lo, hi = float(d.min()), float(d.max())
        a = 4.0 / (hi - lo)
        g.conv3.weight.mul_(a)
        g.conv3.bias.fill_(-1.5 - a * lo)


# ------------------------------------------------------------------------------------------------ whole frames
@pytest.mark.parametrize("variant", [0, 1], indirect=True)
@pytest.mark.parametrize("upscale", [2, 4])
@pytest.mark.parametrize("blocks", [2, 16])
def test_whole_frames(S, variant, upscale, blocks):
    g = _generator(S, upscale_factor=upscale, num_residuals=blocks)
    frames = _frames(2, 203, 317, 3)
    out = g.upscale_u8(frames)
    s = g.num_upsample_stages
    assert out.dtype == torch.uint8 and tuple(out.shape) == (2, 203 << s, 317 << s, 3)
    eng = g.last_engine()
    assert (eng.N, eng.H, eng.W) == (2, 203, 317)             # one call, no chunking at this size
    assert torch.equal(out, _contract(S, g, frames))


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
def test_streamed_in_chunks(S, variant):
    g = _generator(S)
    frames = _frames(5, 40, 24, 3)
    g.stream_budget_bytes = int(_ws(g, 40, 24) * 2.6)          # chunks of 2 frames: 2 + 2 + 1
    try:
        assert g._stream_chunk(5, 40, 24, frames.device) == 2
        out = g.upscale_u8(frames)
        assert g.last_engine().N == 1                           # the ragged last chunk
        assert (2, 40, 24, False) in g._rt["engines"]
        ref = _contract(S, g, frames)
    finally:
        g.stream_budget_bytes = 6 << 30
    assert torch.equal(out, ref)


# ------------------------------------------------------------------------------------------------ spatial windows
TILED = [
    # (x shape, (h, w) of the one-window workspace the tile budget is set to)
    pytest.param((1, 203, 317, 3), (120, 160), id="2d-grid"),
    pytest.param((2, 203, 317, 3), (203, 180), id="strips"),
]


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
@pytest.mark.parametrize("shape,win", TILED)
def test_tiled(S, variant, shape, win):
    g = _generator(S)
    frames = _frames(*shape)
    budget = _ws(g, *win)
    g.tile_budget_bytes = budget
    try:
        out = g.upscale_u8(frames)
        win_h, win_w, _, tiles = g._rt[("tiles", shape[0], shape[1], shape[2], budget)]
        eng = g.last_engine()
        assert (eng.H, eng.W) == (win_h, win_w)
        ref = _contract(S, g, frames)
    finally:
        g.tile_budget_bytes = None
    assert len(tiles) > shape[0]
    if win[0] < shape[1]:
        assert win_h < shape[1] and win_w < shape[2]            # a 2-D grid of windows
    else:
        assert win_h == shape[1] and win_w < shape[2]           # full-height strips
    assert torch.equal(out, ref)
    assert torch.equal(out, _contract(S, g, frames))            # and the whole-frame forward's


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
def test_windows_of_three_frames_per_call(S, variant):
    """Engine of N = 4 windows; 3 frames x 3 windows = 9 windows, interleaved so that each of the first two calls holds
    windows of all 3 frames; calls of 4, 4 and a ragged 1."""
    from srgan_b200 import tiling as T
    g = _generator(S)
    frames = _frames(3, 96, 301, 3)
    halo = T.tile_halo(g.num_residuals, g.num_upsample_stages)
    win_w = 180
    cols = T.axis_tiles(301, win_w, halo, 1)
    assert len(cols) == 3
    tiles = [(f, 0, x0, 0, cx, 96, cw) for (x0, cx, cw) in cols for f in range(3)]
    assert len({t[0] for t in tiles[0:4]}) == 3 and len({t[0] for t in tiles[4:8]}) == 3
    eng = g._engine(4, 96, win_w, False, frames.device, False)
    eng.bind(g._rt["flat"], None, g._rt["flat_buf"])
    S.check(S.lib().srg_generator_pack(eng.handle, S._lib.stream_ptr()))
    out = torch.zeros(3, 96 * 4, 301 * 4, 3, dtype=torch.uint8, device="cuda")
    for i in range(0, len(tiles), 4):
        T.forward_tiles_u8(eng.handle, frames, tiles[i:i + 4], out, S._lib.stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(out, _contract(S, g, frames))


# ------------------------------------------------------------------------------------------------ quantisation
@pytest.mark.parametrize("variant", [0, 1], indirect=True)
@pytest.mark.parametrize("tiled", [False, True], ids=["whole", "tiled"])
def test_both_clamp_bounds(S, variant, tiled):
    g = _generator(S, num_residuals=2)
    frames = _frames(2, 64, 203, 3)
    x = S.transformers.to_tensor(frames)
    _spread_output(g, x)
    with torch.no_grad():
        sr = g(x)
    assert float(sr.min()) < -1 and float(sr.max()) > 2
    inside = ((sr > 0) & (sr < 1)).float().mean()
    assert inside > 0.05                                         # the interior is exercised too
    if tiled:
        g.tile_budget_bytes = _ws(g, 64, 120)
    try:
        out = g.upscale_u8(frames)
        ref = _contract(S, g, frames)
    finally:
        g.tile_budget_bytes = None
    assert torch.equal(out, ref)
    assert bool((out == 0).any()) and bool((out == 255).any())


# ------------------------------------------------------------------------------------------------ CUDA graph
def test_forward_tiles_u8_captures_into_a_cuda_graph(S):
    from srgan_b200 import tiling as T
    g = _generator(S)
    frames = _frames(2, 203, 317, 3)
    halo = T.tile_halo(g.num_residuals, g.num_upsample_stages)
    win_h, win_w, _, tiles = T.plan_tiles(2, 203, 317, halo, lambda h, w: _ws(g, h, w), _ws(g, 120, 160))
    eng = g._engine(3, win_h, win_w, False, frames.device, False)
    eng.bind(g._rt["flat"], None, g._rt["flat_buf"])
    S.check(S.lib().srg_generator_pack(eng.handle, S._lib.stream_ptr()))
    call = [tiles[0], tiles[len(tiles) // 2 + 1], tiles[-1]]          # windows of both frames
    eager = torch.zeros(2, 203 * 4, 317 * 4, 3, dtype=torch.uint8, device="cuda")
    T.forward_tiles_u8(eng.handle, frames, call, eager, S._lib.stream_ptr())
    replay = torch.zeros_like(eager)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        T.forward_tiles_u8(eng.handle, frames, call, replay, S._lib.stream_ptr())     # warm-up on the capture stream
    torch.cuda.current_stream().wait_stream(side)
    replay.zero_()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        T.forward_tiles_u8(eng.handle, frames, call, replay, S._lib.stream_ptr())
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(replay, eager)
    assert int(eager.count_nonzero()) > 0


# ------------------------------------------------------------------------------------------------ forward unchanged
def test_forward_and_engines_unchanged_by_upscale_u8(S):
    g = _generator(S)
    frames = _frames(5, 40, 24, 3)
    x = S.transformers.to_tensor(frames)
    g.stream_budget_bytes = int(_ws(g, 40, 24) * 2.6)
    try:
        with torch.no_grad():
            a = g(x).clone()
            pools = {k: list(v) for k, v in g._rt["engines"].items()}
            u = g.upscale_u8(frames)
            after_u8 = {k: list(v) for k, v in g._rt["engines"].items()}
            b = g(x).clone()
    finally:
        g.stream_budget_bytes = 6 << 30
    assert after_u8.keys() == pools.keys()
    assert all(len(after_u8[k]) == len(pools[k]) and all(p is q for p, q in zip(after_u8[k], pools[k])) for k in pools)
    assert torch.equal(a, b)
    assert torch.equal(u, _q(a))
    assert not u.requires_grad and u.grad_fn is None


# ------------------------------------------------------------------------------------------------ memory at 8K
def test_8k_frame_at_4gib_stays_within_budget(S):
    torch.manual_seed(9)
    g = S.SRResNet().cuda().eval()                 # fresh module: no engine yet
    frames = _frames(1, 4320, 7680, 3, seed=5)
    budget = 4 << 30
    g.tile_budget_bytes = budget
    try:
        torch.cuda.synchronize()
        before = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        out = g.upscale_u8(frames)
        torch.cuda.synchronize()
        rise = torch.cuda.max_memory_allocated() - before
        assert rise < budget + frames.numel() + out.numel() + (64 << 20), rise
        assert g.last_engine().H < 4320 or g.last_engine().W < 7680
        with torch.no_grad():
            sr = g(S.transformers.to_tensor(frames))
    finally:
        g.tile_budget_bytes = None
    for r in range(0, sr.shape[2], 2160):                  # quantise in bands: no SR-sized temporaries
        assert torch.equal(out[:, r:r + 2160], _q(sr[:, :, r:r + 2160])), r
