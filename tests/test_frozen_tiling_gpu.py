"""GPU tests of eval-mode autograd within a memory budget (SRResNet.grad_budget_bytes): bitwise equality with a Python
reference built from the existing entry points (crop each window -> srg_generator_forward_frozen -> srg_generator_backward_ex
on a crop-masked d(SR) -> add each window's input gradient over its window, in order), agreement with the whole-frame
frozen path and the float64 oracle, the memory bound at 1080p, and the autograd semantics of the path (input-only
backward, gradient hook, live graphs, in-place changes, a module used twice).  Every module carries the trained-like
BatchNorm state of tests/bn_affine_state.py."""
import copy
import os
import sys
from ctypes import c_void_p

import pytest
import torch

from oracle import srgan_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bn_affine_state as B  # noqa: E402  (tests/bn_affine_state.py)

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda")


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


def _state(seed, **kw):
    return B.bn_affine_state(O.init_srresnet_state(seed, **kw), seed)


def _module(S, seed=3, **kw):
    g = S.SRResNet(**kw)
    g.load_state_dict(_state(seed, **kw))
    return g.cuda().eval()


def _ws(g, h, w, n=1):
    return g._train_ws_bytes(n, h, w, DEV)


def _inputs(g, shape, seed=5):
    gen = torch.Generator().manual_seed(seed)
    s = g.num_upsample_stages
    x = torch.rand(*shape, generator=gen)
    dsr = torch.randn(shape[0], 3, shape[2] << s, shape[3] << s, generator=gen) * 1e-3
    return x.cuda(), dsr.cuda()


def _run(g, x, dsr, budget):
    """one eval-mode forward + backward with x.requires_grad under `budget`: (SR, x.grad, {name: .grad})"""
    g.grad_budget_bytes = budget
    try:
        xx = x.clone().requires_grad_()
        y = g(xx)
        y.backward(dsr)
        torch.cuda.synchronize()
        grads = {k: (p.grad.clone() if p.grad is not None else None) for k, p in g.named_parameters()}
        for p in g.parameters():
            p.grad = None
        return y.detach().clone(), xx.grad.clone(), grads
    finally:
        g.grad_budget_bytes = None


def _plan(g, x, budget):
    g.grad_budget_bytes = budget
    try:
        return g._frozen_tiles_plan(x.shape[0], x.shape[2], x.shape[3], DEV)
    finally:
        g.grad_budget_bytes = None


def _reference(S, g, x, dsr, plan):
    """existing entry points only, each call through an engine of as many windows as the call has"""
    win_h, win_w, n, tiles = plan
    s = g.num_upsample_stages
    L, rt = S.lib(), g._rt
    st = S._lib.stream_ptr()
    sr = torch.zeros(x.shape[0], 3, x.shape[2] << s, x.shape[3] << s, device=DEV)
    dlr = torch.zeros_like(x)
    total = None
    for i in range(0, len(tiles), n):
        call = tiles[i:i + n]
        m = len(call)
        gbuf = torch.empty_like(rt["flat"])
        eng = g._engine(m, win_h, win_w, False, DEV, False, frozen=True)
        eng.bind(rt["flat"], gbuf, rt["flat_buf"])
        S.check(L.srg_generator_set_grads(eng.handle, c_void_p(gbuf.data_ptr())))
        S.check(L.srg_generator_pack(eng.handle, st))
        xs = torch.stack([x[f, :, y0:y0 + win_h, x0:x0 + win_w] for (f, y0, x0, *_) in call]).contiguous()
        ys = torch.empty(m, 3, win_h << s, win_w << s, device=DEV)
        S.check(L.srg_generator_forward_frozen(eng.handle, c_void_p(xs.data_ptr()), c_void_p(ys.data_ptr()), st))
        ds = torch.zeros_like(ys)
        for j, (f, y0, x0, cy, cx, ch, cw) in enumerate(call):
            hs, ws_ = slice((y0 + cy) << s, (y0 + cy + ch) << s), slice((x0 + cx) << s, (x0 + cx + cw) << s)
            hw, ww = slice(cy << s, (cy + ch) << s), slice(cx << s, (cx + cw) << s)
            sr[f, :, hs, ws_] = ys[j, :, hw, ww]
            ds[j, :, hw, ww] = dsr[f, :, hs, ws_]
        gl = torch.empty_like(xs)
        S.check(L.srg_generator_backward_ex(eng.handle, c_void_p(ds.data_ptr()), 1, c_void_p(gl.data_ptr()), st))
        for j, (f, y0, x0, *_) in enumerate(call):
            dlr[f, :, y0:y0 + win_h, x0:x0 + win_w] += gl[j]
        total = gbuf.clone() if total is None else total + gbuf
    torch.cuda.synchronize()
    grads = {name: total[off:off + k].view(shape) for (name, off, k, shape) in g._ptable}
    return sr, dlr, grads


def _assert_same(a, b):
    assert torch.equal(a[0], b[0]), "SR"
    assert torch.equal(a[1], b[1]), "x.grad"
    bad = [k for k in b[2] if not torch.equal(a[2][k], b[2][k])]
    assert not bad, bad


def cos_ratio(a, b):
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return float(torch.dot(a, b) / (a.norm() * b.norm())), float(a.norm() / b.norm())


def _close(a, b, what, cos_min=0.99, lo=0.98, hi=1.02):
    """x.grad and every parameter gradient within (cos, ratio) bounds; returns the worst cos and ratio seen"""
    bad, worst = [], (1.0, 1.0)
    for name, u, v in [("x", a[1], b[1])] + [(k, a[2][k], b[2][k]) for k in b[2]]:
        c, r = cos_ratio(u, v)
        worst = (min(worst[0], c), r if abs(r - 1) > abs(worst[1] - 1) else worst[1])
        if not (c > cos_min and lo < r < hi):
            bad.append((name, c, r))
    assert not bad, (what, bad)
    print(f"\n{what}: worst cos {worst[0]:.6f}, worst ratio {worst[1]:.6f}")
    return worst


# ------------------------------------------------------------------------------------------------ bitwise vs reference
CASES = [
    # (constructor kwargs, x shape, budget = the frozen workspace of this many windows of this size)
    pytest.param({}, (1, 3, 203, 317), (1, 120, 160), id="2d-grid"),
    pytest.param({}, (1, 3, 203, 317), (1, 203, 180), id="strips"),
    pytest.param({}, (3, 3, 64, 150), (2.2, 64, 150), id="3-frames-ragged"),
    pytest.param({"upscale_factor": 2}, (2, 3, 203, 317), (1, 110, 150), id="x2"),
    pytest.param({"num_residuals": 2}, (2, 3, 203, 317), (1, 110, 150), id="2-blocks"),
]


def _budget(g, spec):
    k, h, w = spec
    return int(k * _ws(g, h, w))


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
@pytest.mark.parametrize("kw,shape,spec", CASES)
def test_budgeted_equals_python_reference(S, variant, kw, shape, spec):
    g = _module(S, **kw)
    x, dsr = _inputs(g, shape)
    budget = _budget(g, spec)
    assert _ws(g, shape[2], shape[3], shape[0]) > budget                  # the budgeted path applies
    plan = _plan(g, x, budget)
    win_h, win_w, n, tiles = plan
    if spec[1] < shape[2]:
        assert win_h < shape[2] and win_w < shape[3]                        # a 2-D grid of windows
    elif spec[2] < shape[3]:
        assert win_h == shape[2] and win_w < shape[3]                       # full-height strips
    else:
        assert (win_h, win_w) == shape[2:] and n == 2 and len(tiles) == 3   # whole frames, calls of 2 + 1
    got = _run(g, x, dsr, budget)
    assert g.last_engine().N == n and _ws(g, win_h, win_w, n) <= budget
    _assert_same(got, _reference(S, g, x, dsr, plan))


@pytest.mark.parametrize("variant", [0, 1], indirect=True)
def test_overlapping_windows_of_two_frames_in_one_call(S, variant):
    """one ABI call: two overlapping windows of frame 0 (their crops do not overlap) and one window of frame 1; d(lr) adds
    the overlap in window order, the parameter gradient sums all three"""
    from srgan_b200 import tiling as T
    g = _module(S, 7, num_residuals=2, upscale_factor=2)
    g._flatten(DEV)
    x, dsr = _inputs(g, (2, 3, 48, 90), seed=8)
    call = [(0, 0, 0, 0, 0, 48, 40), (0, 0, 24, 2, 16, 40, 34), (1, 0, 30, 0, 0, 48, 60)]
    eng = g._frozen_tiles_engine(3, 48, 60, DEV)
    st = S._lib.stream_ptr()
    sr = torch.zeros(2, 3, 96, 180, device=DEV)
    dlr = torch.zeros_like(x)
    T.forward_frozen_tiles(eng.handle, x, call, sr, st)
    T.backward_tiles(eng.handle, dsr, True, dlr, st)
    torch.cuda.synchronize()
    grads = {name: eng.grad_flat[off:off + k].view(shape).clone() for (name, off, k, shape) in g._ptable}
    ref = _reference(S, g, x, dsr, (48, 60, 3, call))
    _assert_same((sr, dlr, grads), ref)


def test_argument_checks_that_need_a_bound_workspace(S):
    from srgan_b200 import tiling as T
    g = _module(S, 9, num_residuals=2, upscale_factor=2)
    g._flatten(DEV)
    x, dsr = _inputs(g, (1, 3, 32, 40))
    st = S._lib.stream_ptr()
    ev = g._engine(1, 32, 40, False, DEV, False)
    ev.bind(g._rt["flat"], None, g._rt["flat_buf"])
    with pytest.raises(RuntimeError, match="needs a training-sized workspace"):
        T.forward_frozen_tiles(ev.handle, x, [(0, 0, 0, 0, 0, 32, 40)], None, st)
    eng = g._frozen_tiles_engine(1, 32, 40, DEV)
    S.check(S.lib().srg_generator_forward_frozen(eng.handle, c_void_p(x.data_ptr()),
                                                 c_void_p(torch.empty(1, 3, 64, 80, device=DEV).data_ptr()), st))
    with pytest.raises(RuntimeError, match="no preceding srg_generator_forward_frozen_tiles"):
        T.backward_tiles(eng.handle, dsr, True, None, st)
    T.forward_frozen_tiles(eng.handle, x, [(0, 0, 0, 0, 0, 32, 40)], None, st)
    with pytest.raises(RuntimeError, match="its backward is srg_generator_backward_tiles"):
        S.check(S.lib().srg_generator_backward_ex(eng.handle, c_void_p(dsr.data_ptr()), 1, None, st))
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ default unchanged
def test_no_budget_or_a_budget_that_fits_changes_nothing(S):
    base = _module(S, 11, num_residuals=2, upscale_factor=2)
    x, dsr = _inputs(base, (2, 3, 40, 56))
    runs = []
    for budget in ("unset", None, _ws(base, 40, 56, 2)):
        g = copy.deepcopy(base)
        if budget != "unset":
            g.grad_budget_bytes = budget
        n0 = g.launch_count()
        xx = x.clone().requires_grad_()
        y = g(xx)
        y.backward(dsr)
        torch.cuda.synchronize()
        runs.append((y.detach(), xx.grad, {k: p.grad for k, p in g.named_parameters()}, g.launch_count() - n0))
    for r in runs[1:]:
        _assert_same(r, runs[0])
        assert r[3] == runs[0][3]


# ------------------------------------------------------------------------------------------------ vs the whole frame
WHOLE = [
    pytest.param({}, (1, 3, 203, 317), (1, 120, 160), id="2d-grid"),
    pytest.param({"upscale_factor": 2}, (2, 3, 203, 317), (1, 110, 150), id="x2"),
    pytest.param({"num_residuals": 2}, (2, 3, 203, 317), (1, 110, 150), id="2-blocks"),
]


@pytest.mark.parametrize("kw,shape,spec", WHOLE)
def test_budgeted_matches_whole_frame_frozen_path(S, kw, shape, spec):
    """d(SR) is the gradient of a pixel loss toward an HR target.  Worst case measured on an NVIDIA B200 (1000 W):
    cos 0.9967 / ratio 0.9990 (2d-grid), 0.9974 / 0.9996 (x2), 0.99992 / 1.00005 (2-blocks).  With a zero-mean random
    d(SR) instead, every gradient is a heavily cancelling sum and the bf16 rounding of the window-border gradients, which
    the whole frame rounds once and the windows once each, moved the 2d-grid case (10 windows of a 203 x 317 frame) to
    cos 0.9929 and ratios 0.977 .. 1.046, outside these bounds."""
    g = _module(S, 13, **kw)
    x, _ = _inputs(g, shape, seed=14)
    s = g.num_upsample_stages
    hr = torch.rand(shape[0], 3, shape[2] << s, shape[3] << s, generator=torch.Generator().manual_seed(15)).cuda()
    with torch.no_grad():
        dsr = (g(x) - hr) * 1e-3
    tiled = _run(g, x, dsr, _budget(g, spec))
    whole = _run(g, x, dsr, None)
    rel = float((tiled[0] - whole[0]).abs().max() / whole[0].abs().max())
    assert rel < 2e-2, rel

    def psnr(a):
        return float(10 * torch.log10(1.0 / torch.mean((a - hr) ** 2)))
    assert abs(psnr(tiled[0]) - psnr(whole[0])) < 0.05
    _close(tiled, whole, f"budgeted vs whole frame {kw} {shape}")


def test_budgeted_matches_oracle_eval_autograd(S):
    """the bounds of test_frozen_gradients_end_to_end_match_oracle_eval_autograd, on a 2-D grid of windows"""
    kw = dict(num_residuals=2, upscale_factor=2)
    sd = _state(17, **kw)
    g = S.SRResNet(**kw)
    g.load_state_dict(sd)
    g = g.cuda().eval()
    x, dsr = _inputs(g, (1, 3, 60, 64), seed=18)
    budget = _ws(g, 40, 40)
    win_h, win_w, _, tiles = _plan(g, x, budget)
    assert win_h < 60 and win_w < 64
    got = _run(g, x, dsr, budget)
    work = O._with_grad(sd)
    xr = x.cpu().clone().requires_grad_()
    yr = O.srresnet_forward(work, xr, training=False)
    keys = O.trainable_keys(work)
    ref = torch.autograd.grad(yr, [xr] + [work[k] for k in keys], grad_outputs=dsr.cpu())
    _close(got, (None, ref[0], dict(zip(keys, ref[1:]))), "budgeted vs fp32 oracle", 0.95, 0.9, 1.1)


# ------------------------------------------------------------------------------------------------ memory at 1080p
def test_1080p_at_12gib_stays_within_budget_and_matches_whole_frame(S):
    g = _module(S, 19)
    x, dsr = _inputs(g, (1, 3, 1080, 1920), seed=20)
    budget = 12 << 30
    g.grad_budget_bytes = budget
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    xx = x.clone().requires_grad_()
    y = g(xx)
    y.backward(dsr)
    torch.cuda.synchronize()
    rise = torch.cuda.max_memory_allocated() - before
    g.grad_budget_bytes = None
    flat = g._rt["flat"].numel() * 4
    # x, SR, d(lr) and two flat gradient buffers (d(SR) was allocated before `before`, so it is not part of the rise)
    bound = budget + x.numel() * 4 + y.numel() * 4 + dsr.numel() * 4 + x.numel() * 4 + 2 * flat + (64 << 20)
    print(f"\n1080p at 12 GiB: peak rise {rise / 2**30:.3f} GiB, bound {bound / 2**30:.3f} GiB")
    assert rise <= bound, (rise, bound)
    assert g.last_engine().H < 1080 or g.last_engine().W < 1920
    tiled = (y.detach(), xx.grad, {k: p.grad for k, p in g.named_parameters()})
    for p in g.parameters():
        p.grad = None
    whole = _run(g, x, dsr, None)                      # 42.3 GB of frozen workspace
    _close(tiled, whole, "1080p at 12 GiB vs whole frame")


# ------------------------------------------------------------------------------------------------ autograd semantics
def _small(S, seed=21):
    g = _module(S, seed, num_residuals=2, upscale_factor=2)
    x, dsr = _inputs(g, (2, 3, 60, 64), seed=seed + 1)
    return g, x, dsr, _ws(g, 40, 40)


def test_input_only_backward(S):
    g, x, dsr, budget = _small(S)
    full = _run(g, x, dsr, budget)
    calls = []
    g.set_grad_hook(lambda m, flat: calls.append(1))
    g.requires_grad_(False)
    only = _run(g, x, dsr, budget)
    assert torch.equal(only[1], full[1])
    assert all(v is None for v in only[2].values())
    assert not calls


def test_gradient_hook_called_once_with_the_sum(S):
    g, x, dsr, budget = _small(S, 23)
    seen = []
    g.set_grad_hook(lambda m, flat: seen.append(flat.clone()))
    g.grad_budget_bytes = budget
    xx = x.clone().requires_grad_()
    g(xx).backward(dsr)
    torch.cuda.synchronize()
    g.grad_budget_bytes = None
    assert len(seen) == 1
    for (name, off, k, shape), p in zip(g._ptable, g._rt["plist"]):
        assert torch.equal(seen[0][off:off + k].view(shape), p.grad), name


def test_two_live_graphs_backward_in_reverse_order(S):
    g, x1, d1, budget = _small(S, 25)
    x2, d2 = _inputs(g, (2, 3, 60, 64), seed=27)
    a = _run(g, x1, d1, budget)
    b = _run(g, x2, d2, budget)
    g.grad_budget_bytes = budget
    xx1, xx2 = x1.clone().requires_grad_(), x2.clone().requires_grad_()
    y1, y2 = g(xx1), g(xx2)
    y2.backward(d2)
    y1.backward(d1)
    torch.cuda.synchronize()
    g.grad_budget_bytes = None
    assert torch.equal(y1, a[0]) and torch.equal(y2, b[0])
    assert torch.equal(xx1.grad, a[1]) and torch.equal(xx2.grad, b[1])
    for k, p in g.named_parameters():
        assert torch.equal(p.grad, b[2][k] + a[2][k]), k


@pytest.mark.parametrize("what", ["parameter", "running_var"])
def test_in_place_change_between_forward_and_backward_raises(S, what):
    g, x, dsr, budget = _small(S, 29)
    g.grad_budget_bytes = budget
    y = g(x.clone().requires_grad_())
    with torch.no_grad():
        if what == "parameter":
            g.residual_blocks[1].conv2.weight.mul_(1.0)
        else:
            g.residual_blocks[0].bn1.running_var.mul_(1.0)
    with pytest.raises(RuntimeError, match="modified in place"):
        y.backward(dsr)
    g.grad_budget_bytes = None


def test_module_used_twice_in_one_graph(S):
    g, x, dsr, budget = _small(S, 31)
    x = x[:1]
    hr = torch.rand(1, 3, 240, 256, generator=torch.Generator().manual_seed(32)).cuda()

    def chain(b):
        g.grad_budget_bytes = b
        try:
            xx = x.clone().requires_grad_()
            y = g(g(xx))
            torch.nn.functional.mse_loss(y, hr).backward()
            torch.cuda.synchronize()
            grads = {k: p.grad.clone() for k, p in g.named_parameters()}
            for p in g.parameters():
                p.grad = None
            return y.detach(), xx.grad, grads
        finally:
            g.grad_budget_bytes = None

    tiled, plain = chain(budget), chain(None)
    rel = float((tiled[0] - plain[0]).abs().max() / plain[0].abs().max())
    assert rel < 2e-2, rel
    _close(tiled, plain, "G(G(x)) budgeted vs whole frame")


def test_deterministic_and_buffers_unchanged(S):
    g, x, dsr, budget = _small(S, 33)
    bufs = {k: v.clone() for k, v in g.state_dict().items() if "running" in k or "num_batches" in k}
    a = _run(g, x, dsr, budget)
    b = _run(g, x, dsr, budget)
    _assert_same(a, b)
    for k, v in g.state_dict().items():
        if k in bufs:
            assert torch.equal(v, bufs[k]), k
