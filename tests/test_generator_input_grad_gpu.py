"""GPU tests of input gradients through SRResNet: conv1's data gradient, the input-only backward, eval-mode autograd with
running BatchNorm statistics ("frozen" BatchNorm) and two chained generators, against torch autograd of the fp32 CPU
oracle (oracle/srgan_oracle.py).  "maxrel" and "cos / ratio" are the measures tests/test_generator_gpu.py uses."""
import copy

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TOL_LAYER = 1e-2       # per layer, same inputs
TOL_WGRAD = 5e-3       # fp32 outputs computed from identical bf16 inputs


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def cos_ratio(got, ref):
    got, ref = got.double().cpu().flatten(), ref.double().cpu().flatten()
    return float(torch.dot(got, ref) / (got.norm() * ref.norm())), float(got.norm() / ref.norm())


def nchw(t):  # engine NHWC bf16 -> NCHW fp32 on the CPU
    return t.float().permute(0, 3, 1, 2).contiguous().cpu()


@pytest.fixture(scope="module")
def S():
    import srgan_b200
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return srgan_b200


@pytest.fixture(scope="module")
def O():
    from oracle import srgan_oracle
    return srgan_oracle


def _seeded(S, seed, **kw):
    torch.manual_seed(seed)
    return S.SRResNet(**kw)


def _warm_running_stats(g, shape, steps=3):
    """give the BatchNorm layers non-trivial running statistics, as a trained generator has (train-mode forwards)"""
    g.train()
    gen = torch.Generator().manual_seed(123)
    with torch.no_grad():
        for _ in range(steps):
            g(torch.rand(*shape, generator=gen).cuda())
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ 1. conv1 data gradient
@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("shape,res", [((2, 3, 16, 24), 16), ((16, 3, 96, 96), 16), ((1, 3, 13, 130), 2),
                                       ((2, 3, 9, 250), 2), ((3, 3, 21, 123), 2)])
def test_conv1_data_gradient_per_layer(S, variant, shape, res):
    """lr.grad against autograd of F.conv2d(lr, W1, b1, padding=4) fed the engine's own d(pre-LeakyReLU): the fold9 path
    (conv9_rows, variant 0) and the generic strip kernel (variant 1), ragged extents included (W > 120 and not a multiple
    of 120, H and W not multiples of 8)."""
    L = S.lib()
    g = _seeded(S, 3, num_residuals=res).cuda()
    g.debug_keep_grads = True
    g.train()
    gen = torch.Generator().manual_seed(4)
    lr = torch.rand(*shape, generator=gen).cuda().requires_grad_()
    old = L.srg_set_conv_variant(variant)
    try:
        y = g(lr)
        y.backward(torch.randn(y.shape, generator=gen).cuda() * 1e-3)
        torch.cuda.synchronize()
    finally:
        L.srg_set_conv_variant(old)
    dpre = nchw(g.last_engine().named_tensor("d_pre_conv1")).double()
    x = lr.detach().cpu().double().requires_grad_()
    ref = torch.autograd.grad(F.conv2d(x, g.conv1.weight.detach().cpu().double(), g.conv1.bias.detach().cpu().double(),
                                       padding=4), x, grad_outputs=dpre)[0]
    assert lr.grad is not None and lr.grad.shape == lr.shape
    assert maxrel(lr.grad, ref) < TOL_LAYER, (shape, variant, maxrel(lr.grad, ref))


# ------------------------------------------------------------------------------------------------ 2. no interference
@pytest.mark.parametrize("trunk_fused", [2, 0])
def test_input_gradient_does_not_change_the_training_step(S, trunk_fused):
    """Same weights and input in train mode, with and without x.requires_grad: output, every parameter gradient and the
    running statistics are bitwise equal; the engine launches exactly two more kernels (the filter pack, the conv)."""
    L = S.lib()
    old = L.srg_set_trunk_fused(trunk_fused)
    try:
        base = _seeded(S, 5)
        gs = [copy.deepcopy(base).cuda().train(), copy.deepcopy(base).cuda().train()]
        gen = torch.Generator().manual_seed(6)
        lr = torch.rand(2, 3, 16, 24, generator=gen).cuda()
        dsr = torch.randn(2, 3, 64, 96, generator=gen).cuda() * 1e-3
        outs = []
        for g, want_dx in zip(gs, (False, True)):
            x = lr.clone().requires_grad_(want_dx)
            y = g(x)
            y.backward(dsr)
            torch.cuda.synchronize()
            outs.append((y.detach().clone(), x.grad))
    finally:
        L.srg_set_trunk_fused(old)
    assert outs[0][1] is None and outs[1][1] is not None
    assert torch.equal(outs[0][0], outs[1][0])
    for (k, p0), p1 in zip(gs[0].named_parameters(), gs[1].parameters()):
        assert torch.equal(p0.grad, p1.grad), k
    for (k, b0), b1 in zip(gs[0].named_buffers(), gs[1].buffers()):
        assert torch.equal(b0, b1), k
    assert gs[1].launch_count() - gs[0].launch_count() == 2


# ------------------------------------------------------------------------------------------------ 3. input-only backward
@pytest.mark.parametrize("trunk_fused", [2, 0])
def test_input_only_backward(S, trunk_fused):
    """Every parameter frozen: x.grad is bitwise the x.grad of the full backward, no .grad appears, the gradient hook is
    not called and fewer kernels run (no weight gradients, bias sums or BatchNorm parameter gradients)."""
    L = S.lib()
    old = L.srg_set_trunk_fused(trunk_fused)
    try:
        base = _seeded(S, 7)
        full, only = copy.deepcopy(base).cuda().train(), copy.deepcopy(base).cuda().train()
        only.requires_grad_(False)
        calls = []
        only.set_grad_hook(lambda m, flat: calls.append(1))
        gen = torch.Generator().manual_seed(8)
        lr = torch.rand(2, 3, 16, 24, generator=gen).cuda()
        dsr = torch.randn(2, 3, 64, 96, generator=gen).cuda() * 1e-3
        xs = []
        for g in (full, only):
            x = lr.clone().requires_grad_()
            g(x).backward(dsr)
            torch.cuda.synchronize()
            xs.append(x.grad)
    finally:
        L.srg_set_trunk_fused(old)
    assert torch.equal(xs[0], xs[1])
    assert all(p.grad is None for p in only.parameters())
    assert only.flat_grads() is None
    assert calls == []
    assert only.launch_count() < full.launch_count()


# ------------------------------------------------------------------------------------------------ 4. end to end, train mode
def test_train_mode_input_gradient_matches_oracle(S, O):
    """x.grad of a default SRResNet in train mode against the oracle's autograd at the golden geometry, fed the same
    upstream gradient (the reconstruction loss's).  The input gradient is the deepest one: direction and scale."""
    g = _seeded(S, 1)
    sd = {k: v.clone() for k, v in g.state_dict().items()}
    gen = torch.Generator().manual_seed(2)
    lr = torch.rand(2, 3, 16, 24, generator=gen)
    hr = torch.rand(2, 3, 64, 96, generator=gen)
    g = g.cuda().train()
    x = lr.cuda().requires_grad_()
    sr = g(x)
    srd = sr.detach().clone().requires_grad_()
    com, tv = S.ReconstructionLoss()(hr.cuda(), srd)
    (com + tv).backward()
    sr.backward(srd.grad)
    torch.cuda.synchronize()
    xr = lr.clone().requires_grad_()
    yr = O.srresnet_forward(O._with_grad(sd), xr, training=True)
    ref = torch.autograd.grad(yr, xr, grad_outputs=srd.grad.cpu())[0]
    cos, ratio = cos_ratio(x.grad, ref)
    assert cos > 0.95 and 0.9 < ratio < 1.1, (cos, ratio)


# ------------------------------------------------------------------------------------------------ 5. frozen BatchNorm (eval)
@pytest.fixture(scope="module")
def frozen_run(S):
    """eval-mode forward + backward of a default SRResNet whose BatchNorm layers carry non-trivial running statistics,
    with every inter-layer gradient kept, plus the no_grad eval output of the same weights."""
    g = _seeded(S, 9).cuda()
    _warm_running_stats(g, (2, 3, 16, 24))
    g.debug_keep_grads = True
    g.eval()
    sd = {k: v.detach().cpu().clone() for k, v in g.state_dict().items()}
    gen = torch.Generator().manual_seed(10)
    lr = torch.rand(2, 3, 16, 24, generator=gen)
    hr = torch.rand(2, 3, 64, 96, generator=gen)
    dsr = torch.randn(2, 3, 64, 96, generator=gen) * 1e-3
    with torch.no_grad():
        y_nograd = g(lr.cuda()).cpu()
    y_detached = g(lr.cuda())                     # grad mode on, input does not require grad
    x = lr.cuda().requires_grad_()
    y = g(x)
    y.backward(dsr.cuda())
    torch.cuda.synchronize()
    eng = g.last_engine()
    T = {name: nchw(eng.named_tensor(name)) for name in eng.tensor_table()}
    grads = {k: p.grad.detach().cpu().clone() for k, p in g.named_parameters()}
    return dict(g=g, sd=sd, lr=lr, hr=hr, dsr=dsr, y_nograd=y_nograd, y_detached=y_detached, y=y, x=x, T=T, grads=grads,
                state_after={k: v.detach().cpu().clone() for k, v in g.state_dict().items()}, eng=eng)


def test_frozen_forward_uses_a_training_workspace_and_keeps_buffers(frozen_run):
    r = frozen_run
    assert r["eng"].frozen and r["eng"].training
    assert r["y"].requires_grad and r["x"].grad is not None
    for k, v in r["sd"].items():
        if not k.endswith((".weight", ".bias")):
            assert torch.equal(v, r["state_after"][k]), k          # running_mean / running_var / num_batches_tracked


def test_eval_without_input_grad_stays_detached(frozen_run):
    r = frozen_run
    assert not r["y_detached"].requires_grad
    assert torch.equal(r["y_detached"].cpu(), r["y_nograd"])


def test_frozen_output_matches_the_folded_eval_output(frozen_run, O):
    r = frozen_run
    y = r["y"].detach().cpu()
    assert maxrel(y, r["y_nograd"]) < 2e-2
    assert abs(O.psnr(y, r["hr"]) - O.psnr(r["y_nograd"], r["hr"])) < 0.05


def test_frozen_batchnorm_backward_per_layer(frozen_run):
    """Per block: d(y) = gamma * inv * d(z), dgamma, dbeta and the now non-zero trunk conv biases against
    F.batch_norm(training=False) / conv autograd, each layer fed the engine's own tensors."""
    r = frozen_run
    sd, T, G = r["sd"], r["T"], r["grads"]

    def bn_eval_bwd(y, p, dz):
        y = y.double().requires_grad_()
        gamma = sd[p + ".weight"].double().requires_grad_()
        beta = sd[p + ".bias"].double().requires_grad_()
        out = F.batch_norm(y, sd[p + ".running_mean"].double(), sd[p + ".running_var"].double(), gamma, beta,
                           training=False, eps=1e-5)
        return torch.autograd.grad(out, (y, gamma, beta), grad_outputs=dz.double())

    dout = T["d_last"]
    for b in range(15, -1, -1):
        p = f"residual_blocks.{b}"
        dy2, dg, db = bn_eval_bwd(T[f"rb{b}.y2"], p + ".bn2", dout)
        assert maxrel(T[f"rb{b}.d_y2"], dy2) < TOL_LAYER, p
        assert maxrel(G[p + ".bn2.weight"], dg) < TOL_WGRAD and maxrel(G[p + ".bn2.bias"], db) < TOL_WGRAD, p
        assert maxrel(G[p + ".conv2.bias"], dy2.sum((0, 2, 3))) < TOL_WGRAD, p
        assert float(G[p + ".conv2.bias"].abs().max()) > 0.0
        dy1, dg, db = bn_eval_bwd(T[f"rb{b}.y1"], p + ".bn1", T[f"rb{b}.d_pre1"])
        assert maxrel(T[f"rb{b}.d_y1"], dy1) < TOL_LAYER, p
        assert maxrel(G[p + ".bn1.weight"], dg) < TOL_WGRAD and maxrel(G[p + ".bn1.bias"], db) < TOL_WGRAD, p
        assert maxrel(G[p + ".conv1.bias"], dy1.sum((0, 2, 3))) < TOL_WGRAD, p
        dout = T[f"rb{b}.d_in"]


def test_frozen_gradients_end_to_end_match_oracle_eval_autograd(frozen_run, O):
    r = frozen_run
    work = O._with_grad(r["sd"])
    xr = r["lr"].clone().requires_grad_()
    yr = O.srresnet_forward(work, xr, training=False)
    keys = O.trainable_keys(work)
    ref = torch.autograd.grad(yr, [xr] + [work[k] for k in keys], grad_outputs=r["dsr"])
    bad = []
    for name, got, want in [("x", r["x"].grad, ref[0])] + [(k, r["grads"][k], v) for k, v in zip(keys, ref[1:])]:
        cos, ratio = cos_ratio(got, want)
        if not (cos > 0.95 and 0.9 < ratio < 1.1):
            bad.append((name, cos, ratio))
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ 6. composition
def test_two_chained_generators_match_oracle(S, O):
    """G2(G1(x)) in train mode under a pixel loss against an HR target (cascade training): G1's parameter gradients and
    x.grad against the oracle's chained autograd."""
    g1, g2 = _seeded(S, 11, num_residuals=2, upscale_factor=2), _seeded(S, 12, num_residuals=2, upscale_factor=2)
    sd1 = {k: v.clone() for k, v in g1.state_dict().items()}
    sd2 = {k: v.clone() for k, v in g2.state_dict().items()}
    gen = torch.Generator().manual_seed(13)
    lr = torch.rand(2, 3, 16, 24, generator=gen)
    hr = torch.rand(2, 3, 64, 96, generator=gen)
    g1, g2 = g1.cuda().train(), g2.cuda().train()
    x = lr.cuda().requires_grad_()
    y = g2(g1(x))
    F.mse_loss(y, hr.cuda()).backward()
    torch.cuda.synchronize()
    w1, w2 = O._with_grad(sd1), O._with_grad(sd2)
    xr = lr.clone().requires_grad_()
    yr = O.srresnet_forward(w2, O.srresnet_forward(w1, xr, training=True), training=True)
    assert maxrel(y.detach(), yr.detach()) < 4e-2
    keys = O.trainable_keys(w1)
    ref = torch.autograd.grad(F.mse_loss(yr, hr), [xr] + [w1[k] for k in keys])
    got = [x.grad] + [dict(g1.named_parameters())[k].grad for k in keys]
    bad = []
    for name, a, b in zip(["x"] + keys, got, ref):
        if name.startswith("residual_blocks.") and ".conv" in name and name.endswith(".bias"):
            assert float(a.abs().max()) == 0.0, name  # in front of a training-mode BatchNorm: mathematically zero
            continue
        cos, ratio = cos_ratio(a, b)
        if not (cos > 0.95 and 0.9 < ratio < 1.1):
            bad.append((name, cos, ratio))
    assert not bad, bad
