"""GPU parity tests of the CUDA discriminator and the GAN-mode steps against the CPU oracle.

Per-layer bound (north_star): max relative error <= 1e-2 with every layer fed the SAME input on both sides.  The
reference network is numerically chaotic end to end (MaxPool argmax ties and InstanceNorm over as few as 3 elements
turn bf16 operand rounding into O(10 %) gradient differences, exactly as for an fp32-vs-bf16 run of the reference
itself), so end-to-end checks on D are on values / direction, the per-stage checks carry the bound.
"""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TOL = 1e-2
KEYS = ["model.0", "model.4", "model.8", "model.12"]
CH = [3, 64, 128, 256, 512]


def maxrel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).abs().max() / max(float(b.abs().max()), 1e-30))


def nchw(t):
    return t.float().permute(0, 3, 1, 2).contiguous().cpu()


def uns2d(xs, Hp, Wp, C):
    """engine operand layout XS[n][h'][w'][(a,b,c)] = z[2h'+a-1][2w'+b-1][c] -> z (NCHW); cells the next conv never
    reads are not materialised and come back 0."""
    n, Hs, Ws, _ = xs.shape
    xs = xs.float().cpu().view(n, Hs, Ws, 2, 2, C)
    z = torch.zeros(n, C, Hp, Wp)
    for a in range(2):
        for b in range(2):
            hs = [h for h in range(Hs) if 0 <= 2 * h + a - 1 < Hp]
            ws = [w for w in range(Ws) if 0 <= 2 * w + b - 1 < Wp]
            if hs and ws:
                blk = xs[:, hs[0]:hs[-1] + 1, ws[0]:ws[-1] + 1, a, b, :].permute(0, 3, 1, 2)
                z[:, :, 2 * hs[0] + a - 1:2 * hs[-1] + a:2, 2 * ws[0] + b - 1:2 * ws[-1] + b:2] = blk
    return z


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


@pytest.fixture(scope="module")
def run(S):
    torch.manual_seed(3)
    d = S.Discriminator()
    sd = {k: v.clone() for k, v in d.state_dict().items()}
    x = torch.rand(1, 3, 940, 940)                 # 940 -> final 3x3 map: the last InstanceNorm sees 9 elements
    d = d.cuda()
    xg = x.cuda().requires_grad_(True)
    out = d(xg)
    torch.manual_seed(5)
    dout = torch.randn(out.shape) * 1e-2
    out.backward(dout.cuda())
    torch.cuda.synchronize()
    eng = d.last_engine()
    T = {k: eng.named_tensor(k).detach().cpu() for k in eng.tensor_table()}
    zin = [x]
    for l in range(1, 4):
        hp, wp = T[f"p{l - 1}"].shape[1:3]
        zin.append(uns2d(T[f"x{l}"], hp, wp, CH[l]))
    grads = {k: p.grad.detach().cpu() for k, p in d.named_parameters()}
    return dict(sd=sd, x=x, out=out.detach().cpu(), dout=dout, T=T, zin=zin, grads=grads, dx=xg.grad.detach().cpu())


def test_forward_stages_isolated(run):
    sd, T, zin = run["sd"], run["T"], run["zin"]
    for l in range(4):
        y = F.conv2d(zin[l], sd[KEYS[l] + ".weight"], sd[KEYS[l] + ".bias"], stride=2, padding=2 if l == 0 else 1)
        assert maxrel(nchw(T[f"y{l}"]), y) < TOL, l                       # strided conv on tensor cores
        assert maxrel(nchw(T[f"p{l}"]), F.max_pool2d(nchw(T[f"y{l}"]), 3, 2)) == 0.0, l      # MaxPool2d(3,2): exact
        xh = F.instance_norm(nchw(T[f"p{l}"]), eps=1e-5)
        if l < 3:
            got = zin[l + 1]
            assert maxrel(got, F.leaky_relu(xh, 0.2) * (got != 0)) < TOL, l   # InstanceNorm + LeakyReLU (bf16 store)
        else:
            assert maxrel(run["out"], torch.sigmoid(xh)) < 1e-4           # InstanceNorm + Sigmoid (fp32)


def test_backward_stages_isolated(run):
    sd, T, zin, G = run["sd"], run["T"], run["zin"], run["grads"]
    dz = run["dout"]
    for l in range(3, -1, -1):
        # pool / InstanceNorm / activation backward from the engine's own fp32 conv output
        y = nchw(T[f"y{l}"]).clone().requires_grad_(True)
        xh = F.instance_norm(F.max_pool2d(y, 3, 2), eps=1e-5)
        z = F.leaky_relu(xh, 0.2) if l < 3 else torch.sigmoid(xh)
        if l < 3:
            z = z * (zin[l + 1] != 0).float()
        z.backward(dz)
        assert maxrel(nchw(T[f"dy{l}"]), y.grad) < TOL, l
        # conv weight / bias / data gradients from the engine's dY
        w = sd[KEYS[l] + ".weight"].clone().requires_grad_(True)
        b = sd[KEYS[l] + ".bias"].clone().requires_grad_(True)
        zi = zin[l].clone().requires_grad_(True)
        F.conv2d(zi, w, b, stride=2, padding=2 if l == 0 else 1).backward(nchw(T[f"dy{l}"]))
        assert maxrel(G[KEYS[l] + ".weight"], w.grad) < 5e-3, l
        assert maxrel(G[KEYS[l] + ".bias"], b.grad) < 5e-3, l
        if l > 0:
            hp, wp = T[f"p{l - 1}"].shape[1:3]
            dzi = uns2d(T[f"dx{l}"], hp, wp, CH[l])
            m = (zin[l] != 0).float()
            assert maxrel(dzi * m, zi.grad * m) < TOL, l
            dz = dzi
        else:
            assert maxrel(run["dx"], zi.grad) < TOL


def test_forward_end_to_end_and_size_rule(S, O, run):
    with torch.no_grad():
        ref = O.discriminator_forward(run["sd"], run["x"])
    assert run["out"].shape == ref.shape
    assert float((run["out"] - ref).abs().mean()) < 2e-2          # end to end; sigmoid map, values in (0, 1)
    d = S.Discriminator().cuda()
    for bad in ((384, 384), (512, 512), (256, 256), (427, 1024)):      # SURVEY Appendix E: the reference raises too
        with pytest.raises(RuntimeError):
            d(torch.rand(1, 3, *bad).cuda())
    assert d(torch.rand(1, 3, 512, 1024).cuda()).shape == (1, 512, 1, 3)
    assert d(torch.rand(2, 3, 684, 684).cuda()).shape == (2, 512, 2, 2)


def test_two_live_forwards_accumulate_like_autograd(S):
    """D(hr) and D(sr) as two separate calls (the reference's form, src/train.py:215-216) must give the same
    parameter gradients as one pass over the concatenated batch (what train_discriminator here does)."""
    torch.manual_seed(9)
    d = S.Discriminator().cuda()
    a, b = torch.rand(1, 3, 428, 700).cuda(), torch.rand(1, 3, 428, 700).cuda()
    loss = S.tanh_mean(d(b), d(a))
    loss.backward()
    g1 = {k: p.grad.clone() for k, p in d.named_parameters()}
    d.zero_grad()
    preds = d(torch.cat([a, b]))
    S.tanh_mean(preds[1:], preds[:1]).backward()
    for k, p in d.named_parameters():
        if k.endswith("weight"):
            assert maxrel(p.grad, g1[k]) < 1e-4, k


def test_tanh_mean_value_and_grads(S):
    torch.manual_seed(1)
    a0, b0 = torch.rand(2, 512, 1, 3), torch.rand(2, 512, 1, 3)
    a, b = a0.clone().cuda().requires_grad_(True), b0.clone().cuda().requires_grad_(True)
    (3.0 * S.tanh_mean(a, b)).backward()
    ar, br = a0.clone().requires_grad_(True), b0.clone().requires_grad_(True)
    ref = torch.mean(torch.tanh(ar - br))
    (3.0 * ref).backward()
    assert abs(float(S.tanh_mean(a, b).detach()) - float(ref.detach())) < 1e-6
    assert maxrel(a.grad, ar.grad) < 1e-5 and maxrel(b.grad, br.grad) < 1e-5


def test_train_discriminator_and_gan_mode_steps(S, O):
    """train_discriminator (src/train.py:206-230) and the GAN-mode generator step (src/train.py:184-192) against
    the oracle's versions.  Geometry LR 235x235 -> HR 940x940 (final D map 3x3): at the reference's native 512x1024
    the last InstanceNorm sees 3 elements and end-to-end gradients are dominated by rounding noise on BOTH sides."""
    torch.manual_seed(4)
    g = S.SRResNet(num_residuals=1)
    d = S.Discriminator()
    g_sd = {k: v.clone() for k, v in g.state_dict().items()}
    d_sd = {k: v.clone() for k, v in d.state_dict().items()}
    lr = torch.rand(1, 3, 235, 235)
    hr = torch.rand(1, 3, 940, 940)
    g, d = g.cuda(), d.cuda()
    d_opt = S.Adam(d.parameters(), lr=5e-5)
    g_opt = S.Adam(g.parameters(), lr=1e-4)
    crit = S.ReconstructionLoss()
    d_before = d.flat_parameters().clone()
    d_loss = S.train_discriminator(d, g, hr.cuda(), lr.cuda(), d_opt)
    ref_loss, ref_grads = O.discriminator_loss_and_grads(d_sd, g_sd, hr, lr)
    assert abs(d_loss - ref_loss) < 0.02                       # mean of tanh over a 512x3x3 map
    moved = (d.flat_parameters() - d_before).abs()
    assert float(moved.max()) <= 5e-5 * 1.001 and float(moved.max()) > 1e-5     # Adam's first step: |dp| <= lr
    # direction of the largest gradient tensor agrees with the oracle's
    gw = dict(d.named_parameters())["model.12.weight"].grad.double().flatten().cpu()
    rw = ref_grads["model.12.weight"].double().flatten()
    assert float(torch.dot(gw, rw) / (gw.norm() * rw.norm())) > 0.5
    losses = S.train_generator(g, d, lr.cuda(), hr.cuda(), None, crit, g_opt, gan_mode=True)
    ref, _, _ = O.generator_loss_and_grads(g_sd, lr, hr, d_sd=d_sd, gan_mode=True)
    assert abs(losses[1] - ref[1]) < 5e-3 * abs(ref[1])       # com_loss
    assert abs(losses[3]) <= 1.0 and abs(losses[0] - (losses[1] + losses[2] + losses[3])) < 1e-5
    assert all(p.grad is None or torch.isfinite(p.grad).all() for p in g.parameters())


def _cos(a, b):
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-300)), float(a.norm() / b.norm().clamp_min(1e-300))


def test_adversarial_steps_match_reference_fixtures(S, golden_dir):
    """train_discriminator (src/train.py:206-230) and the GAN-mode generator objective (src/train.py:184-192) against
    numbers recorded from the UNMODIFIED reference (tests/golden/adversarial.{json,npz}, make_golden.py) at two
    non-degenerate geometries: HR 940x940 (discriminator map 512x3x3) and the native 512x1024 crop (512x1x3).

    What can be pinned end to end is set by the reference's own conditioning, not by this implementation: its fp32
    gradient d(g_d)/d(sr) keeps only cos 0.97 (940x940) / 0.54 (native) with itself when its INPUT is merely rounded to
    bf16 (tests/test_oracle_golden.py::test_discriminator_gradient_conditioning) -- MaxPool argmax flips and an
    InstanceNorm over 9 / 3 elements amplify 2^-9 perturbations.  So: losses to a few percent, gradient norms to 25 %,
    directions as far as that conditioning allows; the per-stage tests above carry the 1e-2 bound on identical inputs."""
    import json
    import os
    import numpy as np
    meta = json.load(open(os.path.join(golden_dir, "adversarial.json")))
    z = np.load(os.path.join(golden_dir, "adversarial.npz"))
    bounds = {"hr940": dict(loss=0.05, dcos=0.80, dratio=0.10, gcos=0.98, acos=0.50, aratio=0.20, fwd=0.985),
              "native": dict(loss=0.12, dcos=0.40, dratio=0.30, gcos=0.85, acos=-1.0, aratio=0.30, fwd=0.95)}
    for tag, rec in meta.items():
        b = bounds[tag]
        torch.manual_seed(14); g = S.SRResNet()
        torch.manual_seed(15); d = S.Discriminator()
        torch.manual_seed(16)
        lr = torch.rand(*rec["lr_shape"]).cuda(); hr = torch.rand(*rec["hr_shape"]).cuda()
        g, d = g.cuda(), d.cuda()
        with torch.no_grad():
            g.eval()
            real0, fake0 = d(hr).cpu(), d(g(lr)).cpu()
        assert real0.shape == tuple(z[f"{tag}/d_real0"].shape)
        assert _cos(real0 - 0.5, torch.from_numpy(z[f"{tag}/d_real0"]) - 0.5)[0] > max(b["fwd"], 0.99), tag
        assert _cos(fake0 - 0.5, torch.from_numpy(z[f"{tag}/d_fake0"]) - 0.5)[0] > b["fwd"], tag
        # three discriminator updates: loss trajectory of the reference function
        d_opt = S.Adam(d.parameters(), lr=5e-5)
        grads = None
        for i, ref in enumerate(rec["d_losses"]):
            loss = S.train_discriminator(d, g, hr, lr, d_opt)
            assert abs(loss - ref) < b["loss"] * abs(ref) + 1e-4, (tag, i, loss, ref)
            if i == 0:
                grads = {k: p.grad.detach().clone() for k, p in d.named_parameters()}
        for k in ("model.0.weight",):
            c, r = _cos(grads[k], torch.from_numpy(z[f"{tag}/d_grad/{k}"]))
            assert c > b["dcos"] and abs(r - 1) < b["dratio"], (tag, k, c, r)
        for k in ("model.4.weight", "model.8.weight", "model.12.weight"):
            c, _ = _cos(grads[k].flatten()[::97], torch.from_numpy(z[f"{tag}/d_grad_sub/{k}"]))
            r = float(grads[k].double().norm()) / rec["d_grad_norms"][k]
            assert c > b["dcos"] and abs(r - 1) < b["dratio"], (tag, k, c, r)
        # GAN-mode generator step with the initial discriminator: com + tv + mean(tanh(D(hr) - D(G(lr))))
        torch.manual_seed(14); g = S.SRResNet().cuda()
        torch.manual_seed(15); d = S.Discriminator().cuda()
        g_opt = S.Adam(g.parameters(), lr=1e-4)
        g_loss, com, tv, g_d = S.train_generator(g, d, lr, hr, None, S.ReconstructionLoss(), g_opt, gan_mode=True)
        gm = rec["gan_mode"]
        assert abs(com - gm["com"]) < 1e-3 * gm["com"] and abs(tv - gm["tv"]) < 2e-2 * gm["tv"], (tag, com, tv)
        assert abs(g_d - gm["g_d"]) < 0.35 * abs(gm["g_d"]) + 1e-4 and g_d * gm["g_d"] > 0, (tag, g_d, gm["g_d"])
        assert abs(g_loss - (com + tv + g_d)) < 1e-5
        gg = {k: p.grad.detach().clone() for k, p in g.named_parameters()}
        for k in ("conv3.weight", "conv3.bias"):
            c, r = _cos(gg[k], torch.from_numpy(z[f"{tag}/g_grad/{k}"]))
            assert c > b["gcos"] and abs(r - 1) < 0.05, (tag, k, c, r)
        for k in ("conv1.weight", "residual_blocks.0.conv1.weight", "upsample.0.weight"):
            assert abs(float(gg[k].double().norm()) / gm["grad_norms"][k] - 1) < 0.25, (tag, k)
        # the adversarial term alone: the gradient that flows through D (input-gradient-only backward) into G
        torch.manual_seed(14); g = S.SRResNet().cuda().train()
        torch.manual_seed(15); d = S.Discriminator().cuda().eval()
        sr = g(lr)
        with d.input_grad_only():
            fake = d(sr)
        with torch.no_grad():
            real = d(hr)
        S.tanh_mean(real, fake).backward()
        for k in ("conv3.weight", "upsample.3.bias"):
            c, r = _cos(dict(g.named_parameters())[k].grad, torch.from_numpy(z[f"{tag}/g_grad_adv/{k}"]))
            assert c > b["acos"] and abs(r - 1) < b["aratio"], (tag, k, c, r)
        for k in ("conv1.weight", "residual_blocks.0.conv1.weight", "upsample.0.weight"):
            n = float(dict(g.named_parameters())[k].grad.double().norm())
            assert abs(n / gm["grad_norms_adv"][k] - 1) < 0.25, (tag, k, n)
        assert all(v is None or torch.isfinite(v).all() for v in (p.grad for p in d.parameters()))


def test_input_grad_only_backward_equals_full_backward(S):
    """Composition pin that is free of the reference's ill-conditioning: the input-gradient-only discriminator backward
    used by the GAN-mode generator step must give exactly the d(sr) of the full backward (same kernels, parameter
    gradients skipped)."""
    torch.manual_seed(31)
    d = S.Discriminator().cuda()
    x0 = torch.rand(1, 3, 512, 1024).cuda()
    w = torch.randn(1, 512, 1, 3).cuda() * 1e-2
    xa = x0.clone().requires_grad_(True)
    d(xa).backward(w)
    xb = x0.clone().requires_grad_(True)
    with d.input_grad_only():
        out = d(xb)
    out.backward(w)
    assert torch.equal(xa.grad, xb.grad)


def test_gan_mode_cuda_graphs_match_eager(S):
    """D step + GAN-mode generator steps replayed from CUDA graphs equal the eagerly enqueued steps bit for bit."""
    crit = S.ReconstructionLoss()
    torch.manual_seed(61)
    lr, hr = torch.rand(1, 3, 107, 171).cuda(), torch.rand(1, 3, 428, 684).cuda()

    def make(graphs):
        gens, opts = [], []
        for s_ in range(2):
            torch.manual_seed(70 + s_)
            g = S.SRResNet(num_residuals=1).cuda()
            gens.append(g)
            opts.append(S.Adam(g.parameters(), lr=1e-3, capturable=True))
        torch.manual_seed(80)
        d = S.Discriminator().cuda()
        d_opt = S.Adam(d.parameters(), lr=1e-4, capturable=True)
        pol = S.MultiGeneratorPolicy(S.PolicyConfig(num_generators=2, force=S.GAN))
        return gens, d, S.MultiGeneratorGAN(gens, opts, crit, discriminator=d, d_optimizer=d_opt, policy=pol,
                                            use_cuda_graphs=graphs)
    ga, da, ta = make(False)
    gb, db, tb = make(True)
    for _ in range(3):
        la = ta.step(lr, hr).clone()
        lb = tb.step(lr, hr).clone()
        torch.cuda.synchronize()
        assert torch.equal(la, lb), (la, lb)
    assert torch.equal(da.flat_parameters(), db.flat_parameters())
    for a, b in zip(ga, gb):
        assert torch.equal(a.flat_parameters(), b.flat_parameters())


def test_l1_mse_bce_match_torch_functional(S):
    """The plain pixel / BCE losses the scope statement names: values and gradients against torch.nn.functional (fp32,
    tolerance 1e-6 relative)."""
    torch.manual_seed(13)
    for shape in [(2, 3, 33, 47), (1, 512, 1, 3), (5,)]:
        a0, b0 = torch.rand(shape) * 0.98 + 0.01, torch.rand(shape)
        for fn, ref in ((S.l1_loss, F.l1_loss), (S.mse_loss, F.mse_loss), (S.bce_loss, F.binary_cross_entropy)):
            a = a0.clone().cuda().requires_grad_(True)
            out = fn(a, b0.cuda())
            (1.5 * out).backward()
            ar = a0.clone().requires_grad_(True)
            r = ref(ar, b0)
            (1.5 * r).backward()
            assert abs(float(out.detach()) - float(r.detach())) <= 2e-6 * max(1.0, abs(float(r.detach()))), (fn.__name__, shape)
            assert maxrel(a.grad, ar.grad) < 1e-5, (fn.__name__, shape)
