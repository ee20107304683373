"""Pins the CPU oracle (oracle/srgan_oracle.py) to outputs of the unmodified reference recorded in
tests/golden/ (made by tests/golden/make_golden.py).  CPU-only."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import srgan_oracle as O


@pytest.fixture(scope="module")
def gj(golden_dir):
    with open(os.path.join(golden_dir, "golden.json")) as f:
        return json.load(f)


def _check_init(sd, ck):
    for k, (s, a) in ck.items():
        v = sd[k].double()
        assert abs(float(v.sum()) - s) <= 1e-9 * max(1.0, abs(a)), k
        assert abs(float(v.abs().sum()) - a) <= 1e-9 * max(1.0, abs(a)), k


def test_seeded_init_matches_reference(gj):
    _check_init(O.init_srresnet_state(1), gj["generator_tiny"]["init_checksum"])
    _check_init(O.init_discriminator_state(3), gj["discriminator_init_checksum"])


def test_generator_forward_loss_grads(gj, golden_dir):
    z = np.load(os.path.join(golden_dir, "generator_tiny.npz"))
    sd = O.init_srresnet_state(1)
    lr = torch.rand(2, 3, 16, 24)
    hr = torch.rand(2, 3, 64, 96)
    with torch.no_grad():
        y_eval = O.srresnet_forward(sd, lr, training=False)
    np.testing.assert_allclose(y_eval.numpy(), z["y_eval"], rtol=0, atol=2e-6)
    losses, grads, sr = O.generator_loss_and_grads(sd, lr, hr)
    np.testing.assert_allclose(sr.numpy(), z["y_train"], rtol=0, atol=5e-6)
    assert abs(losses[1] - float(z["com"])) < 1e-6 and abs(losses[2] - float(z["tv"])) < 1e-7
    np.testing.assert_allclose(sd["residual_blocks.0.bn1.running_mean"].numpy(), z["bn_rm"], atol=1e-7)
    np.testing.assert_allclose(sd["residual_blocks.0.bn1.running_var"].numpy(), z["bn_rv"], atol=1e-7)
    for k in z.files:
        if k.startswith(("grad/", "grad_sub/")):
            ref = z[k]
            got = grads[k.split("/", 1)[1]].numpy()
            if k.startswith("grad_sub/"):
                got = got.flatten()[::97]          # the fixture holds a strided sample of the largest gradients
            assert np.abs(got - ref).max() <= 1e-5 * max(np.abs(ref).max(), 1e-6) + 1e-9, k
    for k, n in gj["generator_tiny"]["grad_norms"].items():
        # biases feeding a training-mode BatchNorm have a mathematically zero gradient: only fp32 noise (~1e-9) there
        assert abs(float(grads[k].double().norm()) - n) <= 2e-5 * max(n, 1e-9) + 2e-8, k


def test_reconstruction_loss_value_and_closed_form_grad(golden_dir):
    z = np.load(os.path.join(golden_dir, "recon_loss.npz"))
    hr, sr = torch.from_numpy(z["hr"]), torch.from_numpy(z["sr"])
    e, t = O.reconstruction_loss(hr, sr)
    assert abs(float(e) - float(z["edge"])) < 1e-7 and abs(float(t) - float(z["tv"])) < 1e-8
    g = O.reconstruction_loss_grad(hr, sr)
    np.testing.assert_allclose(g.numpy(), z["grad"], rtol=0, atol=1e-9)


def test_discriminator_forward_and_size_rule(golden_dir):
    z = np.load(os.path.join(golden_dir, "discriminator_min.npz"))
    sd = O.init_discriminator_state(3)
    x = torch.rand(1, 3, 428, 684)
    assert abs(float(x.double().sum()) - float(z["x_sum"])) < 1e-6
    with torch.no_grad():
        y = O.discriminator_forward(sd, x)
    # the last InstanceNorm normalises over only 1x2 elements: it amplifies fp32 summation-order noise of the conv
    # stack (thread-count dependent) to ~1e-5
    np.testing.assert_allclose(y.numpy(), z["y"], rtol=0, atol=5e-5)
    assert O.discriminator_output_hw(512, 1024) == (1, 3)
    assert O.discriminator_output_hw(684, 684) == (2, 2)
    for bad in ((384, 384), (512, 512), (256, 256), (427, 1024)):
        with pytest.raises(RuntimeError):
            O.discriminator_output_hw(*bad)


def test_cfg1_anchors_four_generator_steps(gj):
    a = gj["cfg1_anchors"]
    sd = O.init_srresnet_state(0)
    O.init_discriminator_state  # D is constructed after G in the reference and consumes RNG before the data
    torch.manual_seed(0)
    sd = O.init_srresnet_state(0)
    _ = O._conv_init(64, 3, 8), O._conv_init(128, 64, 4), O._conv_init(256, 128, 4), O._conv_init(512, 256, 4)
    lr = torch.rand(8, 3, 64, 64)
    hr = torch.rand(8, 3, 256, 256)
    with torch.no_grad():
        y = O.srresnet_forward(sd, lr, training=False)
    assert abs(float(y.double().sum()) - a["eval_sum"]) < 1e-2
    assert abs(float(y[0, 0, 0, 0]) - a["eval_y0000"]) < 1e-6
    keys = O.trainable_keys(sd)
    opt = O.AdamState([sd[k] for k in keys], lr=1e-4)
    for ref in a["steps"][:2]:
        got = O.train_generator_step(sd, opt, lr, hr)
        for g, r in zip(got[:3], ref[:3]):
            assert abs(g - r) <= 2e-5 * abs(r) + 1e-8, (got, ref)


def test_discriminator_step_and_gan_mode(gj):
    dj = gj["d_step"]
    torch.manual_seed(4)
    g_sd = O.init_srresnet_state(4)
    d_sd = {}
    d_sd["model.0.weight"], d_sd["model.0.bias"] = O._conv_init(64, 3, 8)
    d_sd["model.4.weight"], d_sd["model.4.bias"] = O._conv_init(128, 64, 4)
    d_sd["model.8.weight"], d_sd["model.8.bias"] = O._conv_init(256, 128, 4)
    d_sd["model.12.weight"], d_sd["model.12.bias"] = O._conv_init(512, 256, 4)
    lr = torch.rand(*dj["lr_shape"])
    hr = torch.rand(*dj["hr_shape"])
    keys = O.trainable_keys(d_sd)
    opt = O.AdamState([d_sd[k] for k in keys], lr=5e-5)
    for ref in dj["d_losses"]:
        got = O.train_discriminator_step(d_sd, opt, g_sd, hr, lr)
        assert abs(got - ref) <= 1e-4 * abs(ref) + 1e-6, (got, ref)
    for k, (s, a) in dj["d_param_checksum_after"].items():
        # Adam's first steps move every weight by ~lr * sign(grad): weights whose gradient is fp32 noise can go either
        # way depending on the summation order, so the checksum is pinned to 2e-4 rather than to rounding
        assert abs(float(d_sd[k].double().abs().sum()) - a) <= 2e-4 * a, k

    gm = gj["gan_mode"]
    torch.manual_seed(5)
    g_sd = O.init_srresnet_state(5)
    d_sd = {}
    d_sd["model.0.weight"], d_sd["model.0.bias"] = O._conv_init(64, 3, 8)
    d_sd["model.4.weight"], d_sd["model.4.bias"] = O._conv_init(128, 64, 4)
    d_sd["model.8.weight"], d_sd["model.8.bias"] = O._conv_init(256, 128, 4)
    d_sd["model.12.weight"], d_sd["model.12.bias"] = O._conv_init(512, 256, 4)
    losses, grads, _ = O.generator_loss_and_grads(g_sd, lr, hr, d_sd=d_sd, gan_mode=True)
    assert abs(losses[1] - gm["com"]) < 1e-6 and abs(losses[3] - gm["g_d"]) < 1e-6
    for k, n in gm["grad_norms"].items():
        # gradient through D at its smallest valid geometry (last InstanceNorm over 1x2 elements) is sensitive to fp32
        # summation order; pinned to 5e-3
        assert abs(float(grads[k].double().norm()) - n) <= 5e-3 * n + 2e-8, k


def test_image_enhancer_matches_reference(golden_dir):
    z = np.load(os.path.join(golden_dir, "enhancer.npz"))
    x = torch.from_numpy(z["x"])
    np.testing.assert_allclose(O.image_enhancer(x, 1.0).numpy(), z["y1"], rtol=0, atol=1e-6)
    np.testing.assert_allclose(O.image_enhancer(x, 0.5).numpy(), z["y05"], rtol=0, atol=1e-6)


def test_discriminator_gradient_conditioning():
    """Why end-to-end gradient parity through the reference Discriminator cannot be stated at 1e-2: the oracle's OWN fp32
    gradient of the adversarial term w.r.t. the image keeps a cosine of only ~0.5-0.7 with itself at the native 512x1024
    geometry when the input image is rounded to bf16 and nothing else changes (last InstanceNorm over 3 elements, MaxPool
    argmax flips); at 940x940 (9 elements) it stays ~0.97.  The GPU tests therefore bound per-stage errors on identical
    inputs at 1e-2 and end-to-end directions only as far as this conditioning allows."""
    import torch
    from oracle import srgan_oracle as O
    torch.set_num_threads(max(torch.get_num_threads(), 4))
    sd = O.init_discriminator_state(15)

    def grad(x, real):
        x = x.clone().requires_grad_(True)
        torch.mean(torch.tanh(real - O.discriminator_forward(sd, x))).backward()
        return x.grad.double().flatten()

    res = {}
    for (h, w) in ((512, 1024), (940, 940)):
        torch.manual_seed(16)
        hr, sr = torch.rand(1, 3, h, w), torch.rand(1, 3, h, w) * 0.2
        with torch.no_grad():
            real = O.discriminator_forward(sd, hr)
        g0, g1 = grad(sr, real), grad(sr.bfloat16().float(), real)
        res[(h, w)] = float(torch.dot(g0, g1) / (g0.norm() * g1.norm()))
    assert res[(512, 1024)] < 0.9, res          # ill-conditioned: a bf16-sized input perturbation turns the gradient
    assert res[(940, 940)] > 0.9, res
    assert res[(940, 940)] > res[(512, 1024)], res


def test_vgg_perceptual_oracle_matches_reference_fixture(golden_dir):
    """oracle.vgg_features / perceptual_loss (restating src/models.py:123-151, src/utils.py:154-166) against the fixture the
    unmodified reference produced on torchvision-default weights (tests/golden/make_golden.py vgg)."""
    import numpy as np
    import torch
    from oracle import srgan_oracle as O
    z = np.load(os.path.join(golden_dir, "vgg_perceptual.npz"))
    sd = O.init_vgg19_state(int(z["seed"]))
    assert sorted(sd.keys()) == list(z["keys"])
    sr = torch.from_numpy(z["sr"]).requires_grad_(True)
    hr = torch.from_numpy(z["hr"])
    feats = O.vgg_features(sd, hr)
    assert np.allclose(feats["conv3_3"].numpy(), z["conv3_3"], atol=1e-6)
    assert np.allclose(feats["conv4_3"].numpy(), z["conv4_3"], atol=1e-6)
    loss = O.perceptual_loss(sd, sr, hr)
    loss.backward()
    assert abs(float(loss.detach()) - float(z["loss"])) < 1e-7
    assert np.allclose(sr.grad.numpy(), z["grad"], atol=1e-9)
