"""Generate the golden fixtures in this directory by running the UNMODIFIED reference
(/root/reference/src) on fixed seeds.  Run in the build container only (the reference does not
travel to the GPU box):

    python tests/golden/make_golden.py

Off-path imports that are absent here (skimage, matplotlib) are replaced by empty stand-in modules
before ``src.train`` is imported; ``torch.cuda.empty_cache`` is neutralised on CPU (SURVEY 8c).
Nothing in the reference is edited or copied.
"""
import json
import os
import sys
import types

import numpy as np
import torch

REF = "/root/reference"
HERE = os.path.dirname(os.path.abspath(__file__))


def import_reference():
    for name in ("skimage", "skimage.metrics", "matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["skimage.metrics"].structural_similarity = None
    sys.modules["skimage.metrics"].peak_signal_noise_ratio = None
    sys.modules["matplotlib"].pyplot = sys.modules["matplotlib.pyplot"]
    sys.path.insert(0, REF)
    torch.cuda.empty_cache = lambda: None
    import src.models as models
    import src.train as train
    import src.utils as utils
    return models, train, utils


def checksum(sd):
    return {k: [float(v.double().sum()), float(v.double().abs().sum())] for k, v in sd.items()
            if v.dtype.is_floating_point}


def make_enhancer_fixture(models):
    """ImageEnhancer (src/models.py:28-41) on a fixed input; separate file so it can be regenerated on its own:
    python tests/golden/make_golden.py enhancer"""
    torch.manual_seed(6)
    x = torch.rand(2, 3, 18, 26) * 1.4 - 0.2          # values outside [0, 1] exercise the clamp
    np.savez_compressed(os.path.join(HERE, "enhancer.npz"), x=x.numpy(),
                        y1=models.ImageEnhancer().forward(x).numpy(), y05=models.ImageEnhancer(factor=0.5).forward(x).numpy())


def make_adversarial_fixture(models, train, utils):
    """Discriminator step (src/train.py:206-230) and GAN-mode generator term (src/train.py:184-192) at NON-degenerate
    geometries: HR 940 x 940 (discriminator map 512 x 3 x 3) and the reference's native 512 x 1024 crop (512 x 1 x 3,
    src/transformers.py:74).  At the minimum valid size (428 x 684) the last InstanceNorm sees two elements and the sigmoid
    map collapses to a constant, which pins nothing.  python tests/golden/make_golden.py adversarial"""
    out = {}
    arrays = {}
    for tag, (h, w) in (("hr940", (235, 235)), ("native", (128, 256))):
        # ---- two discriminator updates, generator in eval mode (reference function, unmodified)
        torch.manual_seed(14)
        g = models.SRResNet()
        torch.manual_seed(15)
        d = models.Discriminator()
        torch.manual_seed(16)
        lr = torch.rand(1, 3, h, w)
        hr = torch.rand(1, 3, 4 * h, 4 * w)
        d_opt = torch.optim.Adam(d.parameters(), lr=5e-5)
        with torch.no_grad():
            g.eval()
            real0 = d(hr)
            fake0 = d(g(lr))
        d_losses = [train.train_discriminator(d, g, hr, lr, d_opt)]
        torch.autograd.set_detect_anomaly(False)
        grads = {k: p.grad.detach().clone() for k, p in d.named_parameters()}      # gradients of the FIRST update
        for _ in range(2):
            d_losses.append(train.train_discriminator(d, g, hr, lr, d_opt))
            torch.autograd.set_detect_anomaly(False)
        arrays[f"{tag}/d_real0"] = real0.numpy()
        arrays[f"{tag}/d_fake0"] = fake0.numpy()
        for k in ("model.0.weight", "model.0.bias", "model.4.bias"):
            arrays[f"{tag}/d_grad/{k}"] = grads[k].numpy()
        for k in ("model.4.weight", "model.8.weight", "model.12.weight"):
            arrays[f"{tag}/d_grad_sub/{k}"] = grads[k].flatten()[::97].numpy()      # strided sample of the large tensors
        rec = {"lr_shape": [1, 3, h, w], "hr_shape": [1, 3, 4 * h, 4 * w], "seeds": {"g": 14, "d": 15, "data": 16},
               "d_losses": d_losses, "d_grad_norms": {k: float(v.double().norm()) for k, v in grads.items()},
               "d_param_checksum_after": checksum(d.state_dict())}
        # ---- GAN-mode generator objective: com + tv + mean(tanh(D(hr) - D(G(lr)))) (the commented reference lines)
        torch.manual_seed(14)
        g = models.SRResNet()
        torch.manual_seed(15)
        d = models.Discriminator()
        g.train(); d.eval()
        sr = g(lr)
        fake = d(sr)
        with torch.no_grad():
            real = d(hr)
        com, tv = utils.ReconstructionLoss()(hr, sr)
        g_d = torch.mean(torch.tanh(real - fake))
        (com + tv + g_d).backward()
        gg = {k: p.grad.detach() for k, p in g.named_parameters()}
        # the adversarial term alone (gradient through D into G), for a sharper check of the dgrad chain through D
        g.zero_grad()
        sr2 = g(lr)
        torch.mean(torch.tanh(real - d(sr2))).backward()
        ga = {k: p.grad.detach() for k, p in g.named_parameters()}
        for k in ("conv3.weight", "conv3.bias", "upsample.3.bias"):
            arrays[f"{tag}/g_grad/{k}"] = gg[k].numpy()
            arrays[f"{tag}/g_grad_adv/{k}"] = ga[k].numpy()
        rec["gan_mode"] = {"com": com.item(), "tv": tv.item(), "g_d": g_d.item(),
                           "grad_norms": {k: float(v.double().norm()) for k, v in gg.items()},
                           "grad_norms_adv": {k: float(v.double().norm()) for k, v in ga.items()}}
        out[tag] = rec
        print(tag, "d_losses", d_losses, "g_d", g_d.item(), flush=True)
    np.savez_compressed(os.path.join(HERE, "adversarial.npz"), **arrays)
    with open(os.path.join(HERE, "adversarial.json"), "w") as f:
        json.dump(out, f, indent=1)


def make_checkpoint_fixture(models):
    """A checkpoint written the way the reference writes it under DDP (src/train.py:123-125 saves
    ``generator.state_dict()`` of the DDP-wrapped model: every key carries the ``module.`` prefix), for the f-1
    interop test.  Tiny SRResNet (2 residual blocks).  Its parameters are the reference's default initialisation under
    seed 21, which oracle.srgan_oracle.init_srresnet_state reproduces bit for bit, so only the entries that initialisation
    does not give (the BatchNorm buffers moved by one training pass) are stored, in reference_ddp_checkpoint_buffers.pth;
    reference_ddp_checkpoint.json records the key order and a sha256 of every entry, against which tests/conftest.py
    rebuilds the whole checkpoint.  python tests/golden/make_golden.py checkpoint"""
    import hashlib
    torch.manual_seed(21)
    g = models.SRResNet(num_residuals=2)
    init = {k: v.clone() for k, v in g.state_dict().items()}
    g.train()
    with torch.no_grad():
        g(torch.rand(1, 3, 8, 8))             # one training-mode pass: BatchNorm buffers / num_batches_tracked move
    sd = {"module." + k: v for k, v in g.state_dict().items()}
    torch.save({k: v for k, v in sd.items() if not torch.equal(v, init[k[len("module."):]])},
               os.path.join(HERE, "reference_ddp_checkpoint_buffers.pth"))
    meta = {"seed": 21, "num_residuals": 2, "keys": list(sd),
            "entries": {k: [str(v.dtype), list(v.shape), hashlib.sha256(v.numpy().tobytes()).hexdigest()]
                        for k, v in sd.items()}}
    with open(os.path.join(HERE, "reference_ddp_checkpoint.json"), "w") as f:
        json.dump(meta, f, indent=1)
    g.eval()
    x = torch.linspace(0, 1, 3 * 12 * 10).reshape(1, 3, 12, 10)
    with torch.no_grad():
        y = g(x)
    np.savez_compressed(os.path.join(HERE, "reference_ddp_checkpoint_io.npz"), x=x.numpy(), y=y.numpy())


def make_vgg_fixture(models, utils):
    """VGGFeatureExtractor + perceptal_loss (src/models.py:123-151, src/utils.py:154-166), UNMODIFIED, on seeded
    torchvision-default weights: the reference asks torchvision for the ImageNet checkpoint (a download); the one thing
    replaced here is that request -- ``torchvision.models.vgg19`` is wrapped to build the same architecture with
    ``weights=None`` under a fixed seed.  The weights themselves (42 MB for the 12 executed convs) are NOT stored: the
    test rebuilds them with oracle.init_vgg19_state(seed) and this function checks that both constructions agree.
    python tests/golden/make_golden.py vgg"""
    import torchvision
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from oracle import srgan_oracle as O
    real_vgg19 = torchvision.models.vgg19

    def seeded_vgg19(weights=None, **kw):
        torch.manual_seed(31)
        return real_vgg19(weights=None, **kw)

    models.models.vgg19 = seeded_vgg19
    try:
        fe = models.VGGFeatureExtractor()
    finally:
        models.models.vgg19 = real_vgg19
    sd_ref = {k: v.detach().clone() for k, v in fe.state_dict().items()}
    # torchvision builds the classifier's Linear layers after the features, so the feature tensors only depend on the
    # seed and on the conv order: the oracle's own initialiser must reproduce them bit for bit
    sd_or = O.init_vgg19_state(31)
    for k, v in sd_or.items():
        assert torch.equal(v, sd_ref[k]), k
    torch.manual_seed(32)
    sr = torch.rand(2, 3, 40, 24, requires_grad=True)
    hr = torch.rand(2, 3, 40, 24)
    feats = fe(hr)
    loss = utils.perceptal_loss(sr, hr, fe)
    loss.backward()
    # the oracle restatement against the reference, same weights
    sr2 = sr.detach().clone().requires_grad_(True)
    loss_o = O.perceptual_loss(sd_or, sr2, hr)
    loss_o.backward()
    assert abs(float(loss_o) - float(loss)) < 1e-7 and torch.allclose(sr2.grad, sr.grad, atol=1e-9)
    np.savez_compressed(os.path.join(HERE, "vgg_perceptual.npz"), seed=31, sr=sr.detach().numpy(), hr=hr.numpy(),
                        loss=float(loss), grad=sr.grad.numpy(),
                        conv3_3=feats["conv3_3"].detach().numpy(), conv4_3=feats["conv4_3"].detach().numpy(),
                        keys=np.array(sorted(sd_ref.keys())))
    print("vgg fixture: loss", float(loss), "grad max", float(sr.grad.abs().max()), "feature shapes",
          {k: tuple(v.shape) for k, v in feats.items()})


def main():
    torch.set_num_threads(8)
    models, train, utils = import_reference()
    out = {}

    # ---- 1. tiny generator: forward (eval + train), loss, grads ---------------------------------
    torch.manual_seed(1)
    g = models.SRResNet()
    init_ck = checksum(g.state_dict())
    lr = torch.rand(2, 3, 16, 24)
    hr = torch.rand(2, 3, 64, 96)
    g.eval()
    with torch.no_grad():
        y_eval = g(lr)
    g.train()
    y_train = g(lr)
    crit = utils.ReconstructionLoss()
    com, tv = crit(hr, y_train)
    (com + tv).backward()
    grads = {k: p.grad for k, p in g.named_parameters()}
    sel = ["conv1.weight", "conv1.bias", "residual_blocks.0.conv1.weight", "residual_blocks.0.bn1.weight",
           "residual_blocks.0.bn1.bias", "residual_blocks.7.conv2.weight", "residual_blocks.15.bn2.weight",
           "conv2.weight", "upsample.3.bias", "conv3.weight", "conv3.bias"]
    sel_sub = ["upsample.0.weight", "upsample.3.weight"]      # the largest gradients: strided sample, file under 1 MB
    np.savez_compressed(
        os.path.join(HERE, "generator_tiny.npz"),
        y_eval=y_eval.numpy(), y_train=y_train.detach().numpy(),
        com=np.float64(com.item()), tv=np.float64(tv.item()),
        bn_rm=g.residual_blocks[0].bn1.running_mean.numpy(), bn_rv=g.residual_blocks[0].bn1.running_var.numpy(),
        **{"grad/" + k: grads[k].numpy() for k in sel},
        **{"grad_sub/" + k: grads[k].flatten()[::97].numpy() for k in sel_sub},
    )
    out["generator_tiny"] = {
        "seed": 1, "lr_shape": [2, 3, 16, 24], "hr_shape": [2, 3, 64, 96], "init_checksum": init_ck,
        "grad_norms": {k: float(v.double().norm()) for k, v in grads.items()},
    }

    # ---- 2. ReconstructionLoss value + gradient ---------------------------------------------------
    torch.manual_seed(2)
    hr2 = torch.rand(2, 3, 20, 28)
    sr2 = (hr2 + 0.1 * torch.randn(2, 3, 20, 28)).requires_grad_(True)
    e, t = utils.ReconstructionLoss()(hr2, sr2)
    (e + t).backward()
    np.savez_compressed(os.path.join(HERE, "recon_loss.npz"), hr=hr2.numpy(), sr=sr2.detach().numpy(),
                        edge=np.float64(e.item()), tv=np.float64(t.item()), grad=sr2.grad.numpy())

    # ---- 3. cfg1 anchors: 4 x train_generator as-is (SURVEY 8c) -----------------------------------
    torch.manual_seed(0)
    g = models.SRResNet()
    d = models.Discriminator()
    lr = torch.rand(8, 3, 64, 64)
    hr = torch.rand(8, 3, 256, 256)
    g.eval()
    with torch.no_grad():
        y = g(lr)
    anchors = {"eval_sum": float(y.double().sum()), "eval_mean_abs": float(y.double().abs().mean()),
               "eval_y0000": float(y[0, 0, 0, 0]), "steps": []}
    crit = utils.ReconstructionLoss()
    opt = torch.optim.Adam(g.parameters(), lr=1e-4)
    for _ in range(4):
        anchors["steps"].append(list(train.train_generator(g, d, lr, hr, None, crit, opt)))
    torch.autograd.set_detect_anomaly(False)
    out["cfg1_anchors"] = anchors

    # ---- 4. discriminator at its smallest valid geometry (428 x 684) + one D step -----------------
    torch.manual_seed(3)
    d = models.Discriminator()
    out["discriminator_init_checksum"] = checksum(d.state_dict())
    x = torch.rand(1, 3, 428, 684)
    with torch.no_grad():
        yd = d(x)
    np.savez_compressed(os.path.join(HERE, "discriminator_min.npz"), y=yd.numpy(),
                        x_sum=np.float64(x.double().sum()))
    torch.manual_seed(4)
    g = models.SRResNet()
    d = models.Discriminator()
    lr = torch.rand(1, 3, 107, 171)
    hr = torch.rand(1, 3, 428, 684)
    d_opt = torch.optim.Adam(d.parameters(), lr=5e-5)
    d_losses = [train.train_discriminator(d, g, hr, lr, d_opt) for _ in range(2)]
    torch.autograd.set_detect_anomaly(False)
    out["d_step"] = {"seed": 4, "lr_shape": [1, 3, 107, 171], "hr_shape": [1, 3, 428, 684], "d_losses": d_losses,
                     "d_param_checksum_after": checksum(d.state_dict())}

    # ---- 5. GAN-mode generator term (src/train.py:184-192, commented lines restated by the caller) --
    torch.manual_seed(5)
    g = models.SRResNet()
    d = models.Discriminator()
    g.train(); d.eval()
    sr = g(lr)
    fake = d(sr)
    with torch.no_grad():
        real = d(hr)
    com, tv = utils.ReconstructionLoss()(hr, sr)
    g_d = torch.mean(torch.tanh(real - fake))
    (com + tv + g_d).backward()
    out["gan_mode"] = {"seed": 5, "com": com.item(), "tv": tv.item(), "g_d": g_d.item(),
                       "grad_norms": {k: float(p.grad.double().norm()) for k, p in g.named_parameters()}}

    make_enhancer_fixture(models)
    make_adversarial_fixture(models, train, utils)
    make_checkpoint_fixture(models)

    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("golden fixtures written to", HERE)


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "enhancer":
        make_enhancer_fixture(import_reference()[0])
    elif len(sys.argv) > 1 and sys.argv[1] == "adversarial":
        torch.set_num_threads(8)
        make_adversarial_fixture(*import_reference())
    elif len(sys.argv) > 1 and sys.argv[1] == "vgg":
        torch.set_num_threads(8)
        m, _, u = import_reference()
        make_vgg_fixture(m, u)
    elif len(sys.argv) > 1 and sys.argv[1] == "checkpoint":
        make_checkpoint_fixture(import_reference()[0])
    else:
        main()
