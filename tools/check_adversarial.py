"""Developer tool (GPU box): CUDA train_discriminator / GAN-mode train_generator against the reference's own numbers at
non-degenerate geometries (tests/golden/adversarial.{json,npz}, written by make_golden.py from the unmodified reference)."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import srgan_b200 as S  # noqa: E402


def cos(a, b):
    a, b = a.double().flatten().cpu(), b.double().flatten().cpu()
    return float(torch.dot(a, b) / (a.norm() * b.norm()).clamp_min(1e-300)), float(a.norm() / b.norm().clamp_min(1e-300))


def main():
    gd = os.path.join(ROOT, "tests", "golden")
    meta = json.load(open(os.path.join(gd, "adversarial.json")))
    z = np.load(os.path.join(gd, "adversarial.npz"))
    for tag, rec in meta.items():
        print("====", tag, rec["lr_shape"], "->", rec["hr_shape"])
        torch.manual_seed(14); g = S.SRResNet()
        torch.manual_seed(15); d = S.Discriminator()
        torch.manual_seed(16)
        lr = torch.rand(*rec["lr_shape"]); hr = torch.rand(*rec["hr_shape"])
        g, d, lr, hr = g.cuda(), d.cuda(), lr.cuda(), hr.cuda()
        with torch.no_grad():
            g.eval()
            real0, fake0 = d(hr).cpu(), d(g(lr)).cpu()
        for nm, t in (("d_real0", real0), ("d_fake0", fake0)):
            ref = torch.from_numpy(z[f"{tag}/{nm}"])
            print(f"  {nm}: mean|diff| {float((t - ref).abs().mean()):.4e}  max {float((t - ref).abs().max()):.3e}  cos(centered) {cos(t - 0.5, ref - 0.5)[0]:.5f}")
        d_opt = S.Adam(d.parameters(), lr=5e-5)
        losses = []
        for i in range(3):
            losses.append(S.train_discriminator(d, g, hr, lr, d_opt))
            if i == 0:
                grads = {k: p.grad.detach().clone() for k, p in d.named_parameters()}
        print("  d_losses ours", losses, "ref", rec["d_losses"])
        for k in ("model.0.weight",):
            print(f"  d grad {k}: cos/ratio {cos(grads[k], torch.from_numpy(z[f'{tag}/d_grad/{k}']))}")
        for k in ("model.4.weight", "model.8.weight", "model.12.weight"):
            print(f"  d grad {k} (1/97 sample): cos/ratio {cos(grads[k].flatten()[::97], torch.from_numpy(z[f'{tag}/d_grad_sub/{k}']))}  "
                  f"norm ours {float(grads[k].double().norm()):.5f} ref {rec['d_grad_norms'][k]:.5f}")
        # GAN-mode generator step with the INITIAL discriminator
        torch.manual_seed(14); g = S.SRResNet().cuda()
        torch.manual_seed(15); d = S.Discriminator().cuda()
        crit = S.ReconstructionLoss()
        g_opt = S.Adam(g.parameters(), lr=1e-4)
        out = S.train_generator(g, d, lr, hr, None, crit, g_opt, gan_mode=True)
        gm = rec["gan_mode"]
        print(f"  gan step ours (g,com,tv,g_d) {out}  ref com {gm['com']:.7f} tv {gm['tv']:.4e} g_d {gm['g_d']:.4e}")
        gg = {k: p.grad.detach().clone() for k, p in g.named_parameters()}
        for k in ("conv3.weight", "conv3.bias", "upsample.3.bias"):
            print(f"  g grad {k}: cos/ratio {cos(gg[k], torch.from_numpy(z[f'{tag}/g_grad/{k}']))}")
        for k in ("conv1.weight", "residual_blocks.0.conv1.weight", "upsample.0.weight"):
            print(f"  g grad norm {k}: ours {float(gg[k].double().norm()):.5f} ref {gm['grad_norms'][k]:.5f}")
        # adversarial term alone
        torch.manual_seed(14); g = S.SRResNet().cuda().train()
        torch.manual_seed(15); d = S.Discriminator().cuda().eval()
        sr = g(lr)
        with d.input_grad_only():
            fake = d(sr)
        with torch.no_grad():
            real = d(hr)
        S.tanh_mean(real, fake).backward()
        ga = {k: p.grad.detach().clone() for k, p in g.named_parameters()}
        for k in ("conv3.weight", "conv3.bias", "upsample.3.bias"):
            print(f"  g grad (adversarial term only) {k}: cos/ratio {cos(ga[k], torch.from_numpy(z[f'{tag}/g_grad_adv/{k}']))}")
        for k in ("conv1.weight", "residual_blocks.0.conv1.weight", "upsample.0.weight"):
            print(f"  g grad_adv norm {k}: ours {float(ga[k].double().norm()):.5f} ref {gm['grad_norms_adv'][k]:.5f}")


if __name__ == "__main__":
    main()
