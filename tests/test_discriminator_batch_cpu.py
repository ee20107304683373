"""CPU checks of the float64 per-stage discriminator reference (oracle/discriminator_stages.py) that
tests/test_discriminator_batch_gpu.py uses to judge the CUDA engine: the stages composed end to end equal the oracle's
discriminator_forward, the stage backwards composed equal torch autograd in float64, and the engine-layout helpers
invert each other.  No GPU needed."""
import pytest
import torch

from oracle import discriminator_stages as R
from oracle import srgan_oracle as O


@pytest.fixture(scope="module")
def case():
    """Two different samples at 428x700, the smallest geometry whose conv outputs are odd at every stage
    (213x349, 53x87, 13x21, 3x5) and whose final map is 1x2."""
    sd = O.init_discriminator_state(21)
    torch.manual_seed(21)
    x = torch.rand(2, 3, 428, 700)
    x[1] = 0.4 + 0.1 * x[1]                  # a low-contrast sample next to a full-range one
    sd64 = {k: v.double() for k, v in sd.items()}
    return sd, sd64, x


def test_composed_forward_equals_oracle(case):
    """Same arithmetic in float64: equal to 1e-10.  Against the oracle's fp32 evaluation every stage output agrees per
    sample to the oracle's own rounding: below 2e-5 measured for stages 0-2; the final InstanceNorm over 2 elements
    amplifies it to 1.4e-4 (full-range sample) and 9.2e-4 (low-contrast sample), hence 2e-3 there."""
    sd, sd64, x = case
    out64, recs = R.forward(sd64, x.double())
    assert out64.shape == (2, 512, 1, 2)
    assert float((out64 - O.discriminator_forward(sd64, x.double())).abs().max()) < 1e-10
    taps = {}
    O.discriminator_forward(sd, x, taps=taps)
    for l, k in enumerate(R.KEYS):
        for n in range(2):
            ref = recs[l]["out"][n]
            err = float((taps[k][n].double() - ref).abs().max() / ref.abs().max())
            assert err < (1e-4 if l < 3 else 2e-3), (l, n, err)
    assert [tuple(r["y"].shape[2:]) for r in recs] == [(213, 349), (53, 87), (13, 21), (3, 5)]


def test_composed_backward_equals_autograd(case):
    _, sd64, x = case
    torch.manual_seed(22)
    x64 = x.double().requires_grad_(True)
    w = {k: v.clone().requires_grad_(True) for k, v in sd64.items()}
    out = O.discriminator_forward(w, x64)
    dout = torch.randn(out.shape, dtype=torch.float64) * 1e-2
    keys = [k for k in R.KEYS for k in (k + ".weight", k + ".bias")]
    ref = torch.autograd.grad(out, [x64] + [w[k] for k in keys], dout)
    _, recs = R.forward(sd64, x.double())
    dx, grads = R.backward(sd64, recs, dout)
    assert torch.allclose(dx, ref[0], rtol=0, atol=1e-10 * float(ref[0].abs().max()))
    for k, g in zip(keys, ref[1:]):
        scale = float(g.abs().max())
        if k.endswith(".bias"):
            # InstanceNorm removes any per-channel constant its input carries, so every bias gradient is zero in
            # exact arithmetic; both sides return float64 rounding residue
            scale = float(ref[0].abs().max())
        assert float((grads[k] - g).abs().max()) <= 1e-9 * scale, k


def test_leaky_branch_override_only_moves_the_zero_crossing():
    """``positive`` changes the LeakyReLU slope only where it disagrees with xhat's sign; the backward through it
    differs from the default exactly at those elements."""
    torch.manual_seed(23)
    y = torch.randn(2, 8, 9, 11, dtype=torch.float64)
    xhat = R.instance_norm(torch.nn.functional.max_pool2d(y, 3, 2))
    pos = xhat > 0
    assert torch.equal(R.post_forward(y, 1, pos), R.post_forward(y, 1))
    flip = pos.clone()
    flip[1, 3, 0, 0] = ~flip[1, 3, 0, 0]
    dout = torch.randn(xhat.shape, dtype=torch.float64)
    a, b = R.post_backward(y, dout, 1), R.post_backward(y, dout, 1, flip)
    assert not torch.equal(a[1], b[1]) and torch.equal(a[0], b[0])


def test_layout_helpers():
    torch.manual_seed(24)
    for Hp, Wp in ((6, 10), (7, 15), (3, 5)):
        Ho, Wo = (Hp + 2 - 4) // 2 + 1, (Wp + 2 - 4) // 2 + 1
        Hs, Ws = Ho + 1, Wo + 1
        z = torch.randn(3, 8, Hp, Wp)
        xs = R.s2d(z, Hs, Ws)
        assert xs.shape == (3, Hs, Ws, 32)
        back, pad = R.uns2d(xs, Hp, Wp)
        assert torch.equal(back, z) and bool((pad == 0).all())
        # XS[n][h'][w'][(a, b, c)] = z[2h'+a-1][2w'+b-1][c]
        for (h, w, a, b, c) in ((1, 1, 0, 0, 5), (Hs - 1, Ws - 1, 1, 0, 2), (1, 2, 1, 1, 7)):
            hp, wp = 2 * h + a - 1, 2 * w + b - 1
            want = z[1, c, hp, wp] if 0 <= hp < Hp and 0 <= wp < Wp else 0.0
            assert float(xs[1, h, w, (a * 2 + b) * 8 + c]) == float(want)
    # stage-0 unfold: U0[n][h'][w'][((v*2+a)*2+b)*3+c] = x[n][c][2h'+a-2][2(w'+v)+b-2]; a 4-tap stride-1 conv over it
    # with re-indexed weights is the 8x8 / s2 / p2 conv
    x = torch.randn(2, 3, 24, 30, dtype=torch.float64)
    Ho, Wo = (24 + 4 - 8) // 2 + 1, (30 + 4 - 8) // 2 + 1
    u = R.unfold0(x, Ho + 3, Wo)
    assert u.shape == (2, Ho + 3, Wo, 64) and bool((u[..., 48:] == 0).all())
    w = torch.randn(5, 3, 8, 8, dtype=torch.float64)
    wk = torch.zeros(4, 5, 64, dtype=torch.float64)              # [tap u][co][ch]
    for ch in range(48):
        v, rem = divmod(ch, 12)
        a, b, c = rem // 6, (rem % 6) // 3, rem % 3
        for t in range(4):
            wk[t, :, ch] = w[:, c, 2 * t + a, 2 * v + b]
    y = sum(torch.einsum("nhwk,ok->nohw", u[:, t:t + Ho], wk[t]) for t in range(4))
    ref = torch.nn.functional.conv2d(x, w, stride=2, padding=2)
    assert torch.allclose(y, ref, rtol=0, atol=1e-12)
