"""CPU tests of the trained-like BatchNorm state (tests/bn_affine_state.py): it is non-degenerate, and every BatchNorm bug
class that gamma = 1 / beta = 0 hides moves the quantity the GPU tests check (tests/test_bn_affine_gpu.py) by at least 10x
the bound they check it with.  Everything runs on the float64 oracle; no GPU is needed."""
import itertools
import os
import sys

import pytest
import torch

from oracle import srgan_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bn_affine_state as B  # noqa: E402  (tests/bn_affine_state.py)


@pytest.fixture(scope="module")
def states():
    """the same conv weights with the BatchNorm state of generators k = 0..3 (16 blocks)"""
    base = O.init_srresnet_state(5, num_residuals=16)
    return base, [B.bn_affine_state(base, 7, k) for k in range(4)]


@pytest.fixture(scope="module")
def walk(states):
    """float64 train-mode taps of generators 0 and 1 at the GPU tests' small geometry, with random upstream gradients"""
    _, sts = states
    gen = torch.Generator().manual_seed(3)
    x = torch.rand(2, 3, 16, 24, generator=gen, dtype=torch.float64)
    out = []
    for st in sts[:2]:
        taps = {}
        with torch.no_grad():
            O.srresnet_forward(B.to_double(st), x, training=True, update_running=False, taps=taps)
        out.append(taps)
    dz = torch.randn(out[0]["out1"].shape, generator=gen, dtype=torch.float64)
    return out, dz


# ------------------------------------------------------------------------------------------------ the state is non-degenerate
def test_gamma_vectors_pairwise_distinct(states):
    _, sts = states
    vecs = [st[p + ".weight"] for st in sts for p in B.bn_layers(st)]
    assert len(vecs) == 4 * 32
    dmin = min(float((a - b).abs().max()) for a, b in itertools.combinations(vecs, 2))
    assert dmin >= 0.1, dmin
    betas = [st[p + ".bias"] for st in sts for p in B.bn_layers(st)]
    assert min(float((a - b).abs().max()) for a, b in itertools.combinations(betas, 2)) >= 0.1


def test_negative_gamma_in_bn1_and_bn2(states):
    _, sts = states
    for st in sts:
        for p in B.bn_layers(st):
            g = st[p + ".weight"]
            assert int((g < 0).sum()) == 8, p                       # one channel in eight, in front of the ReLU too
            assert 0.3 <= float(g.abs().min()) and float(g.abs().max()) <= 2.0, p


def test_state_leaves_convs_and_is_reproducible(states):
    base, sts = states
    again = B.bn_affine_state(base, 7, 2)
    for key, v in base.items():
        if ".bn" in key:
            assert not torch.equal(sts[0][key], v), key            # every BatchNorm tensor replaced
        else:
            assert torch.equal(sts[0][key], v), key                 # conv weights and biases untouched
        assert torch.equal(again[key], sts[2][key]), key
    for st in sts:
        for p in B.bn_layers(st):
            assert int(st[p + ".num_batches_tracked"]) > 0
            assert float(st[p + ".running_var"].min()) > 0
    assert float(base["residual_blocks.0.bn1.weight"].min()) == 1.0      # the input state is not modified


@pytest.mark.parametrize("training", [False, True])
def test_activation_rms_stays_order_one_through_16_blocks(states, training):
    """per-block RMS of the residual stream within [0.1, 10] of block 0's: a blown-up or collapsed stream would make a
    max-relative bound blind to most of the tensor"""
    _, sts = states
    x = torch.rand(2, 3, 24, 24, generator=torch.Generator().manual_seed(11), dtype=torch.float64)
    for st in sts[:2]:
        taps = {}
        with torch.no_grad():
            O.srresnet_forward(B.to_double(st), x, training=training, update_running=False, taps=taps)
        rms = [float(taps[f"residual_blocks.{b}"].pow(2).mean().sqrt()) for b in range(16)]
        assert all(0.1 <= r / rms[0] <= 10.0 for r in rms), rms


# ------------------------------------------------------------------------------------------------ sensitivity (teeth)
def _layer_io(taps, b, j):
    """(pre-BatchNorm conv output y, the stream entering the block) of layer bn{j} of block b"""
    x_in = taps["out1"] if b == 0 else taps[f"residual_blocks.{b - 1}"]
    return taps[f"residual_blocks.{b}.conv{j}"], x_in


def _bn_out(y, x_in, gamma, beta, j):
    z = B.bn_train(y, gamma, beta)
    return torch.relu(z) if j == 1 else z + x_in


def _each_layer(st):
    for b in range(16):
        for j in (1, 2):
            yield b, j, f"residual_blocks.{b}.bn{j}"


def _min_fwd_change(st, taps, mutate):
    """smallest, over the 32 layers, max-rel change of the BatchNorm(+ReLU / +skip) output when (gamma, beta) of the
    layer are replaced by mutate(b, j, gamma, beta)"""
    worst = float("inf")
    for b, j, p in _each_layer(st):
        y, x_in = _layer_io(taps, b, j)
        g, be = st[p + ".weight"].double(), st[p + ".bias"].double()
        g2, be2 = mutate(b, j, g, be)
        worst = min(worst, B.maxrel(_bn_out(y, x_in, g2, be2, j), _bn_out(y, x_in, g, be, j)))
    return worst


def _min_bwd_change(st, taps, dz, mutate_gamma):
    """smallest max-rel change of the BatchNorm-backward d y when gamma is replaced by mutate_gamma(b, j, gamma)"""
    worst = float("inf")
    for b, j, p in _each_layer(st):
        y, _ = _layer_io(taps, b, j)
        g, be = st[p + ".weight"].double(), st[p + ".bias"].double()
        dy = B.bn_train_bwd(y, g, be, dz)[0]
        dy2 = B.bn_train_bwd(y, mutate_gamma(b, j, g), be, dz)[0]
        worst = min(worst, B.maxrel(dy2, dy))
    return worst


def _other(st, b, j):
    """the neighbouring layer's prefix: bn2 of the same block for bn1, bn1 of the next block (or the previous, at the
    end) for bn2 -- the slip of an off-by-one table entry"""
    if j == 1:
        return f"residual_blocks.{b}.bn2"
    return f"residual_blocks.{b + 1 if b < 15 else b - 1}.bn1"


def test_sensitivity_neighbouring_layer_gamma(states, walk):
    _, sts = states
    st, taps, dz = sts[0], walk[0][0], walk[1]
    fwd = _min_fwd_change(st, taps, lambda b, j, g, be: (st[_other(st, b, j) + ".weight"].double(), be))
    bwd = _min_bwd_change(st, taps, dz, lambda b, j, g: st[_other(st, b, j) + ".weight"].double())
    # the fused backward table's bn2 of block b - 1 replaced by block b's
    bwd_b = min(B.maxrel(B.bn_train_bwd(walk[0][0][f"residual_blocks.{b - 1}.conv2"], st[f"residual_blocks.{b}.bn2.weight"],
                                        st[f"residual_blocks.{b - 1}.bn2.bias"], dz)[0],
                         B.bn_train_bwd(walk[0][0][f"residual_blocks.{b - 1}.conv2"], st[f"residual_blocks.{b - 1}.bn2.weight"],
                                        st[f"residual_blocks.{b - 1}.bn2.bias"], dz)[0]) for b in range(1, 16))
    assert min(fwd, bwd, bwd_b) >= 10 * B.TOL_LAYER, (fwd, bwd, bwd_b)


def test_sensitivity_channel_permutation(states, walk):
    _, sts = states
    st, taps, dz = sts[0], walk[0][0], walk[1]
    fwd = _min_fwd_change(st, taps, lambda b, j, g, be: (torch.roll(g, 1), torch.roll(be, 1)))
    bwd = _min_bwd_change(st, taps, dz, lambda b, j, g: g[torch.arange(64) ^ 1])
    assert min(fwd, bwd) >= 10 * B.TOL_LAYER, (fwd, bwd)


def test_sensitivity_cross_generator(states, walk):
    """generator 1 run with generator 0's BatchNorm parameters / running statistics, on generator 1's own activations"""
    _, sts = states
    s0, s1, taps1, dz = sts[0], sts[1], walk[0][1], walk[1]
    fwd = _min_fwd_change(s1, taps1, lambda b, j, g, be: (s0[f"residual_blocks.{b}.bn{j}.weight"].double(),
                                                          s0[f"residual_blocks.{b}.bn{j}.bias"].double()))
    bwd = _min_bwd_change(s1, taps1, dz, lambda b, j, g: s0[f"residual_blocks.{b}.bn{j}.weight"].double())
    run = float("inf")
    for b, j, p in _each_layer(s1):
        y = taps1[f"residual_blocks.{b}.conv{j}"]
        ok = B.running_update(s1[p + ".running_mean"], s1[p + ".running_var"], y)
        bad = B.running_update(s0[p + ".running_mean"], s0[p + ".running_var"], y)
        run = min(run, B.maxrel(bad[0], ok[0]), B.maxrel(bad[1], ok[1]))
    assert min(fwd, bwd) >= 10 * B.TOL_LAYER and run >= 10 * B.TOL_RUNNING, (fwd, bwd, run)


def test_sensitivity_sign_of_gamma_and_beta(states, walk):
    """A gamma whose sign is lost in front of the ReLU moves the layer by 10x the bound.  A dropped or wrong-signed beta in
    the TRAINING forward's shift is seen with less margin: beta ~ N(0, 0.3) is small next to gamma * x_hat (up to ~6), and
    a bn2 output also carries the skip stream, so a dropped beta moves the weakest layer (a deep bn2) by 2.4e-2 of the
    tensor's largest entry, 2.4x the bound.  The eval fold's beta is checked end to end, where a dropped beta moves the
    output by 10x the bound (test_*_eval_bound_*)."""
    _, sts = states
    st, taps = sts[0], walk[0][0]
    no_beta = _min_fwd_change(st, taps, lambda b, j, g, be: (g, torch.zeros_like(be)))
    neg_beta = _min_fwd_change(st, taps, lambda b, j, g, be: (g, -be))
    abs_gamma = _min_fwd_change(st, taps, lambda b, j, g, be: (g.abs(), be))
    assert abs_gamma >= 10 * B.TOL_LAYER, abs_gamma
    assert no_beta >= 2 * B.TOL_LAYER and neg_beta >= 4 * B.TOL_LAYER, (no_beta, neg_beta)


def test_sensitivity_missing_gamma_factor(states, walk):
    """inv instead of gamma * inv: in the training backward's d y, in the frozen backward's d y and in the frozen path's
    conv-bias gradient dbias = sum(gamma * inv * dz)"""
    _, sts = states
    st, taps, dz = sts[0], walk[0][0], walk[1]
    bwd = _min_bwd_change(st, taps, dz, lambda b, j, g: torch.ones_like(g))
    frozen_dy, frozen_dbias = float("inf"), float("inf")
    for b, j, p in _each_layer(st):
        y = taps[f"residual_blocks.{b}.conv{j}"]
        dy = B.bn_eval_bwd(y, st, p, dz)[0]
        inv = torch.rsqrt(st[p + ".running_var"].double() + B.EPS)
        dy_bad = dz * inv[None, :, None, None]
        frozen_dy = min(frozen_dy, B.maxrel(dy_bad, dy))
        frozen_dbias = min(frozen_dbias, B.maxrel(dy_bad.sum((0, 2, 3)), dy.sum((0, 2, 3))))
    assert min(bwd, frozen_dy) >= 10 * B.TOL_LAYER and frozen_dbias >= 10 * B.TOL_WGRAD, (bwd, frozen_dy, frozen_dbias)


def test_sensitivity_running_update_start(states, walk):
    """the running update started from (0, 1) instead of the loaded statistics"""
    _, sts = states
    st, taps = sts[0], walk[0][0]
    worst = float("inf")
    for b, j, p in _each_layer(st):
        y = taps[f"residual_blocks.{b}.conv{j}"]
        ok = B.running_update(st[p + ".running_mean"], st[p + ".running_var"], y)
        bad = B.running_update(torch.zeros(64), torch.ones(64), y)
        worst = min(worst, B.maxrel(bad[0], ok[0]), B.maxrel(bad[1], ok[1]))
    assert worst >= 10 * B.TOL_RUNNING, worst


def _drop_beta(sd):
    out = dict(sd)
    for p in B.bn_layers(sd):
        out[p + ".bias"] = torch.zeros_like(sd[p + ".bias"])
    return out


@pytest.mark.parametrize("n_res,upscale", [(1, 4), (2, 4), (2, 2), (1, 8)])
def test_shallow_eval_bound_has_headroom_and_sees_a_dropped_beta(n_res, upscale):
    """the eval cases of the GPU tests with n_res <= 2 (TOL_EVAL_SHALLOW / PSNR_EVAL_SHALLOW end to end): bf16 storage
    alone stays inside the bound with margin (measured 0.77e-2 .. 0.98e-2, 53.1 .. 57.0 dB), a beta dropped from the eval
    fold moves the output by 10x the bound (measured 0.22 .. 0.40)"""
    sd = B.bn_affine_state(O.init_srresnet_state(20 + n_res, num_residuals=n_res, upscale_factor=upscale), 20 + n_res)
    x = torch.rand(2, 3, 16, 24, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    if upscale > 4:                 # x16 output: fp32 (1e-6 from float64) keeps the test short
        sd, x = {k: v.float() if v.dtype.is_floating_point else v for k, v in sd.items()}, x.float()
    else:
        sd = B.to_double(sd)
    ref = O.srresnet_forward(sd, x, training=False)
    model = B.eval_forward_bf16_storage(sd, x)
    assert B.maxrel(model, ref) <= 0.6 * B.TOL_EVAL_SHALLOW, B.maxrel(model, ref)
    assert B.psnr_rel(model, ref) >= B.PSNR_EVAL_SHALLOW + 3
    bad = O.srresnet_forward(_drop_beta(sd), x, training=False)
    assert B.maxrel(bad, ref) >= 10 * B.TOL_EVAL_SHALLOW


def test_deep_eval_bound_is_calibrated():
    """TOL_EVAL_DEEP / PSNR_EVAL_DEEP come from the bf16-storage model of the folded eval forward on the DEEP_EVAL case
    (measured max-rel 1.42e-2, 51.4 dB): the model stays inside the bound without it being loose, and a dropped beta
    moves the output by 10x the bound and far below the floor"""
    sd, x = B.deep_eval_case()
    ref = O.srresnet_forward(sd, x, training=False)                       # fp32: 1.4e-6 from the fp64 oracle here
    model = B.eval_forward_bf16_storage(sd, x)
    err, db = B.maxrel(model, ref), B.psnr_rel(model, ref)
    assert B.TOL_EVAL_DEEP / 4 <= err <= B.TOL_EVAL_DEEP, err
    assert B.PSNR_EVAL_DEEP + 3 <= db <= B.PSNR_EVAL_DEEP + 12, db
    bad = O.srresnet_forward(_drop_beta(sd), x, training=False)
    assert B.maxrel(bad, ref) >= 10 * B.TOL_EVAL_DEEP
    assert B.psnr_rel(bad, ref) < B.PSNR_EVAL_DEEP - 20
