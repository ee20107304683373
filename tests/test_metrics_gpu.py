"""GPU tests of the validation metric: srg_image_metrics / image_metrics / calculate_ssim against the fp64 oracle
(oracle.srgan_oracle.psnr, tests/ssim_oracle.ssim; src/utils.py:141-151), its determinism and batch independence, CUDA-graph capture, and
train.compute_score (src/train.py:263-294) on a small generator."""
import math
import os
import sys

import pytest
import torch

from oracle import srgan_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import ssim_oracle  # noqa: E402  (tests/ssim_oracle.py)

pytestmark = pytest.mark.gpu

SHAPES = [(1, 3, 3, 3), (2, 3, 5, 7), (4, 3, 37, 131), (3, 3, 96, 97), (12, 3, 512, 1024)]
KINDS = ["noise", "unclamped", "constant", "flat_bright"]


@pytest.fixture(scope="module")
def S():
    import srgan_b200
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return srgan_b200


def _pair(shape, kind, seed):
    g = torch.Generator().manual_seed(seed)
    hr = torch.rand(shape, generator=g)
    if kind == "noise":                       # SR = HR + noise, clamped like an image
        sr = (hr + 0.03 * torch.randn(shape, generator=g)).clamp(0, 1)
    elif kind == "unclamped":                 # a raw generator output: outside [0, 1]
        sr = 1.5 * hr - 0.25 + 0.1 * torch.randn(shape, generator=g)
    elif kind == "constant":                  # one constant image against another (and against itself below)
        hr = torch.full(shape, 0.375)
        sr = torch.full(shape, 0.625)
    else:                                     # 0.99 + 1e-3 noise: sum x^2 / 27 - ux^2 cancels in fp32
        hr = 0.99 + 1e-3 * torch.randn(shape, generator=g)
        sr = 0.99 + 1e-3 * torch.randn(shape, generator=g)
    return sr, hr


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_matches_fp64_oracle_per_image(S, shape, kind):
    sr, hr = _pair(shape, kind, seed=sum(shape) + KINDS.index(kind))
    psnr, ssim = S.image_metrics(sr.cuda(), hr.cuda())
    assert psnr.dtype == torch.float64 and ssim.dtype == torch.float64 and psnr.shape == ssim.shape == (shape[0],)
    psnr, ssim = psnr.cpu(), ssim.cpu()
    for n in range(shape[0]):
        assert abs(float(ssim[n]) - ssim_oracle.ssim(sr[n], hr[n])) < 1e-6, (n, float(ssim[n]), ssim_oracle.ssim(sr[n], hr[n]))
        assert abs(float(psnr[n]) - O.psnr(sr[n], hr[n])) < 1e-4, (n, float(psnr[n]), O.psnr(sr[n], hr[n]))


@pytest.mark.parametrize("shape", [(2, 3, 5, 7), (2, 3, 40, 64)], ids=["5x7", "40x64"])
def test_identical_images(S, shape):
    x = torch.rand(shape, device="cuda")
    psnr, ssim = S.image_metrics(x, x)
    assert torch.all(torch.isinf(psnr.cpu())) and torch.all(psnr.cpu() > 0)
    assert torch.allclose(ssim.cpu(), torch.ones(shape[0], dtype=torch.float64), rtol=0, atol=1e-6)


@pytest.mark.parametrize("shape", [(5, 3, 37, 131), (6, 3, 64, 248)], ids=["scalar_path", "vector_path"])
def test_deterministic_and_independent_of_batch_position(S, shape):
    g = torch.Generator(device="cuda").manual_seed(7)
    hr = torch.rand(shape, device="cuda", generator=g)
    sr = hr + 0.05 * torch.randn(shape, device="cuda", generator=g)
    p1, s1 = S.image_metrics(sr, hr)
    p2, s2 = S.image_metrics(sr, hr)
    assert torch.equal(p1, p2) and torch.equal(s1, s2)
    perm = torch.randperm(shape[0], generator=torch.Generator().manual_seed(1)).cuda()
    pp, sp = S.image_metrics(sr[perm], hr[perm])
    assert torch.equal(pp, p1[perm]) and torch.equal(sp, s1[perm])
    p3, s3 = S.image_metrics(sr[1:3], hr[1:3])          # a sub-batch (a view at an offset) scores the same
    assert torch.equal(p3, p1[1:3]) and torch.equal(s3, s1[1:3])
    # swapping the arguments: the formulas are symmetric
    pw, sw = S.image_metrics(hr, sr)
    assert torch.equal(pw, p1) and torch.allclose(sw, s1, rtol=0, atol=1e-7)


def test_calculate_ssim_equals_batched_row(S):
    g = torch.Generator(device="cuda").manual_seed(9)
    hr = torch.rand(3, 3, 48, 80, device="cuda", generator=g)
    sr = hr + 0.02 * torch.randn(3, 3, 48, 80, device="cuda", generator=g)
    _, ssim = S.image_metrics(sr, hr)
    for n in range(3):
        assert S.calculate_ssim(sr[n], hr[n]) == float(ssim[n])
    with pytest.raises(RuntimeError, match="3 x H x W"):
        S.calculate_ssim(sr, hr)
    with pytest.raises(RuntimeError, match="C=1"):
        S.image_metrics(sr[:, :1], hr[:, :1])
    with pytest.raises(RuntimeError, match="H=2"):
        S.image_metrics(sr[:, :, :2], hr[:, :, :2])
    with pytest.raises(RuntimeError, match="same shape"):
        S.image_metrics(sr, hr[:2])


def test_cuda_graph_capture_replays_on_new_data(S):
    shape = (4, 3, 64, 128)
    sr_s = torch.rand(shape, device="cuda")
    hr_s = torch.rand(shape, device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        S.image_metrics(sr_s, hr_s)                     # warm-up: caches the scratch outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        psnr_g, ssim_g = S.image_metrics(sr_s, hr_s)
    for seed in (1, 2):
        g = torch.Generator(device="cuda").manual_seed(seed)
        hr = torch.rand(shape, device="cuda", generator=g)
        sr = hr + 0.04 * torch.randn(shape, device="cuda", generator=g)
        sr_s.copy_(sr)
        hr_s.copy_(hr)
        graph.replay()
        p, s = S.image_metrics(sr, hr)
        torch.cuda.synchronize()
        assert torch.equal(psnr_g, p) and torch.equal(ssim_g, s)


class _CountingLoader:
    """(hr, lr) batches like the reference's validation loader; counts how many were pulled."""

    def __init__(self, batches):
        self.batches, self.pulled = batches, 0

    def __iter__(self):
        for b in self.batches:
            self.pulled += 1
            yield b


@pytest.mark.parametrize("training", [True, False], ids=["from_train_mode", "from_eval_mode"])
def test_compute_score_matches_oracle_and_leaves_the_model_alone(S, training):
    torch.manual_seed(5)
    gen = S.SRResNet(num_residuals=1).cuda()
    # non-trivial running statistics and num_batches_tracked first: one training-mode forward
    gen.train()
    with torch.no_grad():
        gen(torch.rand(2, 3, 16, 24, device="cuda"))
    gen.train(training)
    flat = gen.flat_parameters()
    rt = gen._rt
    before = [t.clone() for t in (flat, rt["flat_buf"], rt["nbt"])]
    g = torch.Generator().manual_seed(6)
    batches = []
    for _ in range(4):
        lr = torch.rand(2, 3, 16, 24, generator=g)
        batches.append(((lr.repeat_interleave(4, 2).repeat_interleave(4, 3) + 0.05 * torch.randn(2, 3, 64, 96, generator=g)), lr))
    loader = _CountingLoader(batches)
    avg_psnr, avg_ssim = S.compute_score(gen, loader, torch.device("cuda"), num_batches=3)
    assert loader.pulled == 3
    assert gen.training == training
    for a, b in zip((flat, rt["flat_buf"], rt["nbt"]), before):
        assert torch.equal(a, b)
    # oracle over the same module's eval-mode outputs
    gen.eval()
    ps, ss = [], []
    with torch.no_grad():
        for hr, lr in batches[:3]:
            sr = gen(lr.cuda()).cpu()
            for n in range(hr.shape[0]):
                ps.append(O.psnr(sr[n], hr[n]))
                ss.append(ssim_oracle.ssim(sr[n], hr[n]))
    assert math.isfinite(avg_psnr)
    assert abs(avg_psnr - sum(ps) / len(ps)) < 1e-4
    assert abs(avg_ssim - sum(ss) / len(ss)) < 1e-6
