"""Discriminator parity at the batch sizes it trains at.

The discriminator never runs at batch 1 in a GAN-mode step: train_discriminator concatenates HR and SR into one pass
of batch 2n, and the gan-native workload drives it at N = 24 on 512x1024 crops.  Almost every kernel in
csrc/discriminator.cu computes a per-sample offset that is 0 at N = 1, so the checks here run N in {2, 3} at four
geometries and N = 24 at 512x1024, with samples that differ in kind and scale.

Each stage is judged on its own inputs: the engine's bf16 operand of that stage (``x{l}``), its fp32 conv output
(``y{l}``), its bf16 upstream gradient (``dx{l+1}``) and its bf16 ``dy{l}``, against the float64 stage reference of
oracle/discriminator_stages.py fed exactly those values (and the bf16-rounded weights the GEMMs read).  Errors are per
sample: max|got - ref| / max|ref| over that sample's slice, so a sample with small activations or gradients cannot hide
behind a large one.  Bounds:

* 1e-2 for bf16-stored tensors and conv outputs, 5e-3 for weight and bias gradients, exact for MaxPool, 1e-4 for the
  fp32 sigmoid output.
* LeakyReLU's derivative jumps at 0.  Where xhat is within rounding of 0 the fp32 kernel and a float64 reference may
  take different branches, and one such element moves its dy by 0.8 |dz|, a large fraction of the sample's max.  The
  backward reference therefore takes the branch the engine took, read off the sign of the engine's stored activation
  (z > 0 exactly when the kernel's xhat > 0); the forward checks hold the activation values themselves to 1e-2.

Batch-composition checks need no reference: every op of D is per sample except the parameter-gradient sums, so a
sample's forward and data gradient must not depend on what else is in the batch, bit for bit.

Run with ``-s`` to see the worst per-sample error of every checked quantity next to its bound.
"""
import pytest
import torch
import torch.nn.functional as F

from oracle import discriminator_stages as R
from oracle import srgan_oracle as O

pytestmark = pytest.mark.gpu

GEOMS = {"512x1024": (512, 1024), "684x684": (684, 684), "940x940": (940, 940), "428x700": (428, 700)}
# 512x1024: final map 1x3, the reference's native crop and the gan-native bench.  684x684: 2x2.  940x940: 3x3.
# 428x700: conv outputs odd at every stage (213x349, 53x87, 13x21, 3x5): ragged pooling and space-to-depth edges.
CASES = [(g, n) for g in GEOMS for n in (2, 3)] + [("512x1024", 24)]
KINDS = {2: ("noise", "flat"), 3: ("smooth", "lowcontrast", "flat")}
FOUR = ("noise", "smooth", "flat", "lowcontrast")
TOL, TOL_PARAM, TOL_SIGMOID = 1e-2, 5e-3, 1e-4
TOL_BIAS_SUM = 5e-4       # batch bias gradient vs the sum of single-sample ones, see test_batch_composition_is_bitwise

REPORT = {}


def record(case, what, errs, bound):
    worst = float(errs.max()) if torch.is_tensor(errs) else float(errs)
    key = (case, what)
    REPORT[key] = (max(worst, REPORT.get(key, (0.0,))[0]), bound)
    return worst


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    if REPORT:
        print("\nworst per-sample error (bound)")
        for (case, what), (worst, bound) in sorted(REPORT.items()):
            print(f"  {case:<14} {what:<22} {worst:.3e}  ({bound:.0e})")


@pytest.fixture(scope="module")
def S():
    import srgan_b200
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return srgan_b200


def per_sample(got, ref):
    """max|got - ref| / max|ref| over each sample's slice (dim 0)."""
    got, ref = got.double(), ref.double()
    d = (got - ref).abs().flatten(1).amax(1)
    return d / ref.abs().flatten(1).amax(1).clamp_min(1e-300)


def maxrel(got, ref):
    got, ref = got.double(), ref.double()
    return float((got - ref).abs().max() / ref.abs().max().clamp_min(1e-300))


def nchw(t):
    return t.permute(0, 3, 1, 2)


def image(kind, H, W, seed):
    """One 3 x H x W frame in [0, 1].  noise: uniform.  smooth: a slanted sinusoid per channel.  flat: a constant plus
    1e-3 Gaussian noise, the small-variance InstanceNorm case.  lowcontrast: a uniform-noise frame scaled into
    [0.45, 0.53]."""
    g = torch.Generator().manual_seed(seed)
    if kind == "noise":
        return torch.rand(3, H, W, generator=g)
    if kind == "smooth":
        f = 1.0 + 2.0 * torch.rand(3, 2, generator=g)
        ph = 6.28 * torch.rand(3, generator=g)
        yy = torch.linspace(0, 1, H)[:, None]
        xx = torch.linspace(0, 1, W)[None, :]
        return torch.stack([0.5 + 0.4 * torch.sin(6.28 * (f[c, 0] * yy + f[c, 1] * xx) + ph[c]) for c in range(3)])
    if kind == "flat":
        c = 0.2 + 0.6 * float(torch.rand(1, generator=g))
        return (c + 1e-3 * torch.randn(3, H, W, generator=g)).clamp(0, 1)
    if kind == "lowcontrast":
        return 0.45 + 0.08 * torch.rand(3, H, W, generator=g)
    raise ValueError(kind)


def batch(N, H, W, seed):
    kinds = KINDS.get(N) or tuple(FOUR[n % 4] for n in range(N))
    return torch.stack([image(k, H, W, seed * 1000 + n) for n, k in enumerate(kinds)]), kinds


def upstream(shape, seed):
    """Per-sample upstream gradient of D's output, with sample scales 1, 0.1, 0.01 repeating."""
    g = torch.Generator().manual_seed(seed)
    d = torch.randn(shape, generator=g) * 1e-2
    return d * torch.tensor([10.0 ** -(n % 3) for n in range(shape[0])])[:, None, None, None]


def make_d(S, seed=100):
    torch.manual_seed(seed)
    d = S.Discriminator()
    sd = {k: v.clone() for k, v in d.state_dict().items()}
    return d.cuda(), sd


def fwd_bwd(d, x, dout):
    """D(x) with autograd, then one backward of dout: (out, dx, {name: grad}), all cloned off the engine."""
    xg = x.clone().requires_grad_(True)
    params = list(d.parameters())
    names = [k for k, _ in d.named_parameters()]
    out = d(xg)
    g = torch.autograd.grad(out, [xg] + params, dout)
    return out.detach().clone(), g[0].clone(), {k: v.clone() for k, v in zip(names, g[1:])}


@pytest.fixture(scope="module", params=CASES, ids=[f"{g}-n{n}" for g, n in CASES])
def run(S, request):
    geom, N = request.param
    H, W = GEOMS[geom]
    d, sd = make_d(S)
    x, kinds = batch(N, H, W, seed=N)
    x = x.cuda()
    dout = upstream((N, 512) + O.discriminator_output_hw(H, W), seed=7 + N).cuda()
    out, dx, grads = fwd_bwd(d, x, dout)
    torch.cuda.synchronize()
    eng = d.last_engine()
    T = {k: eng.named_tensor(k).clone() for k in eng.tensor_table()}
    # each stage's operand as the NCHW map it stands for (bf16 values as float64), and the padding cells around it
    zin, pads = [R.bf16(x)], [None]
    for l in range(1, 4):
        hp, wp = T[f"p{l - 1}"].shape[1:3]
        z, pad = R.uns2d(T[f"x{l}"], hp, wp)
        zin.append(z.double())
        pads.append(pad)
    yield dict(case=f"{geom}-n{N}", sd=sd, x=x, kinds=kinds, out=out, dout=dout, dx=dx, grads=grads, T=T, zin=zin,
               pads=pads)
    del T
    torch.cuda.empty_cache()


def test_forward_stages_per_sample(run):
    """Per stage and sample: the stage-0 unfold bitwise, the conv output against the float64 conv of the engine's own
    operand, MaxPool exactly, InstanceNorm + activation against float64 from the engine's own conv output.  The stage
    output is also checked against the whole float64 stage (conv, pool, norm, activation) from the engine's operand:
    1e-2 for the bf16 stages.  For the sigmoid map that composed check's bound is 1e-3, not 1e-4: the fp32 conv
    accumulation (~1e-6 relative to |y3|, 4096-term dot products) passes through an InstanceNorm over 3 elements whose
    1/sqrt(var + eps) reaches 316, so it alone moves the output by up to 1.9e-4 (measured, 24 x 512x1024); the isolated
    check keeps 1e-4."""
    case, sd, T, zin = run["case"], run["sd"], run["T"], run["zin"]
    dev = run["x"].device
    s0 = T["x0"].shape
    assert torch.equal(T["x0"], R.unfold0(run["x"].to(torch.bfloat16), s0[1], s0[2])), "stage-0 unfold"
    for l in range(4):
        w, b = R.stage_params(sd, l, dev)
        ref = R.stage_forward(zin[l], w, b, l)
        y = nchw(T[f"y{l}"])
        assert y.shape == ref["y"].shape
        e = record(case, f"y{l} conv", per_sample(y, ref["y"]), TOL)
        assert e < TOL, (l, e)
        assert torch.equal(nchw(T[f"p{l}"]), F.max_pool2d(y, 3, 2)), l                       # MaxPool2d(3, 2): exact
        iso = R.post_forward(y.double(), l)
        if l < 3:
            got = zin[l + 1]
            assert bool((run["pads"][l + 1] == 0).all()), l                                     # padding cells hold 0
            e = record(case, f"x{l + 1} norm+act", per_sample(got, iso), TOL)
            assert e < TOL, (l, e)
            e = record(case, f"x{l + 1} whole stage", per_sample(got, ref["out"]), TOL)
            assert e < TOL, (l, e)
        else:
            e = record(case, "out norm+sigmoid", per_sample(run["out"], iso), TOL_SIGMOID)
            assert e < TOL_SIGMOID, e
            e = record(case, "out whole stage", per_sample(run["out"], ref["out"]), 1e-3)
            assert e < 1e-3, e
        if l == 0:
            # how small the InstanceNorm variances of the flat frames get (reported, not a bound)
            p = nchw(T["p0"]).double()
            var = p.var(dim=(2, 3), unbiased=False)
            for n, k in enumerate(run["kinds"]):
                if k == "flat":
                    REPORT[(case, "min var0/eps (flat)")] = (float(var[n].min()) / R.EPS, float("nan"))


def test_backward_stages_per_sample(run):
    """Per stage, from the engine's own upstream gradient: d(conv output) through MaxPool + InstanceNorm + activation
    per sample, the weight and bias gradients (summed over the batch, so not per sample), and the data gradient per
    sample -- the bf16 dx{l} for l > 0, the fp32 image gradient for l = 0."""
    case, sd, T, zin, G = run["case"], run["sd"], run["T"], run["zin"], run["grads"]
    dev = run["x"].device
    dz = run["dout"].double()
    for l in range(3, -1, -1):
        y = nchw(T[f"y{l}"])
        positive = zin[l + 1] > 0 if l < 3 else None
        dy_ref = R.post_backward(y, dz, l, positive)
        dy = nchw(T[f"dy{l}"])
        e = record(case, f"dy{l} pool+norm bwd", per_sample(dy, dy_ref), TOL)
        assert e < TOL, (l, e)
        w, _ = R.stage_params(sd, l, dev)
        dzin, dw, db = R.conv_backward(zin[l], w, dy.double(), l)
        e = record(case, f"dW{l}", maxrel(G[R.KEYS[l] + ".weight"], dw), TOL_PARAM)
        assert e < TOL_PARAM, (l, e)
        e = record(case, f"db{l}", maxrel(G[R.KEYS[l] + ".bias"], db), TOL_PARAM)
        assert e < TOL_PARAM, (l, e)
        if l > 0:
            hp, wp = T[f"p{l - 1}"].shape[1:3]
            got = R.uns2d(T[f"dx{l}"], hp, wp)[0]
            e = record(case, f"dx{l} data grad", per_sample(got, dzin), TOL)
            assert e < TOL, (l, e)
            dz = got.double()
        else:
            e = record(case, "dx image grad", per_sample(run["dx"], dzin), TOL)
            assert e < TOL, e


def check_param_sums(case, grads, gsum, weight_bound):
    """Batch parameter gradients against the float64 sum of the single-sample ones; every entry is recorded before
    any is asserted, so a failure still reports them all."""
    bound = {k: weight_bound if k.endswith("weight") else TOL_BIAS_SUM for k in grads}
    errs = {k: record(case, "sum " + k, maxrel(v, gsum[k]), bound[k]) for k, v in grads.items()}
    for k, e in errs.items():
        assert e < bound[k], (k, e)


@pytest.mark.parametrize("geom", ["428x700", "512x1024"])
def test_batch_composition_is_bitwise(S, geom):
    """D(cat[a, b, c])[i] equals D(sample i alone) bit for bit, forward and data gradient with the same upstream
    gradient, and so does every per-sample engine tensor of the backward (dy{l}, dx{l}); a permuted batch gives the
    permuted results.

    Parameter gradients are sums over the batch, so they are compared with the float64 sum of the single-sample ones.
    Weights: 1e-4.  The weight-gradient GEMM accumulates each CTA's share of pixel tiles in fp32 in tensor memory, so
    a batch result is not a reordering of the single-sample sums; each carries its own accumulation error against the
    exact sum.  Measured at stage 0 (the largest): 1.4e-5 here.  Biases: 5e-4.  A bias gradient is zero in exact
    arithmetic, since InstanceNorm removes any per-channel constant of its input, so what the kernels return is the
    sum of dY's bf16 rounding residues, a value far smaller than the terms summed.  Regrouping the fp32 additions of
    that sum moves it by up to 6.1e-5 of its max (measured over both geometries here and N = 24), not 1e-5."""
    H, W = GEOMS[geom]
    d, _ = make_d(S, seed=101)
    x = torch.stack([image(k, H, W, 500 + n) for n, k in enumerate(("smooth", "flat", "noise"))]).cuda()
    dout = upstream((3, 512) + O.discriminator_output_hw(H, W), seed=11).cuda()
    out, dx, grads = fwd_bwd(d, x, dout)

    def grads_of(eng):
        """every dy{l} and the part of every dx{l} that holds a gradient (the image gradient's operand for l = 0)"""
        t = {f"dy{l}": eng.named_tensor(f"dy{l}") for l in range(4)}
        t["dx0"] = eng.named_tensor("dx0")[..., :48]
        for l in range(1, 4):
            hp, wp = eng.named_tensor(f"p{l - 1}").shape[1:3]
            t[f"dx{l}"] = R.uns2d(eng.named_tensor(f"dx{l}"), hp, wp)[0]
        return t

    Tb = {k: v.clone() for k, v in grads_of(d.last_engine()).items()}
    gsum = {k: torch.zeros_like(v, dtype=torch.float64) for k, v in grads.items()}
    for i in range(3):
        o1, dx1, g1 = fwd_bwd(d, x[i:i + 1], dout[i:i + 1])
        assert torch.equal(out[i:i + 1], o1), i
        assert torch.equal(dx[i:i + 1], dx1), i
        for k, v in grads_of(d.last_engine()).items():
            assert torch.equal(Tb[k][i:i + 1], v), (i, k)
        for k, v in g1.items():
            gsum[k] += v.double()
    perm = [2, 0, 1]
    op, dxp, _ = fwd_bwd(d, x[perm], dout[perm])
    assert torch.equal(op, out[perm]) and torch.equal(dxp, dx[perm])
    check_param_sums(f"{geom}-n3", grads, gsum, 1e-4)


def test_param_grads_sum_over_samples_n24(S):
    """At the bench's D batch (24 x 512x1024), each sample's output and data gradient are bitwise its single-sample
    ones.  Parameter gradients are checked against the float64 sum of 24 single-sample gradients.  Here the
    weight-gradient GEMM accumulates 166 pixel tiles per CTA at stage 0, against 7 for a single sample.  The four flat
    frames with weight 1 or 0.1 add terms c * dY that cancel only across all CTAs, since InstanceNorm makes
    sum(dY) = 0.  Measured at stage 0: 5.1e-4 between batch and sum, and 5.4e-4 between the batch and float64 in the
    per-stage test, whose bound is 5e-3; both moved by half between builds whose forward differs in the last bits.
    So weights: 2e-3.  Biases: 5e-4, as in test_batch_composition_is_bitwise."""
    d, _ = make_d(S, seed=102)
    x, _ = batch(24, 512, 1024, seed=24)
    x = x.cuda()
    dout = upstream((24, 512, 1, 3), seed=12).cuda()
    out, dx, grads = fwd_bwd(d, x, dout)
    gsum = {k: torch.zeros_like(v, dtype=torch.float64) for k, v in grads.items()}
    for i in range(24):
        o1, dx1, g1 = fwd_bwd(d, x[i:i + 1], dout[i:i + 1])
        assert torch.equal(out[i:i + 1], o1) and torch.equal(dx[i:i + 1], dx1), i
        for k, v in g1.items():
            gsum[k] += v.double()
    check_param_sums("512x1024-n24", grads, gsum, 2e-3)


@pytest.mark.parametrize("N", [3, 24])
def test_input_grad_only_equals_full_backward(S, N):
    d, _ = make_d(S, seed=103)
    x, _ = batch(N, 512, 1024, seed=30 + N)
    x = x.cuda()
    dout = upstream((N, 512, 1, 3), seed=13).cuda()
    _, dx_full, _ = fwd_bwd(d, x, dout)
    xg = x.clone().requires_grad_(True)
    with d.input_grad_only():
        out = d(xg)
    out.backward(dout)
    assert torch.equal(xg.grad, dx_full)
    assert all(p.grad is None for p in d.parameters())


def test_engine_reuse_across_batch_sizes(S):
    """One module alternating N = 1, 3, 24, 3, 1 (engines pooled per (N, H, W, training)) gives, every call, what a
    fresh module gives for the same call, bit for bit: output, data gradient and every parameter gradient."""
    d, _ = make_d(S, seed=104)
    x, _ = batch(24, 512, 1024, seed=40)
    x = x.cuda()
    dout = upstream((24, 512, 1, 3), seed=14).cuda()
    for N in (1, 3, 24, 3, 1):
        got = fwd_bwd(d, x[:N], dout[:N])
        fresh, _ = make_d(S, seed=104)
        want = fwd_bwd(fresh, x[:N], dout[:N])
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), N
        for k in want[2]:
            assert torch.equal(got[2][k], want[2][k]), (N, k)
        with torch.no_grad():
            assert torch.equal(d(x[:N]), want[0]), N
