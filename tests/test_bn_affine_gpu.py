"""GPU tests of every generator path that consumes BatchNorm gamma / beta / running statistics, with a trained-like state
(tests/bn_affine_state.py: distinct gamma with negative entries, beta, running statistics per layer, channel and
generator) instead of gamma = 1 / beta = 0.  Each check compares a kernel result with F.conv2d / F.batch_norm / autograd
on the CPU fed the engine's own bf16 inputs for that layer (float64 at small sizes, fp32 at cfg2 sizes, where fp32 error
is ~1e-6), with the bounds of tests/test_generator_gpu.py; tests/test_bn_affine_cpu.py shows those bounds see every bug
class a default-initialised state hides."""
import os
import sys

import pytest
import torch
import torch.nn.functional as F

from oracle import srgan_oracle as O

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import bn_affine_state as B  # noqa: E402  (tests/bn_affine_state.py)

pytestmark = pytest.mark.gpu


def nchw(t):  # engine NHWC bf16 -> NCHW fp32 on the CPU
    return t.float().permute(0, 3, 1, 2).contiguous().cpu()


@pytest.fixture(scope="module")
def S():
    import srgan_b200
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return srgan_b200


class Bad(list):
    """collects every check that misses its bound, so that one run reports all of them"""

    def le(self, what, err, bound):
        if not err <= bound:
            self.append((what, err, bound))


def _module(S, sd, **kw):
    g = S.SRResNet(**kw)
    g.load_state_dict(sd)
    return g.cuda()


def _state(seed, k=0, **kw):
    return B.bn_affine_state(O.init_srresnet_state(seed, **kw), seed, k)


def _trunk_names(n_res):
    names = ["out1", "d_last"]
    for b in range(n_res):
        names += [f"rb{b}.{n}" for n in ("y1", "z1", "y2", "out", "d_y2", "d_pre1", "d_y1", "d_in")]
    return names


def check_trunk(bad, tag, T, G, sd, after, blocks, n_res, dt):
    """Per residual block, each step fed the engine's own tensors: forward y1, z1, y2, out; the running statistics after
    the forward against the update formula on the engine's y from the loaded statistics; backward d_y2, d_pre1, d_y1,
    d_in; the BatchNorm parameter gradients; the zero bias gradient of the BatchNorm-preceded convs."""
    for b in blocks:
        p = f"residual_blocks.{b}"
        t = {n: T[f"rb{b}.{n}"].to(dt) for n in ("y1", "z1", "y2", "out", "d_y2", "d_pre1", "d_y1", "d_in")}
        x = (T["out1"] if b == 0 else T[f"rb{b - 1}.out"]).to(dt)
        dout = (T["d_last"] if b == n_res - 1 else T[f"rb{b + 1}.d_in"]).to(dt)
        g1, be1, g2, be2 = (sd[f"{p}.bn{j}.{n}"] for j in (1, 2) for n in ("weight", "bias"))
        bad.le(f"{tag} {p} y1", B.maxrel(t["y1"], B.conv3(x, sd, p + ".conv1")), B.TOL_LAYER)
        bad.le(f"{tag} {p} z1", B.maxrel(t["z1"], F.relu(B.bn_train(t["y1"], g1, be1))), B.TOL_LAYER)
        bad.le(f"{tag} {p} y2", B.maxrel(t["y2"], B.conv3(t["z1"], sd, p + ".conv2")), B.TOL_LAYER)
        bad.le(f"{tag} {p} out", B.maxrel(t["out"], B.bn_train(t["y2"], g2, be2) + x), B.TOL_LAYER)
        for j, y in ((1, t["y1"]), (2, t["y2"])):
            q = f"{p}.bn{j}"
            rm, rv = B.running_update(sd[q + ".running_mean"], sd[q + ".running_var"], y)
            bad.le(f"{tag} {q} running_mean", B.maxrel(after[q + ".running_mean"], rm), B.TOL_RUNNING)
            bad.le(f"{tag} {q} running_var", B.maxrel(after[q + ".running_var"], rv), B.TOL_RUNNING)
        dy2, dg, dbe = B.bn_train_bwd(t["y2"], g2, be2, dout)
        bad.le(f"{tag} {p} d_y2", B.maxrel(t["d_y2"], dy2), B.TOL_LAYER)
        bad.le(f"{tag} {p} bn2.weight grad", B.maxrel(G[p + ".bn2.weight"], dg), B.TOL_WGRAD)
        bad.le(f"{tag} {p} bn2.bias grad", B.maxrel(G[p + ".bn2.bias"], dbe), B.TOL_WGRAD)
        bad.le(f"{tag} {p} conv2.bias grad", float(G[p + ".conv2.bias"].abs().max()), 0.0)
        dp1 = B.conv3_dgrad(t["z1"], sd, p + ".conv2", t["d_y2"]) * (t["z1"] > 0)
        bad.le(f"{tag} {p} d_pre1", B.maxrel(t["d_pre1"], dp1), B.TOL_LAYER)
        dy1, dg, dbe = B.bn_train_bwd(t["y1"], g1, be1, t["d_pre1"])
        bad.le(f"{tag} {p} d_y1", B.maxrel(t["d_y1"], dy1), B.TOL_LAYER)
        bad.le(f"{tag} {p} bn1.weight grad", B.maxrel(G[p + ".bn1.weight"], dg), B.TOL_WGRAD)
        bad.le(f"{tag} {p} bn1.bias grad", B.maxrel(G[p + ".bn1.bias"], dbe), B.TOL_WGRAD)
        bad.le(f"{tag} {p} conv1.bias grad", float(G[p + ".conv1.bias"].abs().max()), 0.0)
        d_in = B.conv3_dgrad(x, sd, p + ".conv1", t["d_y1"]) + dout
        bad.le(f"{tag} {p} d_in", B.maxrel(t["d_in"], d_in), B.TOL_LAYER)


def _cpu_state(g):
    return {k: v.detach().cpu().clone() for k, v in g.state_dict().items()}


def _grads(g):
    return {k: p.grad.detach().cpu().clone() for k, p in g.named_parameters()}


# ------------------------------------------------------------------------------------------------ a. training, per layer
TRAIN_MODES = [pytest.param(0, id="per-layer"), pytest.param(1, id="fused-trunk")]


def _train_run(S, sd, x, dsr, trunk_mode, names):
    L = S.lib()
    old = L.srg_set_trunk_fused(trunk_mode)
    try:
        g = _module(S, sd).train()
        g.debug_keep_grads = True
        y = g(x.cuda())
        y.backward(dsr.cuda())
        torch.cuda.synchronize()
        eng = g.last_engine()
        assert L.srg_generator_trunk_layers(eng.handle) == (33 if trunk_mode else 1)
        assert L.srg_generator_trunk_error(eng.handle) == 0
        T = {n: nchw(eng.named_tensor(n)) for n in names}
        return T, _grads(g), _cpu_state(g)
    finally:
        L.srg_set_trunk_fused(old)


@pytest.mark.parametrize("trunk_mode", TRAIN_MODES)
def test_training_per_layer_all_blocks(S, trunk_mode):
    """2x3x16x24, all 16 blocks, float64 references"""
    sd = _state(31)
    gen = torch.Generator().manual_seed(32)
    x, dsr = torch.rand(2, 3, 16, 24, generator=gen), torch.randn(2, 3, 64, 96, generator=gen) * 1e-3
    T, G, after = _train_run(S, sd, x, dsr, trunk_mode, _trunk_names(16))
    bad = Bad()
    check_trunk(bad, "", T, G, B.to_double(sd), after, range(16), 16, torch.float64)
    assert not bad, bad


@pytest.mark.parametrize("trunk_mode", TRAIN_MODES)
def test_training_per_layer_cfg2(S, trunk_mode):
    """16x3x96x96 (BASELINE configs[1]): blocks 0, 7 and 15, the layers test_full_size_layers_against_fp32_oracle_cfg2
    walks, fp32 references"""
    sd = _state(33)
    gen = torch.Generator().manual_seed(34)
    x, dsr = torch.rand(16, 3, 96, 96, generator=gen), torch.randn(16, 3, 384, 384, generator=gen) * 1e-4
    names = ["out1", "d_last", "rb1.d_in", "rb6.out", "rb8.d_in", "rb14.out"] + \
        [f"rb{b}.{n}" for b in (0, 7, 15) for n in ("y1", "z1", "y2", "out", "d_y2", "d_pre1", "d_y1", "d_in")]
    T, G, after = _train_run(S, sd, x, dsr, trunk_mode, names)
    bad = Bad()
    check_trunk(bad, "", T, G, sd, after, (0, 7, 15), 16, torch.float32)
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ b. multi-generator trunks
@pytest.mark.parametrize("trunk_mode", [pytest.param(0, id="grouped"), pytest.param(1, id="fused-multi")])
@pytest.mark.parametrize("n_res", [2, 16])
@pytest.mark.parametrize("K", [2, 3, 4])
def test_multi_generator_trunk_per_generator(S, K, n_res, trunk_mode):
    """joint_pixel_generator_steps with K generators, each with its own conv weights and BatchNorm state: every
    generator's trunk intermediates, BatchNorm parameter gradients and running statistics against its own state, and
    against generator 0's BatchNorm state they differ by 10x the bound (a generator handed generator 0's parameters fails)."""
    L = S.lib()
    sds = [_state(40 + k, k, num_residuals=n_res) for k in range(K)]
    gens = []
    for sd in sds:
        g = _module(S, sd, num_residuals=n_res)
        g.debug_keep_grads = True
        gens.append(g)
    opts = [S.Adam(g.parameters(), lr=1e-4) for g in gens]
    gen = torch.Generator().manual_seed(50)
    lr, hr = torch.rand(2, 3, 40, 24, generator=gen).cuda(), torch.rand(2, 3, 160, 96, generator=gen).cuda()
    streams = [torch.cuda.Stream() for _ in range(K)]
    old = L.srg_set_trunk_fused(trunk_mode)
    try:
        S.joint_pixel_generator_steps(gens, S.ReconstructionLoss(), opts, lr, hr, streams)
        torch.cuda.synchronize()
    finally:
        L.srg_set_trunk_fused(old)
    names = _trunk_names(n_res)
    bad = Bad()
    apart = []
    for k, g in enumerate(gens):
        eng = g.last_engine()
        if trunk_mode:
            assert L.srg_generator_trunk_layers(eng.handle) == 2 * n_res + 1
            assert L.srg_generator_trunk_error(eng.handle) == 0
        T = {n: nchw(eng.named_tensor(n)) for n in names}
        after = _cpu_state(g)                               # running statistics; the parameters were moved by Adam
        check_trunk(bad, f"gen{k}", T, _grads(g), B.to_double(sds[k]), after, range(n_res), n_res, torch.float64)
        if k == 0:
            continue
        s0, sk = B.to_double(sds[0]), B.to_double(sds[k])
        y1 = T["rb0.y1"].double()
        p = "residual_blocks.0.bn1"
        z0 = F.relu(B.bn_train(y1, s0[p + ".weight"], s0[p + ".bias"]))
        dy0 = B.bn_train_bwd(y1, s0[p + ".weight"], s0[p + ".bias"], T["rb0.d_pre1"].double())[0]
        rm0 = B.running_update(s0[p + ".running_mean"], s0[p + ".running_var"], y1)[0]
        apart.append((k, B.maxrel(T["rb0.z1"], z0), B.maxrel(T["rb0.d_y1"], dy0), B.maxrel(after[p + ".running_mean"], rm0)))
        assert sk[p + ".weight"].ne(s0[p + ".weight"]).all()
    assert not bad, bad
    for k, dz, ddy, drm in apart:
        assert dz >= 10 * B.TOL_LAYER and ddy >= 10 * B.TOL_LAYER and drm >= 10 * B.TOL_RUNNING, (k, dz, ddy, drm)


# ------------------------------------------------------------------------------------------------ c. SyncBatchNorm peer finalize
@pytest.mark.parametrize("trunk_mode", [0, 1])
def test_peer_sync_world1_matches_local_finalize(S, trunk_mode):
    """the fused reduce + exchange + finalize kernel (csrc/peer_sync.cu) with one rank, trained-like state: output,
    every gradient and the running statistics bit-identical to the local finalize"""
    import ctypes
    from ctypes import c_void_p
    L = S.lib()
    ps = c_void_p()
    S._lib.check(L.srg_peer_sync_create(ctypes.byref(ps), 1, 0))
    buf = ctypes.create_string_buffer(64)
    S._lib.check(L.srg_peer_sync_handle(ps, buf))
    S._lib.check(L.srg_peer_sync_connect(ps, buf.raw))
    sd = _state(52, num_residuals=2)
    gen = torch.Generator().manual_seed(51)
    lr = torch.rand(2, 3, 20, 12, generator=gen).cuda()
    dsr = (torch.randn(2, 3, 80, 48, generator=gen) * 1e-3).cuda()
    outs = []
    old = L.srg_set_trunk_fused(trunk_mode)
    try:
        for use_peer in (False, True):
            g = _module(S, sd, num_residuals=2).train()
            if use_peer:
                g.enable_sync_batchnorm(world=1, peer_sync=ps)
            y = g(lr)
            y.backward(dsr)
            torch.cuda.synchronize()
            outs.append((y.detach().clone(), g.flat_grads().clone(),
                         torch.cat([v.flatten().float() for k, v in g.state_dict().items() if "running" in k])))
    finally:
        L.srg_set_trunk_fused(old)
    assert L.srg_peer_sync_error(ps) == 0
    L.srg_peer_sync_destroy(ps)
    for a, b in zip(outs[0], outs[1]):
        assert torch.equal(a, b)


# ------------------------------------------------------------------------------------------------ d. eval forward (folded BN)
def _eval_trunk(sd, out1):
    """the eval-mode trunk (residual blocks with running statistics, conv2, global skip) from a given out1"""
    out = out1
    for b in range(B.num_blocks(sd)):
        p = f"residual_blocks.{b}"
        y = F.relu(F.batch_norm(B.conv3(out, sd, p + ".conv1"), sd[p + ".bn1.running_mean"], sd[p + ".bn1.running_var"],
                                sd[p + ".bn1.weight"], sd[p + ".bn1.bias"], training=False, eps=B.EPS))
        out = F.batch_norm(B.conv3(y, sd, p + ".conv2"), sd[p + ".bn2.running_mean"], sd[p + ".bn2.running_var"],
                           sd[p + ".bn2.weight"], sd[p + ".bn2.bias"], training=False, eps=B.EPS) + out
    return B.conv3(out, sd, "conv2") + out1


EVAL_CASES = [
    # (num_residuals, upscale_factor, input shape); 1x3x256x320 = 320 trunk tiles of 32x8, more than two per CTA
    pytest.param(1, 4, (2, 3, 16, 24), id="1-block"),
    pytest.param(2, 4, (2, 3, 16, 24), id="2-blocks"),
    pytest.param(1, 4, (1, 3, 256, 320), id="1-block-256x320"),
    pytest.param(2, 4, (1, 3, 256, 320), id="2-blocks-256x320"),
    pytest.param(2, 2, (2, 3, 16, 24), id="x2"),
    pytest.param(1, 8, (2, 3, 16, 24), id="x8"),
    pytest.param(16, 4, (4, 3, 64, 64), id="16-blocks"),
]


@pytest.mark.parametrize("n_res,upscale,shape", EVAL_CASES)
def test_eval_forward_against_oracle(S, n_res, upscale, shape):
    """The eval forward (BatchNorm folded into the conv epilogue, bn_eval_coeffs_all_kernel) for conv variants 0 and 1.  End to
    end against O.srresnet_forward(training=False) with the calibrated bounds of bn_affine_state; for 1-2 blocks also
    each stored segment at TOL_LAYER, fed the engine's own input: the folded trunk from out1, every up-sampling stage, the
    output conv."""
    deep = n_res == 16
    if deep:
        sd, x = B.deep_eval_case()
        tol, floor = B.TOL_EVAL_DEEP, B.PSNR_EVAL_DEEP
    else:
        sd = _state(60 + n_res, num_residuals=n_res, upscale_factor=upscale)
        x = torch.rand(*shape, generator=torch.Generator().manual_seed(61))
        tol, floor = B.TOL_EVAL_SHALLOW, B.PSNR_EVAL_SHALLOW
    small = x.numel() <= 4096 and upscale <= 4          # float64 where cheap; fp32 (error ~1e-6) elsewhere
    dt = torch.float64 if small else torch.float32
    ref_sd = B.to_double(sd) if small else sd
    ref = O.srresnet_forward(ref_sd, x.to(dt), training=False)
    g = _module(S, sd, num_residuals=n_res, upscale_factor=upscale).eval()
    L = S.lib()
    bad = Bad()
    figures = []
    for variant in range(2):
        old = L.srg_set_conv_variant(variant)
        try:
            with torch.no_grad():
                y = g(x.cuda()).cpu()
            torch.cuda.synchronize()
            eng = g.last_engine()
            T = {n: nchw(eng.named_tensor(n)).to(dt) for n in ["out1", "trunk"] + [f"up{j}" for j in range(g.num_upsample_stages)]}
        finally:
            L.srg_set_conv_variant(old)
        err, db = B.maxrel(y, ref), B.psnr_rel(y, ref)
        figures.append((variant, err, db))
        bad.le(f"v{variant} end to end", err, tol)
        bad.le(f"v{variant} -PSNR", -db, -floor)
        if not deep:
            bad.le(f"v{variant} trunk", B.maxrel(T["trunk"], _eval_trunk(ref_sd, T["out1"])), B.TOL_LAYER)
        prev = T["trunk"]
        for j, i in enumerate(O.upsample_stage_indices(ref_sd)):
            up = F.relu(F.pixel_shuffle(F.conv2d(prev, ref_sd[f"upsample.{i}.weight"], ref_sd[f"upsample.{i}.bias"], padding=1), 2))
            bad.le(f"v{variant} up{j}", B.maxrel(T[f"up{j}"], up), B.TOL_LAYER)
            prev = T[f"up{j}"]
        bad.le(f"v{variant} conv3", B.maxrel(y, F.conv2d(prev, ref_sd["conv3.weight"], ref_sd["conv3.bias"], padding=4)), B.TOL_LAYER)
    print("eval", n_res, upscale, shape, [(v, f"{e:.3e}", f"{d:.1f} dB") for v, e, d in figures])
    assert not bad, bad


# ------------------------------------------------------------------------------------------------ e. frozen eval autograd
@pytest.fixture(scope="module")
def frozen_run(S):
    """eval-mode forward + backward with x.requires_grad (frozen BatchNorm), every inter-layer gradient kept"""
    sd = _state(70)
    g = _module(S, sd).eval()
    g.debug_keep_grads = True
    gen = torch.Generator().manual_seed(71)
    lr = torch.rand(2, 3, 16, 24, generator=gen)
    dsr = torch.randn(2, 3, 64, 96, generator=gen) * 1e-3
    x = lr.cuda().requires_grad_()
    y = g(x)
    y.backward(dsr.cuda())
    torch.cuda.synchronize()
    eng = g.last_engine()
    assert eng.frozen
    T = {name: nchw(eng.named_tensor(name)) for name in eng.tensor_table()}
    return dict(g=g, sd=sd, lr=lr, dsr=dsr, x=x, T=T, grads=_grads(g), after=_cpu_state(g))


def test_frozen_batchnorm_backward_per_layer(frozen_run):
    """d y = gamma * inv * d z, dgamma, dbeta and the conv-bias gradient sum(d y) (RF_BN_BWD_FROZEN) per block against
    F.batch_norm(training=False) autograd in float64, fed the engine's tensors; the buffers stay as loaded"""
    r = frozen_run
    sd, T, G = B.to_double(r["sd"]), r["T"], r["grads"]
    bad = Bad()
    dout = T["d_last"]
    for b in range(15, -1, -1):
        p = f"residual_blocks.{b}"
        for j, y, dz, dyk in ((2, f"rb{b}.y2", dout, f"rb{b}.d_y2"), (1, f"rb{b}.y1", T[f"rb{b}.d_pre1"], f"rb{b}.d_y1")):
            dy, dg, dbe = B.bn_eval_bwd(T[y].double(), sd, f"{p}.bn{j}", dz.double())
            bad.le(f"{p} d_y{j}", B.maxrel(T[dyk], dy), B.TOL_LAYER)
            bad.le(f"{p} bn{j}.weight grad", B.maxrel(G[f"{p}.bn{j}.weight"], dg), B.TOL_WGRAD)
            bad.le(f"{p} bn{j}.bias grad", B.maxrel(G[f"{p}.bn{j}.bias"], dbe), B.TOL_WGRAD)
            bad.le(f"{p} conv{j}.bias grad", B.maxrel(G[f"{p}.conv{j}.bias"], dy.sum((0, 2, 3))), B.TOL_WGRAD)
        dout = T[f"rb{b}.d_in"]
    assert not bad, bad
    for k, v in r["sd"].items():
        if not k.endswith((".weight", ".bias")):
            assert torch.equal(v, r["after"][k]), k


def test_frozen_gradients_end_to_end_match_oracle_eval_autograd(frozen_run):
    r = frozen_run
    work = O._with_grad(r["sd"])
    xr = r["lr"].clone().requires_grad_()
    yr = O.srresnet_forward(work, xr, training=False)
    keys = O.trainable_keys(work)
    ref = torch.autograd.grad(yr, [xr] + [work[k] for k in keys], grad_outputs=r["dsr"])
    bad = []
    for name, got, want in [("x", r["x"].grad, ref[0])] + [(k, r["grads"][k], v) for k, v in zip(keys, ref[1:])]:
        got, want = got.double().cpu().flatten(), want.double().flatten()
        cos, ratio = float(torch.dot(got, want) / (got.norm() * want.norm())), float(got.norm() / want.norm())
        if not (cos > 0.95 and 0.9 < ratio < 1.1):
            bad.append((name, cos, ratio))
    assert not bad, bad


@pytest.mark.parametrize("mode", ["frozen", "train-fused", "train-per-layer"])
def test_input_only_backward_is_bit_identical(S, mode):
    """every parameter frozen: x.grad bitwise equal to the full backward's, with the trained-like state"""
    import copy
    L = S.lib()
    old = L.srg_set_trunk_fused(0 if mode == "train-per-layer" else 2)
    try:
        base = S.SRResNet()
        base.load_state_dict(_state(72))
        full, only = copy.deepcopy(base).cuda(), copy.deepcopy(base).cuda()
        only.requires_grad_(False)
        gen = torch.Generator().manual_seed(73)
        lr = torch.rand(2, 3, 16, 24, generator=gen).cuda()
        dsr = (torch.randn(2, 3, 64, 96, generator=gen) * 1e-3).cuda()
        xs = []
        for g in (full, only):
            g.train(mode != "frozen")
            x = lr.clone().requires_grad_()
            g(x).backward(dsr)
            torch.cuda.synchronize()
            xs.append(x.grad)
    finally:
        L.srg_set_trunk_fused(old)
    assert torch.equal(xs[0], xs[1])
    assert all(p.grad is None for p in only.parameters())


# ------------------------------------------------------------------------------------------------ f. tiled and streamed eval
def test_tiled_and_streamed_eval_against_oracle(S):
    """The 2-blocks case of test_tiling_gpu (2x3x203x317, windows sized for a 110x150 workspace): the tiled output against
    the fp32 oracle (bounds of d) and bitwise equal to the whole frame; a chunk-streamed call bitwise equal to the unchunked."""
    sd = _state(80, num_residuals=2)
    x = torch.rand(2, 3, 203, 317, generator=torch.Generator().manual_seed(81))
    g = _module(S, sd, num_residuals=2).eval()
    xc = x.cuda()
    g.tile_budget_bytes, g.stream_budget_bytes = None, None
    with torch.no_grad():
        full = g(xc).clone()
        g.tile_budget_bytes = g._eval_ws_bytes(110, 150, xc.device)
        tiled = g(xc).clone()
        win_h, win_w, _, tiles = g._rt[("tiles", 2, 203, 317, g.tile_budget_bytes)]
        assert len(tiles) > 2 and (win_h < 203 or win_w < 317)
        g.tile_budget_bytes = None
        g.stream_budget_bytes = int(g._eval_ws_bytes(203, 317, xc.device) * 1.5)     # one frame per chunk
        streamed = g(xc).clone()
        assert g.last_engine().N == 1
    g.stream_budget_bytes = 6 << 30
    torch.cuda.synchronize()
    assert torch.equal(tiled, full)
    assert torch.equal(streamed, full)
    ref = O.srresnet_forward(sd, x, training=False)
    err, db = B.maxrel(tiled, ref), B.psnr_rel(tiled, ref)
    print("tiled", f"{err:.3e}", f"{db:.1f} dB")
    assert err <= B.TOL_EVAL_SHALLOW and db >= B.PSNR_EVAL_SHALLOW, (err, db)
