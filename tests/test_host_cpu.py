"""CPU-only tests: the C-ABI library loads and exports every symbol include/srgan_b200.h declares (no compute calls),
the engine's parameter table equals the reference's state_dict layout, and the nn.Module surface keeps the reference's
constructor / init / key conventions."""
import ctypes
import os
import re

import pytest
import torch

import srgan_b200 as S
from oracle import srgan_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "srgan_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(srg_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"srg_allreduce_f64_fn"}
    assert len(declared) >= 30
    S.build()
    lib = ctypes.CDLL(S._lib.SO_PATH)
    missing = [n for n in sorted(declared) if not hasattr(lib, n)]
    assert not missing, missing
    # the ctypes table binds exactly the declared set
    assert set(S._lib.EXPORTS) == declared, set(S._lib.EXPORTS) ^ declared
    assert S.lib().srg_abi_version() == 1


def test_engine_parameter_table_matches_reference_state_dict():
    torch.manual_seed(0)
    g = S.SRResNet()
    eng = S.models._GeneratorEngine(2, 16, 24, 16, 2, True, torch.device("cpu"))   # create() needs no device
    table = eng.param_table()
    named = list(g.named_parameters())
    assert [t[0] for t in table] == [k for k, _ in named]
    assert [t[3] for t in table] == [tuple(p.shape) for _, p in named]
    assert sum(t[2] for t in table) == 1549315                       # SURVEY Appendix A
    offs = [t[1] for t in table]
    assert offs == sorted(offs) and all(o % 4 == 0 for o in offs)     # 16-byte aligned slots
    bufs = eng.buffer_table()
    assert len(bufs) == 64 and sum(b[2] for b in bufs) == 4096
    assert bufs[0][0] == "residual_blocks.0.bn1.running_mean" and bufs[1][0] == "residual_blocks.0.bn1.running_var"
    assert eng.param_elems >= 1549315


def test_module_init_and_keys_equal_oracle_restated_reference():
    for seed, kw in [(1, {}), (5, dict(num_residuals=2, upscale_factor=2))]:
        torch.manual_seed(seed)
        g = S.SRResNet(**kw)
        sd = g.state_dict()
        ref = O.init_srresnet_state(seed, **kw)
        assert list(sd.keys()) == list(ref.keys())
        for k in sd:
            assert torch.equal(sd[k].float(), ref[k].float()), k


def test_upscale_factor_quirk_and_unsupported_widths():
    assert S.SRResNet(upscale_factor=2).num_upsample_stages == 1
    assert S.SRResNet(upscale_factor=3).num_upsample_stages == 1
    assert S.SRResNet(upscale_factor=4).num_upsample_stages == 2
    assert S.SRResNet(upscale_factor=8, num_residuals=1).num_upsample_stages == 4
    with pytest.raises(NotImplementedError):
        S.SRResNet(in_channels=1)


def test_no_cpu_fallback():
    g = S.SRResNet(num_residuals=1)
    with pytest.raises(RuntimeError):
        g(torch.rand(1, 3, 8, 8))
    with pytest.raises(RuntimeError):
        g.conv1(torch.rand(1, 3, 8, 8))            # holders never compute
    with pytest.raises(RuntimeError):
        S.ReconstructionLoss()(torch.rand(1, 3, 8, 8), torch.rand(1, 3, 8, 8))


def test_state_dict_roundtrip_with_ddp_prefix():
    """Checkpoints written by the reference carry DDP's "module." prefix (src/train.py:123-125); evaluation strips it
    (src/evaluation.py:26-29).  Same convention works here."""
    torch.manual_seed(2)
    a = S.SRResNet(num_residuals=2)
    ck = {"module." + k: v.clone() for k, v in a.state_dict().items()}
    b = S.SRResNet(num_residuals=2)
    b.load_state_dict({k.replace("module.", "", 1): v for k, v in ck.items()})
    for (k1, v1), (k2, v2) in zip(a.state_dict().items(), b.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)


def test_discriminator_engine_tables_and_size_rule():
    torch.manual_seed(3)
    d = S.Discriminator()
    ref = O.init_discriminator_state(3)
    assert list(d.state_dict().keys()) == list(ref.keys())
    for k in ref:
        assert torch.equal(d.state_dict()[k], ref[k]), k
    eng = S.models._DiscriminatorEngine(2, 512, 1024, True, torch.device("cpu"))     # create() needs no device
    assert eng.out_hw == O.discriminator_output_hw(512, 1024) == (1, 3)
    table = eng.param_table()
    assert [t[0] for t in table] == [k for k, _ in d.named_parameters()]
    assert sum(t[2] for t in table) == 2765760                                        # SURVEY Appendix A
    for hw in ((684, 684), (428, 684), (940, 940), (512, 1024)):
        assert S.models._DiscriminatorEngine(1, hw[0], hw[1], False, torch.device("cpu")).out_hw == O.discriminator_output_hw(*hw)
    for bad in ((384, 384), (512, 512), (256, 256), (427, 1024)):
        with pytest.raises(RuntimeError):
            S.models._DiscriminatorEngine(1, bad[0], bad[1], False, torch.device("cpu"))
        with pytest.raises(RuntimeError):
            O.discriminator_output_hw(*bad)


def test_reference_checkpoint_interop(tmp_path):
    """f-1: files written like the reference's training run (DDP 'module.' prefix, src/train.py:123-125) load into the
    modules, with or without the prefix (src/evaluation.py:24-31); the resume protocol divides both LRs by 5."""
    torch.manual_seed(8)
    g = S.SRResNet(num_residuals=2)
    d = S.Discriminator()
    gp, dp = str(tmp_path / "Training_generator_model_0.pth"), str(tmp_path / "Training_discriminator_model_0.pth")
    S.save_reference_checkpoint(g, gp)
    S.save_reference_checkpoint(d, dp, ddp_prefix=False)
    assert all(k.startswith("module.") for k in torch.load(gp, weights_only=True))
    g2, d2 = S.SRResNet(num_residuals=2), S.Discriminator()
    S.load_reference_checkpoint(g2, gp)
    S.load_reference_checkpoint(d2, dp)
    for a, b in zip(g.state_dict().values(), g2.state_dict().values()):
        assert torch.equal(a, b)
    for a, b in zip(d.state_dict().values(), d2.state_dict().values()):
        assert torch.equal(a, b)
    assert S.resume_learning_rates(1e-4, 5e-5) == (2e-5, 1e-5)


def test_batched_weight_gradient_plan_covers_every_layer_tile_once():
    """Host arithmetic behind wgrad3_batched_kernel / wgrad_reduce_batched_kernel (srg_wgrad_batched_plan, no device work):
    the contiguous per-CTA ranges cover every (layer, tile) exactly once, every (layer, slot) partial set has exactly
    one writer, slots stay below max_slots, and the slots the reduce kernel sums for a layer (first .. last CTA touching
    it) are exactly the slots that get written."""
    L = S.lib()
    for (n, h, w, layers) in [(16, 96, 96, 33), (2, 40, 20, 3), (1, 9, 5, 1), (4, 96, 48, 5), (32, 128, 128, 33), (3, 33, 17, 7),
                              (1, 16, 8, 33)]:
        t, g, per, ms = (ctypes.c_int() for _ in range(4))
        assert L.srg_wgrad_batched_plan(n, h, w, layers, ctypes.byref(t), ctypes.byref(g), ctypes.byref(per), ctypes.byref(ms)) == 0
        T, G, P, M = t.value, g.value, per.value, ms.value
        assert T == n * ((h + 15) // 16) * ((w + 7) // 8)
        total = T * layers
        assert G >= 1 and (G - 1) * P < total <= G * P              # no empty CTA, everything covered
        writers = {}
        covered = 0
        for c in range(G):
            lo, hi = c * P, min((c + 1) * P, total)
            covered += hi - lo
            for layer in range(lo // T, (hi - 1) // T + 1):
                slot = c - (layer * T) // P
                assert 0 <= slot < M, (n, h, w, layers, c, layer, slot, M)
                assert (layer, slot) not in writers
                writers[(layer, slot)] = c
        assert covered == total
        for layer in range(layers):
            c_first, c_last = (layer * T) // P, ((layer + 1) * T - 1) // P
            assert {s_ for (l_, s_) in writers if l_ == layer} == set(range(c_last - c_first + 1)), (n, h, w, layers, layer)


def test_conv9_rows_schedule_applies_every_row_tap_once_per_output_row():
    """The conv9_rows schedule the kernel evaluates (srg_conv9_rows_window is the same inline function): over the 16
    input rows of a tile every output row (block) 0..7 receives each of the 9 row taps exactly once, from the input row
    the convolution prescribes (h_out + kh - 4), through the filter slot that holds tap kh; a block's first touch is
    the `fresh` one and it is the kh = 0 tap; the blocks of one MMA are contiguous and at most 256 columns wide."""
    L = S.lib()
    seen = {j: [] for j in range(8)}
    first = {}
    for ri in range(16):
        jlo, jhi, slot, fresh = (ctypes.c_int() for _ in range(4))
        assert L.srg_conv9_rows_window(ri, ctypes.byref(jlo), ctypes.byref(jhi), ctypes.byref(slot), ctypes.byref(fresh)) == 0
        jlo, jhi, slot, fresh = jlo.value, jhi.value, slot.value, fresh.value
        assert 0 <= jlo <= jhi <= 7 and (jhi - jlo + 1) * 32 <= 256
        for j in range(jlo, jhi + 1):
            s_j = slot + (j - jlo)                      # consecutive slots for consecutive blocks
            kh = 8 - s_j                                # slot s holds tap kh = 8 - s
            assert 0 <= kh <= 8
            assert (ri - 4) == j + kh - 4               # input row h0 + ri - 4 == output row h0 + j shifted by tap kh
            seen[j].append(kh)
            if j not in first:
                first[j] = (ri, kh, fresh and j == jhi)
    for j in range(8):
        assert sorted(seen[j]) == list(range(9)), (j, seen[j])
        assert first[j][1] == 0 and first[j][2], (j, first[j])       # first touch = tap kh 0, flagged fresh
    assert L.srg_conv9_rows_window(16, None, None, None, None) != 0


def test_reference_written_checkpoint_fixture_loads_on_cpu(reference_ddp_checkpoint):
    """f-1 on the host side: the reference-written DDP checkpoint (module. prefix) maps onto the drop-in module's keys."""
    import torch
    import srgan_b200 as S
    g = S.SRResNet(num_residuals=2)
    sd = torch.load(reference_ddp_checkpoint, map_location="cpu", weights_only=True)
    assert all(k.startswith("module.") for k in sd)
    res = S.load_reference_checkpoint(g, sd)
    assert not res.missing_keys and not res.unexpected_keys
    mine = g.state_dict()
    assert set(mine) == {k[len("module."):] for k in sd}
    for k, v in sd.items():
        assert torch.equal(mine[k[len("module."):]].cpu(), v), k


def test_engine_is_released_when_the_autograd_node_dies_without_backward():
    """models._release_on_death: a grad-enabled forward whose output is dropped frees its engine; the finalizer of an
    OLD node (nodes also die after backward) must not release an engine a newer forward has re-acquired; the plain
    True that train.py's phase-split step writes is never mistaken for a token."""
    import gc
    M = S.models

    class Eng:
        busy = False

    class Fn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, eng_box, x):
            ctx.eng = eng_box[0]
            M._release_on_death(ctx, eng_box[0])
            return x * 2

        @staticmethod
        def backward(ctx, g):
            M._release_if(ctx.eng, ctx.busy_token)
            return None, g * 2

    eng = Eng()
    x = torch.ones(3, requires_grad=True)
    t1 = M._acquire(eng)
    y = Fn.apply([eng], x)
    assert eng.busy == t1 and t1 >= 2
    del y
    gc.collect()
    assert eng.busy is False                           # dropped without backward: released
    M._acquire(eng)
    y1 = Fn.apply([eng], x)
    y1.sum().backward()
    assert eng.busy is False                           # released by backward, node y1 still alive
    t3 = M._acquire(eng)
    y2 = Fn.apply([eng], x)
    del y1
    gc.collect()
    assert eng.busy == t3                              # the old node's death leaves the new owner alone
    eng.busy = True                                    # train.joint_pixel_generator_steps marks engines like this
    del y2
    gc.collect()
    assert eng.busy is True
