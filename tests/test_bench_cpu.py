"""CPU-only checks of bench.py's contract: the workload per GPU count (BASELINE configs[1] on one GPU, configs[2] = global
batch 256 on N > 1), and the reference arm's JSON line (rank 0 prints it, the other ranks exit 0 without work).  The
reference arm is run here at a tiny LR size so that the test takes seconds; it executes the unmodified reference from
oracle/_ref when that copy exists and the oracle port otherwise -- as the checker's CPU baseline, never as the product."""
import importlib.util
import json
import os
import subprocess
import sys
import types

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _args(**kw):
    base = dict(workload="cfg2", batch=None, lr_size=96, generators=3, gpus=1)
    base.update(kw)
    return types.SimpleNamespace(**base)


@pytest.mark.parametrize("world,per_gpu", [(1, 16), (2, 128), (4, 64), (8, 32)])
def test_workload_per_gpu_count_follows_baseline_configs(monkeypatch, world, per_gpu):
    B = _bench_module()
    monkeypatch.setenv("WORLD_SIZE", str(world))
    b, h, w = B.geometry(_args())
    assert (b, h, w) == (per_gpu, 96, 96)
    name = B.workload_name(_args())
    assert name.startswith("cfg2" if world == 1 else f"cfg3 (global batch 256 over {world} GPUs)")
    assert B.geometry(_args(batch=16))[0] == 16                       # --batch pins the per-GPU batch (weak scaling)
    assert B.geometry(_args(workload="gan-native")) == (12, 128, 256)  # src/train.py:94, src/transformers.py:74


def test_dump_outputs_keeps_small_arrays_and_samples_large_ones_the_same_way(tmp_path, monkeypatch):
    import numpy as np
    import torch
    B = _bench_module()
    monkeypatch.setattr(B, "DUMP_BUDGET_BYTES", 1 << 20)
    big = torch.arange(1 << 20, dtype=torch.float64)
    for run in ("a", "b"):
        B.dump_outputs(str(tmp_path / run), {"losses": torch.ones(3, 4), "state": big})
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["losses.npy", "state.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 1 << 20
    losses = np.load(tmp_path / "a" / "losses.npy")
    assert losses.dtype == np.float32 and losses.shape == (3, 4)
    state = np.load(tmp_path / "a" / "state.npy")
    assert state.dtype == np.float32 and 0 < state.size < big.numel()
    share = ((1 << 20) - 2 * 1024 - losses.nbytes) // 4             # the budget left once the small array is whole
    idx = np.unique(np.random.default_rng(0).integers(0, big.numel(), share))
    assert np.array_equal(state, idx.astype(np.float32))            # element i of the arange is i
    assert np.array_equal(state, np.load(tmp_path / "b" / "state.npy"))


def test_steps_below_one_and_dumps_of_the_reference_arm_are_refused():
    for flags in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "unused"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *flags], cwd=ROOT, capture_output=True,
                           text=True, timeout=60)
        assert r.returncode == 2 and "error" in r.stderr, flags


def _run_reference_arm(env_extra, *flags):
    env = dict(os.environ)
    env.update(env_extra)
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
           "--lr-size", "16", "--ref-sample-batch", "1", "--generators", "1", *flags]
    return subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=300)


def test_reference_arm_prints_the_contract_line():
    r = _run_reference_arm({"WORLD_SIZE": "1", "RANK": "0"})
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "srgan_train_lr_patches_per_sec" and line["unit"] == "patches/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["cpu_baseline"]["value"] == line["value"] == line["e2e"]["value"]
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    cfg = line["config"]
    assert cfg["batch_per_gpu"] == 16 and cfg["global_batch"] == 16 and cfg["sample_batch"] == 1 and cfg["lr_hw"] == [16, 16]


def test_reference_arm_other_ranks_exit_without_work():
    r = _run_reference_arm({"WORLD_SIZE": "2", "RANK": "1"}, "--gpus", "2")
    assert r.returncode == 0 and r.stdout.strip() == ""
