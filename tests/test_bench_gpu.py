"""bench.py --dump-outputs on the GPU: what it writes is the state the timed steps left, and the same on every run."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--batch", "2", "--lr-size", "16", "--warmup", "0", "--no-e2e", "--no-hbm", "--no-cpu-baseline"]


def _dump(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), *SMALL,
                        "--dump-outputs", str(out)], cwd=ROOT, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    return {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}


def test_dump_outputs_hold_the_trained_state_and_repeat(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import srgan_b200 as S
    a, b, c = _dump(tmp_path / "a", 1), _dump(tmp_path / "b", 1), _dump(tmp_path / "c", 2)
    assert sorted(a) == ["generator0_state", "generator1_state", "generator2_state", "losses"]
    assert a["losses"].shape == (3, 4) and a["losses"].dtype == np.float32 and np.isfinite(a["losses"]).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k                        # seeded inputs and weights: identical files
        assert not np.array_equal(a[k], c[k]), k                    # one more timed step: other losses, other state
    for i in range(3):
        torch.manual_seed(i)                                        # the seed bench.py builds generator i with
        g = S.SRResNet()
        init = torch.cat([v.reshape(-1).float() for v in g.state_dict().values() if v.is_floating_point()]).numpy()
        got = a[f"generator{i}_state"]
        assert got.shape == init.shape and np.isfinite(got).all()
        assert np.mean(got != init) > 0.9, i                        # Adam moved the weights; BatchNorm buffers moved
