import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def reference_ddp_checkpoint(tmp_path_factory):
    """Path of the reference-written DDP checkpoint (make_golden.py:make_checkpoint_fixture), rebuilt whole: the
    parameters from the seeded default initialisation, the BatchNorm buffers from reference_ddp_checkpoint_buffers.pth,
    every entry checked against the dtype, shape and sha256 the reference's file recorded, saved in its key order."""
    import hashlib
    import json
    import torch
    from oracle import srgan_oracle as O
    with open(os.path.join(GOLDEN, "reference_ddp_checkpoint.json")) as f:
        meta = json.load(f)
    stored = torch.load(os.path.join(GOLDEN, "reference_ddp_checkpoint_buffers.pth"), map_location="cpu", weights_only=True)
    init = O.init_srresnet_state(meta["seed"], num_residuals=meta["num_residuals"])
    sd = {}
    for k in meta["keys"]:
        v = stored[k] if k in stored else init[k[len("module."):]]
        assert [str(v.dtype), list(v.shape), hashlib.sha256(v.numpy().tobytes()).hexdigest()] == meta["entries"][k], k
        sd[k] = v
    path = tmp_path_factory.mktemp("checkpoint") / "reference_ddp_checkpoint.pth"
    torch.save(sd, path)
    return str(path)
