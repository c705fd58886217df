import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
REFERENCE_DIR = os.environ.get("BGSB_REFERENCE_DIR", "/root/reference")    # a checkout of the original project, if one is at hand


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    # a `gpu` test must never silently pass on a box without a GPU
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def clips():
    z = np.load(os.path.join(GOLDEN_DIR, "clips.npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def golden():
    with open(os.path.join(GOLDEN_DIR, "golden.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def oracle():
    from oracle import restate
    restate.build()
    return restate


def stress_sequence(n=200, h=48, w=64, seed=7):
    """Mode-churn stress input of SURVEY A.4: 7-colour palette, 15 % switch probability, +-2 noise."""
    rng = np.random.default_rng(seed)
    pal = rng.integers(0, 256, (7, 3)).astype(np.int16)
    idx = rng.integers(0, 7, (h, w))
    out = []
    for _ in range(n):
        sw = rng.random((h, w)) < 0.15
        idx = np.where(sw, rng.integers(0, 7, (h, w)), idx)
        f = pal[idx] + rng.integers(-2, 3, (h, w, 3))
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


def drift_sequence(n, seed):
    """83 x 57 noisy static scene (+-8) crossed by a drifting solid block of a random colour."""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (57, 83, 3), dtype=np.uint8)
    frames = []
    for t in range(n):
        f = np.clip(base.astype(np.int16) + rng.integers(-8, 9, base.shape), 0, 255).astype(np.uint8)
        f[5 + t // 2:25 + t // 2, 10 + t:40 + t] = rng.integers(0, 256, 3)
        frames.append(f)
    return frames
