"""bench.py contract checks: the reference arm prints ONE JSON line with the agreed keys, the product arm refuses to run
without a CUDA device (no CPU fallback), and on a GPU --dump-outputs writes what the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "MOG2 Mpixel/s at 1080p" and d["unit"] == "Mpixel/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1"],
             env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_dump_outputs_needs_the_product_arm(tmp_path):
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "1", "--dump-outputs", str(tmp_path)])
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_frame(tmp_path, oracle):
    """--dump-outputs after W warm-up and K timed steps of F frames == the oracle after (W + K) * F frames of the same
    synthetic stream: the dump is the timed path's last output, and --steps sets how many steps ran."""
    from tracking_b200 import synth
    F, K, Wm = 3, 2, 3
    r = _run(["--steps", str(K), "--warmup", str(Wm), "--frames-per-step", str(F), "--headline-only", "--no-e2e",
              "--no-parity", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)])
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == K
    fg, bg = np.load(tmp_path / "foreground_mask.npy"), np.load(tmp_path / "background_image.npy")
    assert fg.dtype == bg.dtype == np.float32 and fg.shape == (1080, 1920) and bg.shape == (1080, 1920, 3)
    o = oracle.MixtureOfGaussianV2BGS()
    for t in range((Wm + K) * F):                  # the benchmark cycles 128 resident frames; fewer are used here
        ofg, obg = o.process(oracle.synth_frame(1920, 1080, t, synth.SEED0))
    assert np.array_equal(fg, ofg) and np.array_equal(bg, obg)


def test_product_arm_needs_a_cuda_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present")
    r = _run(["--steps", "1", "--warmup", "1"])
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
