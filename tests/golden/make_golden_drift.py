#!/usr/bin/env python
"""Golden vectors for the DP package's plugins and SigmaDeltaBGS on the drift sequences of tests/conftest.py.

    python tests/golden/make_golden_drift.py

Writes tests/golden/golden_drift.json: SHA-256 of each plugin's output masks, their count and their foreground pixels,
for the parameter sets of make_golden_dpz.py / make_golden_dp.py.  The masks come from the reference's own classes when
oracle/_ref/libdp_ref.so has been built (`make -C oracle ref REFERENCE=<checkout of the original project>`), otherwise
from the C restatement; "source" records which.  tests/test_oracle_pin.py compares the restatement with the reference
build frame by frame where that library exists, and with this file where it does not.
"""
import hashlib
import importlib.util
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import restate  # noqa: E402

DPZ_FRAMES, DPZ_SEED = 60, 5
DP_FRAMES, DP_SEED = 50, 11
W, H = 83, 57


def _load(name, path):
    spec = importlib.util.spec_from_file_location(name, path)
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def record(plugin, frames):
    """{"masks_sha256", "n_masks", "foreground_pixels"} of `plugin`'s outputs over `frames`."""
    hs, n, fgsum = hashlib.sha256(), 0, 0
    for f in frames:
        fg, _ = plugin.process(f)
        if fg is None:                                   # SigmaDeltaBGS: the first frame only initialises
            continue
        hs.update(fg.tobytes())
        n += 1
        fgsum += int((fg != 0).sum())
    if hasattr(plugin, "close"):
        plugin.close()
    return {"masks_sha256": hs.hexdigest(), "n_masks": n, "foreground_pixels": fgsum}


def main():
    cf = _load("cf", os.path.join(ROOT, "tests", "conftest.py"))
    dpz = _load("mgdz", os.path.join(HERE, "make_golden_dpz.py"))
    dp = _load("mgd", os.path.join(HERE, "make_golden_dp.py"))
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libdp_ref.so"))
    out = {"generator": "tests/golden/make_golden_drift.py",
           "source": ("oracle/_ref/libdp_ref.so: the reference's own classes compiled by `make -C oracle ref`" if have_ref else
                      "the C restatement (oracle/c/bgs_oracle.c); oracle/_ref/libdp_ref.so was not built when this file "
                      "was written.  The frame-by-frame comparison with the reference build on these sequences is "
                      "tests/test_oracle_pin.py::*_reference_build_live, which runs where that library exists"),
           "sequences": {"DPZivkovicAGMMBGS": {"frames": DPZ_FRAMES, "seed": DPZ_SEED},
                         "others": {"frames": DP_FRAMES, "seed": DP_SEED}},
           "plugins": {}}
    frames = cf.drift_sequence(DPZ_FRAMES, DPZ_SEED)
    out["plugins"]["DPZivkovicAGMMBGS"] = {
        json.dumps(kw, sort_keys=True): record(restate.ReferenceDPZivkovic(W, H, **kw) if have_ref else
                                               restate.DPZivkovicAGMMBGS(**kw), frames)
        for kw in dpz.PARAMS}
    frames = cf.drift_sequence(DP_FRAMES, DP_SEED)
    for name, (kind, order, sets) in dp.PLUGINS.items():
        entry = {}
        for kw in sets:
            full = dict(dp.DEFAULTS[name], **kw)
            p = dp.make_ref(kind, W, H, [full[k] for k in order]) if have_ref else getattr(restate, name)(**kw)
            entry[json.dumps(kw, sort_keys=True)] = record(p, frames)
        out["plugins"][name] = entry
    with open(os.path.join(HERE, "golden_drift.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote golden_drift.json (%s)" % ("reference build" if have_ref else "C restatement"))


if __name__ == "__main__":
    main()
