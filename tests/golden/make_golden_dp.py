#!/usr/bin/env python
"""Golden vectors for DPAdaptiveMedianBGS / DPMeanBGS / DPWrenGABGS / DPPratiMediodBGS / SigmaDeltaBGS from a build of the REFERENCE's own sources.

With a checkout of the original project:  make -C oracle ref REFERENCE=<checkout> && python tests/golden/make_golden_dp.py
Writes tests/golden/golden_dp.json: SHA-256 of the plugins' output masks (the high-threshold masks of
package_bgs/dp/{AdaptiveMedianBGS,MeanBGS,WrenGA,PratiMediodBGS}.cpp and package_bgs/bl/sdLaMa091.cpp, driven as the DP*BGS::process wrappers do) on the committed clips
and on the deterministic stress sequence of tests/conftest.py, for several parameter sets.
"""
import hashlib
import importlib.util
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import restate  # noqa: E402

F32 = lambda v: float(np.float32(v))        # the wrappers' defaults are float literals read into doubles
# plugin -> (kind, parameter order of the reference's parameter class, parameter sets)
PLUGINS = {
    "DPAdaptiveMedianBGS": ("median", ("threshold", "samplingRate", "learningFrames"),
                            [{}, {"threshold": 10, "samplingRate": 2}, {"threshold": 200, "samplingRate": 3}, {"threshold": 25, "samplingRate": 1}]),
    "DPMeanBGS": ("mean", ("threshold", "alpha", "learningFrames"),
                  [{}, {"threshold": 300, "alpha": 0.9}, {"threshold": 1200, "alpha": 0.5}, {"threshold": 50, "alpha": 0.999}]),
    "DPWrenGABGS": ("wren", ("threshold", "alpha", "learningFrames"),
                    [{}, {"threshold": 3.0, "alpha": 0.2}, {"threshold": 20.0, "alpha": 0.05}, {"threshold": 0.5, "alpha": 0.9}]),
    "DPPratiMediodBGS": ("prati", ("threshold", "samplingRate", "historySize", "weight"),
                         [{}, {"threshold": 10, "samplingRate": 1, "historySize": 4}, {"threshold": 20, "samplingRate": 3, "historySize": 7, "weight": 1},
                          {"threshold": 5, "samplingRate": 20}]),
    "SigmaDeltaBGS": ("sigmadelta", ("ampFactor", "minVar", "maxVar"),
                      [{}, {"ampFactor": 3, "minVar": 2, "maxVar": 40}, {"ampFactor": 2, "minVar": 300, "maxVar": 700}, {"ampFactor": 5, "minVar": 1}]),
}
DEFAULTS = {"DPAdaptiveMedianBGS": {"threshold": 40, "samplingRate": 7, "learningFrames": 30},
            "DPMeanBGS": {"threshold": 2700, "alpha": F32(1e-6), "learningFrames": 30},
            "DPWrenGABGS": {"threshold": 12.25, "alpha": F32(0.005), "learningFrames": 30},
            "DPPratiMediodBGS": {"threshold": 30, "samplingRate": 5, "historySize": 16, "weight": 5},
            "SigmaDeltaBGS": {"ampFactor": 1, "minVar": 15, "maxVar": 255}}


def make_ref(kind, w, h, params):
    """The compiled reference class for a plugin (package_bgs/dp/*, or package_bgs/bl/sdLaMa091.cpp for "sigmadelta")."""
    if kind == "sigmadelta":
        return restate.ReferenceSigmaDelta(w, h, *params)
    return restate.ReferenceDPSimple(kind, w, h, *params)


def sequences():
    spec = importlib.util.spec_from_file_location("cf", os.path.join(ROOT, "tests", "conftest.py"))
    cf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cf)
    z = np.load(os.path.join(HERE, "clips.npz"))
    return {"video_clip": list(z["video_clip"]), "png_clip": list(z["png_clip"]), "stress_120x40x52": cf.stress_sequence(120, 40, 52)}


def main():
    out = {"generator": "tests/golden/make_golden_dp.py",
           "source": "oracle/_ref/libdp_ref.so = /root/reference/package_bgs/dp/{AdaptiveMedianBGS,MeanBGS,WrenGA,PratiMediodBGS,Image}.cpp compiled by `make -C oracle ref`",
           "plugins": {}}
    seqs = sequences()
    for plugin, (kind, order, sets) in PLUGINS.items():
        pentry = {}
        for name, frames in seqs.items():
            h, w = frames[0].shape[:2]
            entry = {}
            for kw in sets:
                full = dict(DEFAULTS[plugin], **kw)
                ref = make_ref(kind, w, h, [full[k] for k in order])
                hs = hashlib.sha256()
                fgsum = 0
                for f in frames:
                    fg, _ = ref.process(f)
                    if fg is None:                       # SigmaDeltaBGS: the first frame only initialises
                        continue
                    hs.update(fg.tobytes())
                    fgsum += int((fg != 0).sum())
                ref.close()
                entry[json.dumps(kw, sort_keys=True)] = {"masks_sha256": hs.hexdigest(), "foreground_pixels": fgsum}
            pentry[name] = {"n_frames": len(frames), "shape": list(frames[0].shape), "params": entry}
        out["plugins"][plugin] = pentry
    with open(os.path.join(HERE, "golden_dp.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote golden_dp.json")


if __name__ == "__main__":
    main()
