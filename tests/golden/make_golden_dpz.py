#!/usr/bin/env python
"""Golden vectors for DPZivkovicAGMMBGS from a build of the REFERENCE's own sources.

With a checkout of the original project:  make -C oracle ref REFERENCE=<checkout> && python tests/golden/make_golden_dpz.py
Writes tests/golden/golden_dpz.json: SHA-256 of the plugin's output masks (the high-threshold mask of
package_bgs/dp/ZivkovicAGMM.cpp, driven as DPZivkovicAGMMBGS::process does) on the committed clips and on the
deterministic stress sequence of tests/conftest.py, for several parameter sets.
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

PARAMS = [{}, {"alpha": 0.05, "threshold": 9.0, "gaussians": 5}, {"alpha": 0.3, "gaussians": 2},
          {"alpha": 0.01, "threshold": 12.5, "gaussians": 4}]


def sequences():
    spec = importlib.util.spec_from_file_location("cf", os.path.join(ROOT, "tests", "conftest.py"))
    cf = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cf)
    z = np.load(os.path.join(HERE, "clips.npz"))
    return {"video_clip": list(z["video_clip"]), "png_clip": list(z["png_clip"]), "stress_120x40x52": cf.stress_sequence(120, 40, 52)}


def main():
    out = {"generator": "tests/golden/make_golden_dpz.py",
           "source": "oracle/_ref/libdp_ref.so = /root/reference/package_bgs/dp/{ZivkovicAGMM,Image}.cpp compiled by `make -C oracle ref`",
           "sequences": {}}
    for name, frames in sequences().items():
        h, w = frames[0].shape[:2]
        entry = {}
        for kw in PARAMS:
            ref = restate.ReferenceDPZivkovic(w, h, **kw)
            hs = hashlib.sha256()
            fgsum = 0
            for f in frames:
                fg, _ = ref.process(f)
                hs.update(fg.tobytes())
                fgsum += int((fg != 0).sum())
            ref.close()
            entry[json.dumps(kw, sort_keys=True)] = {"masks_sha256": hs.hexdigest(), "foreground_pixels": fgsum}
        out["sequences"][name] = {"n_frames": len(frames), "shape": list(frames[0].shape), "params": entry}
    with open(os.path.join(HERE, "golden_dpz.json"), "w") as f:
        json.dump(out, f, indent=1)
    print("wrote golden_dpz.json")


if __name__ == "__main__":
    main()
