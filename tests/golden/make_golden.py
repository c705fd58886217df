"""Generates the golden fixtures of tests/golden/ from the reference's own data files.

Needs a checkout of the original project ($BGSB_REFERENCE_DIR, else /root/reference) and cv2 4.13; the outputs are
committed, so the tests need neither the original project nor any video decoding:

    BGSB_REFERENCE_DIR=<checkout of the original project> python tests/golden/make_golden.py

Inputs  : $BGSB_REFERENCE_DIR/dataset/video.avi  (320x176, 374 frames; BASELINE config 1)
          $BGSB_REFERENCE_DIR/frames/1..51.png   (320x240; read by Demo2.cpp:148-151)
Oracle  : oracle/cv2_chain.py -- the reference plugins replayed call-for-call on OpenCV 4.13
          (the library the plugins delegate all arithmetic to).
Outputs : clips.npz     small crops of consecutive decoded frames (inputs for every test)
          golden.json   SHA-256 of every output on the clips AND on the full sequences, plus
                        the CC / blob tables of selected frames.
"""
from __future__ import annotations

import hashlib
import json
import os
import sys
import zipfile

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import cv2_chain as ref          # noqa: E402
from oracle import blobdetect as ref_bd      # noqa: E402

REF = os.environ.get("BGSB_REFERENCE_DIR", "/root/reference")
NAMES = {0: "FrameDifferenceBGS", 1: "StaticFrameDifferenceBGS", 2: "WeightedMovingMeanBGS",
         3: "WeightedMovingVarianceBGS", 5: "MixtureOfGaussianV2BGS", 6: "AdaptiveBackgroundLearning"}


def save_npz_lzma(path, **arrays):
    """np.savez with LZMA members (np.load reads them): the clips stay under 1 MB, where savez_compressed's deflate
    needs 1.3 MB."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_LZMA) as z:
        for name, a in arrays.items():
            with z.open(name + ".npy", "w") as f:
                np.lib.format.write_array(f, a)


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run_algo(aid, frames, **kw):
    a = ref.ALGOS[aid](**kw)
    fgs, bgs, first = [], [], None
    for i, f in enumerate(frames):
        fg, bg = a.process(f)
        if fg is not None:
            if first is None:
                first = i
            fgs.append(fg)
        if bg is not None:
            bgs.append(bg)
    return {"first_fg_frame": first, "n_fg": len(fgs), "n_bg": len(bgs), "fg_sha256": sha(fgs),
            "bg_sha256": sha(bgs) if bgs else None, "fg_pixels_set": int(sum(int((m > 0).sum()) for m in fgs))}, fgs


def pipeline_tables(fgs, zero_border):
    """FD mask -> OPEN(3x3) -> canonical labels + external rects, for a few frames."""
    out = []
    for i in sorted({min(5, len(fgs) - 1), min(12, len(fgs) - 1), min(20, len(fgs) - 1), len(fgs) - 1}):
        m = ref.morph(ref.morph(fgs[i], "erode"), "dilate")
        n, lab = ref.canonical_labels(m if not zero_border else _zb(m))
        rects, _ = ref.external_contour_rects(m, zero_border)
        out.append({"frame": i, "open_sha256": sha([m]), "n_components": int(n), "labels_sha256": sha([lab]),
                    "external_rects_findcontours_order": [list(map(int, r)) for r in rects]})
    return out


def _zb(m):
    m = m.copy()
    m[0, :] = 0; m[-1, :] = 0; m[:, 0] = 0; m[:, -1] = 0
    return m


def blob_sequence(fgs):
    bd = ref_bd.CvBlobDetectorCC(zero_border=True)
    seq = []
    for m in fgs:
        m2 = ref.morph(ref.morph(m, "erode"), "dilate")
        res, nb = bd.DetectNewBlob(m2, [])
        seq.append({"result": res, "new": [round(v, 4) for v in nb.tuple()] if nb else None,
                    "frame_blobs": [[round(v, 4) for v in b.tuple()] for b in bd.lists[0]]})
    return seq


def main():
    cap = cv2.VideoCapture(os.path.join(REF, "dataset", "video.avi"))
    video = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        video.append(f)
    assert len(video) == 374 and video[0].shape == (176, 320, 3)
    pngs = [cv2.imread(os.path.join(REF, "frames", "%d.png" % i)) for i in range(1, 52)]
    assert all(p is not None and p.shape == (240, 320, 3) for p in pngs)

    # ragged sizes on purpose (190 = 5*32+30, 126; 150x101)
    video_clip = np.stack([f[24:150, 0:190] for f in video[56:88]])          # 32 x 126 x 190 x 3
    png_clip = np.stack([f[60:161, 80:230] for f in pngs[0:16]])             # 16 x 101 x 150 x 3
    save_npz_lzma(os.path.join(HERE, "clips.npz"), video_clip=video_clip, png_clip=png_clip)

    golden = {"generator": "tests/golden/make_golden.py", "opencv": cv2.__version__,
              "decoder_note": "video.avi decoded by cv2.VideoCapture (FFMPEG) in the build container",
              "sequences": {}}
    seqs = {"video_clip": list(video_clip), "png_clip": list(png_clip), "video_full": video, "png_full": pngs}
    for sname, frames in seqs.items():
        entry = {"shape": list(np.asarray(frames[0]).shape), "n_frames": len(frames), "input_sha256": sha(frames),
                 "algos": {}}
        for aid, name in NAMES.items():
            res, fgs = run_algo(aid, frames)
            entry["algos"][name] = res
            if aid == 0:
                fd_fgs = fgs
            res_raw, _ = run_algo(aid, frames, enableThreshold=False)
            entry["algos"][name + ":enableThreshold=0"] = res_raw
        entry["fd_open_ccl"] = {"zero_border_0": pipeline_tables(fd_fgs, False),
                                "zero_border_1": pipeline_tables(fd_fgs, True)}
        if sname in ("video_clip", "video_full"):
            entry["fd_open_blobdetector_restated_unpinned"] = blob_sequence(fd_fgs)
        golden["sequences"][sname] = entry
        print(sname, "done")
    with open(os.path.join(HERE, "golden.json"), "w") as f:
        json.dump(golden, f, indent=1)
    print("wrote", os.path.join(HERE, "golden.json"))


if __name__ == "__main__":
    main()
