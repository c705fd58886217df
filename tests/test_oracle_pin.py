"""Pin the oracle before trusting it (CPU only).

The reference holds no golden vectors or known-answer tests for this path (SURVEY 4, 8c), so the
pins are (1) OpenCV itself -- the library the reference plugins delegate every arithmetic step to --
replayed call-for-call (oracle/cv2_chain.py) and (2) SHA-256 hashes of those OpenCV outputs on the
reference's own data files, committed in tests/golden/golden.json by tests/golden/make_golden.py.
"""
import hashlib
import os

import numpy as np
import pytest

from conftest import REFERENCE_DIR, drift_sequence, stress_sequence

NAMES = {0: "FrameDifferenceBGS", 1: "StaticFrameDifferenceBGS", 2: "WeightedMovingMeanBGS",
         3: "WeightedMovingVarianceBGS", 5: "MixtureOfGaussianV2BGS", 6: "AdaptiveBackgroundLearning"}


def sha(arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def run(algo_cls, frames, **kw):
    a = algo_cls(**kw)
    fgs, bgs = [], []
    for f in frames:
        fg, bg = a.process(f)
        if fg is not None:
            fgs.append(fg)
        if bg is not None:
            bgs.append(bg)
    return fgs, bgs


@pytest.mark.parametrize("seq", ["video_clip", "png_clip"])
@pytest.mark.parametrize("aid", [0, 1, 2, 3, 5, 6])
@pytest.mark.parametrize("thr", [True, False])
def test_c_oracle_matches_golden_hashes(oracle, clips, golden, seq, aid, thr):
    frames = list(clips[seq])
    g = golden["sequences"][seq]
    assert sha(frames) == g["input_sha256"]
    key = NAMES[aid] + ("" if thr else ":enableThreshold=0")
    fgs, bgs = run(oracle.ALGOS[aid], frames, enableThreshold=thr)
    exp = g["algos"][key]
    assert len(fgs) == exp["n_fg"] and len(bgs) == exp["n_bg"]
    assert sha(fgs) == exp["fg_sha256"]                       # bit-exact masks
    if exp["bg_sha256"]:
        assert sha(bgs) == exp["bg_sha256"]                   # byte-exact background model


@pytest.mark.parametrize("aid", [0, 1, 2, 3, 5, 6])
def test_c_oracle_matches_opencv_live(oracle, clips, aid):
    """Same comparison against cv2 running live (the image on the GPU box has cv2 too)."""
    from oracle import cv2_chain
    for frames in (list(clips["video_clip"]), stress_sequence(120)):
        for thr in (True, False):
            a, b = run(cv2_chain.ALGOS[aid], frames, enableThreshold=thr), run(oracle.ALGOS[aid], frames, enableThreshold=thr)
            assert len(a[0]) == len(b[0]) and len(a[1]) == len(b[1])
            for x, y in zip(a[0] + a[1], b[0] + b[1]):
                assert np.array_equal(x, y)


@pytest.mark.skipif(not os.path.isdir(REFERENCE_DIR),
                    reason="needs a checkout of the original project at $BGSB_REFERENCE_DIR or /root/reference")
@pytest.mark.parametrize("aid", [0, 1, 2, 3, 5, 6])
def test_c_oracle_full_reference_sequences(oracle, golden, aid):
    """All 374 frames of dataset/video.avi and all 51 frames/N.png (BASELINE config 1 inputs)."""
    import cv2
    cap = cv2.VideoCapture(os.path.join(REFERENCE_DIR, "dataset", "video.avi"))
    video = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        video.append(f)
    pngs = [cv2.imread(os.path.join(REFERENCE_DIR, "frames", "%d.png" % i)) for i in range(1, 52)]
    for name, frames in (("video_full", video), ("png_full", pngs)):
        g = golden["sequences"][name]
        assert sha(frames) == g["input_sha256"], "decoder produced different frames than the golden run"
        fgs, bgs = run(oracle.ALGOS[aid], frames)
        assert sha(fgs) == g["algos"][NAMES[aid]]["fg_sha256"]
        if bgs:
            assert sha(bgs) == g["algos"][NAMES[aid]]["bg_sha256"]


def test_gray_formula_matches_opencv(oracle):
    import cv2
    rng = np.random.default_rng(0)
    img = rng.integers(0, 256, (512, 512, 3), dtype=np.uint8)
    img[:16, :16] = 255
    img[16:32, :16] = 0
    assert np.array_equal(oracle.gray_bgr(img, 0), cv2.cvtColor(img, cv2.COLOR_BGR2GRAY))
    # 2.4 constants differ from 4.x by at most one level (SURVEY Appendix B)
    d = oracle.gray_bgr(img, 1).astype(int) - oracle.gray_bgr(img, 0).astype(int)
    assert np.abs(d).max() <= 1 and 0 < (d != 0).mean() < 0.01


def test_abl_exhaustive_pairs_against_opencv(oracle):
    """Every (input, background) byte pair: the fp64 blend of A.2 reproduces cv2.addWeighted ties."""
    from oracle import cv2_chain
    inp, bg = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8))
    frame0 = np.repeat(bg[:, :, None], 3, 2).copy()
    frame1 = np.repeat(inp[:, :, None], 3, 2).copy()
    a, b = cv2_chain.AdaptiveBackgroundLearning(), oracle.AdaptiveBackgroundLearning()
    for f in (frame0, frame1):
        fa, ba = a.process(f)
        fb, bb = b.process(f)
    assert np.array_equal(fa, fb) and np.array_equal(ba, bb)


@pytest.mark.parametrize("kw", [{}, {"learningFrames": 3}, {"learningFrames": -1, "alphaDetection": 0.3, "threshold": 10},
                                {"learningFrames": 5, "alphaLearn": 0.5, "threshold": 40}])
def test_asbl_restatement_against_opencv(oracle, clips, kw):
    """AdaptiveSelectiveBackgroundLearning (USTC_BGS type 7): the C restatement vs the OpenCV call chain
    (cvtColor, absdiff, convertScaleAbs, threshold, medianBlur, addWeighted) on the reference clip, on a
    noisy moving scene, and on every (gray input, model) byte pair."""
    from oracle import cv2_chain
    rng = np.random.default_rng(3)
    h, w = 97, 131
    base = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    moving = []
    for t in range(14):
        f = np.clip(base.astype(np.int16) + rng.integers(-30, 31, (h, w, 3)), 0, 255).astype(np.uint8)
        f[10 + 4 * t:40 + 4 * t, 20 + 5 * t:60 + 5 * t] = 255 - base[10 + 4 * t:40 + 4 * t, 20 + 5 * t:60 + 5 * t]
        moving.append(f)
    inp, bg = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8))
    pairs = [np.repeat(bg[:, :, None], 3, 2).copy(), np.repeat(inp[:, :, None], 3, 2).copy()]   # gray(v,v,v) == v
    for frames in (list(clips["video_clip"]), moving, pairs):
        a, b = cv2_chain.AdaptiveSelectiveBackgroundLearning(**kw), oracle.AdaptiveSelectiveBackgroundLearning(**kw)
        for i, f in enumerate(frames):
            fa, ba = a.process(f)
            fb, bb = b.process(f)
            assert np.array_equal(fa, fb) and np.array_equal(ba, bb), i


DPZ_PARAMS = [{}, {"alpha": 0.05, "threshold": 9.0, "gaussians": 5}, {"alpha": 0.3, "gaussians": 2},
              {"alpha": 0.01, "threshold": 12.5, "gaussians": 4}]


@pytest.mark.parametrize("kw", DPZ_PARAMS)
def test_dpzivkovic_restatement_matches_reference_golden(oracle, clips, kw):
    """orc_dpz_apply vs the masks a build of the reference's OWN ZivkovicAGMM sources produced
    (tests/golden/golden_dpz.json, written by make_golden_dpz.py from oracle/_ref/libdp_ref.so)."""
    import hashlib
    import json
    import os
    from conftest import stress_sequence
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_dpz.json")))
    seqs = {"video_clip": list(clips["video_clip"]), "png_clip": list(clips["png_clip"]),
            "stress_120x40x52": stress_sequence(120, 40, 52)}
    for name, frames in seqs.items():
        o = oracle.DPZivkovicAGMMBGS(**kw)
        hs = hashlib.sha256()
        for f in frames:
            fg, bg = o.process(f)
            assert bg is None
            hs.update(fg.tobytes())
        assert hs.hexdigest() == g["sequences"][name]["params"][json.dumps(kw, sort_keys=True)]["masks_sha256"], name


@pytest.mark.parametrize("kw", DPZ_PARAMS)
def test_dpzivkovic_restatement_matches_reference_build_live(oracle, kw):
    """The same on a sequence the golden file above does not hold: frame by frame against the compiled reference itself
    where oracle/_ref/libdp_ref.so has been built (`make -C oracle ref`), else against tests/golden/golden_drift.json."""
    frames = drift_sequence(60, 5)
    o = oracle.DPZivkovicAGMMBGS(**kw)
    try:
        ref = oracle.ReferenceDPZivkovic(83, 57, **kw)
    except FileNotFoundError:
        _assert_drift_golden(o, frames, "DPZivkovicAGMMBGS", kw)
        return
    for i, f in enumerate(frames):
        assert np.array_equal(o.process(f)[0], ref.process(f)[0]), i
    ref.close()


def _assert_drift_golden(plugin, frames, name, kw):
    import json
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_drift.json")))
    want = g["plugins"][name][json.dumps(kw, sort_keys=True)]
    hs, n, fgsum = hashlib.sha256(), 0, 0
    for f in frames:
        fg, bg = plugin.process(f)
        assert bg is None
        if fg is not None:
            hs.update(fg.tobytes())
            n += 1
            fgsum += int((fg != 0).sum())
    assert (n, fgsum, hs.hexdigest()) == (want["n_masks"], want["foreground_pixels"], want["masks_sha256"]), (name, kw)


def _dp_simple_cases():
    import importlib.util
    import os
    spec = importlib.util.spec_from_file_location("mgd", os.path.join(os.path.dirname(__file__), "golden", "make_golden_dp.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.parametrize("plugin", ["DPAdaptiveMedianBGS", "DPMeanBGS", "DPWrenGABGS", "DPPratiMediodBGS", "SigmaDeltaBGS"])
def test_dp_simple_restatements_match_reference_golden(oracle, clips, plugin):
    """orc_dp_median / orc_dp_mean / orc_dp_wren vs the masks a build of the reference's OWN AdaptiveMedianBGS / MeanBGS /
    WrenGA sources produced (tests/golden/golden_dp.json, written by make_golden_dp.py from oracle/_ref/libdp_ref.so):
    both clips and the stress sequence, four parameter sets each (incl. a median threshold whose doubled value wraps in
    the reference's unsigned char member)."""
    import hashlib
    import json
    import os
    from conftest import stress_sequence
    m = _dp_simple_cases()
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "golden_dp.json")))["plugins"][plugin]
    seqs = {"video_clip": list(clips["video_clip"]), "png_clip": list(clips["png_clip"]),
            "stress_120x40x52": stress_sequence(120, 40, 52)}
    for kw in m.PLUGINS[plugin][2]:
        seen = 0
        for name, frames in seqs.items():
            o = getattr(oracle, plugin)(**kw)
            hs = hashlib.sha256()
            fgsum = 0
            for f in frames:
                fg, bg = o.process(f)
                assert bg is None
                if fg is None:                                   # SigmaDeltaBGS: the first frame only initialises
                    continue
                hs.update(fg.tobytes())
                fgsum += int((fg != 0).sum())
            want = g[name]["params"][json.dumps(kw, sort_keys=True)]
            assert fgsum == want["foreground_pixels"] and hs.hexdigest() == want["masks_sha256"], (name, kw)
            assert fgsum < len(frames) * frames[0].shape[0] * frames[0].shape[1], (name, kw)
            seen += fgsum
        assert seen > 0, kw                                  # (PratiMediod gives no mask before frame historySize: the 16-frame clip stays empty)


@pytest.mark.parametrize("plugin", ["DPAdaptiveMedianBGS", "DPMeanBGS", "DPWrenGABGS", "DPPratiMediodBGS", "SigmaDeltaBGS"])
def test_dp_simple_restatements_match_reference_build_live(oracle, plugin):
    """The same on a sequence the golden file above does not hold: frame by frame against the compiled reference itself
    where oracle/_ref/libdp_ref.so has been built (`make -C oracle ref`), else against tests/golden/golden_drift.json."""
    m = _dp_simple_cases()
    kind, order, sets = m.PLUGINS[plugin]
    frames = drift_sequence(50, 11)
    for kw in sets:
        full = dict(m.DEFAULTS[plugin], **kw)
        o = getattr(oracle, plugin)(**kw)
        try:
            ref = m.make_ref(kind, 83, 57, [full[k] for k in order])
        except (FileNotFoundError, AttributeError):      # no reference build, or one older than this plugin
            _assert_drift_golden(o, frames, plugin, kw)
            continue
        for i, f in enumerate(frames):
            a, b = o.process(f)[0], ref.process(f)[0]
            assert (a is None) == (b is None) and (a is None or np.array_equal(a, b)), (kw, i)
        ref.close()


def test_morph_and_ccl_against_opencv(oracle):
    from oracle import cv2_chain
    rng = np.random.default_rng(3)
    for trial in range(25):
        h, w = int(rng.integers(5, 90)), int(rng.integers(5, 130))
        m = (rng.random((h, w)) < rng.choice([0.05, 0.3, 0.5, 0.7])).astype(np.uint8) * 255
        for op in ("erode", "dilate"):
            for it in (0, 1, 2, 3):
                assert np.array_equal(cv2_chain.morph(m, op, it) if it else m, oracle.morph(m, op, it))
        n1, l1 = cv2_chain.canonical_labels(m)
        for zb in (False, True):
            n2, l2, st, ext = oracle.ccl8(m, zb)
            if not zb:
                assert n1 == n2 and np.array_equal(l1, l2)
            rects, _ = cv2_chain.external_contour_rects(m, zb)
            mine = [(int(s[0]), int(s[1]), int(s[2] - s[0] + 1), int(s[3] - s[1] + 1)) for s, e in zip(st, ext) if e]
            # findContours lists external contours in reverse raster order of their first pixels
            assert list(reversed(mine)) == [tuple(r) for r in rects]


def test_rect_moments_against_opencv(oracle):
    import cv2
    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (70, 90), dtype=np.uint8)
    for (x, y, w, h) in ((0, 0, 90, 70), (3, 5, 40, 33), (88, 69, 2, 1)):
        m = cv2.moments(img[y:y + h, x:x + w], False)
        got = oracle.rect_moments(img, (x, y, w, h))
        assert got == [int(m[k]) for k in ("m00", "m10", "m01", "m20", "m02", "m11")]


def test_golden_ccl_tables(oracle, clips, golden):
    """FD -> OPEN(3x3) -> canonical labels on the clip reproduces the committed OpenCV results."""
    frames = list(clips["video_clip"])
    fgs, _ = run(oracle.FrameDifferenceBGS, frames)
    for zb in (0, 1):
        for row in golden["sequences"]["video_clip"]["fd_open_ccl"]["zero_border_%d" % zb]:
            m = oracle.morph(oracle.morph(fgs[row["frame"]], "erode"), "dilate")
            assert sha([m]) == row["open_sha256"]
            n, lab, st, ext = oracle.ccl8(m, bool(zb))
            assert n == row["n_components"] and sha([lab]) == row["labels_sha256"]
            mine = [[int(s[0]), int(s[1]), int(s[2] - s[0] + 1), int(s[3] - s[1] + 1)] for s, e in zip(st, ext) if e]
            assert list(reversed(mine)) == row["external_rects_findcontours_order"]


def test_blobdetector_restatement_reproduces_committed_sequence(oracle, clips, golden):
    """Regression pin only: the list logic of CvBlobDetectorCC is 'restated, unpinned' (oracle/blobdetect.py)."""
    from oracle import blobdetect, cv2_chain
    frames = list(clips["video_clip"])
    fgs, _ = run(oracle.FrameDifferenceBGS, frames)
    bd = blobdetect.CvBlobDetectorCC(zero_border=True)
    exp = golden["sequences"]["video_clip"]["fd_open_blobdetector_restated_unpinned"]
    for m, e in zip(fgs, exp):
        m2 = cv2_chain.morph(cv2_chain.morph(m, "erode"), "dilate")
        res, nb = bd.DetectNewBlob(m2, [])
        assert res == e["result"]
        assert [[round(v, 4) for v in b.tuple()] for b in bd.lists[0]] == e["frame_blobs"]
