"""The C restatement against OpenCV (cv2 4.13, live) away from the default parameters.

The GPU is compared with the restatement, so a parameter the restatement misreads would be copied by the kernels
without any test noticing.  These pins close that gap: every MOG2 key (seeded draws plus named edges: learning rates
>= 1 that re-initialise the model, also switched within one stream, varMin > varMax, histories 1 and 2, rates below
1e-4), and the threshold / weight / alpha keys of FD, StaticFD, WMM, WMV, ABL and ASBL.  The draws are those of
tests/param_draws.py, which the GPU sweeps (test_gpu_param_space.py) use too.

Known divergence, left out of the draws: for float inputs cv2 4.13's addWeighted rounds fma(x, alpha, y * beta) (as
measured over all pairs of input bytes), while the restatement (ABL, ASBL's learning phase) rounds the double sum
x * alpha + y * beta.  At alpha 0.05 (the default), 0.25, 0.5 or 0.7 both give the same byte for every pair; at alpha
0.3, 19 of the 65536 pairs differ by one.  test_blend_forms_agree_at_the_swept_alphas pins which alphas are safe."""
import numpy as np
import pytest

from conftest import stress_sequence
from param_draws import MOG2_FRAMES, alphas_per_frame, asbl_draws, mog2_draws, scene, simple_draws

MOG2 = mog2_draws()


def mog2_inputs(name):
    """Both input kinds for a draw: the moving-blob scene and the mode-churn stress sequence (ragged sizes)."""
    seed = sum(map(ord, name))
    return (scene(np.random.default_rng(seed), MOG2_FRAMES, 40, 56),
            stress_sequence(MOG2_FRAMES, 23, 37, seed=seed))


@pytest.mark.parametrize("name", sorted(MOG2))
def test_mog2_restatement_matches_opencv_across_parameters(oracle, name):
    """Raw mask ({0, shadowValue, 255}) and background image on every frame, alpha changed between frames as scheduled."""
    from oracle import cv2_chain
    d = MOG2[name]
    alphas = alphas_per_frame(d)
    for frames in mog2_inputs(name):
        o = oracle.MixtureOfGaussianV2BGS(enableThreshold=False, **d["model"])
        c = cv2_chain.MixtureOfGaussianV2BGS(enableThreshold=False, **d["model"])
        for t, f in enumerate(frames):
            o.alpha = c.alpha = alphas[t]
            ofg, obg = o.process(f)
            cfg, cbg = c.process(f)
            assert np.array_equal(ofg, cfg), (name, t, int((ofg != cfg).sum()))
            assert np.array_equal(obg, cbg), (name, t, int((obg != cbg).sum()))


def test_mog2_thresholded_output_at_every_threshold_edge(oracle):
    """The wrapper's threshold on top of the raw mask, at the shadow value's neighbours."""
    from oracle import cv2_chain
    frames = stress_sequence(16, 20, 30, seed=11)
    for thr in (0, 126, 127, 128, 254, 255):
        for sv in (0, 127, 255):
            o = oracle.MixtureOfGaussianV2BGS(enableThreshold=True, threshold=thr, shadowValue=sv)
            c = cv2_chain.MixtureOfGaussianV2BGS(enableThreshold=True, threshold=thr, shadowValue=sv)
            for t, f in enumerate(frames):
                a, b = o.process(f), c.process(f)
                assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), (thr, sv, t)


def test_mog2_reinitialisation_restarts_the_automatic_rate(oracle):
    """alpha >= 1 re-initialises the model; alpha < 0 afterwards counts its rate 1/min(2 nframes, history) from there, so
    a restatement that kept counting from the first frame would diverge from OpenCV on the frames after the switch."""
    from oracle import cv2_chain
    frames = stress_sequence(20, 16, 24, seed=5)
    o = oracle.MixtureOfGaussianV2BGS(enableThreshold=False, history=50)
    c = cv2_chain.MixtureOfGaussianV2BGS(enableThreshold=False, history=50)
    for t, f in enumerate(frames):
        o.alpha = c.alpha = 1.0 if t == 10 else -1.0
        a, b = o.process(f), c.process(f)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), t
        if t == 10:
            assert o.nframes == 1 and (o.nmodes == 1).all()       # one mode per pixel, as after a first frame


@pytest.mark.parametrize("cls,kw", simple_draws(), ids=lambda v: v if isinstance(v, str) else
                         ",".join("%s=%s" % kv for kv in sorted(v.items())))
def test_simple_plugins_match_opencv_across_parameters(oracle, cls, kw):
    from oracle import cv2_chain
    frames = scene(np.random.default_rng(31), 10, 21, 35) + stress_sequence(6, 21, 35, seed=2)
    okw = {k: (bool(v) if k.startswith("enable") else v) for k, v in kw.items()}
    o, c = getattr(oracle, cls)(**okw), getattr(cv2_chain, cls)(**okw)
    for t, f in enumerate(frames):
        a, b = o.process(f), c.process(f)
        for x, y in zip(a, b):
            assert (x is None) == (y is None), t
            if x is not None:
                assert np.array_equal(x, y), (t, int((x != y).sum()))


@pytest.mark.parametrize("i", range(len(asbl_draws())))
def test_asbl_matches_opencv_across_parameters(oracle, i):
    from oracle import cv2_chain
    kw = asbl_draws()[i]
    frames = scene(np.random.default_rng(40 + i), 14, 19, 33)
    o = oracle.AdaptiveSelectiveBackgroundLearning(**kw)
    c = cv2_chain.AdaptiveSelectiveBackgroundLearning(**kw)
    for t, f in enumerate(frames):
        a, b = o.process(f), c.process(f)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), (kw, t)


def test_blend_forms_agree_at_the_swept_alphas():
    """Every ABL / ASBL alpha the sweeps use gives the same background byte whether the blend is rounded from the double
    sum (the restatement) or as cv2.addWeighted rounds it, over all 65536 pairs of input bytes."""
    import cv2
    s = np.float32(1. / 255.)
    x, y = np.meshgrid(np.arange(256, dtype=np.float32) * s, np.arange(256, dtype=np.float32) * s, indexing="ij")
    alphas = {kw["alpha"] for c, kw in simple_draws() if c == "AdaptiveBackgroundLearning"}
    alphas |= {kw[k] for kw in asbl_draws() for k in ("alphaLearn", "alphaDetection")}
    for a in sorted(alphas):
        cvw = cv2.addWeighted(x, a, y, 1 - a, 0)
        dsum = (x.astype(np.float64) * a + y.astype(np.float64) * (1 - a)).astype(np.float32)
        assert np.array_equal(cv2.convertScaleAbs(cvw, alpha=255.), cv2.convertScaleAbs(dsum, alpha=255.)), a
