"""Seeded parameter draws shared by the oracle pins against OpenCV (test_oracle_param_pins.py) and the GPU sweeps against
the oracle (test_gpu_param_space.py), so that every value the restatement is pinned at is also a value the kernels are
compared at.

A MOG2 draw is a dict: "schedule" is a list of (frames, alpha) segments (alpha is the per-call learning rate and may
change between segments), "model" holds cv::BackgroundSubtractorMOG2's own parameters under their bgsb_set_param keys,
plus "enableThreshold" and "threshold" of the wrapper."""
import numpy as np


def scene(rng, n, h, w):
    """noisy background with drifting brightness, a few moving bright / dark blobs, occasional palette flips"""
    base = rng.integers(30, 200, (h, w, 3)).astype(np.int16)
    yy, xx = np.mgrid[0:h, 0:w]
    out = []
    for t in range(n):
        f = base + rng.integers(-4, 5, (h, w, 3)) + int(6 * np.sin(t / 3.0))
        for b in range(3):
            cy, cx = (7 * t + 31 * b) % h, (11 * t + 17 * b) % w
            m = (yy - cy) ** 2 + (xx - cx) ** 2 < (5 + 2 * b) ** 2
            f[m] = (250, 10 + 60 * b, 128) if b != 1 else f[m] // 2            # b == 1: a shadow-like darker copy
        if t % 9 == 8:
            f[:, : w // 3] = base[:, : w // 3][..., ::-1]
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


MOG2_FRAMES = 24              # every schedule covers this many frames; segment edges sit on multiples of 8


def mog2_edge_draws():
    """Named edges: re-initialising rates (alpha >= 1, also inside a stream), varMin > varMax, short histories, rates
    below 1e-4 and an automatic rate over a long history."""
    d = {}

    def add(name, schedule, **model):
        thr = model.pop("enableThreshold", 0)
        d[name] = dict(schedule=schedule, model=model, enableThreshold=thr, threshold=model.pop("threshold", 15))

    add("alpha_1", [(24, 1.0)])
    add("alpha_1.5", [(24, 1.5)])
    add("alpha_3_history_1", [(24, 3.0)], history=1)
    add("alpha_1_history_2", [(24, 1.0)], history=2)
    add("alpha_1_thresholded", [(24, 1.0)], enableThreshold=1, threshold=100)
    add("switch_0.05_1_0.05", [(8, 0.05), (8, 1.0), (8, 0.05)])
    add("switch_1_auto", [(8, 1.0), (16, -1.0)])
    add("switch_1_auto_history_10", [(8, 1.0), (16, -1.0)], history=10)
    add("varMin_gt_varMax", [(24, 0.05)], varMin=50.0, varMax=10.0)
    add("varMin_gt_varMax_wide", [(24, 0.2)], varMin=300.0, varMax=0.5, varInit=40.0)
    add("history_1_auto", [(24, -1.0)], history=1)
    add("history_2_auto", [(24, -1.0)], history=2)
    add("alpha_0", [(24, 0.0)])
    add("alpha_1e-5", [(24, 1e-5)])
    add("alpha_9e-5_varMin_gt_varMax", [(24, 9e-5)], varMin=20.0, varMax=2.0)
    add("auto_history_1e5", [(24, -1.0)], history=100000)
    return d


def random_mog2_draw(rng):
    alphas = [-1.0, 0.0, 1e-5, 1e-4, 1e-3, 0.01, 0.05, 0.2, 0.5, 0.999999, 1.0, 1.5]
    lengths = ([24], [8, 16], [8, 8, 8])[int(rng.integers(0, 3))]
    schedule = [(n, float(rng.choice(alphas))) for n in lengths]
    model = {"history": int(rng.choice([1, 2, 3, 10, 500, 100000])),
             "varThreshold": float(rng.choice([0.0, 1.0, 4.0, 16.0, 64.0, 1000.0])),
             "varThresholdGen": float(rng.choice([0.0, 1.0, 3.0, 9.0, 100.0, 1000.0])),
             "backgroundRatio": float(rng.choice([0.0, 0.3, 0.9, 1.0, 2.0])),
             "varInit": float(rng.choice([0.5, 5.0, 15.0, 100.0, 1000.0])),
             "varMin": float(rng.choice([0.0, 1.0, 4.0, 20.0, 100.0])),
             "varMax": float(rng.choice([1.0, 10.0, 75.0, 500.0])),
             "complexityReductionThreshold": float(rng.choice([0.0, 0.05, 0.5, 5.0])),
             "shadowThreshold": float(rng.choice([0.0, 0.5, 0.9, 1.5])),
             "detectShadows": int(rng.integers(0, 2)),
             "shadowValue": int(rng.choice([0, 1, 127, 255]))}
    return dict(schedule=schedule, model=model, enableThreshold=int(rng.integers(0, 2)),
                threshold=int(rng.choice([0, 1, 126, 127, 200, 254, 255])))


def mog2_draws(n_random=20, seed=4100):
    d = mog2_edge_draws()
    rng = np.random.default_rng(seed)
    for i in range(n_random):
        d["random_%d" % i] = random_mog2_draw(rng)
    return d


def alphas_per_frame(draw):
    out = []
    for n, a in draw["schedule"]:
        out += [a] * n
    assert len(out) == MOG2_FRAMES
    return out


def segments(draw, T):
    """(first frame, frame count, alpha) of the calls that feed a draw in batches of at most T frames; a batch never
    spans a change of alpha (alpha is a per-call parameter)."""
    out, t0 = [], 0
    for n, a in draw["schedule"]:
        for k in range(0, n, T):
            out.append((t0 + k, min(T, n - k), a))
        t0 += n
    return out


# ---- the simpler plugins: (reference class name, keyword draws), the keys being those of bgsb_set_param ----

def simple_draws():
    """FD, StaticFD, WMM, WMV and ABL at threshold edges, with and without the threshold, weighted and not."""
    out = []
    for thr in (0, 1, 127, 254, 255):
        for en in (0, 1):
            out.append(("FrameDifferenceBGS", dict(enableThreshold=en, threshold=thr)))
            out.append(("StaticFrameDifferenceBGS", dict(enableThreshold=en, threshold=thr)))
            for ew in (0, 1):
                out.append(("WeightedMovingMeanBGS", dict(enableWeight=ew, enableThreshold=en, threshold=thr)))
                out.append(("WeightedMovingVarianceBGS", dict(enableWeight=ew, enableThreshold=en, threshold=thr)))
    for alpha in (0.0, 1e-4, 0.05, 0.5, 1.0):
        for thr, en in ((15, 1), (0, 1), (255, 1), (15, 0)):
            out.append(("AdaptiveBackgroundLearning", dict(alpha=alpha, enableThreshold=en, threshold=thr)))
    return out


def asbl_draws(n=24, seed=4200):
    # (no alpha 0.3: there cv2 4.13's float addWeighted rounds 19 of the 65536 byte pairs differently from the
    # restatement's double sum; see test_oracle_param_pins.py)
    rng = np.random.default_rng(seed)
    out = [dict(learningFrames=lf, alphaLearn=al, alphaDetection=ad, threshold=thr)
           for lf, al, ad, thr in ((0, 0.05, 0.05, 25), (-1, 0.5, 0.5, 25), (1, 1.0, 0.0, 0), (5, 0.0, 1.0, 254),
                                   (3, 0.25, 0.7, 255), (100000, 0.05, 0.05, 1))]
    for _ in range(n - len(out)):
        out.append(dict(learningFrames=int(rng.choice([-1, 0, 1, 2, 5, 90])),
                        alphaLearn=float(rng.choice([0.0, 1e-4, 0.05, 0.25, 0.7, 0.999, 1.0])),
                        alphaDetection=float(rng.choice([0.0, 1e-4, 0.05, 0.25, 0.7, 0.999, 1.0])),
                        threshold=int(rng.choice([0, 1, 10, 25, 127, 254, 255]))))
    return out


def dp_draws(seed=4300):
    """DPZivkovic, the four DP models and SigmaDelta: named edges first, then seeded draws.  (class name, kwargs)."""
    rng = np.random.default_rng(seed)
    out = []
    for g in (1, 2, 3, 4, 5):
        out.append(("DPZivkovicAGMMBGS", dict(gaussians=g, threshold=25.0, alpha=0.001)))
    for thr, a in ((0.0, 0.001), (25.0, 0.0), (25.0, 1.0), (1000.0, 0.5), (9.5, 0.05)):
        out.append(("DPZivkovicAGMMBGS", dict(gaussians=int(rng.integers(1, 6)), threshold=thr, alpha=a)))
    for sr in (1, 2, 7, 1000):
        out.append(("DPAdaptiveMedianBGS", dict(threshold=int(rng.choice([0, 10, 40, 255])), samplingRate=sr,
                                                learningFrames=int(rng.choice([0, 1, 30])))))
    for thr, a, lf in ((2700, float(np.float32(1e-6)), 30), (0, 0.5, 0), (100000, 1.0, 1), (300, 0.05, 5)):
        out.append(("DPMeanBGS", dict(threshold=thr, alpha=a, learningFrames=lf)))
    for thr, a, lf in ((12.25, float(np.float32(0.005)), 30), (0.0, 0.5, 0), (1000.0, 1.0, 1), (4.0, 0.05, 5)):
        out.append(("DPWrenGABGS", dict(threshold=thr, alpha=a, learningFrames=lf)))
    for sr, hs in ((1, 1), (1, 64), (1000, 16), (3, 4), (5, 16)):
        out.append(("DPPratiMediodBGS", dict(threshold=int(rng.choice([0, 10, 30, 255])), samplingRate=sr, historySize=hs,
                                             weight=int(rng.choice([1, 5])))))
    for amp, vmin, vmax in ((0, 15, 255), (1, 15, 255), (4, 100, 10), (2, 300, 1000), (16, 0, 0), (1, 2, 300)):
        out.append(("SigmaDeltaBGS", dict(ampFactor=amp, minVar=vmin, maxVar=vmax)))
    return out
