"""TEST INFRASTRUCTURE ONLY - call-for-call replay of the reference plugins with cv2.

The reference's per-pixel arithmetic does not live in /root/reference: every one of the four
IBGS plugins is a thin wrapper over un-vendored OpenCV calls (SURVEY.md section 8c).  This
module replays each wrapper with the OpenCV build that *is* importable in this image
(opencv-python-headless 4.13.0), one cv2 call per reference C++ call, so that the C
restatement in oracle/c/bgs_oracle.c and the CUDA path can be pinned against the library
the reference actually delegates to.

Nothing under tracking_b200/ may import this module (tests/test_layout.py enforces it).
It is used by tests/, by tests/golden/make_golden.py, by __graft_entry__.smoke() and by
bench.py's cpu_baseline / --impl reference legs.

MatExpr lowering (SURVEY.md Appendix A, verified against cv2 4.13 in tests/test_oracle_pin.py):
  a*X + b*Y  -> cv2.addWeighted(X, a, Y, b, 0)
  E + c*Z    -> cv2.scaleAdd(Z, c, E)
  w*X        -> X.convertTo(alpha=w)  == cv2.multiply / numpy fp32 multiply by float32(w)
"""
from __future__ import annotations

import numpy as np
import cv2


def _thr(img, enable, threshold):
    # cv::threshold(src, dst, thr, 255, THRESH_BINARY): dst = src > thr ? 255 : 0
    if not enable:
        return img
    return cv2.threshold(img, threshold, 255, cv2.THRESH_BINARY)[1]


class FrameDifferenceBGS:
    """package_bgs/FrameDifferenceBGS.cpp:29-61."""

    def __init__(self, enableThreshold=True, threshold=15):
        self.enableThreshold, self.threshold = enableThreshold, threshold
        self.prev = None

    def process(self, img):
        if img is None or img.size == 0:          # :31-32
            return None, None
        if self.prev is None:                      # :39-43
            self.prev = img.copy()
            return None, None
        fg = cv2.absdiff(self.prev, img)           # :45
        if fg.ndim == 3 and fg.shape[2] == 3:
            fg = cv2.cvtColor(fg, cv2.COLOR_BGR2GRAY)   # :47-48
        fg = _thr(fg, self.enableThreshold, self.threshold)  # :50-51
        self.prev = img.copy()                     # :58
        return fg, None


class StaticFrameDifferenceBGS:
    """package_bgs/StaticFrameDifferenceBGS.cpp:29-57."""

    def __init__(self, enableThreshold=True, threshold=15):
        self.enableThreshold, self.threshold = enableThreshold, threshold
        self.bg = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        if self.bg is None:                        # :34-35
            self.bg = img.copy()
        fg = cv2.absdiff(img, self.bg)             # :42
        if fg.ndim == 3 and fg.shape[2] == 3:
            fg = cv2.cvtColor(fg, cv2.COLOR_BGR2GRAY)        # :44-45
        fg = _thr(fg, self.enableThreshold, self.threshold)  # :47-48
        return fg, self.bg.copy()                  # :53-54


class WeightedMovingMeanBGS:
    """package_bgs/WeightedMovingMeanBGS.cpp:30-103."""

    def __init__(self, enableWeight=True, enableThreshold=True, threshold=15):
        self.enableWeight, self.enableThreshold, self.threshold = enableWeight, enableThreshold, threshold
        self.p1 = None
        self.p2 = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        if self.p1 is None:                        # :40-44
            self.p1 = img.copy()
            return None, None
        if self.p2 is None:                        # :46-51
            self.p2 = self.p1.copy()
            self.p1 = img.copy()
            return None, None
        s = np.float32(1.0 / 255.0)
        x0 = img.astype(np.float32) * s            # :53-60
        x1 = self.p1.astype(np.float32) * s
        x2 = self.p2.astype(np.float32) * s
        if self.enableWeight:                      # :61-62  (A*.5 + B*.3) -> addWeighted, + C*.2 -> scaleAdd
            bg_f = cv2.scaleAdd(x2, 0.2, cv2.addWeighted(x0, 0.5, x1, 0.3, 0))
        else:                                      # :64     (A + B) -> add, (t + C)/3.0 -> addWeighted(t,1/3.,C,1/3.)
            bg_f = cv2.addWeighted(cv2.add(x0, x1), 1. / 3.0, x2, 1. / 3.0, 0)
        bg = _to_u8(bg_f)                          # :70
        fg = cv2.absdiff(img, bg)                  # :76
        if fg.ndim == 3 and fg.shape[2] == 3:
            fg = cv2.cvtColor(fg, cv2.COLOR_BGR2GRAY)        # :78-79
        fg = _thr(fg, self.enableThreshold, self.threshold)  # :81-82
        self.p2 = self.p1                          # :90-91
        self.p1 = img.copy()
        return fg, bg


class AdaptiveBackgroundLearning:
    """package_bgs/AdaptiveBackgroundLearning.cpp:30-83 (limit == -1 branch; the limit>0
    branch is dead because `counter` only advances inside it, :52,60-61)."""

    def __init__(self, alpha=0.05, enableThreshold=True, threshold=15):
        self.alpha, self.enableThreshold, self.threshold = alpha, enableThreshold, threshold
        self.bg = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        if self.bg is None:                                    # :40-41
            self.bg = img.copy()
        s = 1.0 / 255.0
        in_f = img.astype(np.float32) * np.float32(s)          # convertTo(CV_32F, 1./255.) :43-44
        bg_f = self.bg.astype(np.float32) * np.float32(s)      # :46-47
        diff_f = cv2.absdiff(in_f, bg_f)                       # :49-50
        bg_f = cv2.addWeighted(in_f, self.alpha, bg_f, 1 - self.alpha, 0)   # :54
        new_bg = _to_u8(bg_f)                                  # :56-57
        self.bg = new_bg                                       # :58
        fg = _to_u8(diff_f)                                    # :64-65
        if fg.ndim == 3 and fg.shape[2] == 3:
            fg = cv2.cvtColor(fg, cv2.COLOR_BGR2GRAY)          # :67-68
        fg = _thr(fg, self.enableThreshold, self.threshold)    # :70-71
        return fg, self.bg.copy()                              # :79-80


class AdaptiveSelectiveBackgroundLearning:
    """package_bgs/AdaptiveSelectiveBackgroundLearning.cpp:30-105 (USTC_BGS type 7, ustc_src/ustc_bgs.cpp:15).
    Defaults are those of loadConfig() (:121-125), which runs before the first saveConfig (:43-46) and
    therefore overrides the constructor's threshold 15 / learningFrames -1."""

    def __init__(self, learningFrames=90, alphaLearn=0.05, alphaDetection=0.05, threshold=25):
        self.learningFrames, self.alphaLearn, self.alphaDetection = learningFrames, alphaLearn, alphaDetection
        self.threshold = threshold
        self.counter = 0
        self.bg = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        gray = cv2.cvtColor(img, cv2.COLOR_BGR2GRAY) if img.ndim == 3 else img.copy()   # :36-39
        if self.bg is None:                                    # :47-48
            self.bg = gray.copy()
        s = 1.0 / 255.0
        in_f = gray.astype(np.float32) * np.float32(s)         # :50-51
        bg_f = self.bg.astype(np.float32) * np.float32(s)      # :53-54
        diff_f = cv2.absdiff(in_f, bg_f)                       # :56-57
        fg = _to_u8(diff_f)                                    # :59-60  (255/(maxVal-minVal) = 255, -minVal = -0)
        _, fg = cv2.threshold(fg, self.threshold, 255, cv2.THRESH_BINARY)   # :62
        fg = cv2.medianBlur(fg, 3)                             # :63
        if self.learningFrames > 0 and self.counter <= self.learningFrames:   # :65-71
            bg_f = cv2.addWeighted(in_f, self.alphaLearn, bg_f, 1 - self.alphaLearn, 0)
            self.counter += 1
        else:                                                  # :72-90: double arithmetic, stored to float
            a = float(self.alphaDetection)
            upd = (a * in_f.astype(np.float64) + (1 - a) * bg_f.astype(np.float64)).astype(np.float32)
            bg_f = np.where(fg == 0, upd, bg_f)
        self.bg = _to_u8(bg_f)                                 # :92-94
        return fg, self.bg.copy()                              # :102-103 (single-channel background model)


def _to_u8(img_f):
    """Mat::convertTo(CV_8U, 255.0, 0): saturate_cast<uchar>(x*255) with round-half-even."""
    # cv2 does not expose Mat::convertTo directly; cv2.convertScaleAbs computes
    # saturate_cast<uchar>(|x*alpha+beta|), identical on the non-negative inputs every call
    # site guarantees (absdiff / sqrt / convex blend of non-negative values).
    return cv2.convertScaleAbs(img_f, alpha=255.0, beta=0.0)


class WeightedMovingVarianceBGS:
    """package_bgs/WeightedMovingVarianceBGS.cpp:30-117,126-138."""

    def __init__(self, enableWeight=True, enableThreshold=True, threshold=15):
        self.enableWeight, self.enableThreshold, self.threshold = enableWeight, enableThreshold, threshold
        self.p1 = None
        self.p2 = None

    @staticmethod
    def _wvar(x_f, mean_f, weight):                # computeWeightedVariance :126-138
        d = cv2.absdiff(x_f, mean_f)
        p = cv2.pow(d, 2.0)
        return p * np.float32(weight)              # weight * Mat -> convertTo(alpha=weight)

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        if self.p1 is None:                        # :40-44
            self.p1 = img.copy()
            return None, None
        if self.p2 is None:                        # :46-51
            self.p2 = self.p1.copy()
            self.p1 = img.copy()
            return None, None
        s = np.float32(1.0 / 255.0)
        x0 = img.astype(np.float32) * s            # :53-60
        x1 = self.p1.astype(np.float32) * s
        x2 = self.p2.astype(np.float32) * s
        if self.enableWeight:                      # :66-70
            w = (0.5, 0.3, 0.2)
        else:
            w = (0.3, 0.3, 0.3)
        mean = cv2.scaleAdd(x2, w[2], cv2.addWeighted(x0, w[0], x1, w[1], 0))
        v = self._wvar(x0, mean, w[0]) + self._wvar(x1, mean, w[1])   # :78-91 (left-assoc sum)
        v = v + self._wvar(x2, mean, w[2])
        sd = cv2.sqrt(v)                           # :95
        fg = _to_u8(sd)                            # :99
        if fg.ndim == 3 and fg.shape[2] == 3:
            fg = cv2.cvtColor(fg, cv2.COLOR_BGR2GRAY)   # :102-103
        fg = _thr(fg, self.enableThreshold, self.threshold)  # :105-106
        self.p2 = self.p1                          # :113-114
        self.p1 = img.copy()
        return fg, None


class MixtureOfGaussianV2BGS:
    """package_bgs/MixtureOfGaussianV2BGS.cpp:29-74.  `cv::BackgroundSubtractorMOG2 mog;`
    default-constructed (history 500, varThreshold 16, shadows on) -> cv2.createBackgroundSubtractorMOG2()."""

    # bgsb_set_param keys of the model's own parameters -> cv::BackgroundSubtractorMOG2 setters
    SETTERS = {"history": "setHistory", "varThreshold": "setVarThreshold", "varThresholdGen": "setVarThresholdGen",
               "backgroundRatio": "setBackgroundRatio", "varInit": "setVarInit", "varMin": "setVarMin", "varMax": "setVarMax",
               "complexityReductionThreshold": "setComplexityReductionThreshold", "shadowThreshold": "setShadowThreshold",
               "detectShadows": "setDetectShadows", "shadowValue": "setShadowValue"}

    def __init__(self, alpha=0.05, enableThreshold=True, threshold=15, **model):
        self.alpha, self.enableThreshold, self.threshold = alpha, enableThreshold, threshold
        self.mog = cv2.createBackgroundSubtractorMOG2()
        for k, v in model.items():
            if k == "detectShadows":
                v = bool(v)
            elif k in ("history", "shadowValue"):
                v = int(v)
            getattr(self.mog, self.SETTERS[k])(v)

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        fg = self.mog.apply(img, learningRate=self.alpha)     # :56
        bg = self.mog.getBackgroundImage()                    # :58-59
        fg = _thr(fg, self.enableThreshold, self.threshold)   # :61-62
        return fg, bg


ALGOS = {
    0: FrameDifferenceBGS,            # ustc_src/ustc_bgs.cpp:8
    1: StaticFrameDifferenceBGS,      # ustc_src/ustc_bgs.cpp:9   (sibling plugin, SURVEY 8f N3)
    2: WeightedMovingMeanBGS,         # ustc_src/ustc_bgs.cpp:10  (sibling plugin, SURVEY 8f N3)
    3: WeightedMovingVarianceBGS,     # ustc_src/ustc_bgs.cpp:11
    5: MixtureOfGaussianV2BGS,        # ustc_src/ustc_bgs.cpp:13
    6: AdaptiveBackgroundLearning,    # ustc_src/ustc_bgs.cpp:14
}


# --- stage 2 / 3 ---------------------------------------------------------------------------

def morph(mask, op, iterations=1):
    """cv::erode / cv::dilate(mask, dst, cv::Mat(), Point(-1,-1), iterations): 3x3 rect."""
    if op == "erode":
        return cv2.erode(mask, None, iterations=iterations)
    if op == "dilate":
        return cv2.dilate(mask, None, iterations=iterations)
    raise ValueError(op)


def canonical_labels(mask):
    """8-connected labels numbered by raster-first pixel (SURVEY.md A.6 'Canonical labels')."""
    n, lab = cv2.connectedComponentsWithAlgorithm((mask > 128).astype(np.uint8), 8, cv2.CV_32S, cv2.CCL_WU)
    # canonicalise defensively: renumber by min linear index
    if n > 1:
        h, w = lab.shape
        flat = lab.ravel()
        first = np.full(n, flat.size, np.int64)
        idx = np.nonzero(flat)[0]
        np.minimum.at(first, flat[idx], idx)
        order = np.argsort(first[1:], kind="stable")
        remap = np.zeros(n, np.int32)
        remap[1 + order] = np.arange(1, n, dtype=np.int32)
        lab = remap[lab]
    return n - 1, lab.astype(np.int32)


def external_contour_rects(mask, zero_border):
    """Steps 1-2 of CvBlobDetectorCC::DetectNewBlob (SURVEY.md A.6): threshold 128, then
    cvFindContours(RETR_EXTERNAL); returns bounding rects in the order findContours lists them."""
    ib = cv2.threshold(mask, 128, 255, cv2.THRESH_BINARY)[1]
    if zero_border:        # OpenCV <= 3.1 zeroes the outer 1-px frame before tracing
        ib = ib.copy()
        ib[0, :] = 0; ib[-1, :] = 0; ib[:, 0] = 0; ib[:, -1] = 0
    contours, _ = cv2.findContours(ib, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)
    return [cv2.boundingRect(c) for c in contours], contours
