"""TEST INFRASTRUCTURE ONLY - Python face of the C restatement (oracle/c/bgs_oracle.c).

Classes carry the reference's plugin names and `process(img) -> (fg|None, bg|None)`
mirrors `IBGS::process(in, fg, bgModel)` (package_bgs/IBGS.h:24): `None` stands for
"output left untouched" (the reference returns early without writing, e.g.
package_bgs/FrameDifferenceBGS.cpp:39-43).

Only tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs may import this.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "_build", "libbgs_oracle.so")
_lib = None


def build(force=False):
    src = os.path.join(_HERE, "c", "bgs_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-B" if force else "-s"], stdout=subprocess.DEVNULL)
    return _LIB_PATH


class Mog2Params(C.Structure):
    _fields_ = [("K", C.c_int), ("Tb", C.c_float), ("Tg", C.c_float), ("TB", C.c_float),
                ("varInit", C.c_float), ("varMin", C.c_float), ("varMax", C.c_float),
                ("CT", C.c_float), ("tau", C.c_float), ("detect_shadows", C.c_int),
                ("shadow_value", C.c_int), ("history", C.c_int)]


def build_ref(reference=os.environ.get("BGSB_REFERENCE_DIR", "/root/reference")):
    """Compile the reference's own DP-package models and Sigma-Delta library into oracle/_ref/libdp_ref.so (`make ref`) when a
    checkout of the original project is there ($BGSB_REFERENCE_DIR, else /root/reference); returns True if the library exists afterwards."""
    here = os.path.dirname(os.path.abspath(__file__))
    if os.path.exists(os.path.join(reference, "package_bgs", "dp", "ZivkovicAGMM.cpp")):
        subprocess.run(["make", "-C", here, "ref", "REFERENCE=" + reference], check=True, stdout=subprocess.DEVNULL)
    return os.path.exists(os.path.join(here, "_ref", "libdp_ref.so"))


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        u8p, f32p, i32p = C.POINTER(C.c_uint8), C.POINTER(C.c_float), C.POINTER(C.c_int32)
        L.orc_gray_bgr.argtypes = [u8p, C.c_int, C.c_int, u8p]
        L.orc_fd.argtypes = [u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p]
        L.orc_sfd.argtypes = [u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p]
        L.orc_wmm.argtypes = [u8p, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p, u8p]
        L.orc_abl.argtypes = [u8p, u8p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, u8p]
        L.orc_asbl.argtypes = [u8p, u8p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, u8p, u8p]
        L.orc_dpz_apply.argtypes = [u8p, C.c_int, C.c_int, C.c_double, C.c_double, f32p, u8p, u8p]
        L.orc_dp_median.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p, u8p]
        L.orc_dp_mean.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_double, f32p, u8p]
        L.orc_dp_wren.argtypes = [u8p, C.c_int, C.c_int, C.c_double, C.c_double, f32p, u8p]
        L.orc_sigma_delta.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p, u8p, u8p]
        L.orc_dp_prati_subtract.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p, u8p, u8p]
        L.orc_dp_prati_update.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p, i32p, u8p]
        L.orc_wmv.argtypes = [u8p, u8p, u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, u8p]
        L.orc_mog2_default_params.argtypes = [C.POINTER(Mog2Params)]
        L.orc_mog2_learning_rate.argtypes = [C.c_double, C.c_int, C.c_int]
        L.orc_mog2_learning_rate.restype = C.c_double
        L.orc_mog2_apply.argtypes = [u8p, C.c_int, C.c_double, C.POINTER(Mog2Params), f32p, f32p, u8p, u8p]
        L.orc_mog2_background.argtypes = [C.c_int, C.POINTER(Mog2Params), f32p, f32p, u8p, u8p]
        L.orc_morph3x3.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, u8p]
        L.orc_ccl8.argtypes = [u8p, C.c_int, C.c_int, C.c_int, i32p, C.c_int, i32p, u8p]
        L.orc_ccl8.restype = C.c_int
        L.orc_rect_moments.argtypes = [u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.POINTER(C.c_uint64)]
        L.orc_synth_frame.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint32, u8p]
        L.orc_synth_churn_frame.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint32, u8p]
        _lib = L
    return _lib


def _u8(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def _f32(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _dense(img):
    img = np.ascontiguousarray(img, dtype=np.uint8)
    assert img.ndim == 3 and img.shape[2] == 3, "plugins take BGR 8UC3 (PreProcessor.cpp:56)"
    return img


def gray_bgr(img, variant=0):
    img = _dense(img)
    out = np.empty(img.shape[:2], np.uint8)
    lib().orc_gray_bgr(_u8(img), out.size, variant, _u8(out))
    return out


class FrameDifferenceBGS:
    def __init__(self, enableThreshold=True, threshold=15, gray_variant=0):
        self.enableThreshold, self.threshold, self.gray_variant = enableThreshold, threshold, gray_variant
        self.prev = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        if self.prev is None:
            self.prev = img.copy()
            return None, None
        fg = np.empty(img.shape[:2], np.uint8)
        lib().orc_fd(_u8(self.prev), _u8(img), fg.size, int(self.enableThreshold), self.threshold,
                     self.gray_variant, _u8(fg))
        self.prev = img.copy()
        return fg, None


class StaticFrameDifferenceBGS:
    """package_bgs/StaticFrameDifferenceBGS.cpp:29-57 (sibling plugin, SURVEY 8f N3)."""

    def __init__(self, enableThreshold=True, threshold=15, gray_variant=0):
        self.enableThreshold, self.threshold, self.gray_variant = enableThreshold, threshold, gray_variant
        self.bg = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        if self.bg is None:
            self.bg = img.copy()
        fg = np.empty(img.shape[:2], np.uint8)
        lib().orc_sfd(_u8(self.bg), _u8(img), fg.size, int(self.enableThreshold), self.threshold,
                      self.gray_variant, _u8(fg))
        return fg, self.bg.copy()


class WeightedMovingMeanBGS:
    """package_bgs/WeightedMovingMeanBGS.cpp:30-103 (sibling plugin, SURVEY 8f N3)."""

    def __init__(self, enableWeight=True, enableThreshold=True, threshold=15, gray_variant=0):
        self.enableWeight, self.enableThreshold, self.threshold = enableWeight, enableThreshold, threshold
        self.gray_variant = gray_variant
        self.p1 = None
        self.p2 = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        if self.p1 is None:
            self.p1 = img.copy()
            return None, None
        if self.p2 is None:
            self.p2 = self.p1
            self.p1 = img.copy()
            return None, None
        fg = np.empty(img.shape[:2], np.uint8)
        bg = np.empty(img.shape, np.uint8)
        lib().orc_wmm(_u8(img), _u8(self.p1), _u8(self.p2), fg.size, int(self.enableWeight),
                      int(self.enableThreshold), self.threshold, self.gray_variant, _u8(fg), _u8(bg))
        self.p2 = self.p1
        self.p1 = img.copy()
        return fg, bg


class AdaptiveBackgroundLearning:
    def __init__(self, alpha=0.05, enableThreshold=True, threshold=15, gray_variant=0):
        self.alpha, self.enableThreshold, self.threshold = alpha, enableThreshold, threshold
        self.gray_variant = gray_variant
        self.bg = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        if self.bg is None:
            self.bg = img.copy()
        fg = np.empty(img.shape[:2], np.uint8)
        lib().orc_abl(_u8(img), _u8(self.bg), fg.size, float(self.alpha), int(self.enableThreshold),
                      self.threshold, self.gray_variant, _u8(fg))
        return fg, self.bg.copy()


def abl_blend_table_24(alpha):
    """PARITY UNPINNED (no OpenCV 2.4 in this image).  New background byte of AdaptiveBackgroundLearning for every
    (input byte x = row, background byte y = column) as OpenCV 2.4 computes `alpha*in_f + (1-alpha)*bg_f`
    (AdaptiveBackgroundLearning.cpp:54): addWeighted on CV_32F in fp32 with the scalars cast to float (SURVEY
    Appendix B), then convertTo(CV_8U, 255) = round-half-even + saturate (:56-58)."""
    x = (np.arange(256, dtype=np.float32) * np.float32(1. / 255.))[:, None]
    y = (np.arange(256, dtype=np.float32) * np.float32(1. / 255.))[None, :]
    a, b = np.float32(alpha), np.float32(1. - alpha)
    nb = (x * a).astype(np.float32) + (y * b).astype(np.float32)
    return np.clip(np.rint(nb.astype(np.float32) * np.float32(255.)), 0, 255).astype(np.uint8)


class AdaptiveSelectiveBackgroundLearning:
    """USTC_BGS type 7; defaults = loadConfig()'s (AdaptiveSelectiveBackgroundLearning.cpp:121-125)."""

    def __init__(self, learningFrames=90, alphaLearn=0.05, alphaDetection=0.05, threshold=25, gray_variant=0):
        self.learningFrames, self.alphaLearn, self.alphaDetection = learningFrames, alphaLearn, alphaDetection
        self.threshold, self.gray_variant = threshold, gray_variant
        self.counter = 0
        self.bg = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        if self.bg is None:
            self.bg = np.empty((h, w), np.uint8)
            lib().orc_gray_bgr(_u8(img), h * w, self.gray_variant, _u8(self.bg))
        learning = self.learningFrames > 0 and self.counter <= self.learningFrames
        if learning:
            self.counter += 1
        fg = np.empty((h, w), np.uint8)
        scratch = np.empty(2 * h * w, np.uint8)
        lib().orc_asbl(_u8(img), _u8(self.bg), w, h, float(self.alphaLearn if learning else self.alphaDetection),
                       0 if learning else 1, int(self.threshold), self.gray_variant, _u8(fg), _u8(scratch))
        return fg, self.bg.copy()


class DPZivkovicAGMMBGS:
    """USTC_BGS type 11 (package_bgs/dp/DPZivkovicAGMMBGS.cpp); defaults of its loadConfig (:97-100).
    Never writes img_bgmodel."""

    def __init__(self, threshold=25.0, alpha=0.001, gaussians=3):
        self.threshold, self.alpha, self.gaussians = threshold, alpha, gaussians
        self.modes = None
        self.nmodes = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        if self.modes is None:                               # InitModel: everything zero (ZivkovicAGMM.cpp:77-91)
            self.modes = np.zeros((h * w, self.gaussians, 5), np.float32)
            self.nmodes = np.zeros(h * w, np.uint8)
        fg = np.empty((h, w), np.uint8)
        lib().orc_dpz_apply(_u8(img), h * w, self.gaussians, float(self.threshold), float(self.alpha),
                            self.modes.ctypes.data_as(C.POINTER(C.c_float)), _u8(self.nmodes), _u8(fg))
        return fg, None


class ReferenceDPZivkovic:
    """The reference's own ZivkovicAGMM class, compiled from the original project's sources by `make -C oracle ref`
    (oracle/_ref/libdp_ref.so).  Raises FileNotFoundError when that build is absent."""

    def __init__(self, w, h, threshold=25.0, alpha=0.001, gaussians=3):
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "libdp_ref.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.L = C.CDLL(path)
        self.L.dpz_ref_create.restype = C.c_void_p
        self.L.dpz_ref_create.argtypes = [C.c_int, C.c_int, C.c_double, C.c_double, C.c_int]
        self.L.dpz_ref_process.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
        self.L.dpz_ref_destroy.argtypes = [C.c_void_p]
        self.w, self.h = w, h
        self.p = self.L.dpz_ref_create(w, h, float(threshold), float(alpha), int(gaussians))

    def process(self, img):
        img = _dense(img)
        fg = np.empty((self.h, self.w), np.uint8)
        self.L.dpz_ref_process(self.p, _u8(img), _u8(fg))
        return fg, None

    def close(self):
        if self.p:
            self.L.dpz_ref_destroy(self.p)
            self.p = None


class DPAdaptiveMedianBGS:
    """USTC_BGS type 9 (package_bgs/dp/DPAdaptiveMedianBGS.cpp); defaults of its loadConfig (:101-104).  Never writes
    img_bgmodel.  `learningFrames` has no effect: the wrapper clears the low mask before Update (:69-70)."""

    def __init__(self, threshold=40, samplingRate=7, learningFrames=30):
        self.threshold, self.samplingRate, self.learningFrames = threshold, samplingRate, learningFrames
        self.median = None
        self.frame = 0

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        first = self.median is None
        if first:                                            # parameters are handed over once (:56-59)
            self.median = np.zeros((h, w, 3), np.uint8)
            self._thr, self._rate = int(self.threshold), int(self.samplingRate)
        fg = np.empty((h, w), np.uint8)
        lib().orc_dp_median(_u8(img), h * w, int(first), self.frame, self._thr, self._rate, _u8(self.median), _u8(fg))
        self.frame += 1
        return fg, None


class DPMeanBGS:
    """USTC_BGS type 12 (package_bgs/dp/DPMeanBGS.cpp); defaults of its loadConfig (:103-106)."""

    def __init__(self, threshold=2700, alpha=float(np.float32(1e-6)), learningFrames=30):
        self.threshold, self.alpha, self.learningFrames = threshold, alpha, learningFrames
        self.mean = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        first = self.mean is None
        if first:
            self.mean = np.zeros((h, w, 3), np.float32)
            self._thr, self._alpha = int(self.threshold), float(self.alpha)
        fg = np.empty((h, w), np.uint8)
        lib().orc_dp_mean(_u8(img), h * w, int(first), self._thr, self._alpha, self.mean.ctypes.data_as(C.POINTER(C.c_float)), _u8(fg))
        return fg, None


class DPWrenGABGS:
    """USTC_BGS type 13 (package_bgs/dp/DPWrenGABGS.cpp); defaults of its loadConfig (:103-106)."""

    def __init__(self, threshold=12.25, alpha=float(np.float32(0.005)), learningFrames=30):
        self.threshold, self.alpha, self.learningFrames = threshold, alpha, learningFrames
        self.state = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        first = self.state is None
        if first:
            self.state = np.zeros((h, w, 4), np.float32)     # mu[3], var[0]
            self._thr, self._alpha = float(self.threshold), float(self.alpha)
        fg = np.empty((h, w), np.uint8)
        lib().orc_dp_wren(_u8(img), h * w, int(first), self._thr, self._alpha, self.state.ctypes.data_as(C.POINTER(C.c_float)), _u8(fg))
        return fg, None


class DPPratiMediodBGS:
    """USTC_BGS type 14 (package_bgs/dp/DPPratiMediodBGS.cpp); defaults of its loadConfig (:104-108)."""

    def __init__(self, threshold=30, samplingRate=5, historySize=16, weight=5):
        self.threshold, self.samplingRate, self.historySize, self.weight = threshold, samplingRate, historySize, weight
        self.samples = None
        self.frame = 0

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        if self.samples is None:                             # parameters are handed over once (:57-62)
            self._thr, self._rate, self._H = int(self.threshold), int(self.samplingRate), int(self.historySize)
            self.samples = np.zeros((self._H, h, w, 3), np.uint8)
            self.dist = np.zeros((self._H, h, w), np.int32)
            self.median = np.zeros((h, w, 3), np.uint8)
            self.n, self.pos = 0, 0
        fg = np.empty((h, w), np.uint8)
        scratch = np.empty(2 * h * w, np.uint8)
        lib().orc_dp_prati_subtract(_u8(img), w, h, self.frame, self._thr, self._H, _u8(self.median), _u8(fg), _u8(scratch))
        if self.frame % self._rate == 0:
            lib().orc_dp_prati_update(_u8(img), h * w, self.n, self.pos, self._H, _u8(self.samples),
                                      self.dist.ctypes.data_as(C.POINTER(C.c_int32)), _u8(self.median))
            if self.n == self._H:
                self.pos = (self.pos + 1) % self._H
            else:
                self.n += 1
                self.pos = 0
        self.frame += 1
        return fg, None


class SigmaDeltaBGS:
    """USTC_BGS type 35 (package_bgs/bl/SigmaDeltaBGS.cpp); defaults of its loadConfig (:68-70).  The first frame only
    initialises the model (no outputs); parameters are applied before every frame; never writes img_bgmodel."""

    def __init__(self, ampFactor=1, minVar=15, maxVar=255):
        self.ampFactor, self.minVar, self.maxVar = ampFactor, minVar, maxVar
        self.Mt = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        h, w = img.shape[:2]
        first = self.Mt is None
        if first:
            self.Mt = np.zeros((h, w, 3), np.uint8)
            self.Vt = np.zeros((h, w, 3), np.uint8)
        fg = np.empty((h, w), np.uint8)
        lib().orc_sigma_delta(_u8(img), w, h, int(first), int(self.ampFactor), int(self.minVar), int(self.maxVar),
                              _u8(self.Mt), _u8(self.Vt), _u8(fg))
        return (None, None) if first else (fg, None)


class ReferenceSigmaDelta:
    """The reference's own sdLaMa091 implementation (oracle/_ref/libdp_ref.so, oracle/ref_dp/sd_ref.cpp), driven as
    SigmaDeltaBGS::process does.  Raises FileNotFoundError / AttributeError when that build is absent or older."""

    def __init__(self, w, h, ampFactor=1, minVar=15, maxVar=255):
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "libdp_ref.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.L = C.CDLL(path)
        self.L.sd_ref_create.restype = C.c_void_p
        self.L.sd_ref_create.argtypes = [C.c_int, C.c_int]
        self.L.sd_ref_process.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8), C.c_int, C.c_int, C.c_int]
        self.L.sd_ref_destroy.argtypes = [C.c_void_p]
        self.w, self.h = w, h
        self.ampFactor, self.minVar, self.maxVar = ampFactor, minVar, maxVar
        self.p = self.L.sd_ref_create(w, h)

    def process(self, img):
        img = _dense(img)
        fg = np.empty((self.h, self.w), np.uint8)
        ok = self.L.sd_ref_process(self.p, _u8(img), _u8(fg), int(self.ampFactor), int(self.minVar), int(self.maxVar))
        return (fg, None) if ok else (None, None)

    def close(self):
        if self.p:
            self.L.sd_ref_destroy(self.p)
            self.p = None


class ReferenceDPSimple:
    """The reference's own AdaptiveMedianBGS / MeanBGS / WrenGA / PratiMediodBGS classes ("median" / "mean" / "wren" / "prati"), compiled from
    the original project's sources by `make -C oracle ref` (oracle/_ref/libdp_ref.so) and driven as their DP*BGS::process wrappers do.
    Raises FileNotFoundError when that build is absent."""

    def __init__(self, kind, w, h, *params):
        path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref", "libdp_ref.so")
        if not os.path.exists(path):
            raise FileNotFoundError(path)
        self.L = C.CDLL(path)
        pre = {"median": "dpmed", "mean": "dpmean", "wren": "dpwren", "prati": "dpprati"}[kind]
        sig = {"median": [C.c_int, C.c_int, C.c_int], "mean": [C.c_int, C.c_double, C.c_int], "wren": [C.c_double, C.c_double, C.c_int],
               "prati": [C.c_int, C.c_int, C.c_int, C.c_int]}[kind]
        self._create, self._process, self._destroy = (getattr(self.L, pre + "_ref_" + n) for n in ("create", "process", "destroy"))
        self._create.restype = C.c_void_p
        self._create.argtypes = [C.c_int, C.c_int] + sig
        self._process.argtypes = [C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8)]
        self._destroy.argtypes = [C.c_void_p]
        self.w, self.h = w, h
        self.p = self._create(w, h, *params)

    def process(self, img):
        img = _dense(img)
        fg = np.empty((self.h, self.w), np.uint8)
        self._process(self.p, _u8(img), _u8(fg))
        return fg, None

    def close(self):
        if self.p:
            self._destroy(self.p)
            self.p = None


class WeightedMovingVarianceBGS:
    def __init__(self, enableWeight=True, enableThreshold=True, threshold=15, gray_variant=0):
        self.enableWeight, self.enableThreshold, self.threshold = enableWeight, enableThreshold, threshold
        self.gray_variant = gray_variant
        self.p1 = None
        self.p2 = None

    def process(self, img):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        if self.p1 is None:
            self.p1 = img.copy()
            return None, None
        if self.p2 is None:
            self.p2 = self.p1
            self.p1 = img.copy()
            return None, None
        fg = np.empty(img.shape[:2], np.uint8)
        lib().orc_wmv(_u8(img), _u8(self.p1), _u8(self.p2), fg.size, int(self.enableWeight),
                      int(self.enableThreshold), self.threshold, self.gray_variant, _u8(fg))
        self.p2 = self.p1
        self.p1 = img.copy()
        return fg, None


class MixtureOfGaussianV2BGS:
    """MOG2 wrapper (package_bgs/MixtureOfGaussianV2BGS.cpp:56-62) over orc_mog2_*."""

    # bgsb_set_param keys of the model's own parameters -> orc_mog2_params fields
    KEYS = {"varThreshold": "Tb", "varThresholdGen": "Tg", "backgroundRatio": "TB", "varInit": "varInit", "varMin": "varMin",
            "varMax": "varMax", "complexityReductionThreshold": "CT", "shadowThreshold": "tau", "detectShadows": "detect_shadows",
            "shadowValue": "shadow_value", "history": "history"}

    def __init__(self, alpha=0.05, enableThreshold=True, threshold=15, **model):
        self.alpha, self.enableThreshold, self.threshold = alpha, enableThreshold, threshold
        self.params = Mog2Params()
        lib().orc_mog2_default_params(C.byref(self.params))
        for k, v in model.items():
            field = self.KEYS[k]
            setattr(self.params, field, type(getattr(self.params, field))(v))
        self.nframes = 0
        self.shape = None

    def _init(self, shape):
        h, w = shape
        K = self.params.K
        self.shape = shape
        self.gmm = np.zeros((h * w, K, 2), np.float32)
        self.mean = np.zeros((h * w, K, 3), np.float32)
        self.nmodes = np.zeros(h * w, np.uint8)
        self.nframes = 0

    def process(self, img, want_raw=False):
        if img is None or img.size == 0:
            return None, None
        img = _dense(img)
        if self.shape != img.shape[:2] or self.alpha >= 1:   # apply(): needToInitialize on a size change or learningRate >= 1
            self._init(img.shape[:2])
        self.nframes += 1
        lr = lib().orc_mog2_learning_rate(float(self.alpha), self.nframes, self.params.history)
        npx = img.shape[0] * img.shape[1]
        raw = np.empty(img.shape[:2], np.uint8)
        lib().orc_mog2_apply(_u8(img), npx, lr, C.byref(self.params), _f32(self.gmm), _f32(self.mean),
                             _u8(self.nmodes), _u8(raw))
        bg = np.empty(img.shape, np.uint8)
        lib().orc_mog2_background(npx, C.byref(self.params), _f32(self.gmm), _f32(self.mean),
                                  _u8(self.nmodes), _u8(bg))
        fg = raw
        if self.enableThreshold:
            fg = np.where(raw > self.threshold, 255, 0).astype(np.uint8)
        if want_raw:
            return fg, bg, raw
        return fg, bg


ALGOS = {0: FrameDifferenceBGS, 1: StaticFrameDifferenceBGS, 2: WeightedMovingMeanBGS,
         3: WeightedMovingVarianceBGS, 5: MixtureOfGaussianV2BGS,
         6: AdaptiveBackgroundLearning, 7: AdaptiveSelectiveBackgroundLearning,
         9: DPAdaptiveMedianBGS, 11: DPZivkovicAGMMBGS, 12: DPMeanBGS, 13: DPWrenGABGS,
         14: DPPratiMediodBGS, 35: SigmaDeltaBGS}   # ids of ustc_src/ustc_bgs.cpp:8-25


def morph(mask, op, iterations=1):
    mask = np.ascontiguousarray(mask, np.uint8)
    out = np.empty_like(mask)
    h, w = mask.shape
    lib().orc_morph3x3(_u8(mask), w, h, {"erode": 0, "dilate": 1}[op], iterations, _u8(out))
    return out


def ccl8(mask, zero_border=False):
    """-> (n, labels int32 HxW, stats n x 6 [xmin,ymin,xmax,ymax,area,first_idx], external n)"""
    mask = np.ascontiguousarray(mask, np.uint8)
    h, w = mask.shape
    labels = np.empty((h, w), np.int32)
    cap = h * w // 2 + 2
    stats = np.zeros((cap, 6), np.int32)
    ext = np.zeros(cap, np.uint8)
    n = lib().orc_ccl8(_u8(mask), w, h, int(zero_border), labels.ctypes.data_as(C.POINTER(C.c_int32)), cap,
                       stats.ctypes.data_as(C.POINTER(C.c_int32)), _u8(ext))
    return n, labels, stats[:n].copy(), ext[:n].copy()


def rect_moments(img, rect):
    img = np.ascontiguousarray(img, np.uint8)
    h, w = img.shape
    out = (C.c_uint64 * 6)()
    x, y, rw, rh = rect
    lib().orc_rect_moments(_u8(img), w, h, x, y, rw, rh, out)
    return [int(v) for v in out]


def synth_frame(w, h, t, seed):
    out = np.empty((h, w, 3), np.uint8)
    lib().orc_synth_frame(w, h, t, seed & 0xFFFFFFFF, _u8(out))
    return out


def synth_churn_frame(w, h, t, seed):
    out = np.empty((h, w, 3), np.uint8)
    lib().orc_synth_churn_frame(w, h, t, seed & 0xFFFFFFFF, _u8(out))
    return out
