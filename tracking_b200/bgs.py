"""Host-side mirror of the reference's plugin interface, on top of the C ABI.

Same class names, parameter names and early-return behaviour as the reference plugins
(package_bgs/{FrameDifferenceBGS,AdaptiveBackgroundLearning,WeightedMovingVarianceBGS,
MixtureOfGaussianV2BGS}.cpp) so that parity tests read like reference usage:

    bgs = MixtureOfGaussianV2BGS()
    fg, bgmodel = bgs.process(frame_bgr)       # IBGS::process(in, fg, bgModel), IBGS.h:24

`None` for an output means "left untouched" (the reference returns before copyTo, e.g.
FrameDifferenceBGS.cpp:39-43).  All arithmetic happens in CUDA kernels behind libbgsb200.so;
this module only moves numpy / torch buffers across ctypes.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


def yuv_frame(img, fmt, nstreams=1):
    """Check a YUV 4:2:0 frame for "inputFormat" fmt (capi.INPUT_NV12 / INPUT_I420): the (3h/2, w) uint8 image that
    cv::cvtColor reads, with a leading stream axis for a group.  -> (array with unit-stride rows, h, w, grouped); NV12
    rows may be padded (the row stride is passed on), I420 planes are made dense."""
    if fmt not in (capi.INPUT_NV12, capi.INPUT_I420):
        raise ValueError("inputFormat %r is not a YUV format" % (fmt,))
    img = np.asarray(img)
    grouped = img.ndim == 3
    if img.dtype != np.uint8 or img.ndim not in (2, 3):
        raise ValueError("YUV 4:2:0 input takes (3h/2, w) uint8 frames (a stream group: (nstreams, 3h/2, w))")
    if grouped and img.shape[0] != nstreams:
        raise ValueError("expected %d frames" % nstreams)
    if not grouped and nstreams != 1:
        raise ValueError("stream group needs [nstreams, 3h/2, w]")
    rows, w = img.shape[-2], img.shape[-1]
    if rows == 0 or w == 0 or rows % 3 or w % 2:         # (3h/2 rows: h = 2 rows / 3 is even whenever 3 divides rows)
        raise ValueError("YUV 4:2:0 frames have 3h/2 rows of w bytes with w and h even (got %d x %d)" % (rows, w))
    h = 2 * rows // 3
    dense = img.strides[-1] == 1 and (fmt == capi.INPUT_NV12 or img.strides[-2] == w)
    if not dense or (grouped and img.strides[0] != img.strides[1] * rows):
        img = np.ascontiguousarray(img)
    return img, h, w, grouped


class _Plugin:
    ALGO = None
    PARAMS = ()
    BG_CHANNELS = 3            # channels of img_bgmodel (AdaptiveSelectiveBackgroundLearning: 1)
    input_format = capi.INPUT_BGR     # "inputFormat": the layout process / submit / process_fanout take

    def __init__(self, device=0, nstreams=1, **params):
        self._h = C.c_void_p()
        self.device, self.nstreams = device, nstreams
        capi.check(capi.lib().bgsb_create_group(C.byref(self._h), self.ALGO, device, nstreams))
        for k, v in params.items():
            self.set(k, v)

    # -- parameters: XML key names of saveConfig/loadConfig ---------------------------------
    def set(self, key, value):
        capi.check(capi.lib().bgsb_set_param(self._h, key.encode(), float(value)))
        if key == "inputFormat":
            self.input_format = int(value)

    def get(self, key):
        v = C.c_double()
        capi.check(capi.lib().bgsb_get_param(self._h, key.encode(), C.byref(v)))
        return v.value

    def reset(self):
        capi.check(capi.lib().bgsb_reset(self._h))

    @property
    def frame_count(self):
        n = C.c_int64()
        capi.check(capi.lib().bgsb_frame_count(self._h, C.byref(n)))
        return n.value

    def close(self):
        if self._h:
            capi.lib().bgsb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- IBGS::process, host buffers -------------------------------------------------------
    def process(self, img_input, want_bg=True):
        """img_input: HxWx3 uint8 BGR (a group takes nstreams x H x W x 3); with "inputFormat" NV12 / I420 the
        (3h/2) x W YUV image (a group: nstreams x 3h/2 x W).  Returns (img_output | None, img_bgmodel | None)."""
        if img_input is None or img_input.size == 0:      # `if(img_input.empty()) return;`
            return None, None
        if self.input_format != capi.INPUT_BGR:
            img, h, w, grouped = yuv_frame(img_input, self.input_format, self.nstreams)
            stride = img.strides[-2]
        else:
            img = np.asarray(img_input)
            if img.dtype != np.uint8 or img.shape[-1] != 3:
                raise ValueError("plugins take BGR 8UC3 frames")
            grouped = img.ndim == 4
            if grouped and img.shape[0] != self.nstreams:
                raise ValueError("expected %d frames" % self.nstreams)
            if not grouped and self.nstreams != 1:
                raise ValueError("stream group needs [nstreams,H,W,3]")
            h, w = img.shape[-3], img.shape[-2]
            if img.strides[-1] != 1 or img.strides[-2] != 3 or (grouped and img.strides[0] != img.strides[1] * h):
                img = np.ascontiguousarray(img)
            stride = img.strides[-3]
        lead = (self.nstreams,) if grouped else ()
        fg = np.empty(lead + (h, w), np.uint8)
        bgshape = (h, w, 3) if self.BG_CHANNELS == 3 else (h, w)
        bg = np.empty(lead + bgshape, np.uint8) if want_bg else None
        fv, bv = C.c_int(0), C.c_int(0)
        capi.check(capi.lib().bgsb_process(self._h, _ptr(img), w, h, stride, _ptr(fg), w,
                                           _ptr(bg) if bg is not None else None, self.BG_CHANNELS * w,
                                           C.byref(fv), C.byref(bv)))
        return (fg if fv.value else None), (bg if bv.value else None)

    # -- pipelined ingest (capture loop) ----------------------------------------------------------
    def submit(self, img_input, fg_out, bg_out=None):
        """Queue one frame (bgsb_submit): like process(), but returns once the work is enqueued; the upload of the
        next frame overlaps this frame's download.  img_input / fg_out / bg_out are caller-owned C-contiguous uint8
        arrays (page-locked ones from pinned_empty() to really overlap) that must stay untouched until wait().
        With "inputFormat" NV12 / I420, img_input is the C-contiguous (3h/2) x W YUV image.
        Returns (fg_valid, bg_valid): whether fg_out / bg_out will be written for this frame."""
        img = np.asarray(img_input)
        if self.input_format != capi.INPUT_BGR:
            if img.ndim != 2 or not img.flags.c_contiguous:
                raise ValueError("submit takes one C-contiguous (3h/2, w) YUV 4:2:0 frame")
            img, h, w, _ = yuv_frame(img, self.input_format)
            stride = w
        else:
            if img.dtype != np.uint8 or img.ndim != 3 or img.shape[-1] != 3 or not img.flags.c_contiguous:
                raise ValueError("submit takes one C-contiguous BGR 8UC3 frame")
            h, w = img.shape[:2]
            stride = w * 3
        if fg_out.dtype != np.uint8 or fg_out.shape != (h, w) or not fg_out.flags.c_contiguous:
            raise ValueError("fg_out must be a C-contiguous HxW uint8 array")
        bgshape = (h, w, 3) if self.BG_CHANNELS == 3 else (h, w)
        if bg_out is not None and (bg_out.dtype != np.uint8 or bg_out.shape != bgshape or not bg_out.flags.c_contiguous):
            raise ValueError("bg_out must be a C-contiguous uint8 array of shape %r" % (bgshape,))
        fv, bv = C.c_int(0), C.c_int(0)
        capi.check(capi.lib().bgsb_submit(self._h, _ptr(img), w, h, stride, _ptr(fg_out), w,
                                          _ptr(bg_out) if bg_out is not None else None, self.BG_CHANNELS * w,
                                          C.byref(fv), C.byref(bv)))
        self._keep = getattr(self, "_keep", [])
        self._keep.append((img, fg_out, bg_out))          # the arrays outlive the queued copies
        return bool(fv.value), bool(bv.value)

    def wait(self):
        """All submitted frames' outputs are in their arrays (bgsb_wait)."""
        capi.check(capi.lib().bgsb_wait(self._h))
        self._keep = []

    # -- device buffers (torch tensors or raw pointers) -----------------------------------------
    def process_dev(self, d_bgr, w, h, d_fg, d_bg=None, stream=0):
        """d_bgr: device pointer to [nstreams][h][w][3] (with "inputFormat" NV12 / I420: [nstreams][3h/2][w])."""
        fv, bv = C.c_int(0), C.c_int(0)
        capi.check(capi.lib().bgsb_process_dev(self._h, C.c_void_p(d_bgr), w, h, C.c_void_p(d_fg),
                                               C.c_void_p(d_bg) if d_bg else None,
                                               C.byref(fv), C.byref(bv), C.c_void_p(stream)))
        return bool(fv.value), bool(bv.value)

    def process_batch_dev(self, d_frames, T, w, h, d_fg, d_bg=None, bg_last_only=False, stream=0):
        """d_frames: device pointer to [nstreams][T][h][w][3] (with "inputFormat" NV12 / I420: [nstreams][T][3h/2][w])."""
        first, bv = C.c_int(0), C.c_int(0)
        capi.check(capi.lib().bgsb_process_batch_dev(self._h, C.c_void_p(d_frames), T, w, h, C.c_void_p(d_fg),
                                                     C.c_void_p(d_bg) if d_bg else None, int(bg_last_only),
                                                     C.byref(first), C.byref(bv), C.c_void_p(stream)))
        return first.value, bool(bv.value)

    def trace_last(self):
        """Stage times of the last traced process() call (set("trace", 1) first): dict of ms."""
        t = capi.Trace()
        capi.check(capi.lib().bgsb_trace_last(self._h, C.byref(t)))
        return dict(frame=t.frame, wall_ms=t.wall_ms, upload_ms=t.upload_ms, kernel_ms=t.kernel_ms,
                    download_ms=t.download_ms, bands=t.bands)

    def state_bytes(self):
        n = C.c_size_t()
        capi.check(capi.lib().bgsb_state_bytes(self._h, C.byref(n)))
        return n.value


class FrameDifferenceBGS(_Plugin):
    """package_bgs/FrameDifferenceBGS.cpp; keys enableThreshold, threshold (:78-80)."""
    ALGO = capi.ALGO_FRAME_DIFFERENCE


class StaticFrameDifferenceBGS(_Plugin):
    """package_bgs/StaticFrameDifferenceBGS.cpp (sibling plugin, SURVEY 8f N3); keys enableThreshold, threshold."""
    ALGO = capi.ALGO_STATIC_FRAME_DIFFERENCE


class WeightedMovingMeanBGS(_Plugin):
    """package_bgs/WeightedMovingMeanBGS.cpp (sibling plugin, SURVEY 8f N3); keys enableWeight, enableThreshold, threshold."""
    ALGO = capi.ALGO_WEIGHTED_MOVING_MEAN


class WeightedMovingVarianceBGS(_Plugin):
    """package_bgs/WeightedMovingVarianceBGS.cpp; keys enableWeight, enableThreshold, threshold (:155-158)."""
    ALGO = capi.ALGO_WEIGHTED_MOVING_VARIANCE


class AdaptiveBackgroundLearning(_Plugin):
    """package_bgs/AdaptiveBackgroundLearning.cpp; keys alpha, limit, enableThreshold, threshold (:103-108)."""
    ALGO = capi.ALGO_ADAPTIVE_BG_LEARNING


class AdaptiveSelectiveBackgroundLearning(_Plugin):
    """package_bgs/AdaptiveSelectiveBackgroundLearning.cpp (USTC_BGS type 7); keys learningFrames, alphaLearn,
    alphaDetection, threshold (:108-126).  Gray model: img_bgmodel is single-channel."""
    ALGO = capi.ALGO_ADAPTIVE_SELECTIVE_BG_LEARNING
    BG_CHANNELS = 1


class DPZivkovicAGMMBGS(_Plugin):
    """package_bgs/dp/DPZivkovicAGMMBGS.cpp (USTC_BGS type 11): the reference's own Zivkovic adaptive GMM; keys
    threshold, alpha, gaussians (:86-100).  Never writes img_bgmodel."""
    ALGO = capi.ALGO_DP_ZIVKOVIC_AGMM


class DPAdaptiveMedianBGS(_Plugin):
    """package_bgs/dp/DPAdaptiveMedianBGS.cpp (USTC_BGS type 9): McFarlane & Schofield's adaptive median; keys threshold,
    samplingRate, learningFrames (:88-104).  Never writes img_bgmodel."""
    ALGO = capi.ALGO_DP_ADAPTIVE_MEDIAN


class DPMeanBGS(_Plugin):
    """package_bgs/dp/DPMeanBGS.cpp (USTC_BGS type 12): temporal mean; keys threshold, alpha, learningFrames (:86-106).
    Never writes img_bgmodel."""
    ALGO = capi.ALGO_DP_MEAN


class DPWrenGABGS(_Plugin):
    """package_bgs/dp/DPWrenGABGS.cpp (USTC_BGS type 13): Wren's single Gaussian per pixel; keys threshold, alpha,
    learningFrames (:86-106).  Never writes img_bgmodel."""
    ALGO = capi.ALGO_DP_WREN_GA


class DPPratiMediodBGS(_Plugin):
    """package_bgs/dp/DPPratiMediodBGS.cpp (USTC_BGS type 14): temporal medoid over a ring of sampled frames (Cucchiara /
    Calderara / Prati); keys threshold, samplingRate, historySize, weight (:90-110).  No mask before frame historySize;
    never writes img_bgmodel."""
    ALGO = capi.ALGO_DP_PRATI_MEDIOD


class SigmaDeltaBGS(_Plugin):
    """package_bgs/bl/SigmaDeltaBGS.cpp (USTC_BGS type 35): the Sigma-Delta estimator of Lacassagne / Manzanera
    (package_bgs/bl/sdLaMa091.cpp); keys ampFactor, minVar, maxVar (:56-70), applied before every frame.  The first frame
    only initialises the model (no outputs); never writes img_bgmodel."""
    ALGO = capi.ALGO_SIGMA_DELTA


class MixtureOfGaussianV2BGS(_Plugin):
    """package_bgs/MixtureOfGaussianV2BGS.cpp; keys alpha, enableThreshold, threshold (:92-95)."""
    ALGO = capi.ALGO_MOG2

    def export_state(self, stream_index=0):
        """-> (planes float32 [25, npx], nmodes uint8 [npx]); plane q = mode*5 + {w,var,muB,muG,muR}."""
        npx = self.state_bytes() // 101
        planes = np.empty((25, npx), np.float32)
        nm = np.empty(npx, np.uint8)
        capi.check(capi.lib().bgsb_mog2_export_state(self._h, stream_index,
                                                     planes.ctypes.data_as(capi.f32p), nm.ctypes.data_as(capi.u8p)))
        return planes, nm

    def import_state(self, planes, nmodes, w, h, nframes, stream_index=0):
        planes = np.ascontiguousarray(planes, np.float32)
        nmodes = np.ascontiguousarray(nmodes, np.uint8)
        capi.check(capi.lib().bgsb_mog2_import_state(self._h, stream_index, w, h, nframes,
                                                     planes.ctypes.data_as(capi.f32p), nmodes.ctypes.data_as(capi.u8p)))


class _PinnedOwner:
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        try:
            capi.lib().bgsb_host_free(self.ptr)
        except Exception:
            pass


def pinned_empty(shape, write_combined=False):
    """uint8 numpy array on page-locked host memory (bgsb_host_alloc); freed with the array."""
    n = int(np.prod(shape))
    p = C.c_void_p()
    capi.check(capi.lib().bgsb_host_alloc(C.byref(p), max(n, 1), int(write_combined)))
    owner = _PinnedOwner(p)
    buf = (C.c_uint8 * max(n, 1)).from_address(p.value)
    buf._owner = owner
    arr = np.frombuffer(buf, dtype=np.uint8, count=n).reshape(shape)
    return arr


def process_fanout(plugins, img_input, want_bg=True):
    """FrameProcessor::process (FrameProcessor.cpp:169-215): every plugin on the same frame, one upload.
    Returns [(img_output | None, img_bgmodel | None), ...] exactly as plugin.process(img_input) would for each.
    With "inputFormat" NV12 / I420 (the same on every plugin) img_input is the (3h/2) x W YUV image."""
    if img_input is None or img_input.size == 0:
        return [(None, None) for _ in plugins]
    fmt = plugins[0].input_format if plugins else capi.INPUT_BGR
    if fmt != capi.INPUT_BGR:
        img, h, w, _ = yuv_frame(img_input, fmt)
    else:
        img = np.asarray(img_input)
        if img.dtype != np.uint8 or img.ndim != 3 or img.shape[-1] != 3:
            raise ValueError("fan-out takes one BGR 8UC3 frame")
        if img.strides[-1] != 1 or img.strides[-2] != 3:
            img = np.ascontiguousarray(img)
        h, w = img.shape[:2]
    n = len(plugins)
    fgs = [np.empty((h, w), np.uint8) for _ in plugins]
    bgs = [np.empty((h, w, 3) if p.BG_CHANNELS == 3 else (h, w), np.uint8) if want_bg else None for p in plugins]
    ctxs = (C.c_void_p * n)(*[p._h for p in plugins])
    fgp = (C.c_void_p * n)(*[f.ctypes.data for f in fgs])
    fgst = (C.c_size_t * n)(*[w] * n)
    bgp = (C.c_void_p * n)(*[(b.ctypes.data if b is not None else None) for b in bgs])
    bgst = (C.c_size_t * n)(*[p.BG_CHANNELS * w for p in plugins])
    fv, bv = (C.c_int * n)(), (C.c_int * n)()
    capi.check(capi.lib().bgsb_process_fanout(ctxs, n, _ptr(img), w, h, img.strides[0], fgp, fgst, bgp, bgst, fv, bv))
    return [((fgs[k] if fv[k] else None), (bgs[k] if bv[k] else None)) for k in range(n)]


# integer ids of the USTC_BGS factory (ustc_src/ustc_bgs.cpp:8-14)
ALGOS = {0: FrameDifferenceBGS, 1: StaticFrameDifferenceBGS, 2: WeightedMovingMeanBGS,
         3: WeightedMovingVarianceBGS, 5: MixtureOfGaussianV2BGS, 6: AdaptiveBackgroundLearning,
         7: AdaptiveSelectiveBackgroundLearning, 9: DPAdaptiveMedianBGS, 11: DPZivkovicAGMMBGS, 12: DPMeanBGS,
         13: DPWrenGABGS, 14: DPPratiMediodBGS, 35: SigmaDeltaBGS}


class USTC_BGS:
    """CvFGDetector adapter (ustc_src/ustc_bgs.{h,cpp}): Process(img) then GetMask()."""

    def __init__(self, type, device=0):
        if type not in ALGOS:                   # CV_Assert(type>=0 && type<=37), .cpp:6
            raise ValueError("USTC_BGS type %r is not on the B200 hot path (0 FD, 1 StaticFD, 2 WMM, 3 WMV, 5 MOG2, 6 ABL, 7 ASBL, 9 DPAdaptiveMedian, 11 DPZivkovicAGMM, 12 DPMean, 13 DPWrenGA, 14 DPPratiMediod, 35 SigmaDelta)" % type)
        self.bgs = ALGOS[type](device=device)
        self.frameNum = 0
        self.img_mask = None
        self.img_bkgmodel = None

    def Process(self, pImg):                    # ustc_bgs.cpp:87-113
        fg, bg = self.bgs.process(pImg)
        if fg is not None:
            self.img_mask = fg
        if bg is not None:
            self.img_bkgmodel = bg
        self.frameNum += 1

    def GetMask(self):                          # ustc_bgs.cpp:79-85; NULL until a mask exists
        if self.frameNum == 0:
            return None
        return self.img_mask

    def Release(self):                          # ustc_bgs.cpp:75-77
        self.bgs.close()
