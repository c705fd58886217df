"""Host-side mirror of the device-resident foreground pipeline (bgsb_pipeline_*, include/bgsb200.h):

    IBGS::process -> erode / dilate chain -> steps 1-2 of CvBlobDetectorCC::DetectNewBlob

for a group of camera streams, i.e. one iteration of the reference's main loop per stream
(ustc_src/trackingMain.cpp:161-166) -- BASELINE config 4.  Device pointers in, device outputs; component
tables are fetched per stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .blobs import _ops, detect_streams


class ForegroundPipeline:
    def __init__(self, algo=capi.ALGO_MOG2, device=0, nstreams=1, morph=(("erode", 1), ("dilate", 1)), **params):
        self._h = C.c_void_p()
        self.device, self.nstreams, self.algo = device, nstreams, algo
        capi.check(capi.lib().bgsb_pipeline_create(C.byref(self._h), algo, device, nstreams))
        self.set_morph(morph)
        for k, v in params.items():
            self.set(k, v)
        self._shape = None

    def set(self, key, value):
        capi.check(capi.lib().bgsb_pipeline_set_param(self._h, key.encode(), float(value)))

    def set_morph(self, chain):
        ops, n = _ops(chain)
        capi.check(capi.lib().bgsb_pipeline_set_morph(self._h, ops, n))

    @property
    def bgs_handle(self):
        """The plugin context inside (bgsb_ctx *), e.g. for bgsb_mog2_export_state."""
        return C.c_void_p(capi.lib().bgsb_pipeline_bgs(self._h))

    def close(self):
        if self._h:
            capi.lib().bgsb_pipeline_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process_dev(self, d_frames, w, h, d_mask=None, d_bg=None, d_labels=None, stream=0):
        """d_frames: device pointer to [nstreams][h][w][3].  -> (mask_valid, bg_valid)."""
        v, bv = C.c_int(0), C.c_int(0)
        capi.check(capi.lib().bgsb_pipeline_process_dev(self._h, C.c_void_p(d_frames), w, h,
                                                        C.c_void_p(d_mask) if d_mask else None,
                                                        C.c_void_p(d_bg) if d_bg else None,
                                                        C.c_void_p(d_labels) if d_labels else None,
                                                        C.byref(v), C.byref(bv), C.c_void_p(stream)))
        self._shape = (w, h)
        return bool(v.value), bool(bv.value)

    def join_dev(self, stream=0):
        """`stream` waits for all clean-up / labelling work enqueued so far (they run on the pipeline's own stream)."""
        capi.check(capi.lib().bgsb_pipeline_join_dev(self._h, C.c_void_p(stream)))

    def components(self, stream_index=0):
        n = C.c_int(0)
        capi.check(capi.lib().bgsb_pipeline_components(self._h, stream_index, None, 0, C.byref(n)))
        comps = (capi.Component * max(n.value, 1))()
        capi.check(capi.lib().bgsb_pipeline_components(self._h, stream_index, comps, max(n.value, 1), C.byref(n)))
        return [dict(label=c.label, first_index=c.first_index, x=c.x, y=c.y, w=c.w, h=c.h, area=c.area,
                     external=c.external) for c in comps[:n.value]]

    def rect_moments(self, rects, stream_index=0):
        if not rects:
            return []
        flat = np.ascontiguousarray(np.asarray(rects, np.int32).reshape(-1))
        out = (C.c_uint64 * (6 * len(rects)))()
        capi.check(capi.lib().bgsb_pipeline_rect_moments(self._h, stream_index, flat.ctypes.data_as(capi.i32p),
                                                         len(rects), out))
        return [[int(out[6 * i + j]) for j in range(6)] for i in range(len(rects))]

    def detect(self, detectors, old_blobs=None):
        """DetectNewBlob for every stream of the last frame on the labelling already done: detectors[s] is stream s's
        blobs.CvBlobDetectorCC, old_blobs[s] its tracked blobs [(x, y, w, h)] (None: none anywhere).
        -> per stream (result, new_blob | None, frame_blobs)."""
        if len(detectors) != self.nstreams:
            raise ValueError("one detector per stream")
        return detect_streams(capi.lib().bgsb_pipeline_detect, (self._h,), detectors, old_blobs)

    def export_mog2_state(self, stream_index=0):
        if self.algo != capi.ALGO_MOG2 or self._shape is None:
            raise ValueError("no MOG2 state")
        npx = self._shape[0] * self._shape[1]
        planes = np.empty((25, npx), np.float32)
        nm = np.empty(npx, np.uint8)
        capi.check(capi.lib().bgsb_mog2_export_state(self.bgs_handle, stream_index,
                                                     planes.ctypes.data_as(capi.f32p), nm.ctypes.data_as(capi.u8p)))
        return planes, nm
