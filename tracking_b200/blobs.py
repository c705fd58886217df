"""Host-side mirror of the mask post-processing + CvBlobDetector stage, on top of the C ABI.

    erode / dilate      cv::erode / cv::dilate(mask, cv::Mat(), Point(-1,-1), iterations)
    ConnectedComponents steps 1-2 of CvBlobDetectorCC::DetectNewBlob (+ exact ROI moments)
    CvBlobDetectorCC    cvCreateBlobDetectorCC() (ustc_src/trackingMain.cpp:56,626)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi

ERODE, DILATE = capi.MORPH_ERODE, capi.MORPH_DILATE


def _ops(chain):
    flat = []
    for op, it in chain:
        flat += [{"erode": ERODE, "dilate": DILATE}.get(op, op), int(it)]
    return (C.c_int * len(flat))(*flat), len(flat) // 2


def morph(mask, chain):
    """mask: HxW uint8 {0,255}; chain: [("erode", 1), ("dilate", 1)] = OPEN 3x3."""
    mask = np.ascontiguousarray(mask, np.uint8)
    h, w = mask.shape
    out = np.empty_like(mask)
    ops, n = _ops(chain)
    capi.check(capi.lib().bgsb_morph(C.c_void_p(mask.ctypes.data), w, h, w, ops, n, C.c_void_p(out.ctypes.data), w))
    return out


def morph_dev(d_mask, w, h, nimages, chain, d_out, stream=0):
    ops, n = _ops(chain)
    capi.check(capi.lib().bgsb_morph_dev(C.c_void_p(d_mask), w, h, nimages, ops, n, C.c_void_p(d_out),
                                         C.c_void_p(stream)))


def erode(mask, iterations=1):
    return morph(mask, [("erode", iterations)])


def dilate(mask, iterations=1):
    return morph(mask, [("dilate", iterations)])


class ConnectedComponents:
    def __init__(self, max_w, max_h, device=0, max_images=1):
        self._h = C.c_void_p()
        self.max_w, self.max_h, self.max_images = max_w, max_h, max_images
        capi.check(capi.lib().bgsb_ccl_create_batch(C.byref(self._h), device, max_w, max_h, max_images))

    def set(self, key, value):
        capi.check(capi.lib().bgsb_ccl_set_param(self._h, key.encode(), float(value)))

    def close(self):
        if self._h:
            capi.lib().bgsb_ccl_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def label(self, mask, zero_border=False, want_labels=True):
        """-> (n, labels int32 HxW | None, components list of dict)"""
        mask = np.ascontiguousarray(mask, np.uint8)
        h, w = mask.shape
        labels = np.empty((h, w), np.int32) if want_labels else None
        cap = ((w + 1) // 2) * ((h + 1) // 2) + 64          # the most 8-connected components an image can hold
        comps = (capi.Component * cap)()
        n = C.c_int(0)
        capi.check(capi.lib().bgsb_ccl_label(self._h, C.c_void_p(mask.ctypes.data), w, h, w, int(zero_border),
                                             C.c_void_p(labels.ctypes.data) if want_labels else None, comps, cap,
                                             C.byref(n)))
        out = [dict(label=c.label, first_index=c.first_index, x=c.x, y=c.y, w=c.w, h=c.h, area=c.area,
                    external=c.external) for c in comps[:n.value]]
        return n.value, labels, out

    def label_dev(self, d_mask, w, h, zero_border=False, d_labels=None, stream=0):
        capi.check(capi.lib().bgsb_ccl_label_dev(self._h, C.c_void_p(d_mask), w, h, int(zero_border),
                                                 C.c_void_p(d_labels) if d_labels else None, C.c_void_p(stream)))

    def label_batch_dev(self, d_masks, w, h, nimages, zero_border=False, d_labels=None, stream=0):
        """nimages dense masks back to back -> one launch sequence for all of them."""
        capi.check(capi.lib().bgsb_ccl_label_batch_dev(self._h, C.c_void_p(d_masks), w, h, nimages, int(zero_border),
                                                       C.c_void_p(d_labels) if d_labels else None, C.c_void_p(stream)))

    def components(self, image=0):
        n = C.c_int(0)
        capi.check(capi.lib().bgsb_ccl_components_of(self._h, image, None, 0, C.byref(n)))
        comps = (capi.Component * max(n.value, 1))()
        capi.check(capi.lib().bgsb_ccl_components_of(self._h, image, comps, max(n.value, 1), C.byref(n)))
        return [dict(label=c.label, first_index=c.first_index, x=c.x, y=c.y, w=c.w, h=c.h, area=c.area,
                     external=c.external) for c in comps[:n.value]]

    def rect_moments(self, rects):
        """rects: [(x,y,w,h)] on the mask last labelled -> [[m00,m10,m01,m20,m02,m11]] (exact ints)."""
        if not rects:
            return []
        flat = np.ascontiguousarray(np.asarray(rects, np.int32).reshape(-1))
        out = (C.c_uint64 * (6 * len(rects)))()
        capi.check(capi.lib().bgsb_ccl_rect_moments(self._h, flat.ctypes.data_as(capi.i32p), len(rects), out))
        return [[int(out[6 * i + j]) for j in range(6)] for i in range(len(rects))]


def detect_streams(fn, handle_args, detectors, old_blobs):
    """bgsb_pipeline_detect / bgsb_pool_detect: per stream (result, new_blob | None, frame_blobs), or None for a stream
    whose status is not BGSB_OK (its detector did not advance).  old_blobs: None or per stream a list of (x, y, w, h)."""
    S = len(detectors)
    bds = (C.c_void_p * S)(*[d._h for d in detectors])
    old_arrs = [(capi.Blob * max(len(o), 1))(*[capi.Blob(*o_[:4], 0) for o_ in o]) for o in (old_blobs or [()] * S)]
    olds = (C.POINTER(capi.Blob) * S)(*[C.cast(a, C.POINTER(capi.Blob)) for a in old_arrs])
    n_old = (C.c_int * S)(*[len(o) for o in (old_blobs or [()] * S)])
    new, fr = (capi.Blob * S)(), (capi.Blob * (10 * S))()
    res, n_fr, status = (C.c_int * S)(), (C.c_int * S)(), (C.c_int * S)()
    rc = fn(*handle_args, bds, olds, n_old, new, res, fr, n_fr, status)
    if rc not in (capi.OK, capi.ERR_CAPACITY):
        capi.check(rc)
    out = []
    for s, d in enumerate(detectors):
        if status[s] != capi.OK:
            out.append(None)
            continue
        d.frame_blobs = [(b.x, b.y, b.w, b.h) for b in fr[10 * s:10 * s + n_fr[s]]]
        nb = (new[s].x, new[s].y, new[s].w, new[s].h) if res[s] else None
        out.append((res[s], nb, d.frame_blobs))
    return out


class CvBlobDetectorCC:
    """DetectNewBlob(pImg, pFGMask, pNewBlobList, pOldBlobList) -> int."""

    def __init__(self, device=0, **params):
        self._h = C.c_void_p()
        capi.check(capi.lib().bgsb_blobdetector_create(C.byref(self._h), device))
        for k, v in params.items():
            capi.check(capi.lib().bgsb_blobdetector_set_param(self._h, k.encode(), float(v)))
        self.frame_blobs = []

    def close(self):
        if self._h:
            capi.lib().bgsb_blobdetector_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _call(self, fn, head, tail, old_blobs):
        old = (capi.Blob * max(len(old_blobs), 1))(*[capi.Blob(*b) for b in old_blobs])
        new = (capi.Blob * 4)()
        fr = (capi.Blob * 16)()
        n_new, res, n_fr = C.c_int(0), C.c_int(0), C.c_int(0)
        capi.check(fn(self._h, *head, old, len(old_blobs), new, 4, C.byref(n_new), C.byref(res), fr, 16,
                      C.byref(n_fr), *tail))
        self.frame_blobs = [(b.x, b.y, b.w, b.h) for b in fr[:n_fr.value]]
        nb = [(b.x, b.y, b.w, b.h) for b in new[:n_new.value]]
        return res.value, (nb[0] if nb else None)

    def DetectNewBlob(self, fg_mask, old_blobs=()):
        m = np.ascontiguousarray(fg_mask, np.uint8)
        h, w = m.shape
        old = [(b[0], b[1], b[2], b[3], 0) for b in old_blobs]
        return self._call(capi.lib().bgsb_blobdetector_detect, (C.c_void_p(m.ctypes.data), w, h, w), (), old)

    def DetectNewBlob_dev(self, d_mask, w, h, old_blobs=(), stream=0):
        old = [(b[0], b[1], b[2], b[3], 0) for b in old_blobs]
        return self._call(capi.lib().bgsb_blobdetector_detect_dev, (C.c_void_p(d_mask), w, h),
                          (C.c_void_p(stream),), old)
