"""Camera streams over GPUs (SURVEY 8e): stream s lives on GPU s mod G; streams never exchange data.

`StreamPool` is the product-level owner of N camera streams on the GPUs one process can see (bgsb_pool_*,
csrc/pool.cu): one host worker thread and one stream-group pipeline per GPU, page-locked frame / mask / table rings, so
that the upload of the next frame set overlaps the kernels of this one and the download of the previous one.  It is the
reference's per-camera main loop (ustc_src/trackingMain.cpp:161-166: query frame, USTC_BGS::Process, clean-up,
DetectNewBlob) run for many cameras at once.

Across processes (one process per GPU, e.g. under torchrun) the same rule shards the streams: `shard_streams`; ranks
never communicate on the data path, torch.distributed is used by bench.py only for the start/stop barrier and the
max-over-ranks of the timed region.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi
from .blobs import _ops, detect_streams


def shard_streams(nstreams: int, world_size: int, rank: int):
    """Stream ids owned by `rank` (round robin: s mod world_size == rank)."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad rank/world_size")
    return list(range(rank, nstreams, world_size))


def streams_per_rank(nstreams: int, world_size: int):
    return [len(shard_streams(nstreams, world_size, r)) for r in range(world_size)]


def aggregate_throughput(units_per_rank, seconds_per_rank):
    """Whole-job throughput = all units / slowest rank's time (max over ranks)."""
    return float(sum(units_per_rank)) / max(seconds_per_rank)


class StreamPool:
    """N camera streams of one geometry on `devices` (default: every visible GPU).

        pool = StreamPool(capi.ALGO_MOG2, nstreams=64, w=1920, h=1080, ring=3)
        pool.frame_buffer(s, slot)[...] = frame          # capture side, page-locked memory
        pool.submit(slot)                                # every stream's frame of `slot` is in place
        valid = pool.wait(slot)
        blobs = pool.components(s, slot)                 # bounding boxes / areas / external flags of stream s

    With submit(slot, detect=True), detect(slot, detectors, old_blobs) then runs DetectNewBlob for every stream.
    """

    def __init__(self, algo, nstreams, w, h, devices=None, ring=2, morph=None, **params):
        L = capi.lib()
        if devices is None:
            n = C.c_int(0)
            capi.check(L.bgsb_device_count(C.byref(n)))
            devices = list(range(max(1, n.value)))
        self.devices = list(devices)
        self.nstreams, self.w, self.h, self.ring = nstreams, w, h, ring
        self._h = C.c_void_p()
        dv = (C.c_int * len(self.devices))(*self.devices)
        capi.check(L.bgsb_pool_create(C.byref(self._h), algo, nstreams, dv, len(self.devices), w, h, ring))
        if morph is not None:
            ops, n = _ops(morph)
            capi.check(L.bgsb_pool_set_morph(self._h, ops, n))
        for k, v in params.items():
            capi.check(L.bgsb_pool_set_param(self._h, k.encode(), float(v)))
        self.input_format = int(params.get("inputFormat", capi.INPUT_BGR))
        rows = C.c_int(0)
        capi.check(L.bgsb_pool_info(self._h, None, None, C.byref(rows)))
        self.table_rows = rows.value

    def close(self):
        if self._h:
            capi.lib().bgsb_pool_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def device_of(self, stream):
        d = C.c_int(0)
        capi.check(capi.lib().bgsb_pool_device_of(self._h, stream, C.byref(d)))
        return d.value

    def frame_buffer(self, stream, slot):
        """(h, w, 3) uint8 view of the page-locked buffer the capture side fills for (stream, slot); with "inputFormat"
        NV12 / I420 the (3h/2, w) view of the YUV 4:2:0 image."""
        p = capi.lib().bgsb_pool_frame_buffer(self._h, stream, slot)
        if not p:
            raise IndexError("stream / slot out of range")
        shape = (self.h, self.w, 3) if self.input_format == capi.INPUT_BGR else (self.h * 3 // 2, self.w)
        buf = (C.c_uint8 * int(np.prod(shape))).from_address(p)
        return np.frombuffer(buf, dtype=np.uint8).reshape(shape)

    def submit(self, slot, want_masks=False, detect=False):
        """want_masks: download the cleaned masks (mask()); detect: keep them on the device for detect()."""
        flags = (capi.POOL_MASKS if want_masks else 0) | (capi.POOL_DETECT if detect else 0)
        capi.check(capi.lib().bgsb_pool_submit(self._h, slot, flags))

    def wait(self, slot):
        v = C.c_int(0)
        capi.check(capi.lib().bgsb_pool_wait(self._h, slot, C.byref(v)))
        return bool(v.value)

    def mask(self, stream, slot):
        p = capi.lib().bgsb_pool_mask(self._h, stream, slot)
        if not p:
            return None
        buf = (C.c_uint8 * (self.h * self.w)).from_address(p)
        return np.frombuffer(buf, dtype=np.uint8).reshape(self.h, self.w)

    def detect(self, slot, detectors, old_blobs=None):
        """DetectNewBlob for every stream of a waited-for slot submitted with detect=True: detectors[s] is stream s's
        blobs.CvBlobDetectorCC, old_blobs[s] its tracked blobs [(x, y, w, h)] (None: none anywhere).  -> per stream
        (result, new_blob | None, frame_blobs), or None for a stream with more than table_rows components (its detector
        did not advance; raise "tableRows")."""
        if len(detectors) != self.nstreams:
            raise ValueError("one detector per stream")
        return detect_streams(capi.lib().bgsb_pool_detect, (self._h, slot), detectors, old_blobs)

    def components(self, stream, slot):
        n = C.c_int(0)
        comps = (capi.Component * self.table_rows)()
        capi.check(capi.lib().bgsb_pool_components(self._h, stream, slot, comps, self.table_rows, C.byref(n)))
        return [dict(label=c.label, first_index=c.first_index, x=c.x, y=c.y, w=c.w, h=c.h, area=c.area,
                     external=c.external) for c in comps[:n.value]]
