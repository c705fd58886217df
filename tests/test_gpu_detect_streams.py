"""DetectNewBlob for every stream of a pipeline (bgsb_pipeline_detect) and of a stream pool (bgsb_pool_detect) on the
labelling they already ran, against oracle/blobdetect.py on the oracle chain's cleaned mask and against a separate
bgsb_blobdetector_detect on the same mask; the batched moments kernels against numpy; which kernels and copies a detect
call makes."""
import collections
import ctypes as C
import json
import os
import warnings

import numpy as np
import pytest

from tracking_b200 import capi

pytestmark = pytest.mark.gpu

OPEN = (("erode", 1), ("dilate", 1))
MOG2, FD, WMV = capi.ALGO_MOG2, capi.ALGO_FRAME_DIFFERENCE, capi.ALGO_WEIGHTED_MOVING_VARIANCE


def walk(clip, s, t):
    return clip[(t * (1 + s % 3) + 5 * s) % len(clip)]          # a different walk per stream (as test_gpu_pool.py)


class Reference:
    """Per stream: the oracle plugin and chain, oracle/blobdetect.py and a bgsb_blobdetector fed the same mask."""

    def __init__(self, oracle, algo, chain, S, plugin_kw=None, zero_border=True):
        from oracle import blobdetect
        from tracking_b200 import blobs
        self.oracle, self.chain = oracle, chain
        self.plugins = [oracle.ALGOS[algo](**(plugin_kw or {})) for _ in range(S)]
        self.obd = [blobdetect.CvBlobDetectorCC(zero_border=zero_border) for _ in range(S)]
        self.sep = [blobs.CvBlobDetectorCC(zeroBorder=int(zero_border)) for _ in range(S)]
        self.dets = [blobs.CvBlobDetectorCC(zeroBorder=int(zero_border)) for _ in range(S)]
        self.tracked = [[] for _ in range(S)]

    def mask(self, s, frame):
        fg, _ = self.plugins[s].process(frame)
        if fg is None:
            return None
        for op, it in self.chain:
            fg = self.oracle.morph(fg, op, it)
        return fg

    def check(self, s, mask, got, where):
        from oracle import blobdetect
        tracked = self.tracked[s]
        ores, onb = self.obd[s].DetectNewBlob(mask, [blobdetect.Blob(*b) for b in tracked])
        sres, snb = self.sep[s].DetectNewBlob(mask, tracked)
        res, nb, frame = got
        assert res == ores == sres, where
        assert frame == [b.tuple() for b in self.obd[s].lists[0]] == self.sep[s].frame_blobs, where
        if res:
            assert nb == onb.tuple() == snb, where
            tracked.append(nb)                  # the new blob becomes a tracked one, as the tracker would do
            del tracked[:-3]


def run_pipeline(oracle, clips, algo, chain, S=5, nframes=32, plugin_kw=None):
    import torch
    from tracking_b200.pipeline import ForegroundPipeline
    clip = clips["video_clip"]
    h, w = clip.shape[1:3]
    pipe = ForegroundPipeline(algo, nstreams=S, morph=chain, **(plugin_kw or {}))
    ref = Reference(oracle, algo, chain, S, {"enableThreshold": False} if plugin_kw else None)
    results = 0
    for t in range(nframes):
        frames = [walk(clip, s, t) for s in range(S)]
        d_in = torch.from_numpy(np.stack(frames)).cuda()
        valid, _ = pipe.process_dev(d_in.data_ptr(), w, h)
        masks = [ref.mask(s, frames[s]) for s in range(S)]
        assert valid == (masks[0] is not None)
        if not valid:
            with pytest.raises(capi.BgsbError) as e:
                pipe.detect(ref.dets, ref.tracked)
            assert e.value.code == capi.ERR_STATE
            continue
        got = pipe.detect(ref.dets, ref.tracked)
        for s in range(S):
            ref.check(s, masks[s], got[s], (algo, chain, t, s))
            results += got[s][0]
    pipe.close()
    return results


@pytest.mark.parametrize("algo", [MOG2, FD, WMV])
@pytest.mark.parametrize("chain", [OPEN, ()], ids=["open", "nochain"])
def test_pipeline_detect_matches_oracle_and_single_detector(oracle, clips, algo, chain):
    run_pipeline(oracle, clips, algo, chain)


def test_pipeline_detect_raw_mask_weighs_shadows(oracle, clips):
    """MOG2 with enableThreshold = 0 and no chain: the moments weigh the raw mask (shadow pixels 127)."""
    run_pipeline(oracle, clips, MOG2, (), S=3, nframes=20, plugin_kw={"enableThreshold": 0})


def _raw_detect(pipe_h, dets, S):
    bds = (C.c_void_p * S)(*dets)
    new, res, st = (capi.Blob * S)(), (C.c_int * S)(), (C.c_int * S)()
    return capi.lib().bgsb_pipeline_detect(pipe_h, bds, None, None, new, res, None, None, st)


def test_pipeline_detect_refusals(clips):
    import torch
    from tracking_b200 import blobs
    from tracking_b200.pipeline import ForegroundPipeline
    clip = clips["video_clip"]
    h, w = clip.shape[1:3]
    S = 2
    dets = [blobs.CvBlobDetectorCC() for _ in range(S)]
    d_in = lambda t: torch.from_numpy(np.stack([clip[t], clip[t + 1]])).cuda()
    # warm-up frame: no mask, no detector advances
    fd = ForegroundPipeline(FD, nstreams=S)
    assert fd.process_dev(d_in(0).data_ptr(), w, h)[0] is False
    assert _raw_detect(fd._h, [d._h for d in dets], S) == capi.ERR_STATE
    assert fd.process_dev(d_in(1).data_ptr(), w, h)[0] is True
    assert _raw_detect(fd._h, [dets[0]._h, None], S) == capi.ERR_ARG                 # NULL detector
    assert _raw_detect(fd._h, [dets[0]._h, dets[0]._h], S) == capi.ERR_ARG           # one detector for two streams
    odd = blobs.CvBlobDetectorCC(zeroBorder=0)
    assert _raw_detect(fd._h, [dets[0]._h, odd._h], S) == capi.ERR_ARG               # labelled with zeroBorder 1
    assert _raw_detect(fd._h, [d._h for d in dets], S) == capi.OK
    fd.close()
    # threshold off with a chain: the reference weighs a grey-level cleaned mask the pipeline does not compute
    raw = ForegroundPipeline(MOG2, nstreams=S, morph=OPEN, enableThreshold=0)
    raw.process_dev(d_in(2).data_ptr(), w, h)
    with pytest.raises(capi.BgsbError) as e:
        raw.detect(dets)
    assert e.value.code == capi.ERR_ARG
    raw.close()
    # the pipeline's own zeroBorder 0 with matching detectors
    zb = ForegroundPipeline(MOG2, nstreams=S, zeroBorder=0)
    zb.process_dev(d_in(3).data_ptr(), w, h)
    with pytest.raises(capi.BgsbError):
        zb.detect(dets)
    zb.detect([blobs.CvBlobDetectorCC(zeroBorder=0) for _ in range(S)])
    zb.close()


def run_pool(oracle, clips, devices, nstreams, ring, want_masks, nframes=32, algo=MOG2):
    from tracking_b200.streams import StreamPool
    clip = clips["video_clip"]
    h, w = clip.shape[1:3]
    pool = StreamPool(algo, nstreams, w, h, devices=devices, ring=ring, morph=OPEN)
    ref = Reference(oracle, algo, OPEN, nstreams)

    def check(t):
        slot = t % ring
        valid = pool.wait(slot)
        masks = [ref.mask(s, walk(clip, s, t)) for s in range(nstreams)]
        assert valid == (masks[0] is not None)
        if not valid:
            return
        if want_masks:
            assert all(np.array_equal(pool.mask(s, slot), masks[s]) for s in range(nstreams))
        got = pool.detect(slot, ref.dets, ref.tracked)
        for s in range(nstreams):
            ref.check(s, masks[s], got[s], (devices, ring, want_masks, t, s))

    for t in range(nframes):
        if t >= ring:
            check(t - ring)
        slot = t % ring
        for s in range(nstreams):
            pool.frame_buffer(s, slot)[...] = walk(clip, s, t)
        pool.submit(slot, want_masks, detect=True)
    for t in range(max(0, nframes - ring), nframes):
        check(t)
    pool.close()


@pytest.mark.parametrize("ring", [1, 3])
@pytest.mark.parametrize("want_masks", [False, True])
def test_pool_detect_one_group(oracle, clips, ring, want_masks):
    run_pool(oracle, clips, [0], 5, ring, want_masks)


@pytest.mark.parametrize("want_masks", [False, True])
def test_pool_detect_two_groups_on_one_device(oracle, clips, want_masks):
    run_pool(oracle, clips, [0, 0], 5, 3, want_masks, algo=FD)


def test_pool_detect_two_devices(oracle, clips):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU on this box (two groups on one device are covered above)")
    run_pool(oracle, clips, [0, 1], 6, 3, False)


def test_pool_detect_refusals(clips):
    from tracking_b200 import blobs
    from tracking_b200.streams import StreamPool
    clip = clips["video_clip"]
    h, w = clip.shape[1:3]
    pool = StreamPool(FD, 2, w, h, devices=[0], ring=2)
    dets = [blobs.CvBlobDetectorCC() for _ in range(2)]
    with pytest.raises(capi.BgsbError) as e:
        pool.detect(0, dets)                                      # nothing submitted / waited for
    assert e.value.code == capi.ERR_STATE
    for t in range(3):
        for s in range(2):
            pool.frame_buffer(s, t % 2)[...] = clip[t + s]
        pool.submit(t % 2, detect=(t != 2))
        valid = pool.wait(t % 2)
        with pytest.raises(capi.BgsbError) as e:
            if t == 0:
                assert not valid
                pool.detect(0, dets)                              # warm-up frame
            elif t == 1:
                pool.detect(1, [dets[0], dets[0]])                # one detector for two streams
            else:
                pool.detect(0, dets)                              # submitted without detect
        assert e.value.code == (capi.ERR_ARG if t == 1 else capi.ERR_STATE), t
    assert pool.detect(1, dets)[0] is not None
    with pytest.raises(capi.BgsbError):
        pool.detect(1, [dets[0], blobs.CvBlobDetectorCC(zeroBorder=0)])
    assert capi.lib().bgsb_pool_submit(pool._h, 0, 4) == capi.ERR_ARG     # unknown flag bit
    pool.close()
    with pytest.raises(capi.BgsbError):
        StreamPool(FD, 2, w, h, devices=[0], ring=2, tableRows=0)


def salt_frames(n, h, w, seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(60, 200, (h, w, 3)).astype(np.uint8)
    out = []
    for _ in range(n):
        f = base.copy()
        f[rng.random((h, w)) < 0.004] = 255
        out.append(f)
    return out


@pytest.mark.parametrize("table_rows", [32, 4096])
def test_pool_detect_table_capacity(oracle, clips, table_rows):
    """A salt-noise stream with more components than "tableRows": BGSB_ERR_CAPACITY for that stream only, its detector
    does not advance; with the rows raised it matches too."""
    from tracking_b200.streams import StreamPool
    clip = clips["video_clip"]
    h, w = clip.shape[1:3]
    S, noisy = 3, 1
    salt = salt_frames(8, h, w, 5)
    frame = lambda s, t: salt[t] if s == noisy else walk(clip, s, t)
    pool = StreamPool(FD, S, w, h, devices=[0], ring=1, morph=(), tableRows=table_rows)
    assert pool.table_rows == table_rows
    ref = Reference(oracle, FD, (), S)
    over = 0
    for t in range(len(salt)):
        for s in range(S):
            pool.frame_buffer(s, 0)[...] = frame(s, t)
        pool.submit(0, detect=True)
        masks = [ref.mask(s, frame(s, t)) for s in range(S)]
        if not pool.wait(0):
            continue
        got = pool.detect(0, ref.dets, ref.tracked)
        for s in range(S):
            if got[s] is None:
                assert s == noisy and table_rows == 32
                assert ref.dets[s].frame_blobs == []              # never advanced
                over += 1
                continue
            if s == noisy:
                assert len(pool.components(s, 0)) > 32
            ref.check(s, masks[s], got[s], (table_rows, t, s))
    assert over == (len(salt) - 1 if table_rows == 32 else 0)
    pool.close()


# ---------------------------------------------------------------------------------------------------------------------
# the batched moments kernels

def numpy_moments(img, rect):
    x, y, rw, rh = rect
    h, w = img.shape
    out = [0] * 6
    if rw <= 0 or rh <= 0:
        return out
    xa, xb, ya, yb = max(x, 0), min(x + rw, w), max(y, 0), min(y + rh, h)
    if xa >= xb or ya >= yb:
        return out
    v = img[ya:yb, xa:xb].astype(np.int64)
    xx = np.arange(xa, xb, dtype=np.int64) - x
    yy = (np.arange(ya, yb, dtype=np.int64) - y)[:, None]
    return [int(v.sum()), int((v * xx).sum()), int((v * yy).sum()), int((v * xx * xx).sum()), int((v * yy * yy).sum()),
            int((v * xx * yy).sum())]


def moment_rects(w, h, seed):
    rng = np.random.default_rng(seed)
    rects = [(0, 0, w, h), (0, 0, 0, 5), (3, 4, 7, 0), (5, 5, -3, 4), (w, 0, 5, h), (0, h, w, 3), (-9, -9, 5, 5),
             (-5, 3, 40, 9), (w - 17, 2, 40, 11), (7, -6, 50, 13), (11, h - 4, 33, 20), (-3, -2, w + 9, h + 7),
             (w - 1, h - 1, 1, 1), (1, 0, w - 2, 1)]
    for _ in range(40):
        x, y = int(rng.integers(-30, w)), int(rng.integers(-10, h))
        rects.append((x, y, int(rng.integers(1, w + 40)), int(rng.integers(1, h + 10))))
    return rects


def test_moments_kernel_bytes_on_seven_images(oracle):
    """rect_moments_kernel on grey-level byte masks (every value weighs) whose rows start off the 16-byte grid."""
    import torch
    from tracking_b200 import blobs
    h, w, S = 41, 1283, 7
    rng = np.random.default_rng(3)
    masks = rng.integers(0, 256, (S, h, w)).astype(np.uint8)
    masks[rng.random((S, h, w)) < 0.4] = 0
    d = torch.from_numpy(masks).cuda()
    cc = blobs.ConnectedComponents(w, h, max_images=S)
    cc.label_batch_dev(d.data_ptr(), w, h, S)
    for s in range(S):
        rects = moment_rects(w, h, s)
        flat = np.ascontiguousarray(np.asarray(rects, np.int32).reshape(-1))
        out = (C.c_uint64 * (6 * len(rects)))()
        capi.check(capi.lib().bgsb_ccl_rect_moments_of(cc._h, s, flat.ctypes.data_as(capi.i32p), len(rects), out))
        for i, r in enumerate(rects):
            assert list(out[6 * i:6 * i + 6]) == numpy_moments(masks[s], r), (s, r)
    cc.close()


def test_moments_kernel_bits_on_seven_streams(oracle):
    """rect_moments_bits_kernel on the pipeline's bit-packed masks of 7 streams, rows of 41 words."""
    import torch
    from tracking_b200.pipeline import ForegroundPipeline
    h, w, S = 37, 1301, 7
    rng = np.random.default_rng(4)
    pipe = ForegroundPipeline(MOG2, nstreams=S, morph=())
    d_mask = torch.zeros((S, h, w), dtype=torch.uint8, device="cuda")
    a = rng.integers(0, 256, (S, h, w, 3)).astype(np.uint8)
    b = np.where(rng.random((S, h, w, 1)) < 0.4, a ^ 128, a)       # the model has learnt `a`: 40 % foreground
    for f in (a, b):
        d_in = torch.from_numpy(f).cuda()
        assert pipe.process_dev(d_in.data_ptr(), w, h, d_mask.data_ptr())[0]
    masks = d_mask.cpu().numpy()
    assert 0.05 < (masks > 0).mean() < 0.95
    for s in range(S):
        rects = moment_rects(w, h, 10 + s)
        got = pipe.rect_moments(rects, s)
        for r, g in zip(rects, got):
            assert g == numpy_moments(masks[s], r), (s, r)
    pipe.close()


# ---------------------------------------------------------------------------------------------------------------------
# what a detect call runs and copies

def profiled(fn, tmpdir):
    """-> (Counter of library kernels, list of (kind, bytes) of the memory copies), fn's result"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
    path = os.path.join(str(tmpdir), "trace.json")
    prof.export_chrome_trace(path)
    with open(path) as f:
        trace = json.load(f)
    kernels, copies = collections.Counter(), []
    for e in trace.get("traceEvents", []):
        if e.get("cat") == "kernel" and "_kernel" in e.get("name", ""):
            name = [p for p in e["name"].replace("(", " ").replace("<", " ").replace(":", " ").split() if p.endswith("_kernel")]
            kernels[name[0]] += 1
        elif e.get("cat") == "gpu_memcpy":
            copies.append((e["name"], int(e["args"]["bytes"])))
    return kernels, copies, out


def test_detect_runs_one_moments_launch_and_copies_no_mask(tmp_path):
    import torch
    from tracking_b200 import blobs
    from tracking_b200.pipeline import ForegroundPipeline
    from tracking_b200.streams import StreamPool
    h, w, S = 1080, 1920, 3
    mask_bytes = h * w
    d = torch.empty((S, 4, h, w, 3), dtype=torch.uint8, device="cuda")
    capi.check(capi.lib().bgsb_synth_frames_dev(C.c_void_p(d.data_ptr()), S, 4, w, h, 0, 11, None))
    frames = d.cpu().numpy()
    pipe = ForegroundPipeline(MOG2, nstreams=S)
    dets = [blobs.CvBlobDetectorCC() for _ in range(S)]
    for t in range(4):
        f = torch.from_numpy(np.ascontiguousarray(frames[:, t])).cuda()
        pipe.process_dev(f.data_ptr(), w, h)
        torch.cuda.synchronize()
        if t == 3:
            kernels, copies, got = profiled(lambda: pipe.detect(dets), tmp_path)
        else:
            pipe.detect(dets)
    assert sum(len(f) for _, _, f in got) > 0
    assert dict(kernels) == {"ccl_gather_kernel": 1, "rect_moments_bits_kernel": 1}, dict(kernels)
    h2d = [b for k, b in copies if "HtoD" in k]
    d2h = [b for k, b in copies if "DtoH" in k]
    assert len(h2d) == 1 and h2d[0] % 32 == 0, copies                 # the records
    assert len(d2h) == 2 and d2h[1] == 48 * h2d[0] // 32, copies      # the tables, then the sums
    assert max(b for _, b in copies) < mask_bytes, copies
    pipe.close()

    groups = 2
    pool = StreamPool(MOG2, S, w, h, devices=[0] * groups, ring=1)
    dets = [blobs.CvBlobDetectorCC() for _ in range(S)]
    for t in range(4):
        for s in range(S):
            pool.frame_buffer(s, 0)[...] = frames[s, t]
        pool.submit(0, detect=True)
        pool.wait(0)
        if t == 3:
            kernels, copies, got = profiled(lambda: pool.detect(0, dets), tmp_path)
        else:
            pool.detect(0, dets)
    assert all(g is not None for g in got)
    assert dict(kernels) == {"rect_moments_kernel": groups}, dict(kernels)
    h2d = sorted(b for k, b in copies if "HtoD" in k)
    d2h = sorted(b for k, b in copies if "DtoH" in k)
    assert len(h2d) == groups and [48 * b // 32 for b in h2d] == d2h, copies
    assert max(b for _, b in copies) < mask_bytes, copies
    pool.close()
