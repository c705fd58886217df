"""YUV 4:2:0 input ("inputFormat" NV12 / I420) on every entry path.

A YUV frame must give exactly what cv::cvtColor(COLOR_YUV2BGR_NV12 / _I420) followed by the BGR path gives.  Each test
feeds a YUV context and a BGR context fed the restated conversion (tests/yuv_restate.py, pinned against cv2 on all
2^24 triples by tests/test_yuv_input.py) in lockstep and requires identical masks, background images and (MOG2)
model state, and equality with the oracle's plugins.  The kernel rows check by name (torch.profiler) that the
conversion kernel (csrc/ingest/yuv420.cu) runs where it should and that the plugin kernels are the BGR run's, and by the
library's own launch counter (bgsb_kernel_launch_count) that it adds exactly one launch per band / call / frame set and
that no BGR call launches it.
"""
import collections
import glob
import os
import re
import warnings

import numpy as np
import pytest

from oracle import restate
from tracking_b200 import capi
from yuv_restate import yuv420_to_bgr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NV12, I420, BGR = capi.INPUT_NV12, capi.INPUT_I420, capi.INPUT_BGR
FMTS = [NV12, I420]
AIDS = [0, 1, 2, 3, 5, 6, 7, 9, 11, 12, 13, 14, 35]
CONVERT = "yuv420_to_bgr_kernel"
SENTINEL, GUARD = 0xA5, 64

KERNEL_DECL = re.compile(r"__global__\s+(?:void\s+)?(?:__launch_bounds__\([^)]*\)\s*)?(?:void\s+)?(\w+)\s*\(")
KERNEL_NAME = re.compile(r"\w+_kernel")

# every __global__ of csrc/ingest/ and the rows below that expect it
INGEST_ROWS = {CONVERT: ["test_conversion_kernel_runs_once_per_band_call_and_frame_set",
                         "test_every_triple_through_mog2_frame_zero"]}


def kernels_in(pattern):
    names = set()
    for path in sorted(glob.glob(os.path.join(ROOT, "tracking_b200", "csrc", pattern))):
        with open(path) as f:
            names.update(KERNEL_DECL.findall(f.read()))
    return names


def test_every_ingest_kernel_is_expected_by_a_row():
    found = kernels_in(os.path.join("ingest", "*.cu"))
    assert found, "no ingest kernels found"
    assert found <= set(INGEST_ROWS), "ingest kernels without a row here: %s" % sorted(found - set(INGEST_ROWS))
    names = set(globals())
    for k, rows in INGEST_ROWS.items():
        assert rows and all(r in names for r in rows), (k, rows)


# ---------------------------------------------------------------------------------------------------------------------
# helpers

def yuv_scene(n, h, w, seed):
    """n frames of a noisy static scene crossed by a bright and a dark block, relit on every fifth frame, as Y / U / V
    planes -> list of (Y, U, V)"""
    rng = np.random.default_rng(seed)
    by = rng.integers(30, 220, (h, w)).astype(np.int16)
    bu = rng.integers(60, 200, (h // 2, w // 2)).astype(np.int16)
    bv = rng.integers(60, 200, (h // 2, w // 2)).astype(np.int16)
    out = []
    for t in range(n):
        Y = by + rng.integers(-6, 7, (h, w))
        U = bu + rng.integers(-3, 4, bu.shape)
        V = bv + rng.integers(-3, 4, bv.shape)
        if t % 5 == 4:
            Y += 30
        y, x = (4 * t) % max(h - 8, 2) // 2 * 2, (8 * t) % max(w - 12, 2) // 2 * 2
        Y[y:y + 8, x:x + 12] = 250
        U[y // 2:y // 2 + 4, x // 2:x // 2 + 6] = 30
        V[y // 2:y // 2 + 4, x // 2:x // 2 + 6] = 220
        Y[(y + h // 2) % h:(y + h // 2) % h + 6, (x + w // 3) % w:(x + w // 3) % w + 10] //= 3
        out.append(tuple(np.clip(a, 0, 255).astype(np.uint8) for a in (Y, U, V)))
    return out


def pack(planes, fmt):
    Y, U, V = planes
    h, w = Y.shape
    if fmt == I420:
        return np.concatenate([Y.reshape(-1), U.reshape(-1), V.reshape(-1)]).reshape(h * 3 // 2, w)
    return np.concatenate([Y, np.stack([U, V], -1).reshape(h // 2, w)], 0)


def to_bgr(planes):
    return yuv420_to_bgr(pack(planes, NV12), NV12)


def frames_of(n, h, w, seed, fmt):
    """-> (YUV frames of fmt, the restated BGR frames)"""
    sc = yuv_scene(n, h, w, seed)
    return [pack(p, fmt) for p in sc], [to_bgr(p) for p in sc]


def eq(a, b, what):
    assert (a is None) == (b is None), "%s: validity %s vs %s" % (what, a is None, b is None)
    if a is not None:
        d = np.flatnonzero(np.asarray(a).reshape(-1) != np.asarray(b).reshape(-1))
        assert d.size == 0, "%s: %d bytes differ, first at %s" % (what, d.size, d[:5].tolist())


def plugin(aid, fmt=BGR, **kw):
    import tracking_b200 as tb
    p = tb.ALGOS[aid](**kw)
    if fmt != BGR:
        p.set("inputFormat", fmt)
    return p


def oracles(aid, n=1):
    return [restate.ALGOS[aid]() for _ in range(n)]


def launches(fn):
    """-> (kernels the library launched during fn(), as counted by bgsb_kernel_launch_count; fn's result)"""
    n0 = capi.kernel_launch_count()
    out = fn()
    return capi.kernel_launch_count() - n0, out


def profiled(fn):
    """Run fn() under the CUDA profiler; -> (Counter of library kernel names, fn's result)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    known = kernels_in("*.cu") | kernels_in(os.path.join("ingest", "*.cu"))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore", UserWarning)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        events = prof.events()
    seen = collections.Counter()
    for e in events:
        if e.device_type == torch.autograd.DeviceType.CUDA:
            m = KERNEL_NAME.search(e.name)
            if m and m.group(0) in known:
                seen[m.group(0)] += 1
    return seen, out


class Guarded:
    """`n` bytes at byte offset `off` inside a larger uint8 device allocation; everything around them is SENTINEL."""

    def __init__(self, n, off):
        import torch
        self.n, self.off = n, off
        self.base = torch.full((GUARD + off + n + GUARD,), SENTINEL, dtype=torch.uint8, device="cuda")
        self.view = self.base[GUARD + off:GUARD + off + n]

    @property
    def ptr(self):
        return self.view.data_ptr()

    def put(self, arr):
        import torch
        self.view.copy_(torch.from_numpy(np.ascontiguousarray(arr).reshape(-1)))

    def get(self, shape):
        return self.view.cpu().numpy().reshape(shape)

    def check(self, what):
        b = self.base.cpu().numpy()
        assert (b[:GUARD + self.off] == SENTINEL).all() and (b[GUARD + self.off + self.n:] == SENTINEL).all(), \
            "%s: guard bytes changed" % what


# ---------------------------------------------------------------------------------------------------------------------
# the conversion itself, exhaustively

def every_triple_planes():
    H = W = 4096
    by, bx = np.mgrid[0:H // 2, 0:W // 2]
    blk = by * (W // 2) + bx
    uv, yg = blk % 65536, blk // 65536
    U, V = (uv & 255).astype(np.uint8), (uv >> 8).astype(np.uint8)
    Y = np.empty((H, W), np.uint8)
    for dy in range(2):
        for dx in range(2):
            Y[dy::2, dx::2] = (yg * 4 + dy * 2 + dx).astype(np.uint8)
    return Y, U, V


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_every_triple_through_mog2_frame_zero(fmt):
    """MOG2's frame-0 background image is the frame itself (SURVEY A.4): on the 4096 x 4096 frame that holds every
    (Y, U, V) triple it must equal the restated conversion byte for byte -- host path (banded) and device path."""
    import torch
    img = pack(every_triple_planes(), fmt)
    want = yuv420_to_bgr(img, fmt)
    h, w = want.shape[:2]
    p = plugin(5, fmt)
    fg, bg = p.process(img)
    eq(bg, want, "host background")
    q = plugin(5, fmt)
    d = torch.from_numpy(img).cuda()
    dfg = torch.empty((h, w), dtype=torch.uint8, device="cuda")
    dbg = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
    q.process_dev(d.data_ptr(), w, h, dfg.data_ptr(), dbg.data_ptr())
    torch.cuda.synchronize()
    eq(dbg.cpu().numpy(), want, "device background")


# ---------------------------------------------------------------------------------------------------------------------
# host paths: bgsb_process (small ragged and banded), bgsb_submit, fan-out

@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("h,w", [(98, 130), (600, 700)])
def test_process_all_plugins(fmt, h, w):
    yuv, bgr = frames_of(5, h, w, seed=h + fmt, fmt=fmt)
    for aid in AIDS:
        p, r, o = plugin(aid, fmt), plugin(aid), oracles(aid)[0]
        for t in range(len(yuv)):
            fg, bg = p.process(yuv[t])
            rfg, rbg = r.process(bgr[t])
            ofg, obg = o.process(bgr[t])
            eq(fg, rfg, "aid %d t %d mask vs BGR" % (aid, t))
            eq(bg, rbg, "aid %d t %d background vs BGR" % (aid, t))
            eq(fg, ofg, "aid %d t %d mask vs oracle" % (aid, t))
            if obg is not None and bg is not None:
                eq(bg, obg, "aid %d t %d background vs oracle" % (aid, t))
        if aid == 5:
            for a, b in zip(p.export_state(), r.export_state()):
                eq(a, b, "MOG2 state")
        p.close(); r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_strided_nv12_and_groups_on_the_host_path(fmt):
    """NV12 rows `stride` apart (padded), and a group of 3 streams back to back"""
    import tracking_b200 as tb
    h, w, S = 66, 90, 3
    seqs = [frames_of(4, h, w, seed=40 + s, fmt=fmt) for s in range(S)]
    p = tb.ALGOS[5](nstreams=S, inputFormat=fmt)
    os_ = oracles(5, S)
    for t in range(4):
        img = np.stack([seqs[s][0][t] for s in range(S)])
        if fmt == NV12:
            wide = np.zeros((S, h * 3 // 2, w + 22), np.uint8)
            wide[:, :, :w] = img
            img = wide[:, :, :w]
        fg, bg = p.process(img)
        for s in range(S):
            ofg, obg = os_[s].process(seqs[s][1][t])
            eq(fg[s], ofg, "stream %d mask" % s)
            eq(bg[s], obg, "stream %d background" % s)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_submit_all_plugins(fmt):
    from tracking_b200.bgs import pinned_empty
    h, w, n = 98, 130, 5
    yuv, bgr = frames_of(n, h, w, seed=7 + fmt, fmt=fmt)
    for aid in AIDS:
        p, r = plugin(aid, fmt), plugin(aid)
        bgch = p.BG_CHANNELS
        ins, fgs, bgs_, valid = [], [], [], []
        for t in range(n):
            a = pinned_empty(yuv[t].shape)
            a[...] = yuv[t]
            f = pinned_empty((h, w))
            b = pinned_empty((h, w, 3) if bgch == 3 else (h, w))
            valid.append(p.submit(a, f, b))
            ins.append(a); fgs.append(f); bgs_.append(b)
        p.wait()
        for t in range(n):
            rfg, rbg = r.process(bgr[t])
            eq(fgs[t] if valid[t][0] else None, rfg, "aid %d t %d submit mask" % (aid, t))
            eq(bgs_[t] if valid[t][1] else None, rbg, "aid %d t %d submit background" % (aid, t))
        p.close(); r.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("h,w", [(98, 130), (600, 700)])
def test_fanout_all_plugins(fmt, h, w):
    from tracking_b200.bgs import process_fanout
    yuv, bgr = frames_of(4, h, w, seed=3 * h + fmt, fmt=fmt)
    ps = [plugin(aid, fmt) for aid in AIDS]
    os_ = [oracles(aid)[0] for aid in AIDS]
    for t in range(len(yuv)):
        got = process_fanout(ps, yuv[t])
        for k, aid in enumerate(AIDS):
            ofg, obg = os_[k].process(bgr[t])
            eq(got[k][0], ofg, "fan-out aid %d t %d mask" % (aid, t))
            if obg is not None and got[k][1] is not None:
                eq(got[k][1], obg, "fan-out aid %d t %d background" % (aid, t))
    # each context then goes on on its own
    fg, _ = ps[4].process(yuv[0])
    eq(fg, os_[4].process(bgr[0])[0], "MOG2 after fan-out")
    for p in ps:
        p.close()


# ---------------------------------------------------------------------------------------------------------------------
# device paths: process_dev (guard bytes, misaligned offsets), process_batch_dev (T = 3 on a group of 3)

@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("off", [0, 3])
def test_process_dev_all_plugins_guarded(fmt, off):
    h, w, n = 66, 130, 4
    yuv, bgr = frames_of(n, h, w, seed=11 + off + fmt, fmt=fmt)
    for aid in AIDS:
        p, o = plugin(aid, fmt), oracles(aid)[0]
        bgch = p.BG_CHANNELS
        fg = Guarded(h * w, off + 5)
        bg = Guarded(h * w * bgch, off + 7)
        for t in range(n):
            fr = Guarded(yuv[t].size, off + t)       # a different alignment on every call
            fr.put(yuv[t])
            fg.view.fill_(SENTINEL); bg.view.fill_(SENTINEL)
            fv, bv = p.process_dev(fr.ptr, w, h, fg.ptr, bg.ptr)
            ofg, obg = o.process(bgr[t])
            eq(fg.get((h, w)) if fv else None, ofg, "aid %d t %d dev mask" % (aid, t))
            if obg is not None and bv:
                eq(bg.get(obg.shape), obg, "aid %d t %d dev background" % (aid, t))
            for g, what in ((fr, "frame"), (fg, "mask"), (bg, "background")):
                g.check("aid %d %s" % (aid, what))
        p.close()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_process_batch_dev_all_plugins(fmt):
    import torch
    import tracking_b200 as tb
    h, w, S, T, nb = 34, 98, 3, 3, 2
    seqs = [frames_of(T * nb, h, w, seed=21 + s + fmt, fmt=fmt) for s in range(S)]
    for aid in AIDS:
        p = tb.ALGOS[aid](nstreams=S, inputFormat=fmt)
        r = tb.ALGOS[aid](nstreams=S)
        bgch = p.BG_CHANNELS
        for b in range(nb):
            d = torch.from_numpy(np.stack([np.stack(seqs[s][0][b * T:(b + 1) * T]) for s in range(S)])).cuda()
            db = torch.from_numpy(np.stack([np.stack(seqs[s][1][b * T:(b + 1) * T]) for s in range(S)])).cuda()
            outs = []
            for ctx, frames in ((p, d), (r, db)):
                fg = torch.zeros((S, T, h, w), dtype=torch.uint8, device="cuda")
                bg = torch.zeros((S, T, h, w) + ((3,) if bgch == 3 else ()), dtype=torch.uint8, device="cuda")
                first, bv = ctx.process_batch_dev(frames.data_ptr(), T, w, h, fg.data_ptr(), bg.data_ptr())
                torch.cuda.synchronize()
                outs.append((first, bv, fg.cpu().numpy(), bg.cpu().numpy()))
            (f0, b0, fg0, bg0), (f1, b1, fg1, bg1) = outs
            assert (f0, b0) == (f1, b1)
            eq(fg0[:, f0:], fg1[:, f0:], "aid %d batch %d masks" % (aid, b))
            if b0:
                eq(bg0[:, f0:], bg1[:, f0:], "aid %d batch %d backgrounds" % (aid, b))
        if aid == 5:
            for s in range(S):
                for a, c in zip(p.export_state(s), r.export_state(s)):
                    eq(a, c, "MOG2 state stream %d" % s)
        p.close(); r.close()


# ---------------------------------------------------------------------------------------------------------------------
# format switching

@pytest.mark.gpu
@pytest.mark.parametrize("aid", [0, 3, 5, 35])
def test_alternating_formats_equal_the_bgr_run(aid):
    import torch
    h, w, n = 66, 98, 9
    sc = yuv_scene(n, h, w, seed=50 + aid)
    bgr = [to_bgr(x) for x in sc]
    host, dev, ref = plugin(aid), plugin(aid), plugin(aid)
    fmts = [BGR, NV12, I420]
    bgch = ref.BG_CHANNELS
    for t in range(n):
        fmt = fmts[t % 3]
        frame = bgr[t] if fmt == BGR else pack(sc[t], fmt)
        host.set("inputFormat", fmt); dev.set("inputFormat", fmt)
        fg, bg = host.process(frame)
        d = torch.from_numpy(np.ascontiguousarray(frame)).cuda()
        dfg = torch.zeros((h, w), dtype=torch.uint8, device="cuda")
        dbg = torch.zeros((h, w, 3) if bgch == 3 else (h, w), dtype=torch.uint8, device="cuda")
        fv, bv = dev.process_dev(d.data_ptr(), w, h, dfg.data_ptr(), dbg.data_ptr())
        torch.cuda.synchronize()
        rfg, rbg = ref.process(bgr[t])
        eq(fg, rfg, "host mask t %d" % t)
        eq(bg, rbg, "host background t %d" % t)
        eq(dfg.cpu().numpy() if fv else None, rfg, "dev mask t %d" % t)
        eq(dbg.cpu().numpy() if bv else None, rbg, "dev background t %d" % t)


# ---------------------------------------------------------------------------------------------------------------------
# pipeline and pool

@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("algo", [5, 0])
def test_pipeline_equals_the_bgr_run(fmt, algo):
    import torch
    from tracking_b200 import blobs
    from tracking_b200.pipeline import ForegroundPipeline
    h, w, S, n = 120, 160, 2, 6
    seqs = [frames_of(n, h, w, seed=60 + s + fmt, fmt=fmt) for s in range(S)]
    py = ForegroundPipeline(algo, nstreams=S, inputFormat=fmt)
    pb = ForegroundPipeline(algo, nstreams=S)
    dy = [blobs.CvBlobDetectorCC() for _ in range(S)]
    db = [blobs.CvBlobDetectorCC() for _ in range(S)]
    for t in range(n):
        outs = []
        for pipe, k in ((py, 0), (pb, 1)):
            d = torch.from_numpy(np.stack([seqs[s][k][t] for s in range(S)])).cuda()
            lab = torch.zeros((S, h, w), dtype=torch.int32, device="cuda")
            v, _ = pipe.process_dev(d.data_ptr(), w, h, d_labels=lab.data_ptr())
            torch.cuda.synchronize()
            outs.append((v, lab.cpu().numpy()))
        assert outs[0][0] == outs[1][0]
        if not outs[0][0]:
            continue
        eq(outs[0][1], outs[1][1], "labels t %d" % t)
        for s in range(S):
            assert py.components(s) == pb.components(s), "table stream %d t %d" % (s, t)
        assert py.detect(dy) == pb.detect(db), "detect t %d" % t


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_pool_equals_the_bgr_run(fmt):
    from tracking_b200 import blobs
    from tracking_b200.streams import StreamPool
    h, w, S, n = 96, 128, 4, 5
    seqs = [frames_of(n, h, w, seed=70 + s + fmt, fmt=fmt) for s in range(S)]
    py = StreamPool(5, S, w, h, devices=[0, 0], ring=2, inputFormat=fmt)
    pb = StreamPool(5, S, w, h, devices=[0, 0], ring=2)
    assert py.table_rows == pb.table_rows == 256
    assert py.frame_buffer(0, 0).shape == (h * 3 // 2, w)
    dy = [blobs.CvBlobDetectorCC() for _ in range(S)]
    db = [blobs.CvBlobDetectorCC() for _ in range(S)]
    for t in range(n):
        slot = t % 2
        for pool, k in ((py, 0), (pb, 1)):
            for s in range(S):
                pool.frame_buffer(s, slot)[...] = seqs[s][k][t]
            pool.submit(slot, want_masks=True, detect=True)
        vy, vb = py.wait(slot), pb.wait(slot)
        assert vy == vb
        if not vy:
            continue
        for s in range(S):
            eq(py.mask(s, slot), pb.mask(s, slot), "pool mask stream %d t %d" % (s, t))
            assert py.components(s, slot) == pb.components(s, slot)
        assert py.detect(slot, dy) == pb.detect(slot, db), "pool detect t %d" % t
    with pytest.raises(capi.BgsbError) as e:
        capi.check(capi.lib().bgsb_pool_set_param(py._h, b"inputFormat", float(BGR)))
    assert e.value.code == capi.ERR_ARG and b"before the first submit" in capi.lib().bgsb_last_error()
    py.close(); pb.close()


# ---------------------------------------------------------------------------------------------------------------------
# refusals

def refused(fn, text):
    with pytest.raises(capi.BgsbError) as e:
        fn()
    assert e.value.code == capi.ERR_ARG, e.value
    assert text in str(e.value), str(e.value)


@pytest.mark.gpu
def test_refusals():
    import ctypes as C
    import torch
    from tracking_b200.bgs import process_fanout
    from tracking_b200.pipeline import ForegroundPipeline
    from tracking_b200.streams import StreamPool
    L = capi.lib()
    p = plugin(5, NV12)
    refused(lambda: p.set("inputFormat", 3), "inputFormat is 0")
    refused(lambda: p.set("inputFormat", -1), "inputFormat is 0")
    refused(lambda: p.set("retainInput", 1), "retainInput cannot be combined")
    fd = plugin(0)
    fd.set("retainInput", 1)
    refused(lambda: fd.set("inputFormat", NV12), "cannot be combined with retainInput")
    img = np.zeros((8 * 3 // 2, 10), np.uint8)
    fg = np.zeros((8, 10), np.uint8)
    bg = np.zeros((8, 10, 3), np.uint8)
    v = C.c_int()

    def host(call, ctx, w, h, stride):
        return lambda: capi.check(getattr(L, call)(ctx._h, img.ctypes.data, w, h, stride, fg.ctypes.data, w,
                                                   bg.ctypes.data, 3 * w, C.byref(v), C.byref(v)))
    for call in ("bgsb_process", "bgsb_submit"):
        refused(host(call, p, 9, 8, 10), "even width and height")
        refused(host(call, p, 10, 7, 10), "even width and height")
        q = plugin(5, I420)
        refused(host(call, q, 10, 8, 12), "stride must equal w")
        q.close()
    d = torch.zeros(4096, dtype=torch.uint8, device="cuda")
    refused(lambda: p.process_dev(d.data_ptr(), 9, 8, d.data_ptr()), "even width and height")
    refused(lambda: p.process_batch_dev(d.data_ptr(), 2, 10, 7, d.data_ptr()), "even width and height")
    # fan-out: one format for all contexts, even sizes
    a, b = plugin(5, NV12), plugin(0)
    refused(lambda: process_fanout([a, b], img), "share one")
    fgp = (C.c_void_p * 1)(fg.ctypes.data)
    fst = (C.c_size_t * 1)(9)
    ctx = (C.c_void_p * 1)(a._h)
    refused(lambda: capi.check(L.bgsb_process_fanout(ctx, 1, img.ctypes.data, 9, 8, 10, fgp, fst, None, None, None, None)),
            "even width and height")
    pipe = ForegroundPipeline(5, nstreams=1, inputFormat=I420)
    refused(lambda: pipe.process_dev(d.data_ptr(), 10, 9), "even width and height")
    refused(lambda: StreamPool(5, 2, 9, 8, devices=[0], ring=2, inputFormat=NV12), "even width and height")
    refused(lambda: StreamPool(5, 2, 10, 8, devices=[0], ring=2, inputFormat=5), "inputFormat is 0")
    assert p.get("inputFormat") == NV12 and fd.get("inputFormat") == BGR
    for x in (p, fd, a, b):
        x.close()
    pipe.close()


# ---------------------------------------------------------------------------------------------------------------------
# which kernels run

def kernel_rows(fmt):
    """the body of test_conversion_kernel_runs_once_per_band_call_and_frame_set, in a fresh process"""
    import torch
    import tracking_b200 as tb
    from tracking_b200.pipeline import ForegroundPipeline
    # bgsb_process, banded (1080p with the background image: 3 bands) and whole (small frame)
    for (h, w) in ((1080, 1920), (66, 98)):
        yuv, bgr = frames_of(3, h, w, seed=80, fmt=fmt)
        p, r = plugin(5, fmt, trace=1), plugin(5, trace=1)
        for t in range(2):
            p.process(yuv[t]); r.process(bgr[t])
        # the library's own launch counter: one conversion per band, nothing else added (the host path's kernels run
        # on the context's streams, whose activity records torch.profiler does not reliably deliver late in a long
        # session; the kernel names are checked on the device paths below)
        ny, _ = launches(lambda: p.process(yuv[2]))
        bands = p.trace_last()["bands"]
        nb, _ = launches(lambda: r.process(bgr[2]))
        assert (h, bands) != (1080, 1), "the 1080p frame was not banded"
        assert r.trace_last()["bands"] == bands
        assert ny - nb == bands, (ny, nb, bands)
        p.close(); r.close()
    # process_dev and process_batch_dev: once per call; pipeline: once per frame set
    h, w, S, T = 66, 98, 3, 3
    seqs = [frames_of(T, h, w, seed=90 + s, fmt=fmt) for s in range(S)]
    for T_ in (1, T):
        p = tb.ALGOS[5](nstreams=S, inputFormat=fmt)
        r = tb.ALGOS[5](nstreams=S)
        d = torch.from_numpy(np.stack([np.stack(seqs[s][0][:T_]) for s in range(S)])).cuda()
        db = torch.from_numpy(np.stack([np.stack(seqs[s][1][:T_]) for s in range(S)])).cuda()
        fg = torch.zeros((S, T_, h, w), dtype=torch.uint8, device="cuda")
        for _ in range(2):
            got, _ = profiled(lambda: p.process_batch_dev(d.data_ptr(), T_, w, h, fg.data_ptr()))
            ref, _ = profiled(lambda: r.process_batch_dev(db.data_ptr(), T_, w, h, fg.data_ptr()))
            assert CONVERT in got and CONVERT not in ref
            assert {k for k in got if k != CONVERT} == set(ref), (got, ref)
            ny, _ = launches(lambda: p.process_batch_dev(d.data_ptr(), T_, w, h, fg.data_ptr()))
            nb, _ = launches(lambda: r.process_batch_dev(db.data_ptr(), T_, w, h, fg.data_ptr()))
            assert ny - nb == 1, (T_, ny, nb)
        p.close(); r.close()
    pipes = [ForegroundPipeline(5, nstreams=S, inputFormat=fmt), ForegroundPipeline(5, nstreams=S)]
    for t in range(T):
        runs, counts = [], []
        for pipe, k in zip(pipes, (0, 1)):
            d = torch.from_numpy(np.stack([seqs[s][k][t] for s in range(S)])).cuda()
            call = lambda: (pipe.process_dev(d.data_ptr(), w, h), pipe.join_dev())  # noqa: E731
            runs.append(profiled(call)[0] if t != 1 else None)
            if t == 1:
                counts.append(launches(call)[0])
        if t == 1:
            assert counts[0] - counts[1] == 1, counts       # one conversion launch per frame set
        else:
            assert CONVERT in runs[0] and CONVERT not in runs[1]
            assert {k for k in runs[0] if k != CONVERT} == set(runs[1]), runs
    # a BGR context that once took YUV frames launches no conversion again
    p = plugin(5, fmt)
    p.process(frames_of(1, h, w, seed=1, fmt=fmt)[0][0])
    p.set("inputFormat", BGR)
    bgr0 = frames_of(1, h, w, seed=1, fmt=fmt)[1][0]
    r = plugin(5)
    r.process(bgr0)
    assert launches(lambda: p.process(bgr0))[0] == launches(lambda: r.process(bgr0))[0]
    print("ok kernel rows")


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", FMTS)
def test_conversion_kernel_runs_once_per_band_call_and_frame_set(fmt):
    """Runs in a child process: late in a long test session torch.profiler has been seen to deliver none or only part
    of a call's kernel records, so the rows start from a fresh profiler state, as a standalone run of this file does."""
    import subprocess
    import sys
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_yuv_input as m; m.kernel_rows(%d)"
            % (ROOT, os.path.join(ROOT, "tests"), fmt))
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
    assert "ok kernel rows" in res.stdout, res.stdout
