"""The PreProcessor's 7x7 Gaussian blur ("gaussianBlur" 1) on every entry path.

A blurred context must give exactly what cv::GaussianBlur(img, Size(7, 7), 1.5) followed by the unblurred path gives.
Each test runs a blur context fed raw frames beside a blur-off context fed the restated blur (tests/gauss_restate.py,
pinned against cv2 by tests/test_gaussian_blur.py) in lockstep and requires identical masks, background images and
(MOG2) model state, and equality with the oracle's plugins fed cv2.GaussianBlur frames.  The kernel rows check by name
(torch.profiler) that the blur kernel (csrc/prep/gauss7.cu) runs where it should and that the plugin kernels are the
unblurred run's, and by the library's own launch counter that it adds exactly one launch per band / call / frame set
and that no blur-off call launches it.

The file's name sorts it after test_gpu_kernel_routes.py on purpose: that file reads kernel names from torch.profiler in
the test process, and when this file's many launches ran between an earlier in-process profiler session
(test_gpu_detect_streams.py) and it, the profiler delivered no kernel records to its rows.
"""
import os

import numpy as np
import pytest

from gauss_restate import gauss7
from test_gpu_yuv_input import (AIDS, KERNEL_NAME, SENTINEL, Guarded, eq, kernels_in, launches, oracles, pack,
                                refused, yuv_scene)
from tracking_b200 import capi
from yuv_restate import yuv420_to_bgr

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NV12, I420, BGR = capi.INPUT_NV12, capi.INPUT_I420, capi.INPUT_BGR
BLUR = "gauss7_kernel"

# every __global__ of csrc/prep/ and the rows below that expect it
PREP_ROWS = {BLUR: ["test_blur_kernel_runs_once_per_band_call_and_frame_set",
                    "test_kernel_exactly_through_mog2_frame_zero", "test_kernel_exactly_on_guarded_device_frames"]}


def test_every_prep_kernel_is_expected_by_a_row():
    found = kernels_in(os.path.join("prep", "*.cu"))
    assert found, "no pre-processing kernels found"
    assert found <= set(PREP_ROWS), "pre-processing kernels without a row here: %s" % sorted(found - set(PREP_ROWS))
    names = set(globals())
    for k, rows in PREP_ROWS.items():
        assert rows and all(r in names for r in rows), (k, rows)


# ---------------------------------------------------------------------------------------------------------------------
# helpers

def profiled(fn):
    """Run fn() under the CUDA profiler; -> (Counter of library kernel names, fn's result)."""
    import collections
    import warnings
    import torch
    from torch.profiler import ProfilerActivity, profile
    known = kernels_in("*.cu") | kernels_in(os.path.join("ingest", "*.cu")) | kernels_in(os.path.join("prep", "*.cu"))
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


def blurred(img):
    """the restated blur, equal to cv2.GaussianBlur(img, (7, 7), 1.5) (tests/test_gaussian_blur.py; kernel_rows checks
    it again on this file's frames, in its own process)"""
    return gauss7(img)


def scene(n, h, w, seed):
    """n BGR frames: noise over a static scene, a moving bright block, a relit frame every fifth, and rows that change
    sharply every 32 rows (host-path bands start on multiples of 32 rows)"""
    rng = np.random.default_rng(seed)
    base = rng.integers(20, 230, (h, w, 3)).astype(np.int16)
    stripe = ((np.arange(h) // 32) % 2 * 90 - 45).astype(np.int16)[:, None, None]
    out = []
    for t in range(n):
        f = base + stripe + rng.integers(-8, 9, (h, w, 3))
        if t % 5 == 4:
            f += 25
        y, x = (5 * t) % max(h - 10, 1), (9 * t) % max(w - 14, 1)
        f[y:y + 10, x:x + 14] = 255
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


def adversarial(h, w):
    """impulses at corners and edges, 0/255 checkerboards of pixels and of channels, all-255 rows and columns"""
    yy, xx = np.mgrid[0:h, 0:w]
    f = (((yy[..., None] + xx[..., None] + np.arange(3)) & 1) * 255).astype(np.uint8)
    f[h // 3:h // 2] = ((((yy + xx) & 1) * 255).astype(np.uint8))[h // 3:h // 2, :, None]
    f[:, w // 3:w // 3 + 5] = 255
    f[2 * h // 3:2 * h // 3 + 4] = 0
    for y, x in ((0, 0), (0, w - 1), (h - 1, 0), (h - 1, w - 1), (h // 2, 0), (0, w // 2), (h - 1, w // 2), (h // 2, w - 1)):
        f[max(y - 1, 0):y + 2, max(x - 1, 0):x + 2] = 0
        f[y, x] = (255, 255, 255)
    return f


def plugin(aid, blur=1, fmt=BGR, **kw):
    import tracking_b200 as tb
    p = tb.ALGOS[aid](**kw)
    if fmt != BGR:
        p.set("inputFormat", fmt)
    if blur:
        p.set("gaussianBlur", 1)
    return p


def bg_of_frame_zero(img, host):
    """MOG2's frame-0 background image is its input frame (SURVEY A.4): the blurred frame the plugin saw"""
    import torch
    h, w = img.shape[:2]
    p = plugin(5)
    if host:
        _, bg = p.process(img)
    else:
        d = torch.from_numpy(np.ascontiguousarray(img)).cuda()
        dfg = torch.empty((h, w), dtype=torch.uint8, device="cuda")
        dbg = torch.empty((h, w, 3), dtype=torch.uint8, device="cuda")
        p.process_dev(d.data_ptr(), w, h, dfg.data_ptr(), dbg.data_ptr())
        torch.cuda.synchronize()
        bg = dbg.cpu().numpy()
    p.close()
    return bg


# ---------------------------------------------------------------------------------------------------------------------
# the kernel itself, exactly

@pytest.mark.parametrize("h,w", [(1080, 1920), (1081, 1923), (37, 53), (5, 9), (3, 3), (1, 7), (7, 1), (1, 1), (4, 300)])
def test_kernel_exactly_through_mog2_frame_zero(h, w):
    rng = np.random.default_rng(h * 3 + w)
    for what, img in (("noise", rng.integers(0, 256, (h, w, 3), dtype=np.uint8)), ("adversarial", adversarial(h, w))):
        want = blurred(img)
        for host in (True, False):
            eq(bg_of_frame_zero(img, host), want, "%d x %d %s %s" % (h, w, what, "host" if host else "device"))


@pytest.mark.parametrize("off", [0, 1, 3, 8])
@pytest.mark.parametrize("h,w", [(66, 130), (40, 1921), (9, 5)])
def test_kernel_exactly_on_guarded_device_frames(off, h, w):
    """misaligned frame and output buffers with 0xA5 guard bytes around them: the guard bytes must not change"""
    rng = np.random.default_rng(off + h)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    img[: h // 2] = adversarial(h, w)[: h // 2]
    p = plugin(5)
    fr = Guarded(img.size, off)
    fr.put(img)
    fg, bg = Guarded(h * w, off + 1), Guarded(h * w * 3, off + 2)
    p.process_dev(fr.ptr, w, h, fg.ptr, bg.ptr)
    eq(bg.get((h, w, 3)), blurred(img), "device background off %d" % off)
    for g, what in ((fr, "frame"), (fg, "mask"), (bg, "background")):
        g.check(what)
    assert (fr.get((h, w, 3)) == img).all(), "the caller's frame was modified"
    p.close()


# ---------------------------------------------------------------------------------------------------------------------
# lockstep parity: host paths

def lockstep(aid, frames, blur_run, ref_run, what):
    o = oracles(aid)[0]
    for t, f in enumerate(frames):
        b = blurred(f)
        fg, bg = blur_run(f)
        rfg, rbg = ref_run(b)
        ofg, obg = o.process(b)
        eq(fg, rfg, "%s aid %d t %d mask vs blur-off" % (what, aid, t))
        eq(bg, rbg, "%s aid %d t %d background vs blur-off" % (what, aid, t))
        eq(fg, ofg, "%s aid %d t %d mask vs oracle" % (what, aid, t))
        if obg is not None and bg is not None:
            eq(bg, obg, "%s aid %d t %d background vs oracle" % (what, aid, t))


@pytest.mark.parametrize("h,w", [(98, 131), (600, 700)])
def test_process_all_plugins(h, w):
    """ragged (98 x 131: odd pitch) and banded (600 x 700: bands of 224 rows with the background image, 320 without;
    rows change sharply at every multiple of 32; kernel_rows checks that the frame is banded)"""
    frames = scene(5, h, w, seed=h)
    for aid in AIDS:
        p, r = plugin(aid), plugin(aid, blur=0)
        lockstep(aid, frames, p.process, r.process, "process")
        if aid == 5:
            for a, b in zip(p.export_state(), r.export_state()):
                eq(a, b, "MOG2 state")
        p.close(); r.close()


def test_submit_all_plugins():
    from tracking_b200.bgs import pinned_empty
    h, w, n = 98, 130, 5
    frames = scene(n, h, w, seed=7)
    for aid in AIDS:
        p, r = plugin(aid), plugin(aid, blur=0)
        bgch = p.BG_CHANNELS
        ins, fgs, bgs_, valid = [], [], [], []
        for t in range(n):
            a = pinned_empty(frames[t].shape)
            a[...] = frames[t]
            f = pinned_empty((h, w))
            b = pinned_empty((h, w, 3) if bgch == 3 else (h, w))
            valid.append(p.submit(a, f, b))
            ins.append(a); fgs.append(f); bgs_.append(b)
        p.wait()
        for t in range(n):
            rfg, rbg = r.process(blurred(frames[t]))
            eq(fgs[t] if valid[t][0] else None, rfg, "aid %d t %d submit mask" % (aid, t))
            eq(bgs_[t] if valid[t][1] else None, rbg, "aid %d t %d submit background" % (aid, t))
        if aid == 5:
            for a, b in zip(p.export_state(), r.export_state()):
                eq(a, b, "MOG2 state")
        p.close(); r.close()


@pytest.mark.parametrize("h,w", [(98, 130), (600, 700)])
def test_fanout_all_plugins(h, w):
    from tracking_b200.bgs import process_fanout
    frames = scene(4, h, w, seed=3 * h)
    ps = [plugin(aid) for aid in AIDS]
    os_ = [oracles(aid)[0] for aid in AIDS]
    for t in range(len(frames)):
        b = blurred(frames[t])
        got = process_fanout(ps, frames[t])
        for k, aid in enumerate(AIDS):
            ofg, obg = os_[k].process(b)
            eq(got[k][0], ofg, "fan-out aid %d t %d mask" % (aid, t))
            if obg is not None and got[k][1] is not None:
                eq(got[k][1], obg, "fan-out aid %d t %d background" % (aid, t))
    fg, _ = ps[4].process(frames[0])
    eq(fg, os_[4].process(blurred(frames[0]))[0], "MOG2 after fan-out")
    for p in ps:
        p.close()


# ---------------------------------------------------------------------------------------------------------------------
# device paths

@pytest.mark.parametrize("off", [0, 3])
def test_process_dev_all_plugins_guarded(off):
    h, w, n = 66, 131, 4
    frames = scene(n, h, w, seed=11 + off)
    for aid in AIDS:
        p, o = plugin(aid), oracles(aid)[0]
        bgch = p.BG_CHANNELS
        fg = Guarded(h * w, off + 5)
        bg = Guarded(h * w * bgch, off + 7)
        for t in range(n):
            fr = Guarded(frames[t].size, off + t)
            fr.put(frames[t])
            fg.view.fill_(SENTINEL); bg.view.fill_(SENTINEL)
            fv, bv = p.process_dev(fr.ptr, w, h, fg.ptr, bg.ptr)
            ofg, obg = o.process(blurred(frames[t]))
            eq(fg.get((h, w)) if fv else None, ofg, "aid %d t %d dev mask" % (aid, t))
            if obg is not None and bv:
                eq(bg.get(obg.shape), obg, "aid %d t %d dev background" % (aid, t))
            for g, what in ((fr, "frame"), (fg, "mask"), (bg, "background")):
                g.check("aid %d %s" % (aid, what))
        p.close()


def test_process_batch_dev_all_plugins():
    """T = 3 on a group of 3 streams whose frames differ: a read across a frame or stream boundary would show"""
    import torch
    import tracking_b200 as tb
    h, w, S, T, nb = 34, 98, 3, 3, 2
    seqs = [scene(T * nb, h, w, seed=21 + 5 * s) for s in range(S)]
    for aid in AIDS:
        p = tb.ALGOS[aid](nstreams=S, gaussianBlur=1)
        r = tb.ALGOS[aid](nstreams=S)
        bgch = p.BG_CHANNELS
        for b in range(nb):
            raw = np.stack([np.stack(seqs[s][b * T:(b + 1) * T]) for s in range(S)])
            d = torch.from_numpy(raw).cuda()
            db = torch.from_numpy(np.stack([np.stack([blurred(f) for f in x]) for x in raw])).cuda()
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
            assert (d.cpu().numpy() == raw).all(), "the caller's frames were modified"
        if aid == 5:
            for s in range(S):
                for a, c in zip(p.export_state(s), r.export_state(s)):
                    eq(a, c, "MOG2 state stream %d" % s)
        p.close(); r.close()


# ---------------------------------------------------------------------------------------------------------------------
# YUV input with the blur: decode, then the PreProcessor

@pytest.mark.parametrize("fmt", [NV12, I420])
@pytest.mark.parametrize("h,w", [(98, 130), (600, 700)])
def test_yuv_then_blur(fmt, h, w):
    import torch
    sc = yuv_scene(4, h, w, seed=h + fmt)
    for aid in (0, 3, 5, 35):
        p, dev = plugin(aid, fmt=fmt), plugin(aid, fmt=fmt)
        r, o = plugin(aid, blur=0), oracles(aid)[0]
        for t, planes in enumerate(sc):
            img = pack(planes, fmt)
            b = blurred(yuv420_to_bgr(pack(planes, NV12), NV12))
            fg, bg = p.process(img)
            d = torch.from_numpy(img).cuda()
            dfg = torch.zeros((h, w), dtype=torch.uint8, device="cuda")
            dbg = torch.zeros((h, w, 3) if p.BG_CHANNELS == 3 else (h, w), dtype=torch.uint8, device="cuda")
            fv, bv = dev.process_dev(d.data_ptr(), w, h, dfg.data_ptr(), dbg.data_ptr())
            torch.cuda.synchronize()
            rfg, rbg = r.process(b)
            ofg, _ = o.process(b)
            eq(fg, rfg, "aid %d t %d host mask" % (aid, t))
            eq(bg, rbg, "aid %d t %d host background" % (aid, t))
            eq(fg, ofg, "aid %d t %d host mask vs oracle" % (aid, t))
            eq(dfg.cpu().numpy() if fv else None, rfg, "aid %d t %d dev mask" % (aid, t))
            eq(dbg.cpu().numpy() if bv else None, rbg, "aid %d t %d dev background" % (aid, t))
        for x in (p, dev, r):
            x.close()


# ---------------------------------------------------------------------------------------------------------------------
# a change takes effect from the next frame

@pytest.mark.parametrize("aid", [0, 3, 2, 5, 35])
def test_toggling_the_blur_on_at_frame_k(aid):
    import torch
    h, w, n, k = 66, 98, 7, 3
    frames = scene(n, h, w, seed=50 + aid)
    host, dev, ref = plugin(aid, blur=0), plugin(aid, blur=0), plugin(aid, blur=0)
    bgch = ref.BG_CHANNELS
    for t in range(n):
        on = k <= t < n - 1                     # on from frame k, off again for the last frame
        host.set("gaussianBlur", int(on)); dev.set("gaussianBlur", int(on))
        fg, bg = host.process(frames[t])
        d = torch.from_numpy(frames[t]).cuda()
        dfg = torch.zeros((h, w), dtype=torch.uint8, device="cuda")
        dbg = torch.zeros((h, w, 3) if bgch == 3 else (h, w), dtype=torch.uint8, device="cuda")
        fv, bv = dev.process_dev(d.data_ptr(), w, h, dfg.data_ptr(), dbg.data_ptr())
        torch.cuda.synchronize()
        rfg, rbg = ref.process(blurred(frames[t]) if on else frames[t])
        eq(fg, rfg, "host mask t %d" % t)
        eq(bg, rbg, "host background t %d" % t)
        eq(dfg.cpu().numpy() if fv else None, rfg, "dev mask t %d" % t)
        eq(dbg.cpu().numpy() if bv else None, rbg, "dev background t %d" % t)
    for x in (host, dev, ref):
        x.close()


# ---------------------------------------------------------------------------------------------------------------------
# pipeline and pool

@pytest.mark.parametrize("algo", [5, 0])
def test_pipeline_equals_the_blur_off_run(algo):
    import torch
    from tracking_b200 import blobs
    from tracking_b200.pipeline import ForegroundPipeline
    h, w, S, n = 120, 160, 2, 6
    seqs = [scene(n, h, w, seed=60 + s) for s in range(S)]
    py = ForegroundPipeline(algo, nstreams=S, gaussianBlur=1)
    pb = ForegroundPipeline(algo, nstreams=S)
    dy = [blobs.CvBlobDetectorCC() for _ in range(S)]
    db = [blobs.CvBlobDetectorCC() for _ in range(S)]
    for t in range(n):
        outs = []
        for pipe, blur in ((py, True), (pb, False)):
            d = torch.from_numpy(np.stack([seqs[s][t] if blur else blurred(seqs[s][t]) for s in range(S)])).cuda()
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
    py.close(); pb.close()


def test_pool_equals_the_blur_off_run():
    from tracking_b200 import blobs
    from tracking_b200.streams import StreamPool
    h, w, S, n = 96, 128, 4, 5
    seqs = [scene(n, h, w, seed=70 + s) for s in range(S)]
    py = StreamPool(5, S, w, h, devices=[0, 0], ring=2, gaussianBlur=1)
    pb = StreamPool(5, S, w, h, devices=[0, 0], ring=2)
    dy = [blobs.CvBlobDetectorCC() for _ in range(S)]
    db = [blobs.CvBlobDetectorCC() for _ in range(S)]
    for t in range(n):
        slot = t % 2
        for pool, blur in ((py, True), (pb, False)):
            for s in range(S):
                pool.frame_buffer(s, slot)[...] = seqs[s][t] if blur else blurred(seqs[s][t])
            pool.submit(slot, want_masks=True, detect=True)
        vy, vb = py.wait(slot), pb.wait(slot)
        assert vy == vb
        if not vy:
            continue
        for s in range(S):
            eq(py.mask(s, slot), pb.mask(s, slot), "pool mask stream %d t %d" % (s, t))
            assert py.components(s, slot) == pb.components(s, slot)
        assert py.detect(slot, dy) == pb.detect(slot, db), "pool detect t %d" % t
    py.close(); pb.close()


# ---------------------------------------------------------------------------------------------------------------------
# refusals

def test_refusals():
    from tracking_b200.bgs import process_fanout
    from tracking_b200.streams import StreamPool
    p = plugin(0)
    for bad in (2, -1, 0.5):
        refused(lambda: p.set("gaussianBlur", bad), "gaussianBlur is 0 or 1")
    refused(lambda: p.set("retainInput", 1), "cannot be combined with gaussianBlur")
    q = plugin(0, blur=0)
    q.set("retainInput", 1)
    refused(lambda: q.set("gaussianBlur", 1), "cannot be combined with retainInput")
    assert p.get("gaussianBlur") == 1 and q.get("gaussianBlur") == 0
    a, b = plugin(5), plugin(0, blur=0)
    img = np.zeros((8, 10, 3), np.uint8)
    refused(lambda: process_fanout([a, b], img), "share one \"gaussianBlur\"")
    refused(lambda: process_fanout([b, a], img), "share one \"gaussianBlur\"")
    refused(lambda: StreamPool(5, 2, 10, 8, devices=[0], ring=2, gaussianBlur=3), "gaussianBlur is 0 or 1")
    for x in (p, q, a, b):
        x.close()


# ---------------------------------------------------------------------------------------------------------------------
# which kernels run

def kernel_rows():
    """the body of test_blur_kernel_runs_once_per_band_call_and_frame_set, in a fresh process"""
    import torch
    import tracking_b200 as tb
    from tracking_b200.pipeline import ForegroundPipeline
    # bgsb_process, banded (1080p with the background image: 3 bands) and whole (small frame)
    for (h, w) in ((1080, 1920), (66, 98)):
        frames = scene(3, h, w, seed=80)
        p, r = plugin(5, trace=1), plugin(5, blur=0, trace=1)
        for t in range(2):
            p.process(frames[t]); r.process(frames[t])
        ny, _ = launches(lambda: p.process(frames[2]))
        bands = p.trace_last()["bands"]
        nb, _ = launches(lambda: r.process(frames[2]))
        assert (h, bands) != (1080, 1), "the 1080p frame was not banded"
        assert r.trace_last()["bands"] == bands
        assert ny - nb == bands, (ny, nb, bands)
        p.close(); r.close()
    # FD's warm-up frame launches no plugin kernel, but the blur runs: its output becomes the history
    fd = plugin(0)
    assert launches(lambda: fd.process(scene(1, 66, 98, seed=1)[0]))[0] == 1
    fd.close()
    # process_dev and process_batch_dev: once per call; pipeline: once per frame set
    h, w, S, T = 66, 98, 3, 3
    seqs = [scene(T, h, w, seed=90 + s) for s in range(S)]
    for T_ in (1, T):
        p = tb.ALGOS[5](nstreams=S, gaussianBlur=1)
        r = tb.ALGOS[5](nstreams=S)
        d = torch.from_numpy(np.stack([np.stack(seqs[s][:T_]) for s in range(S)])).cuda()
        fg = torch.zeros((S, T_, h, w), dtype=torch.uint8, device="cuda")
        for _ in range(2):
            got, _ = profiled(lambda: p.process_batch_dev(d.data_ptr(), T_, w, h, fg.data_ptr()))
            ref, _ = profiled(lambda: r.process_batch_dev(d.data_ptr(), T_, w, h, fg.data_ptr()))
            assert BLUR in got and BLUR not in ref
            assert {k for k in got if k != BLUR} == set(ref), (got, ref)
            ny, _ = launches(lambda: p.process_batch_dev(d.data_ptr(), T_, w, h, fg.data_ptr()))
            nb, _ = launches(lambda: r.process_batch_dev(d.data_ptr(), T_, w, h, fg.data_ptr()))
            assert ny - nb == 1, (T_, ny, nb)
        p.close(); r.close()
    pipes = [ForegroundPipeline(5, nstreams=S, gaussianBlur=1), ForegroundPipeline(5, nstreams=S)]
    for t in range(T):
        runs, counts = [], []
        d = torch.from_numpy(np.stack([seqs[s][t] for s in range(S)])).cuda()
        for pipe in pipes:
            call = lambda: (pipe.process_dev(d.data_ptr(), w, h), pipe.join_dev())  # noqa: E731
            runs.append(profiled(call)[0] if t != 1 else None)
            if t == 1:
                counts.append(launches(call)[0])
        if t == 1:
            assert counts[0] - counts[1] == 1, counts       # one blur launch per frame set
        else:
            assert BLUR in runs[0] and BLUR not in runs[1]
            assert {k for k in runs[0] if k != BLUR} == set(runs[1]), runs
    # a context whose blur was switched off launches no blur kernel again
    f0 = seqs[0][0]
    p = plugin(5)
    p.process(f0)
    p.set("gaussianBlur", 0)
    r = plugin(5, blur=0)
    r.process(f0)
    assert launches(lambda: p.process(f0))[0] == launches(lambda: r.process(f0))[0]
    # the restatement the lockstep tests feed the blur-off contexts is cv2's blur on their frames
    import cv2
    for f in scene(2, 98, 131, seed=98) + scene(1, 600, 700, seed=600) + [adversarial(37, 53)]:
        eq(gauss7(f), cv2.GaussianBlur(f, (7, 7), 1.5), "restatement vs cv2")
    q = plugin(5, trace=1)
    q.process(scene(1, 600, 700, seed=600)[0])
    assert q.trace_last()["bands"] > 1, "the 600 x 700 frame was not banded"
    q.close()
    print("ok kernel rows")


def test_blur_kernel_runs_once_per_band_call_and_frame_set():
    """Runs in a child process, as the YUV rows do: late in a long test session torch.profiler has been seen to deliver
    none or only part of a call's kernel records."""
    import subprocess
    import sys
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_prep_gaussian_blur as m; m.kernel_rows()"
            % (ROOT, os.path.join(ROOT, "tests")))
    res = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-6000:]
    assert "ok kernel rows" in res.stdout, res.stdout
