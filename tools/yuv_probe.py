"""YUV 4:2:0 input ("inputFormat" NV12 / I420) against BGR at 1080p.  GPU box, measurement tooling.

    python tools/yuv_probe.py [--out profiles/r6_yuv_probe.jsonl] [--reps 3]

BGR and YUV legs alternate in one process, on the same frames (the BGR legs are fed the restated conversion of the
YUV frames, so the plugin does the same work).  Records, with the card's name and power limit:
  * convert   : the conversion kernel (yuv420_to_bgr_kernel) at 1 and 16 x 1080p, median of its torch.profiler durations
                inside process_batch_dev calls of FrameDifference, as GB/s on 4.5 B/px and as a share of 6539.5 GB/s (the
                copy rate measured on this card type, DESIGN 3.1).  1 x 1080p (9.3 MB) fits the 126 MB L2, 16 x does not.
  * host      : 1080p MOG2 through bgsb_process and bgsb_submit (page-locked buffers), mask + background and mask
                only, microseconds per frame over a host clock that ends in a synchronise
  * dev       : 16 x 1080p FD and MOG2 through process_batch_dev (T = 1), CUDA events per call: the extra pass's cost
  * pool      : the stream pool's host path (config 4: MOG2 + OPEN, tables back) at 64 x 1080p, ring 2, one GPU, Gpx/s
"""
import argparse
import json
import os
import subprocess
import sys
import time
import warnings

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import tracking_b200 as tb  # noqa: E402
from tracking_b200 import capi  # noqa: E402
from tracking_b200.bgs import pinned_empty  # noqa: E402
from tracking_b200.streams import StreamPool  # noqa: E402
from yuv_restate import yuv420_to_bgr  # noqa: E402  (the conversion the BGR legs are fed, tests/yuv_restate.py)

W, H, NF = 1920, 1080, 8
NV12, I420, BGR = capi.INPUT_NV12, capi.INPUT_I420, capi.INPUT_BGR
PEAK_GBS = 6539.5
NAMES = {BGR: "bgr", NV12: "nv12", I420: "i420"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def scene(n, seed=1):
    """n 1080p frames of a noisy scene with moving blocks, as NV12 / I420 images and their BGR conversion"""
    rng = np.random.default_rng(seed)
    by = rng.integers(30, 220, (H, W)).astype(np.int16)
    bu = rng.integers(60, 200, (H // 2, W // 2)).astype(np.uint8)
    bv = rng.integers(60, 200, (H // 2, W // 2)).astype(np.uint8)
    out = {BGR: [], NV12: [], I420: []}
    for t in range(n):
        Y = by + rng.integers(-5, 6, (H, W))
        for k in range(6):
            y, x = (37 * t + 150 * k) % (H - 80), (91 * t + 300 * k) % (W - 120)
            Y[y:y + 80, x:x + 120] = 240 - 30 * k
        Y = np.clip(Y, 0, 255).astype(np.uint8)
        nv = np.concatenate([Y, np.stack([bu, bv], -1).reshape(H // 2, W)], 0)
        out[NV12].append(nv)
        out[I420].append(np.concatenate([Y.reshape(-1), bu.reshape(-1), bv.reshape(-1)]).reshape(H * 3 // 2, W))
        out[BGR].append(yuv420_to_bgr(nv, NV12))
    return out


def convert_leg(frames, S, reps):
    """median duration of the conversion kernel inside process_batch_dev (FD) calls on S streams"""
    from torch.profiler import ProfilerActivity, profile
    rec = {}
    for fmt in (NV12, I420):
        p = tb.ALGOS[0](nstreams=S, inputFormat=fmt)
        d = torch.from_numpy(np.stack([frames[fmt][s % NF] for s in range(S)])).cuda()
        fg = torch.empty((S, H, W), dtype=torch.uint8, device="cuda")
        for _ in range(5):
            p.process_batch_dev(d.data_ptr(), 1, W, H, fg.data_ptr())
        torch.cuda.synchronize()
        durs = []
        for _ in range(reps):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", UserWarning)
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(50):
                        p.process_batch_dev(d.data_ptr(), 1, W, H, fg.data_ptr())
                    torch.cuda.synchronize()
            durs += [e.time_range.elapsed_us() for e in prof.events() if "yuv420_to_bgr_kernel" in e.name]
        us = float(np.median(durs))
        gbs = S * W * H * 4.5 / (us * 1e-6) / 1e9
        rec[NAMES[fmt]] = dict(kernel_us_median=us, launches=len(durs), gb_per_s=gbs, share_of_peak=gbs / PEAK_GBS)
        p.close()
    return rec


def host_leg(frames, want_bg, reps, n=200):
    """1080p MOG2, us per frame: bgsb_process and bgsb_submit (page-locked buffers), BGR / NV12 / I420 alternating"""
    res = {}
    bufs = {}
    for fmt in (BGR, NV12, I420):
        ins = []
        for f in frames[fmt]:
            a = pinned_empty(f.shape)
            a[...] = f
            ins.append(a)
        bufs[fmt] = ins
    fgs = [pinned_empty((H, W)) for _ in range(2)]
    bgs = [pinned_empty((H, W, 3)) if want_bg else None for _ in range(2)]
    for _ in range(reps):
        for fmt in (BGR, NV12, I420):
            for mode in ("process", "submit"):
                p = tb.ALGOS[5]() if fmt == BGR else tb.ALGOS[5](inputFormat=fmt)
                for t in range(10):
                    p.process(bufs[fmt][t % NF], want_bg=want_bg)
                t0 = time.perf_counter()
                for t in range(n):
                    if mode == "process":
                        p.process(bufs[fmt][t % NF], want_bg=want_bg)
                    else:
                        p.submit(bufs[fmt][t % NF], fgs[t & 1], bgs[t & 1])
                        if t % 16 == 15:
                            p.wait()
                p.wait()
                us = (time.perf_counter() - t0) / n * 1e6
                res.setdefault("%s_%s_us" % (mode, NAMES[fmt]), []).append(us)
                p.close()
    return res


def dev_leg(frames, S, reps, n=50):
    res = {}
    ds = {fmt: torch.from_numpy(np.stack([frames[fmt][s % NF] for s in range(S)])).cuda() for fmt in (BGR, NV12, I420)}
    fg = torch.empty((S, H, W), dtype=torch.uint8, device="cuda")
    bg = torch.empty((S, H, W, 3), dtype=torch.uint8, device="cuda")
    for _ in range(reps):
        for aid, name in ((0, "fd"), (5, "mog2")):
            for fmt in (BGR, NV12, I420):
                p = tb.ALGOS[aid](nstreams=S) if fmt == BGR else tb.ALGOS[aid](nstreams=S, inputFormat=fmt)
                call = lambda: p.process_batch_dev(ds[fmt].data_ptr(), 1, W, H, fg.data_ptr(),  # noqa: E731
                                                   bg.data_ptr() if aid == 5 else None)
                for _ in range(5):
                    call()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(n):
                    call()
                e1.record()
                torch.cuda.synchronize()
                res.setdefault("%s_%s_us" % (name, NAMES[fmt]), []).append(e0.elapsed_time(e1) / n * 1e3)
                p.close()
    return res


def pool_leg(frames, S, reps, n=60):
    res = {}
    for _ in range(reps):
        for fmt in (BGR, NV12):
            kw = {} if fmt == BGR else dict(inputFormat=fmt)
            pool = StreamPool(5, S, W, H, devices=[0], ring=2, morph=(("erode", 1), ("dilate", 1)), **kw)
            for slot in range(2):
                for s in range(S):
                    pool.frame_buffer(s, slot)[...] = frames[fmt][(s + slot) % NF]
            for t in range(4):
                pool.submit(t % 2)
                pool.wait(t % 2)
            pool.submit(0)
            t0 = time.perf_counter()
            for t in range(1, n + 1):
                pool.submit(t % 2)
                pool.wait((t - 1) % 2)
            pool.wait(n % 2)
            sec = (time.perf_counter() - t0) / n
            res.setdefault("gpx_per_s_%s" % NAMES[fmt], []).append(S * W * H / sec / 1e9)
            res.setdefault("frame_set_ms_%s" % NAMES[fmt], []).append(sec * 1e3)
            pool.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r6_yuv_probe.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    frames = scene(NF)
    base = dict(card=card(), geometry="%dx%d" % (W, H))
    lines = []
    for S in (1, 16):
        lines.append(dict(base, leg="convert", streams=S, **convert_leg(frames, S, a.reps)))
    for want_bg in (True, False):
        lines.append(dict(base, leg="host_mog2", background=want_bg, **host_leg(frames, want_bg, a.reps)))
    lines.append(dict(base, leg="dev", streams=16, **dev_leg(frames, 16, a.reps)))
    lines.append(dict(base, leg="pool_config4", streams=64, ring=2, **pool_leg(frames, 64, a.reps)))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main()
