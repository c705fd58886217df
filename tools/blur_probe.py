"""The PreProcessor's Gaussian blur ("gaussianBlur" 1) at 1080p, blur off and on alternating in one process.  GPU box,
measurement tooling.

    python tools/blur_probe.py [--out profiles/r8_blur_probe.jsonl] [--reps 3]

Records, with the card's name and power limit:
  * kernel    : gauss7_kernel alone on 16 x 1080p device-resident frames (200 MB, more than the 126 MB L2), median of its
                torch.profiler durations inside process_batch_dev calls of FrameDifference, as GB/s on 6 B/px (3 read +
                3 written) and as a share of 6539.5 GB/s (the copy rate measured on this card type, DESIGN 3.1)
  * host      : 1080p MOG2 through bgsb_submit (queued) and bgsb_process (banded), page-locked buffers, mask + background
                and mask only, microseconds per frame over a host clock that ends in a synchronise
  * pool      : the stream pool's host path (config 4: MOG2 + OPEN, tables back) at 64 x 1080p, ring 2, one GPU, Gpx/s
  * cv2       : cv2.GaussianBlur(img, (7, 7), 1.5) on one 1080p BGR frame on this host's CPU, 1 thread and the default
                thread count: the per-frame cost the device blur removes
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
from tracking_b200.bgs import pinned_empty  # noqa: E402
from tracking_b200.streams import StreamPool  # noqa: E402

W, H, NF = 1920, 1080, 8
PEAK_GBS = 6539.5
NAMES = {0: "off", 1: "on"}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(0)


def scene(n, seed=1):
    """n 1080p BGR frames of a noisy scene with moving blocks"""
    rng = np.random.default_rng(seed)
    base = rng.integers(30, 220, (H, W, 3)).astype(np.int16)
    out = []
    for t in range(n):
        f = base + rng.integers(-5, 6, (H, W, 3))
        for k in range(6):
            y, x = (37 * t + 150 * k) % (H - 80), (91 * t + 300 * k) % (W - 120)
            f[y:y + 80, x:x + 120] = 240 - 30 * k
        out.append(np.clip(f, 0, 255).astype(np.uint8))
    return out


def kernel_leg(frames, S, reps):
    from torch.profiler import ProfilerActivity, profile
    p = tb.ALGOS[0](nstreams=S, gaussianBlur=1)
    d = torch.from_numpy(np.stack([frames[s % NF] for s in range(S)])).cuda()
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
        durs += [e.time_range.elapsed_us() for e in prof.events() if "gauss7_kernel" in e.name]
    p.close()
    us = float(np.median(durs))
    gbs = S * W * H * 6 / (us * 1e-6) / 1e9
    return dict(kernel_us_median=us, kernel_us_min=float(np.min(durs)), launches=len(durs), gb_per_s=gbs,
                share_of_peak=gbs / PEAK_GBS)


def host_leg(frames, want_bg, reps, n=200):
    res = {}
    ins = []
    for f in frames:
        a = pinned_empty(f.shape)
        a[...] = f
        ins.append(a)
    fgs = [pinned_empty((H, W)) for _ in range(2)]
    bgs = [pinned_empty((H, W, 3)) if want_bg else None for _ in range(2)]
    for _ in range(reps):
        for blur in (0, 1):
            for mode in ("submit", "process"):
                p = tb.ALGOS[5](gaussianBlur=blur, trace=1)
                for t in range(10):
                    p.process(ins[t % NF], want_bg=want_bg)
                bands = p.trace_last()["bands"]
                t0 = time.perf_counter()
                for t in range(n):
                    if mode == "process":
                        p.process(ins[t % NF], want_bg=want_bg)
                    else:
                        p.submit(ins[t % NF], fgs[t & 1], bgs[t & 1])
                        if t % 16 == 15:
                            p.wait()
                p.wait()
                res.setdefault("%s_blur_%s_us" % (mode, NAMES[blur]), []).append((time.perf_counter() - t0) / n * 1e6)
                res["process_bands"] = bands
                p.close()
    return res


def pool_leg(frames, S, reps, n=60):
    res = {}
    for _ in range(reps):
        for blur in (0, 1):
            pool = StreamPool(5, S, W, H, devices=[0], ring=2, morph=(("erode", 1), ("dilate", 1)), gaussianBlur=blur)
            for slot in range(2):
                for s in range(S):
                    pool.frame_buffer(s, slot)[...] = frames[(s + slot) % NF]
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
            res.setdefault("gpx_per_s_blur_%s" % NAMES[blur], []).append(S * W * H / sec / 1e9)
            res.setdefault("frame_set_ms_blur_%s" % NAMES[blur], []).append(sec * 1e3)
            pool.close()
    return res


def cv2_leg(frames, n=50):
    import cv2
    res = dict(cv2_version=cv2.__version__, cpus=os.cpu_count())
    old = cv2.getNumThreads()
    for threads in (1, old):
        cv2.setNumThreads(threads)
        for f in frames[:3]:
            cv2.GaussianBlur(f, (7, 7), 1.5)
        t0 = time.perf_counter()
        for t in range(n):
            cv2.GaussianBlur(frames[t % NF], (7, 7), 1.5)
        res["ms_per_frame_%d_threads" % threads] = (time.perf_counter() - t0) / n * 1e3
    cv2.setNumThreads(old)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_blur_probe.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    frames = scene(NF)
    base = dict(card=card(), geometry="%dx%d" % (W, H))
    lines = [dict(base, leg="kernel", streams=16, **kernel_leg(frames, 16, a.reps))]
    for want_bg in (True, False):
        lines.append(dict(base, leg="host_mog2", background=want_bg, **host_leg(frames, want_bg, a.reps)))
    lines.append(dict(base, leg="pool_config4", streams=64, ring=2, **pool_leg(frames, 64, a.reps)))
    lines.append(dict(base, leg="cv2_host", **cv2_leg(frames)))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        for ln in lines:
            f.write(json.dumps(ln) + "\n")
            print(json.dumps(ln))


if __name__ == "__main__":
    main()
