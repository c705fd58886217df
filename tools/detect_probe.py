"""DetectNewBlob for a stream group at 1080p, synthetic streams (bgsb_synth_frames_dev).  GPU box, measurement tooling.

    python tools/detect_probe.py [--streams 8,64] [--out FILE.jsonl]

Per stream count, MOG2 + OPEN 3x3, the same frames for every variant:
  * pipeline_detect : frame set = bgsb_pipeline_process_dev + bgsb_pipeline_detect (device events and a host clock
                      around the whole loop, which ends in a synchronise; detect itself synchronises twice)
  * per_stream      : the route without it: process_dev with d_mask, then bgsb_blobdetector_detect_dev per stream
                      (each labels its mask again); the two routes' results are compared on every frame set
  * pool            : bgsb_pool submit / wait per frame set (ring 2, one GPU) with flags 0, with BGSB_POOL_DETECT (the
                      device mask kept, no detect call: the cost of the retention) and with detect called
  * moments kernels : the batched kernels of one detect call (one launch for all streams: bits after OPEN, bytes with
                      FrameDifference and no chain) against the former grid(nrects, 16) form of the kernels, launched
                      once per stream on the same masks and rectangles (torch.profiler kernel durations)
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tracking_b200 import blobs, capi, synth  # noqa: E402
from tracking_b200.pipeline import ForegroundPipeline  # noqa: E402
from tracking_b200.streams import StreamPool  # noqa: E402

W, H, NT = 1920, 1080, 8

# The moments kernels as they were before the batched form (one image, grid(nrects, 16)), for the A/B only.
OLD_SRC = r'''
#include <cuda_runtime.h>
#include <stdint.h>
__device__ void reduce6(unsigned long long (&m)[6], unsigned long long *out)
{
    __shared__ unsigned long long red[6][8];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int i = 0; i < 6; i++) {
        unsigned long long v = m[i];
        for (int off = 16; off > 0; off >>= 1) v += __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) red[i][wid] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        unsigned long long v = 0;
        for (int i = 0; i < 8; i++) v += red[threadIdx.x][i];
        if (v) atomicAdd(out + threadIdx.x, v);
    }
}
__global__ void __launch_bounds__(256) old_rect_moments_kernel(const uint8_t *mask, int w, int h, const int *rects,
                                                               unsigned long long *out)
{
    const int ri = blockIdx.x;
    const int rx = rects[4 * ri], ry = rects[4 * ri + 1], rw = rects[4 * ri + 2], rh = rects[4 * ri + 3];
    unsigned long long m[6] = {0, 0, 0, 0, 0, 0};
    for (int yy = blockIdx.y; yy < rh; yy += gridDim.y) {
        int y = ry + yy;
        if (y < 0 || y >= h) continue;
        const uint8_t *row = mask + (size_t)y * w;
        unsigned long long r0 = 0, r1 = 0, r2 = 0;
        for (int xx = threadIdx.x; xx < rw; xx += blockDim.x) {
            int x = rx + xx;
            if (x < 0 || x >= w) continue;
            unsigned long long v = row[x];
            r0 += v; r1 += v * xx; r2 += v * (unsigned long long)xx * xx;
        }
        m[0] += r0; m[1] += r1; m[2] += r0 * yy; m[3] += r2; m[4] += r0 * (unsigned long long)yy * yy; m[5] += r1 * yy;
    }
    reduce6(m, out + 6 * ri);
}
__global__ void __launch_bounds__(256) old_rect_moments_bits_kernel(const unsigned *bits, int w, int h, int wpr,
                                                                    const int *rects, unsigned long long *out)
{
    const int ri = blockIdx.x;
    const int rx = rects[4 * ri], ry = rects[4 * ri + 1], rw = rects[4 * ri + 2], rh = rects[4 * ri + 3];
    const int xa = max(rx, 0), xb = min(rx + rw, w);
    unsigned long long m[6] = {0, 0, 0, 0, 0, 0};
    if (xa < xb) {
        const int k0 = xa >> 5, k1 = (xb - 1) >> 5;
        for (int yy = blockIdx.y; yy < rh; yy += gridDim.y) {
            const int y = ry + yy;
            if (y < 0 || y >= h) continue;
            unsigned long long r0 = 0, r1 = 0, r2 = 0;
            for (int k = k0 + (int)threadIdx.x; k <= k1; k += blockDim.x) {
                unsigned v = bits[(size_t)y * wpr + k];
                if (k == k0) v &= 0xffffffffu << (xa & 31);
                if (k == k1 && (xb & 31)) v &= 0xffffffffu >> (32 - (xb & 31));
                while (v) {
                    const int b = __ffs(v) - 1; v &= v - 1;
                    const unsigned long long xx = (unsigned long long)(k * 32 + b - rx);
                    r0 += 255ull; r1 += 255ull * xx; r2 += 255ull * xx * xx;
                }
            }
            m[0] += r0; m[1] += r1; m[2] += r0 * yy; m[3] += r2; m[4] += r0 * (unsigned long long)yy * yy; m[5] += r1 * yy;
        }
    }
    reduce6(m, out + 6 * ri);
}
extern "C" int old_moments(const void *src, int bits, int w, int h, const int *rects, int n, unsigned long long *out,
                           cudaStream_t st)
{
    if (bits) old_rect_moments_bits_kernel<<<dim3(n, 16), 256, 0, st>>>((const unsigned *)src, w, h, (w + 31) / 32, rects, out);
    else old_rect_moments_kernel<<<dim3(n, 16), 256, 0, st>>>((const uint8_t *)src, w, h, rects, out);
    return (int)cudaGetLastError();
}
'''


def build_old(tmp):
    src, so = os.path.join(tmp, "old_moments.cu"), os.path.join(tmp, "old_moments.so")
    with open(src, "w") as f:
        f.write(OLD_SRC)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-shared", "-Xcompiler", "-fPIC",
                           src, "-o", so])
    lib = C.CDLL(so)
    lib.old_moments.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return lib


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def frames_dev(S):
    st = torch.cuda.current_stream().cuda_stream
    fr = torch.empty((NT, S, H, W, 3), dtype=torch.uint8, device="cuda")
    for t in range(NT):
        synth.frames_dev(fr[t].data_ptr(), S, 1, W, H, t0=t, stream=st)
    torch.cuda.synchronize()
    return fr


def timed(step, iters):
    """-> (device-event us, host-clock us) per iteration; the host clock ends after a synchronise"""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for i in range(iters):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) / iters * 1e6
    return e0.elapsed_time(e1) / iters * 1e3, host


def routes(S, fr, iters):
    st = torch.cuda.current_stream().cuda_stream
    a, b = ForegroundPipeline(5, nstreams=S), ForegroundPipeline(5, nstreams=S)
    da, db = [blobs.CvBlobDetectorCC() for _ in range(S)], [blobs.CvBlobDetectorCC() for _ in range(S)]
    d_mask = torch.empty((S, H, W), dtype=torch.uint8, device="cuda")
    out_a, out_b = [], []

    def step_a(i):
        a.process_dev(fr[i % NT].data_ptr(), W, H, stream=st)
        out_a.append([(r, nb, list(f)) for r, nb, f in a.detect(da)])

    def step_b(i):
        b.process_dev(fr[i % NT].data_ptr(), W, H, d_mask.data_ptr(), stream=st)
        res = []
        for s in range(S):
            r, nb = db[s].DetectNewBlob_dev(d_mask.data_ptr() + s * W * H, W, H, stream=st)
            res.append((r, nb, list(db[s].frame_blobs)))
        out_b.append(res)

    for i in range(2 * NT):                    # settle the model; both routes see the same frames
        step_a(i); step_b(i)
    ta, tb_ = timed(step_a, iters), timed(step_b, iters)
    same = out_a == out_b
    blobs_per_set = sum(len(f) for _, _, f in out_a[-1])
    a.close(); b.close()
    return dict(pipeline_detect_us=ta, per_stream_detect_dev_us=tb_, routes_identical=same,
                frame_blobs_last_set=blobs_per_set)


def pool_cost(S, fr, iters):
    host = [fr[t].cpu().numpy() for t in range(2)]
    out = {}
    for mode in ("plain", "retain", "detect"):
        pool = StreamPool(5, S, W, H, devices=[0], ring=2)
        for slot in range(2):
            for s in range(S):
                pool.frame_buffer(s, slot)[...] = host[slot][s]
        dets = [blobs.CvBlobDetectorCC() for _ in range(S)]

        def step(i):
            slot = i % 2
            if i >= 2:
                pool.wait(slot)
                if mode == "detect":
                    pool.detect(slot, dets)
            pool.submit(slot, detect=mode != "plain")

        for i in range(8):
            step(i)
        # (the two slots hold frames 0 and 1 of the synthetic streams: the video alternates between them)
        out[mode] = timed(lambda i: step(i + 8), iters)
        pool.wait(0); pool.wait(1)
        pool.close()
    return {"pool_%s_us" % k: v for k, v in out.items()}


def kernel_times(prof_fn, names):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        prof_fn()
        torch.cuda.synchronize()
    with tempfile.NamedTemporaryFile(suffix=".json") as f:
        prof.export_chrome_trace(f.name)
        ev = json.load(open(f.name))["traceEvents"]
    d = [e["dur"] for e in ev if e.get("cat") == "kernel" and any(n in e["name"] for n in names)]
    return sum(d), len(d)


def cluster_rects(comps):
    """detect_rects of csrc/blobdetect.cu: external rects in reverse raster order, partitioned, united"""
    from oracle.blobdetect import _partition
    rects = [(c["x"], c["y"], c["w"], c["h"]) for c in reversed(comps) if c["external"]]
    ncls, cls = _partition(rects)
    q = [None] * ncls
    for r, k in zip(rects, cls):
        R = q[k]
        q[k] = r if R is None else (min(R[0], r[0]), min(R[1], r[1]), max(R[0] + R[2], r[0] + r[2]) - min(R[0], r[0]),
                                    max(R[1] + R[3], r[1] + r[3]) - min(R[1], r[1]))
    return q


def moments_ab(S, fr, old, reps=5):
    st = torch.cuda.current_stream().cuda_stream
    out = {}
    for form, algo, chain in (("bits", 5, (("erode", 1), ("dilate", 1))), ("bytes", 0, ())):
        pipe = ForegroundPipeline(algo, nstreams=S, morph=chain)
        dets = [blobs.CvBlobDetectorCC() for _ in range(S)]
        d_mask = torch.empty((S, H, W), dtype=torch.uint8, device="cuda")
        for i in range(2 * NT):
            pipe.process_dev(fr[i % NT].data_ptr(), W, H, d_mask.data_ptr(), stream=st)
            if i:
                pipe.detect(dets)
        torch.cuda.synchronize()
        new = [kernel_times(lambda: pipe.detect(dets), ["rect_moments"]) for _ in range(reps)]
        rects = [cluster_rects(pipe.components(s)) for s in range(S)]
        if form == "bits":
            m = (d_mask > 128).to(torch.int64)
            pad = (W + 31) // 32 * 32 - W
            m = torch.nn.functional.pad(m, (0, pad)).view(S, H, -1, 32)
            src = (m << torch.arange(32, device="cuda")).sum(-1).to(torch.int32).contiguous()
            stride = src[0].numel() * 4
        else:
            src, stride = d_mask, W * H
        d_rects = [torch.tensor(np.asarray(r, np.int32).reshape(-1), device="cuda") for r in rects]
        d_out = torch.zeros(6 * max(1, max(len(r) for r in rects)), dtype=torch.int64, device="cuda")

        def launch_old():
            for s in range(S):
                if rects[s]:
                    rc = old.old_moments(C.c_void_p(src.data_ptr() + s * stride), int(form == "bits"), W, H,
                                         C.c_void_p(d_rects[s].data_ptr()), len(rects[s]), C.c_void_p(d_out.data_ptr()),
                                         C.c_void_p(st))
                    assert rc == 0, rc
        launch_old()
        oldt = [kernel_times(launch_old, ["old_rect_moments"]) for _ in range(reps)]
        area = sum(max(0, min(x + w, W) - max(x, 0)) * max(0, min(y + h, H) - max(y, 0)) for r in rects for x, y, w, h in r)
        out[form] = dict(records=sum(len(r) for r in rects), clipped_area_px=area,
                         new_us_median=float(np.median([t for t, _ in new])), new_launches=new[0][1],
                         old_us_median=float(np.median([t for t, _ in oldt])), old_launches=oldt[0][1])
        pipe.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--streams", default="8,64")
    ap.add_argument("--iters", type=int, default=24)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    old = build_old(tempfile.mkdtemp(prefix="detect_probe_"))
    rows = []
    for S in [int(v) for v in args.streams.split(",")]:
        fr = frames_dev(S)
        row = dict(card=card(), streams=S, geometry="%dx%d" % (W, H))
        row.update(routes(S, fr, args.iters))
        row.update(pool_cost(S, fr, args.iters))
        row["moments_kernels"] = moments_ab(S, fr, old)
        del fr
        torch.cuda.empty_cache()
        print(json.dumps(row), flush=True)
        rows.append(row)
    if args.out:
        with open(args.out, "w") as f:
            f.writelines(json.dumps(r) + "\n" for r in rows)


if __name__ == "__main__":
    main()
