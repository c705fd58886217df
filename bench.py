#!/usr/bin/env python
"""Headline benchmark: MOG2 Mpixel/s at 1080p (BASELINE.json metric), one camera stream per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the timed headline path returned for the last frame of its last step (rank 0): the mask
as DIR/foreground_mask.npy and the background image as DIR/background_image.npy, float32.  The synthetic input is seeded,
so two builds run with the same arguments can be compared output for output.

A "step" is one pass of the hot path over one batch of synthetic input: FRAMES_PER_STEP
consecutive 1920x1080 BGR frames of one camera stream, advanced frame by frame (T = 1, the judged
roofline configuration: 209 algorithmic bytes per pixel per frame, SURVEY 8d) through
MixtureOfGaussianV2BGS -- mask + background image produced for every frame, exactly what
`IBGS::process` returns.  Frames are resident in HBM when the timed region starts (K-GEN).

Multi-GPU: independent camera streams, no data-path collective; torch.distributed (NCCL) is used only for the
barriers and the max-over-ranks of the timed regions.  The headline scales weakly (one stream per GPU).

The ONE JSON line also carries
  parity       the benchmark's own code paths run the first frames of the streams they are timed on; outputs must hash to
               the committed oracle values (tests/golden/bench_hashes.json) or the run aborts
  e2e          the same metric through the host-buffer C-ABI call bgsb_process (pinned host frames,
               H2D + kernel + D2H of mask and background inside the timed region), and its queued form
  roofline     achieved algorithmic HBM GB/s of the MOG2 kernel vs the measured copy peak, on live bytes and on the
               dense 209 B/px of SURVEY 8(d); the same for 16 HBM-resident streams and for a mode-churn stream on which
               the dense figure is real (all 5 modes live)
  config4      BASELINE config 4, the north-star target: MOG2 -> OPEN 3x3 -> connected components, 64 x 1080p streams
               sharded over the N GPUs (strong scaling: 64 / N streams per GPU), device-resident and through the
               StreamPool with host frames; per-stage split
  config5      BASELINE config 5: MOG2 3840x2160, 16 streams per GPU, temporal batches T = 1 and T = 16
  cpu_baseline the reference's CPU path (OpenCV calls replayed call-for-call by oracle/cv2_chain.py,
               the reference C++ itself cannot be built in this image) timed on this box's host cores
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 1920, 1080
NPX = W * H
FRAMES_PER_STEP = 1024        # 34 s of 30 fps video per step; ~23 ms of GPU time, so that K >= 10 steps span several
                               # nvidia-smi clock samples
NFRAMES_RESIDENT = 128          # distinct synthetic frames kept in HBM (796 MB) and cycled
MOG2_BYTES_PER_PX = 209         # dense model: in 3 + state 101 read + 101 write + mask 1 + bg 3  (SURVEY 8d)
MOG2_FIXED_BYTES_PER_PX = 9     # in 3 + nmodes 1 read + 1 write + mask 1 + bg 3
MOG2_BYTES_PER_LIVE_MODE = 40   # weight, variance, 3-vector mean: 20 B read + 20 B written
PIPE_DENSE_BYTES_PER_PX = 218   # SURVEY 8d: 209 + 2 x 2 (OPEN on byte masks) + 5 (CC)
C4_STREAMS = 64                 # BASELINE config 4
C5_STREAMS_PER_GPU = 16         # BASELINE config 5 (128 streams on 8 GPUs)
METRIC = "MOG2 Mpixel/s at 1080p"
UNIT = "Mpixel/s"
WORKLOAD = "MixtureOfGaussianV2 (MOG2, K=5) on one synthetic 1920x1080 BGR stream per GPU, T=1"


_STDOUT_FD = None


def emit(text):
    """The contract's one line, on the process's original stdout."""
    sys.stdout.flush()
    if _STDOUT_FD is None:
        print(text, flush=True)
    else:
        os.write(_STDOUT_FD, (text + "\n").encode())


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def config_dict(world):
    """Identical for both arms (the reference arm times a bounded sample of it, described in its cpu_baseline.sample)."""
    return {"workload": WORKLOAD, "frames_per_step": FRAMES_PER_STEP, "resolution": [W, H], "temporal_batch": 1,
            "streams_per_gpu": 1, "unique_frames": NFRAMES_RESIDENT,
            "parallelism": "independent camera streams, %d GPU(s), no collective" % world,
            "l2": "inputs larger than L2: 209 MB model state + 796 MB of resident frames cycled"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t_begin=None, t_end=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(2)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        rows = [r for (ts, r) in self.rows if t_begin is None or (t_begin <= ts <= t_end + 0.15)]
        window = "timed region"
        if len(rows) < 2:            # region shorter than the sampling period: widen to the load phase around it
            rows = [r for (ts, r) in self.rows if t_begin is None or (t_begin - 1.0 <= ts <= t_end + 1.0)]
            window = "timed region +-1 s (region shorter than 2 samples)"
        for r in rows:
            try:
                sm.append(float(r[0])); smax = float(r[1])
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm), "window": window}


# =====================================================================================================================
# reference arm / CPU baseline
# =====================================================================================================================
def cpu_reference_run(steps, warmup_frames, sample_frames, threads, nuniq=NFRAMES_RESIDENT):
    """The reference's CPU path on this box: MixtureOfGaussianV2BGS::process replayed with OpenCV
    (mog(in, fg, 0.05) + getBackgroundImage + threshold) on the SAME synthetic stream the GPU arm times (same
    generator, same seed, the same ring of `nuniq` frames cycled)."""
    import cv2
    from oracle import cv2_chain, restate
    from tracking_b200 import synth
    cv2.setNumThreads(threads)
    restate.build()
    frames = [restate.synth_frame(W, H, t, synth.SEED0) for t in range(nuniq)]      # C twin of K-GEN, byte-identical
    bgs = cv2_chain.MixtureOfGaussianV2BGS()
    k = 0
    for _ in range(warmup_frames):
        bgs.process(frames[k % nuniq]); k += 1
    t0 = time.perf_counter()
    for _ in range(steps * sample_frames):
        bgs.process(frames[k % nuniq]); k += 1
    dt = time.perf_counter() - t0
    return steps * sample_frames * NPX / dt / 1e6, dt, cv2.getNumThreads()


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # bounded sample of a 1024-frame step: 32 frames per step keeps `--steps 20 --warmup 5` at about 15-20 s of CPU work
    sample = 32
    warm_frames = max(50, args.warmup * sample)
    val, dt, threads = cpu_reference_run(args.steps, warm_frames, sample, cores)
    v1, dt1, _ = cpu_reference_run(1, 50, 96, 1)
    import cv2
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(args.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port",
                             "sample": "%d of the %d frames of each step, x %d steps, after %d warm-up frames, on the same "
                                       "synthetic 1080p stream and the same ring of %d unique frames as the GPU arm; "
                                       "OpenCV %s calls of MixtureOfGaussianV2BGS::process replayed call-for-call (reference "
                                       "C++ not buildable here: needs OpenCV 2.4 headers), %d host cores"
                                       % (sample, FRAMES_PER_STEP, args.steps, warm_frames, NFRAMES_RESIDENT, cv2.__version__, cores),
                             "one_thread": {"value": v1, "unit": UNIT, "cores": 1,
                                            "sample": "96 frames after 50 warm-up frames, cv2.setNumThreads(1), %.1f s" % dt1}},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(json.dumps(line))
    return 0


# =====================================================================================================================
# our arm
# =====================================================================================================================
class Ctx:
    """rank / world / barrier / max-over-ranks helpers shared by the legs."""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def sum_over_ranks(self, values):
        t = self.torch.tensor(list(values), dtype=self.torch.float64, device="cuda")
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def timed(self, fn, iters):
        """CUDA-event time of `iters` calls on torch's current stream, bracketed by barriers; this rank's ms."""
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(iters):
            fn(i)
        e1.record()
        self.barrier()
        return e0.elapsed_time(e1)


def bind_cpus(ctx):
    """Each rank keeps to its own share of the host cores (and allocates its pinned buffers after that), so that the
    ranks' copy engines are fed from disjoint cores.  The pool's B200 boxes expose one NUMA node; on a two-socket host
    the same split keeps a rank on the socket its cores belong to."""
    try:
        cores = sorted(os.sched_getaffinity(0))
        per = max(1, len(cores) // ctx.world)
        mine = cores[ctx.local * per:(ctx.local + 1) * per] or cores
        os.sched_setaffinity(0, mine)
        return {"cores": len(mine), "first": mine[0], "of": len(cores)}
    except Exception as e:       # not fatal: the measurement still stands, only less tidy
        return {"error": str(e)}


def table_hash_update(h, comps):
    import numpy as np
    rows = np.array([(c["x"], c["y"], c["w"], c["h"], c["area"], c["first_index"], c["external"]) for c in comps],
                    np.int32).reshape(-1, 7)
    h.update(np.int32(len(comps)).tobytes() + rows.tobytes())


def parity_check(ctx, my_c4_streams):
    """The timed code paths on the first frames of the streams they are timed on, against committed oracle hashes."""
    import tracking_b200 as tb
    from tracking_b200 import synth
    from tracking_b200.pipeline import ForegroundPipeline
    torch = ctx.torch
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "bench_hashes.json")))
    st = torch.cuda.current_stream().cuda_stream
    out = {"source": "tests/golden/bench_hashes.json (C oracle, pinned to OpenCV 4.13)"}
    # headline path: bgsb_process_dev, one stream, T = 1
    seed = synth.SEED0 + ctx.rank
    exp = gold["mog2"]["by_seed"].get(str(seed))
    nf = gold["mog2"]["frames"]
    if exp is not None:
        d = torch.empty((nf, H, W, 3), dtype=torch.uint8, device="cuda")
        synth.frames_dev(d.data_ptr(), 1, nf, W, H, t0=0, seed0=seed, stream=st)
        fg = torch.empty((H, W), dtype=torch.uint8, device="cuda")
        bg = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
        p = tb.MixtureOfGaussianV2BGS(device=ctx.local)
        for t in range(nf):
            p.process_dev(d[t].data_ptr(), W, H, fg.data_ptr(), bg.data_ptr(), stream=st)
            torch.cuda.synchronize()
            got = hashlib.sha256(fg.cpu().numpy().tobytes() + bg.cpu().numpy().tobytes()).hexdigest()
            if got != exp[t]:
                raise SystemExit("bench.py: PARITY FAILURE -- MOG2 frame %d of stream seed %d differs from the oracle" % (t, seed))
        p.close()
        del d, fg, bg
        out["mog2_frames_checked"] = nf
    # config-4 path: the pipeline object on this rank's streams
    nf = gold["pipeline"]["frames"]
    S = len(my_c4_streams)
    d = torch.empty((nf, S, H, W, 3), dtype=torch.uint8, device="cuda")
    for t in range(nf):
        for i, s in enumerate(my_c4_streams):
            synth.frames_dev(d[t, i].data_ptr(), 1, 1, W, H, t0=t, seed0=synth.SEED0 + s, stream=st)
    pipe = ForegroundPipeline(5, device=ctx.local, nstreams=S)
    hs = [hashlib.sha256() for _ in range(S)]
    for t in range(nf):
        pipe.process_dev(d[t].data_ptr(), W, H, None, None, None, stream=st)
        for i in range(S):
            table_hash_update(hs[i], pipe.components(i))
    for i, s in enumerate(my_c4_streams):
        if hs[i].hexdigest() != gold["pipeline"]["by_seed"][str(synth.SEED0 + s)]:
            raise SystemExit("bench.py: PARITY FAILURE -- pipeline component tables of stream %d differ from the oracle" % s)
    pipe.close()
    del d
    torch.cuda.empty_cache()
    out["pipeline_streams_checked"] = S
    out["pipeline_frames_checked"] = nf
    out["ok"] = True
    return out


def dump_outputs(outdir, arrays):
    """Device arrays -> outdir/<name>.npy as float32 (the caller has synchronised the stream that wrote them)."""
    import numpy as np
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(outdir, name + ".npy"), a.cpu().numpy().astype(np.float32))
    log("bench.py: wrote %s to %s" % (", ".join(n + ".npy" for n in arrays), outdir))


def headline(ctx, args):
    import tracking_b200 as tb
    from tracking_b200 import capi, synth
    torch = ctx.torch
    F, K, Wm = args.frames_per_step, args.steps, args.warmup
    stream = torch.cuda.current_stream().cuda_stream
    frames = torch.empty((NFRAMES_RESIDENT, H, W, 3), dtype=torch.uint8, device="cuda")
    synth.frames_dev(frames.data_ptr(), 1, NFRAMES_RESIDENT, W, H, t0=0, seed0=synth.SEED0 + ctx.rank, stream=stream)
    d_fg = torch.empty((H, W), dtype=torch.uint8, device="cuda")
    d_bg = torch.empty((H, W, 3), dtype=torch.uint8, device="cuda")
    bgs = tb.MixtureOfGaussianV2BGS(device=ctx.local, kernelVariant=args.kernel_variant)
    fptr = [frames[i].data_ptr() for i in range(NFRAMES_RESIDENT)]
    fgp, bgp = d_fg.data_ptr(), d_bg.data_ptr()

    def step(i):
        base = (i * F) % NFRAMES_RESIDENT
        for t in range(F):
            bgs.process_dev(fptr[(base + t) % NFRAMES_RESIDENT], W, H, fgp, bgp, stream=stream)

    sampler = ClockSampler(ctx.local)
    if ctx.rank == 0:
        sampler.start()          # nvidia-smi needs ~0.3 s before its first sample: start it ahead of the warm-up
    for i in range(Wm):
        step(i)
    ctx.barrier()
    t_begin = time.perf_counter()
    launches0 = capi.kernel_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for i in range(K):
        step(Wm + i)
    ev1.record()
    ctx.barrier()
    t_end = time.perf_counter()
    clocks = sampler.stop(t_begin, t_end) if ctx.rank == 0 else None
    launches = capi.kernel_launch_count() - launches0
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, {"foreground_mask": d_fg, "background_image": d_bg})
    ms = ev0.elapsed_time(ev1)
    ms_max = ctx.max_over_ranks([ms])[0]
    _, nm_host = bgs.export_state()
    res = {"ms": ms, "ms_max": ms_max, "launches": launches, "clocks": clocks, "mean_modes": float(nm_host.mean()),
           "share_5_modes": float((nm_host == 5).mean()), "frames": frames}
    bgs.close()
    return res


def run_e2e(ctx, args, frames):
    """bgsb_process / bgsb_submit with host buffers: the IBGS::process boundary."""
    import ctypes as C
    import tracking_b200 as tb
    from tracking_b200 import capi
    torch = ctx.torch
    F, K = args.frames_per_step, args.steps
    nh = 16
    h_in = torch.empty((nh, H, W, 3), dtype=torch.uint8).pin_memory()
    h_in.copy_(frames[:nh].cpu())
    h_fg = torch.empty((H, W), dtype=torch.uint8).pin_memory()
    h_bg = torch.empty((H, W, 3), dtype=torch.uint8).pin_memory()
    e2e_bgs = tb.MixtureOfGaussianV2BGS(device=ctx.local)
    L = capi.lib()
    fv, bv = C.c_int(0), C.c_int(0)
    inp = [C.c_void_p(h_in[i].data_ptr()) for i in range(nh)]
    ofg, obg = C.c_void_p(h_fg.data_ptr()), C.c_void_p(h_bg.data_ptr())

    def e2e_step(i, with_bg=True):
        for t_ in range(F):
            rc = L.bgsb_process(e2e_bgs._h, inp[(i * F + t_) % nh], W, H, W * 3, ofg, W, obg if with_bg else None, W * 3,
                                C.byref(fv), C.byref(bv))
            if rc:
                capi.check(rc)

    def wall(fn, n):
        ctx.barrier()
        t0 = time.perf_counter()
        for i in range(n):
            fn(i)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    Ke = max(2, min(K, 10))
    for i in range(2):
        e2e_step(i)
    dt = wall(e2e_step, Ke)
    assert int(h_fg.max()) in (0, 255)
    dt_mask = wall(lambda i: e2e_step(i, False), max(2, Ke // 2))

    # the same frames through the queued form of the call (bgsb_submit / bgsb_wait, the capture-loop ingest): the
    # upload of frame t+1 overlaps the download of frame t; one wait per step
    nq = 4
    q_fg = torch.empty((nq, H, W), dtype=torch.uint8).pin_memory()
    q_bg = torch.empty((nq, H, W, 3), dtype=torch.uint8).pin_memory()
    qfg = [C.c_void_p(q_fg[i].data_ptr()) for i in range(nq)]
    qbg = [C.c_void_p(q_bg[i].data_ptr()) for i in range(nq)]

    def queued_step(i):
        for t_ in range(F):
            rc = L.bgsb_submit(e2e_bgs._h, inp[(i * F + t_) % nh], W, H, W * 3, qfg[t_ % nq], W, qbg[t_ % nq], W * 3,
                               C.byref(fv), C.byref(bv))
            if rc:
                capi.check(rc)
        capi.check(L.bgsb_wait(e2e_bgs._h))

    queued_step(0)
    dtq = wall(queued_step, Ke)
    assert int(q_fg.max()) in (0, 255)
    dt, dt_mask, dtq = ctx.max_over_ranks([dt, dt_mask * Ke / max(2, Ke // 2), dtq])
    world = ctx.world
    e2e_bgs.close()
    return {"value": world * Ke * F * NPX / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": F * NPX * 3, "d2h_bytes_per_step": F * NPX * 4,
            "steps": Ke, "us_per_frame": dt / (Ke * F) * 1e6,
            "queued": {"value": world * Ke * F * NPX / dtq / 1e6, "unit": UNIT, "us_per_frame": dtq / (Ke * F) * 1e6,
                       "note": "bgsb_submit / bgsb_wait: same frames, same copies per frame, frames queued so that "
                               "the next upload overlaps this frame's download; one wait per step"},
            "mask_only": {"value": world * Ke * F * NPX / dt_mask / 1e6, "unit": UNIT, "d2h_bytes_per_step": F * NPX,
                          "note": "bgsb_process with bg = NULL: what a tracker-only caller (USTC_BGS -> CvBlobTracker) needs back"},
            "note": "bgsb_process (IBGS::process boundary): pinned host BGR frame in, mask + background image out, "
                    "synchronous per frame; upload/kernel/download of 3 row bands (2 without the background image) overlap inside the call"}


def copy_ceiling(ctx):
    """What this rank's PCIe link sustains with the OTHER ranks doing the same at the same time (bgsb_copy_probe): one
    1080p frame up (6.2 MB) and mask + background down (8.3 MB) per iteration from page-locked memory, alone and both
    directions at once on two streams, no kernel.  A synchronous call cannot beat up + down per frame, a queued one cannot
    beat the duplex figure; the e2e values are reported as fractions of the duplex ceiling."""
    import ctypes as C
    from tracking_b200 import capi
    up, dn, both = C.c_double(0), C.c_double(0), C.c_double(0)
    ctx.barrier()
    capi.check(capi.lib().bgsb_copy_probe(ctx.local, NPX * 3, NPX * 4, 200, C.byref(up), C.byref(dn), C.byref(both)))
    u, d, b = ctx.max_over_ranks([up.value, dn.value, both.value])
    return {"duplex_us_per_frame": b * 1e6, "h2d_us_per_frame": u * 1e6, "d2h_us_per_frame": d * 1e6,
            "ceiling_mpixel_s": ctx.world * NPX / b / 1e6, "serial_ceiling_mpixel_s": ctx.world * NPX / (u + d) / 1e6,
            "h2d_gbs_per_gpu": NPX * 3 / u / 1e9, "d2h_gbs_per_gpu": NPX * 4 / d / 1e9,
            "note": "copy-only, all ranks at once, slowest rank: frame up + mask and background down per iteration; "
                    "serial = up then down (the bound of a synchronous call without banding), duplex = both at once"}


def mog2_workload(ctx, S, w, h, T, nres, iters, churn=False, want_bg=True):
    """Device-resident MOG2 on S streams of w x h per GPU; returns this rank's figures for one frame set (all S streams)."""
    import tracking_b200 as tb
    from tracking_b200 import capi, synth
    torch = ctx.torch
    st = torch.cuda.current_stream().cuda_stream
    npx = w * h
    gen = synth.churn_frames_dev if churn else synth.frames_dev
    # ring of nres time steps; batch layout [S][T][h][w][3] per launch
    nb = max(1, nres // T)
    ring = torch.empty((nb, S, T, h, w, 3), dtype=torch.uint8, device="cuda")
    for b in range(nb):
        for s in range(S):
            gen(ring[b, s].data_ptr(), 1, T, w, h, t0=b * T, seed0=synth.SEED0 + ctx.rank * 1000 + s, stream=st)
    fg = torch.empty((S, T, h, w), dtype=torch.uint8, device="cuda")
    bg = torch.empty((S, T, h, w, 3), dtype=torch.uint8, device="cuda") if want_bg else None
    p = tb.MixtureOfGaussianV2BGS(device=ctx.local, nstreams=S)
    bgp = bg.data_ptr() if want_bg else None

    def step(i):
        p.process_batch_dev(ring[i % nb].data_ptr(), T, w, h, fg.data_ptr(), bgp, stream=st)

    warm = max(2 * nb, (60 + T - 1) // T)              # >= 60 frames: mode counts settle (SURVEY 8d asks for 50)
    for i in range(warm):
        step(i)
    l0 = capi.kernel_launch_count()
    ms = ctx.timed(lambda i: step(warm + i), iters)
    launches = capi.kernel_launch_count() - l0
    import numpy as np
    nm = np.concatenate([p.export_state(s)[1] for s in range(min(S, 2))])
    p.close()
    del ring, fg, bg
    torch.cuda.empty_cache()
    frames_done = iters * T
    return {"ms": ms, "launches": launches, "px": S * npx * frames_done, "mean_modes": float(nm.mean()),
            "share_5_modes": float((nm == 5).mean()), "T": T, "S": S, "frames": frames_done}


def mog2_figures(ctx, r, peak, T):
    """Aggregate (all ranks) throughput + this rank's byte figures for a mog2_workload result."""
    ms_max = ctx.max_over_ranks([r["ms"]])[0]
    px_all = ctx.sum_over_ranks([r["px"]])[0]
    live = (MOG2_FIXED_BYTES_PER_PX - 2) + (2 + MOG2_BYTES_PER_LIVE_MODE * r["mean_modes"]) / T      # in 3 + mask 1 + bg 3 per frame; state once per batch
    dense = 7 + 202.0 / T
    rate = r["px"] / (r["ms"] * 1e-3)                    # this rank, px/s
    return {"mpixel_s": px_all / (ms_max * 1e-3) / 1e6, "us_per_frame_per_stream": r["ms"] * 1e3 / (r["frames"] * r["S"]),
            "mean_live_modes_per_px": r["mean_modes"], "share_of_px_with_5_modes": r["share_5_modes"],
            "live_bytes_per_px_frame": live, "live_gbs_per_gpu": rate * live / 1e9, "frac_live": rate * live / 1e9 / peak,
            "dense_bytes_per_px_frame": dense, "dense_gbs_per_gpu": rate * dense / 1e9, "frac_section8d": rate * dense / 1e9 / peak,
            "launches": r["launches"]}


def config4(ctx, args, my_streams, peak):
    """MOG2 -> OPEN 3x3 -> connected components on this rank's share of the 64 streams (strong scaling)."""
    import numpy as np
    import tracking_b200 as tb
    from tracking_b200 import blobs, capi, synth
    from tracking_b200.pipeline import ForegroundPipeline
    from tracking_b200.streams import StreamPool
    torch = ctx.torch
    st = torch.cuda.current_stream().cuda_stream
    S = len(my_streams)
    NT = 24                                              # frame sets kept resident and cycled (24 x S x 6.2 MB)
    frames = torch.empty((NT, S, H, W, 3), dtype=torch.uint8, device="cuda")
    for t in range(NT):
        for i, s in enumerate(my_streams):
            synth.frames_dev(frames[t, i].data_ptr(), 1, 1, W, H, t0=t, seed0=synth.SEED0 + s, stream=st)
    pipe = ForegroundPipeline(5, device=ctx.local, nstreams=S)

    def step(i):
        pipe.process_dev(frames[i % NT].data_ptr(), W, H, None, None, None, stream=st)

    warm = 3 * NT
    for i in range(warm):
        step(i)
    iters = 2 * NT

    def timed_step(i):
        step(warm + i)
        if i == iters - 1:
            pipe.join_dev(st)        # clean-up + labelling run on the pipeline's own stream: the closing event waits for them

    l0 = capi.kernel_launch_count()
    ms = ctx.timed(timed_step, iters)
    launches = capi.kernel_launch_count() - l0
    ncomp0 = len(pipe.components(0))
    nm = pipe.export_mog2_state(0)[1]
    mean_modes = float(nm.mean())
    pipe.close()

    # stage split on the same frames: plugin alone (packed mask is what the pipeline's plugin launch writes, so the byte-mask
    # kernel is timed as its stand-in), clean-up alone, labelling alone (on the cleaned masks of the last frame set)
    p = tb.MixtureOfGaussianV2BGS(device=ctx.local, nstreams=S)
    fg = torch.empty((S, H, W), dtype=torch.uint8, device="cuda")
    clean = torch.empty((S, H, W), dtype=torch.uint8, device="cuda")
    for i in range(warm):
        p.process_dev(frames[i % NT].data_ptr(), W, H, fg.data_ptr(), None, stream=st)
    ms_mog = ctx.timed(lambda i: p.process_dev(frames[(warm + i) % NT].data_ptr(), W, H, fg.data_ptr(), None, stream=st), iters)
    chain = [("erode", 1), ("dilate", 1)]
    ms_morph = ctx.timed(lambda i: blobs.morph_dev(fg.data_ptr(), W, H, S, chain, clean.data_ptr(), stream=st), iters)
    cc = blobs.ConnectedComponents(W, H, device=ctx.local, max_images=S)
    ms_cc = ctx.timed(lambda i: cc.label_batch_dev(clean.data_ptr(), W, H, S, True, None, stream=st), iters)
    cc.close()
    p.close()
    del fg, clean
    torch.cuda.empty_cache()

    # host path: the StreamPool with page-locked frame rings (capture side = frames already in the pool's buffers)
    e2e = None
    if not args.no_e2e:
        ring = 3
        pool = StreamPool(capi.ALGO_MOG2, S, W, H, devices=[ctx.local], ring=ring)
        host = frames[:ring].cpu().numpy()
        for k in range(ring):
            for i in range(S):
                pool.frame_buffer(i, k)[...] = host[k, i]
        del host
        n_e2e = 5 * ring

        def pool_run(n):
            # keep ring - 1 frame sets in flight; slot buffers are "refilled" by the capture side in place
            for t in range(n):
                if t >= ring - 1:
                    pool.wait((t - (ring - 1)) % ring)
                pool.submit(t % ring, False)
            for t in range(max(0, n - (ring - 1)), n):
                pool.wait(t % ring)

        pool_run(2 * ring)
        ctx.barrier()
        t0 = time.perf_counter()
        pool_run(n_e2e)
        dt = time.perf_counter() - t0
        assert len(pool.components(0, (n_e2e - 1) % ring)) >= 0
        pool.close()
        dt_max = ctx.max_over_ranks([dt])[0]
        px_all = ctx.sum_over_ranks([S * NPX * n_e2e])[0]
        e2e = {"value": px_all / dt_max / 1e6, "unit": UNIT, "ms_per_frame_set": dt / n_e2e * 1e3,
               "h2d_bytes_per_frame_set": S * NPX * 3, "d2h_bytes_per_frame_set": S * (256 + 1) * 32,
               "note": "StreamPool (bgsb_pool_*): pinned host frames in, component tables out, ring of %d frame sets, "
                       "upload / kernels / download on three streams; PCIe-bound (6.2 MB per frame up)" % ring}
    del frames
    torch.cuda.empty_cache()

    ms_max, mog_max, morph_max, cc_max = ctx.max_over_ranks([ms, ms_mog, ms_morph, ms_cc])
    px_all = ctx.sum_over_ranks([S * NPX * iters])[0]
    live_bpp = (MOG2_FIXED_BYTES_PER_PX - 4) + MOG2_BYTES_PER_LIVE_MODE * mean_modes + 0.125 * 4      # no byte mask / bg image; packed rows: plugin, memset, clean-up in + out
    rate = S * NPX * iters / (ms * 1e-3)
    return {"workload": "MOG2 -> OPEN 3x3 -> connected components (bgsb_pipeline), 1080p, %d streams sharded over %d GPU(s)" % (C4_STREAMS, ctx.world),
            "scaling": "strong", "streams_total": C4_STREAMS, "streams_this_gpu": S,
            "value": px_all / (ms_max * 1e-3) / 1e6, "unit": UNIT, "ms_per_frame_set": ms_max / iters,
            "launches_per_frame_set": launches / iters, "components_stream0": ncomp0, "mean_live_modes_per_px": mean_modes,
            "live_bytes_per_px": live_bpp, "live_gbs_per_gpu": rate * live_bpp / 1e9, "frac_live": rate * live_bpp / 1e9 / peak,
            "dense_bytes_per_px": PIPE_DENSE_BYTES_PER_PX, "dense_gbs_per_gpu": rate * PIPE_DENSE_BYTES_PER_PX / 1e9,
            "frac_section8d": rate * PIPE_DENSE_BYTES_PER_PX / 1e9 / peak,
            "stage_ms_per_frame_set": {"mog2_byte_mask_kernel": mog_max / iters, "open_3x3_byte_masks": morph_max / iters,
                                       "cc_byte_masks_table_only": cc_max / iters,
                                       "pipeline_minus_mog2": (ms_max - mog_max) / iters,
                                       "note": "stages timed alone through the byte-mask entry points; inside the pipeline the "
                                               "mask is bit-packed between them, so clean-up + labelling cost what "
                                               "pipeline_minus_mog2 says"},
            "e2e": e2e}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from tracking_b200 import capi
    from tracking_b200.streams import shard_streams

    ctx = Ctx()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (there is no CPU fallback for the product path)")
    torch.cuda.set_device(ctx.local)
    affinity = bind_cpus(ctx)
    if ctx.world > 1:
        # NCCL prints its version banner on stdout at communicator creation, and rank 0's stdout is the ONE JSON line
        # of the contract: from here on file descriptor 1 is stderr, the line goes to the saved descriptor (emit()).
        global _STDOUT_FD
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=torch.device("cuda", ctx.local))
    capi.lib()
    peak, peak_src = measured_peak_gbs()
    my_c4 = shard_streams(C4_STREAMS, ctx.world, ctx.rank)

    parity = parity_check(ctx, my_c4) if not args.no_parity else None

    # ---- headline ----
    hd = headline(ctx, args)
    F, K, Wm = args.frames_per_step, args.steps, args.warmup
    total_px = ctx.world * K * F * NPX
    value = total_px / (hd["ms_max"] * 1e-3) / 1e6
    launch_ms = hd["ms"] / max(hd["launches"], 1)
    live_bpp = MOG2_FIXED_BYTES_PER_PX + MOG2_BYTES_PER_LIVE_MODE * hd["mean_modes"]
    alg_bytes = live_bpp * NPX
    achieved = alg_bytes / (launch_ms * 1e-3) / 1e9
    dense_gbs = MOG2_BYTES_PER_PX * NPX / (launch_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "mog2_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = "static: ncu --set full capture committed as profiles/mog2_traffic.json (%s); not measured in this run" % tj.get("source", "")
        except Exception:
            traffic = None

    # ---- host-buffer legs ----
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(ctx, args, hd["frames"])
        ceil = copy_ceiling(ctx)
        e2e["copy_ceiling"] = ceil
        e2e["frac_of_copy_ceiling"] = e2e["value"] / ceil["ceiling_mpixel_s"]
        e2e["queued"]["frac_of_copy_ceiling"] = e2e["queued"]["value"] / ceil["ceiling_mpixel_s"]
        e2e["cpu_affinity"] = affinity
    del hd["frames"]
    torch.cuda.empty_cache()

    # ---- the other roofline workloads + BASELINE configs 4 and 5 ----
    extra_w, c4, c5 = [], None, None
    if not args.headline_only:
        r16 = mog2_workload(ctx, 16, W, H, 1, 24, 48)
        f16 = mog2_figures(ctx, r16, peak, 1)
        f16["name"] = "16 x 1080p streams per GPU, T = 1 (model state 3.3 GB: HBM-resident, mog2_t1_kernel<.,0,true>)"
        rch = mog2_workload(ctx, 1, W, H, 1, 32, 256, churn=True)
        fch = mog2_figures(ctx, rch, peak, 1)
        fch["name"] = "one 1080p mode-churn stream, T = 1: five colours per pixel redrawn every 2nd frame (the dense case)"
        extra_w = [f16, fch]
        c4 = config4(ctx, args, my_c4, peak)
        c5 = {"workload": "MOG2 3840x2160, %d streams per GPU (%d in all), temporal batches" % (C5_STREAMS_PER_GPU, C5_STREAMS_PER_GPU * ctx.world),
              "scaling": "weak", "streams_per_gpu": C5_STREAMS_PER_GPU, "by_T": {}}
        for T in (1, 16):
            r5 = mog2_workload(ctx, C5_STREAMS_PER_GPU, 3840, 2160, T, 16, 16 if T == 1 else 2)
            c5["by_T"][str(T)] = mog2_figures(ctx, r5, peak, T)
        c5["value"] = c5["by_T"]["16"]["mpixel_s"]
        c5["unit"] = UNIT

    cpu = None
    if ctx.rank == 0 and ctx.world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        # about 10 s of wall clock on all host cores, about 4 s on one
        v, cdt, threads = cpu_reference_run(16, 50, 24, cores)
        v1, cdt1, _ = cpu_reference_run(1, 50, 96, 1)
        cpu = {"value": v, "unit": UNIT, "cores": threads, "kind": "port",
               "sample": "384 frames (16 steps x 24) of the same synthetic 1080p stream (same ring of %d unique frames) after "
                         "50 warm-up frames; OpenCV call-for-call replay of MixtureOfGaussianV2BGS::process on %d host "
                         "cores, %.1f s" % (NFRAMES_RESIDENT, cores, cdt),
               "one_thread": {"value": v1, "unit": UNIT, "cores": 1, "sample": "96 frames after 50 warm-up frames, %.1f s" % cdt1}}

    if ctx.rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": ctx.world, "steps": K, "warmup": Wm,
                "ms_per_step": hd["ms_max"] / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": config_dict(ctx.world),
                "clocks": hd["clocks"],
                "e2e": e2e,
                "gpu_launches": int(hd["launches"]),
                "parity": parity,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_src,
                             "kernel": "mog2_t1_kernel<SHADOWS,0,GROUP>", "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_bytes, "launch_ms": launch_ms,
                             "frac_of_8TBs_nominal": achieved / 8000.0,
                             "mean_live_modes_per_px": hd["mean_modes"], "share_of_px_with_5_modes": hd["share_5_modes"],
                             "algorithmic_bytes_per_px_live": live_bpp,
                             "algorithmic_bytes_per_px_section8d": MOG2_BYTES_PER_PX,
                             "achieved_section8d_gbs": dense_gbs, "frac_section8d": dense_gbs / peak,
                             "note": "achieved / frac use the LIVE bytes (9 + 40 * mean live modes per pixel): like the reference's "
                                     "`mode < nmodes` loop the kernel never touches dead modes, so the 209 B/px of SURVEY 8(d) "
                                     "(frac_section8d, > 1 on this stream) are not moved; one 1080p stream half-lives in the "
                                     "126 MB L2, i.e. this workload is issue/latency-bound -- the HBM-bound figure is the "
                                     "16-stream workload below, the dense one the churn workload",
                             "workloads": extra_w},
                "config4": c4, "config5": c5,
                "cpu_baseline": cpu}
        emit(json.dumps(line))
    if ctx.world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: skip the host-buffer legs")
    ap.add_argument("--no-parity", action="store_true", help="profiling runs: skip the oracle-hash self-check")
    ap.add_argument("--headline-only", action="store_true", help="profiling runs: only the headline workload")
    ap.add_argument("--frames-per-step", type=int, default=FRAMES_PER_STEP)
    ap.add_argument("--kernel-variant", type=int, default=0, help="0 production MOG2 kernel, 1 straight restatement (A/B)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the headline path's mask and background image of its last timed frame as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.warmup < 3:
        args.warmup = 3          # timing rule: W >= 3
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
