"""ABL: lookup-table kernels vs arithmetic kernel, 1 and 16 streams of 1080p (GPU box, measurement tooling).
Table 1 is the production routing, 2 the per-thread table kernel, 0 the arithmetic kernel; --table1 runs table 1 only."""
import os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tracking_b200 as tb
from tracking_b200 import synth
w, h, NT = 1920, 1080, 6
st = torch.cuda.current_stream().cuda_stream
for S in (1, 16):
    frames = torch.empty((NT, S, h, w, 3), dtype=torch.uint8, device="cuda")
    for t in range(NT):
        synth.frames_dev(frames[t].data_ptr(), S, 1, w, h, t0=t, stream=st)
    fg = torch.empty((S, h, w), dtype=torch.uint8, device="cuda")
    bg = torch.empty((S, h, w, 3), dtype=torch.uint8, device="cuda")
    ref = None
    for table in ((1,) if "--table1" in sys.argv else (1, 2, 0)):
        p = tb.AdaptiveBackgroundLearning(nstreams=S, ablTable=table)
        k = [0]
        def run(n):
            for _ in range(n):
                p.process_dev(frames[k[0] % NT].data_ptr(), w, h, fg.data_ptr(), bg.data_ptr(), stream=st); k[0] += 1
        run(8)
        torch.cuda.synchronize(); e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 60
        e0.record(); run(n); e1.record(); torch.cuda.synchronize()
        dt = e0.elapsed_time(e1) / n * 1e-3
        sig = (int(fg.long().sum()), int(bg.long().sum()))
        if ref is None: ref = sig
        print("S=%d table=%d  %.1f us/step  %.0f GB/s (10 B/px)  same_result=%s" % (S, table, dt * 1e6, S * w * h * 10 / dt / 1e9, sig == ref))
        p.close()
