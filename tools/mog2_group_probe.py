"""MOG2 T = 1 on S x 1080p streams (byte mask + background image), steady state: us per frame-stream.  python tools/mog2_group_probe.py S"""
import json, os, sys
import torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import tracking_b200 as tb
from tracking_b200 import synth
S = int(sys.argv[1]) if len(sys.argv) > 1 else 16
W, H = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (1920, 1080)
NF = 24 if W * H * S < 40e6 else 8
st = torch.cuda.current_stream().cuda_stream
d = torch.empty((NF, S, H, W, 3), dtype=torch.uint8, device="cuda")
for t in range(NF):
    synth.frames_dev(d[t].data_ptr(), S, 1, W, H, t0=t, stream=st)
fg = torch.empty((S, H, W), dtype=torch.uint8, device="cuda"); bg = torch.empty((S, H, W, 3), dtype=torch.uint8, device="cuda")
p = tb.MixtureOfGaussianV2BGS(nstreams=S)
for k in range(4 * NF):
    p.process_dev(d[k % NF].data_ptr(), W, H, fg.data_ptr(), bg.data_ptr(), stream=st)
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
n = 4 * NF
e0.record()
for k in range(n):
    p.process_dev(d[k % NF].data_ptr(), W, H, fg.data_ptr(), bg.data_ptr(), stream=st)
e1.record(); torch.cuda.synchronize()
us = e0.elapsed_time(e1) / n * 1e3
print(json.dumps(dict(streams=S, geometry=[W, H], us_per_frame_set=us, us_per_frame_stream=us / S, gpx_s=S * W * H / us / 1e3)))
