#!/usr/bin/env python
"""Device-resident throughput of frames whose rows are not 8-byte aligned (1918x1078); the library copies them to a
16-byte row pitch first.  Run on the GPU box: python tools/oddsize_probe.py"""
import os, sys, time, json
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "h264-h265-to-jpeg_b200")]
import torch
import h2j_b200
from bench import make_frames_torch
dev = torch.device("cuda", 0)
w, h, n = 1918, 1078, 256
d, fb, stride = make_frames_torch(64, w, h, dev)
d = d.repeat(n // 64, 1).contiguous()
with h2j_b200.Encoder(max_width=w, max_height=h, max_batch=n, n_slots=1) as e:
    for _ in range(2):
        e.submit_device(0, d.data_ptr(), stride, n, w, h); e.collect_device(0)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(5):
        e.submit_device(0, d.data_ptr(), stride, n, w, h); e.collect_device(0)
    torch.cuda.synchronize(); dt = (time.perf_counter() - t0) / 5
print(json.dumps({"1918x1078_batch256_frames_per_s": round(n / dt)}))
