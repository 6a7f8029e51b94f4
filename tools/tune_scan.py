"""Time the heat-map scan alone (CUDA events, inputs >> L2) and print achieved HBM GB/s."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vatlq
from vatlq import ops, synth

dev = "cuda:0"
for frames in [int(x) for x in os.environ.get("SCAN_FRAMES", "60000,1080").split(",")]:
    H, ip, inx, bb = synth.device_pool(frames, dev, seed=1)
    for _ in range(3):
        ops.heatmap_scan(H, ip, inx, bb)
    reps = 10 if frames > 10000 else 200
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        ops.heatmap_scan(H, ip, inx, bb)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    print(f"scan frames={frames} {ms:.3f} ms  {frames * 208896 / ms / 1e6:.0f} GB/s")
    del H
