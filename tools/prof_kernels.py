"""Short driver for ncu captures at bench scale: one heat-map scan, the 8f kernels, and a core-set
selection long enough to reach the pruned steady state.
    ncu --set full --clock-control none --import-source on -k regex:'pass_kernel_tma|pairs_plan' \
        --launch-skip 1500 -c 8 -o gpurun_out/prof_coreset python tools/prof_kernels.py
    ncu --set full --clock-control none -k regex:'scan_tma|entropy_kernel|cos_colsum_kernel|cos_rowsum' -c 6 \
        -o gpurun_out/prof_stream python tools/prof_kernels.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vatlq
from vatlq import ops, synth

frames = int(os.environ.get("PROF_FRAMES", 20000))
rows = int(os.environ.get("PROF_ROWS", 170000))
k = int(os.environ.get("PROF_K", 5200))
batch = int(os.environ.get("PROF_BATCH", 16))
dev = "cuda:0"
H, ip, inx, bb = synth.device_pool(frames, dev, seed=1)
for _ in range(2):
    r = ops.heatmap_scan(H, ip, inx, bb)
ops.heatmap_entropy(H)
torch.cuda.synchronize()
mp = ops.peak_uncertainty(H[:4000])
torch.cuda.synchronize()
del H
X = synth.pool_embeddings(rows, device=dev)
ops.cosine_rowsum(X)
unc = synth.pool_unc(rows, device=dev)
picks, st = ops.coreset_select(X, unc, [], k, 0.0, 0.01, batch=batch)
torch.cuda.synchronize()
print("ok", st, ops.prune_stats())
if os.environ.get("PROF_TC", "1") != "0":      # the tensor-core labelled-set initialisation (tc_prefilter / tc_rescore)
    lab = torch.from_numpy(synth.pool_labeled(rows, int(os.environ.get("PROF_LABELLED", rows // 10)))).to(dev)
    md = torch.empty(rows, dtype=torch.float64, device=dev)
    print("tc init", ops.coreset_init_tc(X, lab, md, 0, rows)[:2])
