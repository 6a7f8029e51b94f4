"""Short driver for ncu captures of the K-Means filter kernels and the MPE / Margin fast path:
    ncu --set full --clock-control none --import-source on -k regex:'km_gemm_kernel|peak_unc_reg_kernel' -c 8 \
        -o gpurun_out/prof_kmeans python tools/prof_kmeans.py
Launch order: 3 x peak_unc_reg_kernel, 12 seeding distance GEMMs (km_gemm_kernel<128,16,..,1>), 3 assignment GEMMs
(km_gemm_kernel<64,64,2,2,0>)."""
import ctypes as C
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
import vatlq
from vatlq import ops, synth

dev = "cuda:0"
n, k = int(os.environ.get("PROF_ROWS", 100000)), int(os.environ.get("PROF_K", 5000))
H, ip, inx, bb = synth.device_pool(int(os.environ.get("PROF_FRAMES", 20000)), dev, seed=1)
for _ in range(3):
    ops.peak_uncertainty(H)
torch.cuda.synchronize()
del H
L = vatlq._lib.lib()
p = lambda t: C.c_void_p(t.data_ptr())
X = synth.pool_embeddings(n, kind="weak", seed=2, device=dev)
d = X.shape[1]
ws = torch.empty(int(L.vatlq_kmeans_workspace_bytes(n, d, k)), dtype=torch.uint8, device=dev)
st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
cid = torch.empty(k, dtype=torch.int32, device=dev)
closest = torch.empty(n, dtype=torch.float64, device=dev)
trials = 2 + int(np.log(k))
rand = torch.rand(11 * trials, dtype=torch.float64, device=dev)
assert L.vatlq_kmeans_pp(p(X), n, d, None, 12, 0, p(rand), trials, p(cid), p(closest), p(ws), ws.numel(), st) == 0
torch.cuda.synchronize()
Cr = X[torch.randperm(n, device=dev)[:k]].double().contiguous()
labels = torch.empty(n, dtype=torch.int32, device=dev)
for _ in range(3):
    assert L.vatlq_kmeans_assign(p(X), n, d, p(Cr), k, p(labels), None, None, p(ws), ws.numel(), st) == 0
torch.cuda.synchronize()
print("ok", int(labels.max()))
