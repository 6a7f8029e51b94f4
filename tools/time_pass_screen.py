"""The paired pass with the TF32 screen off / on / in verify mode on the counter-based bench pools: per-launch time
of a round's update of min_d (CUDA events around every pass launch, the figure bench.py reports as
roofline.avg_launch_us), the fraction f of the screened rows listed for the exact fp64 arithmetic, verify
violations (must be 0) and whether the pick lists agree.  One JSON line per (pool, mode).
    python tools/time_pass_screen.py [rows] [k] > pass_screen.json"""
import ctypes as C
import hashlib
import json
import os
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vatlq
from vatlq import ops, synth

rows = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
k = int(sys.argv[2]) if len(sys.argv) > 2 else rows // 20
dev = torch.device("cuda:0")
lib = vatlq._lib.lib()
print(json.dumps({"gpu": torch.cuda.get_device_name(0), "rows": rows, "k": k}), flush=True)
for kind in ("clustered", "weak", "iid"):
    X = synth.pool_embeddings(rows, device=dev, kind=kind)
    unc = synth.pool_unc(rows, device=dev)
    ops.coreset_select(X, unc, [], min(k, 300), 0.0, 0.01)   # warm-up (module load, workspace)
    torch.cuda.synchronize()
    ref = None
    for mode in ("off", "on", "verify"):
        ops.set_screen(mode)
        ops.screen_stats(reset=True)
        lib.vatlq_profile_passes(1)
        lib.vatlq_profile_read(None, None, None, 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        picks, st = ops.coreset_select(X, unc, [], k, 0.0, 0.01)
        e1.record()
        torch.cuda.synchronize()
        tot, n_pass, n_picks = C.c_double(), C.c_int64(), C.c_int64()
        lib.vatlq_profile_read(C.byref(tot), C.byref(n_pass), C.byref(n_picks), 1)
        lib.vatlq_profile_passes(0)
        ops.set_screen("env")
        sc = ops.screen_stats(reset=True)
        h = hashlib.sha256(picks.cpu().numpy().tobytes()).hexdigest()
        ref = ref or h
        print(json.dumps({"pool": kind, "screen": mode, "ms": e0.elapsed_time(e1), "rounds": st.rounds,
                          "pass_launches_timed": n_pass.value, "avg_launch_us": 1e3 * tot.value / max(1, n_pass.value),
                          "rows_screened": sc["screened"], "rows_listed": sc["listed"],
                          "f": sc["listed"] / sc["screened"] if sc["screened"] else None,
                          "verify_violations": sc["violations"], "picks_equal": h == ref}), flush=True)
    del X, unc
