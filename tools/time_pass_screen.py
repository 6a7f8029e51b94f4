"""The paired pass with the fp16 screen off / on / in verify mode on the counter-based bench pools: per-launch time
of a round's update of min_d (CUDA events around every pass launch, the figure bench.py reports as
roofline.avg_launch_us), the fraction f of the screened rows listed for the exact fp64 arithmetic, verify
violations (must be 0) and whether the pick lists agree.  With the screen on it also gives the bytes a launch
moves (fp16 screen rows + listed fp32 rows + 40 B of state per row) and their fraction of the 6.65 TB/s HBM
figure bench.py uses, and the time of the fill of the fp16 copy (torch.profiler, one call per pool).  The first
line names the card and its power limit.  One JSON line per (pool, mode).
    python tools/time_pass_screen.py [rows] [k] > pass_screen.json"""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import vatlq
from vatlq import ops, synth

HBM_GBS = 6650.0   # bench.py's fallback HBM figure
rows = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
k = int(sys.argv[2]) if len(sys.argv) > 2 else rows // 20
dev = torch.device("cuda:0")
lib = vatlq._lib.lib()
smi = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(json.dumps({"gpu": torch.cuda.get_device_name(0), "nvidia_smi": smi, "rows": rows, "k": k}), flush=True)


def fill_ms(X, unc):
    """Device time of half_copy_kernel in one short selection (the copy is filled once per call)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ops.coreset_select(X, unc, [], 64, 0.0, 0.01)
        torch.cuda.synchronize()
    us = [e.device_time_total for e in prof.key_averages() if "half_copy_kernel" in e.key]
    return us[0] / 1e3 if us else None


for kind in ("clustered", "weak", "iid"):
    X = synth.pool_embeddings(rows, device=dev, kind=kind)
    unc = synth.pool_unc(rows, device=dev)
    ops.coreset_select(X, unc, [], min(k, 300), 0.0, 0.01)   # warm-up (module load, workspace)
    torch.cuda.synchronize()
    fms = fill_ms(X, unc)
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
        avg_us = 1e3 * tot.value / max(1, n_pass.value)
        rec = {"pool": kind, "screen": mode, "ms": e0.elapsed_time(e1), "rounds": st.rounds,
               "pass_launches_timed": n_pass.value, "avg_launch_us": avg_us,
               "rows_screened": sc["screened"], "rows_listed": sc["listed"],
               "f": sc["listed"] / sc["screened"] if sc["screened"] else None,
               "verify_violations": sc["violations"], "picks_equal": h == ref}
        if mode == "on":
            # the paired launches screen every streamed row once; the solo launches of the round do no work here
            nl = max(1, n_pass.value)
            moved = (sc["screened"] * (2048 * 2 + 40) + sc["listed"] * 2048 * 4) / nl
            rec.update({"bytes_per_launch": moved, "hbm_frac": moved / (avg_us * 1e-6) / (HBM_GBS * 1e9),
                        "fill_ms": fms})
        print(json.dumps(rec), flush=True)
    del X, unc
