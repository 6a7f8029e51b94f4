"""Core-set selection on fp32, fp16 and bf16 features of the config-4 (170 000 frames) and config-5 (1 M frames)
feature pools: selection time per dtype (CUDA events around ops.coreset_select, dtypes alternating within each
repetition after one warm-up call each), the peak bytes allocated by one call, and the sha256 of the picks.  The 16-bit
pools are the fp32 pool rounded once; each 16-bit run's picks must equal those of the fp32 run on its exact upcast
(`upcast_sha256`).  The card's name and power limit are read in the same run.  Round 0 as in bench.py: no labelled
rows, k = 5 % of the pool, batch 16, lambda 0.01.

    python tools/time_coreset_dtypes.py [--reps 3] [--configs 4,5] [--out F]"""
import argparse
import hashlib
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

FRAMES = {4: 170000, 5: 1000000}
DT = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def sha(picks):
    return hashlib.sha256(picks.cpu().numpy().tobytes()).hexdigest()


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--reps", type=int, default=3)
    p.add_argument("--configs", default="4,5")
    p.add_argument("--out", default=None)
    a = p.parse_args()
    from vatlq import ops, synth
    dev = torch.device("cuda:0")
    out = {"card": card(), "configs": {}}
    for cfg in [int(c) for c in a.configs.split(",")]:
        n = FRAMES[cfg]
        k = int(n * 0.05)
        X32 = synth.pool_embeddings(n, d=2048, seed=2, kind="clustered", device=dev)
        unc = synth.pool_unc(n, device=dev)
        pools = {"fp32": X32, "fp16": X32.half(), "bf16": X32.bfloat16()}
        run = lambda X: ops.coreset_select(X, unc, [], k, 0.0, 0.01, batch=16)
        res = {}
        for name, X in pools.items():          # warm-up, hashes, peak bytes (one call each)
            torch.cuda.synchronize()
            torch.cuda.reset_peak_memory_stats(dev)
            base = torch.cuda.memory_allocated(dev)
            picks, st = run(X)
            torch.cuda.synchronize()
            res[name] = {"picks_sha256": sha(picks), "peak_call_bytes": torch.cuda.max_memory_allocated(dev) - base,
                         "X_bytes": X.numel() * X.element_size(), "passes": st.passes, "rounds": st.rounds, "ms": []}
            if name != "fp32":
                up, _ = run(X.float())
                res[name]["upcast_sha256"] = sha(up)
                res[name]["equal_to_upcast"] = res[name]["picks_sha256"] == res[name]["upcast_sha256"]
                torch.cuda.empty_cache()
        for _ in range(a.reps):                  # alternating dtypes
            for name, X in pools.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                run(X)
                e1.record()
                torch.cuda.synchronize()
                res[name]["ms"].append(round(e0.elapsed_time(e1), 2))
        for r in res.values():
            r["ms_median"] = sorted(r["ms"])[len(r["ms"]) // 2]
        out["configs"][f"config{cfg}"] = {"frames": n, "k": k, "dtypes": res}
        print(json.dumps({f"config{cfg}": out["configs"][f"config{cfg}"]}), flush=True)
        del pools, X32
        torch.cuda.empty_cache()
    print(json.dumps({"card": out["card"]}))
    if a.out:
        with open(a.out, "w") as fh:
            json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
