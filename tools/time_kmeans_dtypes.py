"""fp32 vs fp16 / bf16 embeddings in the K-Means filter (kmeans.py over vatlq_kmeans_*_dt) at 3 000 x 2048 (k = 150),
20 000 x 2048 (k = 1 000) and 100 000 x 2048 (k = 5 000): the fp32 entries, the native 16-bit entries, and
"bf16 -> .float() -> fp32" (what a bf16 caller paid before the 16-bit entries existed; the upcast is counted).  For each
variant: the whole kmeans_fit_select call, the k-means++ seeding alone (vatlq_kmeans_pp), one assignment step alone
(vatlq_kmeans_assign against the final centres) and the peak of torch.cuda.max_memory_allocated during the whole call
above what was allocated before it.  CUDA events around each call, median of --reps runs after one warm-up of every
variant, the variants alternating within each repetition.  The 16-bit results are checked bit for bit against the fp32
path on the upcast at every timed size.  The card's name, power limit and max SM clock are read in the same run.

    python tools/time_kmeans_dtypes.py [--sizes 3000:150,20000:1000,100000:5000] [--reps 3]
                                       [--out profiles/r08_kmeans_dtypes.json]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

D = 2048
TAGS = ("fp32", "bf16", "fp16", "bf16+upcast")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def at_size(n, k, reps, dev):
    from vatlq import _lib, kmeans as KM, ops, synth
    L = _lib.lib()
    X32 = synth.pool_embeddings(n, d=D, seed=2, kind="weak", device=dev)
    pools = {"fp32": X32, "fp16": X32.half(), "bf16": X32.bfloat16()}
    ws = torch.empty(int(L.vatlq_kmeans_workspace_bytes(n, D, k)), dtype=torch.uint8, device=dev)
    labels = torch.empty(n, dtype=torch.int32, device=dev)
    cid = torch.empty(k, dtype=torch.int32, device=dev)
    closest = torch.empty(n, dtype=torch.float64, device=dev)
    trials = 2 + int(np.log(k))
    rand = torch.rand((k - 1) * trials, dtype=torch.float64, device=dev, generator=torch.Generator(dev).manual_seed(1))
    st = lambda: C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def src(tag):
        """the X the kernels read: the pool itself, or for "+upcast" a fresh fp32 copy made inside the timed window"""
        return pools[tag.split("+")[0]].float() if "+" in tag else pools[tag]

    def call(name, X, *args):
        if X.dtype == torch.float32:
            _lib.check(getattr(L, name)(_p(X), *args), name)
        else:
            _lib.check(getattr(L, name + "_dt")(_p(X), ops.EMBEDDING_DTYPES[X.dtype], *args), name + "_dt")

    results = {}

    def whole(tag):
        results[tag] = KM.kmeans_fit_select(src(tag), k)

    def seeding(tag):
        call("vatlq_kmeans_pp", src(tag), n, D, None, k, 0, _p(rand), trials, _p(cid), _p(closest), _p(ws), ws.numel(), st())

    def assign(tag):
        call("vatlq_kmeans_assign", src(tag), n, D, _p(results["fp32"].centers), k, _p(labels), None, None, _p(ws), ws.numel(),
             st())

    steps = {"whole_call": whole, "seeding": seeding, "assign": assign}
    for t in TAGS:                                        # warm-up of every variant (and results[t] for the checks)
        for f in steps.values():
            timed(lambda: f(t))
    ref16 = {s: KM.kmeans_fit_select(pools[s].float(), k) for s in ("fp16", "bf16")}
    same = {}
    for s in ("fp16", "bf16"):
        a, b = results[s], ref16[s]
        same[s] = bool(a.query_rows == b.query_rows and torch.equal(a.labels, b.labels) and torch.equal(a.centers, b.centers)
                       and torch.equal(a.center_ids, b.center_ids) and a.n_iter == b.n_iter)
    times = {t: {s: [] for s in steps} for t in TAGS}
    for _ in range(reps):
        for t in TAGS:
            for s, f in steps.items():
                times[t][s].append(timed(lambda: f(t)))
    out = {"n": n, "k": k, "d": D, "trials": trials, "n_iter": results["fp32"].n_iter,
           "bit_equal_to_upcast": same, "x_bytes": {t: n * D * pools[t.split("+")[0]].element_size() for t in TAGS}}
    for t in TAGS:
        rec = {s: {"ms_median": float(np.median(v)), "ms_all": v} for s, v in times[t].items()}
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        whole(t)
        torch.cuda.synchronize()
        rec["peak_extra_bytes"] = torch.cuda.max_memory_allocated() - base
        rec["max_memory_allocated"] = torch.cuda.max_memory_allocated()
        out[t] = rec
    up = torch.empty_like(X32)
    out["upcast_alone_ms"] = float(np.median([timed(lambda: up.copy_(pools["bf16"])) for _ in range(max(reps, 3))]))
    del up
    for t in TAGS[1:]:
        out[f"{t}_vs_fp32"] = {s: out["fp32"][s]["ms_median"] / out[t][s]["ms_median"] for s in steps}
    print(n, k, {t: {s: round(out[t][s]["ms_median"], 2) for s in steps} for t in TAGS}, "bit-equal", same, flush=True)
    del pools, X32, ws
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="3000:150,20000:1000,100000:5000")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_kmeans_dtypes.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import vatlq  # noqa: F401
    dev = torch.device("cuda:0")
    res = {"card": card(), "reps": a.reps, "pool": "synth.pool_embeddings(kind='weak', seed=2), d = 2048",
           "l2": "X is 12-25 MB at 3 000 rows (L2-resident in every dtype), 82-164 MB at 20 000 (fits the 126 MB L2 "
                 "in 16 bits only) and 0.4-0.8 GB at 100 000; no flush between calls"}
    print(json.dumps(res["card"]), flush=True)
    res["sizes"] = [at_size(*(int(v) for v in s.split(":")), a.reps, dev) for s in a.sizes.split(",")]
    s = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(s)
    print(s)


if __name__ == "__main__":
    main()
