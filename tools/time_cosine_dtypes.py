"""fp32 vs fp16 / bf16 embeddings in the Influence / Diversity cosine row sums (vatlq_cosine_colsum_dt +
vatlq_cosine_rowsum_dt) at 170 000 and 1 000 000 rows x 2048: the fp32 kernels, the native 16-bit kernels, and
"upcast, then fp32" (X.float() into a preallocated buffer, then the fp32 kernels: what a 16-bit estimator cost before
the 16-bit kernels existed).  Each pass runs over all rows and over a row list of 90 % of them (the Influence call
of a round with 10 % labelled).  CUDA events around each call, median of --reps runs after one warm-up of every
variant, the variants alternating within each repetition; X (0.7-8.2 GB) is far larger than the 126 MB L2.

Bytes are the algorithm's: each pass reads every listed row once (m * d * sizeof(T)) plus the row list (8 B per row);
the upcast also reads the 16-bit X and writes the fp32 copy.  The 16-bit outputs are checked bit for bit against the
fp32 kernels on the upcast at every timed size.

    python tools/time_cosine_dtypes.py [--rows 170000,1000000] [--reps 7] [--out profiles/r07_cosine_dtypes.json]"""
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
COPY_PEAK = 6.55e12              # B/s, device-to-device copy measured on B200 (DESIGN §4.1)
HBM_PEAK = 7.7e12                # B/s, HGX B200 data sheet, one GPU
DT = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


class Cosine:
    """the two C calls on preallocated buffers (no allocation inside the timed window)"""

    def __init__(self, m, dev):
        from vatlq import _lib
        self.L, self.check = _lib.lib(), _lib.check
        self.ws_bytes = self.L.vatlq_cosine_workspace_bytes(D)
        self.ws = torch.empty(self.ws_bytes, dtype=torch.uint8, device=dev)
        self.S = torch.empty(D, dtype=torch.float64, device=dev)
        self.out = torch.empty(m, dtype=torch.float64, device=dev)

    def colsum(self, X, rows):
        from vatlq import ops
        n = X.shape[0]
        m = n if rows is None else rows.numel()
        self.check(self.L.vatlq_cosine_colsum_dt(_p(X), ops.EMBEDDING_DTYPES[X.dtype], n, D, _p(rows), m, _p(self.S),
                                                 _p(self.ws), self.ws_bytes, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   "vatlq_cosine_colsum_dt")

    def rowsum(self, X, rows):
        from vatlq import ops
        n = X.shape[0]
        m = n if rows is None else rows.numel()
        self.check(self.L.vatlq_cosine_rowsum_dt(_p(X), ops.EMBEDDING_DTYPES[X.dtype], n, D, _p(rows), m, _p(self.S),
                                                 float(m), _p(self.out), C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                   "vatlq_cosine_rowsum_dt")


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def at_size(n, reps, dev):
    from vatlq import synth
    X32 = synth.pool_embeddings(n, d=D, seed=2, kind="clustered", device=dev)
    pools = {"fp32": X32, "fp16": X32.half(), "bf16": X32.bfloat16()}
    up = torch.empty_like(X32)
    lab = synth.pool_labeled(n, n // 10)
    keep = np.ones(n, bool)
    keep[lab] = False
    row_lists = {"all": None, "rows90": torch.from_numpy(np.nonzero(keep)[0]).to(dev)}
    cos = Cosine(n, dev)
    res = {"rows": n, "d": D}
    for rl, rows in row_lists.items():
        m = n if rows is None else rows.numel()
        # bit-for-bit check of the 16-bit outputs against the fp32 kernels on the upcast, at this size
        same = {}
        for s in ("fp16", "bf16"):
            outs = []
            for X in (pools[s], pools[s].float()):
                cos.colsum(X, rows)
                cos.rowsum(X, rows)
                outs.append((cos.S.clone(), cos.out[:m].clone()))
            same[s] = all(torch.equal(a.view(torch.int64), b.view(torch.int64)) for a, b in zip(*outs))
        tags = ["fp32", "bf16", "fp16", "bf16+upcast", "fp16+upcast"]

        def variant(tag):
            if "+" not in tag:
                X = pools[tag]
                return {"colsum": lambda: cos.colsum(X, rows), "rowsum": lambda: cos.rowsum(X, rows)}
            src = pools[tag.split("+")[0]]
            return {"upcast": lambda: up.copy_(src), "colsum": lambda: cos.colsum(up, rows),
                    "rowsum": lambda: cos.rowsum(up, rows)}

        runs = {t: variant(t) for t in tags}
        times = {t: {k: [] for k in runs[t]} for t in tags}
        for t in tags:                                    # warm-up of every variant
            for f in runs[t].values():
                timed(f)
        for _ in range(reps):
            for t in tags:
                for k, f in runs[t].items():
                    times[t][k].append(timed(f))
        out = {"m": m, "bit_equal_to_upcast": same}
        for t in tags:
            es = 2 if t != "fp32" else 4
            ev = 4 if "+" in t else es                    # the kernels of "upcast, then fp32" read fp32
            row_list = 0 if rows is None else 8 * m
            pass_bytes = m * D * ev + row_list
            rec = {}
            total = 0.0
            for k, v in times[t].items():
                ms = float(np.median(v))
                total += ms
                b = n * D * (es + 4) if k == "upcast" else pass_bytes
                rec[k] = {"ms_median": ms, "ms_all": v, "bytes": b, "GB_per_s": b / ms / 1e6,
                          "share_of_copy_peak": b / ms * 1e3 / COPY_PEAK, "share_of_hbm_datasheet": b / ms * 1e3 / HBM_PEAK}
            need = 2 * m * D * es + 2 * row_list              # the bytes the two passes must read in T
            rec["total"] = {"ms_median": total, "bytes_needed": need, "GB_per_s_of_needed": need / total / 1e6}
            out[t] = rec
        for s in ("fp16", "bf16"):
            out[f"{s}_native_vs_fp32_speedup"] = out["fp32"]["total"]["ms_median"] / out[s]["total"]["ms_median"]
            out[f"{s}_native_vs_upcast_speedup"] = out[f"{s}+upcast"]["total"]["ms_median"] / out[s]["total"]["ms_median"]
        res[rl] = out
        print(n, rl, {t: round(out[t]["total"]["ms_median"], 3) for t in tags}, "bit-equal", same, flush=True)
    del pools, up, X32
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", default="170000,1000000")
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r07_cosine_dtypes.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    import vatlq  # noqa: F401
    dev = torch.device("cuda:0")
    res = {"card": card(), "reps": a.reps, "copy_peak_B_per_s": COPY_PEAK, "hbm_datasheet_B_per_s": HBM_PEAK,
           "l2": "X (0.7-8.2 GB) is far larger than the 126 MB L2; no flush between passes"}
    print(json.dumps(res["card"]), flush=True)
    res["sizes"] = [at_size(int(n), a.reps, dev) for n in a.rows.split(",")]
    s = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(s)
    print(s)


if __name__ == "__main__":
    main()
