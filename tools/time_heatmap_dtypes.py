"""fp32 vs fp16 / bf16 heat maps on the device: scan, Entropy and MPE / Margin on the 170 000-frame bench pool
(native 16-bit kernels, and "upcast then the fp32 kernel", which is what a 16-bit estimator cost before they
existed), the stage count of the 16-bit scan, the 1 M-frame pool resident in bf16 (no ring) through the whole
config-5 query, and the chunked host-to-device path.  CUDA events; every variant is warmed up and the variants
alternate within each repetition; the pool (17.8-35.5 GB) is far larger than L2.

    python tools/time_heatmap_dtypes.py [--frames 170000] [--reps 5] [--stage-libs a.so,b.so] [--no-1m] [--out F]

--stage-libs: libvatlq.so builds that differ only in -DVQ_SCAN_STAGES16 (each timed in its own process)."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

COPY_PEAK = 6.55e12              # B/s, device-to-device copy measured on B200 (DESIGN §4.1)
CHUNK = 8192                     # frames per batch of the "upcast, then fp32" path (an estimator batch)
DT = {"fp32": torch.float32, "fp16": torch.float16, "bf16": torch.bfloat16}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def timed(fn, reps_inner=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps_inner):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps_inner


def bench_pool(frames, dev):
    from vatlq import synth
    segs, bb, ip, inx, X, _ = synth.rank_pool(frames, 0, frames, dev, "clustered")
    assert len(segs) == 1
    return segs[0][1], bb, ip, inx, X


def kernels_on_pool(H32, reps):
    """scan / entropy / peaks: fp32, native 16-bit, and 16-bit upcast per CHUNK then fp32"""
    from vatlq import ops
    n = H32.shape[0]
    pools = {"fp32": H32, "fp16": H32.half(), "bf16": H32.bfloat16()}
    buf = torch.empty((CHUNK,) + tuple(H32.shape[1:]), dtype=torch.float32, device=H32.device)
    fr = H32[0].numel()
    ops_ = {"scan": lambda H: ops.heatmap_scan(H), "entropy": ops.heatmap_entropy,
            "peaks": lambda H: ops.peak_uncertainty(H)}

    def run(op, tag):
        f = ops_[op]
        if tag in ("fp32", "fp16", "bf16"):
            return lambda: f(pools[tag])
        src = pools[tag.split("+")[0]]

        def up():
            for a in range(0, n, CHUNK):
                b = min(n, a + CHUNK)
                buf[:b - a].copy_(src[a:b])
                f(buf[:b - a])
        return up

    tags = ["fp32", "bf16", "fp16", "bf16+upcast", "fp16+upcast"]
    times = {op: {t: [] for t in tags} for op in ops_}
    for op in ops_:
        for t in tags:
            timed(run(op, t))                       # warm-up of every shape
    for _ in range(reps):
        for op in ops_:
            for t in tags:
                times[op][t].append(timed(run(op, t)))
    out = {}
    for op in ops_:
        out[op] = {}
        for t in tags:
            ms = float(np.median(times[op][t]))
            es = 4 if t == "fp32" else 2
            byts = n * fr * (es if "+" not in t else (2 + 4 + 4))     # upcast: read 2, write 4, kernel reads 4
            out[op][t] = {"ms_median": ms, "ms_all": times[op][t], "frames_per_s": n / ms * 1e3,
                          "bytes": byts, "GB_per_s": byts / ms / 1e6, "share_of_copy_peak": byts / ms * 1e3 / COPY_PEAK}
        for s in ("fp16", "bf16"):
            out[op][f"{s}_native_vs_upcast_speedup"] = out[op][f"{s}+upcast"]["ms_median"] / out[op][s]["ms_median"]
            out[op][f"{s}_native_vs_fp32_speedup"] = out[op]["fp32"]["ms_median"] / out[op][s]["ms_median"]
    del pools, buf
    return out


def scan_only(frames, reps):
    """bf16 scan time of the library this process loaded (VATLQ_LIB): one --stage-libs variant"""
    from vatlq import ops
    H = bench_pool(frames, "cuda:0")[0].bfloat16()
    torch.cuda.empty_cache()
    timed(lambda: ops.heatmap_scan(H))
    ms = float(np.median([timed(lambda: ops.heatmap_scan(H)) for _ in range(reps)]))
    return {"ms_median": ms, "GB_per_s": frames * H[0].numel() * 2 / ms / 1e6}


def _sha(p):
    return hashlib.sha256(np.asarray(p, dtype="<i8").tobytes()).hexdigest()


def resident_1m(dev):
    """config 5 (1 M frames, k = 50 000) with the pool resident in bf16, every frame materialised (104.4 GB), then the
    fp32 path on the exact upcast of the same content in today's ring form (250 000 frames, 52 GB)"""
    import vatlq
    from vatlq import ops, synth
    z = np.load(os.path.join(ROOT, "tests", "golden", "coreset_scale_c5.npz"))
    n, k, moks = int(z["n"]), int(z["k_full"]), float(z["moks"])
    ring = synth.HEAT_RING
    tid, pos, ip, inx = synth.pool_tracks(n, seed=0, ring=ring)
    bb = synth.pool_boxes(n, 0, n, seed=0, device=dev)
    X = synth.pool_embeddings(n, 0, n, seed=2, kind="clustered", device=dev)
    ipd, inxd = torch.from_numpy(ip).to(dev), torch.from_numpy(inx).to(dev)
    W = synth.ae_weights(42, 4)
    lab = synth.pool_labeled(n, int(n * float(z["labeled_frac"]))).tolist()
    out = {"n": n, "k": k}
    # (1) bf16, 1 M distinct frames
    Hb = torch.empty((n, 17, 64, 48), dtype=torch.bfloat16, device=dev)
    for a in range(0, n, 25000):
        b = min(n, a + 25000)
        Hb[a:b] = synth.pool_heatmaps(tid, pos, a, b, seed=0, device=dev, ring=ring)
    torch.cuda.synchronize()
    out["bf16_pool_bytes"] = Hb.numel() * 2
    ops.heatmap_scan(Hb[:1024], ipd[:1024], inxd[:1024], bb[:1024])
    out["bf16_scan_ms"] = timed(lambda: ops.heatmap_scan(Hb, ipd, inxd, bb))
    vatlq.run_query(Hb[:4096], bb[:4096], ipd[:4096], inxd[:4096], X[:4096], W, [], 64, moks, 0.01, batch=16, device=dev)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = vatlq.run_query(Hb, bb, ipd, inxd, X, W, lab, k, moks, 0.01, batch=16, device=dev)
    torch.cuda.synchronize()
    out["bf16_query_s"] = time.perf_counter() - t0
    out["bf16_pick_sha256"] = _sha(r.picks.cpu().numpy())
    out["bf16_peak_mem_GB"] = torch.cuda.max_memory_allocated(dev) / 1e9
    del Hb, r
    torch.cuda.empty_cache()
    # (2) fp32 ring form of the exact upcast of the same content
    R = synth.pool_heatmaps(tid, pos, 0, ring, seed=0, device=dev, ring=ring)
    R.copy_(R.bfloat16())
    segs = [(a, R[:min(ring, n - a)]) for a in range(0, n, ring)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = vatlq.run_query(segs, bb, ipd, inxd, X, W, lab, k, moks, 0.01, batch=16, device=dev)
    torch.cuda.synchronize()
    out["fp32_ring_upcast_query_s"] = time.perf_counter() - t0
    out["fp32_ring_upcast_pick_sha256"] = _sha(r.picks.cpu().numpy())
    out["pick_hashes_equal"] = out["bf16_pick_sha256"] == out["fp32_ring_upcast_pick_sha256"]
    del R, segs, r, X
    torch.cuda.empty_cache()
    return out


def h2d_chunked(H32, bb, ip, inx, reps):
    """QueryPass.score_chunk fed from pinned host memory (a host ring of CHUNK frames, cycled over the pool)"""
    import vatlq
    from vatlq import synth
    n = H32.shape[0]
    dev = H32.device
    out = {}
    for tag in ("fp32", "bf16", "fp32", "bf16")[:2 * max(1, min(reps, 2))]:
        host = H32[:CHUNK].to(DT[tag]).cpu().pin_memory()
        qp = vatlq.QueryPass(n, dev, ae_weights=synth.ae_weights(42, 4), uncertainty="THC+WPU")

        def feed():
            qp._carry = None
            for a in range(0, n, CHUNK):
                b = min(n, a + CHUNK)
                qp.score_chunk(a, host[:b - a].to(dev, non_blocking=True), bb[a:b], ip[a:b], inx[a:b])
        feed()
        ms = timed(feed)
        rec = out.setdefault(tag, {"ms": [], "h2d_bytes": n * H32[0].numel() * (4 if tag == "fp32" else 2)})
        rec["ms"].append(ms)
        del host, qp
    for rec in out.values():
        rec["ms_median"] = float(np.median(rec["ms"]))
        rec["frames_per_s"] = n / rec["ms_median"] * 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=170000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--stage-libs", default="")
    ap.add_argument("--scan-only", action="store_true")
    ap.add_argument("--no-1m", action="store_true")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    if a.scan_only:
        print(json.dumps(scan_only(a.frames, a.reps)))
        return
    import vatlq  # noqa: F401
    dev = torch.device("cuda:0")
    res = {"card": card(), "frames": a.frames, "reps": a.reps, "upcast_chunk": CHUNK, "copy_peak_B_per_s": COPY_PEAK}
    print(json.dumps(res["card"]), flush=True)
    if a.stage_libs:
        res["scan_bf16_stages"] = {}
        for lib in a.stage_libs.split(","):
            p = subprocess.run([sys.executable, __file__, "--scan-only", "--frames", str(a.frames), "--reps", str(a.reps)],
                               capture_output=True, text=True, env=dict(os.environ, VATLQ_LIB=lib))
            res["scan_bf16_stages"][os.path.basename(os.path.dirname(lib))] = (
                json.loads(p.stdout.strip().splitlines()[-1]) if p.returncode == 0 else p.stderr[-2000:])
            print(lib, res["scan_bf16_stages"][os.path.basename(os.path.dirname(lib))], flush=True)
    H32, bb, ip, inx, X = bench_pool(a.frames, dev)
    del X
    res["kernels"] = kernels_on_pool(H32, a.reps)
    for op, r in res["kernels"].items():
        print(op, {t: round(v["ms_median"], 3) for t, v in r.items() if isinstance(v, dict)}, flush=True)
    res["h2d_chunked"] = h2d_chunked(H32, bb, ip, inx, a.reps)
    print("h2d", {t: round(v["ms_median"], 1) for t, v in res["h2d_chunked"].items()}, flush=True)
    del H32, bb, ip, inx
    torch.cuda.empty_cache()
    if not a.no_1m:
        res["resident_1m_c5"] = resident_1m(dev)
        print("1M", json.dumps(res["resident_1m_c5"]), flush=True)
    s = json.dumps(res, indent=1)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(s)
    print(s)


if __name__ == "__main__":
    main()
