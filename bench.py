#!/usr/bin/env python
"""bench.py — the AL query pass (THC + local-peak + WPU + fusion + core-set) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 1..5] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One "step" = one complete query over a fixed synthetic pool.  `--config` picks BASELINE.json's
configs[config-1]:
    1  THC + local-peak + coordinates on 256 frames (the reference's own CPU-runnable case)
    2  WPU on 10 000 poses
    3  core-set selection of 5 % from 100 000 x 2048 features
    4  full THC+WPU+core-set query over the PoseTrack21-sized pool (170 000 frames)
    5  full query over the 1 M-frame pool (the north_star target; the default)
The pool is ONE global, counter-based synthetic pool (vatl4pose-wacv2024_b200/synth.py `pool_*`): every
rank cuts its contiguous frame range out of it, so N = 1/2/4/8 process the same pool (strong scaling) and
must select the same frames: every line carries `picks_sha256`, and where tests/golden/ holds the
REFERENCE's pick list for the configuration (oracle/pin_scale.py) the run fails (exit code 3) if the
picks differ.  `value` = frames of the pool / time of one query with the pool resident in HBM; `e2e` =
the same query through the public API with the pool in pinned host memory (H2D copies of heat maps /
boxes / flags / features and the D2H read of the picks inside the timed region).  ONE JSON line on rank 0.
`--dump-outputs DIR` writes what the last timed step returned (picks, scores, keypoints; a seeded sample of rows
where an array is large) as .npy files: the inputs are fixed by the arguments, so two builds can be compared.
"""
from __future__ import annotations

import argparse
import dataclasses
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import warnings

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "unlabeled frames scored+selected/sec per AL query"
UNIT = "frames/s"
D = 2048
FRAME_BYTES = 17 * 64 * 48 * 4
LAM = 0.01
CONFIG_FRAMES = {1: 256, 2: 10000, 3: 100000, 4: 170000, 5: 1000000}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--config", type=int, default=5, choices=[1, 2, 3, 4, 5], help="BASELINE.json configs[config-1]")
    p.add_argument("--frames", type=int, default=None, help="pool size (whole job); default: the config's")
    p.add_argument("--query-frac", type=float, default=0.05)
    p.add_argument("--labeled-frac", type=float, default=0.0, help="already-labelled fraction (0 = round 0)")
    p.add_argument("--moks", type=float, default=None, help="mean OKS of the last queries (default 0 at round 0, else 0.6)")
    p.add_argument("--feat-kind", default="clustered", choices=["clustered", "weak", "iid"],
                   help="feature pool: 30-frame clusters at 30:1 separation (SURVEY recipe), 3:1, or i.i.d. rows")
    p.add_argument("--batch", type=int, default=None,
                   help="core-set picks per round (1 = GEMV form, 8 = one pass per round, 16 = two passes per round); default 16")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-prune", action="store_true", help="core-set passes stream every tile (exact pruning off)")
    p.add_argument("--no-p2p", action="store_true", help="multi-GPU: ncclAllGather per round instead of the peer-memory mailbox")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-controls", action="store_true", help="skip the data-dependence control queries (roofline.controls)")
    p.add_argument("--cpu-frames", type=int, default=4096, help="frames of the CPU scoring sample")
    p.add_argument("--cpu-greedy-steps", type=int, default=20, help="greedy steps of the CPU core-set sample")
    p.add_argument("--cpu-rows", type=int, default=200000, help="rows of the CPU core-set sample (cost per step is linear in rows)")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write what the last timed step computed as DIR/<name>.npy (rank 0; at most 64 MB in all)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        p.error("--dump-outputs needs --impl ours")
    return a


def sha_picks(picks) -> str:
    return hashlib.sha256(np.asarray(picks, dtype="<i8").tobytes()).hexdigest()


DUMP_BYTES = 64 << 20


def result_arrays(res) -> dict:
    """The arrays and numbers a caller receives in a result dataclass (run statistics left out)."""
    return {f.name: getattr(res, f.name) for f in dataclasses.fields(res) if f.name not in ("stats", "extra")}


def dump_outputs(out_dir: str, outputs: dict):
    """Write each output as out_dir/<name>.npy: float32 stays float32, everything else becomes float64 (which holds
    the integer indices exactly).  Every output gets an equal share of the 64 MB; one larger than its share is
    replaced by a fixed sample of its rows (seed 0, ascending), whose indices go to <name>_rows.npy, so that two
    builds run with the same arguments dump the same elements."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    arrays = {}
    for name, v in outputs.items():
        if v is None:
            continue
        t = v.detach() if isinstance(v, torch.Tensor) else torch.as_tensor(np.asarray(v))
        arrays[name] = t.reshape(1) if t.dim() == 0 else t
    share = DUMP_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        t = t if t.dtype in (torch.float32, torch.float64) else t.to(torch.float64)
        row_bytes = t.numel() // max(1, t.shape[0]) * t.element_size()
        if t.shape[0] * row_bytes > share:
            m = share // (row_bytes + 8)
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], m, replace=False))
            t = t.index_select(0, torch.from_numpy(rows).to(t.device))
            np.save(os.path.join(out_dir, f"{name}_rows.npy"), rows.astype(np.float64))
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """SM clock and clock-event (throttle) reasons sampled DURING the timed region: through NVML
    (nvidia_ml_py, one sample every 20 ms) when it loads, else `nvidia-smi` every 200 ms (the recipe's
    clocks line; one call takes longer than a short timed region, hence NVML first)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None
        self.source = "nvidia-smi"
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._max = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
            self._nvml = pynvml
            self.source = "nvml"
        except Exception:
            self._nvml = None

    def _run_nvml(self):
        nv = self._nvml
        masks = [nv.nvmlClocksEventReasonHwSlowdown, nv.nvmlClocksEventReasonHwThermalSlowdown,
                 nv.nvmlClocksEventReasonSwThermalSlowdown, nv.nvmlClocksEventReasonSwPowerCap]
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                self.rows.append([str(sm), str(self._max)] + ["Active" if r & m else "Not Active" for m in masks])
            except Exception:
                pass
            self._stop.wait(0.02)

    def _run_smi(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.rows.append(f)
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run_nvml if self._nvml else self._run_smi, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"], "source": self.source}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        reasons = [nm for k, nm in enumerate(self.NAMES) if any(r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.rows), "source": self.source}


# ------------------------------------------------------------------------------------ CPU arm
def blas_threads():
    try:
        from threadpoolctl import threadpool_info
        return max([int(t.get("num_threads", 1)) for t in threadpool_info() if t.get("user_api") == "blas"] or [1])
    except Exception:
        return None


def cpu_reference_arm(config: int, n_pool: int, k: int, moks: float, cpu_frames: int, greedy_steps: int, cpu_rows: int,
                      seed: int = 0):
    """Time the oracle port of the reference's CPU path on a bounded sample of the workload and
    extrapolate to the whole query:  t = n/fps_scoring + k * t_greedy_step  (cost per greedy step is
    constant in the step index and linear in the rows; BASELINE.md §3).  Returns (frames_per_s, detail)."""
    import torch
    from oracle import vatl_oracle as O
    import vatlq
    synth = vatlq.synth
    cores = os.cpu_count() or 1
    det = {"cores": cores, "torch_threads": torch.get_num_threads(), "blas_threads": blas_threads()}
    parts = []
    t_query = 0.0
    if config in (1, 2, 4, 5):
        m = min(cpu_frames, n_pool)
        ids, ip, inx = synth.track_flags(m, np.random.default_rng(seed), 30.0)
        ae = O.make_autoencoder(synth.ae_weights(42, 4))
        want = {1: ("coords", "thc", "peak"), 2: ("wpu",)}.get(config, ("coords", "thc", "wpu", "peak"))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            if config == 2:      # WPU on given poses (compute_hybrid + WholeBodyAE + MSE per pose)
                kp, bb = synth.poses(m, seed=1)
                kl = kp.reshape(m, 51).astype(np.float64)
                for i in range(8):
                    O.wpu_item(ae, bb[i].tolist(), kl[i], True)
                t0 = time.perf_counter()
                for i in range(m):
                    O.wpu_item(ae, bb[i].tolist(), kl[i], True)
                t_score = time.perf_counter() - t0
            else:
                H = synth.heatmaps(m, seed=seed, track_ids=ids)
                boxes = synth.boxes_xyxy(m, seed)
                O.score_pool(H[:8], boxes[:8], ip[:8], inx[:8], ae, want=want)            # warm-up
                t0 = time.perf_counter()
                O.score_pool(H, boxes, ip, inx, ae, want=want)
                t_score = time.perf_counter() - t0
        det["scoring_frames_per_s"] = m / t_score
        t_query += n_pool / det["scoring_frames_per_s"]
        parts.append(f"scoring loop on {m} frames")
    if config in (3, 4, 5):
        rows = min(cpu_rows, n_pool)
        X = synth.embeddings(rows, d=D, seed=2).astype(np.float64)          # float64 features like ActiveLearning.py:270
        unc = np.random.default_rng(3).uniform(0, 1, rows)
        O.coreset_select(X, unc.copy(), [], 1, moks, LAM)                  # warm-up (BLAS threads, page faults)
        t0 = time.perf_counter()
        O.coreset_select(X, unc.copy(), [], greedy_steps, moks, LAM)
        t_step = (time.perf_counter() - t0) / greedy_steps * (n_pool / rows)
        det["greedy_step_s"] = t_step
        t_query += k * t_step
        parts.append(f"first {greedy_steps} greedy steps on {rows} rows" +
                     (f" scaled x{n_pool / rows:.2f} to N={n_pool} (cost per step is linear in rows)" if rows < n_pool else ""))
    det["extrapolated_query_s"] = t_query
    det["sample"] = " + ".join(parts) + f", extrapolated linearly to the whole query (t = N/fps + k*t_step, k={k})"
    return n_pool / t_query, det


def ncu_traffic(kernel: str, rows: int):
    """dram__bytes_read+write per launch of `kernel` from the committed ncu captures (profiles/ncu_traffic.json),
    valid only for the shape it was captured at (an entry is quoted when its `rows` equals this rank's); else None."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[kernel]
        for e in (t if isinstance(t, list) else [t]):
            if int(e["rows"]) == int(rows):
                return e["bytes_per_launch"]
    except Exception:
        pass
    return None


def golden_for(config: int, n: int, lab_frac: float, moks: float, kind: str):
    """The reference's pick list for this configuration, if oracle/pin_scale.py pinned one."""
    tags = {3: ["c3", "c3lab"], 4: ["c4", "c4lab"], 5: ["c5"]}.get(config, [])
    for tag in tags:
        f = os.path.join(ROOT, "tests", "golden", f"coreset_scale_{tag}.npz")
        if not os.path.exists(f):
            continue
        z = np.load(f)
        if (int(z["n"]) == n and abs(float(z["labeled_frac"]) - lab_frac) < 1e-12 and abs(float(z["moks"]) - moks) < 1e-12
                and str(z["kind"]) == kind):
            return tag, z["picks"].astype(np.int64), int(z["k_full"])
    return None, None, None


def check_golden(config, n, k, lab_frac, moks, kind, picks):
    tag, gold, k_full = golden_for(config, n, lab_frac, moks, kind)
    if tag is None:
        return {"pinned": False, "note": "no reference pick list is committed for this configuration"}
    m = min(len(gold), len(picks))
    ok = bool(k == k_full and m > 0 and np.array_equal(np.asarray(picks[:m]), gold[:m]))
    first_diff = None if ok or m == 0 else int(np.argmax(np.asarray(picks[:m]) != gold[:m]))
    return {"pinned": True, "golden": f"tests/golden/coreset_scale_{tag}.npz", "reference_picks_compared": int(m),
            "whole_list": bool(m == k), "ok": ok, "first_difference_at": first_diff,
            "source": "the reference's ActiveLearning.coreset_selection run on this pool (oracle/pin_scale.py)"}


def peak_hbm():
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        if "hbm_gbs" in peaks:
            return float(peaks["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------ main
def main():
    a = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if a.batch is None:
        a.batch = 16    # 16 picks per round: one paired pass (two CTAs per tile, 8 centres each) per read of X
    n = a.frames if a.frames is not None else CONFIG_FRAMES[a.config]
    n_lab = int(n * a.labeled_frac)
    k = int(n * (a.labeled_frac + a.query_frac)) - n_lab
    moks = a.moks if a.moks is not None else (0.0 if n_lab == 0 else 0.6)
    what = {1: "THC + local-peak + coordinates (heat-map scan)", 2: "WPU (hybrid feature + auto-encoder + MSE)",
            3: "core-set selection", 4: "full THC+WPU+core-set query", 5: "full THC+WPU+core-set query"}[a.config]
    workload = f"config {a.config}: {what}, {n} frames"
    if a.config in (1, 4, 5):
        workload += " x 17 x 64x48 fp32 heat maps"
    if a.config >= 3:
        workload += f" + {D}-d features ({a.feat_kind}), select {k} ({a.query_frac:.0%}), labelled {n_lab}, moks {moks}"
    config = {"workload": workload, "baseline_config": a.config, "frames": n, "parallelism": f"frame-range sharding x{world}",
              "pool": "one global counter-based pool sliced per rank (same pool and same picks at every N)"}
    if a.config >= 3:
        config.update({"k": k, "feat_dim": D, "feat_kind": a.feat_kind, "labelled": n_lab, "moks": moks, "unc_lambda": LAM,
                       "coreset_batch": a.batch,
                       "candidate_exchange": "none" if world == 1 else ("ncclAllGather" if a.no_p2p else "peer-memory mailbox (NVLink stores + flags)"),
                       "coreset_pruning": "off" if a.no_prune else "exact (segments of consecutive rows + triangle inequality; picks unchanged)"})
    config["arithmetic"] = ("heat-map scores in f32 (THC, peaks, coordinates, WPU MLP), hybrid feature / fusion / distances / selection in f64 "
                            "(fp64 tensor-core DMMA over the fp32 features); TF32 tcgen05 only as an error-bounded pre-selection")
    config["l2"] = ("inputs (heat maps >= 26 GB and features >= 1 GB per rank) exceed the 126 MB L2" if a.config >= 4 else
                    ("features (819 MB) exceed the 126 MB L2" if a.config == 3 else
                     "L2 flushed between timed iterations (a 256 MB buffer is rewritten)"))

    if a.impl == "reference":
        if rank != 0:
            return
        import torch  # noqa: F401
        vals, det = [], None
        for _ in range(a.steps):
            v, det = cpu_reference_arm(a.config, n, k, moks, a.cpu_frames, a.cpu_greedy_steps, a.cpu_rows)
            vals.append(v)
        v = statistics.median(vals)
        cb = {"value": v, "unit": UNIT, "cores": det["cores"], "kind": "port", "sample": det["sample"],
              "blas_threads": det["blas_threads"], "torch_threads": det["torch_threads"]}
        for key in ("scoring_frames_per_s", "greedy_step_s"):
            if key in det:
                cb[key] = det[key]
        line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": 1e3 * n / v, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "note": "oracle port of the reference's CPU path (the reference is Python; /root/reference is absent on the GPU box)"}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as td
    import vatlq

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        td.init_process_group("nccl", device_id=dev)
    assert world == a.gpus or world == 1, "launch with torchrun --nproc-per-node N for --gpus N"
    if a.config <= 3:
        line, rc = small_config(a, n, k, moks, config, rank, world, dev)
    else:
        line, rc = full_query(a, n, n_lab, k, moks, config, rank, world, local, dev)
    if rank == 0:
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        td.barrier()
        td.destroy_process_group()
    if rc:
        sys.exit(rc)


def cpu_baseline_entry(a, n, k, moks):
    try:
        v, det = cpu_reference_arm(a.config, n, k, moks, a.cpu_frames, a.cpu_greedy_steps, a.cpu_rows)
        cb = {"value": v, "unit": UNIT, "cores": det["cores"], "kind": "port", "sample": det["sample"],
              "blas_threads": det["blas_threads"], "torch_threads": det["torch_threads"]}
        for key in ("scoring_frames_per_s", "greedy_step_s"):
            if key in det:
                cb[key] = det[key]
        return cb
    except Exception as exc:
        return {"value": None, "error": repr(exc)[:300]}


def pass_roofline(lib, nl, streamed_frac, steps, ms_step, prune, no_prune, dmma_peak_fma):
    """roofline of the dominant kernel (the core-set pass over X) from the library's per-launch CUDA-event timing.
    A pass streams `streamed_frac` of the owned rows once and multiplies every streamed 8-row tile with the launch's
    centres on the fp64 tensor cores (DMMA): both the HBM and the fp64-tensor fraction are reported, `bound` names the
    resource that is closer to its measured peak."""
    import ctypes as C
    tot_ms, n_pass, n_picks = C.c_double(), C.c_int64(), C.c_int64()
    lib.vatlq_profile_read(C.byref(tot_ms), C.byref(n_pass), C.byref(n_picks), 1)
    if not (n_pass.value > 0 and tot_ms.value > 0):
        return None
    peak_gbs, peak_src = peak_hbm()
    per_step_bytes = nl * D * 4 + 16 * nl            # SURVEY.md §8d: one greedy step over the owned rows
    # what ONE pass must move: the rows of X it streams (all of them without pruning; the pruned tiles are
    # provably unaffected and never read) + xx r, min_d r/w, unc r/w, score w (fp64 each)  (DESIGN.md §4.4)
    per_pass_bytes = nl * D * 4 * streamed_frac + 40 * nl
    picks_per_launch = n_picks.value / n_pass.value
    avg_s = tot_ms.value / n_pass.value * 1e-3
    gbs = per_pass_bytes / avg_s / 1e9
    fma = nl * streamed_frac * D * picks_per_launch / avg_s          # algorithmic fp64 FMAs (padding centres not counted)
    hbm = {"achieved": gbs, "peak": peak_gbs, "unit": "GB/s", "frac": gbs / peak_gbs, "peak_source": peak_src}
    tens = {"achieved": 2 * fma / 1e12, "peak": 2 * dmma_peak_fma / 1e12, "unit": "TFLOP/s (fp64, mma.sync.m8n8k4 DMMA)",
            "frac": fma / dmma_peak_fma if dmma_peak_fma else None,
            "peak_source": "measured live by vatlq_measure_fp64_mma (saturating DMMA kernel; MEASURED_PEAKS.json has no fp64 figure)"}
    use_t = tens["frac"] is not None and tens["frac"] > hbm["frac"]
    top = tens if use_t else hbm
    return {"kernel": "pass_kernel_tma (core-set distance update: TMA-staged tiles, fp64 tensor-core DMMA, row finishing; "
                      "paired form: 16 centres per read of X by a cluster of two CTAs)",
            "bound": "tensor" if use_t else "hbm", "achieved": top["achieved"], "peak": top["peak"],
            "unit": "TFLOP/s" if use_t else "GB/s", "frac": top["frac"],
            "traffic": ncu_traffic("pass_kernel" if no_prune else "pass_kernel_pruned", nl),
            "peak_source": top["peak_source"], "hbm": hbm, "fp64_tensor": tens,
            "avg_launch_us": avg_s * 1e6, "launches_timed": n_pass.value,
            "algorithmic_bytes_per_launch": per_pass_bytes, "streamed_fraction_of_X": streamed_frac,
            "unpruned_bytes_per_launch": nl * D * 4 + 40 * nl, "segments": prune["segments"],
            "greedy_steps_per_launch": picks_per_launch, "algorithmic_bytes_per_greedy_step": per_step_bytes,
            "greedy_equivalent_gbs": picks_per_launch * per_step_bytes / avg_s / 1e9,
            "share_of_step": tot_ms.value / steps / ms_step,
            "note": "a launch applies greedy_steps_per_launch greedy steps for ONE read of the rows it streams (exact batching; "
                    "the exact triangle filter skips the other rows): hbm charges those bytes once, fp64_tensor counts the "
                    "8-row x centre x 2048 FMAs of the streamed tiles; greedy_equivalent_gbs is SURVEY 8d's per-step bytes x steps / time"}


def run_controls(a, n, dev):
    """Data-dependence controls (single GPU, core-set only, one query each on a pool of <= 170 000 rows): the
    headline pool's 30:1 cluster separation is what lets the exact triangle filter skip tiles, so the same
    selection is also timed with pruning off, on a 3:1 pool, on i.i.d. rows and in a later AL round."""
    import torch
    import vatlq
    from vatlq import ops, synth
    nc = min(n, 170000)
    kc = int(nc * a.query_frac)
    out = {"pool_rows": nc, "k": kc, "what": "core-set selection only (ops.coreset_select), one query each"}
    cases = [("clustered_30to1", "clustered", 0.0, 0.0, False), ("no_prune", "clustered", 0.0, 0.0, True),
             ("weak_3to1", "weak", 0.0, 0.0, False), ("iid", "iid", 0.0, 0.0, False),
             ("labelled10_moks0.6", "clustered", 0.1, 0.6, False)]
    X = None
    last_kind = None
    for tag, kind, labf, mk, noprune in cases:
        try:
            if kind != last_kind:
                X = None
                X = synth.pool_embeddings(nc, d=D, seed=2, kind=kind, device=dev)
                last_kind = kind
            lab = synth.pool_labeled(nc, int(nc * labf))
            unc = synth.pool_unc(nc, device=dev)
            if lab.size:
                unc[torch.from_numpy(lab).to(dev)] = 0.0
            kk = int(nc * (labf + a.query_frac)) - lab.size
            ops.set_prune("off" if noprune else "env")
            ops.prune_stats(reset=True)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            picks, st = ops.coreset_select(X, unc, lab, kk, mk, LAM, batch=a.batch)
            e1.record()
            torch.cuda.synchronize()
            pr = ops.prune_stats(reset=True)
            out[tag] = {"ms": e0.elapsed_time(e1), "frames_per_s": nc / (e0.elapsed_time(e1) * 1e-3),
                        "streamed_fraction": pr["streamed"] / pr["tiles"] if pr["tiles"] else 1.0,
                        "passes": st.passes, "rounds": st.rounds, "picks": st.picks, "labelled": int(lab.size), "moks": mk,
                        "picks_sha256": sha_picks(picks.cpu().numpy())}
        except Exception as exc:
            out[tag] = {"error": repr(exc)[:200]}
        finally:
            ops.set_prune("env")
    return out


def full_query(a, n, n_lab, k, moks, config, rank, world, local, dev):
    import ctypes as C
    import torch
    import torch.distributed as td
    import vatlq
    from vatlq import dist as vd, ops, synth

    lo, hi = vd.shard_range(n, rank, world)
    nl = hi - lo
    segs, bb, ip, inx, Xl, distinct = synth.rank_pool(n, lo, hi, dev, a.feat_kind)
    config["heat_maps"] = (f"{nl} items per rank backed by {distinct} distinct resident frames"
                           + (f" (content period {synth.HEAT_RING} items: {n} x 208 896 B exceeds one GPU's HBM; "
                              "every item is scanned from HBM)" if n > synth.HEAT_RING else ""))
    W = synth.ae_weights(42, 4)
    labeled = synth.pool_labeled(n, n_lab).tolist()
    comm = vd.Comm(use_p2p=not a.no_p2p) if world > 1 else None
    lib = vatlq._lib.lib()
    lib.vatlq_profile_passes(1)
    if a.no_prune:
        ops.set_prune("off")

    def step_resident():
        if world == 1:
            return vatlq.run_query(segs, bb, ip, inx, Xl, W, labeled, k, moks, LAM, batch=a.batch, device=dev)
        return vd.distributed_query(segs, bb, ip, inx, Xl, W, labeled, n, k, moks, LAM, batch=a.batch, comm=comm)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            td.barrier()
            torch.cuda.synchronize()

    for _ in range(a.warmup):
        res = step_resident()
    barrier()
    lib.vatlq_profile_read(None, None, None, 1)
    ops.prune_stats(reset=True)
    launches0 = vatlq._lib.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        barrier()
        ev0.record()
        for _ in range(a.steps):
            res = step_resident()
        ev1.record()
        barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
    if world > 1:
        td.all_reduce(ms, op=td.ReduceOp.MAX)
    ms_step = float(ms.item()) / a.steps
    launches = vatlq._lib.launch_count() - launches0
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, result_arrays(res))
    prune = ops.prune_stats(reset=True)
    streamed_frac = prune["streamed"] / prune["tiles"] if prune["tiles"] else 1.0
    dmma_peak = ops.measure_fp64_mma(dev)
    roof = pass_roofline(lib, nl, streamed_frac, a.steps, ms_step, prune, a.no_prune, dmma_peak)
    lib.vatlq_profile_passes(0)
    st = res.stats
    picks_ref = res.picks.clone()
    picks_host = picks_ref.cpu().numpy()
    peak_gbs, _ = peak_hbm()

    # every rank must hold the same list (each replays the same plan); compare hashes across ranks
    digest = sha_picks(picks_host)
    same_all = True
    if world > 1:
        hs = [None] * world
        td.all_gather_object(hs, digest)
        same_all = len(set(hs)) == 1
    parity = check_golden(a.config, n, k, a.labeled_frac, moks, a.feat_kind, picks_host)
    parity["all_ranks_equal"] = same_all

    # ---- the same kernel with pruning off (one extra query, not part of `value`)
    if roof is not None and not a.no_prune and world == 1:
        unpruned = None
        try:
            ops.set_prune("off")
            lib.vatlq_profile_passes(1)
            lib.vatlq_profile_read(None, None, None, 1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            r2 = step_resident()
            e1.record()
            torch.cuda.synchronize()
            t2, n2, p2 = C.c_double(), C.c_int64(), C.c_int64()
            lib.vatlq_profile_read(C.byref(t2), C.byref(n2), C.byref(p2), 1)
            if n2.value > 0 and t2.value > 0:
                full = nl * D * 4 + 40 * nl
                s2 = t2.value / n2.value * 1e-3
                fma2 = nl * D * (p2.value / n2.value) / s2
                unpruned = {"hbm_gbs": full / s2 / 1e9, "hbm_frac": full / s2 / 1e9 / peak_gbs,
                            "fp64_tensor_tflops": 2 * fma2 / 1e12, "fp64_tensor_frac": fma2 / dmma_peak if dmma_peak else None,
                            "avg_launch_us": s2 * 1e6,
                            "launches_timed": n2.value, "algorithmic_bytes_per_launch": full,
                            "traffic": ncu_traffic("pass_kernel", nl), "query_ms": e0.elapsed_time(e1),
                            "picks_equal_pruned_run": bool(torch.equal(r2.picks, picks_ref))}
        except Exception as exc:  # report, never hide; the headline numbers above are unaffected
            unpruned = {"error": repr(exc)[:200]}
        finally:
            try:
                lib.vatlq_profile_passes(0)
                ops.set_prune("env")
                ops.prune_stats(reset=True)
            except Exception:
                pass
        roof["unpruned_pass"] = unpruned
        roof["note"] += ("; with exact pruning a launch streams only streamed_fraction_of_X of the rows, so its fixed "
                         "costs weigh more: unpruned_pass is the same kernel timed in one extra query with pruning off")

    # ---- the streaming kernel: heat-map scan, timed alone on this rank's items
    def scan_all():
        for pos, seg in segs:
            e = pos + seg.shape[0]
            ops.heatmap_scan(seg, ip[pos:e], inx[pos:e], bb[pos:e])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scan_all()
    reps = 3
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        scan_all()
    e1.record()
    torch.cuda.synchronize()
    scan_s = e0.elapsed_time(e1) / reps * 1e-3
    scan_roof = {"kernel": "heat-map scan (THC + local peaks + argmax) + scan_finalize", "bound": "hbm",
                 "achieved": nl * FRAME_BYTES / scan_s / 1e9,
                 "peak": peak_gbs, "unit": "GB/s", "frac": nl * FRAME_BYTES / scan_s / 1e9 / peak_gbs,
                 "traffic": ncu_traffic("scan", nl),
                 "algorithmic_bytes_per_frame": FRAME_BYTES, "frames": nl, "ms": scan_s * 1e3,
                 "share_of_step": scan_s * 1e3 / ms_step}

    # ---- end to end: pool in pinned host memory, copies inside the timed region
    e2e = None
    if not a.no_e2e:
        try:
            e2e = run_e2e(a, segs, ip, inx, bb, Xl, W, labeled, n, nl, k, moks, world, comm, dev, picks_ref)
        except Exception as exc:  # report, never hide
            e2e = {"value": None, "unit": UNIT, "error": repr(exc)[:300]}

    controls = None
    if world == 1 and not a.no_controls and roof is not None:
        segs.clear()          # (the heat maps are no longer needed: leave the memory to the control pools)
        del Xl
        torch.cuda.empty_cache()
        controls = run_controls(a, n, dev)
        roof["controls"] = controls

    line = None
    rc = 0
    if rank == 0:
        line = {"metric": METRIC, "value": n / (ms_step * 1e-3), "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config, "clocks": clk.summary(), "gpu_launches": int(launches),
                "picks_sha256": digest, "parity": parity,
                "roofline": roof, "roofline_scan": scan_roof, "e2e": e2e,
                "coreset": {"passes_over_X": st.passes, "picks": st.picks, "rounds": st.rounds,
                            "fallback_rounds": st.fallback_empty + st.fallback_overflow,
                            "mean_candidates": st.candidates / max(1, st.rounds - st.fallback_empty - st.fallback_overflow),
                            "ms_per_round": (ms_step - scan_s * 1e3) / max(1, st.rounds),
                            "us_per_round": {"waiting_for_peer_blocks": st.ns_wait / 1e3 / max(1, st.rounds),
                                             "candidate_tiles": st.ns_tiles / 1e3 / max(1, st.rounds),
                                             "planner": st.ns_plan / 1e3 / max(1, st.rounds)}}}
        if world == 1 and not a.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline_entry(a, n, k, moks)
    if not same_all or (parity.get("pinned") and not parity.get("ok")):
        rc = 3
    if comm is not None:
        comm.close()
    return line, rc


def run_e2e(a, segs, ip, inx, bb, Xl, W, labeled, n, nl, k, moks, world, comm, dev, picks_ref):
    """The same query through the public API with HOST inputs: every step streams this rank's heat maps
    from pinned host memory through a ring of three device staging buffers (copy stream overlapped with the
    scan), copies boxes, flags and features, and reads the picks back."""
    import torch
    import torch.distributed as td
    from vatlq import dist as vd, ops
    from vatlq.query import QueryPass
    chunk = 4096
    frame_elems = 17 * 64 * 48
    # host budget: all ranks of the box together pin at most ~40 % of the available host memory
    try:
        avail = [int(l.split()[1]) * 1024 for l in open("/proc/meminfo") if l.startswith("MemAvailable")][0]
    except Exception:
        avail = 64 << 30
    if os.environ.get("VATLQ_BENCH_HOST_GB"):          # (tests of the reduced-ring path)
        avail = int(float(os.environ["VATLQ_BENCH_HOST_GB"]) * (1 << 30) / 0.4) * max(1, world)
    budget_frames = max(chunk, int(0.4 * avail / max(1, world) / FRAME_BYTES) // chunk * chunk)
    # pinned host copies of the distinct heat-map buffers (segments that view one ring share one host copy)
    uniq = {}
    for _, seg in segs:
        uniq.setdefault(seg.untyped_storage().data_ptr(), seg)
    need_frames = sum(torch.empty(0, dtype=sg.dtype, device=dev).set_(sg.untyped_storage()).numel() // frame_elems for sg in uniq.values())
    exact = need_frames <= budget_frames
    hsegs = []
    if exact:
        host = {}
        for base, seg in uniq.items():
            full = torch.empty(0, dtype=seg.dtype, device=dev).set_(seg.untyped_storage())
            hb = torch.empty(full.shape, dtype=seg.dtype, pin_memory=True)
            step = chunk * frame_elems
            for s in range(0, full.numel(), step):
                hb[s:s + step].copy_(full[s:s + step])
            host[base] = hb
        torch.cuda.synchronize()
        for pos, seg in segs:
            hb = host[seg.untyped_storage().data_ptr()]
            off = seg.storage_offset()
            hsegs.append((pos, hb[off:off + seg.numel()].view(seg.shape)))
    else:
        # the rank's distinct frames do not fit the host budget: a pinned ring of budget_frames frames is cycled
        # (same bytes per step over PCIe; the scores then differ from the resident run, so the pick check is skipped)
        first = segs[0][1]
        R = min(budget_frames, first.shape[0] // chunk * chunk) or min(budget_frames, first.shape[0])
        ring = torch.empty((R,) + tuple(first.shape[1:]), dtype=first.dtype, pin_memory=True)
        for s in range(0, R, chunk):
            ring[s:s + chunk].copy_(first[s:s + chunk])
        torch.cuda.synchronize()
        for pos, seg in segs:
            m = seg.shape[0]
            for s in range(0, m, R):
                hsegs.append((pos + s, ring[:min(R, m - s)]))
    Xh = torch.empty(Xl.shape, dtype=Xl.dtype, pin_memory=True); Xh.copy_(Xl)
    bbh, iph, inxh = bb.cpu().pin_memory(), ip.cpu().pin_memory(), inx.cpu().pin_memory()
    torch.cuda.synchronize()
    nbuf = 3
    stage = [torch.empty((chunk, 17, 64, 48), dtype=torch.float32, device=dev) for _ in range(nbuf)]
    Xd = torch.empty_like(Xl)
    copy_stream = torch.cuda.Stream(device=dev)
    lab = np.asarray(labeled, dtype=np.int64)
    rank = td.get_rank() if world > 1 else 0
    lo, hi = vd.shard_range(n, rank, world)
    pieces = [(pos + s, hs[s:s + chunk]) for pos, hs in hsegs for s in range(0, hs.shape[0], chunk)]

    def step():
        main = torch.cuda.current_stream()
        filled = [None] * len(pieces)
        freed = [None] * nbuf
        qp = QueryPass(nl, dev, ae_weights=W, uncertainty="THC+WPU")
        with torch.cuda.stream(copy_stream):
            bd = bbh.to(dev, non_blocking=True); ipd = iph.to(dev, non_blocking=True); ind = inxh.to(dev, non_blocking=True)
        hp = hn = None
        if world > 1:   # the frames next to the range come from the neighbours' host buffers via their GPUs
            f0 = pieces[0][1][0].to(dev, non_blocking=True)
            f1 = pieces[-1][1][-1].to(dev, non_blocking=True)
            hp, hn = vd.exchange_halo(f0, f1, rank, world)

        def issue(i):
            b = i % nbuf
            with torch.cuda.stream(copy_stream):
                if freed[b] is not None:
                    copy_stream.wait_event(freed[b])
                m = pieces[i][1].shape[0]
                stage[b][:m].copy_(pieces[i][1], non_blocking=True)
                e = torch.cuda.Event(); e.record(copy_stream); filled[i] = e

        for i in range(min(nbuf, len(pieces))):
            issue(i)
        for i, (pos, hs) in enumerate(pieces):
            b = i % nbuf
            m = hs.shape[0]
            main.wait_event(filled[i])
            qp.score_chunk(pos, stage[b][:m], bd[pos:pos + m], ipd[pos:pos + m], ind[pos:pos + m],
                           halo_prev=hp if pos == 0 else None, halo_next=hn if pos + m == nl else None)
            e = torch.cuda.Event(); e.record(main); freed[b] = e
            if i + nbuf < len(pieces):
                issue(i + nbuf)
        with torch.cuda.stream(copy_stream):
            Xd.copy_(Xh, non_blocking=True)
            ex = torch.cuda.Event(); ex.record(copy_stream)
        unl = torch.ones(nl, dtype=torch.uint8, device=dev)
        mine = lab[(lab >= lo) & (lab < hi)] - lo
        if mine.size:
            unl[torch.from_numpy(mine).to(dev)] = 0
        unc_l = qp.fuse(unl, "const", labeled_ratio=lab.size / n, group=None if world == 1 else td.group.WORLD,
                        n_unlabeled_global=n - lab.size)
        main.wait_event(ex)
        X = vd.allgather_rows(Xd, n, world) if world > 1 else Xd
        unc = vd.allgather_rows(unc_l, n, world) if world > 1 else unc_l
        picks, _ = ops.coreset_select(X, unc, lab, k, moks, LAM, batch=a.batch,
                                      comm=comm.handle if comm is not None else None,
                                      row_range=(lo, hi) if world > 1 else None)
        return picks.cpu()      # D2H read of the result

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            td.barrier()
            torch.cuda.synchronize()

    p = step()
    same = bool(torch.equal(p, picks_ref.cpu())) if exact else None
    reps = max(1, min(a.steps, 3))
    sync()
    t0 = time.perf_counter()
    for _ in range(reps):
        p = step()
    sync()
    dt = torch.tensor([(time.perf_counter() - t0) / reps], dtype=torch.float64, device=dev)
    if world > 1:
        td.all_reduce(dt, op=td.ReduceOp.MAX)
    h2d = nl * FRAME_BYTES + nl * (16 + 2) + nl * D * 4
    return {"value": n / float(dt.item()), "unit": UNIT, "ms_per_step": float(dt.item()) * 1e3,
            "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(k * 8), "steps": reps,
            "h2d_gbs": h2d / float(dt.item()) / 1e9,
            "picks_equal_resident_run": same, "host_frames_exact": exact,
            "api": "vatlq.QueryPass.score_chunk + fuse + ops.coreset_select (host pinned inputs streamed through "
                   "3 staging buffers, per rank)"}


# ------------------------------------------------------------------------------------ configs 1-3
def small_config(a, n, k, moks, config, rank, world, dev):
    """BASELINE configs 1-3 (single stage each), one GPU: resident `value`, host-buffer `e2e`, roofline of the
    stage's kernel, the CPU port beside it.  The L2 is flushed between timed iterations where the input fits it."""
    import ctypes as C
    import torch
    import vatlq
    from vatlq import ops, synth
    assert world == 1, "configs 1-3 are single-GPU cases (BASELINE.json)"
    lib = vatlq._lib.lib()
    peak_gbs, peak_src = peak_hbm()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    parity = None
    digest = None
    extra = {}
    if a.config == 1:
        tid, pos, ipn, inxn = synth.pool_tracks(n, seed=0)
        H = synth.pool_heatmaps(tid, pos, 0, n, seed=0, device=dev)
        bb = synth.pool_boxes(n, seed=0, device=dev)
        ip, inx = torch.from_numpy(ipn).to(dev), torch.from_numpy(inxn).to(dev)
        run = lambda: ops.heatmap_scan(H, ip, inx, bb)
        hH, hb = H.cpu().pin_memory(), bb.cpu().pin_memory()

        def run_host():
            r = ops.heatmap_scan(hH.to(dev, non_blocking=True), ip, inx, hb.to(dev, non_blocking=True))
            return r.thc.cpu(), r.peak_mean.cpu(), r.kpts.cpu()
        h2d, d2h = n * FRAME_BYTES + n * 16, n * (4 + 4 + 17 * 12)
        alg_bytes = n * FRAME_BYTES
        kernel = "scan_tma_64x48 + scan_finalize (THC + local peaks + argmax, one read of the heat maps)"
        bound_note = "256 frames = 53 MB: about 8 us of HBM time, the launch floor dominates"
    elif a.config == 2:
        kp, bx = synth.poses(n, seed=1)
        kpd, bxd = torch.from_numpy(kp).to(dev), torch.from_numpy(bx).to(dev)
        w, ind, z = ops.pack_ae_weights(synth.ae_weights(42, 4), dev)
        run = lambda: ops.wpu(kpd, bxd, w, ind, z, drop_ears=True, check_status=False)
        hk, hb = torch.from_numpy(kp).pin_memory(), torch.from_numpy(bx).pin_memory()
        run_host = lambda: ops.wpu(hk.to(dev, non_blocking=True), hb.to(dev, non_blocking=True), w, ind, z, drop_ears=True).cpu()
        h2d, d2h = n * 55 * 4, n * 4
        alg_bytes = n * 224
        kernel = "wpu_kernel (fp64 hybrid feature, 8 fused Linear layers in fp32 FMA, sigmoid, MSE)"
        bound_note = ("10 000 poses = 2.2 MB and 56 MFLOP: launch-latency-bound; the FP32 pipe, not HBM and not the tensor pipe, "
                      "is the relevant unit (layer widths 42-24-12-7-4 are below one MMA tile, 1e-5 rules out single-pass TF32)")
        extra["flops_per_pose"] = 5248
    else:
        X = synth.pool_embeddings(n, d=D, seed=2, kind=a.feat_kind, device=dev)
        lab = synth.pool_labeled(n, int(n * a.labeled_frac))
        unc = synth.pool_unc(n, device=dev)
        if lab.size:
            unc[torch.from_numpy(lab).to(dev)] = 0.0
        if a.no_prune:
            ops.set_prune("off")
        lib.vatlq_profile_passes(1)
        state = {}

        def run():
            state["picks"], state["st"] = ops.coreset_select(X, unc, lab, k, moks, LAM, batch=a.batch)
            return state["picks"]
        hX, hu = X.cpu().pin_memory(), unc.cpu().pin_memory()
        run_host = lambda: ops.coreset_select(hX.to(dev, non_blocking=True), hu.to(dev, non_blocking=True), lab, k, moks, LAM,
                                              batch=a.batch)[0].cpu()
        h2d, d2h = n * D * 4 + n * 8, k * 8
        kernel = None
        bound_note = None
    for _ in range(max(3, a.warmup)):
        run()
    torch.cuda.synchronize()
    if a.config == 3:
        lib.vatlq_profile_read(None, None, None, 1)
        ops.prune_stats(reset=True)
    launches0 = vatlq._lib.launch_count()
    times = []
    with ClockSampler(dev.index or 0) as clk:
        for _ in range(a.steps):
            if a.config < 3:
                flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = run()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
    launches = vatlq._lib.launch_count() - launches0
    ms_step = sum(times) / len(times)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, result_arrays(out) if dataclasses.is_dataclass(out)
                     else {{2: "wpu", 3: "picks"}[a.config]: out})
    if a.config == 3:
        prune = ops.prune_stats(reset=True)
        sf = prune["streamed"] / prune["tiles"] if prune["tiles"] else 1.0
        roof = pass_roofline(lib, n, sf, a.steps, ms_step, prune, a.no_prune, ops.measure_fp64_mma(dev))
        lib.vatlq_profile_passes(0)
        picks_host = state["picks"].cpu().numpy()
        digest = sha_picks(picks_host)
        parity = check_golden(3, n, k, a.labeled_frac, moks, a.feat_kind, picks_host)
        st = state["st"]
        extra["coreset"] = {"passes_over_X": st.passes, "picks": st.picks, "rounds": st.rounds,
                            "fallback_rounds": st.fallback_empty + st.fallback_overflow, "ms_per_round": ms_step / max(1, st.rounds)}
    else:
        achieved = alg_bytes / (ms_step * 1e-3) / 1e9
        roof = {"kernel": kernel, "bound": "hbm", "achieved": achieved, "peak": peak_gbs, "unit": "GB/s",
                "frac": achieved / peak_gbs, "traffic": None, "peak_source": peak_src, "avg_launch_us": ms_step * 1e3,
                "algorithmic_bytes_per_launch": alg_bytes, "note": bound_note,
                "timing": "CUDA events around the whole operator call (launch floor included), L2 flushed before each"}
    # e2e: host buffers, copies inside the timed region
    run_host()
    torch.cuda.synchronize()
    reps = max(1, min(a.steps, 5))
    t0 = time.perf_counter()
    for _ in range(reps):
        run_host()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    e2e = {"value": n / dt, "unit": UNIT, "ms_per_step": dt * 1e3, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "steps": reps, "api": "vatlq.ops operator call with pinned host inputs, results read back"}
    line = {"metric": METRIC, "value": n / (ms_step * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": a.steps, "warmup": max(3, a.warmup),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": {1: "f32", 2: "f32", 3: "f64"}[a.config],
            "data": "synthetic", "config": config, "clocks": clk.summary(), "gpu_launches": int(launches),
            "roofline": roof, "e2e": e2e, **extra}
    if digest is not None:
        line["picks_sha256"] = digest
        line["parity"] = parity
    if not a.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline_entry(a, n, k, moks)
    rc = 3 if (parity and parity.get("pinned") and not parity.get("ok")) else 0
    return line, rc


if __name__ == "__main__":
    main()
