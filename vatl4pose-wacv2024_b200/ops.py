"""Batched device operators of the query pass: thin torch-tensor wrappers over the C ABI.

Every function takes CUDA tensors (borrowed pointers go straight into libvatlq), launches on
torch's current stream and returns CUDA tensors.  Nothing here computes on the CPU and nothing
falls back: a missing library or a non-CUDA tensor raises.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib

J, HM_H, HM_W = 17, 64, 48


def _stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _cuda(t: torch.Tensor, dtype, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.VatlqError(f"{name} must be a CUDA tensor (the query pass has no CPU path)")
    if t.dtype != dtype:
        raise _lib.VatlqError(f"{name} must be {dtype}, got {t.dtype}")
    return t.contiguous()


# heat-map element types and their VATLQ_* codes: 16-bit maps are read as they are, and every result equals the
# fp32 path's on their exact upcast, bit for bit (include/vatlq.h)
HEATMAP_DTYPES = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}
# embedding element types of the core-set, pairwise-distance and cosine row-sum entries: the same contract, for X
EMBEDDING_DTYPES = HEATMAP_DTYPES


def _embeddings(t: torch.Tensor, name: str) -> torch.Tensor:
    """A CUDA (n,d) embedding tensor in one of EMBEDDING_DTYPES, contiguous."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.VatlqError(f"{name} must be a CUDA tensor (the query pass has no CPU path)")
    if t.dtype not in EMBEDDING_DTYPES:
        raise _lib.VatlqError(f"{name} must be torch.float32, torch.float16 or torch.bfloat16, got {t.dtype}")
    return t.contiguous()


def _heatmaps(t: torch.Tensor, name: str) -> torch.Tensor:
    """A CUDA heat-map tensor in one of HEATMAP_DTYPES, contiguous."""
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise _lib.VatlqError(f"{name} must be a CUDA tensor (the query pass has no CPU path)")
    if t.dtype not in HEATMAP_DTYPES:
        raise _lib.VatlqError(f"{name} must be torch.float32, torch.float16 or torch.bfloat16, got {t.dtype}")
    return t.contiguous()


def _flags(t, n: int, dev, name: str):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t))
    t = t.to(device=dev).to(torch.uint8).contiguous()
    if t.numel() != n:
        raise _lib.VatlqError(f"{name} must have {n} entries")
    return t


@dataclass
class ScanResult:
    thc: torch.Tensor        # (n,) fp32
    peak_sum: torch.Tensor   # (n,) fp32
    peak_cnt: torch.Tensor   # (n,) int32
    peak_mean: torch.Tensor  # (n,) fp32 (NaN where no peak survives)
    coords_hm: torch.Tensor  # (n,J,2) fp32 heat-map-space coordinates
    kpts: torch.Tensor | None  # (n,J,3) fp32 image-space x, y, score (needs boxes)


def heatmap_scan(H: torch.Tensor, is_prev=None, is_next=None, boxes_xyxy: torch.Tensor | None = None,
                 halo_prev: torch.Tensor | None = None, halo_next: torch.Tensor | None = None) -> ScanResult:
    """THC + local-peak statistics + argmax/quarter-pixel coordinates of a whole pool in one pass
    (vatlq_heatmap_scan_dt).  H (n,J,h,w) fp32 / fp16 / bf16 CUDA (halos of the same dtype); flags length n;
    boxes (n,4) fp32 xyxy.  Outputs are fp32 whatever H's dtype."""
    H = _heatmaps(H, "H")
    if H.dim() != 4:
        raise _lib.VatlqError("H must be (n,J,h,w)")
    n, nj, h, w = H.shape
    dev = H.device
    ip = _flags(is_prev, n, dev, "is_prev")
    inx = _flags(is_next, n, dev, "is_next")
    bb = None if boxes_xyxy is None else _cuda(boxes_xyxy.to(dev), torch.float32, "boxes_xyxy")
    if bb is not None and tuple(bb.shape) != (n, 4):
        raise _lib.VatlqError("boxes_xyxy must be (n,4)")
    hp = None if halo_prev is None else _cuda(halo_prev, H.dtype, "halo_prev")
    hn = None if halo_next is None else _cuda(halo_next, H.dtype, "halo_next")
    for t, nm in ((hp, "halo_prev"), (hn, "halo_next")):
        if t is not None and t.numel() != nj * h * w:
            raise _lib.VatlqError(f"{nm} must be one (J,h,w) frame")
    L = _lib.lib()
    ws_bytes = L.vatlq_heatmap_scan_workspace_bytes(n, nj)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    out = ScanResult(
        thc=torch.empty(n, dtype=torch.float32, device=dev),
        peak_sum=torch.empty(n, dtype=torch.float32, device=dev),
        peak_cnt=torch.empty(n, dtype=torch.int32, device=dev),
        peak_mean=torch.empty(n, dtype=torch.float32, device=dev),
        coords_hm=torch.empty((n, nj, 2), dtype=torch.float32, device=dev),
        kpts=None if bb is None else torch.empty((n, nj, 3), dtype=torch.float32, device=dev))
    with torch.cuda.device(dev):
        _lib.check(L.vatlq_heatmap_scan_dt(_ptr(H), HEATMAP_DTYPES[H.dtype], _ptr(ip), _ptr(inx), n, nj, h, w, _ptr(hp),
                                           _ptr(hn), _ptr(bb), _ptr(out.thc), _ptr(out.peak_sum), _ptr(out.peak_cnt),
                                           _ptr(out.peak_mean), _ptr(out.coords_hm), _ptr(out.kpts), _ptr(ws), ws_bytes,
                                           _stream()), "vatlq_heatmap_scan_dt")
    return out


def thc3(cur: torch.Tensor, prev: torch.Tensor | None, nxt: torch.Tensor | None, is_prev, is_next) -> torch.Tensor:
    """Strict three-tensor THC (separately forwarded prev/next crops, ActiveLearning.py:293-297).
    cur / prev / next: one dtype of HEATMAP_DTYPES."""
    cur = _heatmaps(cur, "cur")
    n, nj, h, w = cur.shape
    dev = cur.device
    prev = None if prev is None else _cuda(prev, cur.dtype, "prev")
    nxt = None if nxt is None else _cuda(nxt, cur.dtype, "next")
    ip = _flags(is_prev, n, dev, "is_prev")
    inx = _flags(is_next, n, dev, "is_next")
    out = torch.empty(n, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vatlq_thc3_dt(_ptr(cur), _ptr(prev), _ptr(nxt), HEATMAP_DTYPES[cur.dtype], _ptr(ip),
                                            _ptr(inx), n, nj, h, w, _ptr(out), _stream()), "vatlq_thc3_dt")
    return out


def pack_ae_weights(weights, device) -> tuple[torch.Tensor, int, int]:
    """Pack the 8 Linear layers of a WholeBodyAE into the flat layout vatlq_wpu expects.
    `weights`: a state_dict (encoder.{0,2,4,6}/decoder.{0,2,4,6}.{weight,bias}), an nn.Module
    with .state_dict(), or a list of 8 (W[out,in], b[out]) pairs."""
    if hasattr(weights, "state_dict"):
        weights = weights.state_dict()
    if isinstance(weights, dict):
        pairs = []
        for part in ("encoder", "decoder"):
            for k in (0, 2, 4, 6):
                pairs.append((weights[f"{part}.{k}.weight"], weights[f"{part}.{k}.bias"]))
    else:
        pairs = list(weights)
    if len(pairs) != 8:
        raise _lib.VatlqError("WholeBodyAE has 8 Linear layers")
    flat = []
    for Wm, b in pairs:
        Wm = torch.as_tensor(np.asarray(Wm) if not isinstance(Wm, torch.Tensor) else Wm).detach().float().cpu()
        b = torch.as_tensor(np.asarray(b) if not isinstance(b, torch.Tensor) else b).detach().float().cpu()
        flat += [Wm.reshape(-1), b.reshape(-1)]
    in_dim = int(pairs[0][0].shape[1])
    z_dim = int(pairs[3][0].shape[0])
    dims = [in_dim, 24, 12, 7, z_dim, 7, 12, 24, in_dim]
    for (Wm, _), a, b in zip(pairs, dims[:-1], dims[1:]):
        if tuple(Wm.shape) != (b, a):
            raise _lib.VatlqError(f"unexpected AE layer shape {tuple(Wm.shape)}, wanted {(b, a)}")
    packed = torch.cat(flat).contiguous().to(device)
    assert packed.numel() == _lib.lib().vatlq_wpu_weight_count(in_dim, z_dim)
    return packed, in_dim, z_dim


def wpu(kpts: torch.Tensor, boxes_xyxy: torch.Tensor, packed_weights: torch.Tensor, in_dim: int, z_dim: int,
        drop_ears: bool = False, return_features: bool = False, check_status: bool = True,
        return_status: bool = False):
    """Whole-body pose unnaturalness of every pose (vatlq_wpu).  kpts (n,17,3) fp32 CUDA."""
    kpts = _cuda(kpts, torch.float32, "kpts")
    n = kpts.shape[0]
    if kpts.numel() != n * 51:
        raise _lib.VatlqError("kpts must be (n,17,3)")
    dev = kpts.device
    bb = _cuda(boxes_xyxy.to(dev), torch.float32, "boxes_xyxy")
    wts = _cuda(packed_weights, torch.float32, "weights")
    out = torch.empty(n, dtype=torch.float32, device=dev)
    feat = torch.empty((n, in_dim), dtype=torch.float32, device=dev) if return_features else None
    status = torch.empty(n, dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vatlq_wpu(_ptr(kpts), _ptr(bb), _ptr(wts), in_dim, z_dim, int(drop_ears), _ptr(out),
                                        _ptr(feat), _ptr(status), n, _stream()), "vatlq_wpu")
    if check_status:
        bad = int(status.max().item()) if n else 0
        if bad:  # the reference's AssertionErrors (hybrid_feature.py:25,31)
            raise AssertionError("height of human body must be positive!" if bad == 1
                                 else "at least one visible keypoint is required!")
    if return_status:
        return (out, feat, status) if return_features else (out, status)
    return (out, feat) if return_features else out


FUSE_MODES = {"const": 0, "increase": 1, "decrease": 2, "single": 3}


def fuse_scores(thc: torch.Tensor, wpu_: torch.Tensor | None, unlabeled: torch.Tensor | None,
                mode: str = "const", labeled_ratio: float = 0.0, group=None) -> torch.Tensor:
    """Min-max / combine / min-max of ActiveLearning.py:490-516 on the device, float64.
    Returns unc (n,) fp64 with 0 at labelled rows.  `group`: a torch.distributed group whose
    ranks hold disjoint shards of the pool (statistics are all-reduced with MIN)."""
    thc = _cuda(thc, torch.float32, "thc")
    n = thc.numel()
    dev = thc.device
    w = None if wpu_ is None else _cuda(wpu_, torch.float32, "wpu")
    m = FUSE_MODES["single"] if w is None else FUSE_MODES[mode]
    unl = _flags(unlabeled, n, dev, "unlabeled")
    L = _lib.lib()
    s1 = torch.empty(4, dtype=torch.float64, device=dev)
    s2 = torch.empty(2, dtype=torch.float64, device=dev)
    u = torch.empty(n, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.vatlq_fuse_stats(_ptr(thc), _ptr(w), _ptr(unl), n, _ptr(s1), _stream()), "vatlq_fuse_stats")
        if group is not None:
            torch.distributed.all_reduce(s1, op=torch.distributed.ReduceOp.MIN, group=group)
        _lib.check(L.vatlq_fuse_combine(_ptr(thc), _ptr(w), _ptr(unl), n, _ptr(s1), m, float(labeled_ratio),
                                        _ptr(u), _ptr(s2), _stream()), "vatlq_fuse_combine")
        if group is not None:
            torch.distributed.all_reduce(s2, op=torch.distributed.ReduceOp.MIN, group=group)
        _lib.check(L.vatlq_fuse_final(_ptr(unl), n, _ptr(s2), _ptr(u), _stream()), "vatlq_fuse_final")
    return u


RULES = {"w_unc": 0, "fixed_lambda": 1, "dist": 2}


@dataclass
class CoresetStats:
    passes: int
    picks: int
    rounds: int
    fallback_empty: int
    fallback_overflow: int
    candidates: int
    rounds_launched: int
    batch: int
    ns_wait: int = 0        # waiting for the peers' candidate blocks (summed over the rounds)
    ns_tiles: int = 0       # candidate x candidate distance tiles
    ns_plan: int = 0        # the planner (greedy replay on the candidates)
    tiles: int = 0          # 8-row tiles the passes of this call saw ...
    tiles_streamed: int = 0  # ... and streamed (the rest was pruned exactly)
    prune_violations: int = 0   # verify mode only: rows of flagged tiles whose min_d moved (must be 0)
    segments: int = 0


TC_INIT_MIN_LABELED = 256     # below this the exact passes are cheaper than two GEMM sweeps
_tc_init_stats = {"calls": 0, "fallbacks": 0, "pairs": 0, "violations": 0}


def coreset_init_tc(X: torch.Tensor, lab: torch.Tensor, min_d: torch.Tensor, lo: int, hi: int, verify: bool = False,
                    want_tmin: bool = False):
    """min_d[lo:hi] = distance to the nearest labelled row through the TF32 tcgen05 GEMM + exact re-scoring
    (vatlq_coreset_init_tc).  Returns (ok, stats dict, tmin or None); ok False = candidate list overflow."""
    n, d = X.shape
    L = _lib.lib()
    ws_bytes = L.vatlq_coreset_init_tc_workspace_bytes(n, hi - lo, lab.numel())
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=X.device)
    st = (C.c_int64 * 4)()
    tmin = torch.empty(hi - lo, dtype=torch.float32, device=X.device) if want_tmin else None
    with torch.cuda.device(X.device):
        rc = L.vatlq_coreset_init_tc(_ptr(X), n, d, lo, hi, _ptr(lab), lab.numel(), _ptr(min_d), _ptr(ws), ws_bytes,
                                     1 if verify else 0, C.cast(st, C.c_void_p), _ptr(tmin), _stream())
    stats = {"pairs": int(st[0]), "capacity": int(st[1]), "violations": int(st[2]), "groups": int(st[3])}
    _tc_init_stats["calls"] += 1
    _tc_init_stats["pairs"] += stats["pairs"]
    _tc_init_stats["violations"] += stats["violations"]
    if rc == _lib.ESTATE:
        _tc_init_stats["fallbacks"] += 1
        return False, stats, tmin
    _lib.check(rc, "vatlq_coreset_init_tc")
    return True, stats, tmin


def coreset_select(X: torch.Tensor, unc: torch.Tensor, labeled, k: int, moks: float, lam: float,
                   rule: str = "w_unc", first_pick: int = -1, batch: int = 16, comm=None,
                   row_range: tuple[int, int] | None = None, return_state: bool = False, tc_init: bool | None = None):
    """k-center greedy selection (vatlq_coreset_init_dt + vatlq_coreset_select_dt).
    X (n,d) CUDA in one of EMBEDDING_DTYPES (replicated on every rank when comm is given): a 16-bit X is read as it
    is and gives, bit for bit, the picks, min_d, unc and counting stats of its fp32 upcast.  unc (n,) fp64 CUDA — a
    private copy is made, like the caller's deepcopy at ActiveLearning.py:612-613.
    tc_init: labelled-set initialisation on the TF32 tcgen05 GEMM (coreset_init_tc, fp32 X only); None picks it for
    fp32 X at d = 2048 with >= TC_INIT_MIN_LABELED labelled rows.  A 16-bit X takes the exact fp64 init (at
    L = 17 000 about 204 ms against 39 ms, DESIGN.md §4.5); tc_init=True with a 16-bit X raises.
    Returns the picks as an int64 CUDA tensor in pick order (and stats / min_d / unc)."""
    X = _embeddings(X, "X")
    dt = EMBEDDING_DTYPES[X.dtype]
    if tc_init and dt != _lib.F32:
        raise _lib.VatlqError("tc_init=True needs an fp32 X (the tcgen05 init is TF32); use tc_init=None for 16-bit X")
    n, d = X.shape
    dev = X.device
    unc = _cuda(unc, torch.float64, "unc").clone()
    if unc.numel() != n:
        raise _lib.VatlqError("unc must have n entries")
    lab = torch.as_tensor(np.asarray(list(labeled) if not isinstance(labeled, (np.ndarray, torch.Tensor)) else
                                     (labeled.cpu().numpy() if isinstance(labeled, torch.Tensor) else labeled),
                                     dtype=np.int64)).to(dev)
    lo, hi = (0, n) if row_range is None else row_range
    L = _lib.lib()
    ws_bytes = L.vatlq_coreset_workspace_bytes_dt(n, d, batch, dt)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    min_d = torch.empty(n, dtype=torch.float64, device=dev)
    out = torch.empty(max(k, 1), dtype=torch.int64, device=dev)
    stats = (C.c_int64 * 16)()
    if tc_init is None:    # the labelled-set contraction on the tcgen05 tensor cores when it is large enough to pay
        tc_init = dt == _lib.F32 and d == 2048 and lab.numel() >= TC_INIT_MIN_LABELED and hi > lo
    done = False
    if tc_init and lab.numel() > 0:
        done, _, _ = coreset_init_tc(X, lab, min_d, lo, hi)
    with torch.cuda.device(dev):
        if not done:
            _lib.check(L.vatlq_coreset_init_dt(_ptr(X), dt, n, d, lo, hi, _ptr(lab) if lab.numel() else None,
                                               lab.numel(), _ptr(min_d), _ptr(ws), ws_bytes, _stream()),
                       "vatlq_coreset_init_dt")
        _lib.check(L.vatlq_coreset_select_dt(_ptr(X), dt, n, d, lo, hi, _ptr(min_d), _ptr(unc), RULES[rule], float(moks),
                                             float(lam), lab.numel(), int(first_pick), int(k), int(batch), _ptr(out),
                                             C.c_void_p(comm) if comm else None, _ptr(ws), ws_bytes,
                                             C.cast(stats, C.c_void_p), _stream()), "vatlq_coreset_select_dt")
    picks = out[:k]
    st = CoresetStats(*[int(v) for v in stats][:15])
    if return_state:
        return picks, st, min_d, unc
    return picks, st


PRUNE_MODES = {"env": -1, "off": 0, "on": 1, "verify": 2}


def set_prune(mode: str = "env", min_rows: int = -1):
    """Exact pruning of the core-set passes (include/vatlq.h): "env" (VATLQ_PRUNE), "off", "on" or
    "verify"; min_rows < 0 keeps VATLQ_PRUNE_MIN_ROWS (default 8192 owned rows)."""
    _lib.check(_lib.lib().vatlq_coreset_set_prune(PRUNE_MODES[mode], int(min_rows)), "vatlq_coreset_set_prune")


def prune_stats(reset: bool = False) -> dict:
    """Tiles seen / streamed by the passes, verify violations and the segment count of the last call."""
    out = (C.c_int64 * 4)()
    _lib.check(_lib.lib().vatlq_coreset_prune_stats(C.cast(out, C.c_void_p), int(reset)), "vatlq_coreset_prune_stats")
    return {"tiles": int(out[0]), "streamed": int(out[1]), "violations": int(out[2]), "segments": int(out[3])}


SCREEN_MODES = {"env": -1, "off": 0, "on": 1, "verify": 2}


def set_screen(mode: str = "env"):
    """fp16 screen of the 16-pick rounds (include/vatlq.h): "env" (VATLQ_PASS_SCREEN), "off", "on" or "verify"."""
    _lib.check(_lib.lib().vatlq_coreset_set_screen(SCREEN_MODES[mode]), "vatlq_coreset_set_screen")


def screen_stats(reset: bool = False) -> dict:
    """Rows screened / listed for the exact fp64 pass and verify violations, since the last reset."""
    out = (C.c_int64 * 3)()
    _lib.check(_lib.lib().vatlq_coreset_screen_stats(C.cast(out, C.c_void_p), int(reset)), "vatlq_coreset_screen_stats")
    return {"screened": int(out[0]), "listed": int(out[1]), "violations": int(out[2])}


def pairwise_dist(X: torch.Tensor, centers) -> torch.Tensor:
    """(n,m) fp64 Euclidean distances of every row to X[centers] with the library's canonical
    fp64 arithmetic (sklearn order: sqrt(max(0, -2 x.c + |x|^2 + |c|^2))).  X in any of EMBEDDING_DTYPES."""
    X = _embeddings(X, "X")
    n, d = X.shape
    c = torch.as_tensor(np.asarray(centers, dtype=np.int64)).to(X.device)
    out = torch.empty((n, c.numel()), dtype=torch.float64, device=X.device)
    ws = torch.empty(n, dtype=torch.float64, device=X.device)
    with torch.cuda.device(X.device):
        _lib.check(_lib.lib().vatlq_pairwise_dist_dt(_ptr(X), EMBEDDING_DTYPES[X.dtype], n, d, _ptr(c), c.numel(), _ptr(out),
                                                     _ptr(ws), n * 8, _stream()), "vatlq_pairwise_dist_dt")
    return out


# ----------------------------------------------------------------------------------------
# SURVEY.md §8f "next" rows: HP / TPC / Entropy uncertainties, Influence / Diversity scores
# ----------------------------------------------------------------------------------------

def pose_uncertainty(coords_hm: torch.Tensor, kpts: torch.Tensor, boxes_xyxy: torch.Tensor, is_prev=None, is_next=None,
                     hm_shape=(HM_H, HM_W), halo_prev_xy: torch.Tensor | None = None,
                     halo_next_xy: torch.Tensor | None = None, want_hp: bool = True, want_tpc: bool = True):
    """HP (ActiveLearning.py:329-330) and TPC (:333-344,736-745) of every item from the scan's
    outputs (vatlq_pose_unc).  Returns (hp, tpc), fp32 (n,) CUDA tensors (None when not wanted)."""
    kpts = _cuda(kpts, torch.float32, "kpts")
    n, nj = kpts.shape[0], kpts.shape[1]
    dev = kpts.device
    xy = _cuda(coords_hm, torch.float32, "coords_hm")
    bb = _cuda(boxes_xyxy.to(dev), torch.float32, "boxes_xyxy")
    if tuple(xy.shape) != (n, nj, 2) or tuple(bb.shape) != (n, 4):
        raise _lib.VatlqError("coords_hm must be (n,J,2) and boxes_xyxy (n,4)")
    ip = _flags(is_prev, n, dev, "is_prev")
    inx = _flags(is_next, n, dev, "is_next")
    hpx = None if halo_prev_xy is None else _cuda(halo_prev_xy, torch.float32, "halo_prev_xy")
    hnx = None if halo_next_xy is None else _cuda(halo_next_xy, torch.float32, "halo_next_xy")
    for t, nm in ((hpx, "halo_prev_xy"), (hnx, "halo_next_xy")):
        if t is not None and t.numel() != nj * 2:
            raise _lib.VatlqError(f"{nm} must be (J,2)")
    hp = torch.empty(n, dtype=torch.float32, device=dev) if want_hp else None
    tpc = torch.empty(n, dtype=torch.float32, device=dev) if want_tpc else None
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vatlq_pose_unc(_ptr(xy), _ptr(kpts), _ptr(bb), _ptr(ip), _ptr(inx), n, nj,
                                             int(hm_shape[0]), int(hm_shape[1]), _ptr(hpx), _ptr(hnx), _ptr(hp),
                                             _ptr(tpc), _stream()), "vatlq_pose_unc")
    return hp, tpc


def heatmap_entropy(H: torch.Tensor) -> torch.Tensor:
    """Entropy uncertainty (ActiveLearning.py:790-796) of every frame (vatlq_heatmap_entropy_dt); H in any of
    HEATMAP_DTYPES, fp32 (n,) out."""
    H = _heatmaps(H, "H")
    if H.dim() != 4:
        raise _lib.VatlqError("H must be (n,J,h,w)")
    n, nj, h, w = H.shape
    out = torch.empty(n, dtype=torch.float32, device=H.device)
    ws = torch.empty(max(n * nj, 1), dtype=torch.float32, device=H.device)
    with torch.cuda.device(H.device):
        _lib.check(_lib.lib().vatlq_heatmap_entropy_dt(_ptr(H), HEATMAP_DTYPES[H.dtype], n, nj, h, w, _ptr(out), _ptr(ws),
                                                       ws.numel() * 4, _stream()), "vatlq_heatmap_entropy_dt")
    return out


def cosine_rowsum(X: torch.Tensor, rows=None, group=None) -> torch.Tensor:
    """Row sums of the cosine-distance matrix of X[rows] (all rows when None): the Influence score
    before normalisation (ActiveLearning.py:471-475) / the Diversity score (:582-585), fp64 (m,).
    X (n,d) CUDA in one of EMBEDDING_DTYPES (vatlq_cosine_*_dt): a 16-bit X is read as it is and gives, bit for bit,
    the row sums of its fp32 upcast.  `group`: ranks hold disjoint row sets of one pool; the column sums are
    all-reduced."""
    X = _embeddings(X, "X")
    dt = EMBEDDING_DTYPES[X.dtype]
    n, d = X.shape
    dev = X.device
    r = None
    m = n
    if rows is not None:
        r = rows if isinstance(rows, torch.Tensor) else torch.as_tensor(np.asarray(rows, dtype=np.int64))
        r = r.to(device=dev, dtype=torch.int64).contiguous()
        m = r.numel()
    L = _lib.lib()
    ws_bytes = L.vatlq_cosine_workspace_bytes(d)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=dev)
    S = torch.empty(d, dtype=torch.float64, device=dev)
    out = torch.empty(m, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(L.vatlq_cosine_colsum_dt(_ptr(X), dt, n, d, _ptr(r), m, _ptr(S), _ptr(ws), ws_bytes, _stream()),
                   "vatlq_cosine_colsum_dt")
        m_total = m
        if group is not None:
            torch.distributed.all_reduce(S, group=group)
            cnt = torch.tensor([m], dtype=torch.int64, device=dev)
            torch.distributed.all_reduce(cnt, group=group)
            m_total = int(cnt.item())
        _lib.check(L.vatlq_cosine_rowsum_dt(_ptr(X), dt, n, d, _ptr(r), m, _ptr(S), float(m_total), _ptr(out),
                                            _stream()), "vatlq_cosine_rowsum_dt")
    return out


def minmax_f64(v: torch.Tensor, mask=None, group=None) -> torch.Tensor:
    """(v - min) / (max - min) over the rows with mask != 0, 0 elsewhere, fp64 (the influence
    normalisation of ActiveLearning.py:477); returns a new tensor."""
    v = _cuda(v, torch.float64, "v").clone()
    n = v.numel()
    mk = _flags(mask, n, v.device, "mask")
    s2 = torch.empty(2, dtype=torch.float64, device=v.device)
    L = _lib.lib()
    with torch.cuda.device(v.device):
        _lib.check(L.vatlq_minmax_stats_f64(_ptr(v), _ptr(mk), n, _ptr(s2), _stream()), "vatlq_minmax_stats_f64")
        if group is not None:
            torch.distributed.all_reduce(s2, op=torch.distributed.ReduceOp.MIN, group=group)
        _lib.check(L.vatlq_fuse_final(_ptr(mk), n, _ptr(s2), _ptr(v), _stream()), "vatlq_fuse_final")
    return v


def blend_scores(unc: torch.Tensor, infl: torch.Tensor, combine_weight: float, mask=None) -> torch.Tensor:
    """combine_weight * unc + (1 - combine_weight) * influence (ActiveLearning.py:519), fp64."""
    unc = _cuda(unc, torch.float64, "unc")
    infl = _cuda(infl, torch.float64, "infl")
    n = unc.numel()
    if infl.numel() != n:
        raise _lib.VatlqError("unc and infl must have the same length")
    mk = _flags(mask, n, unc.device, "mask")
    out = torch.empty(n, dtype=torch.float64, device=unc.device)
    with torch.cuda.device(unc.device):
        _lib.check(_lib.lib().vatlq_fuse_blend(_ptr(unc), _ptr(infl), _ptr(mk), n, float(combine_weight), _ptr(out), _stream()),
                   "vatlq_fuse_blend")
    return out


def oks(kpts: torch.Tensor, gt_kpts: torch.Tensor, bbox_ann_xyxy: torch.Tensor) -> torch.Tensor:
    """OKS of every predicted pose against its ground truth (al_metric.py:42-69; call site
    ActiveLearning.py:309), fp64 (n,).  kpts / gt_kpts (n,17,3) fp32, bbox_ann (n,4) xyxy fp32."""
    kpts = _cuda(kpts, torch.float32, "kpts")
    n = kpts.shape[0]
    dev = kpts.device
    gt = _cuda(gt_kpts.to(dev).reshape(n, 51), torch.float32, "gt_kpts")
    bb = _cuda(bbox_ann_xyxy.to(dev).reshape(n, 4), torch.float32, "bbox_ann_xyxy")
    if kpts.numel() != n * 51 or gt.numel() != n * 51:
        raise _lib.VatlqError("kpts and gt_kpts must be (n,17,3)")
    out = torch.empty(n, dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vatlq_oks(_ptr(kpts), _ptr(gt), _ptr(bb), n, _ptr(out), _stream()), "vatlq_oks")
    return out


def peak_uncertainty(H: torch.Tensor, want_mpe: bool = True, want_margin: bool = True):
    """MPE / Margin uncertainties (ActiveLearning.py:762-788) of every frame (vatlq_peak_unc_dt): H in any of
    HEATMAP_DTYPES, fp32 (n,) each."""
    H = _heatmaps(H, "H")
    if H.dim() != 4:
        raise _lib.VatlqError("H must be (n,J,h,w)")
    n, nj, h, w = H.shape
    mpe = torch.empty(n, dtype=torch.float32, device=H.device) if want_mpe else None
    mar = torch.empty(n, dtype=torch.float32, device=H.device) if want_margin else None
    ws = torch.empty(max(int(_lib.lib().vatlq_peak_workspace_bytes(n, nj, h, w)), 16), dtype=torch.uint8, device=H.device)
    with torch.cuda.device(H.device):
        _lib.check(_lib.lib().vatlq_peak_unc_dt(_ptr(H), HEATMAP_DTYPES[H.dtype], n, nj, h, w, _ptr(mpe), _ptr(mar), _ptr(ws),
                                                ws.numel(), _stream()), "vatlq_peak_unc_dt")
    return mpe, mar


def rank_scores(score: torch.Tensor, mask=None, descending: bool = True, count: int | None = None) -> torch.Tensor:
    """Row ids with mask != 0 ordered by score (descending by default), equal scores in ascending id order — the
    candidate order of ActiveLearning.py:527-530 — computed on the device (vatlq_rank_scores).  Returns the first
    `count` ids (all masked-in rows when None) as an int64 CUDA tensor."""
    score = _cuda(score, torch.float64, "score")
    n = score.numel()
    mk = _flags(mask, n, score.device, "mask")
    m = n if mk is None else int(mk.sum().item())
    out = torch.empty(max(n, 1), dtype=torch.int64, device=score.device)
    L = _lib.lib()
    ws_bytes = L.vatlq_rank_workspace_bytes(n)
    ws = torch.empty(max(ws_bytes, 1), dtype=torch.uint8, device=score.device)
    with torch.cuda.device(score.device):
        _lib.check(L.vatlq_rank_scores(_ptr(score), _ptr(mk), n, int(descending), _ptr(out), _ptr(ws), ws_bytes, _stream()),
                   "vatlq_rank_scores")
    return out[:m if count is None else min(m, int(count))]


def measure_fp64_mma(device=None) -> float:
    """fp64 tensor-core (DMMA) peak of the device in FMA/s, measured live (vatlq_measure_fp64_mma)."""
    dev = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
    ws = torch.empty(4 * 256 * 8 * 1024, dtype=torch.uint8, device=dev)
    out = C.c_double()
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().vatlq_measure_fp64_mma(C.byref(out), _ptr(ws), ws.numel(), _stream()), "vatlq_measure_fp64_mma")
    return float(out.value)
