"""The query pass as one device-resident pipeline: scan -> WPU -> fusion -> core-set.

`QueryPass` is what `ActiveLearning.eval_and_query` (active_learning.py) drives; it is also the
public functional entry point (`run_query`) that bench.py times end to end.  A pool can be fed
in chunks (the way the estimator produces it, batch by batch): the last frame of a chunk is
kept as the halo of the next one, so THC never needs the whole pool resident.

Multi-GPU: every rank owns a contiguous range of the id-sorted pool.  THC needs the frame on
each side of the range (one (17,64,48) halo, exchanged with rank+-1), fusion all-reduces six
doubles, and the greedy selection exchanges one candidate block per round (see dist.py).
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np
import torch

from . import _lib, ops


@dataclass
class QueryResult:
    picks: torch.Tensor                 # (k,) int64, pick order, global indices
    thc: torch.Tensor | None            # (n_local,) fp32
    wpu: torch.Tensor | None            # (n_local,) fp32
    peak_mean: torch.Tensor | None      # (n_local,) fp32
    kpts: torch.Tensor | None           # (n_local,17,3) fp32
    unc: torch.Tensor | None            # fused score, fp64 (n_global when gathered)
    combine_weight: float | None        # mean local-peak value over unlabelled items
    stats: object = None
    extra: dict = field(default_factory=dict)


def _require_cuda(dev: torch.device):
    if dev.type != "cuda":
        raise _lib.VatlqError("QueryPass needs a CUDA device")


SINGLE_UNCERTAINTIES = ("HP", "TPC", "Entropy", "MPE", "Margin")   # one fp32 score per item, min-max normalised (:511-516)
FILTERS = ("None", "Diversity", "Coreset", "K-Means", "weighted")   # the filters `select` runs (:533-614)


def classify_uncertainty(name: str) -> tuple[str | None, bool, bool]:
    """(single, use_thc, use_wpu) of an uncertainty name, in the dispatch order of ActiveLearning.py:329-401: exact
    names first, then the substring tests.  In the elif order of the reference a name containing "THC" is THC (even
    "THC_WPU..."); only the exact string "THC+WPU" enables the two-criterion path (:345,364,403,494).  All three
    empty: "None", or a name without a device path."""
    single = name if name in SINGLE_UNCERTAINTIES else None
    use_thc = single is None and "THC" in name
    use_wpu = single is None and (name == "THC+WPU" or ("WPU" in name and "THC" not in name))
    return single, use_thc, use_wpu


def unlabelled_mask(n: int, labeled, device) -> torch.Tensor:
    """uint8 (n,) on `device`: 1 on every row whose id is not in `labeled`."""
    lab = np.asarray(labeled, dtype=np.int64)
    unl = torch.ones(n, dtype=torch.uint8, device=device)
    if lab.size:
        unl[torch.from_numpy(lab).to(device)] = 0
    return unl


def influence(X: torch.Tensor, unl: torch.Tensor, group=None) -> torch.Tensor:
    """Influence representativeness (ActiveLearning.py:467-475): row sums of the cosine-distance graph of the
    unlabelled rows, min-max normalised over them; fp64 (len(unl),), 0 on labelled rows.  X holds the rows `unl`
    masks, in any of ops.EMBEDDING_DTYPES (a 16-bit X gives the bits of its fp32 upcast).  `group`: the ranks hold
    disjoint row ranges of one pool (column sums and min / max are all-reduced)."""
    rows = torch.nonzero(unl, as_tuple=False).flatten()
    infl = torch.zeros(unl.numel(), dtype=torch.float64, device=unl.device)
    infl[rows] = ops.minmax_f64(ops.cosine_rowsum(X, rows=rows, group=group), group=group)
    return infl


def select(score: torch.Tensor, unl: torch.Tensor, X, k: int, filter: str, *, labeled=(), moks: float = 0.0,
           lam: float = 0.01, rule: str = "w_unc", first_pick: int = -1, batch: int = 16, comm=None,
           row_range: tuple[int, int] | None = None, w_unc: float = 1.0, combine_weight: float | None = None, group=None):
    """The filter stage after fusion (ActiveLearning.py:527-614) over the whole pool: `score` fp64 (n,), `unl` its
    uint8 unlabelled mask, X the (n, d) embeddings or a function returning them (called only by the filters that
    read X).  With at most one unlabelled item every filter returns the score-ordered top k (:533-534, 541-542).
    None: the top k by score, in id order.  Diversity: of the top 8k by score (in id order), the k of least cosine
    row sum (:581-590).  Coreset: ops.coreset_select (labeled, moks, lam, rule, first_pick, batch, comm, row_range;
    :609-614).  K-Means / weighted: kmeans_fit_select on the unlabelled rows in id order (:593-608); weighted first
    drops duplicate rows (np.unique(axis=0), which also sorts them), weighs each row 1 + w_unc * combine_weight *
    score and maps the chosen rows of that sorted matrix straight through the candidate ids (:553-580, kept as the
    reference has it); both clamp k to the rows they cluster, like the reference clamps query_size.
    X may be fp32, fp16 or bf16 for every filter: it is read as it is and the picks equal those of its fp32 upcast.
    `group`: the ranks hold the same X and share the K-Means assignment step.
    Returns (picks, k, stats): int64 ids on score's device in the reference's order, the k the filter used, and
    its CoresetStats or K-Means {"n_iter", "relocations"} (None for the other filters)."""
    n_unl = int(unl.sum().item())
    if n_unl <= 1 or filter == "None":
        return torch.sort(ops.rank_scores(score, unl, descending=True, count=k)).values, k, None
    X = X() if callable(X) else X
    if filter == "Diversity":
        cand = torch.sort(ops.rank_scores(score, unl, descending=True, count=8 * k)).values
        return cand[ops.rank_scores(ops.cosine_rowsum(X, rows=cand), None, descending=False, count=k)], k, None
    if filter == "Coreset":
        picks, st = ops.coreset_select(X, score, labeled, k, moks, lam, rule=rule, batch=batch, first_pick=first_pick,
                                       comm=comm, row_range=row_range)
        return picks, k, st
    if filter not in ("K-Means", "weighted"):
        raise ValueError(f"Filter type is not supported: {filter}")
    from . import kmeans as KM
    cand = torch.nonzero(unl, as_tuple=False).flatten()
    emb = X[cand]
    k = min(k, n_unl)
    weight = None
    if filter == "weighted":
        eidx = torch.as_tensor(KM.unique_rows_first_index(emb), dtype=torch.int64, device=emb.device)
        emb = emb[eidx]
        weight = (1 + w_unc * combine_weight * score[cand])[eidx].contiguous()
        k = min(k, int(emb.shape[0]))
    res = KM.kmeans_fit_select(emb, k, sample_weight=weight, group=group)
    picks = cand[torch.as_tensor(res.query_rows, dtype=torch.int64, device=cand.device)]
    return picks, k, {"n_iter": res.n_iter, "relocations": res.relocations}


class QueryPass:
    """Device-side state of one AL query over a pool of `n_local` items on this rank."""

    def __init__(self, n_local: int, device, ae_weights=None, uncertainty: str = "THC+WPU",
                 n_joints: int = ops.J, hm_shape=(ops.HM_H, ops.HM_W), keep_kpts: bool = True):
        self.dev = torch.device(device)
        _require_cuda(self.dev)
        _lib.lib()  # fail now, loudly, if the CUDA library is missing
        self.n = int(n_local)
        self.uncertainty = uncertainty
        self.single, self.use_thc, self.use_wpu = classify_uncertainty(uncertainty)
        if not (self.use_thc or self.use_wpu or self.single or uncertainty == "None"):
            raise ValueError("Uncertainty type is not supported by the accelerated path")
        self.nj, self.hm = n_joints, tuple(hm_shape)
        f32 = dict(dtype=torch.float32, device=self.dev)
        self.thc = torch.zeros(self.n, **f32)
        self.wpu = torch.zeros(self.n, **f32) if self.use_wpu else None
        self.peak_sum = torch.zeros(self.n, **f32)
        self.peak_cnt = torch.zeros(self.n, dtype=torch.int32, device=self.dev)
        self.peak_mean = torch.zeros(self.n, **f32)
        pose = self.single in ("HP", "TPC")
        self.kpts = torch.zeros((self.n, n_joints, 3), **f32) if (keep_kpts or self.use_wpu or pose) else None
        self.coords_hm = torch.zeros((self.n, n_joints, 2), **f32) if (keep_kpts or pose) else None
        # HP / TPC are finished from the scan's outputs once every chunk is in; Entropy per chunk
        self.aux = torch.zeros(self.n, **f32) if self.single else None
        self._aux_done = self.single != "TPC" and self.single != "HP"
        self._boxes = torch.zeros((self.n, 4), **f32) if pose else None
        self._flags = torch.zeros((2, self.n), dtype=torch.uint8, device=self.dev) if self.single == "TPC" else None
        self._halo_xy = [None, None]
        self._carry = None        # last frame of the previous chunk (halo_prev of the next)
        self._carry_pos = 0
        self._pending = None      # a chunk whose last frame still waits for its successor
        self._wpu_status = None   # device scalar: worst per-pose status seen so far (checked in fuse())
        self.ae = None
        if self.use_wpu:
            if ae_weights is None:
                raise _lib.VatlqError("WPU needs the WholeBodyAE weights")
            self.set_autoencoder(ae_weights)

    # the AE is re-initialised and fine-tuned after every retrain (ActiveLearning.py:681-685)
    def set_autoencoder(self, ae_weights):
        self.ae = ops.pack_ae_weights(ae_weights, self.dev)

    # ------------------------------------------------------------------ scoring
    def score_chunk(self, pos: int, H: torch.Tensor, boxes_xyxy: torch.Tensor, is_prev, is_next,
                    halo_prev: torch.Tensor | None = None, halo_next: torch.Tensor | None = None):
        """Score pool items [pos, pos+len(H)).  Chunks must arrive in pool order.  `halo_prev` /
        `halo_next` are only for the first / last chunk of a rank's range (frames owned by the
        neighbouring ranks); between chunks the halo is carried automatically: the scan of a
        chunk is given the first frame of the NEXT chunk as halo_next lazily — to keep the
        stream simple the last frame of every chunk is re-scored with the next chunk instead.
        H may be fp32, fp16 or bf16 (ops.HEATMAP_DTYPES); the carried halo frame keeps the chunk's dtype, so every
        chunk of one pool must share it (converting the carried frame to 16 bits would round it)."""
        m = H.shape[0]
        if m == 0:
            return
        if self._carry is not None and pos != self._carry_pos:
            raise _lib.VatlqError("chunks must be fed in pool order")
        if self._carry is not None and H.dtype != self._carry.dtype:
            raise _lib.VatlqError(f"every chunk of a pool must have one heat-map dtype: got {H.dtype} after "
                                  f"{self._carry.dtype}")
        first = self._carry is None
        hp = halo_prev if first else self._carry
        last_chunk = pos + m >= self.n
        res = ops.heatmap_scan(H, is_prev, is_next, boxes_xyxy, halo_prev=hp,
                               halo_next=halo_next if last_chunk else None)
        sl = slice(pos, pos + m)
        self.peak_sum[sl] = res.peak_sum
        self.peak_cnt[sl] = res.peak_cnt
        self.peak_mean[sl] = res.peak_mean
        if self.kpts is not None:
            self.kpts[sl] = res.kpts
        if self.coords_hm is not None:
            self.coords_hm[sl] = res.coords_hm
        if self.use_thc:
            self.thc[sl] = res.thc
            if not first and self._pending is not None:
                # the previous chunk's last item lacked its next frame: redo that one item now
                pH, pbox, pip, pin, php = self._pending
                fix = ops.heatmap_scan(pH, pip, pin, pbox, halo_prev=php, halo_next=H[0])
                self.thc[pos - 1] = fix.thc[0]
            if not last_chunk:
                prev_of_last = H[m - 2] if m >= 2 else hp
                # (device slices of the flags: no host round trip per chunk)
                ip = ops._flags(is_prev, m, self.dev, "is_prev")[m - 1:m].clone()
                inx = ops._flags(is_next, m, self.dev, "is_next")[m - 1:m].clone()
                self._pending = (H[m - 1:m].clone(), boxes_xyxy[m - 1:m].clone(), ip, inx,
                                 None if prev_of_last is None else prev_of_last.clone())
            else:
                self._pending = None
        self._carry = H[m - 1].clone()
        self._carry_pos = pos + m
        if self.single == "Entropy":
            self.aux[sl] = ops.heatmap_entropy(H)
        elif self.single in ("MPE", "Margin"):
            mpe, mar = ops.peak_uncertainty(H, want_mpe=self.single == "MPE", want_margin=self.single == "Margin")
            self.aux[sl] = mpe if self.single == "MPE" else mar
        if self._boxes is not None:
            self._boxes[sl] = boxes_xyxy
        if self._flags is not None:
            self._flags[0, sl] = ops._flags(is_prev, m, self.dev, "is_prev")
            self._flags[1, sl] = ops._flags(is_next, m, self.dev, "is_next")
            # heat-map-space coordinates of the neighbouring ranks' frames (TPC across a shard boundary)
            if first and halo_prev is not None:
                self._halo_xy[0] = ops.heatmap_scan(halo_prev.reshape(1, *H.shape[1:])).coords_hm[0]
            if last_chunk and halo_next is not None:
                self._halo_xy[1] = ops.heatmap_scan(halo_next.reshape(1, *H.shape[1:])).coords_hm[0]
        if self.use_wpu:
            w, ind, z = self.ae
            # invalid poses (hybrid_feature.py:25,31) are reported once, in fuse(): no host sync per chunk
            self.wpu[sl], st = ops.wpu(res.kpts, boxes_xyxy, w, ind, z, drop_ears=not self.use_thc, check_status=False,
                                       return_status=True)
            self._wpu_status = st.max() if self._wpu_status is None else torch.maximum(self._wpu_status, st.max())

    def score_pool(self, H, boxes_xyxy, is_prev, is_next, halo_prev=None, halo_next=None, chunk: int | None = None):
        """Score a pool that is already resident (one scan call, or chunked when asked).  `H` is the
        (n,J,h,w) tensor, or a list of (pos, tensor) segments in pool order that together cover the
        rank's items (a pool whose heat maps are held as several buffers, e.g. a resident ring)."""
        self._carry = None
        self._pending = None
        self._wpu_status = None
        self._halo_xy = [None, None]
        self._aux_done = self.single not in ("HP", "TPC")
        if isinstance(H, (list, tuple)):
            for pos, seg in H:
                e = pos + seg.shape[0]
                self.score_chunk(pos, seg, boxes_xyxy[pos:e], is_prev[pos:e], is_next[pos:e],
                                 halo_prev if pos == 0 else None, halo_next if e >= self.n else None)
            return
        if chunk is None or chunk >= H.shape[0]:
            self.score_chunk(0, H, boxes_xyxy, is_prev, is_next, halo_prev, halo_next)
            return
        n = H.shape[0]
        for a in range(0, n, chunk):
            b = min(n, a + chunk)
            self.score_chunk(a, H[a:b], boxes_xyxy[a:b], is_prev[a:b], is_next[a:b],
                             halo_prev if a == 0 else None, halo_next if b == n else None)

    def single_score(self) -> torch.Tensor:
        """The per-item HP / TPC / Entropy uncertainty (fp32), finished on first use."""
        if not self._aux_done:
            hp, tpc = ops.pose_uncertainty(self.coords_hm, self.kpts, self._boxes,
                                           None if self._flags is None else self._flags[0],
                                           None if self._flags is None else self._flags[1], self.hm,
                                           self._halo_xy[0], self._halo_xy[1],
                                           want_hp=self.single == "HP", want_tpc=self.single == "TPC")
            self.aux.copy_(hp if self.single == "HP" else tpc)
            self._aux_done = True
        return self.aux

    # ------------------------------------------------------------------ fusion
    def fuse(self, unlabeled_mask: torch.Tensor, thc_vs_wpu: str = "const", labeled_ratio: float = 0.0,
             group=None, n_unlabeled_global: int | None = None) -> torch.Tensor:
        """ActiveLearning.py:486-530: combine weight + fused uncertainty (fp64, 0 on labelled rows)."""
        unl = unlabeled_mask.to(self.dev).to(torch.uint8)
        if self._wpu_status is not None:
            bad = int(self._wpu_status.item())
            self._wpu_status = None
            if bad:  # the reference's AssertionErrors (hybrid_feature.py:25,31)
                raise AssertionError("height of human body must be positive!" if bad == 1
                                     else "at least one visible keypoint is required!")
        n_unl = int(unl.sum().item()) if n_unlabeled_global is None else int(n_unlabeled_global)
        self.n_unlabeled = n_unl
        # combine_weight = sum over unlabelled of localpeak_mean / |U|   (:411-412,486-488)
        pm = torch.where(unl.bool(), self.peak_mean.double(), torch.zeros((), dtype=torch.float64, device=self.dev))
        cw = pm.sum()
        if group is not None:
            torch.distributed.all_reduce(cw, group=group)
        self.combine_weight = float(cw.item()) / n_unl if n_unl > 0 else None
        if n_unl in (0, 1) or self.uncertainty == "None":
            return torch.zeros(self.n, dtype=torch.float64, device=self.dev)   # :490-491, :523-524
        if self.use_thc and self.use_wpu:
            return ops.fuse_scores(self.thc, self.wpu, unl, thc_vs_wpu, labeled_ratio, group=group)
        single = self.single_score() if self.single else (self.thc if self.use_thc else self.wpu)
        return ops.fuse_scores(single, None, unl, "single", group=group)


def run_query(H, boxes_xyxy, is_prev, is_next, X, ae_weights, labeled, k: int, moks: float = 0.0,
              lam: float = 0.01, uncertainty: str = "THC+WPU", thc_vs_wpu: str = "const", rule: str = "w_unc",
              batch: int = 16, device="cuda:0", chunk: int | None = None, first_pick: int = -1) -> QueryResult:
    """One full single-GPU query (THC + WPU + fusion + core-set) — the public functional API.
    Inputs may be host numpy arrays / CPU tensors (copied to `device` here, chunk by chunk for
    the heat maps) or CUDA tensors (used in place).  Heat maps may be fp32, fp16 or bf16 (numpy float16,
    torch bfloat16): they are copied and scored in their own dtype, never converted."""
    dev = torch.device(device)

    def to_dev(a, dtype):
        t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
        return t.to(device=dev, dtype=dtype, non_blocking=True)

    n = sum(t.shape[0] for _, t in H) if isinstance(H, (list, tuple)) else H.shape[0]
    qp = QueryPass(n, dev, ae_weights=ae_weights, uncertainty=uncertainty)
    bb = to_dev(boxes_xyxy, torch.float32)
    ip = to_dev(is_prev, torch.uint8)
    inx = to_dev(is_next, torch.uint8)
    on_dev = isinstance(H, (list, tuple)) or (isinstance(H, torch.Tensor) and H.is_cuda)
    if on_dev:
        qp.score_pool(H, bb, ip, inx, chunk=chunk)
    else:
        step = chunk or 8192
        Ht = H if isinstance(H, torch.Tensor) else torch.from_numpy(H)
        qp._carry = None
        for a in range(0, n, step):
            b = min(n, a + step)
            qp.score_chunk(a, Ht[a:b].to(dev, non_blocking=True), bb[a:b], ip[a:b], inx[a:b])
    Xd = to_dev(X, torch.float32)
    lab = np.asarray(list(labeled), dtype=np.int64)
    unl = unlabelled_mask(n, lab, dev)
    unc = qp.fuse(unl, thc_vs_wpu, labeled_ratio=lab.size / max(n, 1))
    picks, st = ops.coreset_select(Xd, unc, lab, k, moks, lam, rule=rule, batch=batch, first_pick=first_pick)
    return QueryResult(picks=picks, thc=qp.thc, wpu=qp.wpu, peak_mean=qp.peak_mean, kpts=qp.kpts, unc=unc,
                       combine_weight=qp.combine_weight, stats=st)
