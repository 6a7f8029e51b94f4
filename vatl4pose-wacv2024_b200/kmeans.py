"""K-Means / weighted K-Means query filters (ActiveLearning.py:593-608, :553-580) on the device.

The reference calls `sklearn.cluster.KMeans(n_clusters=query_size, random_state=318).fit_predict(embeddings
[, sample_weight=weight])` and queries, per cluster, the member closest to its centre.  This module is the host
side of that estimator for this one call: it draws the random numbers from numpy's RandomState in the order
sklearn draws them (sklearn/cluster/_kmeans.py: `_kmeans_plusplus`), decides convergence the way
`_kmeans_single_lloyd` does, and leaves everything data-sized to libvatlq (`csrc/kmeans.cu`).  There is no CPU
path: the embeddings must be a CUDA tensor.  They may be fp32, fp16 or bf16 (ops.EMBEDDING_DTYPES): a 16-bit X is read
as it is by the vatlq_kmeans_*_dt entries and every result (labels, centres, seeds, iteration count, relocations,
picks) equals, bit for bit, that of its fp32 upcast; fp32 X goes through the fp32 entries.

What is reproduced: the labels and therefore the queried rows.  sklearn's centre sums depend on its OpenMP chunking,
so centre coordinates of clusters with three or more members agree to rounding only (tests/test_gpu_kmeans.py checks labels and picks exactly, centres to
1e-9).  The order in which several clusters that became empty in the SAME iteration are re-seeded follows numpy's
argpartition on the device-computed distances, like sklearn.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .ops import EMBEDDING_DTYPES, _cuda, _ptr, _stream, rank_scores


@dataclass
class KMeansResult:
    query_rows: list            # per cluster 0..cluster_num-1: the member closest to its centre (:603)
    labels: torch.Tensor        # (n,) int32
    centers: torch.Tensor       # (k,d) fp64
    n_iter: int
    center_ids: torch.Tensor    # (k,) int32 rows chosen by k-means++
    relocations: int            # empty clusters re-seeded over all iterations


def _i32(n, dev):
    return torch.empty(max(int(n), 1), dtype=torch.int32, device=dev)


def _f64(*shape, dev):
    return torch.empty(shape, dtype=torch.float64, device=dev)


def _x_dtype(t) -> torch.dtype:
    """The dtype `_cuda` checks X against: X's own when the K-Means entries read it, else fp32 (refused as before)."""
    dt = getattr(t, "dtype", None)
    return dt if dt in EMBEDDING_DTYPES else torch.float32


def _call_x(L, name: str, X: torch.Tensor, *args):
    """Call vatlq_kmeans_<name> on X: the fp32 entry for an fp32 X, its _dt form with X's dtype code otherwise."""
    if X.dtype == torch.float32:
        fn, head = name, (_ptr(X),)
    else:
        fn, head = name + "_dt", (_ptr(X), EMBEDDING_DTYPES[X.dtype])
    _lib.check(getattr(L, fn)(*head, *args), fn)


def kmeans_fit_select(X: torch.Tensor, n_clusters: int, sample_weight: torch.Tensor | None = None, random_state: int = 318,
                      max_iter: int = 300, tol: float = 1e-4, group=None, select: bool = True) -> KMeansResult:
    """`KMeans(n_clusters, random_state=random_state).fit_predict(X, sample_weight)` (k-means++ init, n_init = 1,
    Lloyd) + the per-cluster closest member.  X (n,d) CUDA in one of ops.EMBEDDING_DTYPES (a 16-bit X gives, bit for
    bit, the result of X.float()), sample_weight (n,) fp64 CUDA or None.
    group: a torch.distributed group whose ranks all hold the SAME X: the assignment GEMM (the dominant step of a
    Lloyd iteration) is sharded by rows and the labels are all-gathered; seeding and the M step replay identically
    on every rank (deterministic kernels), so every rank returns the same result as a single GPU.
    select=False: the clustering alone (`fit_predict`); query_rows holds -1 for clusters without members instead of
    raising like the reference's per-cluster arg-min does."""
    X = _cuda(X, _x_dtype(X), "X")
    if X.dim() != 2:
        raise _lib.VatlqError("X must be (n,d)")
    n, d = X.shape
    k = int(n_clusters)
    if k < 1:
        raise ValueError(f"The 'n_clusters' parameter of KMeans must be an int in the range [1, inf). Got {k} instead.")
    if n < k:       # sklearn _check_params_vs_input
        raise ValueError(f"n_samples={n} should be >= n_clusters={k}.")
    dev = X.device
    w = None if sample_weight is None else _cuda(sample_weight, torch.float64, "sample_weight")
    if w is not None and w.numel() != n:
        raise _lib.VatlqError("sample_weight must have one entry per row")
    L = _lib.lib()
    st = _stream()
    ws = torch.empty(max(int(L.vatlq_kmeans_workspace_bytes(n, d, k)), 16), dtype=torch.uint8, device=dev)
    wsb = ws.numel()

    # ---- the random stream, consumed exactly like sklearn's _kmeans_plusplus (host: numpy's own generator)
    rs = np.random.RandomState(random_state)
    sw = np.ones(n, dtype=np.float64) if w is None else w.cpu().numpy()
    first = int(rs.choice(n, p=sw / sw.sum()))
    trials = 2 + int(np.log(k))
    rand = rs.uniform(size=max(k - 1, 0) * trials)                 # k-1 successive uniform(size=trials) draws
    rand_d = torch.from_numpy(rand).to(dev) if k > 1 else None
    center_ids, closest = _i32(k, dev), _f64(n, dev=dev)
    with torch.cuda.device(dev):
        tolv, mean = _f64(1, dev=dev), _f64(d, dev=dev)
        _call_x(L, "vatlq_kmeans_mean_var", X, n, d, _ptr(mean), _ptr(tolv), _ptr(ws), wsb, st)
        _call_x(L, "vatlq_kmeans_pp", X, n, d, _ptr(w), k, first, _ptr(rand_d), trials, _ptr(center_ids), _ptr(closest),
                _ptr(ws), wsb, st)
        # centres: `cc` in the centred frame (where sklearn keeps them: X -= X_mean), `centers` = cc + X_mean
        cc, cc_new = _f64(k, d, dev=dev), _f64(k, d, dev=dev)
        centers, centers_new = _f64(k, d, dev=dev), _f64(k, d, dev=dev)
        _call_x(L, "vatlq_kmeans_gather", X, d, _ptr(center_ids), k, _ptr(mean), _ptr(cc), _ptr(centers), st)
        tol_abs = float(tolv.item()) * tol                          # _tolerance: mean(var(X, axis=0)) * tol

        labels = torch.full((n,), -1, dtype=torch.int32, device=dev)
        labels_old = labels.clone()
        sums, wsum, shift = _f64(k, d, dev=dev), _f64(k, dev=dev), _f64(k, dev=dev)
        order, starts = _i32(n, dev), _i32(k + 1, dev)
        flags = torch.zeros(2, dtype=torch.int32, device=dev)       # [changed, n_empty]
        dis = _f64(n, dev=dev)
        strict, n_iter, relocations = False, 0, 0

        world = 1
        if group is not None:
            import torch.distributed as td
            from .dist import allgather_rows, shard_range
            world = td.get_world_size(group)
            lo, hi = shard_range(n, td.get_rank(group), world)

        def assign(into, against, counter):
            if world == 1:
                _call_x(L, "vatlq_kmeans_assign", X, n, d, _ptr(centers), k, _ptr(into), _ptr(against), _ptr(counter),
                        _ptr(ws), wsb, st)
                return
            if hi > lo:                                             # this rank's rows only (in X's own dtype)
                _call_x(L, "vatlq_kmeans_assign", X[lo:hi], hi - lo, d, _ptr(centers), k, _ptr(into[lo:hi]),
                        None if against is None else _ptr(against[lo:hi]), _ptr(counter), _ptr(ws), wsb, st)
            elif counter is not None:
                counter.zero_()
            into[:n].copy_(allgather_rows(into[lo:hi], n, world, group))
            if counter is not None:
                td.all_reduce(counter, op=td.ReduceOp.SUM, group=group)

        def average(argmax_w):
            _lib.check(L.vatlq_kmeans_average(_ptr(sums), _ptr(wsum), k, d, argmax_w, _ptr(mean), _ptr(cc), _ptr(cc_new),
                                              _ptr(centers_new), _ptr(shift), st), "vatlq_kmeans_average")

        for it in range(max_iter):                                  # _kmeans_single_lloyd
            n_iter = it + 1
            assign(labels, labels_old, flags[0:1])
            _call_x(L, "vatlq_kmeans_update", X, n, d, _ptr(w), _ptr(mean), _ptr(labels), k, _ptr(sums), _ptr(wsum), _ptr(order),
                    _ptr(starts), _ptr(flags[1:2]), _ptr(ws), wsb, st)
            average(-1)                                             # the common case: no empty cluster
            changed, n_empty = (int(v) for v in flags.cpu().tolist())
            if n_empty:                                             # _relocate_empty_clusters_dense (rare)
                wsum_h = wsum.cpu().numpy()
                empty = np.where(wsum_h == 0)[0].astype(np.int32)
                _call_x(L, "vatlq_kmeans_rowdist", X, n, d, _ptr(centers), _ptr(labels), _ptr(dis), st)
                dist_h = dis.cpu().numpy()
                far = np.argpartition(dist_h, -len(empty))[:-len(empty) - 1:-1].astype(np.int32)
                if dist_h.max() != 0:
                    e_d, f_d = torch.from_numpy(empty).to(dev), torch.from_numpy(np.ascontiguousarray(far)).to(dev)
                    _call_x(L, "vatlq_kmeans_relocate", X, d, _ptr(w), _ptr(mean), _ptr(labels), _ptr(e_d), _ptr(f_d), len(empty),
                            _ptr(sums), _ptr(wsum), st)
                    relocations += len(empty)
                    wsum_h = wsum.cpu().numpy()
                average(int(np.argmax(wsum_h)) if (wsum_h == 0).any() else -1)
            centers, centers_new = centers_new, centers
            cc, cc_new = cc_new, cc
            if changed == 0:                                        # np.array_equal(labels, labels_old)
                strict = True
                break
            center_shift = shift.cpu().numpy()
            if (center_shift ** 2).sum() <= tol_abs:
                break
            labels, labels_old = labels_old, labels                 # labels_old[:] = labels
        else:
            labels, labels_old = labels_old, labels                 # max_iter reached: the last labels were swapped away
        if not strict:                                              # rerun the E step so labels match the centres
            assign(labels, None, None)

        # ---- per cluster the member closest to its centre (:599-603)
        _call_x(L, "vatlq_kmeans_update", X, n, d, _ptr(w), _ptr(mean), _ptr(labels), k, _ptr(sums), _ptr(wsum), _ptr(order),
                _ptr(starts), _ptr(flags[1:2]), _ptr(ws), wsb, st)
        _call_x(L, "vatlq_kmeans_rowdist", X, n, d, _ptr(centers), _ptr(labels), _ptr(dis), st)
        picks = _i32(k, dev)
        _lib.check(L.vatlq_kmeans_pick(_ptr(dis), _ptr(order), _ptr(starts), k, _ptr(picks), st), "vatlq_kmeans_pick")
        picks_h = picks[:k].cpu().numpy()
    if not select:
        return KMeansResult([int(v) for v in picks_h], labels[:n], centers, n_iter, center_ids[:k], relocations)
    cluster_num = int((picks_h >= 0).sum())                         # len(np.unique(cluster_idxs))
    rows = []
    for i in range(cluster_num):                                    # `for i in range(cluster_num)` of the reference
        if picks_h[i] < 0:                                          # dis[cluster_idxs == i] is empty there too
            raise ValueError("attempt to get argmin of an empty sequence")
        rows.append(int(picks_h[i]))
    return KMeansResult(rows, labels[:n], centers, n_iter, center_ids[:k], relocations)


def unique_rows_first_index(E: torch.Tensor) -> np.ndarray:
    """`np.unique(E, axis=0, return_index=True)[1]`: the first-occurrence index of every distinct row, in
    lexicographic row order (ActiveLearning.py:555).  Rows are ordered on the device by their first column (stable
    radix sort, ties in ascending row order); only runs of rows that share the first column are compared in full,
    on the host, which for embeddings means duplicates.  A 16-bit E gives the indices of E.float(): its first column
    widens exactly to fp64, and the runs go to the host as fp32 (numpy has no bf16)."""
    E = _cuda(E, _x_dtype(E), "E")
    m = E.shape[0]
    if m == 0:
        return np.zeros(0, dtype=np.int64)
    col0 = E[:, 0].to(torch.float64).contiguous()
    order = rank_scores(col0, None, descending=False).cpu().numpy()
    v = col0.cpu().numpy()[order]
    same = np.flatnonzero(v[1:] == v[:-1])
    if same.size == 0:
        return order.astype(np.int64)
    out = []
    run_start = np.flatnonzero(np.r_[True, v[1:] != v[:-1]])
    run_end = np.r_[run_start[1:], m]
    for a, b in zip(run_start, run_end):
        if b - a == 1:
            out.append(int(order[a]))
            continue
        ids = np.sort(order[a:b])                                   # ascending row ids: lexsort is stable on them
        rows = E[torch.as_tensor(ids, device=E.device)].float().cpu().numpy()
        lex = np.lexsort(rows.T[::-1])
        ids, rows = ids[lex], rows[lex]
        keep = np.r_[True, np.any(rows[1:] != rows[:-1], axis=1)]
        out.extend(int(i) for i in ids[keep])
    return np.asarray(out, dtype=np.int64)
