#!/usr/bin/env python
"""Pin `oracle/vatl_oracle.py` against the reference itself and write tests/golden/*.npz.

Runs ONLY in the build container (needs /root/reference).  It imports the reference's own
functions with the import-stub recipe of SURVEY.md §8c, feeds them seeded inputs and the
edge-case vectors of SURVEY.md §8a, checks that the oracle restatement reproduces every
output bit-for-bit, and stores inputs + REFERENCE outputs as golden fixtures.  The
fixtures travel to the GPU box; /root/reference does not.

    python oracle/pin_against_reference.py            # verify + (re)write fixtures
"""
from __future__ import annotations

import importlib
import os
import sys
import warnings
from types import SimpleNamespace
from unittest.mock import MagicMock

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("VATL_REFERENCE", "/root/reference")
GOLD = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)

from oracle import golden_inputs as GI  # noqa: E402  (the heat maps and features are rebuilt, not stored)


def import_reference():
    sys.path[:0] = [REF, os.path.join(REF, "ALiPy")]
    for name in ("matplotlib", "matplotlib.pyplot", "matplotlib.ticker", "matplotlib.colors",
                 "skimage", "skimage.feature", "seaborn", "umap", "annoy", "easydict",
                 "pycocotools", "pycocotools.coco", "pycocotools.cocoeval", "optuna",
                 "prettytable", "cachetools"):
        try:
            importlib.import_module(name)
        except Exception:
            sys.modules[name] = MagicMock()
    import active_learning  # noqa: F401  (reference package)
    from active_learning import ActiveLearning as AL
    from active_learning.local_peak import localpeak_mean, localpeak_values
    from active_learning.Whole_body_AE.hybrid_feature import compute_hybrid
    from active_learning.Whole_body_AE.AutoEncoder import WholeBodyAE
    from alphapose.utils.transforms import heatmap_to_coord_simple, get_max_pred
    from alphapose.utils.bbox import bbox_xyxy_to_xywh
    from alipy.index import IndexCollection
    return SimpleNamespace(AL=AL, localpeak_mean=localpeak_mean, localpeak_values=localpeak_values,
                           compute_hybrid=compute_hybrid, WholeBodyAE=WholeBodyAE,
                           heatmap_to_coord_simple=heatmap_to_coord_simple, get_max_pred=get_max_pred,
                           bbox_xyxy_to_xywh=bbox_xyxy_to_xywh, IndexCollection=IndexCollection)


def same(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(a, b, equal_nan=True), (what, np.abs(a.astype(np.float64) - b).max())


def ref_autoencoder(R, weights):
    """WholeBodyAE(z_dim) with first/last layers resized to the weights' in_dim (the call site
    feeds 42-d features although AutoEncoder.py:12 says 38; SURVEY.md §8c caveat)."""
    import torch
    import torch.nn as nn
    import io, contextlib
    z = weights[3][0].shape[0]
    with contextlib.redirect_stdout(io.StringIO()):
        ae = R.WholeBodyAE(z_dim=z)
    ind = weights[0][0].shape[1]
    ae.encoder[0] = nn.Linear(ind, 24)
    ae.decoder[6] = nn.Linear(24, ind)
    lin = [m for m in list(ae.encoder) + list(ae.decoder) if isinstance(m, nn.Linear)]
    with torch.no_grad():
        for m, (W, b) in zip(lin, weights):
            m.weight.copy_(torch.from_numpy(W))
            m.bias.copy_(torch.from_numpy(b))
    return ae.eval()


def pin_next_rows(R, O, synth):
    """SURVEY.md §8f rows: HP / TPC / Entropy (reference methods compute_tpc / compute_entropy
    called unbound; the HP expression of :330 evaluated as written), Influence / Diversity /
    top-k (the sklearn calls of :469-477, :527-540, :581-590 evaluated as written)."""
    from sklearn.neighbors import KNeighborsTransformer
    H, ip, inx, boxes, rng = GI.next_inputs()
    n = H.shape[0]
    fake = SimpleNamespace(heatmap_to_coord=R.heatmap_to_coord_simple, eval_joints=list(range(17)),
                           hm_size=[64, 48], norm_type=None)
    hp_ref, tpc_ref, ent_ref, ent_pos_ref = [], [], [], []
    Hpos = np.abs(H) + np.float32(1e-3)          # a non-negative pool: finite entropies
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for i in range(n):
            box = boxes[i].tolist()
            pose_coords, pose_scores = R.heatmap_to_coord_simple(H[i], box)
            hp_ref.append(float(-np.sum(pose_scores)))                                   # :330
            thresh = 0.01 * np.sqrt((box[2] - box[0]) * (box[3] - box[1]))               # :334
            tpc = 0
            has_p, has_n = bool(ip[i]) and i > 0, bool(inx[i]) and i < n - 1
            if has_p:
                tpc += R.AL.compute_tpc(fake, pose_coords, H[i - 1], box, thresh)
            if has_n:
                tpc += R.AL.compute_tpc(fake, pose_coords, H[i + 1], box, thresh)
                if not has_p:
                    tpc *= 2
            elif has_p:
                tpc *= 2
            tpc_ref.append(float(tpc))
            ent_ref.append(float(R.AL.compute_entropy(fake, H[i])))
            ent_pos_ref.append(float(R.AL.compute_entropy(fake, Hpos[i])))
        same(hp_ref, O.pose_unc_pool(H, boxes, ip, inx, "HP"), "HP")
        same(tpc_ref, O.pose_unc_pool(H, boxes, ip, inx, "TPC"), "TPC")
        same(ent_ref, O.pose_unc_pool(H, boxes, ip, inx, "Entropy"), "Entropy raw")
        same(ent_pos_ref, O.pose_unc_pool(Hpos, boxes, ip, inx, "Entropy"), "Entropy positive")
    assert len(set(tpc_ref)) > 3, tpc_ref

    # Influence / Diversity / top-k on clustered and i.i.d. embeddings
    out = dict(boxes=boxes, is_prev=ip, is_next=inx, hp=np.array(hp_ref), tpc=np.array(tpc_ref),
               entropy_raw=np.array(ent_ref), entropy_pos=np.array(ent_pos_ref))
    for tag, clustered in (("clu", True), ("iid", False)):
        N, k = 400, 20
        X32 = GI.next_features(clustered)
        X = X32.astype(np.float64)
        lab = sorted(rng.choice(N, 60, replace=False).tolist())
        unl = [i for i in range(N) if i not in set(lab)]
        unc_score = rng.uniform(0, 1, len(unl))
        cw = 0.37
        knn = KNeighborsTransformer(mode="distance", metric="cosine", n_neighbors=len(unl) - 1)   # :471
        infl = np.asarray(np.sum(knn.fit_transform(X[unl]), axis=1)).flatten()                  # :472-473
        rowsum_ref = infl.copy()
        infl = (infl - np.min(infl)) / (np.max(infl) - np.min(infl))                            # :475
        same(infl, O.influence_scores(X, unl), f"influence {tag}")
        total = cw * unc_score + (1 - cw) * infl                                                # :519
        same(total, O.total_score(unc_score, infl, cw), f"total {tag}")
        score_dict = dict((idx, sc) for idx, sc in zip(unl, total))                              # :527
        srt = sorted(score_dict.items(), key=lambda x: x[1], reverse=True)                       # :529
        score_dict = dict((int(idx), sc) for idx, sc in srt)
        top_ref = sorted(list(score_dict.keys())[:k])                                            # :534
        same(top_ref, O.topk_select(unl, total, k), f"topk {tag}")
        cand = sorted(list(score_dict.keys())[:8 * k])                                           # :538
        knn = KNeighborsTransformer(mode="distance", metric="cosine", n_neighbors=len(cand) - 1)  # :583
        div = np.asarray(np.sum(knn.fit_transform(X[cand]), axis=1)).flatten()
        dd = dict((idx, sc) for idx, sc in zip(cand, div))
        dd = dict((int(idx), sc) for idx, sc in sorted(dd.items(), key=lambda x: x[1]))          # :587-588
        div_ref = list(dd.keys())[:k]                                                            # :589
        same(div_ref, O.diversity_select(X, unl, total, k), f"diversity {tag}")
        out.update({f"{tag}_labeled": np.array(lab, np.int64), f"{tag}_unc": unc_score,
                    f"{tag}_cw": np.float64(cw), f"{tag}_k": np.int64(k), f"{tag}_rowsum": rowsum_ref,
                    f"{tag}_influence": infl, f"{tag}_total": total, f"{tag}_topk": np.array(top_ref, np.int64),
                    f"{tag}_div_rowsum": div, f"{tag}_diversity": np.array(div_ref, np.int64)})
    np.savez_compressed(os.path.join(GOLD, "next.npz"), **out)


def pin_oks(R, O, synth):
    """OKS (active_learning/al_metric.py:42-69, call site ActiveLearning.py:309) and the mOKS of a query list
    (get_retrain_id, :852-858): the reference's functions on seeded poses, incl. the no-visible-joint branch."""
    from active_learning.al_metric import compute_OKS
    rng = np.random.default_rng(17)
    n = 96
    kp, bb = synth.poses(n, seed=3)
    gt = kp.copy()
    gt[:, :, :2] += rng.normal(0, 8.0, (n, 17, 2)).astype(np.float32)
    gt[:, :, 2] = (rng.random((n, 17)) < 0.75).astype(np.float32) * 2
    gt[3, :, 2] = 0                      # nothing visible: distance to the doubled box
    gt[4, :, 2] = 0; kp[4, :, 0] += 900   # ... with predictions far outside it
    gt[7] = kp[7]; gt[7, :, 2] = 1       # perfect prediction -> 1.0
    ref = []
    for i in range(n):
        box = R.bbox_xyxy_to_xywh(bb[i].tolist())
        k = kp[i].reshape(-1).tolist()
        g = gt[i].reshape(-1).tolist()
        ref.append(float(compute_OKS(box, k, g)))
        same(ref[-1], float(O.compute_oks(O.xyxy_to_xywh(bb[i].tolist()), k, g)), f"oks {i}")
    oks_dict = dict(enumerate(ref))
    q = sorted(rng.choice(n, 20, replace=False).tolist())
    fake = SimpleNamespace(labeled_id=R.IndexCollection([1, 2, 3]), unlabeled_id=R.IndexCollection(list(range(4, n))),
                           finish_acc=0.8, finish_margin=0.05)
    import io, contextlib
    with contextlib.redirect_stdout(io.StringIO()):
        retrain_ref, moks_ref = R.AL.get_retrain_id(fake, q, oks_dict)
    same(moks_ref, O.mean_oks_of_queries(q, oks_dict), "mOKS of the queries")
    np.savez_compressed(os.path.join(GOLD, "oks.npz"), kpts=kp, gt=gt, boxes=bb, oks=np.array(ref), query=np.array(q, np.int64),
                        moks=np.float64(moks_ref), retrain=np.array(retrain_ref, np.int64))
    print("OKS pinned:", len(ref), "items, mOKS", moks_ref)


def pin_peaks(R, O, synth):
    """MPE / Margin: the reference's compute_mpe / compute_margin (ActiveLearning.py:762-788) called unbound, with
    the RESTATED peak_local_max standing in for skimage.feature.peak_local_max (scikit-image is not installed
    here: the restatement's parity with the library is unpinned; everything around it is the reference's code)."""
    sys.modules["active_learning.ActiveLearning"].peak_local_max = O.peak_local_max   # (the module, not the class)
    H = GI.peaks_inputs()
    fake = SimpleNamespace()
    mpe = np.array([float(R.AL.compute_mpe(fake, H[i])) for i in range(len(H))])
    mar = np.array([float(R.AL.compute_margin(fake, H[i])) for i in range(len(H))])
    same(mpe, [O.mpe_item(H[i]) for i in range(len(H))], "MPE")
    same(mar, [O.margin_item(H[i]) for i in range(len(H))], "Margin")
    np.savez_compressed(os.path.join(GOLD, "peaks.npz"), mpe=mpe, margin=mar)
    print("MPE / Margin pinned (peak_local_max restated):", mpe[:3], mar[:3])


def _reference_branch(src_lines, head):
    """The statements of one `elif self.filter==...:` branch of eval_and_query, de-indented, as a code object."""
    import textwrap
    start = next(i for i, l in enumerate(src_lines) if l.strip().startswith(head))
    ind = len(src_lines[start]) - len(src_lines[start].lstrip())
    body = []
    for l in src_lines[start + 1:]:
        if l.strip() and (len(l) - len(l.lstrip())) <= ind:
            break
        body.append(l)
    return compile(textwrap.dedent("".join(body)), f"<reference {head}>", "exec")


def kmeans_cases(synth):
    """(tag, X fp32 (n,2048), candidate_list, total_score over the candidates, query_size, w_unc, combine_weight)."""
    out = []
    for tag, kind, n, n_lab, k, seed in (("clustered", "clustered", 600, 60, 27, 2), ("weak", "weak", 900, 0, 45, 4),
                                         ("iid", "iid", 500, 100, 20, 5), ("pairs", "iid", 240, 0, 150, 6),
                                         ("one", "clustered", 200, 0, 1, 7), ("all", "weak", 64, 0, 64, 8)):
        X = synth.pool_embeddings(n, kind=kind, seed=seed)
        lab = set(synth.pool_labeled(n, n_lab, seed=seed).tolist())
        cand = [i for i in range(n) if i not in lab]
        score = synth.pool_unc(n, seed=seed)[cand]
        out.append((tag, dict(kind=kind, n=n, n_lab=n_lab, seed=seed, dup=np.zeros(0, np.int64)), X, cand, score, k, 0.7, 0.35))
    # duplicated rows (np.unique has work to do; two-member clusters of identical rows)
    n, seed = 400, 9
    X = synth.pool_embeddings(n, kind="iid", seed=seed)
    dup = np.arange(100, 160)
    X[dup] = X[dup - 100]
    cand = list(range(n))
    out.append(("dups", dict(kind="iid", n=n, n_lab=0, seed=seed, dup=dup), X, cand, synth.pool_unc(n, seed=seed), 120, 1.3, 0.5))
    return out


def pin_kmeans(R, O, synth):
    """K-Means / weighted filters: the reference's OWN statements (ActiveLearning.py:553-580 and :593-608, taken
    from the source file and executed here) against the oracle restatement; sklearn is the same library call in
    both.  Golden: pool parameters (the pools are counter-based), labels and query lists."""
    from sklearn.cluster import KMeans
    with open(os.path.join(REF, "active_learning", "ActiveLearning.py")) as fh:
        src = fh.readlines()
    code = {"K-Means": _reference_branch(src, 'elif self.filter=="K-Means":'),
            "weighted": _reference_branch(src, 'elif self.filter=="weighted":')}
    gold = {}
    for tag, meta, X, cand, score, k, w_unc, cw in kmeans_cases(synth):
        fvecs = X.astype(np.float64)                           # fvecs_matrix is float64 (:270)
        for filt in ("K-Means", "weighted"):
            me = SimpleNamespace(unlabeled_id=SimpleNamespace(index=list(cand)), query_size=k, plot_cluster=False, w_unc=w_unc)
            env = dict(np=np, KMeans=KMeans, self=me, fvecs_matrix=fvecs, candidate_list=list(cand),
                       track_ids_list=np.zeros(len(fvecs)), total_score=score.copy(), combine_weight=cw)
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                exec(code[filt], env)
                if filt == "K-Means":
                    q, qs, lab = O.kmeans_filter(fvecs, cand, k)
                    eidx = np.zeros(0, np.int64)
                else:
                    q, qs, lab, eidx = O.weighted_kmeans_filter(fvecs, cand, score, w_unc, cw, k)
            assert env["query_list"] == q, (tag, filt)
            assert me.query_size == qs, (tag, filt)
            same(env["cluster_idxs"], lab, f"kmeans labels {tag} {filt}")
            key = f"{tag}_{'km' if filt == 'K-Means' else 'wk'}"
            gold[key + "_query"] = np.asarray(q, np.int64)
            gold[key + "_labels"] = np.asarray(lab, np.int32)
            gold[key + "_embed_idx"] = np.asarray(eidx, np.int64)
            gold[key + "_qsize"] = np.int64(qs)
            gold[key + "_niter"] = np.int64(env["cluster_learner"].n_iter_)
        gold[tag + "_meta"] = np.array([meta["n"], meta["n_lab"], meta["seed"], k], np.int64)
        gold[tag + "_kind"] = np.array(meta["kind"])
        gold[tag + "_dup"] = meta["dup"]
        gold[tag + "_w"] = np.array([w_unc, cw])
        print("K-Means / weighted pinned:", tag, len(gold[tag + "_km_query"]), len(gold[tag + "_wk_query"]))
    np.savez_compressed(os.path.join(GOLD, "kmeans.npz"), **gold)


def main():
    if len(sys.argv) > 1 and sys.argv[1] == "kmeans":
        from oracle import vatl_oracle as O
        pin_kmeans(import_reference(), O, importlib.import_module("vatl4pose-wacv2024_b200.synth"))
        return
    if len(sys.argv) > 1 and sys.argv[1] == "peaks":
        from oracle import vatl_oracle as O
        pin_peaks(import_reference(), O, importlib.import_module("vatl4pose-wacv2024_b200.synth"))
        return
    if len(sys.argv) > 1 and sys.argv[1] == "oks":     # only the OKS fixture (the others are unchanged)
        from oracle import vatl_oracle as O
        pin_oks(import_reference(), O, importlib.import_module("vatl4pose-wacv2024_b200.synth"))
        return
    from oracle import vatl_oracle as O
    synth = importlib.import_module("vatl4pose-wacv2024_b200.synth")
    R = import_reference()
    os.makedirs(GOLD, exist_ok=True)
    ns = SimpleNamespace()

    # ---------------- known-answer fragment of local_peak.py:25-31 -------------------
    kat = np.array([[0, 0, 0, 0, 0, 0, 0, 4, 0, 0], [0, 0, 0, 1, 1, 0, 0, 0, 0, 0],
                    [0, 0, 0, 0, 3, 2, 0, 0, 0, 0], [0, 0, 0, 0, 2, 2, 0, 0, 0, 0]])
    same(R.localpeak_values(kat), [4, 3], "KAT ref")
    same(O.localpeak_values(kat), [4, 3], "KAT oracle")

    # ---------------- scan: coords / maxvals / THC / peak mean ------------------------
    H, ip, inx, boxes = GI.scan_inputs()
    n = H.shape[0]
    ref = {"hm_xy": [], "img_xy": [], "maxv": [], "peak": [], "thc": [], "thc3": []}
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for i in range(n):
            box = boxes[i].tolist()
            c_ref, v_ref = R.heatmap_to_coord_simple(H[i], box)
            c_or, v_or = O.heatmap_to_coord(H[i], box)
            same(c_ref, c_or, f"img coords {i}"); same(v_ref, v_or, f"maxvals {i}")
            hm_xy, _ = O.heatmap_coords(H[i])
            p0, _ = R.get_max_pred(H[i]); q0, _ = O.max_pred(H[i]); same(p0, q0, f"max_pred {i}")
            ref["hm_xy"].append(hm_xy); ref["img_xy"].append(c_ref); ref["maxv"].append(v_ref[:, 0])
            pm_ref = R.localpeak_mean(H[i]); pm_or = O.localpeak_mean(H[i])
            same(np.float32(pm_ref), np.float32(pm_or), f"peak mean {i}")
            for j in range(17):
                same(R.localpeak_values(H[i][j]), O.localpeak_values(H[i][j]), f"peaks {i},{j}")
            ref["peak"].append(np.float32(pm_ref))
            # reference call-site logic ActiveLearning.py:345-363 with pool neighbours
            thc = 0
            if ip[i] and i > 0:
                thc += R.AL.compute_thc(ns, H[i], H[i - 1], norm_type="L1")
            if inx[i] and i < n - 1:
                thc += R.AL.compute_thc(ns, H[i], H[i + 1], norm_type="L1")
                if not (ip[i] and i > 0):
                    thc *= 2
            elif ip[i] and i > 0:
                thc *= 2
            ref["thc"].append(float(thc))
    thc_or = O.thc_pool(H, ip, inx)
    same(ref["thc"], thc_or, "thc pool")
    np.savez_compressed(os.path.join(GOLD, "scan.npz"), boxes=boxes, is_prev=ip, is_next=inx,
                        hm_xy=np.stack(ref["hm_xy"]), img_xy=np.stack(ref["img_xy"]),
                        maxv=np.stack(ref["maxv"]), peak=np.array(ref["peak"], np.float32),
                        thc=np.array(ref["thc"], np.float64))

    # ---------------- WPU -------------------------------------------------------------
    import torch
    W = synth.ae_weights(42, 4, seed=318)
    ae_ref = ref_autoencoder(R, W)
    ae_or = O.make_autoencoder(W)
    kp, bb = synth.poses(64, seed=1)
    # also poses that came out of the coord stage (float32 image coords + heat-map scores)
    kp2 = np.concatenate([np.stack(ref["img_xy"][:10]), np.stack(ref["maxv"][:10])[..., None]], axis=2)
    # keep scores positive for the reference's assert (sum(scores) > 0)
    kp = np.concatenate([kp, kp2.astype(np.float32)], axis=0)
    bb = np.concatenate([bb, boxes[:10]], axis=0)
    crit = torch.nn.MSELoss()
    feats, wpu42, wpu38 = [], [], []
    for i in range(kp.shape[0]):
        kl = kp[i].reshape(-1).astype(np.float64).tolist()
        box = R.bbox_xyxy_to_xywh(bb[i].tolist())
        f_ref = R.compute_hybrid(box, np.array(kl))
        f_or = O.hybrid_feature(O.xyxy_to_xywh(bb[i].tolist()), np.array(kl))
        same(f_ref, f_or, f"hybrid {i}")
        same(R.compute_hybrid(box, kl), O.hybrid_feature(O.xyxy_to_xywh(bb[i].tolist()), kl), f"hybrid list {i}")
        with torch.no_grad():
            u = torch.tensor(f_ref).float()
            r = ae_ref(u)
            w42 = float(crit(r, u))                                   # ActiveLearning.py:368-370
            a, b = u.numpy(), r.numpy()                               # :378-386
            a = np.concatenate([a[:3], a[5:20], a[22:]]); b = np.concatenate([b[:3], b[5:20], b[22:]])
            w38 = float(crit(torch.tensor(b).float(), torch.tensor(a).float()))
        same(w42, O.wpu_item(ae_or, bb[i].tolist(), np.array(kl), False), f"wpu42 {i}")
        same(w38, O.wpu_item(ae_or, bb[i].tolist(), kl, True), f"wpu38 {i}")
        feats.append(f_ref); wpu42.append(w42); wpu38.append(w38)
    np.savez_compressed(os.path.join(GOLD, "wpu.npz"), kpts=kp, boxes=bb,
                        feat=np.stack(feats), wpu42=np.array(wpu42), wpu38=np.array(wpu38),
                        **{f"W{k}": w for k, (w, _) in enumerate(W)},
                        **{f"b{k}": b for k, (_, b) in enumerate(W)})

    # ---------------- fusion ----------------------------------------------------------
    rng = np.random.default_rng(5)
    t_u, w_u = rng.uniform(0, 40, 57), rng.uniform(0, 0.2, 57)

    def ref_fuse(t, w, mode, ratio):       # transcription-free: evaluate the reference formulas
        a = (t - np.min(t)) / (np.max(t) - np.min(t))
        b = (w - np.min(w)) / (np.max(w) - np.min(w))
        u = {"const": a + b, "increase": ratio * a + (1 - ratio) * b,
             "decrease": (1 - ratio) * a + ratio * b}[mode]
        return (u - np.min(u)) / (np.max(u) - np.min(u))
    fused = {m: ref_fuse(t_u, w_u, m, 0.15) for m in ("const", "increase", "decrease")}
    for m in fused:
        same(fused[m], O.fuse_scores(t_u, w_u, m, 0.15), f"fuse {m}")
    np.savez_compressed(os.path.join(GOLD, "fuse.npz"), thc=t_u, wpu=w_u, ratio=0.15, **fused,
                        single=O.fuse_scores(t_u))

    # ---------------- core-set --------------------------------------------------------
    cases = {}

    def run_coreset(tag, X32, unc, labeled, k, moks, lam, rule="w_unc", fixed=False, unc_name="THC+WPU"):
        X = X32.astype(np.float64)
        fake = SimpleNamespace(labeled_id=R.IndexCollection(list(labeled)), moks_queried=moks,
                               unc_lambda=lam, uncertainty=unc_name,
                               cfg=SimpleNamespace(VAL=SimpleNamespace(UNC_LAMBDA=lam)),
                               opt=SimpleNamespace(fixed_lambda=fixed), query_size=k)
        import io, contextlib
        with contextlib.redirect_stderr(io.StringIO()):
            picks_ref = R.AL.coreset_selection(fake, X, unc.copy())
        picks_or, md = O.coreset_select(X, unc.copy(), labeled, k, moks, lam, rule)
        same(picks_ref, picks_or, f"coreset {tag}")
        cases[tag] = dict(unc=unc, labeled=np.array(list(labeled), np.int64), k=k, moks=moks,
                          lam=lam, rule=rule, picks=np.array(picks_ref, np.int64), min_d=md)

    rng = np.random.default_rng(3)
    F = GI.coreset_features()
    Xc, Xi, Xd = F["clustered_round0"], F["iid_round0_moks"], F["duplicates"]
    unc_c, unc_i = rng.uniform(0, 1, 600), rng.uniform(0, 1, 500)
    lab20 = sorted(rng.choice(600, 120, replace=False).tolist())
    run_coreset("clustered_round0", Xc, unc_c, [], 60, 0.0, 0.01)
    run_coreset("clustered_lab20", Xc, np.where(np.isin(np.arange(600), lab20), 0.0, unc_c), lab20, 60, 0.6, 0.01)
    run_coreset("iid_round0_moks", Xi, unc_i, [], 50, 0.6, 0.01)
    run_coreset("iid_fixed_lambda", Xi, unc_i, [3, 77, 200], 40, 0.3, 0.01, rule="fixed_lambda", fixed=True)
    run_coreset("iid_dist_only", Xi, unc_i, [5, 9], 40, 0.3, 0.0, rule="dist")
    run_coreset("duplicates", Xd, unc_i, [0], 60, 0.5, 0.01)
    run_coreset("zero_unc", Xc, np.zeros(600), [7], 40, 0.6, 0.01)
    run_coreset("d2048", F["d2048"], rng.uniform(0, 1, 160), [], 30, 0.6, 0.01)
    flat = {}
    for tag, c in cases.items():
        for key, val in c.items():
            flat[f"{tag}/{key}"] = np.asarray(val)
    np.savez_compressed(os.path.join(GOLD, "coreset.npz"), **flat)
    pin_next_rows(R, O, synth)
    pin_oks(R, O, synth)
    pin_peaks(R, O, synth)
    pin_kmeans(R, O, synth)
    print("oracle pinned against the reference; fixtures written to", GOLD)
    for fn in sorted(os.listdir(GOLD)):
        print(f"  {fn}: {os.path.getsize(os.path.join(GOLD, fn)) / 1e6:.2f} MB")


if __name__ == "__main__":
    main()
