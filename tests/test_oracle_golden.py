"""CPU: the oracle restatement reproduces the reference outputs stored in tests/golden/
(written by oracle/pin_against_reference.py from the reference's own functions)."""
import warnings

import numpy as np
import pytest

from oracle import vatl_oracle as O
from conftest import ae_weights_from_gold


def test_known_answer_local_peak():
    # the only known-answer fragment the reference holds: active_learning/local_peak.py:25-31
    kat = np.array([[0, 0, 0, 0, 0, 0, 0, 4, 0, 0], [0, 0, 0, 1, 1, 0, 0, 0, 0, 0],
                    [0, 0, 0, 0, 3, 2, 0, 0, 0, 0], [0, 0, 0, 0, 2, 2, 0, 0, 0, 0]])
    v = O.localpeak_values(kat)
    assert v.tolist() == [4, 3] and v.min() == 3


def test_scan_matches_reference(gold_scan):
    g = gold_scan
    H, boxes = g["H"], g["boxes"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        for i in range(H.shape[0]):
            xy, _ = O.heatmap_coords(H[i])
            c, v = O.heatmap_to_coord(H[i], boxes[i].tolist())
            assert np.array_equal(xy, g["hm_xy"][i])
            assert np.array_equal(c, g["img_xy"][i])
            assert np.array_equal(v[:, 0], g["maxv"][i])
            assert np.array_equal(np.float32(O.localpeak_mean(H[i])), g["peak"][i], equal_nan=True)
    assert np.array_equal(O.thc_pool(H, g["is_prev"], g["is_next"]), g["thc"])


def test_scan_edge_cases(gold_scan):
    g = gold_scan
    e = 10  # first edge frame (see oracle/pin_against_reference.py::edge_maps)
    assert np.isnan(g["peak"][e + 1])                       # every joint negative -> NaN mean
    assert g["hm_xy"][e][3].tolist() == [0.0, 0.0]          # tie -> first index, corner, no shift
    assert g["hm_xy"][e][1].tolist() == [0.0, 0.0]          # max <= 0 -> coordinates zeroed
    assert g["hm_xy"][e][5].tolist() == [2.25, 2.0]         # dx>0 -> +0.25, dy == 0 -> no shift
    assert g["hm_xy"][e][4].tolist() == [1.0, 1.0]          # px == 1 is not strictly interior
    assert g["thc"][e + 3] == 0.0                           # singleton track
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert O.localpeak_values(g["H"][e][0]).tolist() == [1.0, 1.0, 0.5]   # plateau + 0.5 kept, 0.49 dropped
        assert O.localpeak_values(g["H"][e][1]).size == 0                     # all-negative map
        v0 = O.localpeak_values(g["H"][e][2])                                  # max == 0: exact zeros are kept
        assert v0.size > 1 and (v0 == 0).all()


def test_wpu_matches_reference(gold_wpu):
    g = gold_wpu
    ae = O.make_autoencoder(ae_weights_from_gold(g))
    for i in range(g["kpts"].shape[0]):
        kl = g["kpts"][i].reshape(-1).astype(np.float64)
        box = g["boxes"][i].tolist()
        f = O.hybrid_feature(O.xyxy_to_xywh(box), kl)
        assert np.array_equal(f, g["feat"][i])
        assert O.wpu_item(ae, box, kl, False) == g["wpu42"][i]
        assert O.wpu_item(ae, box, kl.tolist(), True) == g["wpu38"][i]


def test_hybrid_asserts():
    kp = np.ones(51)
    with pytest.raises(AssertionError):
        O.hybrid_feature((0, 0, 10, 0), kp)
    kp[2::3] = 0
    with pytest.raises(AssertionError):
        O.hybrid_feature((0, 0, 10, 10), kp)


def test_fusion_matches_reference(gold_fuse):
    g = gold_fuse
    for mode in ("const", "increase", "decrease"):
        assert np.array_equal(O.fuse_scores(g["thc"], g["wpu"], mode, float(g["ratio"])), g[mode])
    assert np.array_equal(O.fuse_scores(g["thc"]), g["single"])
    assert O.fuse_scores(np.array([3.0])).tolist() == [0.0]


# sklearn's distances are BLAS matrix products, whose last bits depend on the CPU's BLAS kernel and thread count:
# the golden holds the bits of the machine that pinned it, so on another CPU the oracle's distances are compared
# within the rounding of ||x||^2 + ||y||^2 - 2 x.y (d(c,c) ~ 1e-7 from cancellation) and the selections exactly.
BLAS_RTOL, BLAS_ATOL = 1e-9, 1e-6


def test_coreset_matches_reference(gold_coreset):
    for tag, c in gold_coreset.items():
        picks, md = O.coreset_select(c["X"].astype(np.float64), c["unc"].copy(), c["labeled"].tolist(), int(c["k"]),
                                     float(c["moks"]), float(c["lam"]), str(c["rule"]))
        assert picks == c["picks"].tolist(), tag
        assert np.allclose(md, c["min_d"], rtol=BLAS_RTOL, atol=BLAS_ATOL), tag


# ---- SURVEY.md §8f rows: HP / TPC / Entropy, Influence / Diversity / top-k ----------------
def test_next_row_uncertainties_match_reference(gold_next):
    g = gold_next
    H, boxes, ip, inx = g["H"], g["boxes"], g["is_prev"], g["is_next"]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        assert np.array_equal(O.pose_unc_pool(H, boxes, ip, inx, "HP"), g["hp"])
        assert np.array_equal(O.pose_unc_pool(H, boxes, ip, inx, "TPC"), g["tpc"])
        assert np.array_equal(O.pose_unc_pool(H, boxes, ip, inx, "Entropy"), g["entropy_raw"], equal_nan=True)
        Hpos = np.abs(H) + np.float32(1e-3)
        assert np.array_equal(O.pose_unc_pool(Hpos, boxes, ip, inx, "Entropy"), g["entropy_pos"])
    assert np.isneginf(g["entropy_raw"]).all()          # raw maps hold negatives: entr(p<0) = -inf
    assert np.isfinite(g["entropy_pos"]).all()
    assert len(set(g["tpc"].tolist())) > 3


def test_influence_diversity_topk_match_reference(gold_next):
    g = gold_next
    for tag in ("clu", "iid"):
        X = g[f"{tag}_X"].astype(np.float64)
        lab = set(g[f"{tag}_labeled"].tolist())
        unl = [i for i in range(X.shape[0]) if i not in lab]
        k, cw = int(g[f"{tag}_k"]), float(g[f"{tag}_cw"])
        assert np.allclose(O.cosine_rowsum(X[unl]), g[f"{tag}_rowsum"], rtol=1e-13, atol=0)       # (BLAS, see above)
        infl = O.influence_scores(X, unl)
        assert np.allclose(infl, g[f"{tag}_influence"], rtol=0, atol=1e-13)
        assert np.array_equal(O.total_score(g[f"{tag}_unc"], g[f"{tag}_influence"], cw), g[f"{tag}_total"])
        total = O.total_score(g[f"{tag}_unc"], infl, cw)
        assert O.topk_select(unl, total, k) == g[f"{tag}_topk"].tolist()
        assert O.diversity_select(X, unl, total, k) == g[f"{tag}_diversity"].tolist()
    assert O.influence_scores(np.zeros((3, 8)), [1]).tolist() == [0.0]


def test_oks_oracle_matches_reference_golden():
    """al_metric.compute_OKS / get_retrain_id's mOKS (reference outputs in tests/golden/oks.npz)."""
    from conftest import load_golden
    from oracle import vatl_oracle as O
    z = load_golden("oks.npz")
    got = [O.compute_oks(O.xyxy_to_xywh(z["boxes"][i].tolist()), z["kpts"][i].reshape(-1).tolist(), z["gt"][i].reshape(-1).tolist())
           for i in range(len(z["oks"]))]
    assert np.array_equal(np.array(got), z["oks"])
    assert z["oks"][7] == 1.0 and z["oks"][4] < 1e-3
    assert O.mean_oks_of_queries(z["query"].tolist(), dict(enumerate(z["oks"].tolist()))) == float(z["moks"])
