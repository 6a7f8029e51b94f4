"""GPU parity of the SURVEY.md §8f rows — HP / TPC / Entropy uncertainties, Influence / Diversity
scores and the top-k / Diversity selections — against the reference outputs in tests/golden/next.npz
(written by oracle/pin_against_reference.py) and against the oracle on larger seeded pools."""
import warnings
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

RTOL = 1e-5   # north_star: scores within 1e-5 relative; counts / indices bit-exact


def _scan(v, H, boxes, ip, inx):
    Hd = torch.from_numpy(H).cuda()
    r = v.ops.heatmap_scan(Hd, ip, inx, torch.from_numpy(boxes).cuda())
    return Hd, r


def test_hp_tpc_match_reference(built_lib, gold_next):
    v, g = built_lib, gold_next
    H, boxes, ip, inx = g["H"], g["boxes"], g["is_prev"], g["is_next"]
    _, r = _scan(v, H, boxes, ip, inx)
    hp, tpc = v.ops.pose_uncertainty(r.coords_hm, r.kpts, torch.from_numpy(boxes).cuda(), ip, inx)
    assert np.array_equal(hp.cpu().numpy().astype(np.float64), g["hp"])        # fp32 sum in numpy's order
    assert np.array_equal(tpc.cpu().numpy().astype(np.float64), g["tpc"])      # integer counts


def test_tpc_halo_equals_whole_pool(built_lib, gold_next):
    """Splitting the pool in two ranges with one-frame halo coordinates changes nothing."""
    v, g = built_lib, gold_next
    H, boxes, ip, inx = g["H"], g["boxes"], g["is_prev"], g["is_next"]
    n = H.shape[0]
    _, r = _scan(v, H, boxes, ip, inx)
    bb = torch.from_numpy(boxes).cuda()
    for cut in (1, 5, n - 1):
        a = v.ops.pose_uncertainty(r.coords_hm[:cut], r.kpts[:cut], bb[:cut], ip[:cut], inx[:cut],
                                   halo_next_xy=r.coords_hm[cut])[1]
        b = v.ops.pose_uncertainty(r.coords_hm[cut:], r.kpts[cut:], bb[cut:], ip[cut:], inx[cut:],
                                   halo_prev_xy=r.coords_hm[cut - 1])[1]
        assert np.array_equal(torch.cat([a, b]).cpu().numpy().astype(np.float64), g["tpc"])


def test_entropy_matches_reference(built_lib, gold_next):
    v, g = built_lib, gold_next
    H = g["H"]
    e_raw = v.ops.heatmap_entropy(torch.from_numpy(H).cuda()).cpu().numpy()
    assert np.array_equal(e_raw.astype(np.float64), g["entropy_raw"])          # -inf: maps hold negatives
    Hpos = np.abs(H) + np.float32(1e-3)
    e_pos = v.ops.heatmap_entropy(torch.from_numpy(Hpos).cuda()).cpu().numpy()
    assert np.allclose(e_pos, g["entropy_pos"], rtol=RTOL, atol=0)
    # generic map shape (not 64x48) and an all-zero map (0/0 -> NaN like scipy)
    rng = np.random.default_rng(3)
    G = rng.uniform(0, 1, (5, 3, 10, 14)).astype(np.float32)
    G[2, 1] = 0
    from oracle import vatl_oracle as O
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref = np.array([O.entropy_item(G[i]) for i in range(5)])
    got = v.ops.heatmap_entropy(torch.from_numpy(G).cuda()).cpu().numpy()
    assert np.isnan(ref[2]) and np.isnan(got[2])
    ok = ~np.isnan(ref)
    assert np.allclose(got[ok], ref[ok], rtol=RTOL, atol=0)


@pytest.mark.parametrize("tag", ["clu", "iid"])
def test_influence_diversity_topk_match_reference(built_lib, gold_next, tag):
    v, g = built_lib, gold_next
    X32 = g[f"{tag}_X"]
    n = X32.shape[0]
    lab = set(g[f"{tag}_labeled"].tolist())
    unl = [i for i in range(n) if i not in lab]
    k, cw = int(g[f"{tag}_k"]), float(g[f"{tag}_cw"])
    X = torch.from_numpy(X32).cuda()
    rows = torch.tensor(unl, dtype=torch.int64, device="cuda")
    rs = v.ops.cosine_rowsum(X, rows=rows)
    assert np.allclose(rs.cpu().numpy(), g[f"{tag}_rowsum"], rtol=1e-10, atol=0)
    infl = v.ops.minmax_f64(rs)
    assert np.allclose(infl.cpu().numpy(), g[f"{tag}_influence"], rtol=0, atol=1e-9)
    # the blend of :519 is one IEEE op per step: bit-exact given the reference's own inputs
    tot = v.ops.blend_scores(torch.from_numpy(g[f"{tag}_unc"]).cuda(), torch.from_numpy(g[f"{tag}_influence"]).cuda(), cw)
    assert np.array_equal(tot.cpu().numpy(), g[f"{tag}_total"])
    # selections from the device-computed influence
    tot = v.ops.blend_scores(torch.from_numpy(g[f"{tag}_unc"]).cuda(), infl, cw).cpu().numpy()
    order = sorted(range(len(unl)), key=lambda t: tot[t], reverse=True)
    assert sorted(unl[t] for t in order[:k]) == g[f"{tag}_topk"].tolist()
    cand = sorted(unl[t] for t in order[:8 * k])
    div = v.ops.cosine_rowsum(X, rows=torch.tensor(cand, dtype=torch.int64, device="cuda")).cpu().numpy()
    assert np.allclose(div, g[f"{tag}_div_rowsum"], rtol=1e-10, atol=0)
    by_div = sorted(range(len(cand)), key=lambda t: div[t])
    assert [cand[t] for t in by_div[:k]] == g[f"{tag}_diversity"].tolist()


def test_cosine_rowsum_full_width_and_zero_rows(built_lib):
    """d = 2048 (the estimator's width), all rows (no index list), zero rows kept as zeros like
    sklearn's normalize, against the O(m^2 d) sklearn graph."""
    from oracle import vatl_oracle as O
    v = built_lib
    X32 = v.synth.embeddings(700, d=2048, seed=9, clustered=True)
    X32[13] = 0
    X32[500] = 0
    ref = O.cosine_rowsum(X32.astype(np.float64))
    got = v.ops.cosine_rowsum(torch.from_numpy(X32).cuda()).cpu().numpy()
    assert np.allclose(got, ref, rtol=1e-10, atol=0)
    Z = torch.zeros((6, 64), device="cuda")               # the reference's all-zero fvecs_matrix (:270,283)
    assert v.ops.cosine_rowsum(Z).cpu().tolist() == [5.0] * 6                 # distance 1 to the others, 0 to itself
    assert O.cosine_rowsum(np.zeros((6, 64))).tolist() == [5.0] * 6


class FakeEstimator(torch.nn.Module):
    def __init__(self, H, X):
        super().__init__()
        self.H, self.X = H, X

    def forward(self, crops):
        return self.H[crops[:, 0, 0, 0].long()]

    def get_embedding(self, crops):
        return self.X[crops[:, 0, 0, 0].long()]


def _loader(n, boxes, ip, inx, bs):
    for a in range(0, n, bs):
        b = min(n, a + bs)
        inps = torch.zeros((b - a, 3, 1, 2, 2))
        inps[:, :, 0, 0, 0] = torch.arange(a, b, dtype=torch.float32)[:, None]
        yield (list(range(a, b)), inps, None, None, None, None, None, boxes[a:b], boxes[a:b], ip[a:b], inx[a:b])


def _cfg_opt(unc, rep, flt):
    cfg = SimpleNamespace(VAL=SimpleNamespace(QUERY_RATIO=[0.05, 0.1, 0.2], W_UNC=1.0, UNC_LAMBDA=0.01),
                          DATA_PRESET=SimpleNamespace(HEATMAP_SIZE=[64, 48]), AE=SimpleNamespace(Z_DIM=4))
    opt = SimpleNamespace(strategy=f"{unc}+{rep}_{flt}filter", uncertainty=unc, representativeness=rep, filter=flt,
                          video_id="0", THCvsWPU="const", fixed_lambda=False, onebyone=False)
    return cfg, opt


@pytest.mark.parametrize("unc,rep,flt", [("HP", "None", "None"), ("TPC", "Influence", "Diversity"),
                                         ("THC", "Influence", "None"), ("None", "Influence", "Coreset"),
                                         ("HP", "Random", "Random"), ("Entropy", "None", "None")])
def test_controller_next_strategies_match_oracle(built_lib, unc, rep, flt):
    """Two AL rounds through the reference-shaped controller with the newly accelerated strategy
    names, against the oracle pipeline (chunked scoring: 50 items per loader batch)."""
    from oracle import vatl_oracle as O
    v = built_lib
    n = 160
    ids, ip, inx = v.synth.track_flags(n, np.random.default_rng(4), 8.0)
    H = v.synth.heatmaps(n, seed=4, track_ids=ids)
    rng = np.random.default_rng(5)
    for i in range(1, n):                      # TPC that discriminates (see the pin script)
        if ip[i] and rng.uniform() < 0.7:
            H[i] = H[i - 1] + rng.normal(0, 1e-4, H[i].shape).astype(np.float32)
            for j in rng.choice(17, size=int(rng.integers(0, 6)), replace=False):
                H[i, j] = np.roll(H[i - 1, j], (int(rng.integers(-2, 3)), int(rng.integers(-2, 3))), axis=(0, 1))
    if unc == "Entropy":
        H = np.abs(H) + np.float32(1e-3)       # raw maps hold negatives: every entropy would be -inf
    boxes = v.synth.boxes_xyxy(n, 4)
    X32 = v.synth.embeddings(n, d=2048, seed=6)
    X = X32.astype(np.float64)
    est = FakeEstimator(torch.from_numpy(H).cuda(), torch.from_numpy(X32).cuda())
    al = v.ActiveLearning(*_cfg_opt(unc, rep, flt), model=est, eval_loader=None, eval_len=n, AE=None)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        if unc == "THC":
            raw = O.thc_pool(H, ip, inx)
        elif unc == "None":
            raw = None
        else:
            raw = O.pose_unc_pool(H, boxes, ip, inx, unc)
        peak = np.array([O.localpeak_mean(H[i]) for i in range(n)], dtype=np.float64)
    want_feat = flt not in ("None", "Random")
    labeled = []
    for rnd in range(2):
        al.eval_loader = _loader(n, boxes, ip, inx, 50)
        np.random.seed(100 + rnd)
        al.eval_and_query()
        np.random.seed(100 + rnd)
        unl = [i for i in range(n) if i not in set(labeled)]
        k = al.query_sizes[rnd] - len(labeled)
        unc_score = None if raw is None else O.fuse_scores(raw[unl])
        Xr = X if want_feat else np.zeros_like(X)
        infl = None
        if rep == "Influence":
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                infl = O.influence_scores(Xr, unl)
        elif rep == "Random":
            infl = np.random.rand(len(unl))
        cw = float(np.mean(peak[unl]))
        total = O.total_score(unc_score, infl, cw)
        if total is None:
            total = np.zeros(len(unl))
        if flt == "None":
            expect = O.topk_select(unl, total, k)
        elif flt == "Diversity":
            expect = O.diversity_select(X, unl, total, k)
        elif flt == "Random":
            cand = sorted(O.candidate_order(unl, total)[:8 * k])
            expect = []
            while len(expect) < k and cand:
                q = int(np.random.choice(cand)); expect.append(q); cand.remove(q)
        else:
            u = np.zeros(n); u[unl] = total
            dist_only = unc == "None"            # _query (:828-833): random first pick, then pure distance
            fp = int(np.random.choice(np.arange(n))) if (dist_only and not labeled) else None
            expect, _ = O.coreset_select(X, u, labeled, k, 0.0, 0.01, rule="dist" if dist_only else "w_unc", first_pick=fp)
        got = al.query_list_list[f"Round{rnd}"]
        if rep == "Influence" and not want_feat:
            assert len(got) == k               # all-zero features: influence is 0/0 = NaN in the reference too
        else:
            assert got == expect, (rnd, got, expect)
        if raw is not None:
            d = al.uncertainty_dict[f"Round{rnd}"]
            assert np.allclose([d[i] for i in range(n)], raw, rtol=RTOL)
        labeled = labeled + got
        assert al.outcome() is None


@pytest.mark.parametrize("kind", ["MPE", "Margin"])
def test_peak_uncertainties_match_oracle(built_lib, kind):
    """MPE / Margin (ActiveLearning.py:762-788) against the oracle, whose compute_mpe / compute_margin were run
    through the REFERENCE's own methods with the restated peak_local_max (golden), plus edge maps: plateaus,
    constant maps (trivial image -> no peak), peaks on the excluded border, ties."""
    v = built_lib
    from conftest import load_golden
    z = load_golden("peaks.npz")
    H = z["H"]
    got_mpe, got_mar = v.ops.peak_uncertainty(torch.from_numpy(H).cuda())
    got = (got_mpe if kind == "MPE" else got_mar).cpu().numpy()
    ref = z["mpe" if kind == "MPE" else "margin"]
    assert np.allclose(got, ref, rtol=1e-5, atol=1e-6), np.abs(got - ref).max()


def test_peak_fast_path_equals_generic(built_lib, monkeypatch):
    """The 64 x 48 paths (register / shuffle: the default; shared-memory staged) against the generic routine (bit-equal), on smooth maps, noise maps, tied
    peaks and plateau maps whose candidate list overflows (redone by the generic routine on a list)."""
    v = built_lib
    rng = np.random.default_rng(21)
    n, nj = 300, 17
    yy, xx = np.mgrid[0:64, 0:48].astype(np.float32)
    H = np.zeros((n, nj, 64, 48), np.float32)
    for i in range(n):
        for j in range(nj):
            kind = (i * nj + j) % 6
            if kind == 0:      # a few gaussians (what an estimator emits)
                for _ in range(int(rng.integers(1, 5))):
                    cy, cx, a = rng.uniform(0, 64), rng.uniform(0, 48), rng.uniform(0.1, 1.0)
                    H[i, j] += a * np.exp(-((yy - cy) ** 2 + (xx - cx) ** 2) / (2 * 2.0 ** 2))
            elif kind == 1:    # noise
                H[i, j] = rng.normal(0, 0.05, (64, 48))
            elif kind == 2:    # two-level plateaus: hundreds of pixels equal their window maximum (overflow)
                H[i, j] = (rng.random((64, 48)) < 0.7).astype(np.float32) * 0.5
            elif kind == 3:    # quantised: many exact ties
                H[i, j] = np.round(rng.normal(0, 1, (64, 48)), 0) * 0.25
            elif kind == 4:    # constant map (trivial image)
                H[i, j] = rng.uniform(-1, 1)
            else:              # constant with a single bump on the excluded border and one inside
                H[i, j, 2, 3] = 1.0
                H[i, j, 30, 20] = 0.5
    Hd = torch.from_numpy(H).cuda()
    fast = v.ops.peak_uncertainty(Hd)
    monkeypatch.setenv("VATLQ_PEAK_GENERIC", "1")
    gen = v.ops.peak_uncertainty(Hd)
    monkeypatch.delenv("VATLQ_PEAK_GENERIC")
    assert torch.equal(fast[0], gen[0]) and torch.equal(fast[1], gen[1])
    monkeypatch.setenv("VATLQ_PEAK_SMEM", "1")         # the shared-memory-staged 64 x 48 variant
    staged = v.ops.peak_uncertainty(Hd)
    monkeypatch.delenv("VATLQ_PEAK_SMEM")
    assert torch.equal(staged[0], gen[0]) and torch.equal(staged[1], gen[1])
    from oracle import vatl_oracle as O
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref_mpe = [O.mpe_item(H[i]) for i in range(12)]
        ref_mar = [O.margin_item(H[i]) for i in range(12)]
    assert np.allclose(fast[0][:12].cpu().numpy(), ref_mpe, rtol=1e-5, atol=1e-6)
    assert np.allclose(fast[1][:12].cpu().numpy(), ref_mar, rtol=1e-5, atol=1e-6)


def test_rank_scores_equals_python_stable_sort(built_lib):
    """vatlq_rank_scores reproduces `sorted(dict.items(), key=score, reverse=True)` over a dict in ascending id order
    (ActiveLearning.py:527-530): ties keep ascending ids; negative values, zeros of both signs, infinities."""
    v = built_lib
    rng = np.random.default_rng(3)
    n = 5000
    s = np.round(rng.normal(0, 1, n), 1)           # many ties
    s[:7] = [0.0, -0.0, np.inf, -np.inf, 1e-300, -1e-300, 0.0]
    mask = (rng.random(n) < 0.7).astype(np.uint8)
    ids = [i for i in range(n) if mask[i]]
    for desc in (True, False):
        expect = [i for i, _ in sorted(((i, s[i]) for i in ids), key=lambda x: x[1], reverse=desc)]
        got = v.ops.rank_scores(torch.from_numpy(s).cuda(), torch.from_numpy(mask).cuda(), descending=desc).cpu().tolist()
        assert got == expect
        assert v.ops.rank_scores(torch.from_numpy(s).cuda(), torch.from_numpy(mask).cuda(), descending=desc, count=17).cpu().tolist() == expect[:17]
    allrows = v.ops.rank_scores(torch.from_numpy(s).cuda()).cpu().tolist()
    assert allrows == [i for i, _ in sorted(enumerate(s), key=lambda x: x[1], reverse=True)]


def test_new_rows_edge_shapes(built_lib):
    """Empty and single-item inputs; MPE / Margin on a non-64x48 map shape (generic path) against the oracle."""
    from oracle import vatl_oracle as O
    v = built_lib
    dev = "cuda:0"
    assert v.ops.oks(torch.zeros((0, 17, 3), device=dev), torch.zeros((0, 17, 3), device=dev), torch.zeros((0, 4), device=dev)).numel() == 0
    assert v.ops.rank_scores(torch.tensor([0.5], dtype=torch.float64, device=dev)).cpu().tolist() == [0]
    assert v.ops.rank_scores(torch.zeros(0, dtype=torch.float64, device=dev)).numel() == 0
    rng = np.random.default_rng(8)
    H = rng.normal(0, 0.05, (3, 5, 40, 30)).astype(np.float32)
    H[0, 0, 20, 15] = 1.0; H[0, 0, 8, 8] = 0.7; H[1, 2] = 0.3      # peaks; a constant (trivial) map
    mpe, mar = v.ops.peak_uncertainty(torch.from_numpy(H).to(dev))
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ref_mpe = [O.mpe_item(H[i]) for i in range(3)]
        ref_mar = [O.margin_item(H[i]) for i in range(3)]
    assert np.allclose(mpe.cpu().numpy(), ref_mpe, rtol=1e-5, atol=1e-6)
    assert np.allclose(mar.cpu().numpy(), ref_mar, rtol=1e-5, atol=1e-6)
