"""CPU: the host logic of the controller (`ActiveLearning.eval_and_query` / `_query`, `QueryPass`: chunk
bookkeeping, strategy dispatch, representativeness / filter branches, index-set updates) driven with
oracle-backed STAND-INS for the device operators.  This is test scaffolding: the product itself has no
CPU path (tests/test_host_logic.py::test_no_cpu_fallback); here every `ops.*` entry the controller calls is
replaced by a function that evaluates the oracle, so the Python around the kernels is checked without a GPU.
The same scenarios run against the real kernels in tests/test_gpu_next.py / test_gpu_query.py."""
import warnings

import numpy as np
import pytest
import torch

from oracle import vatl_oracle as O
from test_kmeans_host_cpu import km_on_cpu  # noqa: F401  (fixture: the K-Means device calls as NumPy stand-ins)


def _install_stand_ins(monkeypatch, v):
    ops, query, AL, _lib = v.ops, v.query, v.active_learning, v._lib
    cpu = torch.device("cpu")
    monkeypatch.setattr(_lib, "lib", lambda: None)
    monkeypatch.setattr(AL, "_dev", lambda: cpu)
    monkeypatch.setattr(query, "_require_cuda", lambda dev: None)
    monkeypatch.setattr(torch.Tensor, "cuda", lambda self, *a, **k: self)

    def _flags(t, n, dev, name):
        if t is None:
            return None
        if not isinstance(t, torch.Tensor):
            t = torch.as_tensor(np.asarray(t))
        return t.to(torch.uint8)

    def heatmap_scan(H, is_prev=None, is_next=None, boxes_xyxy=None, halo_prev=None, halo_next=None):
        Hn = H.numpy()
        n = Hn.shape[0]
        ip = np.zeros(n, np.uint8) if is_prev is None else np.asarray(is_prev)
        inx = np.zeros(n, np.uint8) if is_next is None else np.asarray(is_next)
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            thc = O.thc_pool(Hn, ip, inx, None if halo_prev is None else halo_prev.numpy(),
                             None if halo_next is None else halo_next.numpy())
            pm = np.array([O.localpeak_mean(Hn[i]) for i in range(n)], np.float32)
            xy = np.stack([O.heatmap_coords(Hn[i])[0] for i in range(n)])
            kp = None
            if boxes_xyxy is not None:
                kp = np.zeros((n, 17, 3), np.float32)
                for i in range(n):
                    c, val = O.heatmap_to_coord(Hn[i], [float(x) for x in boxes_xyxy[i]])
                    kp[i, :, :2] = c
                    kp[i, :, 2] = val[:, 0]
        return ops.ScanResult(thc=torch.from_numpy(thc.astype(np.float32)), peak_sum=torch.zeros(n),
                              peak_cnt=torch.zeros(n, dtype=torch.int32), peak_mean=torch.from_numpy(pm),
                              coords_hm=torch.from_numpy(xy), kpts=None if kp is None else torch.from_numpy(kp))

    def heatmap_entropy(H):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return torch.tensor([O.entropy_item(h) for h in H.numpy()], dtype=torch.float32)

    def pose_uncertainty(coords_hm, kpts, boxes, is_prev=None, is_next=None, hm_shape=(64, 48), halo_prev_xy=None,
                         halo_next_xy=None, want_hp=True, want_tpc=True):
        n = kpts.shape[0]
        hp = torch.tensor([O.hp_item(kpts[i, :, 2:3].numpy()) for i in range(n)], dtype=torch.float32) if want_hp else None
        tpc = None
        if want_tpc:
            xy = coords_hm.numpy()
            out = np.zeros(n, np.float32)

            def img(i, pts):   # the decode of transforms.py:568-581 with item i's crop box
                b = [float(x) for x in boxes[i]]
                bw, bh = b[2] - b[0], b[3] - b[1]
                t = O.inverse_affine(np.array([b[0] + bw * .5, b[1] + bh * .5]), np.array([bw, bh]), [hm_shape[1], hm_shape[0]])
                o = np.zeros_like(pts)
                for j in range(pts.shape[0]):
                    o[j] = np.dot(t, np.array([pts[j][0], pts[j][1], 1.]).T)[:2]
                return o
            for i in range(n):
                b = [float(x) for x in boxes[i]]
                th = 0.01 * np.sqrt((b[2] - b[0]) * (b[3] - b[1]))
                has_p = bool(is_prev[i]) and (i > 0 or halo_prev_xy is not None)
                has_n = bool(is_next[i]) and (i < n - 1 or halo_next_xy is not None)
                c, cur = 0, img(i, xy[i])
                if has_p:
                    c += np.count_nonzero(np.linalg.norm(cur - img(i, xy[i - 1] if i > 0 else halo_prev_xy.numpy()), axis=1) > th)
                if has_n:
                    c += np.count_nonzero(np.linalg.norm(cur - img(i, xy[i + 1] if i < n - 1 else halo_next_xy.numpy()), axis=1) > th)
                out[i] = c * (2 if has_p != has_n else 1)
            tpc = torch.from_numpy(out)
        return hp, tpc

    def cosine_rowsum(X, rows=None, group=None):
        Xn = X.numpy().astype(np.float64)
        if rows is not None:
            Xn = Xn[np.asarray(rows)]
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return torch.from_numpy(O.cosine_rowsum(Xn))

    def minmax_f64(vv, mask=None, group=None):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return torch.from_numpy(O._minmax(vv.numpy()))

    def blend_scores(unc, infl, cw, mask=None):
        out = cw * unc.numpy() + (1 - cw) * infl.numpy()
        return torch.from_numpy(out if mask is None else np.where(mask.numpy() != 0, out, 0.0))

    def fuse_scores(thc, wpu_, unl, mode="const", labeled_ratio=0.0, group=None):
        u = unl.numpy().astype(bool)
        out = np.zeros(thc.numel())
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            out[u] = O.fuse_scores(thc.numpy().astype(np.float64)[u],
                                   None if wpu_ is None else wpu_.numpy().astype(np.float64)[u],
                                   mode if wpu_ is not None else "const", labeled_ratio)
        return torch.from_numpy(out)

    def coreset_select(X, unc, labeled, k, moks, lam, rule="w_unc", first_pick=-1, batch=16, comm=None, row_range=None,
                       return_state=False):
        u = unc.numpy().copy()
        picks, _ = O.coreset_select(X.numpy().astype(np.float64), u, list(labeled), k, moks, lam, rule, first_pick)
        p = torch.tensor(picks, dtype=torch.int64)
        return (p, None, None, torch.from_numpy(u)) if return_state else (p, None)

    def wpu(kpts, boxes, packed, in_dim, z_dim, drop_ears=False, return_features=False, check_status=True,
            return_status=False):
        ae = packed[0]   # pack_ae_weights stand-in below keeps the torch module
        out = [O.wpu_item(ae, [float(x) for x in boxes[i]], kpts[i].reshape(-1).double().numpy(), drop_ears)
               for i in range(kpts.shape[0])]
        w = torch.tensor(out, dtype=torch.float32)
        return (w, torch.zeros(len(out), dtype=torch.uint8)) if return_status else w

    def oks(kpts, gt, bann):
        n = kpts.shape[0]
        out = [O.compute_oks(O.xyxy_to_xywh([float(x) for x in bann[i]]), kpts[i].reshape(-1).double().numpy(),
                             gt[i].reshape(-1).double().numpy()) for i in range(n)]
        return torch.tensor(out, dtype=torch.float64)

    def rank_scores(score, mask=None, descending=True, count=None):
        sc = score.numpy()
        idx = [i for i in range(len(sc)) if mask is None or bool(mask[i])]
        order = sorted(idx, key=lambda t: sc[t], reverse=descending)       # the reference's stable sorted() (:529,587)
        return torch.tensor(order if count is None else order[:count], dtype=torch.int64)

    def pack_ae_weights(weights, device):
        return [O.make_autoencoder(weights)], 42, 4

    for name, fn in dict(_flags=_flags, heatmap_scan=heatmap_scan, heatmap_entropy=heatmap_entropy,
                         pose_uncertainty=pose_uncertainty, cosine_rowsum=cosine_rowsum, minmax_f64=minmax_f64,
                         blend_scores=blend_scores, fuse_scores=fuse_scores, coreset_select=coreset_select, wpu=wpu, oks=oks, rank_scores=rank_scores,
                         pack_ae_weights=pack_ae_weights).items():
        monkeypatch.setattr(ops, name, fn)


@pytest.mark.parametrize("unc,rep,flt", [("HP", "None", "None"), ("TPC", "Influence", "Diversity"),
                                         ("THC", "Influence", "None"), ("None", "Influence", "Coreset"),
                                         ("HP", "Random", "Random"), ("Entropy", "None", "None")])
def test_controller_next_strategies_host_logic(built_lib, monkeypatch, unc, rep, flt):
    import test_gpu_next as T
    _install_stand_ins(monkeypatch, built_lib)
    T.test_controller_next_strategies_match_oracle(built_lib, unc, rep, flt)


@pytest.mark.parametrize("unc,flt", [("THC+WPU", "Coreset"), ("THC", "None")])
def test_controller_default_strategies_host_logic(built_lib, monkeypatch, unc, flt):
    import test_gpu_query as T
    _install_stand_ins(monkeypatch, built_lib)
    T.test_two_rounds_match_oracle(built_lib, unc, flt)


@pytest.fixture
def one_rank_group():
    import torch.distributed as td
    td.init_process_group("gloo", store=td.HashStore(), rank=0, world_size=1)
    try:
        yield td.group.WORLD
    finally:
        td.destroy_process_group()


@pytest.mark.parametrize("rep,flt,n_unl", [("Influence", "None", None), ("None", "Diversity", None),
                                           ("None", "K-Means", None), ("Influence", "weighted", None),
                                           ("Influence", "Coreset", None), ("None", "Coreset", None),
                                           ("None", "Coreset", 0), ("None", "Coreset", 1),
                                           ("None", "K-Means", 0), ("None", "K-Means", 1)])
def test_distributed_query_matches_controller_host_logic(km_on_cpu, one_rank_group, monkeypatch, rep, flt, n_unl):
    """dist.distributed_query on a one-rank gloo group picks what ActiveLearning._query picks from the same pool,
    labelled set and rule, with the same scores.  With at most one unlabelled item (n_unl) every filter takes the
    score-ordered top k and nothing is clustered (ActiveLearning.py:533-534, 541-542)."""
    import vatlq as v
    from types import SimpleNamespace
    from vatlq import _lib, dist, kmeans as KM
    fake = _lib.lib()
    _install_stand_ins(monkeypatch, v)
    monkeypatch.setattr(_lib, "lib", lambda: fake)
    monkeypatch.setattr(KM, "rank_scores", v.ops.rank_scores)
    if n_unl is not None:
        def no_clustering(*a, **kw):
            raise AssertionError("a pool with at most one unlabelled item is not clustered")
        monkeypatch.setattr(KM, "kmeans_fit_select", no_clustering)
    n = 60
    ids, ip, inx = v.synth.track_flags(n, np.random.default_rng(3), 6.0)
    H = torch.from_numpy(v.synth.heatmaps(n, seed=3, track_ids=ids))
    boxes = torch.from_numpy(v.synth.boxes_xyxy(n, 3))
    ip, inx = torch.from_numpy(ip.astype(np.uint8)), torch.from_numpy(inx.astype(np.uint8))
    X = v.synth.embeddings(n, d=64, seed=3)
    X[40:45] = X[20:25]                                   # duplicates for the weighted filter's np.unique
    labeled = list(range(0, n, 5)) if n_unl is None else list(range(n - n_unl))
    cfg = SimpleNamespace(VAL=SimpleNamespace(QUERY_RATIO=[0.1, 0.2], W_UNC=0.8, UNC_LAMBDA=0.01),
                          DATA_PRESET=SimpleNamespace(HEATMAP_SIZE=[64, 48]), AE=SimpleNamespace(Z_DIM=4))
    opt = SimpleNamespace(strategy=f"THC+{rep}_{flt}filter", uncertainty="THC", representativeness=rep, filter=flt,
                          video_id="0", THCvsWPU="const", fixed_lambda=False, onebyone=False)
    al = v.ActiveLearning(cfg, opt, eval_len=n)
    al.labeled_id.update(labeled)
    al.unlabeled_id.difference_update(labeled)
    k = al.query_size
    cand = sorted(set(range(n)) - set(labeled))
    fake.n = len(cand) if flt != "weighted" else len(np.unique(X[cand].astype(np.float64), axis=0))
    fake.k = min(k, fake.n)
    qp = v.QueryPass(n, "cpu", uncertainty="THC")
    qp.score_pool(H, boxes, ip, inx)
    al._query(qp, torch.from_numpy(X))
    res = dist.distributed_query(H, boxes, ip, inx, torch.from_numpy(X), None, labeled, n, k, 0.0, al.unc_lambda,
                                 uncertainty="THC", rule="w_unc", representativeness=rep, filter=flt, w_unc=al.w_unc,
                                 group=one_rank_group)
    assert res.picks.tolist() == al.last_query.query_list
    assert len(res.picks) == min(k, len(cand))
    assert torch.equal(res.unc, al.last_query.score)
