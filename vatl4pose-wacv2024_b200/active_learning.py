"""Host-side mirror of the reference's query interface (active_learning/ActiveLearning.py).

Same names, argument meaning and error behaviour as the reference for the ONE path this
package accelerates — `ActiveLearning.eval_and_query()` and the helper callables it uses —
with the per-person Python loop replaced by batched CUDA kernels (ops.py / libvatlq.so).
Everything else of the reference class (dataset building, estimator training, mAP/OSPA
evaluation, plotting) is out of scope and is injected or hooked:

    al = ActiveLearning(cfg, opt)                       # builds estimator / loader / AE through the reference's builders
    al = ActiveLearning(cfg, opt, model=estimator, eval_loader=loader, eval_len=len(dataset), AE=ae)   # or injected
    al.eval_and_query()          # fills labeled_id / unlabeled_id / query_list_list / moks_queried / ...
    al.outcome()                 # None while rounds remain, else the reference's 20-tuple (:203)

Strategy names are the reference's (`opt.uncertainty`, `opt.representativeness`, `opt.filter`,
ActiveLearning.py:329-401,467-481,533-619).  Uncertainties THC*, WPU*, THC+WPU, HP, TPC, Entropy
MPE, Margin and None, representativeness None / Influence / Random and filters None / Coreset / Diversity /
Random / K-Means / weighted run here; names without a device path (see _require_accelerated) raise NotImplementedError
naming the reference code path to use (dispatch to the reference, never a CPU re-implementation
of ours).
"""
from __future__ import annotations

import copy
from types import SimpleNamespace

import numpy as np
import torch
import torch.nn as nn

from . import _lib, ops
from .query import FILTERS, QueryPass, classify_uncertainty, influence, select, unlabelled_mask

__all__ = ["ActiveLearning", "IndexCollection", "WholeBodyAE", "compute_thc", "compute_entropy", "localpeak_mean",
           "heatmap_to_coord_simple", "compute_hybrid", "coreset_selection"]


def _dev():
    if not torch.cuda.is_available():
        raise _lib.VatlqError("no CUDA device: the query pass has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _as_cuda(a, dtype=torch.float32):
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
    return t.to(device=_dev(), dtype=dtype).contiguous()


def embedding_store_dtype(filter_: str, representativeness: str, dtype: torch.dtype) -> torch.dtype:
    """The dtype eval_and_query stores the embeddings in: fp16 / bf16 as they are when only the core-set reads them
    (filter Coreset, representativeness None or Random) — its picks equal those of the exact fp32 upcast, at half
    the memory — fp32 (`.float()`, like the reference) for every other consumer."""
    if dtype in (torch.float16, torch.bfloat16) and filter_ == "Coreset" and representativeness in ("None", "Random"):
        return dtype
    return torch.float32


def _heatmaps(out: torch.Tensor) -> torch.Tensor:
    """The estimator's heat maps as the kernels read them: fp16 / bf16 (autocast or a .half() model) as they are —
    the scores equal those of their exact fp32 upcast — every other dtype as `.float()` like the reference."""
    return (out if out.dtype in (torch.float16, torch.bfloat16) else out.float()).contiguous()


# ----------------------------------------------------------------------------------------
# single-item shims with the reference's signatures (tests read like the reference's code)
# ----------------------------------------------------------------------------------------

def compute_thc(heatmaps, heatmaps_adj, norm_type="L1"):
    """ActiveLearning.compute_thc (ActiveLearning.py:747-760) for one pair of (J,H,W) stacks."""
    if norm_type != "L1":
        raise NotImplementedError("only the L1 norm is on the query path (ActiveLearning.py:346)")
    cur = _as_cuda(heatmaps)[None]
    adj = _as_cuda(heatmaps_adj)[None]
    one = torch.ones(1, dtype=torch.uint8)
    # a single existing neighbour is doubled at the call site (:355-362), not in compute_thc
    return float(ops.thc3(cur, adj, None, one, 1 - one)[0]) / 2.0


def localpeak_mean(heatmaps, filter_size=3, order=0.5):
    """active_learning/local_peak.py:12-22 for one (J,H,W) stack."""
    if filter_size != 3 or order != 0.5:
        raise NotImplementedError("the query path uses filter_size=3, order=0.5 (ActiveLearning.py:412)")
    return float(ops.heatmap_scan(_as_cuda(heatmaps)[None]).peak_mean[0])


def compute_entropy(heatmaps):
    """ActiveLearning.compute_entropy (ActiveLearning.py:790-796) for one (J,H,W) stack."""
    return float(ops.heatmap_entropy(_as_cuda(heatmaps)[None])[0])


def heatmap_to_coord_simple(hms, bbox, hms_flip=None, **kwargs):
    """alphapose/utils/transforms.py:550-583 for one (J,H,W) stack -> (preds (J,2), maxvals (J,1))."""
    h = _as_cuda(hms)
    if hms_flip is not None:
        h = (h + _as_cuda(hms_flip)) / 2
    box = torch.tensor([list(map(float, bbox))], dtype=torch.float32)
    r = ops.heatmap_scan(h[None], boxes_xyxy=box)
    k = r.kpts[0].cpu().numpy()
    return k[:, :2].copy(), k[:, 2:3].copy()


def compute_hybrid(bbox, keypoints):
    """active_learning/Whole_body_AE/hybrid_feature.py:14-58.  bbox is [x,y,w,h]; returns the
    42-d feature as float64 holding the float32 values the auto-encoder is fed (`.float()`,
    ActiveLearning.py:367)."""
    k = np.asarray(keypoints, dtype=np.float32).reshape(1, ops.J, 3)
    x, y, w, h = [float(v) for v in bbox]
    box = torch.tensor([[x, y, x + w - 1, y + h - 1]], dtype=torch.float32)   # inverse of bbox.py:95-97
    dummy = torch.zeros(int(_lib.lib().vatlq_wpu_weight_count(42, 4)), device=_dev())
    _, feat = ops.wpu(_as_cuda(k), box, dummy, 42, 4, return_features=True)
    return feat[0].double().cpu().numpy()


class WholeBodyAE(nn.Module):
    """Layer stack of active_learning/Whole_body_AE/AutoEncoder.py:5-39.  The reference hard-codes
    input_dim=38 while its call site feeds 42 features (SURVEY.md §8a-5); here the width is an
    argument defaulting to what compute_hybrid emits.  `forward` is plain torch (used for
    training, which stays reference code); `unnaturalness` is the fused CUDA scoring path."""

    def __init__(self, z_dim=2, kp_direct=False, input_dim=42):
        super().__init__()
        if kp_direct:
            raise NotImplementedError("kp_direct auto-encoders are not on the query path")
        self.z_dim, self.input_dim = z_dim, input_dim
        self.encoder = nn.Sequential(nn.Linear(input_dim, 24), nn.ReLU(True), nn.Linear(24, 12), nn.ReLU(True),
                                     nn.Linear(12, 7), nn.ReLU(True), nn.Linear(7, z_dim))
        self.decoder = nn.Sequential(nn.Linear(z_dim, 7), nn.ReLU(True), nn.Linear(7, 12), nn.ReLU(True),
                                     nn.Linear(12, 24), nn.ReLU(True), nn.Linear(24, input_dim), nn.Sigmoid())

    def forward(self, x):
        return self.decoder(self.encoder(x))

    def unnaturalness(self, kpts, boxes_xyxy, drop_ears=False):
        w, ind, z = ops.pack_ae_weights(self, _dev())
        return ops.wpu(_as_cuda(kpts).reshape(-1, ops.J, 3), _as_cuda(boxes_xyxy).reshape(-1, 4), w, ind, z, drop_ears)


def forward_with_embedding(model, crops, want_embedding: bool, fuse: bool = True):
    """The estimator's heat maps and, when wanted, its 2048-d embedding for one batch (ActiveLearning.py:277-286).
    The reference runs the backbone twice: `self.model(inps)` and `self.model.module.get_embedding(inps)`, both of
    which start with `self.preact(x)` (alphapose/models/fastpose.py:44-59,70-73, simplepose.py:82-91).  When the
    estimator has that shape (`preact` + `avgpool`), a forward hook keeps the backbone output of the ONE forward and
    the embedding is `flatten(avgpool(out), 1)` of it — `get_embedding`'s own two lines — so the backbone runs once
    (SURVEY 8f-4, producer side).  The estimator itself is untouched; anything else (no `preact`, several replicas
    under DataParallel, fuse=False / `opt.fuse_embedding = False`) takes the reference's two calls."""
    core = model.module if hasattr(model, "module") else model
    if want_embedding and fuse and hasattr(core, "preact") and hasattr(core, "avgpool"):
        grabbed = []
        handle = core.preact.register_forward_hook(lambda mod, inp, out: grabbed.append(out))
        try:
            out = model(crops)
        finally:
            handle.remove()
        if len(grabbed) == 1 and torch.is_tensor(grabbed[0]):
            return out, torch.flatten(core.avgpool(grabbed[0]), 1)
        return out, core.get_embedding(crops)          # replicas / an unexpected call pattern: the reference's second call
    out = model(crops)
    return out, (core.get_embedding(crops) if want_embedding else None)


class IndexCollection:
    """The part of alipy.index.IndexCollection (ALiPy/alipy/index/index_collections.py:26-226)
    the query path uses: an ordered, duplicate-free list of ints with set-speed membership."""

    def __init__(self, data=None):
        self._list, self._set = [], set()
        if data is not None:
            self.update(data)

    @property
    def index(self):
        return list(self._list)   # the reference hands out a copy (:91-95)

    def __len__(self):
        return len(self._list)

    def __contains__(self, v):
        return int(v) in self._set

    def __iter__(self):
        return iter(self._list)

    def add(self, v):
        v = int(v)
        if v not in self._set:
            self._set.add(v)
            self._list.append(v)
        return self

    def discard(self, v):
        v = int(v)
        if v in self._set:
            self._set.remove(v)
            self._list.remove(v)
        return self

    def update(self, other):
        for v in other:
            self.add(v)
        return self

    def difference_update(self, other):
        drop = {int(v) for v in other} & self._set
        if drop:
            self._set -= drop
            self._list = [v for v in self._list if v not in drop]
        return self


def coreset_selection(self, embeddings, uncertainty):
    """ActiveLearning.coreset_selection (ActiveLearning.py:798-850), same `self` attributes:
    labeled_id, moks_queried, unc_lambda, uncertainty (the strategy name), cfg.VAL.UNC_LAMBDA,
    opt.fixed_lambda, query_size.  `uncertainty` (the array) is modified in place like the
    reference (:848).  Returns the list of picked indices in pick order."""
    # (fp16 / bf16 tensors as they are: the selection equals that on their exact fp32 upcast)
    keep = isinstance(embeddings, torch.Tensor) and embeddings.dtype in (torch.float16, torch.bfloat16)
    X = _as_cuda(embeddings, embeddings.dtype if keep else torch.float32)
    if isinstance(embeddings, np.ndarray) and embeddings.dtype == np.float64:
        if not np.array_equal(X.cpu().numpy().astype(np.float64), embeddings):
            raise _lib.VatlqError("embeddings must hold fp32-representable values (ActiveLearning.py:270,286)")
    unc = _as_cuda(uncertainty, torch.float64)
    rule, first_pick = _coreset_rule(self, X.shape[0])
    picks, stats, _, unc_after = ops.coreset_select(
        X, unc, list(self.labeled_id.index), int(self.query_size), float(self.moks_queried), float(self.unc_lambda),
        rule=rule, first_pick=first_pick, batch=int(getattr(self, "coreset_batch", 16)), return_state=True)
    self.coreset_stats = stats
    if isinstance(uncertainty, np.ndarray):
        uncertainty[:] = unc_after.cpu().numpy()
    return [int(i) for i in picks.cpu().tolist()]


def _coreset_rule(self, n: int) -> tuple[str, int]:
    """(rule, first_pick) of the core-set for the strategy of `self` (ActiveLearning.py:815-833): "dist" without an
    uncertainty to weigh, its first pick drawn from np.random like the reference when nothing is labelled;
    "fixed_lambda" / "w_unc" otherwise."""
    if self.uncertainty == "None" or self.cfg.VAL.UNC_LAMBDA == 0:
        return "dist", int(np.random.choice(np.arange(n))) if len(self.labeled_id.index) == 0 else -1
    return ("fixed_lambda" if self.opt.fixed_lambda else "w_unc"), -1


# ----------------------------------------------------------------------------------------
# the controller
# ----------------------------------------------------------------------------------------

_REFERENCE_ONLY_UNC = ("VL4Pose",)                      # the reference's own VL4Pose branch is an unfinished stub (:390-391)


class ActiveLearning:
    """Query-pass controller with the reference's public surface: `ActiveLearning(cfg, opt)`,
    `eval_and_query()`, `outcome()` and the state they mutate (ActiveLearning.py:52-164,253-649,
    166-205).  The estimator, the evaluation data loader and the auto-encoder are injected
    (`model`, `eval_loader`, `AE`); `eval_loader` yields the reference's collate tuple
    (idxs, inps, labels, label_masks, GTkpts, img_ids, ann_ids, bboxes_crop, bboxes_ann, isPrev, isNext)
    (alphapose/datasets/posetrack21.py:207-) in pool order."""

    def __init__(self, cfg, opt, model=None, eval_loader=None, eval_len=None, AE=None, oks_fn=None,
                 eval_hook=None, retrain_hook=None, metrics_hook=None):
        self.round_cnt = 0
        self.cfg, self.opt = cfg, opt
        self.one_by_one = bool(getattr(opt, "onebyone", False))
        self.strategy = opt.strategy
        self.uncertainty = opt.uncertainty
        self.representativeness = opt.representativeness
        self.filter = opt.filter
        self.video_id = getattr(opt, "video_id", None)
        self.get_prenext = getattr(opt, "get_prenext", ("THC" in self.uncertainty or self.uncertainty == "TPC"))
        self.model, self.eval_loader, self.AE = model, eval_loader, AE
        self.oks_fn, self.eval_hook, self.retrain_hook, self.metrics_hook = oks_fn, eval_hook, retrain_hook, metrics_hook
        # dispatch keys: accept exactly the reference's names (:329-401,467-481,533-619)
        if not (any(classify_uncertainty(self.uncertainty)) or self.uncertainty in ("None",) + _REFERENCE_ONLY_UNC):
            raise ValueError("Uncertainty type is not supported")
        if self.representativeness not in ("None", "Influence", "Random"):
            raise ValueError("Representativeness type is not supported")
        if self.filter not in FILTERS + ("Random",):
            raise ValueError("Filter type is not supported")
        if eval_len is None and eval_loader is None:
            self._build_from_reference()          # the two-argument form of the reference (:52-164)
            eval_loader = self.eval_loader
        self.eval_len = int(eval_len if eval_len is not None else len(eval_loader.dataset))
        self.query_ratio = cfg.VAL.QUERY_RATIO
        self.w_unc = cfg.VAL.W_UNC
        self.unc_lambda = cfg.VAL.UNC_LAMBDA
        self.query_sizes = [int(self.eval_len * x) for x in self.query_ratio]
        self.query_size = self.query_sizes[0]
        if self.one_by_one:
            self.query_size = 3
        self.unlabeled_id = IndexCollection(list(range(self.eval_len)))
        self.labeled_id = IndexCollection()
        self.retrain_id = IndexCollection()
        # result members of the reference (:121-137), same names, returned by outcome() (:203)
        self.percentage, self.performance, self.performance_ann = [], [], []
        self.ospa_list, self.ospa_list_ann, self.combine_weight = [], [], []
        self.query_list_list, self.uncertainty_dict, self.influence_dict = {}, {}, {}
        self.uncertainty_mean, self.spearmanr_list, self.corr_list, self.moksQ_list = [], [], [], []
        self.true_labeled_dict, self.false_labeled_dict = {}, {}
        self.true_unlabeled_dict, self.false_unlabeled_dict = {}, {}
        # stopping criteria (:100-105)
        self.is_early_stop = False
        self.finish_acc = float(getattr(opt, "retrain_thresh", 1.0))
        self.finish_margin = 0.05
        self.actual_finish = self.finished_minerror = self.finished_oursc = 100
        self.moks_queried = 0
        self.eval_joints = list(range(ops.J))
        self.hm_size = cfg.DATA_PRESET.HEATMAP_SIZE
        self.coreset_batch = int(getattr(opt, "coreset_batch", 16))
        self.last_query = None
        self.OKS_dict = None

    def _build_from_reference(self):
        """`ActiveLearning(cfg, opt)` exactly as scripts/Run_active_learning.py:165-173 calls it: the
        evaluation dataset / loader, the estimator and the auto-encoder are built by the REFERENCE's
        own builders (ActiveLearning.py:95-99,144-152; they stay reference code), which therefore must
        be importable.  Everything after the estimator's forward runs here."""
        try:
            from alphapose.models import builder                      # noqa: F401  (reference package)
        except Exception as exc:
            raise _lib.VatlqError(
                "ActiveLearning(cfg, opt) builds the dataset, the estimator and the auto-encoder through the "
                "reference's builders (alphapose.models.builder): put the reference checkout on sys.path, or inject "
                "model=, eval_loader=, eval_len= and AE= (see INTEGRATION.md)") from exc
        cfg, opt = self.cfg, self.opt
        ds = builder.build_dataset(cfg.DATASET.EVAL, preset_cfg=cfg.DATA_PRESET, train=False, get_prenext=self.get_prenext)
        self.eval_dataset = ds
        self.eval_loader = torch.utils.data.DataLoader(
            ds, batch_size=cfg.VAL.BATCH_SIZE * getattr(opt, "num_gpu", 1), shuffle=False, num_workers=8, drop_last=False,
            pin_memory=True, collate_fn=ds.my_collate_fn)                                           # (:97-99)
        if self.model is None:
            m = builder.build_sppe(cfg.MODEL, preset_cfg=cfg.DATA_PRESET)                           # (:213-221)
            if not getattr(opt, "from_scratch", False):
                if not cfg.MODEL.PRETRAINED:
                    raise ValueError("No pretrained model is given!")
                m.load_state_dict(torch.load(cfg.MODEL.PRETRAINED))
            self.model = torch.nn.DataParallel(m, device_ids=getattr(opt, "gpus", None)).cuda()     # (:233)
        if self.AE is None and "WPU" in self.strategy:                                              # (:150-152, 886-)
            from active_learning.Whole_body_AE.AutoEncoder import WholeBodyAE as RefAE
            ae = RefAE(z_dim=cfg.AE.Z_DIM)
            pre = getattr(cfg.AE, "PRETRAINED", None)
            if pre:
                ae.load_state_dict(torch.load(pre))
            self.AE = ae

    # -- dispatch guard: names this package does not accelerate stay on the reference ----
    def _require_accelerated(self):
        u = self.uncertainty
        if u in _REFERENCE_ONLY_UNC:
            raise NotImplementedError(
                f"uncertainty '{u}' is not on the accelerated path: run the reference's "
                "ActiveLearning.eval_and_query (active_learning/ActiveLearning.py:329-401) for it")

    @torch.no_grad()
    def eval_and_query(self):
        """ActiveLearning.eval_and_query (:253-649): estimator forward stays the caller's model;
        scoring, fusion and selection run on the device."""
        self._require_accelerated()
        dev = _dev()
        n = self.eval_len
        # embeddings are collected when the filter OR the representativeness needs them (:283)
        want_feat = self.filter not in ("None", "Random") or self.representativeness not in ("None", "Random")
        qp = QueryPass(n, dev, ae_weights=self.AE if classify_uncertainty(self.uncertainty)[2] else None,
                       uncertainty=self.uncertainty)
        # (the reference keeps an all-zero fvecs_matrix otherwise, :270); allocated at the first batch, in
        # embedding_store_dtype of the estimator's embeddings
        X = None
        oks_dev = torch.zeros(n, dtype=torch.float64, device=dev)
        have_gt = True
        m = self.model
        if hasattr(m, "eval"):
            m.eval()
        strict = bool(getattr(self.opt, "strict_prenext", False)) and "THC" in self.uncertainty
        thc_strict = torch.zeros(n, dtype=torch.float32, device=dev) if strict else None
        pos = 0
        for batch in self.eval_loader:
            idxs, inps = batch[0], batch[1]
            bboxes_crop, isPrev, isNext = batch[7], batch[9], batch[10]
            idx_t = torch.as_tensor(np.asarray(idxs)).long()
            b = idx_t.numel()
            if not torch.equal(idx_t, torch.arange(pos, pos + b)):
                raise _lib.VatlqError("eval_loader must walk the id-sorted pool in order (shuffle=False)")
            cur = inps[:, 0].to(dev)
            out, emb = forward_with_embedding(m, cur, want_feat, fuse=bool(getattr(self.opt, "fuse_embedding", True)))
            H = _heatmaps(out[:, self.eval_joints])                       # (:277-281)
            if want_feat:
                if X is None:
                    X = torch.zeros((n, 2048), device=dev,
                                    dtype=embedding_store_dtype(self.filter, self.representativeness, emb.dtype))
                if X.dtype != torch.float32 and emb.dtype != X.dtype:
                    raise _lib.VatlqError(f"the estimator's embeddings changed dtype mid-pool ({X.dtype} -> {emb.dtype})")
                X[pos:pos + b] = emb if emb.dtype == X.dtype else emb.float()   # (:283-286)
            boxes = torch.as_tensor(np.asarray(bboxes_crop), dtype=torch.float32).reshape(b, 4).to(dev)
            ip = torch.as_tensor(np.asarray(isPrev)).to(torch.uint8)
            inx = torch.as_tensor(np.asarray(isNext)).to(torch.uint8)
            qp.score_chunk(pos, H, boxes, ip, inx)
            # OKS of every item against its ground truth (:309, al_metric.py:42-69): the selection weights of
            # the NEXT query (moks_queried) and the stopping criteria come from it
            gt, bann = (batch[4], batch[8]) if len(batch) > 8 else (None, None)
            if gt is not None and bann is not None and self.oks_fn is None:
                gt_t = torch.as_tensor(np.asarray(gt), dtype=torch.float32).reshape(b, 51)
                ba_t = torch.as_tensor(np.asarray(bann), dtype=torch.float32).reshape(b, 4)
                oks_dev[pos:pos + b] = ops.oks(qp.kpts[pos:pos + b], gt_t, ba_t)
            else:
                have_gt = False
            if strict:   # the reference's own three forwards (:293-297)
                Hp = _heatmaps(m(inps[:, 1].to(dev))[:, self.eval_joints])
                Hn = _heatmaps(m(inps[:, 2].to(dev))[:, self.eval_joints])
                thc_strict[pos:pos + b] = ops.thc3(H, Hp, Hn, ip, inx)
            if self.eval_hook is not None:
                self.eval_hook(self, batch, qp.kpts[pos:pos + b])
            pos += b
        if pos != n:
            raise _lib.VatlqError(f"eval_loader produced {pos} items, expected {n}")
        if strict:
            qp.thc.copy_(thc_strict)
        self.OKS_dict = None
        self._strict_oks = True     # a full eval_and_query must be able to derive moks_queried (see _query)
        if have_gt:
            self.OKS_dict = dict(enumerate(oks_dev.cpu().tolist()))
        if self.metrics_hook is not None:   # mAP / OSPA of :438-447 are evaluation (reference code): hooked
            m_ = self.metrics_hook(self, qp.kpts) or {}
            self.performance.append(m_.get("res"))
            self.performance_ann.append(m_.get("res_ann"))
            self.ospa_list.append(m_.get("ospa"))
            self.ospa_list_ann.append(m_.get("ospa_ann"))
        else:
            for lst in (self.performance, self.performance_ann, self.ospa_list, self.ospa_list_ann):
                lst.append(None)
        return self._query(qp, X)

    def _query(self, qp: QueryPass, X):
        """Everything after the per-person loop: :465-649."""
        dev = qp.dev
        n = self.eval_len
        unl_idx = self.unlabeled_id.index
        unl = unlabelled_mask(n, self.labeled_id.index, dev)
        thc_h = qp.thc.cpu().numpy() if qp.use_thc else None
        wpu_h = qp.wpu.cpu().numpy() if qp.use_wpu else None
        if self.uncertainty == "THC+WPU":
            total_unc = float(thc_h.astype(np.float64).sum())
            UNC = {i: [t, w] for i, (t, w) in enumerate(zip(thc_h.tolist(), wpu_h.tolist()))}
        elif qp.use_thc or qp.use_wpu or qp.single:
            v = qp.single_score().cpu().numpy() if qp.single else (thc_h if qp.use_thc else wpu_h)
            total_unc = float(v.astype(np.float64).sum())
            UNC = dict(enumerate(v.tolist()))
        else:
            total_unc, UNC = 0.0, {i: 0 for i in range(n)}
        self.uncertainty_mean.append(total_unc / n)                                   # (:466)
        self.percentage.append(len(self.labeled_id) / n * 100)
        score = qp.fuse(unl, getattr(self.opt, "THCvsWPU", "const"), labeled_ratio=len(self.labeled_id) / n)
        if self.representativeness != "None":                                         # (:467-483)
            unl_t = torch.as_tensor(unl_idx, dtype=torch.int64, device=dev)
            infl = torch.zeros(n, dtype=torch.float64, device=dev)
            if len(unl_idx) in (0, 1):
                infl_u = np.zeros(len(unl_idx))
            elif self.representativeness == "Influence":
                infl = influence(X, unl)
                infl_u = infl[unl_t].cpu().numpy()
            else:                                                                     # "Random" (:476-477)
                infl_u = np.random.rand(len(unl_idx))
                infl[unl_t] = torch.from_numpy(infl_u).to(dev)
            self.influence_dict["Round" + str(self.round_cnt)] = dict(zip(map(int, unl_idx), map(float, infl_u)))
            if len(unl_idx) not in (0, 1):
                if self.uncertainty != "None":                                        # (:517-519)
                    score = ops.blend_scores(score, infl, qp.combine_weight, unl)
                else:                                                                 # (:525-526)
                    score = infl
        if len(unl_idx) > 0:
            self.combine_weight.append(qp.combine_weight)                             # (:486-488)
        if self.uncertainty != "None" and len(unl_idx) not in (0, 1):
            self.uncertainty_dict["Round" + str(self.round_cnt)] = UNC                # (:510,514)
        if self.filter == "Random" and len(unl_idx) > 1:                              # (:591-592, random_query :727-734)
            # unlabelled ids by descending score, ties in id order (sorted() is stable) (:527-530)
            cand = sorted(ops.rank_scores(score, unl, descending=True, count=8 * self.query_size).cpu().tolist())
            query_list = []
            while len(query_list) < self.query_size and len(cand) > 0:
                q = int(np.random.choice(cand))
                query_list.append(q)
                cand.remove(q)
        elif self.filter in ("K-Means", "weighted") and len(unl_idx) > 1:
            query_list = self._kmeans_query(X, score, unl_idx, qp.combine_weight)
        else:
            # (the first pick of "dist" is drawn only when the core-set runs: never with <= 1 unlabelled item)
            rule, first_pick = _coreset_rule(self, n) if self.filter == "Coreset" and len(unl_idx) > 1 else ("w_unc", -1)
            picks, _, stats = select(score, unl, X, self.query_size, self.filter, labeled=list(self.labeled_id.index),
                                     moks=float(self.moks_queried), lam=float(self.unc_lambda), rule=rule,
                                     first_pick=first_pick, batch=self.coreset_batch)
            query_list = [int(i) for i in picks.cpu().tolist()]
            if stats is not None:
                self.coreset_stats = stats
        self.last_query = SimpleNamespace(thc=qp.thc, wpu=qp.wpu, single=qp.aux, peak_mean=qp.peak_mean, kpts=qp.kpts,
                                          score=score, query_list=list(query_list))
        OKS_dict = self.OKS_dict
        if OKS_dict is None and self.oks_fn is not None:
            OKS_dict = dict(enumerate(np.asarray(self.oks_fn(list(range(n)), qp.kpts), dtype=np.float64).tolist()))
            self.OKS_dict = OKS_dict
        if OKS_dict is not None:                                                       # (:620-627)
            r = "Round" + str(self.round_cnt)
            self.true_labeled_dict[r] = self.get_corresponding_id(OKS_dict, true=True, labeled=True)
            self.true_unlabeled_dict[r] = self.get_corresponding_id(OKS_dict, true=True, labeled=False)
            self.false_labeled_dict[r] = self.get_corresponding_id(OKS_dict, true=False, labeled=True)
            self.false_unlabeled_dict[r] = self.get_corresponding_id(OKS_dict, true=False, labeled=False)
        if len(unl_idx) != 0:                                                          # (:629-649)
            if OKS_dict is None:
                w_unc_rule = (self.filter == "Coreset" and self.uncertainty != "None" and self.cfg.VAL.UNC_LAMBDA != 0
                              and not getattr(self.opt, "fixed_lambda", False))
                if w_unc_rule and getattr(self, "_strict_oks", False):
                    raise _lib.VatlqError(
                        "the Coreset filter weighs distance against uncertainty with the mean OKS of the queried items "
                        "(ActiveLearning.py:815-821,858): the loader must deliver GTkpts / bboxes_ann (batch[4], batch[8]) "
                        "or an oks_fn must be given — without them moks_queried would silently stay 0")
                self.moksQ_list.append(self.moks_queried)
            else:
                self.retrain_id = IndexCollection()
                retrain_id, self.moks_queried = self.get_retrain_id(query_list, OKS_dict)
                self.moksQ_list.append(self.moks_queried)
                self.retrain_id.update(retrain_id)
            self.labeled_id.update(query_list)
            self.unlabeled_id.difference_update(query_list)
            self.query_list_list["Round" + str(self.round_cnt)] = list(map(int, query_list))
            if OKS_dict is not None:
                self.actual_finish, self.finished_minerror, self.finished_oursc = self.is_finished(query_list, OKS_dict)
                if self.actual_finish < 100:
                    self.is_early_stop = True                                          # (:646-649)
        return None

    def _kmeans_query(self, X, score, unl_idx, combine_weight):
        """filter K-Means / weighted over the unlabelled ids `unl_idx` (query.select); self.query_size is clamped in
        place like the reference does (:558-561, 564-565)."""
        n = score.numel()
        unl = unlabelled_mask(n, np.setdiff1d(np.arange(n), np.asarray(unl_idx, dtype=np.int64)), score.device)
        picks, self.query_size, self.kmeans_stats = select(score, unl, X, self.query_size, self.filter, w_unc=self.w_unc,
                                                           combine_weight=combine_weight)
        return [int(i) for i in picks.cpu().tolist()]

    # ---- host bookkeeping on the per-item OKS values (tiny; ActiveLearning.py:707-725, 852-884) ----
    def get_retrain_id(self, query_list, OKS_dict):
        """ActiveLearning.get_retrain_id (:852-872): labelled items whose OKS is still low plus the new
        queries; mOKS of the new queries (mean taken in descending-OKS order like the reference)."""
        q = set(int(i) for i in query_list)
        oks_q = sorted((OKS for idx, OKS in OKS_dict.items() if idx in q), reverse=True)
        moks_queried = np.mean(oks_q)
        retrain_id = [idx for idx, OKS in OKS_dict.items() if idx in self.labeled_id and OKS <= self.finish_acc + self.finish_margin]
        retrain_id += list(query_list)
        return retrain_id, moks_queried

    def get_corresponding_id(self, OKS_dict, true=True, labeled=True):
        """ActiveLearning.get_corresponding_id (:874-884)."""
        thresh = self.finish_acc + self.finish_margin
        pool = self.labeled_id if labeled else self.unlabeled_id
        return [idx for idx, OKS in OKS_dict.items() if idx in pool and ((OKS >= thresh) if true else (OKS < thresh))]

    def is_finished(self, query_list, OKS_dict):
        """ActiveLearning.is_finished (:707-725): the three stopping criteria as label percentages."""
        time = (len(self.labeled_id) / self.eval_len) * 100
        vals = np.array(list(OKS_dict.values()))
        if np.all(vals >= self.finish_acc) and time < self.actual_finish:
            self.actual_finish = time
        OKS_q = np.array([OKS_dict[int(i)] for i in query_list])
        if np.mean(OKS_q) >= self.finish_acc and time < self.finished_minerror:
            self.finished_minerror = time
        OKS_lq = np.array([OKS_dict[int(i)] for i in self.labeled_id.index + list(query_list)])
        if np.all(OKS_lq >= self.finish_acc) and time < self.finished_oursc:
            self.finished_oursc = time
        return self.actual_finish, self.finished_minerror, self.finished_oursc

    def outcome(self):
        """ActiveLearning.outcome (:166-205).  Retraining itself (:651-686) is reference code behind
        `retrain_hook(self)`.  Returns None while rounds remain; when finished, the reference's 20-tuple
        (:203) — the evaluation members (performance, ospa) hold what `metrics_hook` delivered (None without)."""
        if self.is_early_stop or self.one_by_one:
            def last(lst):
                return lst[-1] if lst else None
            while len(self.performance) <= len(self.query_ratio):     # pad the remaining rounds (:169-178)
                self.round_cnt += 1
                self.performance.append(last(self.performance))
                self.performance_ann.append(last(self.performance_ann))
                self.ospa_list.append(last(self.ospa_list))
                self.ospa_list_ann.append(last(self.ospa_list_ann))
                self.uncertainty_mean.append(last(self.uncertainty_mean))
                self.percentage.append(self.query_ratio[min(self.round_cnt, len(self.query_ratio)) - 1] * 100)
                self.combine_weight.append(last(self.combine_weight))
                self.moksQ_list.append(last(self.moksQ_list))
            finish = True
        else:
            if self.retrain_hook is not None:
                self.retrain_hook(self)
            self.round_cnt += 1
            if len(self.unlabeled_id) == 0:
                self.eval_and_query()   # final evaluation round (:191-193)
                finish = True
            else:
                if self.round_cnt >= len(self.query_ratio):
                    self.query_size = len(self.unlabeled_id)                          # (:197-198)
                else:
                    self.query_size = self.query_sizes[self.round_cnt] - len(self.labeled_id)   # (:199-200)
                finish = False
        if not finish:
            return None
        return (self.percentage, self.performance, self.performance_ann, self.query_list_list, self.uncertainty_dict,
                self.uncertainty_mean, self.influence_dict, self.combine_weight, self.spearmanr_list, self.corr_list,
                self.true_labeled_dict, self.true_unlabeled_dict, self.false_labeled_dict, self.false_unlabeled_dict,
                self.actual_finish, self.finished_minerror, self.finished_oursc, self.ospa_list, self.ospa_list_ann,
                self.moksQ_list)
