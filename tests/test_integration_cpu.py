"""INTEGRATION.md §A executed: the glue of vatl4pose-wacv2024_b200/integration.py against an object shaped like the
reference's ActiveLearning.  The glue only reads and writes attributes of that object, calls the hooks the test
installs (retrain_model, save_GT_dict, initialize_estimator) and rebuilds its ids with type(ref.labeled_id); so the
stand-in is a bare class, with a distinct subclass of the package's restatement of alipy's IndexCollection, so that
the test sees which type the glue builds, and the bounding-box conversion is the oracle's restatement of alphapose's
bbox_xyxy_to_xywh (pinned against the reference by oracle/pin_against_reference.py)."""
import json
import os
from types import SimpleNamespace

import numpy as np
import pytest
import torch


@pytest.fixture(scope="module")
def R():
    import vatlq
    from oracle import vatl_oracle as O

    class AL:                                        # the reference class, created without its __init__
        pass

    class IndexCollection(vatlq.IndexCollection):    # the reference's alipy IndexCollection
        pass
    return SimpleNamespace(AL=AL, IndexCollection=IndexCollection, bbox_xyxy_to_xywh=O.xyxy_to_xywh)


def _cfg_opt(tmp):
    cfg = SimpleNamespace(VAL=SimpleNamespace(QUERY_RATIO=[0.1, 0.3], W_UNC=1.0, UNC_LAMBDA=0.01),
                          DATA_PRESET=SimpleNamespace(HEATMAP_SIZE=[64, 48]), AE=SimpleNamespace(Z_DIM=4),
                          RETRAIN=SimpleNamespace(BASE=10, ALPHA=20))
    opt = SimpleNamespace(strategy="THC+None_Nonefilter", uncertainty="THC", representativeness="None", filter="None",
                          video_id="0", THCvsWPU="const", fixed_lambda=False, onebyone=False, retrain_thresh=0.9,
                          work_dir=str(tmp))
    return cfg, opt


def test_retrain_hook_drives_the_reference_object(R, tmp_path):
    import vatlq
    from vatlq import integration
    cfg, opt = _cfg_opt(tmp_path)
    ref = R.AL.__new__(R.AL)                         # the reference class, no __init__
    calls = []
    ref.cfg, ref.opt, ref.continual = cfg, opt, True
    ref.labeled_id, ref.unlabeled_id, ref.retrain_id = R.IndexCollection(), R.IndexCollection(list(range(20))), R.IndexCollection()
    ref.model, ref.AE, ref.eval_loader, ref.eval_len = "estimator-v0", "ae-v0", None, 20
    ref.eval_dataset = list(range(20))

    def fake_retrain():
        calls.append((list(ref.retrain_id.index), ref.retrain_epoch, ref.round_cnt))
        ref.model, ref.AE = "estimator-v1", "ae-v1"
    ref.retrain_model = fake_retrain
    al = vatlq.ActiveLearning(cfg, opt, **integration.from_reference(ref, with_metrics=False))
    assert al.model == "estimator-v0" and al.eval_len == 20 and al.query_size == 2
    # state as eval_and_query leaves it after a round with OKS available
    al.labeled_id.update([3, 7]); al.unlabeled_id.difference_update([3, 7]); al.retrain_id.update([3, 7])
    al.moks_queried = 0.75
    assert al.outcome() is None                      # -> retrain_hook -> the reference's retrain_model
    assert calls == [([3, 7], int(20 * (1 - 0.75)), 0)]                      # epoch rule of ActiveLearning.py:183
    assert isinstance(ref.labeled_id, R.IndexCollection) and ref.labeled_id.index == [3, 7]
    assert ref.unlabeled_id.index == [i for i in range(20) if i not in (3, 7)] and ref.moks_queried == 0.75
    assert al.model == "estimator-v1" and al.AE == "ae-v1"                   # the fine-tuned AE is picked up (:681-685)
    assert al.round_cnt == 1 and al.query_size == int(20 * 0.3) - 2
    ref.continual = False                            # non-continual: estimator re-initialised, BASE-scaled epochs (:179-182)
    ref.initialize_estimator = lambda: ("estimator-fresh", "opt", "sched")
    al.outcome()
    assert calls[-1][1] == int(10 * 2 / 20 + 20 * (1 - 0.75))


def test_prediction_records_and_metrics_hook(R, tmp_path):
    import vatlq
    from vatlq import integration
    cfg, opt = _cfg_opt(tmp_path)
    ref = SimpleNamespace(opt=opt, save_GT_dict=lambda gt: (json.dump(gt, open(os.path.join(str(tmp_path), "GT.json"), "w")),
                                                              os.path.join(str(tmp_path), "GT.json"))[1])
    seen = []
    pc = integration.PredictionCollector(ref, evaluate_mAP=lambda p, ann_type, ann_file: (seen.append(("map", p, ann_file)), {"AP": 1.0})[1],
                                         ospa_for_loc=lambda ann_json_path, pr_json_path: (seen.append(("ospa", pr_json_path)), 0.5)[1],
                                         bbox_xyxy_to_xywh=R.bbox_xyxy_to_xywh)
    al = SimpleNamespace(labeled_id=vatlq.IndexCollection([1]), OKS_dict={0: 0.9, 1: 0.8})
    kp = torch.arange(2 * 51, dtype=torch.float32).reshape(2, 17, 3)
    gt = np.ones((2, 17, 3), np.float32)
    batch = ([0, 1], None, None, None, gt, [11, 12], [101, 102], None, np.array([[0, 0, 9, 19], [5, 5, 14, 24]], np.float32), None, None)
    pc.eval_hook(al, batch, kp)
    out = pc.metrics_hook(al, kp)
    assert out == {"res": {"AP": 1.0}, "ospa": 0.5, "res_ann": {"AP": 1.0}, "ospa_ann": 0.5}
    rec = json.load(open(os.path.join(str(tmp_path), "predicted_kpt.json")))
    ann = json.load(open(os.path.join(str(tmp_path), "predicted_kpt_ann.json")))
    # the record layout of ActiveLearning.py:312-326
    assert rec[0]["bbox"] == list(R.bbox_xyxy_to_xywh([0, 0, 9, 19])) == [0, 0, 10, 20] and rec[1]["image_id"] == 12 and rec[1]["id"] == 102
    s = kp[0, :, 2].numpy()
    assert np.isclose(rec[0]["score"], float(np.mean(s) + 1.25 * np.max(s))) and rec[0]["category_id"] == 1
    assert rec[1]["keypoints"] == kp[1].reshape(-1).tolist() and ann[1]["keypoints"] == gt[1].reshape(-1).tolist()   # labelled -> GT (:322-323)
    assert ann[0]["keypoints"] == rec[0]["keypoints"] and rec[0]["OKS"] == 0.9
    assert [s_[0] for s_ in seen] == ["map", "ospa", "map", "ospa"]
