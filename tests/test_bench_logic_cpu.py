"""CPU: the parts of bench.py that decide pass / fail — the pick-list hash, the golden lookup for a configuration and
the parity verdict (a wrong pick list must turn into `ok: False`, which bench.py maps to exit code 3)."""
import numpy as np


def test_golden_lookup_and_parity_verdict():
    import bench
    z = np.load("tests/golden/coreset_scale_c4.npz")
    picks = z["picks"].astype(np.int64)
    assert bench.sha_picks(picks) == str(z["sha256"])
    tag, gold, k_full = bench.golden_for(4, 170000, 0.0, 0.0, "clustered")
    assert tag == "c4" and k_full == 8500 and np.array_equal(gold, picks)
    assert bench.golden_for(4, 170000, 0.1, 0.6, "clustered")[0] == "c4lab"
    assert bench.golden_for(4, 170001, 0.0, 0.0, "clustered")[0] is None          # another pool: nothing pinned
    assert bench.golden_for(4, 170000, 0.0, 0.0, "iid")[0] is None
    ok = bench.check_golden(4, 170000, 8500, 0.0, 0.0, "clustered", picks)
    assert ok["pinned"] and ok["ok"] and ok["whole_list"] and ok["reference_picks_compared"] == 8500
    bad = picks.copy()
    bad[4321], bad[4322] = bad[4322], bad[4321]                                  # same set, wrong order
    v = bench.check_golden(4, 170000, 8500, 0.0, 0.0, "clustered", bad)
    assert v["pinned"] and not v["ok"] and v["first_difference_at"] == 4321
    # a prefix golden (config 5: the CPU produced the first 400 picks of 50 000)
    z5 = np.load("tests/golden/coreset_scale_c5.npz")
    long_list = np.concatenate([z5["picks"], np.arange(10 ** 6 - 49600, 10 ** 6)])
    v5 = bench.check_golden(5, 1000000, 50000, 0.0, 0.0, "clustered", long_list)
    assert v5["ok"] and not v5["whole_list"] and v5["reference_picks_compared"] == 400
    assert not bench.check_golden(5, 1000000, 49999, 0.0, 0.0, "clustered", long_list)["ok"]     # another k: not this workload
    assert bench.check_golden(3, 12345, 10, 0.0, 0.0, "clustered", [1, 2, 3])["pinned"] is False


def test_traffic_table_and_peaks():
    import bench
    assert bench.ncu_traffic("pass_kernel_pruned", 1000000) > 3e9
    assert bench.ncu_traffic("scan", 170000) > 35e9 and bench.ncu_traffic("scan", 123) is None
    gbs, src = bench.peak_hbm()
    assert 3000 < gbs < 9000 and isinstance(src, str)


def test_dump_outputs_budget_and_fixed_sample(tmp_path):
    import torch
    import bench
    from vatlq.query import QueryResult
    n = 1 << 20
    res = QueryResult(picks=torch.arange(5000, 0, -1), thc=torch.rand(n), wpu=torch.rand(n), peak_mean=torch.rand(n),
                      kpts=torch.rand(n, 17, 3), unc=torch.rand(n, dtype=torch.float64), combine_weight=0.25, stats=object())
    out = bench.result_arrays(res)
    assert sorted(out) == ["combine_weight", "kpts", "peak_mean", "picks", "thc", "unc", "wpu"]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["combine_weight.npy", "kpts.npy", "kpts_rows.npy", "peak_mean.npy", "picks.npy", "thc.npy", "unc.npy", "wpu.npy"]
    assert sum(p.stat().st_size for p in (tmp_path / "a").iterdir()) <= 64 << 20
    for f in files:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype in (np.float32, np.float64) and np.array_equal(x, y)
    rows = np.load(tmp_path / "a" / "kpts_rows.npy").astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "kpts.npy"), res.kpts[torch.from_numpy(rows)].numpy())
    assert np.array_equal(np.load(tmp_path / "a" / "picks.npy"), np.arange(5000, 0, -1, dtype=np.float64))
    assert np.array_equal(np.load(tmp_path / "a" / "thc.npy"), res.thc.numpy())
    assert np.load(tmp_path / "a" / "combine_weight.npy").tolist() == [0.25]
