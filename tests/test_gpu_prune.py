"""GPU: the exact pruning of the core-set passes (segments + triangle inequality, coreset.cu
"pruning") must not change a single bit: same picks, same min_d as the unpruned passes, zero
violations in verify mode, and the oracle's pick list on a pool the oracle can finish."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _select(v, X, unc, lab, k, moks, batch, mode, min_rows=0):
    v.ops.set_prune(mode, min_rows)
    v.ops.prune_stats(reset=True)
    try:
        # (tc_init=False: these tests are about the exact passes, including the labelled-set initialisation passes;
        #  the tensor-core initialisation has its own tests in test_gpu_tc.py)
        picks, st, md, _ = v.ops.coreset_select(X, unc, lab, k, moks, 0.01, batch=batch, return_state=True, tc_init=False)
        torch.cuda.synchronize()
    finally:
        v.ops.set_prune("env", -1)
    return picks, md, v.ops.prune_stats(reset=True)


def _ragged_clusters(n, d, seed):
    """Tracks of 1..90 rows (longer than the 64-row segment cap, and singletons)."""
    rng = np.random.default_rng(seed)
    sizes = []
    while sum(sizes) < n:
        sizes.append(int(rng.integers(1, 91)))
    assign = np.repeat(np.arange(len(sizes)), sizes)[:n]
    cen = (np.maximum(rng.standard_normal((len(sizes), d)), 0) * 0.5).astype(np.float32)
    return (cen[assign] + rng.normal(0, 0.01, (n, d)).astype(np.float32)).astype(np.float32)


@pytest.mark.parametrize("batch", [8, 16, 1])
def test_pruned_passes_change_nothing(built_lib, batch):
    v = built_lib
    n, k = 30000, 240 if batch == 1 else 640
    X = v.synth.device_embeddings(n, "cuda:0", seed=7)
    unc = torch.rand(n, dtype=torch.float64, device="cuda:0", generator=torch.Generator("cuda:0").manual_seed(8))
    p_off, md_off, s_off = _select(v, X, unc, [], k, 0.6, batch, "off")
    p_on, md_on, s_on = _select(v, X, unc, [], k, 0.6, batch, "on")
    p_ver, md_ver, s_ver = _select(v, X, unc, [], k, 0.6, batch, "verify")
    assert torch.equal(p_off, p_on) and torch.equal(p_off, p_ver)
    assert torch.equal(md_off, md_on) and torch.equal(md_off, md_ver)       # bit for bit
    assert s_off["segments"] == 0 and s_off["streamed"] == s_off["tiles"] > 0
    assert s_on["segments"] >= n // 64 and s_on["streamed"] < 0.9 * s_on["tiles"]   # clustered pool: tiles were pruned
    assert s_ver["violations"] == 0 and s_ver["streamed"] == s_ver["tiles"]


def test_pruning_with_labelled_set_ragged_tracks_and_iid(built_lib):
    v = built_lib
    rng = np.random.default_rng(3)
    for name, X in (("ragged", _ragged_clusters(12345, 2048, 11)),
                    ("iid", v.synth.embeddings(9001, d=2048, seed=12, clustered=False))):
        n = X.shape[0]
        Xd = torch.from_numpy(X).cuda()
        lab = sorted(rng.choice(n, n // 10, replace=False).tolist())
        u = rng.uniform(0, 1, n); u[lab] = 0
        unc = torch.from_numpy(u).cuda()
        for moks in (0.0, 0.6):
            p_off, md_off, _ = _select(v, Xd, unc, lab, 200, moks, 8, "off")
            p_on, md_on, s_on = _select(v, Xd, unc, lab, 200, moks, 8, "on")
            _, _, s_ver = _select(v, Xd, unc, lab, 200, moks, 8, "verify")
            assert torch.equal(p_off, p_on), (name, moks)
            assert torch.equal(md_off, md_on), (name, moks)
            assert s_ver["violations"] == 0, (name, moks, s_ver)
            assert s_on["streamed"] <= s_on["tiles"]


def test_pruned_selection_matches_oracle(built_lib):
    from oracle import vatl_oracle as O
    v = built_lib
    X = _ragged_clusters(2400, 2048, 5)
    unc = np.random.default_rng(6).uniform(0, 1, 2400)
    ref, md_ref = O.coreset_select(X.astype(np.float64), unc.copy(), [], 120, 0.6, 0.01)
    for batch in (8, 16):
        p, md, s = _select(v, torch.from_numpy(X).cuda(), torch.from_numpy(unc).cuda(), [], 120, 0.6, batch, "on")
        assert p.cpu().tolist() == ref, batch
        assert np.allclose(md.cpu().numpy(), md_ref, rtol=1e-9, atol=1e-6)   # sklearn's d(c,c) is ~1e-7, ours exactly 0
        assert s["streamed"] < s["tiles"]


def test_labelled_set_initialisation_is_pruned_exactly(built_lib):
    """The labelled-set initialisation (vatlq_coreset_init: n_labeled/8 passes) is pruned with the same
    filter: identical min_d / picks with a 20 % labelled set, fewer tiles streamed."""
    v = built_lib
    n = 30000
    X = v.synth.device_embeddings(n, "cuda:0", seed=17)
    rng = np.random.default_rng(18)
    lab = sorted(rng.choice(n, n // 5, replace=False).tolist())
    u = rng.uniform(0, 1, n); u[lab] = 0
    unc = torch.from_numpy(u).cuda()
    p_off, md_off, s_off = _select(v, X, unc, lab, 24, 0.6, 8, "off")
    p_on, md_on, s_on = _select(v, X, unc, lab, 24, 0.6, 8, "on")
    _, md_ver, s_ver = _select(v, X, unc, lab, 24, 0.6, 8, "verify")
    assert torch.equal(p_off, p_on) and torch.equal(md_off, md_on) and torch.equal(md_off, md_ver)
    assert s_ver["violations"] == 0
    assert s_ver["tiles"] > 700 * (n // 8)                 # the 750 initialisation passes were counted (verify collects them)


@pytest.mark.parametrize("batch", [8, 16])
def test_tile_counts_are_the_passes_rows(built_lib, batch):
    """Every pass that applies centres sees each owned 8-row tile once, and nothing else counts as a tile: in
    particular not the segment filter's tiles of anchor rows (batch 8: the solo filter, batch 16: the paired one)."""
    v = built_lib
    n = 20005
    X = torch.from_numpy(_ragged_clusters(n, 2048, 21)).cuda()
    unc = torch.from_numpy(np.random.default_rng(22).uniform(0, 1, n)).cuda()
    v.ops.set_prune("on", 0)
    try:
        _, st = v.ops.coreset_select(X, unc, [], 300, 0.6, 0.01, batch=batch, tc_init=False)
        torch.cuda.synchronize()
    finally:
        v.ops.set_prune("env", -1)
    assert st.passes > 0 and st.tiles_streamed < st.tiles       # tiles were pruned, so the filter ran
    assert st.tiles == st.passes * ((n + 7) // 8), (st.tiles, st.passes)
