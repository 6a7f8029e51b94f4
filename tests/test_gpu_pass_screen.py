"""GPU: the TF32 screen of the paired pass (coreset.cu, "the screen") decides which rows skip the exact fp64
arithmetic; it must not change a single bit: same picks, min_d and uncertainties as with the screen off, and zero
violations in verify mode (rows the screen did not list whose min_d moved anyway)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _select(v, X, unc, lab, k, moks, batch, mode):
    v.ops.set_screen(mode)
    v.ops.screen_stats(reset=True)
    try:
        picks, _, md, u = v.ops.coreset_select(X, unc, lab, k, moks, 0.01, batch=batch, return_state=True)
        torch.cuda.synchronize()
    finally:
        v.ops.set_screen("env")
    return picks, md, u, v.ops.screen_stats(reset=True)


def _bits(t):
    return t.contiguous().view(torch.int64)


def _check(v, X, unc, lab, k, moks, batch, name):
    p_off, md_off, u_off, s_off = _select(v, X, unc, lab, k, moks, batch, "off")
    p_on, md_on, u_on, s_on = _select(v, X, unc, lab, k, moks, batch, "on")
    p_ver, md_ver, u_ver, s_ver = _select(v, X, unc, lab, k, moks, batch, "verify")
    assert torch.equal(p_off, p_on) and torch.equal(p_off, p_ver), name
    assert torch.equal(_bits(md_off), _bits(md_on)) and torch.equal(_bits(md_off), _bits(md_ver)), name
    assert torch.equal(_bits(u_off), _bits(u_on)) and torch.equal(_bits(u_off), _bits(u_ver)), name
    assert s_off["screened"] == 0
    assert s_ver["violations"] == 0, (name, s_ver)
    assert s_on["listed"] <= s_on["screened"]
    if s_on["screened"]:
        print(f"{name}: batch {batch}, listed / screened rows f = {s_on['listed'] / s_on['screened']:.4f} "
              f"({s_on['listed']} / {s_on['screened']})")
    return s_on


@pytest.mark.parametrize("kind", ["clustered", "weak", "iid"])
def test_screen_changes_nothing(built_lib, kind):
    v = built_lib
    n, k = 30001, 480                     # ragged: not a multiple of 8 or 128
    X = v.synth.pool_embeddings(n, d=2048, seed=2, kind=kind, device="cuda:0")
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], k, 0.0, 16, kind)
    assert s["screened"] > 0 and s["listed"] < s["screened"]


@pytest.mark.parametrize("batch", [1, 8])
def test_short_rounds_do_not_screen(built_lib, batch):
    v = built_lib
    n = 12345
    X = v.synth.pool_embeddings(n, d=2048, seed=4, kind="clustered", device="cuda:0")
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], 64 if batch == 1 else 160, 0.0, batch, f"batch {batch}")
    assert s["screened"] == 0


def test_screen_duplicates_nan_rows_and_labelled_round(built_lib):
    v = built_lib
    n = 20011
    rng = np.random.default_rng(9)
    X = v.synth.pool_embeddings(n, d=2048, seed=6, kind="clustered", device="cuda:0").clone()
    dup = rng.choice(n, 400, replace=False)
    X[torch.from_numpy(dup[:200]).cuda()] = X[torch.from_numpy(dup[200:]).cuda()]   # d = 0 ties
    X[17, 5] = float("nan")
    X[9000, :] = float("nan")
    unc = v.synth.pool_unc(n, device="cuda:0")
    _check(v, X, unc, [], 320, 0.0, 16, "duplicates + NaN rows")
    lab = sorted(rng.choice(n, n // 10, replace=False).tolist())
    u = unc.clone()
    u[torch.tensor(lab, device="cuda:0")] = 0
    _check(v, X, u, lab, 320, 0.6, 16, "10 % labelled, mOKS 0.6")
