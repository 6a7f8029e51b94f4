"""The fp16 screen of the paired pass (coreset.cu, "the screen") on inputs where fp16 differs most from fp32:
elements beyond the fp16 range (the copy holds +-Inf), elements in the fp16 subnormal range, a row of huge norm.
Screen on, off and verify must agree bit for bit with zero verify violations.  The CPU tests check the restated
error bound on fp16-rounded dot products at K = 2048 and the workspace size of the copy."""
import numpy as np
import pytest
import torch

from test_gpu_pass_screen import _check

K = 2048
U = 2.0 ** -8
ABS = 2.0 ** -18     # |S~ - S| <= u |x||c| + 2^-18 (|x| + |c|): half of E's 2u and 2^-17 terms


def _pool(v, n, seed, kind="clustered"):
    return v.synth.pool_embeddings(n, d=K, seed=seed, kind=kind, device="cuda:0").clone()


@pytest.mark.gpu
def test_rows_beyond_fp16_range(built_lib):
    """Rows with |x_k| >= 65520 in columns where every other row is 0: their copy holds Inf, they are picked
    early (so the round's centres carry Inf), and every other centre is 0 there (Inf x 0 = NaN in S~)."""
    v = built_lib
    n = 20011
    X = _pool(v, n, 21)
    X[:, :64] = 0
    rng = np.random.default_rng(21)
    big = torch.from_numpy(rng.choice(n, 40, replace=False)).cuda()
    X[big, :64] = torch.from_numpy(rng.choice([-1.0, 1.0], (40, 64)) * rng.uniform(65520, 1e5, (40, 64))).float().cuda()
    unc = v.synth.pool_unc(n, device="cuda:0")
    picks, _, _, _ = v.ops.coreset_select(X, unc, [], 320, 0.0, 0.01, batch=16, return_state=True)
    assert np.isin(big.cpu().numpy(), picks.cpu().numpy()).any()
    _check(v, X, unc, [], 320, 0.0, 16, "beyond fp16 range")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["clustered", "iid"])
def test_fp16_subnormal_pool(built_lib, kind):
    """The whole pool scaled into the fp16 subnormal range (|x_k| < 6.1e-5 for almost every element): the
    absolute term of E is what keeps the screen exact here."""
    v = built_lib
    n = 16007
    X = _pool(v, n, 23, kind)
    X *= 1.5e-5 / X.pow(2).mean().sqrt()     # rms element 1.5e-5
    assert (X.abs() < 6.1e-5).float().mean().item() > 0.99
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], 320, 0.0, 16, f"subnormal {kind}")
    assert s["screened"] > 0


@pytest.mark.gpu
def test_huge_norm_row_and_subnormal_rows(built_lib):
    """A row 10^3 times longer than the rest and a block of rows in the subnormal range among ordinary rows."""
    v = built_lib
    n = 24001
    X = _pool(v, n, 25)
    X[5000] *= 1000.0
    X[7000:7300] *= 1e-4
    unc = v.synth.pool_unc(n, device="cuda:0")
    _check(v, X, unc, [], 480, 0.0, 16, "huge norm + subnormal rows")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["clustered", "iid"])
def test_ragged_pools(built_lib, kind):
    """n = 1 mod 16: the last tile is ragged and the screen's last stage holds a lone tile on one CTA of a pair."""
    v = built_lib
    n = 40017
    X = _pool(v, n, 27, kind)
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], 640, 0.0, 16, f"ragged {kind}")
    assert s["screened"] > 0 and s["listed"] < s["screened"]


def _adversarial(rng):
    """Pairs (x, c) of fp32 vectors at K = 2048 on which fp16 rounding hurts: mixed scales, fp16 subnormals,
    elements just inside the fp16 range, values between fp16 grid points, cancelling sums."""
    out = []
    for t in range(64):
        x = rng.standard_normal(K)
        c = rng.standard_normal(K)
        kind = t % 8
        if kind == 0:      # per-element scales from 2^-30 to 2^14
            x *= 2.0 ** rng.uniform(-30, 14, K)
            c *= 2.0 ** rng.uniform(-30, 14, K)
        elif kind == 1:    # all subnormal in fp16
            x *= 2e-5
            c *= 2e-5
        elif kind == 2:    # subnormal rows against an ordinary centre
            x *= 3e-5
        elif kind == 3:    # near the top of the fp16 range
            x = np.clip(x * 2e4, -65500, 65500)
            c = rng.uniform(-1, 1, K)
        elif kind == 4:    # cancellation: c close to -x, S near -|x|^2 with large terms
            c = -x + 1e-3 * rng.standard_normal(K)
        elif kind == 5:    # cancellation with S close to 0: c orthogonal-ish to x with large terms
            c = x.copy()
            c[K // 2:] *= -1
        elif kind == 6:    # halfway points of the fp16 grid (round-to-nearest-even ties)
            x = (np.round(rng.uniform(1, 2, K) * 1024) + 0.5) / 1024
            c = (np.round(rng.uniform(1, 2, K) * 1024) + 0.5) / 1024 * rng.choice([-1, 1], K)
        else:              # mixed: half the elements subnormal, half ordinary
            x[: K // 2] *= 1e-5
            c[K // 2:] *= 1e-5
        out.append((x.astype(np.float32), c.astype(np.float32)))
    return out


def _fp32_tree_dot(xh, ch):
    """The products of the fp16 operands (exact in fp32), summed in fp32 as the screen does: 16 features per MMA
    step in a sequential chain per K segment of 256, the 8 segments added in fp64."""
    p = (xh.astype(np.float64) * ch.astype(np.float64)).astype(np.float32).reshape(8, 16, 16)
    seg = np.zeros(8, np.float32)
    for s in range(16):
        step = np.zeros(8, np.float32)
        for e in range(16):
            step = (step + p[:, s, e]).astype(np.float32)
        seg = (seg + step).astype(np.float32)
    return float(np.sum(seg.astype(np.float64)))


def test_fp16_bound_on_adversarial_vectors():
    rng = np.random.default_rng(5)
    worst = 0.0
    for x, c in _adversarial(rng):
        xh, ch = x.astype(np.float16), c.astype(np.float16)   # round to nearest even, like cvt.rn
        assert np.isfinite(xh).all() and np.isfinite(ch).all()
        S = float(np.sum(x.astype(np.longdouble) * c.astype(np.longdouble)))   # fp32 x fp32 is exact in fp64
        nx = float(np.sqrt(np.sum(x.astype(np.float64) ** 2)))
        nc = float(np.sqrt(np.sum(c.astype(np.float64) ** 2)))
        bound = U * nx * nc + ABS * (nx + nc)
        exact16 = float(np.sum(xh.astype(np.longdouble) * ch.astype(np.longdouble)))
        for St in (exact16, _fp32_tree_dot(xh, ch)):
            assert abs(St - S) <= bound, (St, S, bound)
            worst = max(worst, abs(St - S) / bound)
    assert worst < 0.5    # the bound keeps a margin of at least 2 on these vectors


def test_rounding_model_of_the_bound():
    """|dv| <= 2^-11 |v| + 2^-25 and |dv| <= |v| for every fp32 value inside the fp16 range."""
    rng = np.random.default_rng(6)
    v = np.concatenate([rng.standard_normal(200000) * 2.0 ** rng.uniform(-40, 15, 200000),
                        np.float32(2.0 ** -14) * rng.uniform(-1, 1, 50000)]).astype(np.float32)
    v = v[np.abs(v) < 65504]
    dv = np.abs(v.astype(np.float16).astype(np.float64) - v.astype(np.float64))
    av = np.abs(v.astype(np.float64))
    assert (dv <= 2.0 ** -11 * av + 2.0 ** -25).all()
    assert (dv <= av).all()
    with np.errstate(over="ignore"):
        assert np.isinf(np.float32(65520).astype(np.float16)) and np.float32(65519).astype(np.float16) == 65504


def test_workspace_holds_the_copy_only_for_paired_rounds(built_lib):
    L = built_lib._lib.lib()
    for n in (1, 30001, 1_000_000):
        base = L.vatlq_coreset_workspace_bytes(n, K, 1)
        for d, batch, extra in ((K, 1, 0), (K, 8, 0), (K, 15, 0), (K, 16, n * 4096), (K, 64, n * 4096),
                                (1024, 16, None), (256, 16, None)):
            got = L.vatlq_coreset_workspace_bytes(n, d, batch)
            if extra is None:
                assert got == L.vatlq_coreset_workspace_bytes(n, d, 1)
            else:
                assert got == base + extra, (n, d, batch)
