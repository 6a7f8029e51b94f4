"""GPU: the core-set on fp16 / bf16 embeddings.  Contract (include/vatlq.h, vatlq_coreset_*_dt): every output for a
16-bit X — picks, min_d, unc and the counting fields of CoresetStats — equals, bit for bit, the output of the same call
on X.float(), in every screen and prune mode; so does pairwise_dist.  The reference here is always the fp32 path on the
exact upcast of the 16-bit pool."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

K = 2048
DTYPES = [torch.float16, torch.bfloat16]
COUNTS = ("passes", "picks", "rounds", "fallback_empty", "fallback_overflow", "candidates", "rounds_launched", "batch",
          "tiles", "tiles_streamed", "prune_violations", "segments")


def _bits(t):
    return t.contiguous().view(torch.int64)


def _select(v, X, unc, lab, k, moks, batch=16, rule="w_unc", first_pick=-1, screen="on", prune="on"):
    v.ops.set_screen(screen)
    v.ops.set_prune(prune)
    v.ops.screen_stats(reset=True)
    v.ops.prune_stats(reset=True)
    try:
        # (tc_init=False: both dtypes through vatlq_coreset_init_dt, the entry the contract is about)
        picks, st, md, u = v.ops.coreset_select(X, unc, lab, k, moks, 0.01, rule=rule, first_pick=first_pick,
                                                batch=batch, return_state=True, tc_init=False)
        torch.cuda.synchronize()
    finally:
        v.ops.set_screen("env")
        v.ops.set_prune("env")
    return picks, st, md, u, v.ops.screen_stats(reset=True), v.ops.prune_stats(reset=True)


def _check(v, X16, unc, lab, k, moks, name, **kw):
    """X16 against its fp32 upcast: every output bit for bit; returns the 16-bit run's screen statistics."""
    assert X16.dtype in DTYPES
    ref = _select(v, X16.float(), unc, lab, k, moks, **kw)
    got = _select(v, X16, unc, lab, k, moks, **kw)
    assert torch.equal(ref[0], got[0]), name
    for f in COUNTS:
        assert getattr(ref[1], f) == getattr(got[1], f), (name, f)
    assert torch.equal(_bits(ref[2]), _bits(got[2])), name
    assert torch.equal(_bits(ref[3]), _bits(got[3])), name
    assert ref[4]["screened"] == got[4]["screened"], (name, ref[4], got[4])
    assert ref[4]["violations"] == 0 and got[4]["violations"] == 0, (name, ref[4], got[4])
    assert ref[5]["violations"] == 0 and got[5]["violations"] == 0, (name, ref[5], got[5])
    assert got[1].prune_violations == 0
    return got[4]


def _pool(v, n, seed, dtype, kind="clustered", d=K):
    return v.synth.pool_embeddings(n, d=d, seed=seed, kind=kind, device="cuda:0").to(dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["clustered", "weak", "iid"])
def test_pools_equal_upcast(built_lib, kind, dtype):
    v = built_lib
    n = 20011                                   # ragged: not a multiple of 8 or 16
    X = _pool(v, n, 31, dtype, kind)
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], 400, 0.0, f"{kind} {dtype}")
    assert s["screened"] > 0 and s["listed"] < s["screened"]


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("batch", [1, 8, 16])
def test_batches(built_lib, batch, dtype):
    v = built_lib
    n = 9001
    X = _pool(v, n, 33, dtype)
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], 48 if batch == 1 else 160, 0.0, f"batch {batch} {dtype}", batch=batch)
    if batch < 16:
        assert s["screened"] == 0                # an unpaired selection (the solo pass) does not screen


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("d", [1000, 256])     # pass_kernel_generic: a ragged last super-step, and a short row
def test_generic_widths(built_lib, d, dtype):
    v = built_lib
    n = 5003
    X = _pool(v, n, 35, dtype, d=d)
    unc = v.synth.pool_unc(n, device="cuda:0")
    lab = np.random.default_rng(35).choice(n, 300, replace=False)
    _check(v, X, unc, lab, 96, 0.6, f"d {d} {dtype}")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rule", ["w_unc", "fixed_lambda", "dist"])
def test_rules_with_labelled_set(built_lib, rule, dtype):
    """A labelled set of 10 % at mOKS 0.6 (the init passes with pruning) and every selection rule."""
    v = built_lib
    n = 20011
    X = _pool(v, n, 37, dtype)
    unc = v.synth.pool_unc(n, device="cuda:0")
    lab = np.random.default_rng(37).choice(n, n // 10, replace=False)
    _check(v, X, unc, lab, 320, 0.6, f"{rule} {dtype}", rule=rule)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("rule", ["w_unc", "fixed_lambda", "dist"])
def test_rules_empty_labelled_set(built_lib, rule, dtype):
    v = built_lib
    n = 12007
    X = _pool(v, n, 39, dtype)
    unc = v.synth.pool_unc(n, device="cuda:0")
    _check(v, X, unc, [], 240, 0.0, f"{rule} {dtype}", rule=rule, first_pick=77 if rule == "dist" else -1)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("prune", ["off", "on", "verify"])
@pytest.mark.parametrize("screen", ["off", "on", "verify"])
def test_screen_and_prune_modes(built_lib, screen, prune, dtype):
    v = built_lib
    n = 16007
    X = _pool(v, n, 41, dtype)
    unc = v.synth.pool_unc(n, device="cuda:0")
    lab = np.random.default_rng(41).choice(n, n // 10, replace=False)
    s = _check(v, X, unc, lab, 256, 0.6, f"screen {screen} prune {prune} {dtype}", screen=screen, prune=prune)
    assert (s["screened"] > 0) == (screen != "off")


@pytest.mark.parametrize("dtype", DTYPES)
def test_duplicate_and_nan_rows(built_lib, dtype):
    v = built_lib
    n = 16007
    X = _pool(v, n, 43, dtype)
    X[100:400] = X[100]                         # d = 0 ties
    X[9000:9020] = X[8999]
    X[12345, 7] = float("nan")
    X[15000] = float("nan")
    unc = v.synth.pool_unc(n, device="cuda:0")
    _check(v, X, unc, [], 320, 0.0, f"duplicates + NaN {dtype}")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["clustered", "iid"])
def test_fp16_subnormal_scale(built_lib, kind, dtype):
    """The pool scaled to an rms element of 1.5e-5: almost every element is an fp16 subnormal."""
    v = built_lib
    n = 16007
    X32 = v.synth.pool_embeddings(n, d=K, seed=45, kind=kind, device="cuda:0")
    X = (X32 * (1.5e-5 / X32.pow(2).mean().sqrt())).to(dtype)
    if dtype == torch.float16:
        assert (X.float().abs() < 6.1e-5).float().mean().item() > 0.99
    unc = v.synth.pool_unc(n, device="cuda:0")
    s = _check(v, X, unc, [], 320, 0.0, f"subnormal {kind} {dtype}")
    assert s["screened"] > 0


def test_bf16_dot_products_overflowing_fp32(built_lib):
    """bf16 rows with elements near 1e30 in 64 columns where the rest of the pool is 0: they are picked early, and
    their dot products with each other overflow fp32 (Inf in the screen's S~).  Such rows must be listed, not
    decided, and the picks must still equal the upcast's."""
    v = built_lib
    n = 20011
    X = _pool(v, n, 47, torch.bfloat16)
    X[:, :64] = 0
    rng = np.random.default_rng(47)
    big = torch.from_numpy(rng.choice(n, 40, replace=False)).cuda()
    X[big, :64] = torch.from_numpy(rng.choice([-1.0, 1.0], (40, 64)) * rng.uniform(1e29, 1e30, (40, 64))).to(
        torch.bfloat16).cuda()
    S = X[big].float() @ X[big].float().T
    assert not torch.isfinite(S).all()          # these dot products do overflow fp32
    unc = v.synth.pool_unc(n, device="cuda:0")
    ref = _select(v, X.float(), unc, [], 320, 0.0)
    assert np.isin(big.cpu().numpy(), ref[0].cpu().numpy()).sum() >= 2
    s = _check(v, X, unc, [], 320, 0.0, "bf16 overflow")
    assert s["listed"] >= 40


@pytest.mark.parametrize("dtype", DTYPES)
def test_default_init_resolution(built_lib, dtype):
    """tc_init=None: the fp32 upcast takes the tcgen05 init (>= 256 labelled rows at d = 2048), the 16-bit X the
    exact init; both give the same bits (the tcgen05 init equals the exact one)."""
    v = built_lib
    n = 12007
    X = _pool(v, n, 53, dtype)
    unc = v.synth.pool_unc(n, device="cuda:0")
    lab = np.random.default_rng(53).choice(n, 600, replace=False)
    a = v.ops.coreset_select(X.float(), unc, lab, 160, 0.6, 0.01, return_state=True)
    b = v.ops.coreset_select(X, unc, lab, 160, 0.6, 0.01, return_state=True)
    assert torch.equal(a[0], b[0]) and torch.equal(_bits(a[2]), _bits(b[2])) and torch.equal(_bits(a[3]), _bits(b[3]))
    with pytest.raises(v._lib.VatlqError, match="tc_init"):
        v.ops.coreset_select(X, unc, lab, 160, 0.6, 0.01, tc_init=True)


@pytest.mark.parametrize("dtype", DTYPES)
def test_workspace_drops_the_copy(built_lib, dtype):
    v = built_lib
    L = v._lib.lib()
    dt = v.ops.EMBEDDING_DTYPES[dtype]
    for n in (30001, 1_000_000):
        f32 = L.vatlq_coreset_workspace_bytes_dt(n, K, 16, v._lib.F32)
        assert f32 == L.vatlq_coreset_workspace_bytes(n, K, 16)
        assert L.vatlq_coreset_workspace_bytes_dt(n, K, 16, dt) == f32 - n * 4096
        for d, batch in ((K, 8), (1000, 16)):
            assert L.vatlq_coreset_workspace_bytes_dt(n, d, batch, dt) == L.vatlq_coreset_workspace_bytes(n, d, batch)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("d", [K, 1000])
def test_pairwise_dist_equal_upcast(built_lib, d, dtype):
    v = built_lib
    n = 3001
    X = _pool(v, n, 49, dtype, d=d)
    X[5] = float("nan")
    centers = [0, 5, 17, 1234, 3000, 17, 2999, 8, 9]
    a = v.ops.pairwise_dist(X.float(), centers)
    b = v.ops.pairwise_dist(X, centers)
    assert torch.equal(_bits(a), _bits(b))


@pytest.mark.parametrize("dtype", DTYPES)
def test_8_byte_aligned_view(built_lib, dtype):
    """A 16-bit X that is 8- but not 16-byte aligned runs at d = 1000 (equal to the upcast) and is refused at
    d = 2048, where the passes copy whole rows with TMA."""
    v = built_lib
    n = 2001
    buf = torch.empty(n * 1000 + 4, dtype=dtype, device="cuda:0")
    buf[4:] = _pool(v, n, 51, dtype, d=1000).reshape(-1)
    X = buf[4:].view(n, 1000)
    assert X.data_ptr() % 16 == 8
    unc = v.synth.pool_unc(n, device="cuda:0")
    _check(v, X, unc, [], 64, 0.0, f"8-byte aligned {dtype}")
    X2 = torch.zeros(n * K + 4, dtype=dtype, device="cuda:0")[4:].view(n, K)
    with pytest.raises(v._lib.VatlqError, match="16-byte"):
        v.ops.coreset_select(X2, unc, [], 8, 0.0, 0.01)
