"""GPU: the Influence / Diversity cosine row sums on fp16 / bf16 embeddings.  Contract (include/vatlq.h,
vatlq_cosine_*_dt): for a 16-bit X the column sums S, the row sums, the min-max-normalised Influence and the Diversity
picks equal, bit for bit, those of the fp32 path on X.float().  The reference here is always the fp32 path on the exact
upcast of the 16-bit pool; values are compared as bit patterns, so NaN outputs compare too."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16]
N = 41001                           # pool size: the row lists pick up to 40 001 of these rows
WIDTHS = (2048, 256, 12, 4)
COUNTS = (1, 7, 8, 9, 40001)


def _bits(t):
    return t.contiguous().view(torch.int64)


def _same(a, b, what):
    assert a.dtype == b.dtype == torch.float64 and a.shape == b.shape, what
    bad = (_bits(a) != _bits(b)).sum().item()
    assert bad == 0, f"{what}: {bad} entries differ"


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _colsum(v, X, rows=None):
    """S of X[rows] through vatlq_cosine_colsum_dt (ops.cosine_rowsum keeps S to itself)"""
    L = v._lib.lib()
    n, d = X.shape
    m = n if rows is None else rows.numel()
    ws_bytes = L.vatlq_cosine_workspace_bytes(d)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=X.device)
    S = torch.empty(d, dtype=torch.float64, device=X.device)
    v._lib.check(L.vatlq_cosine_colsum_dt(_ptr(X), v.ops.EMBEDDING_DTYPES[X.dtype], n, d, _ptr(rows), m, _ptr(S), _ptr(ws),
                                          ws_bytes, C.c_void_p(torch.cuda.current_stream().cuda_stream)),
                 "vatlq_cosine_colsum_dt")
    return S


def _check(v, X16, rows, what):
    """S and the row sums of X16[rows] against those of its upcast, bit for bit; returns the 16-bit row sums"""
    X32 = X16.float()
    _same(_colsum(v, X16, rows), _colsum(v, X32, rows), f"S {what}")
    got = v.ops.cosine_rowsum(X16, rows=rows)
    _same(got, v.ops.cosine_rowsum(X32, rows=rows), f"row sums {what}")
    return got


def _pool(v, kind, d, dtype, n=N, seed=61):
    """the clustered bench pool, an i.i.d. pool, or the clustered pool scaled to an rms element of 1.5e-5 (almost every
    element an fp16 subnormal)"""
    X = v.synth.pool_embeddings(n, d=d, seed=seed, kind="iid" if kind == "iid" else "clustered", device=DEV)
    if kind == "subnormal":
        X = X * (1.5e-5 / X.pow(2).mean().sqrt())
    return X.to(dtype)


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["clustered", "iid", "subnormal"])
def test_sums_equal_upcast(built_lib, kind, dtype):
    """Every width and row count, with a row list (sorted, from a larger pool) and without one (the first m rows)."""
    v = built_lib
    rng = np.random.default_rng(63)
    for d in WIDTHS:
        X = _pool(v, kind, d, dtype)
        if kind == "subnormal" and dtype == torch.float16 and d == 2048:
            assert (X.float().abs() < 6.1e-5).float().mean().item() > 0.99
        for m in COUNTS:
            _check(v, X[:m], None, f"{kind} d={d} m={m} {dtype}")
            rows = torch.from_numpy(np.sort(rng.choice(N, m, replace=False))).to(DEV)
            _check(v, X, rows, f"{kind} d={d} m={m} rows {dtype}")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("kind", ["clustered", "iid", "subnormal"])
def test_influence_and_diversity_equal_upcast(built_lib, kind, dtype):
    """query.influence over the unlabelled rows and the Diversity filter of query.select (the k of least cosine row
    sum among the top 8k by score), 10 % labelled."""
    v = built_lib
    from vatlq import query
    n, k = 40001, 400
    X = _pool(v, kind, 2048, dtype, n=n, seed=65)
    lab = np.random.default_rng(65).choice(n, n // 10, replace=False)
    unl = query.unlabelled_mask(n, lab, DEV)
    _same(query.influence(X, unl), query.influence(X.float(), unl), f"influence {kind} {dtype}")
    score = v.synth.pool_unc(n, device=DEV)
    score[torch.from_numpy(lab).to(DEV)] = 0
    got, k16, _ = query.select(score, unl, X, k, "Diversity")
    ref, k32, _ = query.select(score, unl, X.float(), k, "Diversity")
    assert k16 == k32 == k and got.numel() == k
    assert torch.equal(got, ref), f"Diversity picks {kind} {dtype}"


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("d", [2048, 12])
def test_zero_and_huge_rows(built_lib, d, dtype):
    """All-zero rows (cosine distance 1 to every other row: row sum m - 1) and, in bf16, a row with elements near 3e38
    whose squares overflow fp32 but not the fp64 accumulation."""
    v = built_lib
    m = 4001
    X = _pool(v, "clustered", d, dtype, n=m, seed=67)
    zero = [0, 17, 4000]
    X[zero] = 0
    big = 1234
    if dtype == torch.bfloat16:
        rng = np.random.default_rng(67)
        w = min(d, 64)
        X[big, :w] = torch.from_numpy(rng.choice([-1.0, 1.0], w) * rng.uniform(1e38, 3e38, w)).to(dtype).to(DEV)
        assert not torch.isfinite(X[big].float() ** 2).all()      # these squares do overflow fp32
    for rows in (None, torch.arange(0, m, 3, device=DEV)):
        got = _check(v, X, rows, f"zero / huge rows d={d} {rows is not None} {dtype}")
        assert torch.isfinite(got).all()
        ids = torch.arange(m, device=DEV) if rows is None else rows
        at_zero = torch.isin(ids, torch.tensor(zero, device=DEV))
        assert (got[at_zero] == ids.numel() - 1).all()


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("d", [2048, 256])
def test_nan_row(built_lib, d, dtype):
    """A NaN element propagates as in fp32: S and the row sums hold NaN at the same places, with the same bits."""
    v = built_lib
    m = 3001
    X = _pool(v, "iid", d, dtype, n=m, seed=69)
    X[5, 3] = float("nan")
    for rows in (None, torch.arange(1, m, 2, device=DEV), torch.arange(0, m, 2, device=DEV)):
        got = _check(v, X, rows, f"NaN d={d} {dtype}")
        assert torch.isnan(got).any() == (rows is None or bool((rows == 5).any()))


@pytest.mark.parametrize("dtype", DTYPES)
def test_alignment(built_lib, dtype):
    """A 16-bit X that is 8- but not 16-byte aligned runs (equal to the upcast); a 2-byte-aligned 16-bit view and an
    8-byte-aligned fp32 view are refused."""
    v = built_lib
    n, d = 2001, 256
    buf = torch.empty(n * d + 4, dtype=dtype, device=DEV)
    buf[4:] = _pool(v, "clustered", d, dtype, n=n, seed=71).reshape(-1)
    X = buf[4:].view(n, d)
    assert X.data_ptr() % 16 == 8
    _check(v, X, None, f"8-byte aligned {dtype}")
    _check(v, X, torch.arange(0, n, 5, device=DEV), f"8-byte aligned rows {dtype}")
    with pytest.raises(v._lib.VatlqError, match="aligned"):
        v.ops.cosine_rowsum(buf[1:1 + n * d].view(n, d))
    with pytest.raises(v._lib.VatlqError, match="aligned"):
        v.ops.cosine_rowsum(torch.zeros(n * d + 2, device=DEV)[2:].view(n, d))


def test_unknown_dtype_code(built_lib):
    """An unknown dtype code through the C ABI returns VATLQ_EINVAL and writes nothing."""
    v = built_lib
    L = v._lib.lib()
    n, d = 64, 256
    X = torch.ones((n, d), dtype=torch.bfloat16, device=DEV)
    ws_bytes = L.vatlq_cosine_workspace_bytes(d)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    S = torch.full((d,), 7.0, dtype=torch.float64, device=DEV)
    out = torch.full((n,), 7.0, dtype=torch.float64, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for code in (3, -1, 255):
        assert L.vatlq_cosine_colsum_dt(_ptr(X), code, n, d, None, n, _ptr(S), _ptr(ws), ws_bytes, st) == v._lib.EINVAL
        assert "dtype" in L.vatlq_last_error().decode()
        assert L.vatlq_cosine_rowsum_dt(_ptr(X), code, n, d, None, n, _ptr(S), float(n), _ptr(out), st) == v._lib.EINVAL
        assert "dtype" in L.vatlq_last_error().decode()
    torch.cuda.synchronize()
    assert (S == 7.0).all() and (out == 7.0).all()


# ---- two GPUs: bf16 embedding shards through distributed_query
STRATEGIES = (("THC+WPU", "Influence", "Coreset"), ("THC+WPU", "None", "Diversity"), ("TPC", "Influence", "Diversity"))


def _two_gpu_worker(rank, port, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch.distributed as td
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    td.init_process_group("nccl", rank=rank, world_size=2, device_id=torch.device("cuda", rank))
    try:
        from vatlq import dist, synth
        solo = None
        for r in range(2):                       # (every rank must take part in every new_group call)
            g = td.new_group([r])
            if r == rank:
                solo = g
        n, k = 3000, 40
        dev = torch.device("cuda", rank)
        ids, ip, inx = synth.track_flags(n, np.random.default_rng(4), 12.0)
        H = torch.from_numpy(synth.heatmaps(n, seed=4, track_ids=ids)).to(dev)
        boxes = torch.from_numpy(synth.boxes_xyxy(n, 4)).to(dev)
        ip, inx = torch.from_numpy(ip.astype(np.uint8)).to(dev), torch.from_numpy(inx.astype(np.uint8)).to(dev)
        X16 = synth.pool_embeddings(n, d=256, seed=5, device=dev).to(torch.bfloat16)
        W = synth.ae_weights(42, 4)
        lab = [7, 900, 1501, 2999]
        lo, hi = dist.shard_range(n, rank, 2)
        comm = dist.Comm()
        res = []
        for unc, rep, flt in STRATEGIES:
            kw = dict(uncertainty=unc, representativeness=rep, filter=flt)
            sh = slice(lo, hi)
            multi = dist.distributed_query(H[sh], boxes[sh], ip[sh], inx[sh], X16[sh], W, lab, n, k, 0.3, comm=comm, **kw)
            multi32 = dist.distributed_query(H[sh], boxes[sh], ip[sh], inx[sh], X16[sh].float(), W, lab, n, k, 0.3,
                                             comm=comm, **kw)
            one = dist.distributed_query(H, boxes, ip, inx, X16.float(), W, lab, n, k, 0.3, group=solo, **kw)
            res.append((multi.picks.cpu().tolist() == one.picks.cpu().tolist(),
                        torch.equal(multi.picks, multi32.picks) and torch.equal(_bits(multi.unc), _bits(multi32.unc)),
                        bool(torch.allclose(multi.unc, one.unc, rtol=1e-9, atol=1e-12))))
        comm.close()
        q.put((rank, res))
    finally:
        td.destroy_process_group()


def test_two_gpus_bf16_shards_influence_diversity_match_one_gpu_fp32(built_lib):
    """bf16 embedding shards on two GPUs with Influence and with the Diversity filter: the picks equal those of one
    GPU holding the whole fp32 upcast (the same entry point on a one-rank group), and the scores and picks equal,
    bit for bit, those of the same two-GPU run on fp32 shards."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_two_gpu_worker, args=(r, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    for p in ps:
        p.join(timeout=600)
    for p in ps:
        if p.is_alive():
            p.kill()
    res = sorted(q.get(timeout=5) for _ in ps)
    want = [(True, True, True)] * len(STRATEGIES)
    assert res == [(0, want), (1, want)], res
