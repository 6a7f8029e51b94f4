"""GPU: the K-Means and weighted K-Means filters on fp16 / bf16 embeddings.  Contract (include/vatlq.h,
vatlq_kmeans_*_dt): for a 16-bit X every result equals, bit for bit, that of the same call on X.float() — labels,
center_ids, centres, n_iter, relocations, closest / dis, query rows, np.unique indices — and therefore sklearn's on
X.astype(np.float64).  The reference is always the fp32 path on the exact upcast of the 16-bit pool."""
import ctypes as C
import os
import socket
import sys
import warnings

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from kmeans_cases import CASES, case_inputs     # noqa: E402

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16]


def _bits(t):
    return t.contiguous().view(torch.int64) if t.dtype == torch.float64 else t.contiguous().view(torch.int32)


def _eq(a, b, what):
    assert a.dtype == b.dtype and a.shape == b.shape, what
    bad = (_bits(a) != _bits(b)).sum().item()
    assert bad == 0, f"{what}: {bad} entries differ"


def _same_result(a, b, what):
    assert a.query_rows == b.query_rows, what
    _eq(a.labels, b.labels, f"labels {what}")
    _eq(a.center_ids, b.center_ids, f"center_ids {what}")
    assert torch.equal(a.centers, b.centers), f"centres {what}"
    assert a.n_iter == b.n_iter and a.relocations == b.relocations, what


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


# ---- the reference golden cases with X rounded to 16 bits
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("tag", CASES)
def test_golden_cases_in_16_bits_equal_the_upcast(built_lib, tag, dtype):
    from vatlq import kmeans as KM
    z = np.load(os.path.join(ROOT, "tests", "golden", "kmeans.npz"))
    X, cand, score, k, w_unc, cw = case_inputs(z, tag)
    cand_t = torch.as_tensor(cand, device=DEV)
    emb16 = torch.from_numpy(X).to(DEV).to(dtype)[cand_t]
    emb32 = emb16.float()
    _same_result(KM.kmeans_fit_select(emb16, k), KM.kmeans_fit_select(emb32, k), f"K-Means {tag} {dtype}")
    eidx = KM.unique_rows_first_index(emb16)
    assert np.array_equal(eidx, KM.unique_rows_first_index(emb32))
    e_t = torch.as_tensor(eidx, device=DEV)
    weight = (1 + w_unc * cw * torch.from_numpy(score).to(DEV))[e_t].contiguous()
    kk = min(k, len(eidx))
    _same_result(KM.kmeans_fit_select(emb16[e_t], kk, sample_weight=weight),
                 KM.kmeans_fit_select(emb32[e_t], kk, sample_weight=weight), f"weighted {tag} {dtype}")


# ---- the shapes of test_kmeans_matches_sklearn (d = 36 and 100 are not multiples of 8)
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n,d,k,weighted", [(3000, 2048, 150, False), (2500, 2048, 120, True), (700, 96, 333, False),
                                            (1000, 36, 10, True), (130, 2048, 100, False), (5000, 256, 64, False)])
def test_matches_the_upcast_and_sklearn(built_lib, n, d, k, weighted, dtype):
    from sklearn.cluster import KMeans
    from oracle import vatl_oracle as O
    from vatlq import kmeans as KM
    rng = np.random.default_rng(n + k)
    cen = np.abs(rng.normal(0, 1, (max(n // 25, 1), d)))
    X = (cen[(np.arange(n) // 25) % len(cen)] + rng.normal(0, 0.2, (n, d))).astype(np.float32)
    w = (1 + rng.random(n)) if weighted else None
    X16 = torch.from_numpy(X).to(DEV).to(dtype)
    wd = None if w is None else torch.from_numpy(w).to(DEV)
    res = KM.kmeans_fit_select(X16, k, sample_weight=wd)
    _same_result(res, KM.kmeans_fit_select(X16.float(), k, sample_weight=wd), f"{n}x{d} k={k} {dtype}")
    X64 = X16.float().cpu().numpy().astype(np.float64)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        km = KMeans(n_clusters=k, random_state=318)
        lab = km.fit_predict(X64, sample_weight=w)
        rows = O._closest_member_per_cluster(X64, km, lab)
    assert np.array_equal(res.labels.cpu().numpy(), lab)
    assert res.query_rows == rows
    assert res.n_iter == km.n_iter_


# ---- the relocation pools of test_kmeans_empty_cluster_relocation
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n,nw,k", [(100, 30, 40), (200, 50, 60), (120, 100, 110)])
def test_empty_cluster_relocation(built_lib, n, nw, k, dtype):
    from vatlq import kmeans as KM
    rng = np.random.default_rng(5 + n)
    X16 = torch.from_numpy(np.abs(rng.normal(0, 1, (n, 16))).astype(np.float32)).to(DEV).to(dtype)
    w = np.zeros(n)
    w[rng.choice(n, nw, replace=False)] = 1 + rng.random(nw)
    wd = torch.from_numpy(w).to(DEV)
    res = KM.kmeans_fit_select(X16, k, sample_weight=wd, select=False)
    assert res.relocations > 0
    _same_result(res, KM.kmeans_fit_select(X16.float(), k, sample_weight=wd, select=False), f"relocation {n} {dtype}")


# ---- each entry alone against its fp32 call on the upcast (ragged n, d % 32 != 0)
@pytest.mark.parametrize("dtype", DTYPES)
def test_each_entry_against_the_fp32_call_on_the_upcast(built_lib, dtype):
    v = built_lib
    L = v._lib.lib()
    code = v.ops.EMBEDDING_DTYPES[dtype]
    chk = v._lib.check
    rng = np.random.default_rng(5)
    n, d, k = 1237, 100, 77
    X16 = torch.from_numpy(rng.normal(0, 1, (n, d)).astype(np.float32)).to(DEV).to(dtype)
    X32 = X16.float()
    ws = torch.empty(int(L.vatlq_kmeans_workspace_bytes(n, d, k)), dtype=torch.uint8, device=DEV)
    wsb = ws.numel()
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    f64 = lambda *s: torch.full(s, 7.0, dtype=torch.float64, device=DEV)
    i32 = lambda *s: torch.full(s, -7, dtype=torch.int32, device=DEV)

    def both(fn, *bufs):
        """(16-bit outputs, fp32 outputs) of fn(X, code_or_None, buffers)"""
        a, b = [t.clone() for t in bufs], [t.clone() for t in bufs]
        fn(X16, code, a)
        fn(X32, None, b)
        return a, b

    def call(name, X, code, *args):
        if code is None:
            chk(getattr(L, name)(_ptr(X), *args), name)
        else:
            chk(getattr(L, name + "_dt")(_ptr(X), code, *args), name + "_dt")

    (m16, mv16), (m32, mv32) = both(lambda X, c, o: call("vatlq_kmeans_mean_var", X, c, n, d, _ptr(o[0]), _ptr(o[1]), _ptr(ws), wsb, st),
                                    f64(d), f64(1))
    _eq(m16, m32, "mean")
    _eq(mv16, mv32, "var")
    X64 = X32.cpu().numpy().astype(np.float64)
    assert np.array_equal(m16.cpu().numpy(), X64.mean(axis=0))
    mean = m32
    # k-means++ on the same random stream as kmeans.py draws
    rs = np.random.RandomState(318)
    first = int(rs.choice(n))
    trials = 2 + int(np.log(k))
    rand = torch.from_numpy(rs.uniform(size=(k - 1) * trials)).to(DEV)
    (ids16, cl16), (ids32, cl32) = both(lambda X, c, o: call("vatlq_kmeans_pp", X, c, n, d, None, k, first, _ptr(rand), trials,
                                                             _ptr(o[0]), _ptr(o[1]), _ptr(ws), wsb, st), i32(k), f64(n))
    _eq(ids16, ids32, "center_ids")
    _eq(cl16, cl32, "closest")
    (cc16, cr16), (cc32, cr32) = both(lambda X, c, o: call("vatlq_kmeans_gather", X, c, d, _ptr(ids32), k, _ptr(mean), _ptr(o[0]),
                                                           _ptr(o[1]), st), f64(k, d), f64(k, d))
    _eq(cc16, cc32, "gather Cc")
    _eq(cr16, cr32, "gather Cr")
    Cd = torch.from_numpy(rng.normal(0, 1, (k, d))).to(DEV)
    old = torch.zeros(n, dtype=torch.int32, device=DEV)
    (lab16, ch16), (lab32, ch32) = both(lambda X, c, o: call("vatlq_kmeans_assign", X, c, n, d, _ptr(Cd), k, _ptr(o[0]), _ptr(old),
                                                             _ptr(o[1]), _ptr(ws), wsb, st), i32(n), i32(1))
    _eq(lab16, lab32, "labels")
    _eq(ch16, ch32, "changed")
    labels = lab32
    wv = torch.from_numpy(1 + rng.random(n)).to(DEV)
    a, b = both(lambda X, c, o: call("vatlq_kmeans_update", X, c, n, d, _ptr(wv), _ptr(mean), _ptr(labels), k, _ptr(o[0]), _ptr(o[1]),
                                     _ptr(o[2]), _ptr(o[3]), _ptr(o[4]), _ptr(ws), wsb, st), f64(k, d), f64(k), i32(n), i32(k + 1), i32(1))
    for x, y, what in zip(a, b, ("sums", "wsum", "order", "starts", "n_empty")):
        _eq(x, y, f"update {what}")
    sums, wsum = b[0], b[1]
    emp = torch.tensor([3, 11], dtype=torch.int32, device=DEV)
    far = torch.tensor([5, 1000], dtype=torch.int32, device=DEV)
    a, b = both(lambda X, c, o: call("vatlq_kmeans_relocate", X, c, d, _ptr(wv), _ptr(mean), _ptr(labels), _ptr(emp), _ptr(far), 2,
                                     _ptr(o[0]), _ptr(o[1]), st), sums, wsum)
    _eq(a[0], b[0], "relocate sums")
    _eq(a[1], b[1], "relocate wsum")
    (dis16,), (dis32,) = both(lambda X, c, o: call("vatlq_kmeans_rowdist", X, c, n, d, _ptr(Cd), _ptr(labels), _ptr(o[0]), st), f64(n))
    _eq(dis16, dis32, "dis")
    assert np.array_equal(dis16.cpu().numpy(), ((X64 - Cd.cpu().numpy()[labels.cpu().numpy()]) ** 2).sum(axis=1))


# ---- rounding to bf16 makes duplicates
def test_bf16_rounding_duplicates_in_the_weighted_filter(built_lib):
    """Rows that differ in fp32 but round to the same bf16 row are duplicates for np.unique: the weighted filter's
    de-duplication count and picks equal those on the upcast (and differ from the fp32 pool's count)."""
    v = built_lib
    from vatlq import kmeans as KM
    from vatlq.query import select, unlabelled_mask
    n, k = 600, 30
    X = torch.from_numpy(v.synth.pool_embeddings(n, d=256, kind="weak", seed=21)).to(torch.bfloat16).float().numpy()
    X[300:400] = X[100:200] * np.float32(1 + 2 ** -12)      # bf16 values moved by < half an ulp: they round back
    X32 = torch.from_numpy(X).to(DEV)
    X16 = X32.to(torch.bfloat16)
    assert (X32[300:400] != X32[100:200]).any(1).all() and torch.equal(X16[300:400], X16[100:200])
    unl = unlabelled_mask(n, list(range(0, n, 7)), DEV)
    cand = torch.nonzero(unl).flatten()
    n16 = len(KM.unique_rows_first_index(X16[cand]))
    assert n16 == len(KM.unique_rows_first_index(X16.float()[cand])) < len(KM.unique_rows_first_index(X32[cand]))
    score = torch.from_numpy(v.synth.pool_unc(n, seed=21)).to(DEV) * unl
    got = select(score, unl, X16, k, "weighted", w_unc=0.8, combine_weight=0.4)
    ref = select(score, unl, X16.float(), k, "weighted", w_unc=0.8, combine_weight=0.4)
    assert torch.equal(got[0], ref[0]) and got[1] == ref[1] and got[2] == ref[2]


def test_bf16_rows_of_huge_norm(built_lib):
    """bf16 rows near 1e30 (their squares overflow fp32, not fp64): every result equals the upcast's."""
    v = built_lib
    from vatlq import kmeans as KM
    n, d, k = 2000, 256, 40
    X = torch.from_numpy(v.synth.pool_embeddings(n, d=d, kind="clustered", seed=23)).to(DEV)
    X[::97] *= 1e30
    X16 = X.to(torch.bfloat16)
    assert torch.isfinite(X16).all() and X16.float().abs().max() > 1e29
    res = KM.kmeans_fit_select(X16, k, select=False)
    _same_result(res, KM.kmeans_fit_select(X16.float(), k, select=False), "huge rows")


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("flt", ["K-Means", "weighted"])
def test_query_select_on_16bit(built_lib, flt, dtype):
    v = built_lib
    from vatlq.query import select, unlabelled_mask
    n, k = 1500, 40
    X16 = torch.from_numpy(v.synth.pool_embeddings(n, d=2048, kind="clustered", seed=31)).to(DEV).to(dtype)
    unl = unlabelled_mask(n, list(range(0, n, 11)), DEV)
    score = torch.from_numpy(v.synth.pool_unc(n, seed=31)).to(DEV) * unl
    got = select(score, unl, X16, k, flt, w_unc=0.8, combine_weight=0.4)
    ref = select(score, unl, X16.float(), k, flt, w_unc=0.8, combine_weight=0.4)
    assert torch.equal(got[0], ref[0]) and got[1] == ref[1] and got[2] == ref[2]


# ---- the C ABI's refusals
@pytest.mark.parametrize("dtype", DTYPES)
def test_alignment_and_dtype_errors(built_lib, dtype):
    """A 16-bit X 8- but not 16-byte aligned runs (equal to the upcast); at a 2-byte offset every _dt entry refuses it,
    as it refuses an unknown dtype code, before writing anything; the fp32 _pp and _assign still refuse an 8-byte
    aligned fp32 X."""
    v = built_lib
    L = v._lib.lib()
    from vatlq import kmeans as KM
    n, d, k = 501, 36, 12
    rng = np.random.default_rng(8)
    buf = torch.empty(n * d + 4, dtype=dtype, device=DEV)
    buf[4:] = torch.from_numpy(np.abs(rng.normal(0, 1, n * d)).astype(np.float32)).to(DEV).to(dtype)
    X = buf[4:].view(n, d)
    assert X.data_ptr() % 16 == 8
    _same_result(KM.kmeans_fit_select(X, k), KM.kmeans_fit_select(X.float(), k), f"8-byte aligned {dtype}")
    with pytest.raises(v._lib.VatlqError, match="8-byte aligned"):
        KM.kmeans_fit_select(buf[1:1 + n * d].view(n, d), k)
    code = v.ops.EMBEDDING_DTYPES[dtype]
    ws = torch.empty(int(L.vatlq_kmeans_workspace_bytes(n, d, k)), dtype=torch.uint8, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    out = torch.full((n,), 7.0, dtype=torch.float64, device=DEV)
    lab = torch.zeros(n, dtype=torch.int32, device=DEV)
    Cd = torch.zeros((k, d), dtype=torch.float64, device=DEV)
    bad = buf[1:1 + n * d].view(n, d)
    for x, c, msg in [(X, 3, "dtype"), (X, -1, "dtype"), (bad, code, "8-byte aligned")]:
        assert L.vatlq_kmeans_rowdist_dt(_ptr(x), c, n, d, _ptr(Cd), _ptr(lab), _ptr(out), st) == v._lib.EINVAL
        assert msg in L.vatlq_last_error().decode()
        assert L.vatlq_kmeans_mean_var_dt(_ptr(x), c, n, d, _ptr(out), _ptr(out), _ptr(ws), ws.numel(), st) == v._lib.EINVAL
        assert msg in L.vatlq_last_error().decode()
        assert L.vatlq_kmeans_assign_dt(_ptr(x), c, n, d, _ptr(Cd), k, _ptr(lab), None, None, _ptr(ws), ws.numel(), st) == v._lib.EINVAL
        assert msg in L.vatlq_last_error().decode()
    torch.cuda.synchronize()
    assert (out == 7.0).all() and (lab == 0).all()
    x32 = torch.zeros(n * d + 2, device=DEV)[2:].view(n, d)
    assert x32.data_ptr() % 16 == 8
    assert L.vatlq_kmeans_assign(_ptr(x32), n, d, _ptr(Cd), k, _ptr(lab), None, None, _ptr(ws), ws.numel(), st) == v._lib.EINVAL
    assert "16-byte aligned" in L.vatlq_last_error().decode()
    with pytest.raises(v._lib.VatlqError, match="16-byte aligned"):
        KM.kmeans_fit_select(x32, k)


# ---- two GPUs: bf16 embedding shards through distributed_query with the K-Means filters
FILTERS = ("K-Means", "weighted")


def _two_gpu_worker(rank, port, q):
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
        res = []
        for flt in FILTERS:
            kw = dict(uncertainty="THC+WPU", filter=flt, w_unc=0.8)
            sh = slice(lo, hi)
            multi = dist.distributed_query(H[sh], boxes[sh], ip[sh], inx[sh], X16[sh], W, lab, n, k, 0.3, **kw)
            one = dist.distributed_query(H, boxes, ip, inx, X16.float(), W, lab, n, k, 0.3, group=solo, **kw)
            res.append(multi.picks.cpu().tolist() == one.picks.cpu().tolist() and multi.stats == one.stats)
        q.put((rank, res))
    finally:
        td.destroy_process_group()


def test_two_gpus_bf16_shards_kmeans_filters_match_one_gpu_fp32(built_lib):
    """bf16 embedding shards on two GPUs with the K-Means and weighted filters (the assignment sharded by rows): the
    picks equal those of one GPU holding the whole fp32 upcast."""
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
    assert res == [(0, [True] * len(FILTERS)), (1, [True] * len(FILTERS))], res
