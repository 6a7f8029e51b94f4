"""CPU: the host side of the K-Means filters on fp16 / bf16 embeddings.  kmeans.py must send a 16-bit X to the
vatlq_kmeans_*_dt entries with its dtype code and an fp32 X to the fp32 entries exactly as before; the results on a
16-bit X must be those of its fp32 upcast.  The device calls are the NumPy stand-ins of test_kmeans_host_cpu.py, which
decode a 16-bit X here the way the kernels widen it (fp16 through np.float16, bf16 as the top half of an fp32).  The
argument checks of the _dt entries are exercised on the real library (they refuse before any device work); the kernels
themselves are checked on the GPU (test_gpu_kmeans_half.py)."""
import contextlib
import ctypes as C
import os
import re
import socket
import sys
import warnings

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path[:0] = [ROOT, HERE]
from test_kmeans_host_cpu import FakeLib, _a     # noqa: E402

F32, F16, BF16 = 0, 1, 2
X_ENTRIES = ("vatlq_kmeans_mean_var", "vatlq_kmeans_pp", "vatlq_kmeans_gather", "vatlq_kmeans_assign",
             "vatlq_kmeans_update", "vatlq_kmeans_relocate", "vatlq_kmeans_rowdist")


def _decode(ptr, count, code):
    """count 16-bit values at ptr, widened exactly to fp32"""
    raw = _a(ptr, count, C.c_uint16).copy()
    if code == F16:
        return raw.view(np.float16).astype(np.float32)
    assert code == BF16, code
    return (raw.astype(np.uint32) << 16).view(np.float32)


class HalfFakeLib(FakeLib):
    """FakeLib plus the seven *_dt entries; records which entry each X-reading call went to, with its dtype code."""

    def __init__(self):
        self.calls, self._keep = [], []

    def _dt(self, name, X, code, count, args):
        self.calls.append((name + "_dt", code))
        x = _decode(X, count, code)
        self._keep.append(x)                          # the fp32 stand-in reads it through a raw pointer
        return getattr(FakeLib, name)(self, C.c_void_p(x.ctypes.data), *args)

    def vatlq_kmeans_mean_var_dt(self, X, code, n, d, *rest):
        return self._dt("vatlq_kmeans_mean_var", X, code, n * d, (n, d, *rest))

    def vatlq_kmeans_pp_dt(self, X, code, n, d, *rest):
        return self._dt("vatlq_kmeans_pp", X, code, n * d, (n, d, *rest))

    def vatlq_kmeans_gather_dt(self, X, code, d, *rest):
        return self._dt("vatlq_kmeans_gather", X, code, self.n * d, (d, *rest))

    def vatlq_kmeans_assign_dt(self, X, code, n, d, *rest):
        return self._dt("vatlq_kmeans_assign", X, code, n * d, (n, d, *rest))

    def vatlq_kmeans_update_dt(self, X, code, n, d, *rest):
        return self._dt("vatlq_kmeans_update", X, code, n * d, (n, d, *rest))

    def vatlq_kmeans_relocate_dt(self, X, code, d, *rest):
        return self._dt("vatlq_kmeans_relocate", X, code, self.n * d, (d, *rest))

    def vatlq_kmeans_rowdist_dt(self, X, code, n, d, *rest):
        return self._dt("vatlq_kmeans_rowdist", X, code, n * d, (n, d, *rest))


def _recording(name):
    def call(self, X, *args):
        self.calls.append((name, None))
        return getattr(FakeLib, name)(self, X, *args)
    return call


for _name in X_ENTRIES:
    setattr(HalfFakeLib, _name, _recording(_name))


def _patch(KM, _lib, fake):
    """what the fixtures of test_kmeans_host_cpu.py patch, with HalfFakeLib as the library"""
    _lib.lib = lambda: fake
    KM._cuda = lambda t, dt, name: t.contiguous()
    KM._stream = lambda: None
    torch.cuda.device = lambda dev: contextlib.nullcontext()


@pytest.fixture
def km_half(monkeypatch):
    import vatlq  # noqa: F401
    from vatlq import _lib, kmeans as KM
    fake = HalfFakeLib()
    monkeypatch.setattr(_lib, "lib", lambda: fake)
    monkeypatch.setattr(KM, "_cuda", lambda t, dt, name: t.contiguous())
    monkeypatch.setattr(KM, "_stream", lambda: None)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())

    def run(X, k, w=None, **kw):
        fake.n, fake.k = X.shape[0], k
        fake.calls.clear()
        res = KM.kmeans_fit_select(X, k, sample_weight=None if w is None else torch.from_numpy(w), **kw)
        return res, list(fake.calls)
    return run


def _same(a, b):
    assert a.query_rows == b.query_rows
    assert torch.equal(a.labels, b.labels) and torch.equal(a.center_ids, b.center_ids)
    assert torch.equal(a.centers.view(torch.int64), b.centers.view(torch.int64))
    assert a.n_iter == b.n_iter and a.relocations == b.relocations


def _pools():
    rng = np.random.default_rng(11)
    X = np.abs(rng.normal(0, 1, (300, 24))).astype(np.float32)
    yield X, 40, 1 + rng.random(300), {}
    X = np.abs(rng.normal(0, 1, (100, 16))).astype(np.float32)      # empty clusters: relocation, select=False
    w = np.zeros(100)
    w[rng.choice(100, 30, replace=False)] = 1 + rng.random(30)
    yield X, 40, w, {"select": False}
    yield np.abs(rng.normal(0, 1, (257, 12))).astype(np.float32), 9, None, {}


@pytest.mark.parametrize("dtype,code", [(torch.float16, F16), (torch.bfloat16, BF16)])
def test_16bit_x_goes_to_the_dt_entries_and_gives_the_upcast_result(km_half, dtype, code):
    saw_relocation = False
    for X, k, w, kw in _pools():
        X16 = torch.from_numpy(X).to(dtype)
        got, calls16 = km_half(X16, k, w, **kw)
        ref, calls32 = km_half(X16.float(), k, w, **kw)
        _same(got, ref)
        saw_relocation |= got.relocations > 0
        assert calls16 and all(c == code for _, c in calls16)
        assert {n for n, _ in calls16} <= {e + "_dt" for e in X_ENTRIES}
        assert [n for n, _ in calls16] == [n + "_dt" for n, _ in calls32]     # the same calls, in the same order
        assert all(c is None for _, c in calls32) and {n for n, _ in calls32} <= set(X_ENTRIES)
    assert saw_relocation                               # _relocate_dt and _rowdist_dt were exercised


def test_fp32_x_keeps_the_fp32_entries(km_half):
    X, k, w, kw = next(_pools())
    res, calls = km_half(torch.from_numpy(X), k, w, **kw)
    assert calls and all(c is None and n in X_ENTRIES for n, c in calls)
    assert [n for n, _ in calls[:3]] == ["vatlq_kmeans_mean_var", "vatlq_kmeans_pp", "vatlq_kmeans_gather"]


def test_kmeans_checks_x_through_the_module_cuda_with_its_own_dtype(monkeypatch):
    """kmeans_fit_select / unique_rows_first_index validate X through kmeans._cuda with X's dtype when it is one of
    EMBEDDING_DTYPES and with fp32 otherwise (so an fp64 X is refused with the message it always got)."""
    import vatlq  # noqa: F401
    from vatlq import _lib, kmeans as KM
    seen = []

    def cuda(t, dt, name):
        seen.append((dt, name))
        raise _lib.VatlqError("stop")
    monkeypatch.setattr(KM, "_cuda", cuda)
    for dt in (torch.float32, torch.float16, torch.bfloat16, torch.float64):
        for fn in (lambda t: KM.kmeans_fit_select(t, 2), KM.unique_rows_first_index):
            seen.clear()
            with pytest.raises(_lib.VatlqError):
                fn(torch.zeros((4, 8), dtype=dt))
            assert seen[0][0] == (dt if dt != torch.float64 else torch.float32)


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_unique_rows_first_index_on_16bit(monkeypatch, dtype):
    """np.unique(E.float(), axis=0, return_index=True)[1] for a 16-bit E: rows that differ in fp32 but round to the same
    16-bit row are duplicates, rows that share only their first columns are not."""
    import vatlq  # noqa: F401
    from vatlq import kmeans as KM
    monkeypatch.setattr(KM, "_cuda", lambda t, dt, name: t.contiguous())

    def rank_scores(score, mask=None, descending=True, count=None):
        s = np.where(score.numpy() == 0, 0.0, score.numpy())
        order = np.argsort(-s if descending else s, kind="stable")
        return torch.from_numpy(order if count is None else order[:count])
    monkeypatch.setattr(KM, "rank_scores", rank_scores)
    rng = np.random.default_rng(3)
    E = np.abs(rng.normal(0, 1, (200, 12))).astype(np.float32)
    E[50:80] = E[10:40] * np.float32(1 + 1e-5)        # distinct in fp32, equal after rounding to 16 bits
    E[100:110, 0] = E[5, 0]
    E[120:125, :3] = E[6, :3]
    E[130, 0], E[131, 0] = 0.0, -0.0
    E[131, 1:] = E[130, 1:]
    E16 = torch.from_numpy(E).to(dtype)
    got = KM.unique_rows_first_index(E16)
    _, ref = np.unique(E16.float().numpy(), axis=0, return_index=True)
    assert np.array_equal(got, ref)
    assert len(got) < len(np.unique(E, axis=0))         # the rounding made duplicates
    assert KM.unique_rows_first_index(torch.zeros((0, 4), dtype=dtype)).size == 0


def test_dt_signatures_follow_the_header():
    """The seven *_dt entries are in _lib's table, with the argument types of their declarations in include/vatlq.h,
    i.e. the fp32 entry's with (const void* X, int dtype) in X's place."""
    import vatlq  # noqa: F401
    from vatlq import _lib
    ct = {"int": C.c_int, "int64_t": C.c_int64, "size_t": C.c_size_t, "double": C.c_double, "vatlq_stream_t": C.c_void_p}
    hdr = open(os.path.join(ROOT, "include", "vatlq.h")).read()
    for base in X_ENTRIES:
        name = base + "_dt"
        m = re.search(r"int\s+" + name + r"\(([^)]*)\);", hdr)
        assert m, name
        params = [re.sub(r"\s+", " ", p).strip() for p in m.group(1).split(",")]
        want = [C.c_void_p if "*" in p else ct[p.replace("const ", "").rsplit(" ", 1)[0]] for p in params]
        res, args = _lib.SIGNATURES[name]
        assert res is C.c_int and args == want, name
        assert args[:2] == [C.c_void_p, C.c_int] and args[2:] == _lib.SIGNATURES[base][1][1:], name


ALIGNED, BUF = 0x10000, 0x20000        # fake device addresses: the checks must refuse before touching them
BIG = 1 << 40


def _dt_calls(L):
    """entry -> call(X pointer, dtype) with otherwise valid arguments (n = 64, d = 16, k = 4)"""
    p, n, d, k = C.c_void_p(BUF), 64, 16, 4
    return {
        "vatlq_kmeans_mean_var_dt": lambda x, dt: L.vatlq_kmeans_mean_var_dt(C.c_void_p(x), dt, n, d, p, p, p, BIG, None),
        "vatlq_kmeans_pp_dt": lambda x, dt: L.vatlq_kmeans_pp_dt(C.c_void_p(x), dt, n, d, None, k, 0, p, 3, p, p, p, BIG, None),
        "vatlq_kmeans_gather_dt": lambda x, dt: L.vatlq_kmeans_gather_dt(C.c_void_p(x), dt, d, p, k, p, p, p, None),
        "vatlq_kmeans_assign_dt": lambda x, dt: L.vatlq_kmeans_assign_dt(C.c_void_p(x), dt, n, d, p, k, p, None, None, p, BIG, None),
        "vatlq_kmeans_update_dt": lambda x, dt: L.vatlq_kmeans_update_dt(C.c_void_p(x), dt, n, d, None, p, p, k, p, p, p, p, p, p,
                                                                         BIG, None),
        "vatlq_kmeans_relocate_dt": lambda x, dt: L.vatlq_kmeans_relocate_dt(C.c_void_p(x), dt, d, None, p, p, p, p, 1, p, p, None),
        "vatlq_kmeans_rowdist_dt": lambda x, dt: L.vatlq_kmeans_rowdist_dt(C.c_void_p(x), dt, n, d, p, p, p, None),
    }


@pytest.mark.parametrize("name", [e + "_dt" for e in X_ENTRIES])
def test_dt_entries_refuse_bad_dtype_and_misaligned_16bit_x(built_lib, name):
    _lib = built_lib._lib
    L = _lib.lib()
    call = _dt_calls(L)[name]
    for dt in (3, -1, 255):
        assert call(ALIGNED, dt) == _lib.EINVAL
        msg = L.vatlq_last_error().decode()
        assert msg.startswith(name + ":") and "dtype" in msg, msg
    for x, dt in [(ALIGNED + 2, F16), (ALIGNED + 4, BF16), (ALIGNED + 6, F16)]:
        assert call(x, dt) == _lib.EINVAL, (x, dt)
        msg = L.vatlq_last_error().decode()
        assert msg.startswith(name + ":") and "8-byte aligned" in msg, msg


def test_fp32_entries_keep_their_alignment_rules(built_lib):
    """_pp and _assign refuse an fp32 X that is 8- but not 16-byte aligned, as they always did, now through their _dt
    form; a 16-bit X at the same address passes the alignment check (the null workspace is what refuses it)."""
    _lib = built_lib._lib
    L = _lib.lib()
    p, n, d, k = C.c_void_p(BUF), 64, 16, 4
    x = C.c_void_p(ALIGNED + 8)
    assert L.vatlq_kmeans_pp(x, n, d, None, k, 0, p, 3, p, p, p, BIG, None) == _lib.EINVAL
    assert L.vatlq_last_error().decode() == "vatlq_kmeans_pp_dt: X must be 16-byte aligned"
    assert L.vatlq_kmeans_assign(x, n, d, p, k, p, None, None, p, BIG, None) == _lib.EINVAL
    assert L.vatlq_last_error().decode() == "vatlq_kmeans_assign_dt: X and C must be 16-byte aligned"
    for dt in (F16, BF16):
        assert L.vatlq_kmeans_pp_dt(x, dt, n, d, None, k, 0, p, 3, p, p, None, BIG, None) == _lib.EINVAL
        assert "aligned" not in L.vatlq_last_error().decode()
        assert L.vatlq_kmeans_assign_dt(x, dt, n, d, p, k, p, None, None, None, BIG, None) == _lib.EINVAL
        assert "aligned" not in L.vatlq_last_error().decode()


# ---- world 2, gloo: the row-sharded assignment on a bf16 X
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _sharded_worker(rank, world, port, q):
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(here), here]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    td.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import vatlq  # noqa: F401
        from vatlq import _lib, kmeans as KM
        from test_kmeans_half_cpu import HalfFakeLib, _patch
        from sklearn.cluster import KMeans
        fake = HalfFakeLib()
        _patch(KM, _lib, fake)
        rng = np.random.default_rng(4)                       # identical pool on every rank
        n, d, k = 301, 20, 23                                # ragged shards
        X16 = torch.from_numpy(np.abs(rng.normal(0, 1, (n, d))).astype(np.float32)).to(torch.bfloat16)
        w = 1 + rng.random(n)
        fake.n, fake.k = n, k
        res = KM.kmeans_fit_select(X16, k, sample_weight=torch.from_numpy(w), group=td.group.WORLD)
        ok = all(c == BF16 for _, c in fake.calls) and ("vatlq_kmeans_assign_dt", BF16) in fake.calls
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            km = KMeans(n_clusters=k, random_state=318)
            lab = km.fit_predict(X16.float().numpy().astype(np.float64), sample_weight=w)
        ok &= bool(np.array_equal(res.labels.numpy(), lab)) and res.n_iter == km.n_iter_
        rows = torch.tensor(res.query_rows)
        both = [torch.empty_like(rows) for _ in range(world)]
        td.all_gather(both, rows)
        ok &= all(torch.equal(b, rows) for b in both)        # every rank returns the same picks
        q.put((rank, bool(ok)))
    finally:
        td.destroy_process_group()


def test_row_sharded_assignment_on_bf16_world2():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_sharded_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = [q.get(timeout=180) for _ in ps]
    for p in ps:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)], res
