"""CPU: the host side of the core-set on fp16 / bf16 embeddings — argument checks of the *_dt entry points (no device
needed), the workspace size, the ops layer's dtype rules, the controller's choice of when to keep 16-bit embeddings,
the dtype agreement of distributed_query on two gloo processes, and the screen's error bound for 16-bit X (coreset.cu,
"the screen") on exact products of adversarial vectors at K = 2048.  The kernels are checked on the GPU
(test_gpu_coreset_half.py)."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

K = 2048
ALIGNED, BUF = 0x10000, 0x20000        # fake device addresses: the checks must reject before touching them
BIG = 1 << 40


def _calls(L):
    """name -> call(X pointer, dtype, d) of the three *_dt entry points (min_d / out left null where the X checks come
    first, so an X that passes them is refused by the next check, still before any device work)"""
    return {
        "vatlq_coreset_init_dt": lambda x, dt, d: L.vatlq_coreset_init_dt(
            C.c_void_p(x), dt, 64, d, 0, 64, None, 0, None, C.c_void_p(BUF), BIG, None),
        "vatlq_coreset_select_dt": lambda x, dt, d: L.vatlq_coreset_select_dt(
            C.c_void_p(x), dt, 64, d, 0, 64, None, None, 0, 0.0, 0.01, 0, -1, 4, 16, None, None, C.c_void_p(BUF), BIG,
            None, None),
        "vatlq_pairwise_dist_dt": lambda x, dt, d: L.vatlq_pairwise_dist_dt(
            C.c_void_p(x), dt, 64, d, None, 1, None, C.c_void_p(BUF), BIG, None),
    }


@pytest.mark.parametrize("name", ["vatlq_coreset_init_dt", "vatlq_coreset_select_dt", "vatlq_pairwise_dist_dt"])
def test_dt_entries_reject_bad_dtype_and_alignment(built_lib, name):
    _lib = built_lib._lib
    L = _lib.lib()
    call = _calls(L)[name]
    for x, dt in [(ALIGNED, 3), (ALIGNED, -1), (ALIGNED + 4, _lib.F16), (ALIGNED + 2, _lib.BF16), (ALIGNED + 8, _lib.F32)]:
        assert call(x, dt, 1000) == _lib.EINVAL, (x, dt)
        msg = L.vatlq_last_error().decode()
        assert "dtype" in msg or "aligned" in msg, msg
    for dt in (_lib.F16, _lib.BF16):          # 8 bytes suffice at d = 1000: the next check (a null pointer) refuses
        assert call(ALIGNED + 8, dt, 1000) == _lib.EINVAL
        assert "aligned" not in L.vatlq_last_error().decode()
        if name != "vatlq_pairwise_dist_dt":  # the TMA passes at d = 2048 need 16 bytes in every dtype
            assert call(ALIGNED + 8, dt, K) == _lib.EINVAL and "16-byte" in L.vatlq_last_error().decode()


def test_workspace_bytes_dt(built_lib):
    _lib = built_lib._lib
    L = _lib.lib()
    for n in (1, 30001, 1_000_000):
        for d, batch in ((K, 16), (K, 64), (K, 8), (1000, 16)):
            f32 = L.vatlq_coreset_workspace_bytes(n, d, batch)
            assert L.vatlq_coreset_workspace_bytes_dt(n, d, batch, _lib.F32) == f32
            copy = n * 4096 if (d == K and batch >= 16) else 0
            for dt in (_lib.F16, _lib.BF16):
                assert L.vatlq_coreset_workspace_bytes_dt(n, d, batch, dt) == f32 - copy, (n, d, batch)
    assert L.vatlq_coreset_workspace_bytes_dt(100, K, 16, 3) == 0


def test_ops_dtype_rules(built_lib):
    ops, err = built_lib.ops, built_lib._lib.VatlqError
    assert set(ops.EMBEDDING_DTYPES) == {torch.float32, torch.float16, torch.bfloat16}
    unc = torch.zeros(4, dtype=torch.float64)
    for dt in (torch.float16, torch.bfloat16, torch.float32, torch.float64):
        X = torch.zeros((4, 16), dtype=dt)
        with pytest.raises(err, match="CUDA tensor"):
            ops.coreset_select(X, unc, [], 1, 0.0, 0.01)
        with pytest.raises(err, match="CUDA tensor"):
            ops.pairwise_dist(X, [0])


def test_tc_init_true_refuses_16bit_x(built_lib, monkeypatch):
    """tc_init=True with a 16-bit X raises before any device work (the tcgen05 init is TF32, fp32 X only)."""
    ops, err = built_lib.ops, built_lib._lib.VatlqError
    monkeypatch.setattr(ops, "_embeddings", lambda t, name: t)          # (a CPU tensor stands in for a CUDA one)
    for dt in (torch.float16, torch.bfloat16):
        with pytest.raises(err, match="tc_init"):
            ops.coreset_select(torch.zeros((1000, K), dtype=dt), None, list(range(400)), 8, 0.6, 0.01, tc_init=True)


@pytest.mark.parametrize("filt,rep,dtype,expect", [
    ("Coreset", "None", torch.float16, torch.float16),
    ("Coreset", "Random", torch.bfloat16, torch.bfloat16),
    ("Coreset", "Influence", torch.bfloat16, torch.float32),
    ("Diversity", "None", torch.float16, torch.float32),
    ("K-Means", "None", torch.bfloat16, torch.float32),
    ("weighted", "Random", torch.float16, torch.float32),
    ("Coreset", "None", torch.float32, torch.float32),
    ("Coreset", "None", torch.float64, torch.float32),
])
def test_controller_keeps_16bit_embeddings_only_for_the_coreset(built_lib, filt, rep, dtype, expect):
    from vatlq import active_learning as AL
    assert AL.embedding_store_dtype(filt, rep, dtype) == expect


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, dtypes, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    td.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from vatlq import _lib, dist
        n = 7
        X = (torch.arange(n * 4, dtype=torch.float32).reshape(n, 4) / 8).to(dtypes[rank])
        lo, hi = dist.shard_range(n, rank, world)
        try:
            dist._agree_dtype(X[lo:hi], "distributed_query")
        except _lib.VatlqError as e:
            q.put((rank, "VatlqError", str(e)))
            return
        full = dist.allgather_rows(X[lo:hi], n, world)
        q.put((rank, "ok" if full.dtype == dtypes[rank] and torch.equal(full, X) else "mismatch", ""))
    finally:
        td.destroy_process_group()


def _run2(dtypes):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, dtypes, q)) for r in range(2)]
    for p in ps:
        p.start()
    for p in ps:
        p.join(timeout=120)
    hung = [p.is_alive() for p in ps]
    for p in ps:
        if p.is_alive():
            p.kill()
    assert not any(hung), "dtype agreement hung"
    return sorted(q.get(timeout=5) for _ in ps)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_distributed_query_gathers_16bit_rows_world2(dtype):
    res = _run2([dtype, dtype])
    assert [r[1] for r in res] == ["ok", "ok"], res


def test_distributed_query_dtype_mismatch_raises_on_every_rank():
    res = _run2([torch.float16, torch.float32])
    assert [r[1] for r in res] == ["VatlqError", "VatlqError"], res
    assert all("distributed_query" in r[2] and "different dtypes" in r[2] for r in res), res


# ---- the screen's bound for 16-bit X: |S~ - S| <= 2^-12 |x||c| + 2^-120 (|x| + |c|) + 2^-114 (half of E16's terms)
U16, ABS1, ABS0 = 2.0 ** -12, 2.0 ** -120, 2.0 ** -114


def _round(v, dtype):
    return torch.from_numpy(v).to(dtype).to(torch.float64).numpy()


def _adversarial16(rng, dtype):
    top = 60000.0 if dtype == torch.float16 else 1e19     # (bf16: products up to ~1e38, just inside fp32)
    out = []
    for t in range(48):
        x, c = rng.standard_normal(K), rng.standard_normal(K)
        kind = t % 6
        if kind == 0:      # per-element scales over the whole range of the type
            lo = -24 if dtype == torch.float16 else -60
            x *= 2.0 ** rng.uniform(lo, 14, K)
            c *= 2.0 ** rng.uniform(lo, 14, K)
        elif kind == 1:    # cancellation: c close to -x
            c = -x + 1e-2 * rng.standard_normal(K)
        elif kind == 2:    # S close to 0 with large terms
            c = x.copy()
            c[K // 2:] *= -1
        elif kind == 3:    # near the top of the range
            x = np.clip(x * top / 4, -top, top)
            c = rng.uniform(-1, 1, K)
        elif kind == 4:    # subnormals of the type against ordinary values
            x *= 2e-6 if dtype == torch.float16 else 1e-39
        else:              # all large, same sign: the longest accumulation
            x, c = np.abs(x) * 100, np.abs(c) * 100
        out.append((_round(x, dtype), _round(c, dtype)))
    return out


def _fp32_tree_dot(x, c):
    """Exact products rounded to fp32 (exact for two fp16 or two bf16 values), summed in fp32 as the screen does: 16
    features per MMA step in a sequential chain per K segment of 256, the 8 segments added in fp64."""
    p = (x * c).astype(np.float32).reshape(8, 16, 16)
    seg = np.zeros(8, np.float32)
    for s in range(16):
        step = np.zeros(8, np.float32)
        for e in range(16):
            step = (step + p[:, s, e]).astype(np.float32)
        seg = (seg + step).astype(np.float32)
    return float(np.sum(seg.astype(np.float64)))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16])
def test_16bit_bound_on_adversarial_vectors(dtype):
    rng = np.random.default_rng(9)
    worst = 0.0
    for x, c in _adversarial16(rng, dtype):
        S = float(np.sum(x.astype(np.longdouble) * c.astype(np.longdouble)))
        prod = x * c
        if dtype == torch.float16 or np.all(np.abs(prod[prod != 0]) >= 2.0 ** -126):
            assert np.array_equal(prod.astype(np.float32).astype(np.float64), prod)   # exact in fp32
        nx, nc = float(np.sqrt(np.sum(x * x))), float(np.sqrt(np.sum(c * c)))
        bound = U16 * nx * nc + ABS1 * (nx + nc) + ABS0
        St = _fp32_tree_dot(x, c)
        assert np.isfinite(St)
        assert abs(St - S) <= bound, (St, S, bound)
        worst = max(worst, abs(St - S) / bound)
    assert worst < 0.5    # E16 = 2 x these terms: a margin of at least 2 on these vectors
