"""CPU: the host side of fp16 / bf16 heat maps — argument checks of the *_dt entry points (no device needed), the
ops layer's dtype rules, the controller's pass-through of 16-bit estimator output, and the dtype agreement of the
halo exchange on two gloo processes.  The kernels themselves are checked on the GPU (test_gpu_half.py)."""
import ctypes as C
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as td
import torch.multiprocessing as mp

N, J, HH, WW = 1, 17, 64, 48
ALIGNED, BUF = 0x10000, 0x20000        # fake device addresses: the checks must reject before touching them
BIG = 1 << 30


def _entries(L):
    """name -> call(H pointer, dtype) of the four *_dt entry points on one 17 x 64 x 48 frame"""
    return {
        "vatlq_heatmap_scan_dt": lambda h, dt: L.vatlq_heatmap_scan_dt(
            C.c_void_p(h), dt, None, None, N, J, HH, WW, None, None, None, C.c_void_p(BUF), None, None, None, None, None,
            C.c_void_p(BUF), BIG, None),
        "vatlq_thc3_dt": lambda h, dt: L.vatlq_thc3_dt(C.c_void_p(h), None, None, dt, None, None, N, J, HH, WW,
                                                       C.c_void_p(BUF), None),
        "vatlq_heatmap_entropy_dt": lambda h, dt: L.vatlq_heatmap_entropy_dt(C.c_void_p(h), dt, N, J, HH, WW, C.c_void_p(BUF),
                                                                             C.c_void_p(BUF), BIG, None),
        "vatlq_peak_unc_dt": lambda h, dt: L.vatlq_peak_unc_dt(C.c_void_p(h), dt, N, J, HH, WW, C.c_void_p(BUF), None,
                                                               C.c_void_p(BUF), BIG, None),
    }


@pytest.mark.parametrize("name", ["vatlq_heatmap_scan_dt", "vatlq_thc3_dt", "vatlq_heatmap_entropy_dt", "vatlq_peak_unc_dt"])
def test_dt_entries_reject_bad_dtype_and_alignment(built_lib, name):
    _lib = built_lib._lib
    L = _lib.lib()
    call = _entries(L)[name]
    for h, dt in [(ALIGNED, 3), (ALIGNED, -1), (ALIGNED + 4, _lib.F16), (ALIGNED + 2, _lib.BF16)]:
        assert call(h, dt) == _lib.EINVAL, (h, dt)
        msg = L.vatlq_last_error().decode()
        assert name in msg and ("dtype" in msg or "aligned" in msg), msg
    if name == "vatlq_heatmap_scan_dt":   # the TMA scan needs 16 bytes in every dtype
        assert call(ALIGNED + 8, _lib.BF16) == _lib.EINVAL and "16-byte" in L.vatlq_last_error().decode()


def test_ops_reject_host_and_unsupported_heatmaps(built_lib):
    ops, err = built_lib.ops, built_lib._lib.VatlqError
    for dt in (torch.float16, torch.bfloat16, torch.float32, torch.float64):
        H = torch.zeros((2, J, HH, WW), dtype=dt)
        for fn in (ops.heatmap_scan, ops.heatmap_entropy, ops.peak_uncertainty, lambda t: ops.thc3(t, t, None, [1, 1], None)):
            with pytest.raises(err, match="CUDA tensor"):
                fn(H)
    assert set(ops.HEATMAP_DTYPES) == {torch.float32, torch.float16, torch.bfloat16}


@pytest.mark.parametrize("dtype,expect", [(torch.bfloat16, torch.bfloat16), (torch.float16, torch.float16),
                                          (torch.float64, torch.float32)])
def test_eval_and_query_passes_16bit_heatmaps_through(built_lib, monkeypatch, dtype, expect):
    """The estimator's 16-bit heat maps reach the scan unconverted; any other dtype is `.float()`-ed as before."""
    import test_gpu_query as TQ
    import test_host_controller_cpu as HC
    v = built_lib
    HC._install_stand_ins(monkeypatch, v)
    stand_in, seen = v.ops.heatmap_scan, []

    def recording_scan(H, *a, **k):
        seen.append(H.dtype)
        for key in ("halo_prev", "halo_next"):
            if k.get(key) is not None:
                assert k[key].dtype == H.dtype
                k[key] = k[key].float()
        return stand_in(H.float(), *a, **k)    # (the oracle stand-in computes on numpy fp32)

    monkeypatch.setattr(v.ops, "heatmap_scan", recording_scan)
    n = 40
    ids, ip, inx = v.synth.track_flags(n, np.random.default_rng(3), 8.0)
    H = v.synth.heatmaps(n, seed=3, track_ids=ids)
    boxes = v.synth.boxes_xyxy(n, 3)
    X = v.synth.embeddings(n, d=2048, seed=4)
    cfg, opt = TQ.cfg_opt("THC", "None")
    est = TQ.FakeEstimator(torch.from_numpy(H).to(dtype), torch.from_numpy(X))
    al = v.ActiveLearning(cfg, opt, model=est, eval_loader=TQ.loader(n, boxes, ip, inx, 16), eval_len=n,
                          AE=v.synth.ae_weights(42, 4))
    al.eval_and_query()
    assert len(seen) >= 3 and set(seen) == {expect}, seen
    assert len(al.query_list_list["Round0"]) == al.query_sizes[0]


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
        g = torch.Generator().manual_seed(5)
        n = 6
        H = (torch.randn((n, 3, 4, 4), generator=g) * 1e-3).to(dtypes[rank])   # identical on every rank
        H.view(-1)[:4] = torch.tensor([float("nan"), float("inf"), -0.0, 1e-30]).to(dtypes[rank])
        lo, hi = dist.shard_range(n, rank, world)
        try:
            hp, hn = dist.exchange_halo(H[lo], H[hi - 1], rank, world)
        except _lib.VatlqError as e:
            q.put((rank, "VatlqError", str(e)))
            return
        bits = lambda t: t.view(torch.int16)
        ok = ((hp is None) if lo == 0 else torch.equal(bits(hp), bits(H[lo - 1]))) and \
             ((hn is None) if hi == n else torch.equal(bits(hn), bits(H[hi])))
        q.put((rank, "ok" if ok and (hp if hp is not None else hn).dtype == dtypes[rank] else "mismatch", ""))
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
    assert not any(hung), "exchange_halo hung"
    return sorted(q.get(timeout=5) for _ in ps)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
def test_exchange_halo_16bit_world2(dtype):
    res = _run2([dtype, dtype])
    assert [r[1] for r in res] == ["ok", "ok"], res


def test_exchange_halo_dtype_mismatch_raises_on_every_rank():
    res = _run2([torch.bfloat16, torch.float32])
    assert [r[1] for r in res] == ["VatlqError", "VatlqError"], res
    assert all("different dtypes" in r[2] for r in res), res
