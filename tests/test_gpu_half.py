"""GPU: fp16 / bf16 heat maps.  Contract (include/vatlq.h): every output for a 16-bit H equals, bit for bit, the fp32
path's output for H.float() — compared as bit patterns, so NaN outputs compare too."""
import hashlib
import os
import socket
from types import SimpleNamespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16]


def _same(a, b, what=""):
    if a is None or b is None:
        assert a is None and b is None, what
        return
    a, b = a.contiguous(), b.contiguous()
    assert a.dtype == b.dtype and a.shape == b.shape, what
    iv = {1: torch.uint8, 4: torch.int32, 8: torch.int64}[a.element_size()]
    bad = (a.view(iv) != b.view(iv)).sum().item()
    assert bad == 0, f"{what}: {bad} entries differ"


def _f(t):
    return None if t is None else t.float()


def _scan_eq(ops, H, ip=None, inx=None, boxes=None, hp=None, hn=None):
    r16 = ops.heatmap_scan(H, ip, inx, boxes, halo_prev=hp, halo_next=hn)
    r32 = ops.heatmap_scan(H.float(), ip, inx, boxes, halo_prev=_f(hp), halo_next=_f(hn))
    for f in ("thc", "peak_sum", "peak_cnt", "peak_mean", "coords_hm", "kpts"):
        _same(getattr(r16, f), getattr(r32, f), f)
    return r16


def _special_maps(dtype, n=6, h=64, w=48, seed=0):
    """Synthetic maps plus the corner cases: NaN, +-inf, all-negative, all-zero, -0.0 / +0.0 ties, maxima on the
    border and next to it (quarter-shift edge), 16-bit subnormals, plateaus large enough to overflow the MPE / Margin
    candidate list, tiny sums (Entropy's elementwise branch)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    H = torch.rand((n, 17, h, w), generator=g) * 0.3
    H[0, 0, 10, 10] = float("nan")
    H[0, 1, 12, 12] = float("inf")
    H[0, 2, 14, 14] = float("-inf")
    H[0, 3] = -H[0, 3] - 0.1                      # all negative
    H[0, 4] = 0.0                                 # all zero
    H[0, 5] = -1.0
    H[0, 5, 3:9, 4:9] = 0.0
    H[0, 5, 5, 5:7] = -0.0                        # -0.0 / +0.0 ties at the maximum
    H[0, 6, 0, 17] = 2.0                          # maximum on the border
    H[0, 7, 1, 1] = 2.0                           # quarter-shift edge (x == 1, y == 1: no shift)
    H[0, 8, h - 2, w - 2] = 2.0
    H[0, 9, 2, 2] = 2.0                           # first interior pixel that shifts
    H[0, 9, 2, 3] = 1.0
    H[1, 0] = torch.rand((h, w), generator=g) * 5e-5         # fp16 subnormals
    H[1, 1] = torch.rand((h, w), generator=g) * 1e-39        # bf16 (and fp32) subnormals
    H[1, 2] = torch.rand((h, w), generator=g) * 1e-12        # tiny sum
    H[1, 3] = 1.0
    H[1, 3, 7, 9] = 0.0                           # one plateau over the whole map (candidate list overflow)
    H[1, 4] = (torch.rand((h, w), generator=g) * 4).floor() / 4  # four-level plateaus
    H[1, 5] = 0.5
    H[1, 5, 15, 15] = 0.25                        # and one more plateau
    return H.to(DEV).to(dtype)


@pytest.fixture(scope="module")
def pools(built_lib):
    synth = built_lib.synth
    out = {}
    for n, seed, mean_len in [(256, 0, 30.0), (67, 5, 3.0), (1, 6, 30.0), (2, 7, 30.0)]:
        ids, ip, inx = synth.track_flags(n, np.random.default_rng(seed), mean_len)
        H = torch.from_numpy(synth.heatmaps(n + 2, seed=seed)).to(DEV)
        out[n] = SimpleNamespace(H=H[1:n + 1], hp=H[0], hn=H[n + 1], ip=ip, inx=inx,
                                 boxes=torch.from_numpy(synth.boxes_xyxy(n, seed)).to(DEV))
    return out


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("n", [256, 67, 1, 2])
@pytest.mark.parametrize("halos", [False, True])
def test_scan_equals_fp32_on_upcast(built_lib, pools, dtype, n, halos):
    p = pools[n]
    H = p.H.to(dtype)
    hp, hn = (p.hp.to(dtype), p.hn.to(dtype)) if halos else (None, None)
    _scan_eq(built_lib.ops, H, p.ip, p.inx, p.boxes, hp, hn)
    _scan_eq(built_lib.ops, H)                                     # no flags, no boxes


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("shape", [(64, 48), (20, 24)])          # (20, 24): the generic kernels
def test_special_maps_equal_fp32_on_upcast(built_lib, dtype, shape):
    ops = built_lib.ops
    H = _special_maps(dtype, h=shape[0], w=shape[1])
    n = H.shape[0]
    ip, inx = np.array([0, 1, 1, 1, 0, 1], np.uint8), np.array([1, 1, 1, 0, 1, 0], np.uint8)
    boxes = torch.tensor([[10.0, 20.0, 10.0 + 48 * 3, 20.0 + 64 * 3]] * n, device=DEV)
    r = _scan_eq(ops, H, ip, inx, boxes, hp=H[3], hn=H[2])
    assert torch.isnan(r.thc).any() or torch.isinf(r.thc).any()
    # thc3: separately forwarded neighbours
    prev, nxt = torch.roll(H, 1, 0), torch.roll(H, -1, 0)
    _same(ops.thc3(H, prev, nxt, ip, inx), ops.thc3(H.float(), prev.float(), nxt.float(), ip, inx), "thc3")
    _same(ops.thc3(H, None, nxt, None, inx), ops.thc3(H.float(), None, nxt.float(), None, inx), "thc3 next only")
    e16 = ops.heatmap_entropy(H)
    _same(e16, ops.heatmap_entropy(H.float()), "entropy")
    assert torch.isnan(e16[0]) or torch.isinf(e16[0])
    m16, g16 = ops.peak_uncertainty(H)
    m32, g32 = ops.peak_uncertainty(H.float())
    _same(m16, m32, "mpe")
    _same(g16, g32, "margin")


@pytest.mark.parametrize("dtype", DTYPES)
def test_peak_plateaus_take_the_redo_path(built_lib, dtype):
    """Quantised maps with plateaus: the register kernel's candidate list overflows and the redo kernel runs."""
    ops = built_lib.ops
    H = _special_maps(dtype, n=64, seed=3)
    H[:, :, 8:56, 8:40] = H[:, :, 8:56, 8:40].float().mul(4).round().div(4).to(dtype)
    m16, g16 = ops.peak_uncertainty(H)
    m32, g32 = ops.peak_uncertainty(H.float())
    _same(m16, m32, "mpe")
    _same(g16, g32, "margin")
    os.environ["VATLQ_PEAK_GENERIC"] = "1"
    try:
        mg, gg = ops.peak_uncertainty(H)        # the generic routine alone gives the same result
    finally:
        del os.environ["VATLQ_PEAK_GENERIC"]
    _same(mg, m32, "mpe generic")
    _same(gg, g32, "margin generic")


def test_ops_reject_other_dtypes_and_mixed_halos(built_lib):
    ops, err = built_lib.ops, built_lib._lib.VatlqError
    H = torch.zeros((3, 17, 64, 48), device=DEV, dtype=torch.bfloat16)
    for fn in (ops.heatmap_scan, ops.heatmap_entropy, ops.peak_uncertainty):
        with pytest.raises(err, match="float32, torch.float16 or torch.bfloat16"):
            fn(H.double())
    with pytest.raises(err, match="halo_prev"):
        ops.heatmap_scan(H, halo_prev=H[0].float())
    with pytest.raises(err, match="next"):
        ops.thc3(H, None, H.half(), None, [1, 1, 1])


STRATEGIES = ["THC+WPU", "THC", "TPC", "HP", "Entropy", "MPE", "Margin"]


@pytest.fixture(scope="module")
def qpool(built_lib):
    synth = built_lib.synth
    n = 120
    ids, ip, inx = synth.track_flags(n, np.random.default_rng(11), 6.0)
    return SimpleNamespace(n=n, H=torch.from_numpy(synth.heatmaps(n, seed=11, track_ids=ids)).to(DEV),
                           boxes=synth.boxes_xyxy(n, 11), ip=ip, inx=inx, X=synth.embeddings(n, d=256, seed=12),
                           W=synth.ae_weights(42, 4, seed=318))


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("unc", STRATEGIES)
def test_query_pass_chunks_equal_fp32_on_upcast(built_lib, qpool, dtype, unc):
    v, q = built_lib, qpool
    H = q.H.to(dtype)
    for chunk in (1, 7, 4096):
        args = dict(labeled=[3, 50], k=12, moks=0.4, lam=0.01, uncertainty=unc, device=DEV, chunk=chunk)
        r16 = v.run_query(H, q.boxes, q.ip, q.inx, q.X, q.W, **args)
        r32 = v.run_query(H.float(), q.boxes, q.ip, q.inx, q.X, q.W, **args)
        for f in ("thc", "wpu", "peak_mean", "kpts", "unc"):
            _same(getattr(r16, f), getattr(r32, f), f"{unc} chunk {chunk} {f}")
        assert r16.picks.tolist() == r32.picks.tolist()
        assert r16.combine_weight == r32.combine_weight
    # host arrays: numpy float16 / torch CPU bfloat16, copied chunk by chunk without conversion
    Hh = H.cpu().numpy() if dtype == torch.float16 else H.cpu()
    args["chunk"] = 50
    r = v.run_query(Hh, q.boxes, q.ip, q.inx, q.X, q.W, **args)
    r32 = v.run_query(H.float().cpu().numpy(), q.boxes, q.ip, q.inx, q.X, q.W, **args)
    _same(r.unc, r32.unc, "host input")
    assert r.picks.tolist() == r32.picks.tolist()


@pytest.mark.parametrize("dtype", DTYPES)
def test_query_pass_rejects_mixed_dtypes(built_lib, qpool, dtype):
    v, q = built_lib, qpool
    qp = v.QueryPass(q.n, DEV, ae_weights=q.W, uncertainty="THC+WPU")
    bb = torch.from_numpy(q.boxes).to(DEV)
    ip, inx = torch.from_numpy(q.ip).to(DEV), torch.from_numpy(q.inx).to(DEV)
    qp.score_chunk(0, q.H[:10].to(dtype), bb[:10], ip[:10], inx[:10])
    with pytest.raises(v._lib.VatlqError, match="one heat-map dtype"):
        qp.score_chunk(10, q.H[10:20], bb[10:20], ip[10:20], inx[10:20])
    qp2 = v.QueryPass(q.n, DEV, ae_weights=q.W, uncertainty="THC+WPU")
    with pytest.raises(v._lib.VatlqError, match="halo_prev"):
        qp2.score_chunk(0, q.H[:10].to(dtype), bb[:10], ip[:10], inx[:10], halo_prev=q.H[0])


@pytest.mark.parametrize("strict", [False, True])
def test_eval_and_query_bf16_estimator(built_lib, strict):
    """Two rounds with an estimator that returns bf16 against the same estimator returning .float() of it."""
    import test_gpu_query as TQ
    v = built_lib
    n = 200
    ids, ip, inx = v.synth.track_flags(n, np.random.default_rng(1), 10.0)
    H = torch.from_numpy(v.synth.heatmaps(n, seed=1, track_ids=ids)).to(DEV).to(torch.bfloat16)
    boxes = v.synth.boxes_xyxy(n, 1)
    X = torch.from_numpy(v.synth.embeddings(n, d=2048, seed=2)).to(DEV)
    W = v.synth.ae_weights(42, 4)
    rng = np.random.default_rng(7)
    gt = (np.tile(boxes[:, None, :2], (1, 17, 1)) + rng.normal(0, 20.0, (n, 17, 2))).astype(np.float32)
    gt = np.concatenate([gt, np.full((n, 17, 1), 2.0, np.float32)], axis=2)
    runs = []
    for Hm in (H, H.float()):
        cfg, opt = TQ.cfg_opt("THC+WPU", "Coreset")
        opt.strict_prenext = strict
        al = v.ActiveLearning(cfg, opt, model=TQ.FakeEstimator(Hm, X), eval_loader=None, eval_len=n, AE=W)
        for _ in range(2):
            al.eval_loader = TQ.loader(n, boxes, ip, inx, 64, gt)
            al.eval_and_query()
        runs.append(al)
    a, b = runs
    assert a.query_list_list == b.query_list_list
    assert a.uncertainty_dict == b.uncertainty_dict
    assert a.combine_weight == b.combine_weight
    assert a.uncertainty_mean == b.uncertainty_mean
    assert a.moks_queried == b.moks_queried


def _sha(p):
    return hashlib.sha256(np.asarray(p, dtype="<i8").tobytes()).hexdigest()


def test_bench_pool_bf16_at_scale(built_lib):
    """The 170 000-frame bench pool (config 4) in bf16 against the fp32 path on its upcast."""
    v = built_lib
    synth = v.synth
    n, k = 170000, 8500
    free, _ = torch.cuda.mem_get_info()
    if free < n * synth.FRAME_BYTES * 1.5 + n * 2048 * 4 * 1.2 + (8 << 30):
        pytest.skip("not enough free HBM for this pool")
    segs, bb, ip, inx, X, _ = synth.rank_pool(n, 0, n, DEV, "clustered")
    H16 = [(pos, seg.to(torch.bfloat16)) for pos, seg in segs]
    del segs
    torch.cuda.empty_cache()
    W = synth.ae_weights(42, 4)
    res = {}
    for tag in ("bf16", "fp32"):
        H = H16 if tag == "bf16" else [(pos, seg.float()) for pos, seg in H16]
        r = v.run_query(H, bb, ip, inx, X, W, [], k, 0.0, 0.01, batch=16, device=DEV)
        res[tag] = (float(r.thc.double().sum()), float(r.wpu.double().sum()), int(torch.argmax(r.unc)), _sha(r.picks.cpu().numpy()))
        del H, r
        torch.cuda.empty_cache()
    assert res["bf16"] == res["fp32"], res


def _two_gpu_worker(rank, port, q):
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import torch.distributed as td
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    td.init_process_group("nccl", rank=rank, world_size=2, device_id=torch.device("cuda", rank))
    try:
        import vatlq
        from vatlq import dist, synth
        n, k = 3000, 40
        dev = torch.device("cuda", rank)
        ids, ip, inx = synth.track_flags(n, np.random.default_rng(4), 12.0)
        H = torch.from_numpy(synth.heatmaps(n, seed=4, track_ids=ids)).to(dev).to(torch.bfloat16)
        boxes = synth.boxes_xyxy(n, 4)
        X = synth.embeddings(n, d=256, seed=5)
        W = synth.ae_weights(42, 4)
        lo, hi = dist.shard_range(n, rank, 2)
        comm = dist.Comm()
        r = dist.distributed_query(H[lo:hi], torch.from_numpy(boxes[lo:hi]).to(dev), torch.from_numpy(ip[lo:hi]).to(dev),
                                   torch.from_numpy(inx[lo:hi]).to(dev), torch.from_numpy(X[lo:hi]).to(dev), W, [7, 900], n, k,
                                   moks=0.3, comm=comm)
        comm.close()
        one = vatlq.run_query(H.float(), boxes, ip, inx, X, W, [7, 900], k, 0.3, device=dev)
        q.put((rank, r.picks.cpu().tolist() == one.picks.cpu().tolist()))
    finally:
        td.destroy_process_group()


def test_two_gpus_bf16_shards_match_one_gpu_fp32(built_lib):
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
    assert res == [(0, True), (1, True)], res
