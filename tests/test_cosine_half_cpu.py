"""CPU: the host side of the Influence / Diversity cosine row sums on fp16 / bf16 embeddings — the argument checks of
vatlq_cosine_colsum_dt / vatlq_cosine_rowsum_dt (no device needed: every refused call stops before device work), the
fp32 entries forwarding to them, and the dtype rules of ops.cosine_rowsum.  The kernels are checked on the GPU
(test_gpu_cosine_half.py)."""
import contextlib
import ctypes as C

import pytest
import torch

ALIGNED, BUF = 0x10000, 0x20000        # fake device addresses: the checks must reject before touching them
BIG = 1 << 40


def _calls(L):
    """name -> call(X pointer, dtype, d, m) of the two *_dt entry points on a 64-row X without a row list (m != 64 is
    refused after every X check, still before any device work)"""
    return {
        "vatlq_cosine_colsum_dt": lambda x, dt, d, m: L.vatlq_cosine_colsum_dt(
            C.c_void_p(x), dt, 64, d, None, m, C.c_void_p(BUF), C.c_void_p(BUF), BIG, None),
        "vatlq_cosine_rowsum_dt": lambda x, dt, d, m: L.vatlq_cosine_rowsum_dt(
            C.c_void_p(x), dt, 64, d, None, m, C.c_void_p(BUF), 64.0, C.c_void_p(BUF), None),
    }


def _fp32_calls(L):
    """the same calls through the fp32 entries"""
    return {
        "vatlq_cosine_colsum_dt": lambda x, d, m: L.vatlq_cosine_colsum(
            C.c_void_p(x), 64, d, None, m, C.c_void_p(BUF), C.c_void_p(BUF), BIG, None),
        "vatlq_cosine_rowsum_dt": lambda x, d, m: L.vatlq_cosine_rowsum(
            C.c_void_p(x), 64, d, None, m, C.c_void_p(BUF), 64.0, C.c_void_p(BUF), None),
    }


@pytest.mark.parametrize("name", ["vatlq_cosine_colsum_dt", "vatlq_cosine_rowsum_dt"])
def test_dt_entries_reject_bad_dtype_and_alignment(built_lib, name):
    _lib = built_lib._lib
    L = _lib.lib()
    call = _calls(L)[name]
    for dt in (3, -1):
        assert call(ALIGNED, dt, 2048, 64) == _lib.EINVAL
        assert "dtype" in L.vatlq_last_error().decode()
    for x, dt in [(ALIGNED + 4, _lib.F16), (ALIGNED + 2, _lib.BF16), (ALIGNED + 8, _lib.F32), (ALIGNED + 4, _lib.F32)]:
        assert call(x, dt, 2048, 64) == _lib.EINVAL, (x, dt)
        assert "aligned" in L.vatlq_last_error().decode()
    for dt in (_lib.F16, _lib.BF16):          # 8 bytes suffice in 16 bits: the row-count check is the one that refuses
        for d in (4, 12, 256, 2048):
            assert call(ALIGNED + 8, dt, d, 63) == _lib.EINVAL
            msg = L.vatlq_last_error().decode()
            assert "aligned" not in msg and "m must equal n" in msg, msg
        assert call(ALIGNED, dt, 2052, 64) == _lib.EINVAL and "<= 2048" in L.vatlq_last_error().decode()
        assert call(ALIGNED, dt, 6, 64) == _lib.EINVAL and "multiple of 4" in L.vatlq_last_error().decode()


@pytest.mark.parametrize("name", ["vatlq_cosine_colsum_dt", "vatlq_cosine_rowsum_dt"])
def test_fp32_entries_forward_to_dt(built_lib, name):
    """The fp32 entries are the *_dt calls with VATLQ_F32: each refusal is reported by the *_dt entry, with the same
    message the *_dt call gives for the same arguments."""
    _lib = built_lib._lib
    L = _lib.lib()
    dt_call, f32_call = _calls(L)[name], _fp32_calls(L)[name]
    for x, d, m in [(ALIGNED + 8, 2048, 64), (ALIGNED, 6, 64), (ALIGNED, 4096, 64), (ALIGNED, 2048, 63), (0, 2048, 64)]:
        assert f32_call(x, d, m) == _lib.EINVAL, (x, d, m)
        msg = L.vatlq_last_error().decode()
        assert msg.startswith(name + ":"), msg
        assert dt_call(x, _lib.F32, d, m) == _lib.EINVAL
        assert L.vatlq_last_error().decode() == msg
    assert L.vatlq_cosine_workspace_bytes(2048) == L.vatlq_cosine_workspace_bytes(1024) * 2 > 0


class _LooksCuda(torch.Tensor):
    """A CPU tensor that reports is_cuda: the dtype rules of ops.cosine_rowsum can then be checked past the device
    check without a GPU."""

    @property
    def is_cuda(self):
        return True


class _RecordingLib:
    """Stands in for libvatlq: records the dtype code of every cosine call and reports success."""

    def __init__(self):
        self.codes = []

    def vatlq_cosine_workspace_bytes(self, d):
        return 0

    def vatlq_cosine_colsum_dt(self, X, dtype, *args):
        self.codes.append(("colsum", dtype))
        return 0

    def vatlq_cosine_rowsum_dt(self, X, dtype, *args):
        self.codes.append(("rowsum", dtype))
        return 0


def test_ops_cosine_rowsum_dtype_rules(built_lib, monkeypatch):
    ops, _lib = built_lib.ops, built_lib._lib
    err = _lib.VatlqError
    for dt in (torch.float16, torch.bfloat16, torch.float32, torch.float64):
        with pytest.raises(err, match="CUDA tensor"):
            ops.cosine_rowsum(torch.zeros((4, 16), dtype=dt))
    with pytest.raises(err, match="CUDA tensor"):
        ops.cosine_rowsum(torch.zeros((4, 16)).numpy())
    fake = _RecordingLib()
    monkeypatch.setattr(_lib, "lib", lambda: fake)
    monkeypatch.setattr(ops, "_stream", lambda: None)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    for dt in (torch.float64, torch.int8, torch.float8_e4m3fn):
        with pytest.raises(err, match="torch.float32, torch.float16 or torch.bfloat16"):
            ops.cosine_rowsum(torch.zeros((4, 16)).to(dt).as_subclass(_LooksCuda))
    assert fake.codes == []
    for dt, code in ((torch.float32, _lib.F32), (torch.float16, _lib.F16), (torch.bfloat16, _lib.BF16)):
        fake.codes.clear()
        out = ops.cosine_rowsum(torch.zeros((4, 16), dtype=dt).as_subclass(_LooksCuda), rows=[0, 2])
        assert fake.codes == [("colsum", code), ("rowsum", code)]
        assert out.dtype == torch.float64 and out.shape == (2,)
