"""ctypes binding of libvatlq.so (C ABI in include/vatlq.h).  There is no fallback: a missing
library or a failing call raises."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VATLQ_LIB") or os.path.join(HERE, "libvatlq.so")   # VATLQ_LIB: tuning builds only

_vp, _i64, _int, _sz, _dbl = C.c_void_p, C.c_int64, C.c_int, C.c_size_t, C.c_double

# name -> (restype, argtypes): every symbol include/vatlq.h declares
SIGNATURES = {
    "vatlq_abi_version": (_int, []),
    "vatlq_last_error": (C.c_char_p, []),
    "vatlq_launch_count": (C.c_uint64, []),
    "vatlq_heatmap_scan_workspace_bytes": (_sz, [_i64, _int]),
    "vatlq_heatmap_scan": (_int, [_vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_heatmap_scan_dt": (_int, [_vp, _int, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp,
                                     _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_thc3": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp]),
    "vatlq_thc3_dt": (_int, [_vp, _vp, _vp, _int, _vp, _vp, _i64, _int, _int, _int, _vp, _vp]),
    "vatlq_wpu_weight_count": (_sz, [_int, _int]),
    "vatlq_wpu": (_int, [_vp, _vp, _vp, _int, _int, _int, _vp, _vp, _vp, _i64, _vp]),
    "vatlq_fuse_stats": (_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "vatlq_fuse_combine": (_int, [_vp, _vp, _vp, _i64, _vp, _int, _dbl, _vp, _vp, _vp]),
    "vatlq_fuse_final": (_int, [_vp, _i64, _vp, _vp, _vp]),
    "vatlq_coreset_workspace_bytes": (_sz, [_i64, _int, _int]),
    "vatlq_coreset_init": (_int, [_vp, _i64, _int, _i64, _i64, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vatlq_coreset_init_tc_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "vatlq_coreset_init_tc": (_int, [_vp, _i64, _int, _i64, _i64, _vp, _i64, _vp, _vp, _sz, _int, _vp, _vp, _vp]),
    "vatlq_coreset_select": (_int, [_vp, _i64, _int, _i64, _i64, _vp, _vp, _int, _dbl, _dbl, _i64,
                                    _i64, _i64, _int, _vp, _vp, _vp, _sz, _vp, _vp]),
    "vatlq_coreset_prune_stats": (_int, [_vp, _int]),
    "vatlq_coreset_set_prune": (_int, [_int, _i64]),
    "vatlq_coreset_screen_stats": (_int, [_vp, _int]),
    "vatlq_coreset_set_screen": (_int, [_int]),
    "vatlq_pairwise_dist": (_int, [_vp, _i64, _int, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vatlq_pose_unc": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _int, _vp, _vp, _vp, _vp, _vp]),
    "vatlq_heatmap_entropy": (_int, [_vp, _i64, _int, _int, _int, _vp, _vp, _sz, _vp]),
    "vatlq_heatmap_entropy_dt": (_int, [_vp, _int, _i64, _int, _int, _int, _vp, _vp, _sz, _vp]),
    "vatlq_cosine_workspace_bytes": (_sz, [_int]),
    "vatlq_cosine_colsum": (_int, [_vp, _i64, _int, _vp, _i64, _vp, _vp, _sz, _vp]),
    "vatlq_cosine_rowsum": (_int, [_vp, _i64, _int, _vp, _i64, _vp, _dbl, _vp, _vp]),
    "vatlq_minmax_stats_f64": (_int, [_vp, _vp, _i64, _vp, _vp]),
    "vatlq_fuse_blend": (_int, [_vp, _vp, _vp, _i64, _dbl, _vp, _vp]),
    "vatlq_peak_workspace_bytes": (_sz, [_i64, _int, _int, _int]),
    "vatlq_peak_unc": (_int, [_vp, _i64, _int, _int, _int, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_peak_unc_dt": (_int, [_vp, _int, _i64, _int, _int, _int, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_rank_workspace_bytes": (_sz, [_i64]),
    "vatlq_rank_scores": (_int, [_vp, _vp, _i64, _int, _vp, _vp, _sz, _vp]),
    "vatlq_kmeans_workspace_bytes": (_sz, [_i64, _int, _i64]),
    "vatlq_kmeans_mean_var": (_int, [_vp, _i64, _int, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_kmeans_pp": (_int, [_vp, _i64, _int, _vp, _i64, _i64, _vp, _int, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_kmeans_gather": (_int, [_vp, _int, _vp, _i64, _vp, _vp, _vp, _vp]),
    "vatlq_kmeans_assign": (_int, [_vp, _i64, _int, _vp, _i64, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_kmeans_update": (_int, [_vp, _i64, _int, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "vatlq_kmeans_relocate": (_int, [_vp, _int, _vp, _vp, _vp, _vp, _vp, _int, _vp, _vp, _vp]),
    "vatlq_kmeans_average": (_int, [_vp, _vp, _i64, _int, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "vatlq_kmeans_rowdist": (_int, [_vp, _i64, _int, _vp, _vp, _vp, _vp]),
    "vatlq_kmeans_pick": (_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "vatlq_measure_fp64_mma": (_int, [_vp, _vp, _sz, _vp]),
    "vatlq_oks": (_int, [_vp, _vp, _vp, _i64, _vp, _vp]),
    "vatlq_profile_passes": (_int, [_int]),
    "vatlq_profile_read": (_int, [_vp, _vp, _vp, _int]),
    "vatlq_comm_unique_id": (_int, [_vp]),
    "vatlq_comm_init": (_int, [_vp, _int, _int, C.POINTER(_vp)]),
    "vatlq_comm_mailbox_handle": (_int, [_vp, _vp]),
    "vatlq_comm_attach": (_int, [_vp, _vp, _int]),
    "vatlq_comm_destroy": (_int, [_vp]),
}

_lib = None
EINVAL, ECOMM, ESTATE = -1, -3, -4     # VATLQ_E* of include/vatlq.h
F32, F16, BF16 = 0, 1, 2               # VATLQ_F32 / VATLQ_F16 / VATLQ_BF16: heat-map element types of the *_dt entries


class VatlqError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raises if the CUDA library is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise VatlqError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the query pass)")
        h = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        if h.vatlq_abi_version() != 1:
            raise VatlqError("libvatlq.so ABI version mismatch: rebuild")
        _lib = h
    return _lib


def check(code: int, what: str = ""):
    if code != 0:
        msg = lib().vatlq_last_error().decode(errors="replace")
        raise VatlqError(f"{what or 'libvatlq'} failed with code {code}: {msg}")


def launch_count() -> int:
    return int(lib().vatlq_launch_count())
