"""ctypes binding of libb2s.so (include/b2s.h).  No fallback: a missing library or a
missing CUDA device raises — the product never computes on the CPU.

torch is used for exactly three things here: owning device memory, naming the current
CUDA stream, and (elsewhere) torch.distributed.  No torch op is on the compute path.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from pathlib import Path

_LIB_NAME = "libb2s.so"
_lock = threading.Lock()
_lib = None
_lib_pid = None

IDX_BITS = 22
IDX_MASK = (1 << IDX_BITS) - 1
NONE_KEY = 0xFFFFFFFF
DESC_BYTES = 32
SELECT_MAX_QUERIES = 32768
ABI_VERSION = 5
VARIANT_POPC = 0
VARIANT_I8MMA = 1
VARIANT_I8MMA1 = 2
HAMMING_BEST_ONLY = 0x100      # OR-ed into the variant: fwd_second not needed (cross-check-only matching)

PIPE_IDS = {"popc": 0, "lop3": 1, "iadd": 2, "imnmx": 3, "dfma": 4, "ffma": 5, "imad": 6, "redux": 7, "shfl": 8,
            "vmin_u16x2": 9, "vmin3_u16x2": 10, "viaddmax_u16x2": 11, "setp_sel": 12, "prmt": 13, "ffma2": 14, "ffma2+ffma": 15, "ffma2+2ffma": 16,
            "ffma2+iadd": 17, "ffma2+2iadd": 18, "ffma2_3src": 19,
            "ffma2_s_p_p": 20, "ffma2_s_p_s": 21, "ffma_3src": 22, "ffma2_p_p_q": 23, "ffma2_s_p_samep": 24}


class RecordSink(C.Structure):
    """b2s_record_sink (include/b2s.h): the winner kernel also writes the pair's result record."""
    _fields_ = [("records", C.c_void_p), ("record_bytes", C.c_size_t), ("out_q", C.c_void_p), ("out_t", C.c_void_p),
                ("out_d", C.c_void_p), ("stride", C.c_int), ("pair_id0", C.c_int)]


class B2SError(RuntimeError):
    """libb2s returned a non-zero status."""


def lib_path() -> Path:
    """libb2s.so next to this module; B2S_LIB overrides it (diagnostic builds only, e.g. tools/k3h_check.py)."""
    override = os.environ.get("B2S_LIB")
    return Path(override) if override else Path(__file__).resolve().parent / _LIB_NAME


def _declare(lib):
    vp, i32, u64, sz, dbl = C.c_void_p, C.c_int, C.c_uint64, C.c_size_t, C.c_double
    ip = C.POINTER(C.c_int)
    lib.b2s_abi_version.restype = i32
    lib.b2s_abi_version.argtypes = []
    lib.b2s_launch_count.restype = C.c_ulonglong
    lib.b2s_launch_count.argtypes = []
    lib.b2s_last_error.restype = C.c_char_p
    lib.b2s_last_error.argtypes = []
    lib.b2s_device_info.restype = i32
    lib.b2s_device_info.argtypes = [ip, ip, ip, ip]
    lib.b2s_hamming_workspace_bytes.restype = sz
    lib.b2s_hamming_workspace_bytes.argtypes = [i32, i32]
    lib.b2s_hamming_workspace_bytes_v.restype = sz
    lib.b2s_hamming_workspace_bytes_v.argtypes = [i32, i32, i32, i32, i32, i32]
    lib.b2s_hamming_knn2_batched.restype = i32
    lib.b2s_hamming_knn2_batched.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32,
                                             vp, vp, vp, i32, i32, vp, sz, vp]
    lib.b2s_hamming_shared_workspace_bytes.restype = sz
    lib.b2s_hamming_shared_workspace_bytes.argtypes = [i32, i32, i32, i32, i32, i32]
    lib.b2s_hamming_last_plan.restype = None
    lib.b2s_hamming_last_plan.argtypes = [ip, ip, ip]
    lib.b2s_hamming_knn2_shared.restype = i32
    lib.b2s_hamming_knn2_shared.argtypes = [vp, vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, i32, i32, vp, sz, vp]
    lib.b2s_hamming_set_config.restype = i32
    lib.b2s_hamming_set_config.argtypes = [i32, i32, i32]
    lib.b2s_hamming_get_config.restype = i32
    lib.b2s_hamming_get_config.argtypes = [ip, ip, ip]
    lib.b2s_select_matches.restype = i32
    lib.b2s_select_matches.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, i32, i32,
                                       vp, vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.b2s_record_bytes.restype = sz
    lib.b2s_record_bytes.argtypes = [i32]
    lib.b2s_pose_record_bytes.restype = sz
    lib.b2s_pose_record_bytes.argtypes = [i32]
    lib.b2s_pack_records.restype = i32
    lib.b2s_pack_records.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp, sz, vp]
    lib.b2s_rank_pairs.restype = i32
    lib.b2s_rank_pairs.argtypes = [vp, vp, vp, i32, i32, i32, vp, vp, vp, vp, vp]
    lib.b2s_eight_point_batched.restype = i32
    lib.b2s_eight_point_batched.argtypes = [vp, vp, vp, i32, i32, vp, u64, vp, i32, vp, vp, vp, vp, vp]
    lib.b2s_ransac_score_batched.restype = i32
    lib.b2s_ransac_score_batched.argtypes = [vp, vp, vp, i32, vp, i32, dbl, vp, i32, i32, vp, vp]
    lib.b2s_ransac_score_tc_workspace_bytes.restype = sz
    lib.b2s_ransac_score_tc_workspace_bytes.argtypes = [i32, i32, i32]
    lib.b2s_ransac_score_tc.restype = i32
    lib.b2s_ransac_score_tc.argtypes = [vp, vp, vp, i32, i32, vp, i32, dbl, vp, vp, vp, sz, vp, vp, i32, vp, vp]
    lib.b2s_homography_dlt_batched.restype = i32
    lib.b2s_homography_dlt_batched.argtypes = [vp, vp, vp, i32, i32, vp, u64, vp, i32, vp, vp, vp]
    lib.b2s_homography_score_batched.restype = i32
    lib.b2s_homography_score_batched.argtypes = [vp, vp, vp, i32, vp, i32, dbl, vp, vp, vp]
    lib.b2s_homography_select.restype = i32
    lib.b2s_homography_select.argtypes = [vp, vp, vp, vp, i32, vp, i32, dbl, vp, vp, vp, vp, vp]
    lib.b2s_decompose_essential_batched.restype = i32
    lib.b2s_decompose_essential_batched.argtypes = [vp, vp, vp, vp, vp, i32, i32, vp, vp, vp, vp]
    lib.b2s_refit_essential_batched.restype = i32
    lib.b2s_refit_essential_batched.argtypes = [vp, vp, vp, vp, i32, vp, vp, vp, vp, vp]
    lib.b2s_pose_pick.restype = i32
    lib.b2s_pose_pick.argtypes = [vp, vp, i32, vp, vp, vp]
    lib.b2s_five_point_batched.restype = i32
    lib.b2s_five_point_batched.argtypes = [vp, vp, vp, i32, i32, vp, u64, vp, vp, vp, vp]
    lib.b2s_bow_histogram_batched.restype = i32
    lib.b2s_bow_histogram_batched.argtypes = [vp, vp, i32, i32, vp, i32, vp, vp, vp, vp]
    lib.b2s_bow_cosine.restype = i32
    lib.b2s_bow_cosine.argtypes = [vp, vp, i32, i32, vp, vp]
    lib.b2s_ransac_winner_workspace_bytes.restype = sz
    lib.b2s_ransac_winner_workspace_bytes.argtypes = [i32, i32]
    lib.b2s_ransac_winner_batched.restype = i32
    lib.b2s_ransac_winner_batched.argtypes = [vp, vp, vp, i32, vp, i32, dbl, vp, vp, vp, vp, vp, sz, vp, vp, vp, i32, vp]
    lib.b2s_ransac_select.restype = i32
    lib.b2s_ransac_select.argtypes = [vp, vp, vp, vp, i32, vp, i32, dbl, vp, vp, vp, vp, vp, i32, vp]
    lib.b2s_displacement_median_batched.restype = i32
    lib.b2s_displacement_median_batched.argtypes = [vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, vp]
    lib.b2s_refit_homography_batched.restype = i32
    lib.b2s_refit_homography_batched.argtypes = [vp, vp, vp, vp, i32, vp, vp, vp]
    lib.b2s_robust_pose_decide.restype = i32
    lib.b2s_robust_pose_decide.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32, vp]
    lib.b2s_robust_pose_decide_records.restype = i32
    lib.b2s_robust_pose_decide_records.argtypes = [vp, vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp, vp, i32,
                                                   vp, vp]
    lib.b2s_hamming_kernel_timing.restype = i32
    lib.b2s_hamming_kernel_timing.argtypes = [i32, C.POINTER(C.c_float)]
    lib.b2s_mma_microbench.restype = i32
    lib.b2s_mma_microbench.argtypes = [i32, i32, C.POINTER(dbl), vp]
    lib.b2s_tmem_microbench.restype = i32
    lib.b2s_tmem_microbench.argtypes = [i32, i32, C.POINTER(dbl), vp, vp]
    lib.b2s_pipe_microbench.restype = i32
    lib.b2s_pipe_microbench.argtypes = [i32, i32, i32, C.POINTER(dbl), vp, vp]
    return lib


EXPORTS = (
    "b2s_abi_version", "b2s_launch_count", "b2s_last_error", "b2s_device_info", "b2s_hamming_workspace_bytes", "b2s_hamming_workspace_bytes_v",
    "b2s_hamming_knn2_batched", "b2s_hamming_set_config", "b2s_hamming_get_config",
    "b2s_select_matches", "b2s_eight_point_batched", "b2s_ransac_score_batched",
    "b2s_ransac_select", "b2s_pipe_microbench", "b2s_mma_microbench", "b2s_tmem_microbench",
    "b2s_hamming_kernel_timing", "b2s_ransac_score_tc_workspace_bytes", "b2s_ransac_score_tc",
    "b2s_homography_dlt_batched", "b2s_homography_score_batched", "b2s_homography_select", "b2s_decompose_essential_batched", "b2s_refit_essential_batched", "b2s_pose_pick", "b2s_five_point_batched",
    "b2s_bow_histogram_batched", "b2s_bow_cosine", "b2s_hamming_shared_workspace_bytes", "b2s_hamming_knn2_shared", "b2s_hamming_last_plan",
    "b2s_record_bytes", "b2s_pose_record_bytes", "b2s_pack_records", "b2s_rank_pairs", "b2s_ransac_winner_workspace_bytes", "b2s_ransac_winner_batched",
    "b2s_displacement_median_batched", "b2s_refit_homography_batched", "b2s_robust_pose_decide",
    "b2s_robust_pose_decide_records",
)


def load_library():
    """dlopen libb2s.so (no CUDA call is made).  Raises if it has not been built."""
    global _lib, _lib_pid
    with _lock:
        if _lib is not None and _lib_pid == os.getpid():
            return _lib
        path = lib_path()
        if not path.exists():
            raise B2SError(
                f"{path} is missing — build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C monocular-visual-slam_b200/csrc`. There is no CPU fallback.")
        _lib = _declare(C.CDLL(str(path)))
        _lib_pid = os.getpid()
        if _lib.b2s_abi_version() != ABI_VERSION:
            raise B2SError("libb2s.so ABI version mismatch")
        return _lib


def require_cuda():
    """Import torch lazily and insist on a CUDA device (fork-safe: called on first use only)."""
    import torch

    if not torch.cuda.is_available():
        raise B2SError("b200slam needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def check(status: int):
    if status != 0:
        msg = load_library().b2s_last_error().decode("utf-8", "replace")
        if status == 1:
            raise ValueError(f"libb2s: {msg}")
        raise B2SError(f"libb2s error {status}: {msg}")


def ptr(t) -> int | None:
    """Device (or host) pointer of a torch tensor / numpy array, None passes NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return t.data_ptr()
    return t.ctypes.data


def current_stream() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream
