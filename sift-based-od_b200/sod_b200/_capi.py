"""ctypes binding of libsod_b200.so (declared in include/sod.h).

There is no fallback: if the library is missing or cannot be loaded, importing this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

# SOD_B200_LIB selects another build of the same library (kernel experiments); never a fallback.
_LIB_PATH = Path(os.environ.get("SOD_B200_LIB") or Path(__file__).resolve().parent / "libsod_b200.so")

SOD_OK = 0
DESC_DIM = 128
TILE_ROWS = 128


class SodError(RuntimeError):
    pass


def _load() -> C.CDLL:
    if not _LIB_PATH.exists():
        raise ImportError(
            f"{_LIB_PATH} not built: run `python __graft_entry__.py` (or sod_b200.build.build()); "
            "the CUDA library is the only implementation of the hot path")
    return C.CDLL(str(_LIB_PATH))


lib = _load()

_p = C.c_void_p
_i64 = C.c_int64
_i32 = C.c_int32



class Keypoints(C.Structure):
    _fields_ = [("xy", _p), ("angle", _p), ("octave", _p), ("n", _i64)]


class Scene(C.Structure):
    _fields_ = [("query", Keypoints), ("query_frame", _p), ("frame_wh", _p), ("n_frames", _i32),
                ("model", Keypoints), ("model_image", _p), ("image_centroid", _p), ("image_size", _p),
                ("image_group", _p), ("n_images", _i32), ("groups_per_frame", _i32)]


class HoughOut(C.Structure):
    _fields_ = [("pose", _p), ("base_bin", _p), ("near_edge", _p), ("counters", _p), ("bin_group", _p),
                ("bin_code", _p), ("bin_count", _p), ("bin_offset", _p), ("bin_order", _p),
                ("bin_mean", _p), ("members", _p), ("cap_bins", _i64), ("cap_votes", _i64)]


class AffineOut(C.Structure):
    _fields_ = [("counters", _p), ("valid_bin", _p), ("params", _p), ("votes", _p), ("status", _p),
                ("member_keep", _p), ("cap_valid", _i64), ("cap_votes", _i64)]


class PosesOut(C.Structure):
    _fields_ = [("counters", _p), ("cluster_bins", _p), ("cluster_offset", _p), ("sub_bins", _p), ("sub_first", _p),
                ("pose", _p), ("shape_bin", _p), ("segment", _p), ("cap", _i64)]


class SiftOut(C.Structure):
    _fields_ = [("xy", _p), ("size", _p), ("angle", _p), ("response", _p), ("octave", _p), ("des", _p),
                ("counters", _p), ("cap", _i64)]


class SiftBatchOut(C.Structure):
    _fields_ = [("xy", _p), ("size", _p), ("angle", _p), ("response", _p), ("octave", _p), ("des", _p),
                ("frame", _p), ("count", _p), ("offset", _p), ("overflow", _p), ("rows_overflow", _p),
                ("cap_rows", _i64), ("cap_per_frame", _i64)]


STAGES = {"match": 0, "hough_prep": 1, "hough_vote": 2, "hough_finish": 3, "affine": 4}


def timing_enable(on: bool = True) -> None:
    check(lib.sod_timing_enable(int(on)), "sod_timing_enable")


def timing_read(stage: str) -> list[float]:
    """Durations (ms) of the named stage's launches since the last read; waits for them."""
    buf = (C.c_float * 128)()
    n = int(lib.sod_timing_read(STAGES[stage], C.cast(buf, _p), 128))
    if n < 0:
        check(n, "sod_timing_read")
    return [float(buf[i]) for i in range(n)]


SIGMA_LUT_MIN = -24
SIGMA_LUT_LEN = 49
MAX_BINS = 15
MAX_CLUSTER_BINS = 65536

_PROTOS = {
    "sod_version": (C.c_int, []),
    "sod_last_error": (C.c_char_p, []),
    "sod_device_sm_count": (C.c_int, []),
    "sod_timing_enable": (C.c_int, [_i32]),
    "sod_timing_read": (_i32, [_i32, _p, _i32]),
    "sod_cq_ints": (_i64, [_i64]),
    "sod_pack_u8_from_f32": (C.c_int, [_p, _i64, _p, _p, _p]),
    "sod_db_prepare_workspace_bytes": (C.c_size_t, [_i64]),
    "sod_db_prepare": (C.c_int, [_p, _i64, _p, _p, _p, C.c_size_t, _p]),
    "sod_query_prepare": (C.c_int, [_p, _i64, _p, _p]),
    "sod_match_workspace_bytes": (C.c_size_t, [_i64, _i64]),
    "sod_match_top2": (C.c_int, [_p, _p, _i64, _p, _p, _i64, _i32, _p, _p, _p, C.c_size_t, _p]),
    "sod_row_thr_ints": (_i64, [_i64]),
    "sod_match_top2_range": (C.c_int, [_p, _p, _i64, _p, _p, _i64, _i32, _i64, _i64, _p, _p, _p, _p, C.c_size_t, _p]),
    "sod_match_top2_peer": (C.c_int, [_p, _p, _i64, _p, _p, _i64, _i32, _i64, _i64, _p, _p, _i32, _i64, _p, _p, _p,
                                      C.c_size_t, _p]),
    "sod_top2_merge": (C.c_int, [_p, _p, _i32, _i64, _p, _p, _p, _p, C.c_double, _p]),
    "sod_top2_keys": (C.c_int, [_p, _p, _i64, _i64, _p, _p]),
    "sod_top2_merge_keys": (C.c_int, [_p, _i32, _i64, _p, _p]),
    "sod_top2_from_keys": (C.c_int, [_p, _i64, _p, _p, _p, _p, C.c_double, _p]),
    "sod_exchange_bytes": (C.c_size_t, [_i64, _i32]),
    "sod_exchange_alloc": (C.c_int, [C.c_size_t, C.POINTER(_p)]),
    "sod_exchange_free": (C.c_int, [_p]),
    "sod_ipc_export": (C.c_int, [_p, _p]),
    "sod_ipc_open": (C.c_int, [_p, C.POINTER(_p)]),
    "sod_ipc_close": (C.c_int, [_p]),
    "sod_top2_exchange_peer": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _i64, _p, _p, _p, _p, C.c_double, _p]),
    "sod_bf16_operand_cols": (_i64, [_i32]),
    "sod_bf16_db_rows": (_i64, [_i64]),
    "sod_bf16_prepare": (C.c_int, [_p, _i64, _i32, _i32, _p, _p, _p, _p]),
    "sod_match_bf16_workspace_bytes": (C.c_size_t, [_i64, _i64]),
    "sod_match_top2_bf16": (C.c_int, [_p, _p, _i64, _p, _p, _i64, _i32, _i32, _p, _p, _p, C.c_size_t, _p]),
    "sod_top2_merge_f32": (C.c_int, [_p, _p, _i32, _i64, _p, _p, _p, _p, C.c_double, _p]),
    "sod_pose_adjacency": (C.c_int, [_p, _p, _p, _p, _p, _i64, _p, _p, _p]),
    "sod_angle_adjacency": (C.c_int, [_p, _p, _i64, C.c_double, _p, _p, _p]),
    "sod_final_poses_workspace_bytes": (C.c_size_t, [_i64]),
    "sod_final_poses": (C.c_int, [_p, _p, _i64, _p, C.POINTER(PosesOut), _p, C.c_size_t, _p]),
    "sod_final_poses_records": (C.c_int, [_p, _p, _p, _p, _i64, _p, _i32, C.POINTER(PosesOut), _p, C.c_size_t, _p]),
    "sod_compact_scratch_bytes": (C.c_size_t, [_i64]),
    "sod_compact_matches": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _p, _p, _p, _p]),
    "sod_compact_matches_dev": (C.c_int, [_p, _p, _i64, _p, _i32, _i32, _p, _p, _p, _p, _p]),
    "sod_estimate_pose": (C.c_int, [C.POINTER(Scene), _p, _p, _i64, _i32, _p, _p, _p, _p, _p]),
    "sod_pose_bin_index": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p]),
    "sod_affine_residual_keep": (C.c_int, [_p, _p, _i64, _p, C.c_double, C.c_double, _p, _p]),
    "sod_hough_workspace_bytes": (C.c_size_t, [_i64, _i64]),
    "sod_hough_vote": (C.c_int, [C.POINTER(Scene), _p, _p, _i64, _p, _i32, _p, _i32, C.POINTER(HoughOut), _p,
                                 C.c_size_t, _p]),
    "sod_hough_vote_dims": (C.c_int, [C.POINTER(Scene), _p, _p, _i64, _p, _i32, _i32, _i32, _i32, _p, _i32,
                                      C.POINTER(HoughOut), _p, C.c_size_t, _p]),
    "sod_valid_bin_records": (C.c_int, [C.POINTER(HoughOut), C.POINTER(AffineOut), _p, _p, _p, _p, _p]),
    "sod_affine_verify": (C.c_int, [C.POINTER(Scene), _p, _p, C.POINTER(HoughOut), _i32, _i32, _i32,
                                    C.c_double, C.c_double, _i32, C.POINTER(AffineOut), _p]),
    "sod_sift_workspace_bytes": (C.c_size_t, [_i32, _i32, _i64]),
    "sod_sift_extract": (C.c_int, [_p, _i32, _i32, _i64, C.POINTER(SiftOut), _p, C.c_size_t, _p]),
    "sod_sift_describe": (C.c_int, [_p, _i32, _i32, _i64, _p, _p, _p, _p, _i64, _p, _p, _p, C.c_size_t, _p]),
    "sod_sift_level_offset": (_i64, [_i32, _i32, _i32, _i32, _p]),
    "sod_sift_batch_workspace_bytes": (C.c_size_t, [_i32, _i32, _i32, _i64]),
    "sod_sift_extract_batch": (C.c_int, [_p, _i32, _i32, _i64, _i64, _i32, _i64, C.POINTER(SiftBatchOut), _p,
                                         C.c_size_t, _p]),
    "sod_sift_mixed_workspace_bytes": (C.c_size_t, [_p, _i32, _i64]),
    "sod_sift_extract_mixed": (C.c_int, [_p, _p, _p, _i32, _i64, C.POINTER(SiftBatchOut), _p, C.c_size_t, _p]),
}

SIFT_MAX_MIXED_FRAMES = 64


def _bind() -> None:
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)  # AttributeError here = header and library disagree
        fn.restype = res
        fn.argtypes = args


_bind()

EXPORTED = tuple(_PROTOS)


def check(rc: int, what: str) -> None:
    if rc != SOD_OK:
        msg = lib.sod_last_error().decode("utf-8", "replace")
        raise SodError(f"{what} failed ({rc}): {msg}")
