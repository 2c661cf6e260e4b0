"""CPU-side checks of the boundary: the library builds, loads without a GPU, exports exactly the
functions include/sod.h declares, and argument errors are reported through status codes."""
import re
import subprocess
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _header_functions():
    text = (ROOT / "include" / "sod.h").read_text()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(sod_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from sod_b200 import _capi
    declared = _header_functions()
    assert len(declared) >= 15
    out = subprocess.run(["nm", "-D", "--defined-only", str(_capi._LIB_PATH)], capture_output=True, text=True).stdout
    exported = sorted(set(re.findall(r" T (sod_[a-z0-9_]+)", out)))
    assert exported == declared
    assert sorted(_capi.EXPORTED) == declared          # the ctypes binding covers all of them


def test_library_has_blackwell_code_only():
    from sod_b200 import _capi
    out = subprocess.run(["cuobjdump", "-lelf", str(_capi._LIB_PATH)], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_error_reporting_without_gpu():
    from sod_b200 import _capi
    lib = _capi.lib
    assert lib.sod_version() >= 1000
    assert lib.sod_cq_ints(0) == 0 and lib.sod_cq_ints(1) == 260 and lib.sod_cq_ints(129) == 520
    rc = lib.sod_db_prepare(None, -1, None, None, None, 0, None)
    assert rc == -1 and b"n_rows" in lib.sod_last_error()
    rc = lib.sod_top2_merge(None, None, 1, 10, None, None, None, None, 0.75, None)
    assert rc == -1 and b"null" in lib.sod_last_error()
    assert lib.sod_compact_scratch_bytes(5000) >= 8 * 6


def test_argument_checks_of_the_newer_entry_points_without_gpu():
    """Argument validation happens before any CUDA call, so it is testable on the CPU."""
    from sod_b200 import _capi
    lib = _capi.lib
    assert lib.sod_bf16_operand_cols(0) == 128 and lib.sod_bf16_operand_cols(1) == 384
    assert lib.sod_bf16_db_rows(0) == 0 and lib.sod_bf16_db_rows(1) == 128 and lib.sod_bf16_db_rows(129) == 256
    assert lib.sod_bf16_prepare(None, 4, 2, 1, None, None, None, None) == -1 and b"side" in lib.sod_last_error()
    assert lib.sod_bf16_prepare(None, 4, 0, 1, None, None, None, None) == -1 and b"null" in lib.sod_last_error()
    assert lib.sod_bf16_prepare(None, 0, 0, 1, None, None, None, None) == 0          # nothing to do
    assert lib.sod_match_top2_bf16(None, None, -1, None, None, 0, 1, 0, None, None, None, 0, None) == -1
    assert lib.sod_match_top2(None, None, 3, None, None, 2 ** 31, 0, None, None, None, 0, None) == -1
    assert b"out of range" in lib.sod_last_error()
    assert lib.sod_match_top2(None, None, 3, None, None, 5, 2 ** 31 - 3, None, None, None, 0, None) == -1
    assert b"overflows" in lib.sod_last_error()
    assert lib.sod_top2_merge_f32(None, None, 2, 10, None, None, None, None, 0.75, None) == -1
    assert lib.sod_pose_adjacency(None, None, None, None, None, 65537, None, None, None) == -1
    assert b"65536" in lib.sod_last_error()
    assert lib.sod_angle_adjacency(None, None, 10, 1.0, None, None, None) == -1 and b"null" in lib.sod_last_error()
    assert lib.sod_pose_adjacency(None, None, None, None, None, 0, None, None, None) == 0


def test_key_exchange_entry_points_check_their_arguments_without_gpu():
    from sod_b200 import _capi
    lib = _capi.lib
    assert lib.sod_top2_keys(None, None, 5, 4, None, None) == -1 and b"n_rows" in lib.sod_last_error()
    assert lib.sod_top2_keys(None, None, 0, 0, None, None) == 0                       # nothing to do
    assert lib.sod_top2_keys(None, None, 0, 8, None, None) == -1 and b"null" in lib.sod_last_error()
    assert lib.sod_top2_keys(None, None, 0, 8, 24, None) == -1 and b"aligned" in lib.sod_last_error()
    assert lib.sod_top2_merge_keys(None, -1, 4, None, None) == -1
    assert lib.sod_top2_merge_keys(None, 2, 4, 16, None) == -1 and b"null" in lib.sod_last_error()
    assert lib.sod_top2_merge_keys(None, 2, 0, None, None) == 0
    assert lib.sod_top2_from_keys(None, 4, None, None, None, None, 0.75, None) == -1
    assert lib.sod_row_thr_ints(0) == 0 and lib.sod_row_thr_ints(1) == 256 and lib.sod_row_thr_ints(257) == 512


def test_ctypes_prototypes_have_the_arity_of_the_header():
    """Every prototype bound in _capi.py takes as many arguments as include/sod.h declares."""
    from sod_b200 import _capi
    text = re.sub(r"/\*.*?\*/", "", (ROOT / "include" / "sod.h").read_text(), flags=re.S)
    for name, params in re.findall(r"\b(sod_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        params = params.strip()
        n = 0 if params in ("", "void") else params.count(",") + 1
        assert len(_capi._PROTOS[name][1]) == n, name


def test_product_does_not_import_the_oracle():
    pkg = ROOT / "sift-based-od_b200"
    for f in list(pkg.rglob("*.py")) + list(pkg.rglob("*.cu")) + list(pkg.rglob("*.cuh")):
        text = f.read_text()
        assert "oracle" not in text.lower() or f.name == "build.py", f"{f} mentions the oracle"


def test_graft_entry_build():
    import __graft_entry__ as g
    g.build()


def test_exchange_argument_checks():
    """Entry points added in round 2 reject bad arguments before touching the device (no GPU needed)."""
    import ctypes as C
    from sod_b200._capi import lib
    assert lib.sod_exchange_bytes(1000, 0) == 0 and lib.sod_exchange_bytes(1000, 17) == 0
    assert lib.sod_exchange_bytes(1000, 8) == 512 + 2 * 8 * 1000 * 16
    table = (C.c_void_p * 2)(0, 0)
    assert lib.sod_top2_exchange_peer(None, None, 10, 2, 2, C.cast(table, C.c_void_p), 100, None, None, None, None,
                                      0.75, None) == -1                       # rank out of range
    assert lib.sod_top2_exchange_peer(None, None, 101, 0, 2, C.cast(table, C.c_void_p), 100, None, None, None, None,
                                      0.75, None) == -1 and b"capacity" in lib.sod_last_error()
    assert lib.sod_top2_exchange_peer(None, None, 0, 0, 2, C.cast(table, C.c_void_p), 100, None, None, None, None,
                                      0.75, None) == 0                        # empty batch: nothing to do
    assert lib.sod_timing_read(99, None, 0) == -1
    assert lib.sod_exchange_alloc(16, None) == -1
