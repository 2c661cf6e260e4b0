"""CPU-side checks of the SIFT entry points: sizes, pyramid layout and argument errors, before any CUDA call."""
import ctypes as C

import pytest


def test_workspace_bytes_and_level_offsets():
    from sod_b200._capi import lib
    assert lib.sod_sift_workspace_bytes(0, 10, 0) == 0
    assert lib.sod_sift_workspace_bytes(10, 32769, 0) == 0
    assert lib.sod_sift_workspace_bytes(10, 10, -1) == 0
    assert lib.sod_sift_workspace_bytes(10, 10, (1 << 24) + 1) == 0
    # 1200x900: 10 octaves (cv2 octaves -1..8), six 2400x1800 f32 levels first
    wh = (C.c_int32 * 2)()
    assert lib.sod_sift_level_offset(1200, 900, -1, 0, C.cast(wh, C.c_void_p)) == 0 and tuple(wh) == (2400, 1800)
    assert lib.sod_sift_level_offset(1200, 900, -1, 5, None) == 5 * 2400 * 1800 * 4
    assert lib.sod_sift_level_offset(1200, 900, 0, 0, C.cast(wh, C.c_void_p)) == 6 * 2400 * 1800 * 4
    assert tuple(wh) == (1200, 900)
    assert lib.sod_sift_level_offset(641, 479, 1, 0, C.cast(wh, C.c_void_p)) > 0 and tuple(wh) == (320, 239)
    assert lib.sod_sift_level_offset(1200, 900, 8, 0, None) > 0
    assert lib.sod_sift_level_offset(1200, 900, 9, 0, None) == -1 and b"octave 9" in lib.sod_last_error()
    assert lib.sod_sift_level_offset(1200, 900, 0, 6, None) == -1
    pyramid = lib.sod_sift_workspace_bytes(1200, 900, 0)
    assert 6 * 2400 * 1800 * 4 * 1.33 <= pyramid <= 6 * 2400 * 1800 * 4 * 4 / 3 + 4096
    assert lib.sod_sift_workspace_bytes(1200, 900, 1000) > pyramid + 1000 * (36 + 24 + 8 * 4)


def test_extract_and_describe_reject_bad_arguments_without_gpu():
    from sod_b200._capi import SiftOut, lib
    fake = 1 << 20                         # never dereferenced: validation fails first
    assert lib.sod_sift_extract(None, 10, 10, 10, None, None, 0, None) == -1 and b"null image" in lib.sod_last_error()
    assert lib.sod_sift_extract(fake, 10, 10, 9, None, None, 0, None) == -1 and b"pitch" in lib.sod_last_error()
    assert lib.sod_sift_extract(fake, 0, 10, 10, None, None, 0, None) == -1 and b"out of range" in lib.sod_last_error()
    assert lib.sod_sift_extract(fake, 10, 10, 10, None, None, 0, None) == -1 and b"null out" in lib.sod_last_error()
    out = SiftOut(fake, fake, fake, fake, fake, fake, fake, 0)
    assert lib.sod_sift_extract(fake, 10, 10, 10, C.byref(out), None, 0, None) == -1
    assert b"cap" in lib.sod_last_error()
    out = SiftOut(fake, fake, fake, None, fake, fake, fake, 100)
    assert lib.sod_sift_extract(fake, 10, 10, 10, C.byref(out), None, 0, None) == -1
    assert b"null output" in lib.sod_last_error()
    out = SiftOut(fake, fake, fake, fake, fake, fake, fake, 100)
    need = lib.sod_sift_workspace_bytes(10, 10, 100)
    assert lib.sod_sift_extract(fake, 10, 10, 10, C.byref(out), fake, need - 1, None) == -1
    assert b"workspace" in lib.sod_last_error()
    assert lib.sod_sift_extract(fake, 10, 10, 10, C.byref(out), fake + 16, need, None) == -1   # misaligned
    assert lib.sod_sift_describe(fake, 10, 10, 10, None, None, None, None, 0, None, None, None, 0, None) == 0
    assert lib.sod_sift_describe(fake, 10, 10, 10, None, None, None, None, 3, None, None, None, 0, None) == -1
    assert b"null keypoint" in lib.sod_last_error()
    assert lib.sod_sift_describe(fake, 10, 10, 10, fake, fake, fake, fake, -1, fake, None, fake, 0, None) == -1
    assert lib.sod_sift_describe(fake, 10, 10, 10, fake, fake, fake, fake, 3, fake, None, fake, 0, None) == -1
    assert b"workspace" in lib.sod_last_error()


def test_gpu_sift_rejects_a_bad_capacity():
    from sod_b200.sift import GpuSift
    with pytest.raises(ValueError):
        GpuSift(capacity=0)
