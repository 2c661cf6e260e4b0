"""CPU-side checks of the final-pose entry points: every argument error is reported before any CUDA call, and an
empty input does nothing."""
import ctypes as C

FAKE = 1 << 20                 # never dereferenced: validation fails first


def _out(cap=100, **null):
    from sod_b200._capi import PosesOut
    fields = [name for name, _ in PosesOut._fields_ if name != "cap"]
    return PosesOut(*(None if name in null else FAKE for name in fields), cap)


def test_final_poses_rejects_bad_arguments_without_gpu():
    from sod_b200._capi import PosesOut, lib
    f = lib.sod_final_poses
    ws = lib.sod_final_poses_workspace_bytes(100)
    assert ws > 100 * 4 * 4 and lib.sod_final_poses_workspace_bytes(65537) == 0
    assert lib.sod_final_poses_workspace_bytes(-1) == 0
    assert lib.sod_final_poses_workspace_bytes(65536) >= 65536 * 2048 * 4       # the bit rows of one 65,536-bin segment

    def err(mean=FAKE, seg=None, n=100, n_dev=None, out=None, work=FAKE, work_bytes=ws):
        o = _out() if out is None else out
        assert f(mean, seg, n, n_dev, C.byref(o), work, work_bytes, None) == -1
        return lib.sod_last_error()

    assert b"65536" in err(n=65537)
    assert b"65536" in err(n=-1)
    assert b"null pointer" in err(mean=None)
    assert b"null pointer" in err(work=None)
    assert f(FAKE, None, 100, None, None, FAKE, ws, None) == -1 and b"null pointer: out" in lib.sod_last_error()
    for name, _ in PosesOut._fields_[:-1]:
        assert b"null pointer in out" in err(out=_out(**{name: True})), name
    assert b"out->cap 99 < 100" in err(out=_out(cap=99))
    assert b"workspace too small" in err(work_bytes=ws - 1)
    assert f(None, None, 0, None, None, None, 0, None) == 0                     # n = 0: nothing to do


def test_final_poses_records_rejects_bad_arguments_without_gpu():
    from sod_b200._capi import lib
    f = lib.sod_final_poses_records
    ws = lib.sod_final_poses_workspace_bytes(64)
    names = ("status", "group", "order", "mean", "cap", "n_dev", "gpf", "out", "work", "work_bytes", "stream")

    def call(**kw):
        a = dict(zip(names, (FAKE, FAKE, FAKE, FAKE, 64, FAKE, 3, None, FAKE, ws, None)), **kw)
        o = a["out"] if a["out"] is not None else _out(cap=64)
        return f(*(C.byref(o) if n == "out" else a[n] for n in names))

    def err(**kw):
        assert call(**kw) == -1
        return lib.sod_last_error()

    assert b"65536" in err(cap=65537)
    assert b"groups_per_frame" in err(gpf=0)
    assert b"groups_per_frame" in err(gpf=0, cap=0)                             # checked before the empty no-op
    for name in ("status", "group", "order", "mean", "n_dev", "work"):
        assert b"null pointer" in err(**{name: None}), name
    assert b"null pointer in out" in err(out=_out(cap=64, pose=True))
    assert b"out->cap 63 < 64" in err(out=_out(cap=63))
    assert b"workspace too small" in err(work_bytes=ws - 1)
    assert call(cap=0, status=None, group=None, order=None, mean=None, n_dev=None, work=None) == 0
