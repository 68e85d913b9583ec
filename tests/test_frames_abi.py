"""CPU: the fm_frames layout of include/fm_gpu.h, its binding, and fm_process_frames' argument checks that come before any
device work."""
import ctypes as C

import pytest


@pytest.fixture(scope="module")
def lib():
    from find_motion_b200 import build, _lib
    build.build()
    return _lib.load()


def test_fm_frames_layout():
    from find_motion_b200 import _lib
    F = _lib.fm_frames
    assert C.sizeof(F) == 40
    assert [(n, getattr(F, n).offset) for n, _ in F._fields_] == [
        ("data", 0), ("stream_stride", 8), ("frame_stride", 16), ("row_pitch", 24), ("uv_offset", 32)]


def test_symbol_exported_and_bound(lib):
    from find_motion_b200 import _lib
    assert "fm_process_frames" in _lib.SYMBOLS
    assert hasattr(lib, "fm_process_frames")


def test_null_arguments_refused(lib):
    from find_motion_b200 import _lib
    fr = _lib.fm_frames(0x1000, 0, 0, 0, 0)
    assert lib.fm_process_frames(None, C.byref(fr), 1, None, None, None, None, 0, 0) == -1
    assert b"null" in lib.fm_last_error()
    # the frames are checked before the context is read: a context handle that is never dereferenced
    dummy = C.create_string_buffer(64)
    assert lib.fm_process_frames(C.addressof(dummy), None, 1, None, None, None, None, 0, 0) == -1
    assert b"null" in lib.fm_last_error()
    no_data = _lib.fm_frames(0, 0, 0, 0, 0)
    assert lib.fm_process_frames(C.addressof(dummy), C.byref(no_data), 1, None, None, None, None, 0, 0) == -1
