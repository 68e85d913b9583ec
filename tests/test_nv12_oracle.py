"""CPU: the restatement of NV12 -> BGR (tests/nv12_restated.py) against cv2.cvtColor(COLOR_YUV2BGR_NV12) for every
(Y, U, V) triple and on random frames, and the range check of FM_FLAG_NV12 in fm_ctx_create, which comes before any
device query."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from tests import nv12_restated as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_every_yuv_triple_matches_cv2():
    cv2 = pytest.importorskip("cv2")
    nv = N.exhaustive_planes()
    H = nv.shape[0] * 2 // 3
    Y = nv[:H].astype(np.int64)
    UV = nv[H:].reshape(H // 2, -1, 2).astype(np.int64)
    keys = (Y << 16) | np.repeat(np.repeat((UV[..., 0] << 8) | UV[..., 1], 2, 0), 2, 1)
    assert np.unique(keys).size == 1 << 24                      # the frame does hold every triple
    want = cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12)
    got = N.bgr_from_nv12(nv)
    assert (got == want).all(), int((got != want).any(-1).sum())


# widths that are not multiples of 16 (nor of 8, 4 where possible); tests/test_gpu_nv12.py runs such widths on the GPU
@pytest.mark.parametrize("W,H", [(2, 2), (6, 4), (18, 10), (100, 76), (642, 362), (1000, 562), (1366, 768), (64, 48),
                                 (1920, 1080)])
def test_random_frames_match_cv2(W, H):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(W * 131 + H)
    nv = rng.integers(0, 256, size=(H * 3 // 2, W), dtype=np.uint8)
    assert (N.bgr_from_nv12(nv) == cv2.cvtColor(nv, cv2.COLOR_YUV2BGR_NV12)).all()


def test_synthetic_decoder_output_round_trips_through_cv2():
    """nv12_from_bgr (the GPU tests' decoder stand-in) is the I420 of cv2 with interleaved chroma."""
    cv2 = pytest.importorskip("cv2")
    from find_motion_b200 import synth
    for W, H in ((96, 64), (1000, 562)):           # H/2 odd: the chroma planes do not end on a row of W bytes
        clip = synth.make_clip(W, H, 2, seed=5)
        nv = N.nv12_from_bgr(clip)
        assert nv.shape == (2, H * 3 // 2, W)
        for f, n in zip(clip, nv):
            i420 = cv2.cvtColor(f, cv2.COLOR_BGR2YUV_I420)
            assert (cv2.cvtColor(i420, cv2.COLOR_YUV2BGR_I420) == N.bgr_from_nv12(n)).all()


def test_flag_constant():
    from find_motion_b200 import _lib
    with open(os.path.join(ROOT, "include", "fm_gpu.h")) as f:
        m = re.search(r"#define\s+FM_FLAG_NV12\s+(\d+)", f.read())
    assert m and int(m.group(1)) == _lib.FLAG_NV12 == 512


@pytest.mark.parametrize("W,H", [(641, 480), (640, 481), (1, 2), (1919, 1079)])
def test_odd_geometry_is_refused_before_any_device_query(W, H):
    from find_motion_b200 import build, _lib
    build.build()
    lib = _lib.load()
    cfg = _lib.fm_config(device=0, n_streams=1, frame_width=W, frame_height=H, max_frames=4, fps=30, box_size=1,
                         min_box_scale=50, blur_scale=20, threshold=7, avg=0.1, min_time=0.5, cache_time=1.0,
                         max_components=0, flags=_lib.FLAG_NV12)
    ctx = C.c_void_p()
    assert lib.fm_ctx_create(C.byref(cfg), C.byref(ctx)) == -4          # FM_ERANGE, with or without a device
    assert not ctx.value
    assert b"even" in lib.fm_last_error()


def test_grid_limits_are_refused_before_any_device_query():
    from find_motion_b200 import build, _lib
    build.build()
    lib = _lib.load()
    for S, T in ((65536, 1), (1, 65536)):
        cfg = _lib.fm_config(device=0, n_streams=S, frame_width=64, frame_height=48, max_frames=T, fps=30, box_size=64,
                             min_box_scale=50, blur_scale=20, threshold=7, avg=0.1, min_time=0.5, cache_time=1.0,
                             max_components=0, flags=_lib.FLAG_NV12)
        ctx = C.c_void_p()
        assert lib.fm_ctx_create(C.byref(cfg), C.byref(ctx)) == -4, (S, T)
        assert not ctx.value
