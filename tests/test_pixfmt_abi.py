"""CPU: FM_FLAG_RGB and FM_FLAG_ALPHA in the binding, their refusal together with the other frame formats (fm_ctx_create
makes it before any device query, so it needs no GPU), and fm_debug_rows_plan_format, the rows plan fm_ctx_create builds for each format."""
import ctypes as C

import pytest

from tests.test_rows_plan import BOXES, SIZES


@pytest.fixture(scope="module")
def lib():
    from find_motion_b200 import build, _lib
    build.build()
    return _lib.load()


def _cfg(flags, W=640, H=480):
    from find_motion_b200 import _lib
    return _lib.fm_config(device=0, n_streams=1, frame_width=W, frame_height=H, max_frames=8, fps=30, box_size=100,
                          min_box_scale=50, blur_scale=20, threshold=7, avg=0.1, min_time=0.5, cache_time=2.0,
                          max_components=0, flags=flags)


def test_flag_value():
    from find_motion_b200 import _lib
    assert _lib.FLAG_RGB == 4096 and _lib.FLAG_ALPHA == 8192
    assert "fm_debug_rows_plan_format" in _lib.SYMBOLS


@pytest.mark.parametrize("fmt", ["RGB", "ALPHA"])
@pytest.mark.parametrize("other", ["NV12", "GRAY"])
@pytest.mark.parametrize("W,H", [(640, 480), (333, 217), (1920, 1080)])
def test_format_with_other_format_refused_before_device_query(lib, fmt, other, W, H):
    from find_motion_b200 import _lib
    ctx = C.c_void_p()
    cfg = _cfg(getattr(_lib, "FLAG_" + fmt) | getattr(_lib, "FLAG_" + other), W, H)
    assert lib.fm_ctx_create(C.byref(cfg), C.byref(ctx)) == -1           # FM_EINVAL, not FM_ECUDA
    err = lib.fm_last_error()
    assert b"FM_FLAG_" + fmt.encode() in err and b"FM_FLAG_" + other.encode() in err and not ctx.value


@pytest.mark.parametrize("fmt", [dict(rgb=True), dict(alpha=True), dict(rgb=True, alpha=True)])
@pytest.mark.parametrize("kw", [dict(nv12=True), dict(gray=True)])
def test_engine_refuses_format_with_other_format(lib, fmt, kw):
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    with pytest.raises(_lib.FmError) as e:
        MotionEngine(640, 480, **fmt, **kw)
    assert e.value.code == -1


def _info(info):
    return {f: getattr(info, f) for f, _ in info._fields_}


def _plan_format(lib, W, H, box, flags):
    from find_motion_b200 import _lib
    info = _lib.fm_rows_plan_info()
    _lib.check(lib.fm_debug_rows_plan_format(W, H, box, flags, C.byref(info)))
    return _info(info)


def test_rows_plan_format_refusals(lib):
    from find_motion_b200 import _lib
    info = _lib.fm_rows_plan_info()
    for flags in (_lib.FLAG_NV12, _lib.FLAG_RGB | _lib.FLAG_GRAY, _lib.FLAG_RGB | _lib.FLAG_NV12, _lib.FLAG_ALPHA | _lib.FLAG_GRAY,
                  _lib.FLAG_ALPHA | _lib.FLAG_NV12, _lib.FLAG_UPSCALE, 16384):
        assert lib.fm_debug_rows_plan_format(1920, 1080, 100, flags, C.byref(info)) == -1, flags
    assert lib.fm_debug_rows_plan_format(0, 1080, 100, 0, C.byref(info)) == -1


@pytest.mark.parametrize("W,H", SIZES)
def test_rows_plan_format_matches_channel_plans(lib, W, H):
    """0 and RGB select the three-byte plan of fm_debug_rows_plan (the order moves only the gray weights), GRAY the
    one-byte plan of fm_debug_rows_plan_channels(..., 1, ...); the library self-checks each tap by tap."""
    from find_motion_b200 import _lib
    for box in BOXES:
        if box > W:
            continue
        bgr, gray = _lib.fm_rows_plan_info(), _lib.fm_rows_plan_info()
        _lib.check(lib.fm_debug_rows_plan(W, H, box, C.byref(bgr)))
        _lib.check(lib.fm_debug_rows_plan_channels(W, H, box, 1, C.byref(gray)))
        assert _plan_format(lib, W, H, box, 0) == _info(bgr), (W, H, box)
        assert _plan_format(lib, W, H, box, _lib.FLAG_RGB) == _info(bgr), (W, H, box)
        assert _plan_format(lib, W, H, box, _lib.FLAG_GRAY) == _info(gray), (W, H, box)


@pytest.mark.parametrize("W,H", SIZES)
def test_four_byte_rows_plan_invariants(lib, W, H):
    """The four-byte plan (ALPHA, RGB | ALPHA: the same plan) over tests/test_rows_plan.py's geometries: the library
    re-checks every tap of every column against cv2's table and its TMA box (FM_ERANGE otherwise); here the plan's shape is
    checked against the oracle's tables and the kernel's limits."""
    from find_motion_b200 import _lib
    from oracle import restated as R
    for box in BOXES:
        if box > W:
            continue
        p = _plan_format(lib, W, H, box, _lib.FLAG_ALPHA)
        assert _plan_format(lib, W, H, box, _lib.FLAG_ALPHA | _lib.FLAG_RGB) == p
        w, h = box, int(H * (box / float(W)))
        if h < 1:
            continue
        xt, yt = R.area_tab(W, w), R.area_tab(H, h)
        taps = max(len(t) for t in xt)
        bgr = _plan_format(lib, W, H, box, 0)
        if not p["usable"]:
            sx, sy = W / w, H / h
            integer = abs(sx - round(sx)) < 1e-12 and abs(sy - round(sy)) < 1e-12
            # beyond the BGR plan's reasons: a box row of four-byte pixels wider than TMA's 256 words
            assert W % 4 != 0 or integer or taps < 4 or w == W or not bgr["usable"] or \
                bgr["box_bytes"] * 4 // 3 > 1024 - 64, (W, H, box, p, bgr)
            continue
        assert 1 <= p["box_rows"] <= 160 and p["band_rows"] >= 1
        assert p["box_bytes"] % 16 == 0 and (p["box_bytes"] // 16) % 2 == 1 and p["box_bytes"] <= 1024
        assert p["smem_bytes"] <= 200 * 1024
        assert p["chunk_cols"] in (1, 2) and p["seg_cols"] % p["chunk_cols"] == 0
        assert p["bands"] == -(-h // p["band_rows"]) and p["segs"] == -(-w // p["seg_cols"])
        assert p["max_groups"] == -(-taps // 4)
        rows = max(yt[min(d0 + p["band_rows"], h) - 1][-1][0] - yt[d0][0][0] + 1 for d0 in range(0, h, p["band_rows"]))
        assert rows == p["box_rows"]
        assert p["box_bytes"] >= 4 * taps    # a box row holds every tap of a column, four bytes each
        if bgr["usable"]:                   # the bands depend on the rows only
            assert p["band_rows"] == bgr["band_rows"] and p["box_rows"] == bgr["box_rows"]
