"""CPU: FM_FLAG_GRAY in the binding and the refusal of FM_FLAG_GRAY | FM_FLAG_NV12, which fm_ctx_create makes before any
device query (so it needs no GPU)."""
import ctypes as C

import pytest


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
    assert _lib.FLAG_GRAY == 2048
    flags = [v for k, v in vars(_lib).items() if k.startswith("FLAG_")]
    assert len(set(flags)) == len(flags) and all(v & (v - 1) == 0 for v in flags)


@pytest.mark.parametrize("W,H", [(640, 480), (333, 217), (1920, 1080)])
def test_gray_with_nv12_refused_before_device_query(lib, W, H):
    from find_motion_b200 import _lib
    ctx = C.c_void_p()
    cfg = _cfg(_lib.FLAG_GRAY | _lib.FLAG_NV12, W, H)
    assert lib.fm_ctx_create(C.byref(cfg), C.byref(ctx)) == -1           # FM_EINVAL, not FM_ECUDA
    assert b"FM_FLAG_GRAY" in lib.fm_last_error() and not ctx.value


def test_engine_refuses_gray_with_nv12(lib):
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    with pytest.raises(_lib.FmError) as e:
        MotionEngine(640, 480, gray=True, nv12=True)
    assert e.value.code == -1


def _plan(lib, W, H, box, channels):
    from find_motion_b200 import _lib
    info = _lib.fm_rows_plan_info()
    _lib.check(lib.fm_debug_rows_plan_channels(W, H, box, channels, C.byref(info)))
    return {f: getattr(info, f) for f, _ in info._fields_}


def test_rows_plan_channels_entry(lib):
    from find_motion_b200 import _lib
    info = _lib.fm_rows_plan_info()
    for ch in (0, 2, 4):
        assert lib.fm_debug_rows_plan_channels(1920, 1080, 100, ch, C.byref(info)) == -1
    b = _lib.fm_rows_plan_info()
    _lib.check(lib.fm_debug_rows_plan(1920, 1080, 100, C.byref(b)))
    assert _plan(lib, 1920, 1080, 100, 3) == {f: getattr(b, f) for f, _ in b._fields_}
    assert _plan(lib, 1920, 1080, 100, 1)["usable"] == 1         # the reference's default regime on gray frames


@pytest.mark.parametrize("W,H", __import__("tests.test_rows_plan", fromlist=["SIZES"]).SIZES)
def test_gray_rows_plan_invariants(lib, W, H):
    """The one-channel plan of the row-per-lane resize kernel over tests/test_rows_plan.py's geometries (and the detector
    input width 300): the library re-checks every tap of every column against cv2's table and its TMA box (FM_ERANGE
    otherwise); here the plan's shape is checked against the oracle's tables."""
    from oracle import restated as R
    from tests.test_rows_plan import BOXES
    for box in BOXES:
        if box > W:
            continue
        p = _plan(lib, W, H, box, 1)
        w, h = box, int(H * (box / float(W)))
        if h < 1:
            continue
        xt, yt = R.area_tab(W, w), R.area_tab(H, h)
        taps = max(len(t) for t in xt)
        if not p["usable"]:
            sx, sy = W / w, H / h
            integer = abs(sx - round(sx)) < 1e-12 and abs(sy - round(sy)) < 1e-12
            assert W % 16 != 0 or integer or taps < 4 or w == W, (W, H, box, p)
            continue
        assert W % 16 == 0
        assert 1 <= p["box_rows"] <= 160 and p["band_rows"] >= 1
        assert p["box_bytes"] % 16 == 0 and (p["box_bytes"] // 16) % 2 == 1 and p["box_bytes"] <= 1024
        assert p["smem_bytes"] <= 200 * 1024
        assert p["chunk_cols"] in (1, 2) and p["seg_cols"] % p["chunk_cols"] == 0
        assert p["bands"] == -(-h // p["band_rows"]) and p["segs"] == -(-w // p["seg_cols"])
        assert p["max_groups"] == -(-taps // 4)
        rows = max(yt[min(d0 + p["band_rows"], h) - 1][-1][0] - yt[d0][0][0] + 1 for d0 in range(0, h, p["band_rows"]))
        assert rows == p["box_rows"]
        bgr = _plan(lib, W, H, box, 3)
        if bgr["usable"]:                   # one byte per pixel: never a wider box than BGR's
            assert p["box_bytes"] <= bgr["box_bytes"] and p["band_rows"] == bgr["band_rows"]
