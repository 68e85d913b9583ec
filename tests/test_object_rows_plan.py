"""CPU: the rows-kernel plan of the detector input planes (FM_FLAG_OBJECT_PLANES, W x H -> 300 x oh) is usable for the
usual camera geometries and passes its own tap-by-tap checks (fm_debug_rows_plan needs no device)."""
import ctypes as C

import pytest

from find_motion_b200 import _lib


@pytest.mark.parametrize("W,H", [(1920, 1080), (1280, 720), (3840, 2160)])
def test_object_rows_plan_usable(W, H):
    info = _lib.fm_rows_plan_info()
    _lib.check(_lib.load().fm_debug_rows_plan(W, H, _lib.OBJECT_WIDTH, C.byref(info)))   # FM_ERANGE if a tap check fails
    assert info.usable == 1
    assert info.bands * info.band_rows >= int(H * (_lib.OBJECT_WIDTH / float(W)))
    assert info.segs * info.seg_cols >= _lib.OBJECT_WIDTH
