"""CPU: the premise of FM_FLAG_GRAY's exactness on the pinned cv2.  A gray context on frame G must give what a BGR context
gives on cv2.cvtColor(G, COLOR_GRAY2BGR); that holds because
  * BGR2GRAY(GRAY2BGR(G)) == G (cv2's fixed-point weights sum to 2^15), and
  * INTER_AREA resizes each channel alone: cv2.resize of the three equal channels equals the one-channel cv2.resize of G
    in every channel, at every geometry tests/test_gpu_gray.py runs (decimation by tables, integer ratios, odd sizes,
    upscales), and for the detector input planes (width 300)."""
import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")


def test_gray_round_trip_every_value():
    g = np.arange(256, dtype=np.uint8).reshape(16, 16)
    assert (cv2.cvtColor(cv2.cvtColor(g, cv2.COLOR_GRAY2BGR), cv2.COLOR_BGR2GRAY) == g).all()


# (W, H, box_size): the processing planes of tests/test_gpu_gray.py, and the widths of their detector input planes
GEOMETRIES = [(1920, 1080, 100), (640, 480, 100), (640, 480, 320), (80, 60, 100), (333, 217, 111), (1000, 562, 100),
              (1920, 1080, 300), (640, 480, 300), (80, 60, 300), (333, 217, 300), (1280, 720, 300), (100, 76, 160)]


@pytest.mark.parametrize("W,H,box", GEOMETRIES)
def test_inter_area_per_channel_equals_one_channel(W, H, box):
    rng = np.random.default_rng(W * 7 + H * 3 + box)
    h = int(H * (box / float(W)))                                      # imutils.resize
    for g in (rng.integers(0, 256, size=(H, W), dtype=np.uint8),
              cv2.cvtColor(rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8), cv2.COLOR_BGR2GRAY)):
        one = cv2.resize(g, (box, h), interpolation=cv2.INTER_AREA)
        three = cv2.resize(cv2.cvtColor(g, cv2.COLOR_GRAY2BGR), (box, h), interpolation=cv2.INTER_AREA)
        for ch in range(3):
            assert (three[..., ch] == one).all(), (W, H, box, ch)
        assert (cv2.cvtColor(three, cv2.COLOR_BGR2GRAY) == one).all()
