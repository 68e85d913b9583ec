"""TEST INFRASTRUCTURE ONLY -- CPU restatement of cv2.resize(INTER_AREA) with a destination larger than the source,
what imutils.resize does to a frame narrower than box_size (find_motion.py:492).  There cv2 switches to its
fixed-point linear interpolation with area-style offsets (cv::resize, `area_mode`; SURVEY.md A.1).  Checked against
cv2 byte for byte by tests/test_upscale_oracle.py.

oracle/restated.resize_area covers downscale and identity; `resize_area` here adds the upscale and defers to it
otherwise.  `use_in_oracle(monkeypatch)` makes oracle.restated.StreamOracle (and everything built on it) take it.
"""
from __future__ import annotations

import math

import numpy as np

from oracle import restated as R

_BASE_RESIZE = R.resize_area


def upscale_tab(src: int, dst: int):
    """One axis, dst >= src: per destination index the first source index and the two 11-bit weights (a0, a1)."""
    inv = dst / src                    # double inv_scale, as cv2
    scale = 1.0 / inv
    one = np.float32(1.0)
    coef = np.float32(2048.0)          # INTER_RESIZE_COEF_SCALE
    sx = np.empty(dst, np.int64)
    a = np.empty((dst, 2), np.int64)
    for d in range(dst):
        s = math.floor(d * scale)
        fx = np.float32((d + 1) - (s + 1) * inv)          # double expression, cast to float
        fx = np.float32(0.0) if fx <= 0 else np.float32(fx - np.float32(math.floor(fx)))
        if s >= src - 1:                                   # right / bottom border
            fx, s = np.float32(0.0), src - 1
        sx[d] = s
        a[d, 0] = int(np.rint(np.float32(one - fx) * coef))     # saturate_cast<short>: round half to even
        a[d, 1] = int(np.rint(np.float32(fx * coef)))
    return sx, a


def resize_upscale(img: np.ndarray, w: int, h: int) -> np.ndarray:
    """cv2.resize(img, (w, h), INTER_AREA) for w >= W, h >= H: horizontal taps in int32, then the vertical combine
    in the form cv2's VResizeLinear uses for u8 on every column (SIMD body and scalar tail alike):
    ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2.  The single rounding (b0*h0 + b1*h1 + 2^21) >> 22
    is off by one on a few percent of the pixels."""
    H, W = img.shape[:2]
    xs, xa = upscale_tab(W, w)
    ys, ya = upscale_tab(H, h)
    S = img.astype(np.int64)
    xs1 = np.minimum(xs + 1, W - 1)
    ex = (1, w) + (1,) * (img.ndim - 2)
    hx = (S[:, xs] * xa[:, 0].reshape(ex) + S[:, xs1] * xa[:, 1].reshape(ex)) >> 4     # [H][w](..)
    ys1 = np.minimum(ys + 1, H - 1)
    ey = (h, 1) + (1,) * (img.ndim - 2)
    v = (((ya[:, 0].reshape(ey) * hx[ys]) >> 16) + ((ya[:, 1].reshape(ey) * hx[ys1]) >> 16) + 2) >> 2
    return np.clip(v, 0, 255).astype(np.uint8)


def resize_area(img: np.ndarray, w: int, h: int) -> np.ndarray:
    """cv2.resize(img, (w, h), interpolation=INTER_AREA) for u8 HxWx3 of any size (imutils.resize never asks for
    one axis up and the other down)."""
    H, W = img.shape[:2]
    if (w > W or h > H) and w >= W and h >= H:
        return resize_upscale(img, w, h)
    return _BASE_RESIZE(img, w, h)


def use_in_oracle(monkeypatch) -> None:
    """Route oracle.restated's resize (StreamOracle.process) through `resize_area` for the duration of a test."""
    monkeypatch.setattr(R, "resize_area", resize_area)
