"""CPU: the restatement of cv2's INTER_AREA upscale (tests/upscale_restated.py) -- what imutils.resize does to a
frame narrower than box_size (find_motion.py:492) -- against cv2 itself, byte for byte, and the whole per-frame chain
of StreamOracle against the cv2 call chain on upscaled streams.  Also the FM_FLAG_UPSCALE constant of the C ABI."""
import os
import re

import numpy as np
import pytest

from oracle import restated as R
from tests import upscale_restated as U

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (W, H, width): imutils.resize(frame, width=width) gives height int(H * width / W) >= H
GEOMETRIES = [
    (640, 480, 800), (1280, 720, 1920), (1920, 1080, 3840), (80, 60, 100), (160, 120, 300), (320, 240, 640),
    (1, 1, 100), (97, 31, 100), (7, 1000, 100), (333, 217, 1000), (64, 48, 100), (96, 96, 100), (80, 60, 300),
    (299, 100, 300), (160, 120, 640), (213, 120, 640), (320, 240, 960), (100, 75, 300), (2, 3, 5), (3, 2, 7),
    (1, 5, 3), (5, 1, 8), (17, 13, 100), (31, 29, 300), (640, 360, 1920), (720, 480, 800), (720, 576, 1920),
    (800, 600, 1920), (1024, 768, 1920), (1366, 768, 1920), (1280, 1024, 3840), (1920, 1200, 3840),
    (176, 144, 300), (352, 288, 800), (250, 250, 251), (639, 479, 640), (101, 99, 303), (123, 45, 1000),
    (64, 64, 192), (10, 640, 300), (3, 3, 9), (128, 96, 800), (500, 7, 1920), (1919, 1079, 1920),
]


@pytest.mark.parametrize("W,H,width", GEOMETRIES)
def test_resize_upscale_matches_cv2(W, H, width):
    cv2 = pytest.importorskip("cv2")
    h = int(H * (width / float(W)))
    assert h >= H
    rng = np.random.default_rng(W * 7919 + H * 31 + width)
    img = rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
    want = cv2.resize(img, (width, h), interpolation=cv2.INTER_AREA)
    got = U.resize_area(img, width, h)
    assert got.shape == want.shape and (got == want).all(), int((got != want).sum())
    # saturated and dark frames: every chain at the ends of the range
    for v in (0, 255):
        flat = np.full((H, W, 3), v, np.uint8)
        assert (U.resize_area(flat, width, h) == cv2.resize(flat, (width, h), interpolation=cv2.INTER_AREA)).all()


def test_vertical_rounding_is_cv2s_two_step_form():
    """The single rounding (b0*h0 + b1*h1 + 2^21) >> 22 differs from cv2 on these geometries: the restatement must not."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(3)
    for W, H, width in ((640, 480, 800), (80, 60, 100), (160, 120, 300)):
        h = int(H * (width / float(W)))
        img = rng.integers(0, 256, size=(H, W, 3), dtype=np.uint8)
        xs, xa = U.upscale_tab(W, width)
        ys, ya = U.upscale_tab(H, h)
        S = img.astype(np.int64)
        hx = S[:, xs] * xa[:, 0, None] + S[:, np.minimum(xs + 1, W - 1)] * xa[:, 1, None]
        naive = (ya[:, 0, None, None] * hx[ys] + ya[:, 1, None, None] * hx[np.minimum(ys + 1, H - 1)] + (1 << 21)) >> 22
        want = cv2.resize(img, (width, h), interpolation=cv2.INTER_AREA)
        assert (naive != want).any()
        assert (U.resize_area(img, width, h) == want).all()


def _run_chain(monkeypatch, W, H, n, kw, seed):
    cv2 = pytest.importorskip("cv2")
    U.use_in_oracle(monkeypatch)
    from find_motion_b200 import synth
    from oracle import cv2_chain
    clip = synth.make_clip(W, H, n, seed=seed, fps=kw.get("fps", 30))
    orc = R.StreamOracle(W, H, **kw)
    ref = cv2_chain.Cv2Stream(W, H, **kw)
    assert (orc.w, orc.h) == (kw["box_size"], int(H * (kw["box_size"] / float(W))))
    moved = 0
    for t in range(n):
        rec = orc.process(clip[t], keep_planes=True)
        want = ref.step(clip[t])
        for key in ("gray", "blur", "thresh"):
            assert (rec["planes"][key] == want[key]).all(), (key, t)
        assert (orc.bg == ref.ref_frame).all(), ("bg", t)
        assert rec["areas"] == want["areas"], t
        cnts = cv2.findContours(want["thresh"], mode=cv2.RETR_EXTERNAL, method=cv2.CHAIN_APPROX_SIMPLE)[-2]
        assert rec["boxes"] == sorted(tuple(cv2.boundingRect(c)) for c in cnts), t
        for key in ("movement", "counter", "decay", "cache_len", "wrote", "n_flush"):
            assert rec[key] == want[key], (key, t)
        moved += bool(rec["movement"])
    assert moved > 0                      # the clip's scripted objects were seen


def test_stream_oracle_equals_cv2_chain_low_res_camera(monkeypatch):
    """An 80x60 sensor at the CLI default box_size 100."""
    _run_chain(monkeypatch, 80, 60, 24, dict(fps=6, box_size=100, blur_scale=20, threshold=8, avg=0.2, min_time=0.3,
                                cache_time=0.6), seed=41)


def test_stream_oracle_equals_cv2_chain_with_masks(monkeypatch):
    """320x240 at box 640 with rectangle and polygon masks scaled by box_size / W = 2 (find_motion.py:616)."""
    masks = [((0, 0), (50, 50)), ((0, 0), (0, 50), (50, 0)), ((200, 30), (280, 90)), ((40, 150), (40, 220), (120, 150))]
    _run_chain(monkeypatch, 320, 240, 16, dict(fps=6, box_size=640, blur_scale=32, threshold=8, avg=0.15, min_time=0.3,
                                  cache_time=0.6, mask_areas=masks), seed=42)


def test_derive_params_of_an_upscaled_stream():
    p = R.derive_params(80, 60, box_size=100)
    assert (p["w"], p["h"], p["scale"], p["gaussian"]) == (100, 75, 1.25, 5)


def test_upscale_flag_constant():
    from find_motion_b200 import _lib
    with open(os.path.join(ROOT, "include", "fm_gpu.h")) as f:
        hdr = f.read()
    m = re.search(r"#define\s+FM_FLAG_UPSCALE\s+(\d+)", hdr)
    assert m and int(m.group(1)) == _lib.FLAG_UPSCALE == 128
