"""GPU: frames with a row pitch or a chroma offset of their own (fm_process_frames).  Every case feeds one context the
frames pitched, cropped or split into planes, and a twin context of the same configuration the same frames packed, over
several chained calls (background and counters carry across calls).  Stats, components, the dilated threshold plane
and the float64 background (with KEEP_PLANES also gray and blur), clip frames and detector input planes must be equal,
byte for byte.  The padding around the frames is random, so a kernel that reads it shows."""
import functools

import numpy as np
import pytest

from find_motion_b200 import synth
from tests import nv12_restated as N12

pytestmark = pytest.mark.gpu

TUNE = dict(fps=8, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)
FUSED = dict(box_size=1920, blur_scale=384)           # 1080p full resolution, k = 5: k_fused
WIDE = dict(box_size=1920, blur_scale=20)             # 1080p full resolution, k = 97
DEFAULT = dict(box_size=100, blur_scale=20)           # default mode


@functools.lru_cache(maxsize=4)
def _clip(W, H, n, seed, quiet=False):
    c = synth.make_clip(W, H, n, seed=seed, fps=TUNE["fps"])
    return np.repeat(c[:1], n, axis=0) if quiet else c


def _packed(W, H, S, T, call, nv12, quiet_streams=()):
    """[S, T, H, W, 3] (nv12: [S, T, H * 3 // 2, W]) packed CUDA batch of call `call`."""
    import torch
    n = max(4 * T, 24)                       # up to four calls; at least 24 frames: the blip and the walker
    b = np.stack([_clip(W, H, n, synth.stream_seed(31, s), s in quiet_streams)[call * T:(call + 1) * T] for s in range(S)])
    if nv12:
        b = N12.nv12_from_bgr(b)
    return torch.from_numpy(np.ascontiguousarray(b)).cuda()


def _garbage(n):
    import torch
    return torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda")


def bgr_pitched(pitch, off=0):
    """rows `pitch` bytes apart, frames pitch * H apart, at byte offset `off` of a buffer of random bytes"""
    def feed(p):
        import torch
        S, T, H, W, _ = p.shape
        fs = pitch * H
        v = torch.as_strided(_garbage(S * T * fs + off), (S, T, H, W, 3), (T * fs, fs, pitch, 3, 1), off)
        v.copy_(p)
        return dict(frames=v)
    return feed


def bgr_crop(CW, CH, x0, y0):
    """frames[:, :, y0:y0 + H, x0:x0 + W] of CW x CH canvases"""
    def feed(p):
        S, T, H, W, _ = p.shape
        canvas = _garbage(S * T * CH * CW * 3).view(S, T, CH, CW, 3)
        v = canvas[:, :, y0:y0 + H, x0:x0 + W]
        v.copy_(p)
        return dict(frames=v)
    return feed


def nv12_surfaces(pitch, coded_rows, off=0):
    """decoder-like surfaces: luma pitch `pitch`, chroma after coded_rows luma rows, passed as luma and chroma views"""
    def feed(p):
        import torch
        S, T, R, W = p.shape
        H = R * 2 // 3
        fs = pitch * (coded_rows + coded_rows // 2)
        buf = _garbage(S * T * fs + off)
        luma = torch.as_strided(buf, (S, T, H, W), (T * fs, fs, pitch, 1), off)
        uv = torch.as_strided(buf, (S, T, H // 2, W), (T * fs, fs, pitch, 1), off + pitch * coded_rows)
        luma.copy_(p[:, :, :H])
        uv.copy_(p[:, :, H:])
        return dict(frames=luma, chroma=uv)
    return feed


def nv12_split(pitch, negative):
    """the chroma planes in an allocation of their own, before (negative uv_offset) or after the luma planes"""
    def feed(p):
        import torch
        S, T, R, W = p.shape
        H = R * 2 // 3
        fs = pitch * H
        a, b = _garbage(S * T * fs), _garbage(S * T * fs)
        lo, hi = (a, b) if a.data_ptr() < b.data_ptr() else (b, a)
        lbuf, cbuf = (hi, lo) if negative else (lo, hi)
        luma = torch.as_strided(lbuf, (S, T, H, W), (T * fs, fs, pitch, 1), 0)
        uv = torch.as_strided(cbuf, (S, T, H // 2, W), (T * fs, fs, pitch, 1), 0)
        luma.copy_(p[:, :, :H])
        uv.copy_(p[:, :, H:])
        assert (uv.data_ptr() < luma.data_ptr()) == negative
        return dict(frames=luma, chroma=uv, _keep=(a, b))
    return feed


def _compare_frames(eng, ref, st, rst, nv, keep):
    np.testing.assert_array_equal(st, rst)
    for s, v in enumerate(nv):
        for t in range(v):
            assert eng.components(s, t) == ref.components(s, t), (s, t)
            last = t == v - 1
            a = eng.planes(s, t, gray=keep, blur=keep, thresh=True, bg=last)
            b = ref.planes(s, t, gray=keep, blur=keep, thresh=True, bg=last)
            assert a.keys() == b.keys()
            for k in a:
                assert np.array_equal(a[k], b[k]), (s, t, k)


def _run(W, H, kw, feeds, S=2, T=4, calls=3, nv12=False, keep=False, clips=False, objects=False, ekw=None,
         nvalid=None, quiet_streams=(), expect_front_end=None, moving=True):
    """feeds[i % len(feeds)] lays out call i (None: packed, as the twin gets it)."""
    from find_motion_b200.engine import MotionEngine
    ekw = dict(ekw or {}, keep_planes=keep, device_clips=clips, object_planes=objects, nv12=nv12)
    kw = dict(TUNE, **kw)
    with MotionEngine(W, H, n_streams=S, max_frames=T, **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **ekw, **kw) as ref:
        if expect_front_end is not None:
            assert eng.info["front_end"] == expect_front_end
        contours = 0
        for i in range(calls):
            p = _packed(W, H, S, T, i, nv12, quiet_streams)
            nv = nvalid[i % len(nvalid)] if nvalid else [T] * S
            feed = feeds[i % len(feeds)]
            args = {k: v for k, v in (feed(p) if feed else dict(frames=p)).items() if not k.startswith("_")}
            if clips:
                st, cl = eng.process_clip(n_valid=nv, **args)
                cl = [c.clone() for c in cl]
                rst, rcl = ref.process_clip(p, n_valid=nv)
                for s in range(S):
                    assert cl[s].shape == rcl[s].shape and bool((cl[s] == rcl[s]).all()), (i, s)
            else:
                st = eng.process(n_valid=nv, **args)
                rst = ref.process(p, n_valid=nv)
            _compare_frames(eng, ref, st, rst, nv, keep)
            contours += int(st["n_contours"].sum())
            if objects:
                for (ia, pa), (ib, pb) in zip(eng.object_planes(), ref.object_planes()):
                    assert np.array_equal(ia, ib) and bool((pa == pb).all()), i
        if moving:
            assert contours > 0, "the scene never moved: the comparison says little"
        return eng, ref


# ---- 1080p full resolution, k = 5 (k_fused) ----
def test_fused_pitch_6144():
    _run(1920, 1080, FUSED, [bgr_pitched(6144)], expect_front_end=0)


def test_fused_crop_of_larger_canvas():
    _run(1920, 1080, FUSED, [bgr_crop(2048, 1200, 64, 8)], keep=True, expect_front_end=0)


def test_fused_ragged_including_zero():
    _run(1920, 1080, FUSED, [bgr_pitched(6144)], nvalid=[[4, 4], [0, 3], [2, 0]])


def test_fused_refuses_unaligned_pitch_and_stays_in_step():
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    W, H, S, T = 1920, 1080, 2, 4
    kw = dict(TUNE, **FUSED)
    with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as ref:
        for i in range(3):
            p = _packed(W, H, S, T, i, False)
            if i == 1:
                with pytest.raises(_lib.FmError) as e:
                    eng.process(**bgr_pitched(6144 + 8)(p))
                assert e.value.code == -1 and "row_pitch" in str(e.value)
            args = bgr_pitched(6144)(p) if i else dict(frames=p)
            _compare_frames(eng, ref, eng.process(**args), ref.process(p), [T] * S, False)


def test_no_fused_generic_gray():
    _run(1920, 1080, FUSED, [bgr_pitched(5776)], ekw=dict(no_fused=True), keep=True, calls=2)


# ---- 1080p, k = 97 ----
@pytest.mark.parametrize("pitch", [5888, 5768], ids=["aligned16_tma", "mod16_8"])
def test_k97(pitch):
    _run(1920, 1080, WIDE, [bgr_pitched(pitch)], calls=2, T=3)


@pytest.mark.parametrize("ekw", [dict(umma=True), dict(umma=True, umma_apron=True)], ids=["umma", "umma_apron"])
@pytest.mark.parametrize("pitch", [5888, 5768])
def test_k97_umma(ekw, pitch):
    _run(1920, 1080, WIDE, [bgr_pitched(pitch)], calls=2, T=3, ekw=dict(ekw, no_fused=True))


# ---- default mode (box 100) ----
DEFAULT_LAYOUTS = [(bgr_pitched(5888), {}), (bgr_pitched(5888), dict(no_rows=True)), (bgr_pitched(5764), {}),
                   (bgr_pitched(5761), {}), (bgr_crop(1925, 1090, 3, 1), {})]


@pytest.mark.parametrize("i", range(len(DEFAULT_LAYOUTS)), ids=["rows", "no_rows", "g4_mod16_4", "odd_pitch", "odd_crop"])
def test_default_mode_1080p(i):
    feed, ekw = DEFAULT_LAYOUTS[i]
    _run(1920, 1080, DEFAULT, [feed], ekw=ekw, keep=True)


@pytest.mark.parametrize("pitch", [11776, 11524, 11521], ids=["rows", "g4_mod16_4", "odd_pitch"])
def test_default_mode_4k(pitch):
    _run(3840, 2160, DEFAULT, [bgr_pitched(pitch)], S=1, T=3, calls=2)


def test_integer_ratio_and_upscale():
    _run(200, 112, dict(box_size=100, blur_scale=20), [bgr_pitched(608, off=3)], keep=True, T=6)
    _run(80, 60, dict(box_size=100, blur_scale=20), [bgr_pitched(250, off=1)], keep=True, T=6, ekw=dict(upscale=True))


# ---- NV12 ----
def test_nv12_fused_decoder_surfaces():
    _run(1920, 1080, FUSED, [nv12_surfaces(2048, 1088)], nv12=True, keep=True, expect_front_end=0)


@pytest.mark.parametrize("negative", [True, False], ids=["uv_before", "uv_after"])
def test_nv12_fused_separate_chroma(negative):
    _run(1920, 1080, FUSED, [nv12_split(2048, negative)], nv12=True, calls=2)


@pytest.mark.parametrize("pitch", [1928, 1922], ids=["mod16_8", "mod16_2"])
@pytest.mark.parametrize("kw", [DEFAULT, WIDE], ids=["default", "k97"])
def test_nv12_staged(kw, pitch):
    _run(1920, 1080, kw, [nv12_surfaces(pitch, 1090, off=pitch % 8)], nv12=True, calls=2, T=3)


def test_nv12_overlapping_planes_refused():
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    with MotionEngine(64, 48, n_streams=1, max_frames=2, nv12=True, **dict(TUNE, box_size=64, blur_scale=20)) as eng:
        buf = _garbage(2 * 128 * 80)
        luma = torch.as_strided(buf, (1, 2, 48, 64), (2 * 128 * 80, 128 * 80, 128, 1), 0)
        uv = torch.as_strided(buf, (1, 2, 24, 64), (2 * 128 * 80, 128 * 80, 128, 1), 128 * 40)     # inside the luma rows
        with pytest.raises(_lib.FmError) as e:
            eng.process(luma, chroma=uv)
        assert e.value.code == -1 and "overlaps" in str(e.value)
        luma = torch.as_strided(buf, (1, 2, 48, 64), (2 * 128 * 80, 128 * 80, 128, 1), 128 * 8)
        with pytest.raises(_lib.FmError):          # uv_offset < 0: the chroma rows run into the first luma rows
            eng.process(luma, chroma=torch.as_strided(buf, (1, 2, 24, 64), (2 * 128 * 80, 128 * 80, 128, 1), 0))
        with pytest.raises(AssertionError):        # a chroma view at the luma plane's address (uv_offset 0 means "packed")
            eng.process(luma, chroma=luma[:, :, :24])


# ---- clips ----
CLIP_CASES = {   # (front end, nv12, layouts of the calls in turn; None = packed).  The fused front end reads by TMA only
    "fused_bgr": (FUSED, False, [bgr_pitched(6144)]),
    "fused_bgr_interleaved": (FUSED, False, [bgr_pitched(5776), None]),
    "fused_nv12": (FUSED, True, [nv12_surfaces(2048, 1088)]),
    "fused_nv12_interleaved": (FUSED, True, [None, nv12_surfaces(1936, 1090)]),
    "default_bgr": (DEFAULT, False, [bgr_pitched(6144)]),
    "default_bgr_odd_interleaved": (DEFAULT, False, [bgr_pitched(5761, off=5), None]),
    "default_nv12": (DEFAULT, True, [nv12_surfaces(2048, 1088)]),
    "default_nv12_odd_interleaved": (DEFAULT, True, [None, nv12_surfaces(1922, 1090, off=2)]),
}


@pytest.mark.parametrize("case", list(CLIP_CASES))
def test_clips(case):
    """Stream 1 is quiet, so its frames go to the ring and come back in later calls; T = 6 > cache_frames = 4 (the
    stores of a call overwrite slots its gathers read)."""
    kw, nv12, feeds = CLIP_CASES[case]
    _run(1920, 1080, dict(kw, cache_time=0.5), feeds, T=6, calls=4, nv12=nv12, clips=True, quiet_streams=(1,))


# ---- detector input planes ----
@pytest.mark.parametrize("W,H,kw,feed,ekw", [
    (1920, 1080, DEFAULT, bgr_pitched(5888), {}),                 # k_resize_rows<true>
    (1920, 1080, DEFAULT, bgr_pitched(5764), {}),                 # k_resize_gray with BGR output
    (200, 150, DEFAULT, bgr_pitched(611, off=1), {}),             # W < 300: k_upscale_gray with BGR output
], ids=["rows", "resize_gray", "upscale"])
def test_object_planes(W, H, kw, feed, ekw):
    _run(W, H, kw, [feed], objects=True, ekw=ekw)


def test_object_planes_fused_nv12():
    _run(1920, 1080, FUSED, [nv12_surfaces(2048, 1088)], nv12=True, objects=True, expect_front_end=0)


# ---- MotionEngine ----
def test_engine_crop_view_and_chroma_pair():
    """A torch crop view and a chroma= pair of surface slices give what .contiguous() input gives."""
    import torch
    from find_motion_b200.engine import MotionEngine
    W, H, S, T, Hc = 640, 360, 2, 4, 368
    kw = dict(TUNE, box_size=100, blur_scale=20)
    for nv12 in (False, True):
        with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=nv12, device_clips=True, object_planes=True, **kw) as eng, \
                MotionEngine(W, H, n_streams=S, max_frames=T, nv12=nv12, device_clips=True, object_planes=True, **kw) as ref:
            for i in range(3):
                p = _packed(W, H, S, T, i, nv12)
                if nv12:
                    surf = _garbage(S * T * (Hc * 3 // 2) * 704).view(S, T, Hc * 3 // 2, 704)
                    surf[..., :H, :W] = p[:, :, :H]
                    surf[..., Hc:Hc + H // 2, :W] = p[:, :, H:]
                    a, b = eng.process_clip(surf[..., :H, :W], chroma=surf[..., Hc:Hc + H // 2, :W])
                    a2 = eng.process(surf[..., :H, :W], chroma=surf[..., Hc:Hc + H // 2, :W])
                    assert not surf[..., :H, :W].is_contiguous()
                else:
                    canvas = _garbage(S * T * 400 * 700 * 3).view(S, T, 400, 700, 3)
                    canvas[:, :, 7:7 + H, 13:13 + W] = p
                    view = canvas[:, :, 7:7 + H, 13:13 + W]
                    a, b = eng.process_clip(view)
                    a2 = eng.process(view)
                ra, rb = ref.process_clip(p.contiguous())
                ra2 = ref.process(p.contiguous())
                np.testing.assert_array_equal(a, ra)
                np.testing.assert_array_equal(a2, ra2)
                for x, y in zip(b, rb):
                    assert x.shape == y.shape and bool((x == y).all())
                for (ia, pa), (ib, pb) in zip(eng.object_planes(), ref.object_planes()):
                    assert np.array_equal(ia, ib) and bool((pa == pb).all())
