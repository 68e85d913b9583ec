"""GPU: RGB, BGRA and RGBA input (FM_FLAG_RGB, FM_FLAG_ALPHA).  Such a context must give, on every front end, exactly what
a BGR context of the same tuning gives on cv2.cvtColor(frame, COLOR_RGB2BGR / COLOR_BGRA2BGR / COLOR_RGBA2BGR): every
fm_frame_stats field, every component, the dilated threshold plane, the gray and blur taps and the float64 background, with
as many kernel launches per call on packed frames (four-byte frames: one more on tcgen05, the apron fill, and one fewer where only their rows are 16-byte aligned); its clips are the input frames, alpha included, and its detector input
planes those of the BGR twin.  The frames are synth.make_clip's BGR frames with the channels flipped (RGB, RGBA) and
seeded random alpha bytes appended (BGRA, RGBA), so the BGR twin of each is the synthetic frame itself."""
import ctypes as C

import numpy as np
import pytest

from find_motion_b200 import synth
from tests import clips_restated as CR
from tests.test_gpu_gray import CONFIGS, TUNE, _batch, _masks, _same

pytestmark = pytest.mark.gpu


def _bgr_clips(W, H, S, n, fps, seed=17):
    return np.stack([synth.make_clip(W, H, n, seed=synth.stream_seed(seed, s), fps=fps) for s in range(S)])


FORMATS = ["rgb", "bgra", "rgba"]


def _ekw(fmt):
    return dict(rgb=fmt in ("rgb", "rgba"), alpha=fmt in ("bgra", "rgba"))


def _px(fmt):
    return 4 if fmt in ("bgra", "rgba") else 3


def _conv(bgr, fmt, seed=99):
    """[..., H, W, 3] BGR -> the format's frames: channels flipped for RGB / RGBA (cv2.COLOR_BGR2RGB is this flip), and a
    fourth byte of seeded random (not constant) alpha for BGRA / RGBA"""
    x = bgr[..., ::-1] if fmt in ("rgb", "rgba") else bgr
    if fmt in ("bgra", "rgba"):
        a = np.random.default_rng(seed).integers(0, 256, size=bgr.shape[:-1] + (1,), dtype=np.uint8)
        x = np.concatenate([x, a], axis=-1)
    return np.ascontiguousarray(x)


def _to_bgr(x, fmt):
    """the format's frames -> their BGR twins (cv2.cvtColor ..2BGR): drop the alpha byte, flip R-first orders"""
    x = x[..., :3]
    return x[..., ::-1] if fmt in ("rgb", "rgba") else x


def _pitched(pitch, pad=0):
    """a layout that copies the packed batch into rows `pitch` bytes apart (pad bytes before the first frame)"""
    import torch

    def lay(b):
        S, T, H, W, P = b.shape
        fstride = pitch * H + pad
        raw = torch.zeros(S * T * fstride + pad + 64, dtype=torch.uint8, device=b.device)
        v = raw.as_strided((S, T, H, W, P), (T * fstride, fstride, pitch, P, 1), pad)
        v.copy_(b)
        return v
    return lay


def _crop(pitch_px, rows, x0, y0):
    """a crop view [.., y0:y0 + H, x0:x0 + W] of padded surfaces of rows x pitch_px pixels"""
    def lay(b):
        import torch
        S, T, H, W, P = b.shape
        s = torch.full((S, T, rows, pitch_px, P), 77, dtype=torch.uint8, device=b.device)
        s[:, :, y0:y0 + H, x0:x0 + W] = b
        return s[:, :, y0:y0 + H, x0:x0 + W]
    return lay


def _compare(fmt, W, H, S, T, kw, ekw=None, keep=False, masks=True, layout=None):
    """Three calls and a reset: all frames, a ragged call with stream 0 at n_valid = 0, fm_ctx_reset, all frames.
    layout(batch) -> the device view the engine under test is fed (default: the packed batch)."""
    import torch
    from find_motion_b200.engine import MotionEngine, launch_count
    ekw = dict(ekw or {})
    if masks:
        kw = dict(kw, mask_areas=_masks(W, H))
    plan = [[T] * S, [0] + [max(1, T - s) for s in range(1, S)], "reset", [T] * S]
    clips = _bgr_clips(W, H, S, 3 * T, kw["fps"])
    with MotionEngine(W, H, n_streams=S, max_frames=T, keep_planes=keep, **_ekw(fmt), **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, keep_planes=keep, **ekw, **kw) as ref:
        assert eng.info == ref.info and eng.frame_shape == (H, W, _px(fmt))
        pos, moved = [0] * S, 0
        for i, nv in enumerate(plan):
            if nv == "reset":
                eng.reset()
                ref.reset()
                continue
            b = _batch(clips, pos, nv, T)
            dev = torch.from_numpy(_conv(b, fmt, seed=i)).cuda()
            dev = layout(dev) if layout else dev
            twin = torch.from_numpy(b).cuda()
            torch.cuda.synchronize()
            n0 = launch_count()
            got = eng.process(dev, n_valid=nv)
            n1 = launch_count()
            want = ref.process(twin, n_valid=nv)
            if layout is None:          # a pitched layout may take another front end than the packed twin
                # four-byte frames: on tcgen05 they fill the apron plane (k_pad_gray) where BGR ones feed k_umma_fused
                # directly; on the mma.sync blur, rows of W*4 bytes may be 16-byte aligned where W*3 are not, and then
                # pass 1 reads the frames instead of a gray plane made first (k_gray)
                extra = 0
                if _px(fmt) == 4 and ekw.get("umma"):
                    extra = 1
                elif _px(fmt) == 4 and eng.info["front_end"] == 1 and eng.info["gaussian"] > 1 and (3 * W) % 16 \
                        and (4 * W) % 16 == 0:
                    extra = -1
                assert n1 - n0 == launch_count() - n1 + extra, i
            assert (got == want).all(), (i, np.argwhere(got != want)[:4])
            moved += int(got["movement"].sum())
            _same(eng, ref, S, nv, keep, i)
            pos = [p + v for p, v in zip(pos, nv)]
        assert moved > 0                    # the scripted objects were seen
        return eng.info


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("name", list(CONFIGS))
def test_format_equals_bgr_of_cv2_conversion(name, fmt):
    W, H, S, T, kw, ekw, front_end = CONFIGS[name]
    info = _compare(fmt, W, H, S, T, kw, ekw)
    assert info["front_end"] == front_end


@pytest.mark.parametrize("name", ["1080p_k5_fused", "1080p_k97_wide", "1080p_k97_umma", "330x240_k1", "640x480_default",
                                  "640x480_ratio2", "80x60_upscale"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_keep_planes(name, fmt):
    W, H, _, _, kw, ekw, _ = CONFIGS[name]
    _compare(fmt, W, H, 2, 4, kw, ekw, keep=True)


@pytest.mark.parametrize("name", ["640x480_default", "640x480_ratio2", "80x60_upscale", "1080p_k97_wide", "1080p_k97_umma",
                                  "330x240_k1", "333x217_box111"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_odd_pitch_on_non_fused_front_ends(name, fmt):
    W, H, _, _, kw, ekw, _ = CONFIGS[name]
    _compare(fmt, W, H, 2, 4, kw, ekw, layout=_pitched(_px(fmt) * W + 5, pad=7))


@pytest.mark.parametrize("name", ["1080p_k5_fused", "1080p_default", "1080p_k97_wide", "1080p_k97_umma"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_crops_of_padded_surfaces(name, fmt):
    """Crops of 2048-pixel-wide surfaces read in place equal the packed frames (x0 = 16: 16-byte aligned rows)."""
    W, H, _, _, kw, ekw, _ = CONFIGS[name]
    _compare(fmt, W, H, 2, 4, kw, ekw, layout=_crop(2048, 1100, 16, 4))


@pytest.mark.parametrize("fmt", FORMATS)
def test_fused_refusals(fmt):
    """A fused context refuses rows TMA cannot read, and a non-zero uv_offset, with nothing enqueued."""
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    W, H, _, _, kw, _, _ = CONFIGS["1080p_k5_fused"]
    S, T = 2, 4
    clips = _bgr_clips(W, H, S, 2 * T, kw["fps"])
    with MotionEngine(W, H, n_streams=S, max_frames=T, **_ekw(fmt), **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **_ekw(fmt), **kw) as fresh:
        assert eng.info["front_end"] == 0
        first = torch.from_numpy(_conv(clips[:, :T], fmt)).cuda()
        with pytest.raises(_lib.FmError) as e:
            eng.process(_pitched(_px(fmt) * W + 4)(first))
        assert e.value.code == -1
        fr = _lib.fm_frames(first.data_ptr(), first.stride(0), first.stride(1), 0, 48)
        assert eng._lib.fm_process_frames(eng._ctx, C.byref(fr), T, None, None, None, None, 0, 0) == -1
        assert b"uv_offset" in eng._lib.fm_last_error()
        good = torch.from_numpy(_conv(clips[:, T:], fmt)).cuda()
        assert (eng.process(good) == fresh.process(good)).all()
        _same(eng, fresh, S, [T] * S, False, "after refusal")


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("W,H,kw", [(1920, 1080, dict(TUNE, box_size=1920, blur_scale=384)),
                                    (640, 480, dict(TUNE, box_size=100))])
def test_host_entry_points(W, H, kw, fmt):
    """fm_process_host and fm_submit_host / fm_wait on pinned batches give the stats of the device path."""
    import torch
    from find_motion_b200.engine import MotionEngine, PinnedBatch
    S, T = 2, 8
    clips = _conv(_bgr_clips(W, H, S, 3 * T, kw["fps"]), fmt)
    pin = [PinnedBatch((S, T, H, W, _px(fmt))) for _ in range(2)]
    with MotionEngine(W, H, n_streams=S, max_frames=T, **_ekw(fmt), **kw) as host, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **_ekw(fmt), **kw) as dev:
        want = [dev.process(torch.from_numpy(np.ascontiguousarray(clips[:, i * T:(i + 1) * T])).cuda()) for i in range(3)]
        pin[0].array[...] = clips[:, :T]
        assert (host.process_host(pin[0].array) == want[0]).all()
        pin[1].array[...] = clips[:, T:2 * T]
        host.submit_host(1, pin[1].array)
        pin[0].array[...] = clips[:, 2 * T:]
        host.submit_host(0, pin[0].array, n_valid=[T, T])
        assert (host.wait_host(1) == want[1]).all()
        assert (host.wait_host(0) == want[2]).all()
    for p in pin:
        p.free()


def _run_clips(fmt, W, H, S, n, T, kw, nvalid=None, layout=None):
    """process_clip: every clip frame is, byte for byte, the input frame (alpha included) the schedule of
    tests/clips_restated.py names, and its BGR conversion is the BGR twin context's clip frame."""
    import torch
    from find_motion_b200.engine import MotionEngine
    bgr = _bgr_clips(W, H, S, n, kw["fps"], seed=23)
    clips = _conv(bgr, fmt)
    flushed = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **_ekw(fmt), **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **kw) as ref:
        Cf = eng.info["cache_frames"]
        rings = [CR.RingSim(Cf) for _ in range(S)]
        fed = [[] for _ in range(S)]
        pos, i = [0] * S, 0
        while min(n - p for p in pos) > 0:
            nv = [min(v, n - p) for v, p in zip(nvalid(i) if nvalid else [T] * S, pos)]
            dev = torch.from_numpy(_batch(clips, pos, nv, T)).cuda()
            stats, out = eng.process_clip(layout(dev) if layout else dev, n_valid=nv)
            rstats, rout = ref.process_clip(torch.from_numpy(_batch(bgr, pos, nv, T)).cuda(), n_valid=nv)
            assert (stats == rstats).all(), i
            for s in range(S):
                fed[s] += range(pos[s], pos[s] + nv[s])
                ids = rings[s].call(stats[s], nv[s])
                got = out[s].cpu().numpy()
                assert got.shape == (len(ids), H, W, _px(fmt)), (s, got.shape)
                if ids:
                    assert np.array_equal(got, clips[s][[fed[s][j] for j in ids]]), (i, s, ids)
                    assert np.array_equal(_to_bgr(got, fmt), rout[s].cpu().numpy()), (i, s)
                flushed += int(stats[s]["n_flush"][:nv[s]].sum())
            pos = [p + v for p, v in zip(pos, nv)]
            i += 1
    return Cf, flushed


@pytest.mark.parametrize("fmt", FORMATS)
def test_clips_fused_geometry(fmt):
    Cf, flushed = _run_clips(fmt, 256, 192, 2, 48, 8, dict(TUNE, box_size=256, blur_scale=64))
    assert flushed > 0


@pytest.mark.parametrize("fmt", FORMATS)
def test_clips_call_longer_than_the_cache_ragged_pitched(fmt):
    rng = np.random.default_rng(5)
    sched = [[int(v) for v in rng.integers(0, 33, size=3)] for _ in range(20)]
    sched[0] = [32, 0, 20]
    kw = dict(fps=30, threshold=12, avg=0.3, min_time=0.04, cache_time=0.1, box_size=100)
    Cf, flushed = _run_clips(fmt, 160, 120, 3, 96, 32, kw, nvalid=lambda i: sched[i],
                             layout=_pitched(_px(fmt) * 160 + 5, pad=1))
    assert Cf == 3 and flushed > 0


@pytest.mark.parametrize("fmt", FORMATS)
@pytest.mark.parametrize("W,H,kw", [(1920, 1080, dict(TUNE, box_size=1920, blur_scale=384)),
                                    (640, 480, dict(TUNE, box_size=100)),
                                    (600, 400, dict(TUNE, box_size=100)),
                                    (300, 200, dict(TUNE, box_size=100)),
                                    (80, 60, dict(TUNE, box_size=100))])
@pytest.mark.parametrize("no_rows", [False, True])
def test_object_planes(W, H, kw, no_rows, fmt):
    """The detector input planes are BGR: those of the BGR twin context and cv2.resize of the twins (the rows kernel and
    the table fallback, the integer ratio 2, the 1 x 1 copy and the upscale)."""
    import cv2
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T = 2, 8
    ekw = dict(upscale=True) if kw["box_size"] > W else {}
    bgr = _bgr_clips(W, H, S, 3 * T, kw["fps"])
    planes = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, no_rows=no_rows, **_ekw(fmt), **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, no_rows=no_rows, **ekw, **kw) as ref:
        assert eng.object_shape == ref.object_shape
        oh = eng.object_shape[0]
        for i in range(3):
            tw = np.ascontiguousarray(bgr[:, i * T:(i + 1) * T])
            rd, td = torch.from_numpy(_conv(tw, fmt, seed=i)).cuda(), torch.from_numpy(tw).cuda()   # the planes read the call's frames
            assert (eng.process(rd) == ref.process(td)).all(), i
            got, want = eng.object_planes(), ref.object_planes()
            for s in range(S):
                assert np.array_equal(got[s][0], want[s][0])
                g = got[s][1].cpu().numpy()
                assert np.array_equal(g, want[s][1].cpu().numpy()), (i, s)
                for j, t in enumerate(got[s][0]):
                    assert np.array_equal(g[j], cv2.resize(tw[s, t], (300, oh), interpolation=cv2.INTER_AREA)), (i, s, t)
                planes += len(got[s][0])
    assert planes > 0
