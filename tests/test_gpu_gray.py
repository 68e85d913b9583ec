"""GPU: single-channel gray input (FM_FLAG_GRAY).  A gray context must give, on every front end, exactly what a BGR context
of the same tuning gives on cv2.cvtColor(frame, COLOR_GRAY2BGR): every fm_frame_stats field, every component, the dilated
threshold plane, the gray and blur taps and the float64 background; its clips are the gray input frames and its detector
input planes those of the BGR twins.  The gray frames are cv2.cvtColor(synth.make_clip(...), COLOR_BGR2GRAY)."""
import numpy as np
import pytest

from find_motion_b200 import synth
from tests import clips_restated as CR

pytestmark = pytest.mark.gpu

TUNE = dict(fps=8, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)


def _masks(W, H):
    return [((0, 0), (W // 8, H // 8)), ((W // 2, H // 2), (W // 2, H - 1), (W - 1, H // 2))]


def _gray_clips(W, H, S, n, fps, seed=17):
    import cv2
    return np.stack([np.stack([cv2.cvtColor(f, cv2.COLOR_BGR2GRAY)
                               for f in synth.make_clip(W, H, n, seed=synth.stream_seed(seed, s), fps=fps)])
                     for s in range(S)])


def _twin(g):
    """[..., H, W] gray -> [..., H, W, 3] BGR by cv2 itself: what the BGR context is fed."""
    import cv2
    flat = g.reshape((-1,) + g.shape[-2:])
    out = np.stack([cv2.cvtColor(f, cv2.COLOR_GRAY2BGR) for f in flat])
    return out.reshape(g.shape + (3,))


def _batch(clips, pos, nv, T):
    """[S, T, ...] of the next nv[s] frames of each stream, zeros past n_valid."""
    b = np.zeros((clips.shape[0], T) + clips.shape[2:], np.uint8)
    for s, (p, v) in enumerate(zip(pos, nv)):
        b[s, :v] = clips[s, p:p + v]
    return b


def _same(eng, ref, S, nv, keep, tag):
    for s in range(S):
        a = eng.planes(s, 0, gray=False, blur=False, thresh=False)
        r = ref.planes(s, 0, gray=False, blur=False, thresh=False)
        assert (a["bg"] == r["bg"]).all(), ("bg", tag, s)
        for t in range(nv[s]):
            assert eng.components(s, t) == ref.components(s, t), (tag, s, t)
            a, r = eng.planes(s, t, gray=keep, blur=keep, bg=False), ref.planes(s, t, gray=keep, blur=keep, bg=False)
            for key in a:
                assert (a[key] == r[key]).all(), (key, tag, s, t)


def _compare(W, H, S, T, kw, ekw=None, keep=False, masks=True, layout=None):
    """Three calls and a reset: all frames, a ragged call with stream 0 at n_valid = 0, fm_ctx_reset, all frames.
    layout(batch) -> the device view the gray engine is fed (default: the packed batch)."""
    import torch
    from find_motion_b200.engine import MotionEngine
    ekw = dict(ekw or {})
    if masks:
        kw = dict(kw, mask_areas=_masks(W, H))
    plan = [[T] * S, [0] + [max(1, T - s) for s in range(1, S)], "reset", [T] * S]
    clips = _gray_clips(W, H, S, 3 * T, kw["fps"])
    with MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, keep_planes=keep, **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, keep_planes=keep, **ekw, **kw) as ref:
        assert eng.info == ref.info
        pos, moved = [0] * S, 0
        for i, nv in enumerate(plan):
            if nv == "reset":
                eng.reset()
                ref.reset()
                continue
            b = _batch(clips, pos, nv, T)
            dev = torch.from_numpy(b).cuda()
            got = eng.process(layout(dev) if layout else dev, n_valid=nv)
            want = ref.process(torch.from_numpy(_twin(b)).cuda(), n_valid=nv)
            assert (got == want).all(), (i, np.argwhere(got != want)[:4])
            moved += int(got["movement"].sum())
            _same(eng, ref, S, nv, keep, i)
            pos = [p + v for p, v in zip(pos, nv)]
        assert moved > 0                    # the scripted objects were seen
        return eng.info


CONFIGS = {
    "1080p_k5_fused": (1920, 1080, 8, 16, dict(TUNE, box_size=1920, blur_scale=384), {}, 0),
    "720p_k5_T32": (1280, 720, 2, 32, dict(TUNE, box_size=1280, blur_scale=256), {}, 0),
    "720p_k5_T33": (1280, 720, 2, 33, dict(TUNE, box_size=1280, blur_scale=256), {}, 0),
    "4k_k5": (3840, 2160, 2, 4, dict(TUNE, box_size=3840, blur_scale=768), {}, 0),
    "1080p_k97_wide": (1920, 1080, 2, 8, dict(TUNE, box_size=1920, blur_scale=20), dict(no_umma=True), 1),
    "1080p_k97_umma": (1920, 1080, 2, 8, dict(TUNE, box_size=1920, blur_scale=20), dict(umma=True), 1),
    "330x240_k1": (330, 240, 2, 8, dict(TUNE, box_size=330, blur_scale=400), {}, 1),
    "1000x562_k5_not_fusable": (1000, 562, 2, 8, dict(TUNE, box_size=1000, blur_scale=200), {}, 1),
    "1080p_default": (1920, 1080, 4, 8, dict(TUNE, box_size=100), {}, 2),
    "640x480_default": (640, 480, 2, 8, dict(TUNE, box_size=100), {}, 2),
    "640x480_default_no_rows": (640, 480, 2, 8, dict(TUNE, box_size=100), dict(no_rows=True), 2),
    "640x480_ratio2": (640, 480, 2, 8, dict(TUNE, box_size=320), {}, 2),
    "80x60_upscale": (80, 60, 2, 8, dict(TUNE, box_size=100), dict(upscale=True), 2),
    "333x217_box111": (333, 217, 2, 8, dict(TUNE, box_size=111), {}, 2),
    # the one-channel warp-per-row kernels with tap groups that do not fit registers (k_resize_gray_g4<4, false, 1>, and
    # with 3840-byte segments <8, false, 1>)
    "4k_default_no_rows": (3840, 2160, 2, 4, dict(TUNE, box_size=100), dict(no_rows=True), 2),
    "4k_box32_no_rows": (3840, 2160, 2, 4, dict(TUNE, box_size=32), dict(no_rows=True), 2),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_gray_equals_bgr_of_cv2_conversion(name):
    W, H, S, T, kw, ekw, front_end = CONFIGS[name]
    info = _compare(W, H, S, T, kw, ekw)
    assert info["front_end"] == front_end
    if name == "330x240_k1":
        assert info["gaussian"] == 1


@pytest.mark.parametrize("name", ["1080p_k5_fused", "1080p_k97_wide", "1080p_k97_umma", "330x240_k1", "640x480_default",
                                  "640x480_ratio2", "80x60_upscale"])
def test_gray_keep_planes(name):
    W, H, _, _, kw, ekw, _ = CONFIGS[name]
    _compare(W, H, 2, 4, kw, ekw, keep=True)


def _pitched(pitch, pad=0):
    """a layout that copies the packed batch into rows `pitch` bytes apart (pad bytes before the first frame)"""
    import torch

    def lay(b):
        S, T, H, W = b.shape
        fstride = pitch * H + pad
        raw = torch.zeros(S * T * fstride + pad + 64, dtype=torch.uint8, device=b.device)
        v = raw.as_strided((S, T, H, W), (T * fstride, fstride, pitch, 1), pad)
        v.copy_(b)
        return v
    return lay


@pytest.mark.parametrize("name", ["640x480_default", "640x480_ratio2", "80x60_upscale", "1080p_k97_wide", "1080p_k97_umma",
                                  "330x240_k1", "333x217_box111"])
def test_odd_pitch_on_non_fused_front_ends(name):
    W, H, _, _, kw, ekw, _ = CONFIGS[name]
    _compare(W, H, 2, 4, kw, ekw, layout=_pitched(W + 3, pad=5))


def test_default_mode_pitch_multiple_of_4():
    """rows 4-byte but not 16-byte aligned: not TMA-readable, so the one-channel k_resize_gray_g4 instead of the rows
    kernel"""
    W, H, _, _, kw, ekw, _ = CONFIGS["1080p_default"]
    _compare(W, H, 2, 4, kw, ekw, layout=_pitched(W + 4, pad=8))


@pytest.mark.parametrize("no_rows", [False, True])
def test_default_mode_runs_the_one_channel_rows_kernel(no_rows):
    """the reference's default regime on gray frames takes k_resize_rows (one-channel plan) unless FM_FLAG_NO_ROWS"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from find_motion_b200.engine import MotionEngine
    W, H, S, T = 1920, 1080, 2, 4
    kw = dict(TUNE, box_size=100)
    b = torch.from_numpy(_gray_clips(W, H, S, T, kw["fps"])).cuda()
    with MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, no_rows=no_rows, **kw) as eng:
        eng.process(b)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            eng.process(b)
            torch.cuda.synchronize()
    names = {e.key for e in prof.key_averages()}
    rows = any("k_resize_rows" in n for n in names)
    g4 = any("k_resize_gray_g4" in n for n in names)
    assert (rows, g4) == (not no_rows, no_rows), sorted(n for n in names if n.startswith(("k_", "void k_")))


def test_fused_pitch_multiple_of_16_and_refusal():
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    W, H, _, _, kw, ekw, _ = CONFIGS["1080p_k5_fused"]
    _compare(W, H, 2, 4, kw, ekw, layout=_pitched(W + 48, pad=16))
    S, T = 2, 4
    clips = _gray_clips(W, H, S, 2 * T, kw["fps"])
    with MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, **kw) as fresh:
        assert eng.info["front_end"] == 0
        bad = _pitched(W + 4)(torch.from_numpy(clips[:, :T]).cuda())
        with pytest.raises(_lib.FmError) as e:
            eng.process(bad)
        assert e.value.code == -1
        good = torch.from_numpy(np.ascontiguousarray(clips[:, T:])).cuda()
        assert (eng.process(good) == fresh.process(good)).all()
        _same(eng, fresh, S, [T] * S, False, "after refusal")


@pytest.mark.parametrize("name", ["1080p_k5_fused", "1080p_default", "1080p_k97_wide"])
def test_luma_of_padded_decoder_surfaces(name):
    """The luma plane of NV12 surfaces (pitch 2048, 1088 coded rows, chroma after them) read in place equals the packed
    luma."""
    W, H, _, _, kw, ekw, _ = CONFIGS[name]

    def surf(b):
        import torch
        S, T = b.shape[:2]
        s = torch.full((S, T, 1088 * 3 // 2, 2048), 77, dtype=torch.uint8, device=b.device)
        s[:, :, :H, :W] = b
        return s[:, :, :H, :W]
    _compare(W, H, 2, 4, kw, ekw, layout=surf)


@pytest.mark.parametrize("W,H,kw", [(1920, 1080, dict(TUNE, box_size=1920, blur_scale=384)),
                                    (640, 480, dict(TUNE, box_size=100))])
def test_host_entry_points(W, H, kw):
    """fm_process_host and fm_submit_host / fm_wait on pinned gray batches give the stats of the device path."""
    import torch
    from find_motion_b200.engine import MotionEngine, PinnedBatch
    S, T = 2, 8
    clips = _gray_clips(W, H, S, 3 * T, kw["fps"])
    pin = [PinnedBatch((S, T, H, W)) for _ in range(2)]
    with MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, **kw) as host, \
            MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, **kw) as dev:
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


def _run_clips(W, H, S, n, T, kw, nvalid=None, layout=None):
    """process_clip of a gray context: every clip frame is, byte for byte, the gray input frame the schedule of
    tests/clips_restated.py names, and channel 0 of the BGR twin context's clip frame; the stats equal the twin's."""
    import torch
    from find_motion_b200.engine import MotionEngine
    clips = _gray_clips(W, H, S, n, kw["fps"], seed=23)
    flushed = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, device_clips=True, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **kw) as ref:
        C = eng.info["cache_frames"]
        rings = [CR.RingSim(C) for _ in range(S)]
        fed = [[] for _ in range(S)]
        pos, i = [0] * S, 0
        while min(n - p for p in pos) > 0:
            nv = [min(v, n - p) for v, p in zip(nvalid(i) if nvalid else [T] * S, pos)]
            b = _batch(clips, pos, nv, T)
            dev = torch.from_numpy(b).cuda()
            stats, out = eng.process_clip(layout(dev) if layout else dev, n_valid=nv)
            rstats, rout = ref.process_clip(torch.from_numpy(_twin(b)).cuda(), n_valid=nv)
            assert (stats == rstats).all(), i
            for s in range(S):
                fed[s] += range(pos[s], pos[s] + nv[s])
                ids = rings[s].call(stats[s], nv[s])
                got = out[s].cpu().numpy()
                assert got.shape == (len(ids), H, W), (s, got.shape)
                if ids:
                    assert np.array_equal(got, clips[s][[fed[s][j] for j in ids]]), (i, s, ids)
                    assert np.array_equal(got, rout[s].cpu().numpy()[..., 0]), (i, s)
                flushed += int(stats[s]["n_flush"][:nv[s]].sum())
            pos = [p + v for p, v in zip(pos, nv)]
            i += 1
    return C, flushed


def test_clips_fused_geometry():
    C, flushed = _run_clips(256, 192, 2, 48, 8, dict(TUNE, box_size=256, blur_scale=64))
    assert flushed > 0


def test_clips_call_longer_than_the_cache_ragged_pitched():
    rng = np.random.default_rng(5)
    sched = [[int(v) for v in rng.integers(0, 33, size=3)] for _ in range(20)]
    sched[0] = [32, 0, 20]
    kw = dict(fps=30, threshold=12, avg=0.3, min_time=0.04, cache_time=0.1, box_size=100)
    C, flushed = _run_clips(160, 120, 3, 96, 32, kw, nvalid=lambda i: sched[i], layout=_pitched(163, pad=1))
    assert C == 3 and flushed > 0


@pytest.mark.parametrize("W,H,kw", [(1920, 1080, dict(TUNE, box_size=1920, blur_scale=384)),
                                    (640, 480, dict(TUNE, box_size=100)),
                                    (600, 400, dict(TUNE, box_size=100)),
                                    (300, 200, dict(TUNE, box_size=100)),
                                    (80, 60, dict(TUNE, box_size=100))])
def test_object_planes(W, H, kw):
    """The detector input planes of a gray context equal the BGR twin context's and cv2.resize of the twins (tables,
    the integer ratio 2, the 1 x 1 copy and the upscale)."""
    import cv2
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T = 2, 8
    ekw = dict(upscale=True) if kw["box_size"] > W else {}
    clips = _gray_clips(W, H, S, 3 * T, kw["fps"])
    planes = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, gray=True, object_planes=True, **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, **ekw, **kw) as ref:
        assert eng.object_shape == ref.object_shape
        oh = eng.object_shape[0]
        for i in range(3):
            b = np.ascontiguousarray(clips[:, i * T:(i + 1) * T])
            tw = _twin(b)
            gd, td = torch.from_numpy(b).cuda(), torch.from_numpy(tw).cuda()     # the planes read the call's frames
            assert (eng.process(gd) == ref.process(td)).all(), i
            got, want = eng.object_planes(), ref.object_planes()
            for s in range(S):
                assert np.array_equal(got[s][0], want[s][0])
                g = got[s][1].cpu().numpy()
                assert np.array_equal(g, want[s][1].cpu().numpy()), (i, s)
                for j, t in enumerate(got[s][0]):
                    assert np.array_equal(g[j], cv2.resize(tw[s, t], (300, oh), interpolation=cv2.INTER_AREA)), (i, s, t)
                planes += len(got[s][0])
    assert planes > 0
