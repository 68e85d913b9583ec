"""GPU: find_objects' detector input planes (FM_FLAG_OBJECT_PLANES, MotionEngine.object_planes, csrc/k_objects.cu).
Every plane is compared byte for byte with cv2.resize(raw, (300, oh), INTER_AREA) of the frame the call wrote, on the
seeded synthetic clips, and the frame list with the `wrote` flags of the call's stats."""
import ctypes as C

import cv2
import numpy as np
import pytest

from find_motion_b200 import synth
from tests import nv12_restated as NV

pytestmark = pytest.mark.gpu

TUNE = dict(fps=8, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)


def _oh(W, H):
    return int(H * (300 / float(W)))


def _want(frame, W, H):
    return cv2.resize(frame, (300, _oh(W, H)), interpolation=cv2.INTER_AREA)


def _clips(W, H, S, N, seed=23):
    return np.stack([synth.make_clip(W, H, N, seed=synth.stream_seed(seed, s), fps=TUNE["fps"]) for s in range(S)])


def _check(res, stats, frames, W, H, n_valid=None):
    """res: object_planes() of a call on frames [S, T, H, W, 3] (BGR) with those stats.  -> planes checked"""
    n = 0
    for s, (idx, planes) in enumerate(res):
        nv = stats.shape[1] if n_valid is None else n_valid[s]
        assert list(idx) == list(np.flatnonzero(stats[s]["wrote"][:nv])), s
        got = planes.cpu().numpy()
        assert got.shape == (len(idx), _oh(W, H), 300, 3)
        for i, t in enumerate(idx):
            assert np.array_equal(got[i], _want(frames[s, t], W, H)), (s, t)
        n += len(idx)
    return n


def _rows_usable(W, H):
    from find_motion_b200 import _lib
    if W < 300:
        return False
    info = _lib.fm_rows_plan_info()
    _lib.check(_lib.load().fm_debug_rows_plan(W, H, 300, C.byref(info)))
    return bool(info.usable)


# (W, H, tuning): full resolution k=5 (fused), default mode, k=97; the rows path (1080p, 720p, 4K, 640x480), the
# fallback with tables (1000x700: rows not 16-byte multiples), an integer ratio (600x400 -> 2x), the identity (300 wide),
# the upscale (160x120, 80x60, 203x117)
CONFIGS = [
    (1920, 1080, dict(box_size=1920, blur_scale=384)),
    (1920, 1080, dict(box_size=100, blur_scale=20)),
    (1920, 1080, dict(box_size=1920, blur_scale=20)),
    (1280, 720, dict(box_size=100, blur_scale=20)),
    (3840, 2160, dict(box_size=100, blur_scale=20)),
    (640, 480, dict(box_size=100, blur_scale=20)),
    (1000, 700, dict(box_size=100, blur_scale=20)),
    (600, 400, dict(box_size=100, blur_scale=20)),
    (300, 200, dict(box_size=100, blur_scale=20)),
    (160, 120, dict(box_size=100, blur_scale=20)),
    (80, 60, dict(box_size=80, blur_scale=16)),
    (203, 117, dict(box_size=100, blur_scale=20)),
]


@pytest.mark.parametrize("W,H,kw", CONFIGS, ids=[f"{w}x{h}_b{k['box_size']}_bs{k['blur_scale']}" for w, h, k in CONFIGS])
def test_planes_equal_cv2_for_written_frames(W, H, kw):
    """Over three calls with motion episodes: the planes of exactly the written frames, in order, equal cv2's."""
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, N = 2, 8, 24
    clips = _clips(W, H, S, N)
    dev = torch.from_numpy(clips).cuda()
    written = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, **TUNE, **kw) as eng:
        assert eng.object_shape == (_oh(W, H), 300, 3)
        for t0 in range(0, N, T):
            stats = eng.process(dev[:, t0:t0 + T])
            written += _check(eng.object_planes(), stats, clips[:, t0:t0 + T], W, H)
    assert written > 0, "the clip has motion episodes"


def test_both_resize_paths_are_covered():
    """The configurations above reach the rows kernel and the fallback (fm_debug_rows_plan(W, H, 300))."""
    rows = {(w, h): _rows_usable(w, h) for w, h, _ in CONFIGS}
    assert rows[(1920, 1080)] and rows[(1280, 720)] and rows[(3840, 2160)]
    assert not rows[(1000, 700)] and not rows[(600, 400)] and not rows[(300, 200)]


@pytest.mark.parametrize("W,H,kw,ekw", [
    (1920, 1080, dict(box_size=1920, blur_scale=384), {}),
    (640, 480, dict(box_size=100, blur_scale=20), {}),
    (160, 120, dict(box_size=200, blur_scale=20), dict(upscale=True)),
    (640, 480, dict(box_size=640, blur_scale=20), {}),
])
def test_flag_leaves_results_unchanged(W, H, kw, ekw):
    """With the flag, and object_planes called after every call, stats, contour records and the float64 background
    equal those of a context without the flag."""
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, N = 2, 8, 24
    masks = [((0, 0), (W // 6, H // 6))]
    dev = torch.from_numpy(_clips(W, H, S, N)).cuda()
    with MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, mask_areas=masks, **ekw, **TUNE, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, mask_areas=masks, **ekw, **TUNE, **kw) as ref:
        assert eng.info == ref.info
        for t0 in range(0, N, T):
            a = eng.process(dev[:, t0:t0 + T])
            eng.object_planes()
            b = ref.process(dev[:, t0:t0 + T])
            assert np.array_equal(a, b), t0
            for s in range(S):
                for t in range(T):
                    assert eng.components(s, t) == ref.components(s, t), (t0, s, t)
                assert np.array_equal(eng.planes(s, T - 1, gray=False, blur=False, thresh=False)["bg"],
                                      ref.planes(s, T - 1, gray=False, blur=False, thresh=False)["bg"]), (t0, s)


@pytest.mark.parametrize("W,H,kw,front_end", [
    (1920, 1080, dict(box_size=1920, blur_scale=384), 0),       # fused: the context converts the written frames
    (1920, 1080, dict(box_size=100, blur_scale=20), 2),         # staged: the slot of the call is resized
])
def test_nv12(W, H, kw, front_end):
    """NV12 contexts give the planes of cv2.cvtColor(frame, COLOR_YUV2BGR_NV12)."""
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, N = 2, 8, 24
    nv = np.stack([np.stack([NV.nv12_from_bgr(f) for f in clip]) for clip in _clips(W, H, S, N)])
    bgr = np.stack([np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in clip]) for clip in nv])
    dev = torch.from_numpy(nv).cuda()
    written = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, object_planes=True, **TUNE, **kw) as eng:
        assert eng.info["front_end"] == front_end
        for t0 in range(0, N, T):
            stats = eng.process(dev[:, t0:t0 + T])
            written += _check(eng.object_planes(), stats, bgr[:, t0:t0 + T], W, H)
    assert written > 0


@pytest.mark.parametrize("W,H,kw", [
    (1920, 1080, dict(box_size=100, blur_scale=20)),            # rows kernel, and the fallback for the padded strides
    (1920, 1080, dict(box_size=1920, blur_scale=384)),
    (203, 117, dict(box_size=100, blur_scale=20)),
])
def test_ragged_padded_and_quiet_streams(W, H, kw):
    """Ragged n_valid (including 0), frame and stream strides with padding (not 16-byte multiples), and a stream
    that writes nothing: its part of a sentinel-filled `out` stays untouched."""
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, N = 3, 8, 24
    clips = _clips(W, H, S, N)
    clips[2] = clips[2, :1]                                      # stream 2: a still scene
    fb = H * W * 3
    for pad in (0, 4):
        buf = torch.zeros(S * (T * (fb + pad) + pad) + pad, dtype=torch.uint8, device="cuda")
        frames = torch.as_strided(buf, (S, T, H, W, 3), (T * (fb + pad) + pad, fb + pad, W * 3, 3, 1), pad)
        out = torch.full((S, T + 1, _oh(W, H), 300, 3), 0xA5, dtype=torch.uint8, device="cuda")
        written = 0
        with MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, **TUNE, **kw) as eng:
            pos = [0] * S
            for i, nvalid in enumerate(([8, 8, 8], [5, 0, 8], [3, 8, 0], [8, 8, 8])):
                batch = np.zeros((S, T, H, W, 3), np.uint8)
                for s in range(S):
                    batch[s, :nvalid[s]] = clips[s, pos[s]:pos[s] + nvalid[s]]
                    pos[s] += nvalid[s]
                frames.copy_(torch.from_numpy(batch))
                out.fill_(0xA5)
                if pad and kw["box_size"] == 1920:               # the fused front end reads by TMA: aligned strides only
                    with pytest.raises(Exception):
                        eng.process(frames, n_valid=nvalid)
                    break
                stats = eng.process(frames, n_valid=nvalid)
                res = eng.object_planes(out=out)
                written += _check(res, stats, batch, W, H, nvalid)
                assert not stats["wrote"][2].any()
                assert len(res[2][0]) == 0
                assert bool((out[2] == 0xA5).all())
                for s in range(2):
                    assert bool((out[s, len(res[s][0]):] == 0xA5).all()), (i, s)
            if not (pad and kw["box_size"] == 1920):
                assert written > 0


def test_chained_calls_without_sync():
    """process; object_planes; process; object_planes with no synchronisation in between, on the fused front end whose
    next call starts under the contour tail of the previous one: both calls' planes are right."""
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    W, H, S, T, N = 1920, 1080, 4, 8, 32
    clips = _clips(W, H, S, N)
    dev = torch.from_numpy(clips).cuda()
    kw = dict(box_size=1920, blur_scale=384)
    oh = _oh(W, H)
    written = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, **TUNE, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **TUNE, **kw) as ref:
        assert eng.info["front_end"] == 0
        lib = _lib.load()
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        stats_dev = torch.empty((N // T, S * T * 32), dtype=torch.uint8, device="cuda")
        outs = torch.full((N // T, S, T, oh, 300, 3), 0xA5, dtype=torch.uint8, device="cuda")
        for i in range(N // T):                                  # everything enqueued, nothing waited for
            b = dev[:, i * T:(i + 1) * T]
            _lib.check(lib.fm_process(eng._ctx, b.data_ptr(), b.stride(0), b.stride(1), T, st, stats_dev[i].data_ptr()))
            _lib.check(lib.fm_object_planes(eng._ctx, st, outs[i].data_ptr(), outs[i].stride(0), T))
        torch.cuda.synchronize()
        eng.check()
        for i in range(N // T):
            stats = ref.process(dev[:, i * T:(i + 1) * T])
            got = stats_dev[i].cpu().numpy().view(stats.dtype).reshape(S, T)
            assert np.array_equal(got, stats), i
            res = []
            for s in range(S):
                idx = np.flatnonzero(stats[s]["wrote"])
                res.append((idx, outs[i, s, :len(idx)]))
            written += _check(res, stats, clips[:, i * T:(i + 1) * T], W, H)
    assert written > 0


def test_refusals():
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    W, H, S, T = 640, 480, 2, 4
    kw = dict(TUNE, box_size=100)
    frames = torch.from_numpy(_clips(W, H, S, T)).cuda()
    out = torch.empty((S, T, _oh(W, H), 300, 3), dtype=torch.uint8, device="cuda")
    lib = _lib.load()

    def planes(eng, cap=T, o=out):
        return lib.fm_object_planes(eng._ctx, None, o.data_ptr(), o.stride(0), cap)

    with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as eng:          # no flag
        eng.process(frames)
        assert planes(eng) == -1
    with MotionEngine(W, H, n_streams=S, max_frames=T, object_planes=True, **kw) as eng:
        assert planes(eng) == -1                                              # no call yet
        eng.process(frames)
        assert planes(eng, cap=T - 1) == -1                                   # short capacity
        assert planes(eng) == 0
        eng.process(frames[:, :2])
        assert planes(eng, cap=2, o=out[:, :2]) == 0                          # the last call's n_frames counts
        eng.process_host(frames.cpu().numpy())
        assert planes(eng) == -1                                              # host entry point
        eng.submit_host(0, frames.cpu().numpy())
        eng.wait_host(0)
        assert planes(eng) == -1
        eng.process(frames)
        assert planes(eng) == 0
        torch.cuda.synchronize()
    with pytest.raises(_lib.FmError) as e:                                    # oh = int(10 * 300 / 4000) = 0
        MotionEngine(4000, 10, n_streams=1, max_frames=1, object_planes=True, box_size=4000, blur_scale=800)
    assert e.value.code == -4


def test_launch_counts():
    """fm_process launches the same kernels with the flag as without; fm_object_planes adds the plan and the resize,
    and on a fused NV12 context the conversion."""
    import torch
    from find_motion_b200.engine import MotionEngine, launch_count

    def delta(fn):
        torch.cuda.synchronize()
        n = launch_count()
        fn()
        torch.cuda.synchronize()
        return launch_count() - n

    S, T = 2, 4
    for W, H, kw, nv12, extra in ((1920, 1080, dict(box_size=1920, blur_scale=384), False, 2),
                                  (1920, 1080, dict(box_size=100, blur_scale=20), False, 2),
                                  (160, 120, dict(box_size=100, blur_scale=20), False, 2),
                                  (1920, 1080, dict(box_size=1920, blur_scale=384), True, 3),
                                  (1920, 1080, dict(box_size=100, blur_scale=20), True, 2)):
        clips = _clips(W, H, S, T)
        if nv12:
            clips = np.stack([np.stack([NV.nv12_from_bgr(f) for f in c]) for c in clips])
        b = torch.from_numpy(clips).cuda()
        with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=nv12, object_planes=True, **TUNE, **kw) as eng, \
                MotionEngine(W, H, n_streams=S, max_frames=T, nv12=nv12, **TUNE, **kw) as ref:
            for _ in range(2):
                assert delta(lambda: eng.process(b)) == delta(lambda: ref.process(b)), (W, H, kw, nv12)
                assert delta(lambda: eng.object_planes()) == extra, (W, H, kw, nv12)
