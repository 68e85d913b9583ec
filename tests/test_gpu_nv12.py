"""GPU: NV12 input (FM_FLAG_NV12).  An NV12 context must give, on every front end, exactly what a BGR context of the
same tuning gives on cv2.cvtColor(frame, COLOR_YUV2BGR_NV12): every fm_frame_stats field, every component, the dilated
threshold plane, the gray and blur taps and the float64 background.  The NV12 frames are synthetic decoder output
(synth.make_clip -> COLOR_BGR2YUV_I420 -> interleaved chroma, tests/nv12_restated.py)."""
import numpy as np
import pytest

from find_motion_b200 import synth
from tests import clips_restated as CR
from tests import nv12_restated as N12

pytestmark = pytest.mark.gpu

TUNE = dict(fps=8, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)


def _masks(W, H):
    return [((0, 0), (W // 8, H // 8)), ((W // 2, H // 2), (W // 2, H - 1), (W - 1, H // 2))]


def _nv12_clips(W, H, S, n, fps, seed=17):
    return np.stack([N12.nv12_from_bgr(synth.make_clip(W, H, n, seed=synth.stream_seed(seed, s), fps=fps))
                     for s in range(S)])


def _twin(nv):
    """[..., H * 3 // 2, W] NV12 -> [..., H, W, 3] BGR by cv2 itself: what the BGR context is fed."""
    import cv2
    flat = nv.reshape((-1,) + nv.shape[-2:])
    out = np.stack([cv2.cvtColor(f, cv2.COLOR_YUV2BGR_NV12) for f in flat])
    return out.reshape(nv.shape[:-2] + out.shape[1:])


def _batch(clips, pos, nv, T):
    """[S, T, ...] of the next nv[s] frames of each stream, zeros past n_valid."""
    b = np.zeros((clips.shape[0], T) + clips.shape[2:], np.uint8)
    for s, (p, v) in enumerate(zip(pos, nv)):
        b[s, :v] = clips[s, p:p + v]
    return b


def _compare(W, H, S, T, kw, ekw=None, keep=False, masks=True):
    """Three calls and a reset: all frames, a ragged call with stream 0 at n_valid = 0, fm_ctx_reset, all frames."""
    import torch
    from find_motion_b200.engine import MotionEngine
    ekw = dict(ekw or {})
    if masks:
        kw = dict(kw, mask_areas=_masks(W, H))
    plan = [[T] * S, [0] + [max(1, T - s) for s in range(1, S)], "reset", [T] * S]
    clips = _nv12_clips(W, H, S, 3 * T, kw["fps"])
    with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, keep_planes=keep, **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, keep_planes=keep, **ekw, **kw) as ref:
        assert eng.info == ref.info
        pos, moved = [0] * S, 0
        for i, nv in enumerate(plan):
            if nv == "reset":
                eng.reset()
                ref.reset()
                continue
            b = _batch(clips, pos, nv, T)
            got = eng.process(torch.from_numpy(b).cuda(), n_valid=nv)
            want = ref.process(torch.from_numpy(_twin(b)).cuda(), n_valid=nv)
            assert (got == want).all(), (i, np.argwhere(got != want)[:4])
            moved += int(got["movement"].sum())
            for s in range(S):
                a, r = eng.planes(s, 0, gray=False, blur=False, thresh=False), ref.planes(s, 0, gray=False, blur=False,
                                                                                          thresh=False)
                assert (a["bg"] == r["bg"]).all(), ("bg", i, s)
                for t in range(nv[s]):
                    assert eng.components(s, t) == ref.components(s, t), (i, s, t)
                    a, r = eng.planes(s, t, gray=keep, blur=keep, bg=False), ref.planes(s, t, gray=keep, blur=keep, bg=False)
                    for key in a:
                        assert (a[key] == r[key]).all(), (key, i, s, t)
            pos = [p + v for p, v in zip(pos, nv)]
        assert moved > 0                    # the scripted objects were seen
        return eng.info


CONFIGS = {
    "1080p_k5_fused": (1920, 1080, 8, 16, dict(TUNE, box_size=1920, blur_scale=384), {}),
    "720p_k5_T32": (1280, 720, 2, 32, dict(TUNE, box_size=1280, blur_scale=256), {}),
    "4k_k5": (3840, 2160, 2, 4, dict(TUNE, box_size=3840, blur_scale=768), {}),
    "1080p_k97_wide": (1920, 1080, 2, 8, dict(TUNE, box_size=1920, blur_scale=20), dict(no_umma=True)),
    "1080p_k97_umma": (1920, 1080, 2, 8, dict(TUNE, box_size=1920, blur_scale=20), dict(umma=True)),
    "1080p_default": (1920, 1080, 4, 8, dict(TUNE, box_size=100), {}),
    "640x480_default": (640, 480, 2, 8, dict(TUNE, box_size=100), {}),
    "640x480_ratio2": (640, 480, 2, 8, dict(TUNE, box_size=320), {}),
    "80x60_upscale": (80, 60, 2, 8, dict(TUNE, box_size=100), dict(upscale=True)),
    "1000x562_k5_not_fusable": (1000, 562, 2, 8, dict(TUNE, box_size=1000, blur_scale=200), {}),
    # W % 8 != 0: the byte path of k_nv12_bgr
    "642x362_default": (642, 362, 2, 8, dict(TUNE, box_size=100), {}),
    "100x76_upscale": (100, 76, 2, 8, dict(TUNE, box_size=160), dict(upscale=True)),
}


@pytest.mark.parametrize("name", list(CONFIGS))
def test_nv12_equals_bgr_of_cv2_conversion(name):
    W, H, S, T, kw, ekw = CONFIGS[name]
    info = _compare(W, H, S, T, kw, ekw)
    if name == "1000x562_k5_not_fusable":
        assert info["gaussian"] == 5 and info["front_end"] == 1
    if name.endswith("_fused") or name in ("720p_k5_T32", "4k_k5"):
        assert info["front_end"] == 0


@pytest.mark.parametrize("name", ["1080p_k5_fused", "640x480_default"])
def test_nv12_keep_planes(name):
    W, H, _, _, kw, ekw = CONFIGS[name]
    _compare(W, H, 2, 4, kw, ekw, keep=True)


@pytest.mark.parametrize("W,H,kw", [(256, 192, dict(TUNE, box_size=256, blur_scale=64)),
                                    (320, 240, dict(TUNE, box_size=100))])
def test_planes_match_cv2_chain(W, H, kw):
    """KEEP_PLANES gray and blur, the threshold plane and the background against the reference's cv2 chain run on the
    converted frames."""
    import torch
    from find_motion_b200.engine import MotionEngine
    from oracle import cv2_chain
    T, n = 8, 24
    nv = _nv12_clips(W, H, 1, n, kw["fps"])
    bgr = _twin(nv)
    ref = cv2_chain.Cv2Stream(W, H, **kw)
    with MotionEngine(W, H, n_streams=1, max_frames=T, nv12=True, keep_planes=True, **kw) as eng:
        for t0 in range(0, n, T):
            eng.process(torch.from_numpy(nv[:, t0:t0 + T]).cuda())
            for t in range(T):
                want = ref.step(bgr[0, t0 + t])
                pl = eng.planes(0, t, bg=(t == T - 1))
                for key in ("gray", "blur"):
                    assert (pl[key] == want[key]).all(), (key, t0 + t)
                # fm_debug_planes gives the dilated threshold plane as 0 / 1
                assert ((pl["thresh"] != 0) == (want["thresh"] != 0)).all(), ("thresh", t0 + t)
            assert (pl["bg"] == ref.ref_frame).all(), ("bg", t0)


def test_launches_of_fused_and_staged_paths():
    """The fused path really runs: the 1080p k=5 NV12 context keeps front_end == 0 and adds the same launches per call
    as the BGR fused context.  A staged configuration adds exactly one (the conversion kernel)."""
    import torch
    from find_motion_b200.engine import MotionEngine, launch_count

    def delta(fn):
        torch.cuda.synchronize()
        n = launch_count()
        fn()
        torch.cuda.synchronize()
        return launch_count() - n

    for W, H, kw, front_end, extra in ((1920, 1080, dict(TUNE, box_size=1920, blur_scale=384), 0, 0),
                                       (640, 480, dict(TUNE, box_size=100), 2, 1),
                                       (1000, 562, dict(TUNE, box_size=1000, blur_scale=200), 1, 1)):
        S, T = 2, 4
        nv = _nv12_clips(W, H, S, T, kw["fps"])
        b_nv, b_bgr = torch.from_numpy(nv).cuda(), torch.from_numpy(_twin(nv)).cuda()
        with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, **kw) as eng, \
                MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as ref:
            assert eng.info["front_end"] == ref.info["front_end"] == front_end
            for _ in range(2):
                assert delta(lambda: eng.process(b_nv)) == delta(lambda: ref.process(b_bgr)) + extra, (W, H)


def test_strides_not_multiples_of_8():
    """Padded strides (frame stride and stream stride not multiples of 8) on the staged path and on the fused one,
    where they are refused: the fused NV12 front end reads its frames by TMA, which needs 16-byte aligned strides, as
    the BGR one does."""
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    for W, H, kw, fused in ((640, 480, dict(TUNE, box_size=100), False),
                            (256, 192, dict(TUNE, box_size=256, blur_scale=64), True)):
        S, T = 2, 8
        nv = _nv12_clips(W, H, S, 2 * T, kw["fps"])
        fb = W * H * 3 // 2
        fstride = fb + 4
        sstride = T * fstride + 2
        raw = torch.zeros(S * sstride + 64, dtype=torch.uint8, device="cuda")
        frames = raw.as_strided((S, T, H * 3 // 2, W), (sstride, fstride, W, 1), 6)
        with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, **kw) as eng, \
                MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as ref:
            for t0 in (0, T):
                frames.copy_(torch.from_numpy(nv[:, t0:t0 + T]).cuda())
                want = ref.process(torch.from_numpy(_twin(nv[:, t0:t0 + T])).cuda())
                if fused:
                    with pytest.raises(_lib.FmError) as e:
                        eng.process(frames)
                    assert e.value.code == -1
                    break
                assert (eng.process(frames) == want).all(), t0
                for s in range(S):
                    for t in range(T):
                        assert eng.components(s, t) == ref.components(s, t), (t0, s, t)


def _run_clips(W, H, S, n, T, kw, nvalid=None):
    """process_clip of an NV12 context: every clip frame must be, byte for byte, the NV12 input frame the schedule of
    tests/clips_restated.py names; the stats must equal a BGR context's on the converted frames."""
    import torch
    from find_motion_b200.engine import MotionEngine
    clips = _nv12_clips(W, H, S, n, kw["fps"], seed=23)
    flushed = 0
    with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, device_clips=True, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as ref:
        C = eng.info["cache_frames"]
        rings = [CR.RingSim(C) for _ in range(S)]
        fed = [[] for _ in range(S)]
        pos, i = [0] * S, 0
        while min(n - p for p in pos) > 0:
            nv = [min(v, n - p) for v, p in zip(nvalid(i) if nvalid else [T] * S, pos)]
            b = _batch(clips, pos, nv, T)
            stats, out = eng.process_clip(torch.from_numpy(b).cuda(), n_valid=nv)
            assert (stats == ref.process(torch.from_numpy(_twin(b)).cuda(), n_valid=nv)).all(), i
            for s in range(S):
                fed[s] += range(pos[s], pos[s] + nv[s])
                ids = rings[s].call(stats[s], nv[s])
                got = out[s].cpu().numpy()
                assert got.shape == (len(ids), H * 3 // 2, W), (s, got.shape)
                if ids:
                    assert np.array_equal(got, clips[s][[fed[s][j] for j in ids]]), (i, s, ids)
                flushed += int(stats[s]["n_flush"][:nv[s]].sum())
            pos = [p + v for p, v in zip(pos, nv)]
            i += 1
    return C, flushed


def test_clips_fused_geometry():
    C, flushed = _run_clips(256, 192, 2, 48, 8, dict(TUNE, box_size=256, blur_scale=64))
    assert flushed > 0


def test_clips_call_longer_than_the_cache_ragged():
    rng = np.random.default_rng(5)
    sched = [[int(v) for v in rng.integers(0, 33, size=3)] for _ in range(20)]
    sched[0] = [32, 0, 20]
    kw = dict(fps=30, threshold=12, avg=0.3, min_time=0.04, cache_time=0.1, box_size=100)
    C, flushed = _run_clips(160, 120, 3, 96, 32, kw, nvalid=lambda i: sched[i])
    assert C == 3 and flushed > 0


@pytest.mark.parametrize("W,H,kw", [(1920, 1080, dict(TUNE, box_size=1920, blur_scale=384)),
                                    (640, 480, dict(TUNE, box_size=100))])
def test_host_entry_points(W, H, kw):
    """fm_process_host and fm_submit_host / fm_wait on pinned NV12 batches give the stats of the device path."""
    import torch
    from find_motion_b200.engine import MotionEngine, PinnedBatch
    S, T = 2, 8
    clips = _nv12_clips(W, H, S, 3 * T, kw["fps"])
    pin = [PinnedBatch((S, T, H * 3 // 2, W)) for _ in range(2)]
    with MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, **kw) as host, \
            MotionEngine(W, H, n_streams=S, max_frames=T, nv12=True, **kw) as dev:
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
