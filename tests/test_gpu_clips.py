"""GPU: the device-side look-back cache and fm_process_clip (FM_FLAG_DEVICE_CLIPS, csrc/k_clips.cu).  Every frame
process_clip hands out is compared byte for byte with the seeded synthetic frame that the schedule of
tests/clips_restated.py names, and that schedule with a deque(maxlen=cache_frames) replay of the reference."""
import numpy as np
import pytest

from find_motion_b200 import synth
from tests import clips_restated as CR

pytestmark = pytest.mark.gpu

TUNE = dict(fps=8, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)


def _clips(W, H, S, N, fps, scripts=None, seed=11):
    return np.stack([synth.make_clip(W, H, N, seed=synth.stream_seed(seed, s), fps=fps,
                                     script=None if scripts is None else scripts[s]) for s in range(S)])


class Checker:
    """Ring simulation + deque replay of every stream, fed the stats of every call in order.  fed[s] lists the clip
    frame behind each absolute frame id of stream s."""

    def __init__(self, clips, C):
        self.clips = clips
        self.rings = [CR.RingSim(C) for _ in range(len(clips))]
        self.deques = [CR.DequeReplay(C) for _ in range(len(clips))]
        self.fed = [[] for _ in range(len(clips))]
        self.hazards = 0                  # calls in which a store overwrites a slot a gather of the same call reads
        self.reach = 0                    # most calls back a flushed frame came from
        self.flushed = 0

    def reset(self, s):
        self.deques[s].reset()

    def call(self, stats, n_valid, first, clips_out=None, T=None):
        """first[s]: clip index of the first frame stream s carried in this call (its frames are consecutive)."""
        for s in range(len(self.clips)):
            nv = int(n_valid[s])
            ring = self.rings[s]
            gather, store, _ = CR.schedule(stats[s], nv, ring.base, ring.C)
            ring_slots = {src[1] for src, _ in gather if src[0] == "ring"}
            self.hazards += bool(ring_slots & {slot for _, slot in store})
            if T and gather:
                self.reach = max(self.reach, max((ring.base - b + T - 1) // T for _, b in gather))
            self.flushed += int(stats[s]["n_flush"][:nv].sum())
            self.fed[s] += range(first[s], first[s] + nv)
            ids = ring.call(stats[s], nv)
            assert ids == [i for rec in stats[s][:nv] for i in self.deques[s].frame(rec)], s
            if clips_out is not None:
                got = clips_out[s].cpu().numpy()
                assert got.shape[0] == len(ids), (s, got.shape, len(ids))
                if ids:
                    assert np.array_equal(got, self.clips[s][[self.fed[s][i] for i in ids]]), (s, ids)


def _batch(dev, pos, nv, T):
    """[S, T, H, W, 3] of the next nv[s] frames of each stream (zeros past n_valid)."""
    import torch
    S = dev.shape[0]
    b = torch.zeros((S, T) + tuple(dev.shape[2:]), dtype=torch.uint8, device=dev.device)
    for s in range(S):
        if nv[s]:
            b[s, :nv[s]] = dev[s, pos[s]:pos[s] + nv[s]]
    return b


def _run(W, H, S, N, T, kw, ekw=None, scripts=None, nvalid=None, compare_stats=True):
    """Drive process_clip over N frames per stream in calls of T (nvalid(i) -> per-stream counts of call i) and check
    every output frame; the stats are also compared with process() on a context without the flag."""
    import torch
    from find_motion_b200.engine import MotionEngine
    clips = _clips(W, H, S, N, kw["fps"], scripts)
    dev = torch.from_numpy(clips).cuda()
    ekw = ekw or {}
    with MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **ekw, **kw) as eng, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **ekw, **kw) as ref:
        chk = Checker(clips, eng.info["cache_frames"])
        pos, i = [0] * S, 0
        while min(N - p for p in pos) > 0:
            nv = list(nvalid(i)) if nvalid else [T] * S
            nv = [min(v, N - p) for v, p in zip(nv, pos)]
            batch = _batch(dev, pos, nv, T)
            stats, out = eng.process_clip(batch, n_valid=nv)
            if compare_stats:
                want = ref.process(batch, n_valid=nv)
                assert (stats == want).all(), i
            chk.call(stats, nv, pos, out, T)
            pos = [p + v for p, v in zip(pos, nv)]
            i += 1
    return chk


def test_default_mode():
    chk = _run(320, 240, 2, 48, 8, dict(TUNE, box_size=100))
    assert chk.flushed > 0


def test_full_resolution_fused_k5():
    chk = _run(256, 192, 2, 48, 8, dict(TUNE, box_size=256, blur_scale=64))
    assert chk.flushed > 0


def test_full_resolution_wide_k97():
    chk = _run(388, 240, 1, 40, 8, dict(TUNE, box_size=388, blur_scale=4))
    assert chk.flushed > 0


def test_upscaled_geometry():
    chk = _run(80, 60, 2, 48, 8, dict(TUNE, box_size=100), ekw=dict(upscale=True))
    assert chk.flushed > 0


def test_1080p_cache_longer_than_a_call():
    """8 streams x 16 frames of 1080p, cache_time 1 s at 30 fps: C = 30 > T, and flushes reach back two calls."""
    scripts = [[("walker", 38 + s % 4, 48)] for s in range(8)]
    chk = _run(1920, 1080, 8, 48, 16, dict(fps=30, threshold=12, avg=0.1, min_time=0.1, cache_time=1.0, box_size=100),
               scripts=scripts, compare_stats=False)
    assert chk.reach >= 2, chk.reach


def test_short_cache_long_call():
    """C = 3 with T = 32: several flushes per call, the cache overflowing inside a call, and stores into slots a flush
    of the same call reads (the gathers must run first)."""
    scripts = [[("blip", 5 + s, 8 + s), ("blip", 20, 23), ("blip", 33 + s % 2, 36 + s % 2), ("blip", 50, 53),
                ("blip", 65 - s % 2, 68 - s % 2)] for s in range(4)]
    chk = _run(160, 120, 4, 96, 32, dict(fps=30, threshold=12, avg=0.3, min_time=0.04, cache_time=0.1, box_size=160,
                                         blur_scale=32), scripts=scripts)
    assert chk.flushed > 0 and chk.hazards > 0, (chk.flushed, chk.hazards)


def test_no_cache_and_no_min_time():
    chk = _run(160, 120, 2, 24, 8, dict(TUNE, box_size=100, cache_time=0.0))          # C = 0: no ring at all
    assert chk.flushed == 0
    chk = _run(160, 120, 2, 24, 8, dict(TUNE, box_size=100, min_time=0.0))            # every frame written
    assert chk.flushed == 0


def test_ragged_batches():
    rng = np.random.default_rng(3)
    sched = [[int(v) for v in rng.integers(0, 9, size=3)] for _ in range(40)]
    sched[0] = [8, 0, 3]
    chk = _run(160, 120, 3, 48, 8, dict(TUNE, box_size=100), nvalid=lambda i: sched[i])
    assert chk.flushed > 0


def test_single_frame_calls():
    chk = _run(160, 120, 2, 40, 1, dict(TUNE, box_size=100))
    assert chk.flushed > 0


def test_unaligned_frames():
    """203 x 117: H*W*3 is odd, so neither the output frames nor the input frames are 16-byte aligned."""
    chk = _run(203, 117, 2, 40, 8, dict(TUNE, box_size=203, blur_scale=20))
    assert chk.flushed > 0


def test_padded_strides():
    import torch
    from find_motion_b200.engine import MotionEngine
    W, H, S, N, T = 160, 120, 2, 40, 8
    kw = dict(TUNE, box_size=100)
    clips = _clips(W, H, S, N, kw["fps"])
    fb = W * H * 3
    fstride, sstride = fb + 37, T * (fb + 37) + 101
    raw = torch.zeros(S * sstride + 64, dtype=torch.uint8, device="cuda")
    frames = raw.as_strided((S, T, H, W, 3), (sstride, fstride, W * 3, 3, 1), 7)
    cap = 8 + T + 3
    outbuf = torch.zeros(S * (cap * fb + 5) + 16, dtype=torch.uint8, device="cuda")
    out = outbuf.as_strided((S, cap, H, W, 3), (cap * fb + 5, fb, W * 3, 3, 1), 3)
    with MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **kw) as eng:
        chk = Checker(clips, eng.info["cache_frames"])
        for t0 in range(0, N, T):
            frames.copy_(torch.from_numpy(clips[:, t0:t0 + T]).cuda())
            stats, got = eng.process_clip(frames, out=out)
            chk.call(stats, [T] * S, [t0] * S, got)
    assert chk.flushed > 0


def test_mixed_entry_points_and_reset():
    """process_host, submit_host / wait_host, plain process and submit_reset between process_clip calls: the frames
    those calls cached come out of later flushes."""
    import torch
    from find_motion_b200.engine import MotionEngine
    W, H, S, T, N = 160, 120, 2, 8, 96
    kw = dict(TUNE, box_size=100)
    clips = _clips(W, H, S, N, kw["fps"])
    plan = ["clip", "host", "clip", "submit", "process", "clip", "reset", "clip", "submit_ragged", "clip", "process",
            "clip"]
    with MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **kw) as eng:
        chk = Checker(clips, eng.info["cache_frames"])
        pos = [0] * S                                       # next clip frame of each stream
        for step in plan:
            if step == "reset":
                eng.submit_reset(1)
                torch.cuda.synchronize()
                chk.reset(1)
                continue
            nv = [T, 5] if step == "submit_ragged" else [T] * S      # stream 1 carries 5 frames there
            batch = np.stack([clips[s, pos[s]:pos[s] + T] for s in range(S)])
            if step == "clip":
                stats, out = eng.process_clip(torch.from_numpy(batch).cuda())
                chk.call(stats, nv, pos, out)
            elif step == "host":
                chk.call(eng.process_host(batch), nv, pos)
            elif step in ("submit", "submit_ragged"):
                eng.submit_host(1, batch, n_valid=nv)
                chk.call(eng.wait_host(1), nv, pos)
            elif step == "process":
                chk.call(eng.process(torch.from_numpy(batch).cuda()), nv, pos)
            pos = [p + v for p, v in zip(pos, nv)]
    assert chk.flushed > 0


def test_refusals_and_launch_counts():
    import torch
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine, launch_count
    W, H, S, T = 160, 120, 2, 8
    kw = dict(TUNE, box_size=100)
    frames = torch.from_numpy(_clips(W, H, S, T, kw["fps"])).cuda()
    with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as plain, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **kw) as eng:
        with pytest.raises(_lib.FmError) as e:
            plain.process_clip(frames)
        assert e.value.code == -1
        C = eng.info["cache_frames"]
        small = torch.empty((S, C + T - 1, H, W, 3), dtype=torch.uint8, device="cuda")
        with pytest.raises(_lib.FmError) as e:
            eng.process_clip(frames, out=small)
        assert e.value.code == -1
        eng.process_clip(frames, out=torch.empty((S, C + T, H, W, 3), dtype=torch.uint8, device="cuda"))

        def delta(fn):
            n = launch_count()
            fn()
            torch.cuda.synchronize()
            return launch_count() - n

        d_plain = delta(lambda: plain.process(frames))
        assert delta(lambda: plain.process(frames)) == d_plain
        assert delta(lambda: eng.process(frames)) == d_plain + 2          # plan + ring stores
        assert delta(lambda: eng.process_clip(frames)) == d_plain + 3     # plan + gathers + ring stores


def test_motion_avi_matches_run_vid(tmp_path):
    """run_vid (host path) writes *_motion.avi from an FFV1 clip; writing the clips of the device path with
    cv2.VideoWriter (FFV1) gives a file that decodes to the same frames."""
    cv2 = pytest.importorskip("cv2")
    import torch
    from find_motion_b200.engine import MotionEngine
    from find_motion_b200.video_motion import run_vid
    from tests import helpers
    fx = helpers.load_golden("full_256x192_k5")
    clip = helpers.golden_clip(fx)
    W, H, fps = fx["clip"]["W"], fx["clip"]["H"], fx["kwargs"]["fps"]
    src = str(tmp_path / "clip.avi")
    wr = cv2.VideoWriter(src, cv2.VideoWriter_fourcc(*"FFV1"), fps, (W, H))
    if not wr.isOpened():
        pytest.skip("FFV1 writer not available in this cv2 build")
    for f in clip:
        wr.write(f)
    wr.release()
    cap = cv2.VideoCapture(src)
    decoded = []
    while True:
        ok, f = cap.read()
        if not ok:
            break
        decoded.append(f)
    cap.release()
    if len(decoded) != len(clip) or not all((a == b).all() for a, b in zip(decoded, clip)):
        pytest.skip("FFV1 round trip is not lossless here")
    outdir = tmp_path / "out"
    outdir.mkdir()
    wrote, _, err, _ = run_vid(src, **dict(fx["kwargs"], outdir=str(outdir), codec="FFV1", chunk=8))
    assert err == "" and wrote is True
    host_avi = sorted(outdir.glob("*_motion.avi"))[0]

    T = 8
    dev_avi = str(tmp_path / "device_motion.avi")
    wr = cv2.VideoWriter(dev_avi, cv2.VideoWriter_fourcc(*"FFV1"), fps, (W, H))
    frames = torch.from_numpy(np.stack(decoded)).cuda()
    with MotionEngine(W, H, n_streams=1, max_frames=T, device_clips=True, **fx["kwargs"]) as eng:
        for t0 in range(0, len(decoded), T):
            _, clips = eng.process_clip(frames[None, t0:t0 + T])
            for f in clips[0].cpu().numpy():            # only the written frames leave the GPU
                wr.write(f)
    wr.release()

    def read_all(path):
        cap = cv2.VideoCapture(str(path))
        out = []
        while True:
            ok, f = cap.read()
            if not ok:
                break
            out.append(f)
        cap.release()
        return out

    a, b = read_all(host_avi), read_all(dev_avi)
    assert len(a) == len(b) == fx["writes"] > 0
    assert all((x == y).all() for x, y in zip(a, b))
