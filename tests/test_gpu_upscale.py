"""GPU: frames narrower than box_size (FM_FLAG_UPSCALE, csrc/k_upscale.cu).  The gray plane against cv2's own
resize + cvtColor, whole calls against the cv2 call chain (dilated threshold, stats, contour records, float64
background), the host entry points, the job driver over a folder that mixes a downscaled and an upscaled geometry,
and the detector input plane.  Exact equality throughout."""
import functools

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _want_gray(cv2, frame, box):
    H, W = frame.shape[:2]
    small = cv2.resize(frame, (box, int(H * (box / float(W)))), interpolation=cv2.INTER_AREA)
    return cv2.cvtColor(small, cv2.COLOR_BGR2GRAY)


def test_flag_is_required():
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    with pytest.raises(_lib.FmError) as e:
        MotionEngine(80, 60, box_size=100)
    assert e.value.code == -4
    with MotionEngine(80, 60, box_size=100, upscale=True) as eng:
        assert (eng.w, eng.h, eng.info["front_end"], eng.info["scale"]) == (100, 75, 2, 1.25)
    with MotionEngine(640, 480, box_size=320, upscale=True) as eng:      # the flag changes nothing when downscaling
        assert eng.info["front_end"] == 2


GRAY_GEOMS = [(80, 60, 100), (64, 48, 100), (97, 31, 100), (320, 240, 640), (640, 480, 800), (333, 217, 1000),
              (1280, 720, 1920), (1920, 1080, 3840)]


@pytest.mark.parametrize("W,H,box", GRAY_GEOMS)
def test_gray_plane_matches_cv2(W, H, box):
    cv2 = pytest.importorskip("cv2")
    import torch
    from find_motion_b200.engine import MotionEngine
    rng = np.random.default_rng(W + box)
    S, T = 1, 2
    frames = rng.integers(0, 256, size=(S, T, H, W, 3), dtype=np.uint8)
    frames[0, 1, : H // 2] = 255
    with MotionEngine(W, H, n_streams=S, max_frames=T, box_size=box, keep_planes=True, upscale=True) as eng:
        eng.process(torch.from_numpy(frames).cuda())
        for t in range(T):
            got = eng.planes(0, t, blur=False, thresh=False, bg=False)["gray"]
            want = _want_gray(cv2, frames[0, t], box)
            assert got.shape == want.shape and (got == want).all(), (t, int((got != want).sum()))


def test_gray_plane_ragged_odd_batch_and_strided_frames():
    """S = 3, T = 5 with n_valid = [5, 0, 3], frames taken from a wider batch (stream stride != T * frame bytes)."""
    cv2 = pytest.importorskip("cv2")
    import torch
    from find_motion_b200.engine import MotionEngine
    W, H, box, S, T = 150, 101, 301, 3, 5
    rng = np.random.default_rng(11)
    big = rng.integers(0, 256, size=(S, T + 2, H, W, 3), dtype=np.uint8)
    dev = torch.from_numpy(big).cuda()[:, 1:T + 1]
    nv = [5, 0, 3]
    with MotionEngine(W, H, n_streams=S, max_frames=T, box_size=box, keep_planes=True, upscale=True) as eng:
        stats = eng.process(dev, n_valid=nv)
        for s in range(S):
            for t in range(nv[s]):
                got = eng.planes(s, t, blur=False, thresh=False, bg=False)["gray"]
                assert (got == _want_gray(cv2, big[s, t + 1], box)).all(), (s, t)
            for t in range(nv[s], T):
                assert tuple(stats[s, t]) == (0,) * 8


def _records(cv2, thresh):
    cnts = cv2.findContours(thresh, mode=cv2.RETR_EXTERNAL, method=cv2.CHAIN_APPROX_SIMPLE)[-2]
    return sorted((int(round(2 * cv2.contourArea(c))), tuple(int(v) for v in cv2.boundingRect(c))) for c in cnts)


def _parity(W, H, n, T, kw, seed, **engine_kw):
    cv2 = pytest.importorskip("cv2")
    import torch
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine
    from oracle import cv2_chain
    clip = synth.make_clip(W, H, n, seed=seed, fps=kw.get("fps", 30),
                           script=[("walker", 2, n), ("blip", 1, 4), ("hidden", 0, n)])
    ref = cv2_chain.Cv2Stream(W, H, **kw)
    dev = torch.from_numpy(clip[None]).cuda()
    moved = 0
    with MotionEngine(W, H, n_streams=1, max_frames=T, upscale=True, **engine_kw, **kw) as eng:
        assert eng.info["front_end"] == 2
        for t0 in range(0, n, T):
            t1 = min(n, t0 + T)
            stats = eng.process(dev[:, t0:t1])
            for t in range(t0, t1):
                want = ref.step(clip[t])
                pl = eng.planes(0, t - t0, gray=False, blur=False, bg=False)
                assert (pl["thresh"] == want["thresh"]).all(), (t, int((pl["thresh"] != want["thresh"]).sum()))
                n_all, comps = eng.components(0, t - t0)
                assert n_all == len(comps) and comps == _records(cv2, want["thresh"]), t
                st = stats[0, t - t0]
                assert (int(st["n_contours"]), bool(st["movement"]), int(st["movement_counter"]), int(st["movement_decay"]),
                        int(st["cache_len"]), bool(st["wrote"]), int(st["n_flush"])) == \
                    (len(want["areas"]), want["movement"], want["counter"], want["decay"], want["cache_len"], want["wrote"],
                     want["n_flush"]), t
                moved += bool(want["movement"])
            bg = eng.planes(0, t1 - 1 - t0, gray=False, blur=False, thresh=False)["bg"]
            assert (bg == ref.ref_frame).all(), ("bg", t1)
    assert moved > 0


def test_parity_low_res_camera_default_box():
    _parity(80, 60, 20, 4, dict(fps=6, box_size=100, blur_scale=20, threshold=8, avg=0.2, min_time=0.3, cache_time=0.6),
            seed=51)


@pytest.mark.parametrize("blur_scale", [384, 20])          # k = 5 and k = 97
def test_parity_720p_to_1920_with_masks(blur_scale):
    masks = [((0, 0), (100, 100)), ((0, 0), (0, 100), (100, 0)), ((900, 100), (1100, 300)), ((200, 450), (200, 650), (450, 450))]
    _parity(1280, 720, 8, 4, dict(fps=6, box_size=1920, blur_scale=blur_scale, threshold=8, avg=0.15, min_time=0.3,
                                  cache_time=0.6, mask_areas=masks), seed=52)


@pytest.mark.parametrize("path", ["umma", "no_umma"])
def test_parity_640x480_to_800_both_blur_paths(path):
    _parity(640, 480, 10, 5, dict(fps=6, box_size=800, blur_scale=20, threshold=8, avg=0.2, min_time=0.3, cache_time=0.6),
            seed=53, **{path: True})


def test_host_entry_points_equal_device_entry_point():
    import torch
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine
    W, H, S, T, n = 96, 54, 2, 4, 16
    kw = dict(fps=6, box_size=160, blur_scale=20, threshold=8, avg=0.2, min_time=0.3, cache_time=0.6, upscale=True)
    clips = np.stack([synth.make_clip(W, H, n, seed=60 + s, fps=6) for s in range(S)])
    with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as a, MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as b, \
            MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as c:
        pend = None
        want, got_c = [], []
        for i, t0 in enumerate(range(0, n, T)):
            batch = np.ascontiguousarray(clips[:, t0:t0 + T])
            sa = a.process(torch.from_numpy(batch).cuda())
            sb = b.process_host(batch)
            c.submit_host(i & 1, batch)
            if pend is not None:
                got_c.append(c.wait_host(pend))
            pend = i & 1
            assert (sa == sb).all(), t0
            want.append(sa)
            for s in range(S):
                for t in range(T):
                    assert a.components(s, t) == b.components(s, t)
        got_c.append(c.wait_host(pend))
        assert len(got_c) == len(want) == n // T and all((x == y).all() for x, y in zip(want, got_c))
        assert (a.planes(1, T - 1, gray=False, blur=False, thresh=False)["bg"] ==
                b.planes(1, T - 1, gray=False, blur=False, thresh=False)["bg"]).all()


def test_run_pool_mixed_down_and_upscaled_files(tmp_path, monkeypatch):
    """192x108 files (downscaled to 96) and 64x48 files (upscaled to 96) in one folder: every result tuple and every
    written frame as the oracle loop gives them.  Before the upscale path existed, the 64x48 files came back as
    error tuples."""
    cv2 = pytest.importorskip("cv2")
    from find_motion_b200 import jobs
    from find_motion_b200.video_motion import run_vid
    from tests.test_jobs_host_logic import KW, _clips, expected_writes
    from tests.upscale_restated import use_in_oracle
    use_in_oracle(monkeypatch)                 # expected_writes runs the oracle on the 64x48 clips too
    spec = {"big0": (192, 108, 30, 71), "small0": (64, 48, 26, 72), "big1": (192, 108, 12, 73), "small1": (64, 48, 40, 74)}
    clips = _clips(spec)
    paths = {}
    for name, clip in clips.items():
        p = str(tmp_path / (name + ".avi"))
        wr = cv2.VideoWriter(p, cv2.VideoWriter_fourcc(*"FFV1"), 6, (clip.shape[2], clip.shape[1]))
        if not wr.isOpened():
            pytest.skip("FFV1 writer not available in this cv2 build")
        for f in clip:
            wr.write(f)
        wr.release()
        paths[p] = name
    for p, name in paths.items():
        cap = cv2.VideoCapture(p)
        ok, first = cap.read()
        cap.release()
        if not ok or not (first == clips[name][0]).all():
            pytest.skip("FFV1 round trip is not lossless here")
    outdir = tmp_path / "out"
    outdir.mkdir()
    kw = dict(KW, box_size=96, outdir=str(outdir), codec="FFV1")
    res = jobs.run_pool(functools.partial(run_vid, **kw), 4, list(paths), devices=[0], streams=2, chunk=8)
    assert sorted(r[1] for r in res) == sorted(paths)
    tun = {k: v for k, v in kw.items() if k not in ("outdir", "codec")}
    n_written = 0
    for wrote, path, err, objs in res:
        name = paths[path]
        want = expected_writes(clips[name], tun)
        assert err == "" and objs == () and wrote == (len(want) > 0), (name, err)
        outs = sorted(outdir.glob(name + ".avi_*_motion.avi"))
        assert len(outs) == (1 if want else 0), name
        if want:
            cap = cv2.VideoCapture(str(outs[0]))
            got = []
            while True:
                ok, f = cap.read()
                if not ok:
                    break
                got.append(f)
            cap.release()
            assert len(got) == len(want), name
            for f, t in zip(got, want):
                assert (f == clips[name][t]).all(), (name, t)
            n_written += name.startswith("small")
    assert n_written > 0                     # an upscaled file wrote motion segments


@pytest.mark.parametrize("W", [80, 160, 299])
def test_detector_input_plane_upscaled(W):
    cv2 = pytest.importorskip("cv2")
    from find_motion_b200 import synth
    from find_motion_b200.engine import resize_area
    H = W * 3 // 4 + 1
    frame = synth.make_clip(W, H, 1, seed=W)[0]
    want = cv2.resize(frame, (300, int(H * (300 / float(W)))), interpolation=cv2.INTER_AREA)
    got = resize_area(frame, 300)
    assert got.shape == want.shape and (got == want).all(), int((got != want).sum())
