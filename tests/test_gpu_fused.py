"""GPU parity of the fused stencil+background kernel (K1): tile borders, partial tiles, k in {1,3,5},
full 1080p frames, and A/B equality with the generic multi-kernel front end."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _compare_with_oracle(W, H, n, T, kw, seed, n_streams=1, no_fused=False):
    import torch
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine
    from oracle import restated as R
    clips = np.stack([synth.make_clip(W, H, n, seed=seed + s, fps=kw.get("fps", 30)) for s in range(n_streams)])
    orcs = [R.StreamOracle(W, H, **kw) for _ in range(n_streams)]
    dev = torch.from_numpy(clips).cuda()
    with MotionEngine(W, H, n_streams=n_streams, max_frames=T, keep_planes=True, no_fused=no_fused, **kw) as eng:
        assert eng.info["front_end"] == (1 if no_fused else 0), "fused front end expected unless switched off"
        for t0 in range(0, n, T):
            t1 = min(n, t0 + T)
            stats = eng.process(dev[:, t0:t1])
            for s in range(n_streams):
                for t in range(t0, t1):
                    rec = orcs[s].process(clips[s, t], keep_planes=True)
                    pl = eng.planes(s, t - t0, bg=(t == t1 - 1))
                    for key in ("gray", "blur", "thresh"):
                        assert (pl[key] == rec["planes"][key]).all(), (key, s, t, np.argwhere(pl[key] != rec["planes"][key])[:4])
                    if t == t1 - 1:
                        assert (pl["bg"] == rec["planes"]["bg"]).all(), ("bg", s, t)
                    _, comps = eng.components(s, t - t0)
                    assert sorted(a / 2.0 for a, _ in comps) == rec["areas"], (s, t)
                    st = stats[s, t - t0]
                    assert (bool(st["movement"]), int(st["movement_counter"]), int(st["movement_decay"]),
                            bool(st["wrote"]), int(st["n_flush"]), int(st["cache_len"])) == \
                        (rec["movement"], rec["counter"], rec["decay"], rec["wrote"], rec["n_flush"], rec["cache_len"])


@pytest.mark.parametrize("W,H", [(160, 120), (128, 64), (32, 4), (256, 70), (96, 200), (288, 130)])
def test_fused_tile_borders(W, H):
    kw = dict(fps=6, box_size=W, blur_scale=W // 5, threshold=8, avg=0.15, min_time=0.4, cache_time=1.0,
              min_box_scale=50, mask_areas=[((3, 2), (W // 3, H // 2)), ((W // 2, 0), (W - 1, H // 3), (W // 2, H - 1))])
    _compare_with_oracle(W, H, 14, 5, kw, seed=31)


@pytest.mark.parametrize("k,blur_scale", [(1, 160), (3, 53), (5, 32)])
def test_fused_kernel_sizes(k, blur_scale):
    from oracle import restated as R
    kw = dict(fps=6, box_size=160, blur_scale=blur_scale, threshold=6, avg=0.3, min_time=0.3, cache_time=0.5)
    assert R.derive_params(160, 120, **{a: kw[a] for a in ("fps", "box_size", "blur_scale")})["gaussian"] == k
    _compare_with_oracle(160, 120, 12, 4, kw, seed=40 + k)


def test_fused_avg_out_of_unit_range_still_exact():
    """avg > 1 makes the background leave [0, 255]: the saturating/abs path of convertScaleAbs.  A negative threshold sets
    every threshold bit.  Both take the variant of K1 without the carry form of the threshold test; the negative threshold
    also runs through the generic front end at k = 5 (mma.sync Gaussian, then the separate temporal kernel)."""
    for avg, threshold in ((1.7, 6), (0.3, -1)):
        kw = dict(fps=6, box_size=128, blur_scale=32, threshold=threshold, avg=avg, min_time=0.3, cache_time=0.5)
        _compare_with_oracle(128, 96, 10, 5, kw, seed=77)
    _compare_with_oracle(128, 96, 10, 5, kw, seed=78, no_fused=True)


def test_fused_multi_stream_1080p():
    from find_motion_b200 import synth
    kw = dict(fps=30, box_size=1920, blur_scale=384, threshold=12, avg=0.1, min_time=0.1, cache_time=0.2,
              mask_areas=synth.CFG2_MASKS)
    _compare_with_oracle(1920, 1080, 6, 3, kw, seed=2000, n_streams=2)


def test_fused_equals_generic_front_end():
    import torch
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine
    W, H, n, T = 640, 360, 24, 8
    kw = dict(fps=10, box_size=640, blur_scale=128, threshold=10, avg=0.1, min_time=0.3, cache_time=0.6,
              mask_areas=synth.README_MASKS)
    clips = np.stack([synth.make_clip(W, H, n, seed=90 + s, fps=10) for s in range(3)])
    dev = torch.from_numpy(clips).cuda()
    with MotionEngine(W, H, n_streams=3, max_frames=T, **kw) as a, \
            MotionEngine(W, H, n_streams=3, max_frames=T, no_fused=True, **kw) as b:
        assert a.info["front_end"] == 0 and b.info["front_end"] == 1
        for t0 in range(0, n, T):
            sa, sb = a.process(dev[:, t0:t0 + T]), b.process(dev[:, t0:t0 + T])
            assert (sa == sb).all()
            for s in range(3):
                pa, pb = a.planes(s, T - 1, gray=False, blur=False), b.planes(s, T - 1, gray=False, blur=False)
                assert (pa["thresh"] == pb["thresh"]).all() and (pa["bg"] == pb["bg"]).all()
