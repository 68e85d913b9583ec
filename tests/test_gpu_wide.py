"""GPU parity of the tensor-core wide Gaussian (k_wide.cu): kernel radii below / at / above the plane size,
16-byte-aligned BGR staging and the gray-plane staging, border tiles, partial column tiles, row-group padding,
and the resize front end feeding it.  Everything compared for exact equality with the oracle."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _run(W, H, n, T, kw, seed, n_streams=1, expect_front_end=None, **engine_kw):
    import torch
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine
    from oracle import restated as R
    clips = np.stack([synth.make_clip(W, H, n, seed=seed + s, fps=kw.get("fps", 30)) for s in range(n_streams)])
    orcs = [R.StreamOracle(W, H, **kw) for _ in range(n_streams)]
    dev = torch.from_numpy(clips).cuda()
    with MotionEngine(W, H, n_streams=n_streams, max_frames=T, keep_planes=True, **engine_kw, **kw) as eng:
        if expect_front_end is not None:
            assert eng.info["front_end"] == expect_front_end
        for t0 in range(0, n, T):
            t1 = min(n, t0 + T)
            stats = eng.process(dev[:, t0:t1])
            for s in range(n_streams):
                for t in range(t0, t1):
                    rec = orcs[s].process(clips[s, t], keep_planes=True)
                    pl = eng.planes(s, t - t0, bg=(t == t1 - 1))
                    for key in ("gray", "blur", "thresh"):
                        assert (pl[key] == rec["planes"][key]).all(), \
                            (key, s, t, np.argwhere(pl[key] != rec["planes"][key])[:4])
                    if t == t1 - 1:
                        assert (pl["bg"] == rec["planes"]["bg"]).all(), ("bg", s, t)
                    _, comps = eng.components(s, t - t0)
                    assert sorted(a / 2.0 for a, _ in comps) == rec["areas"], (s, t)
                    st = stats[s, t - t0]
                    assert (bool(st["movement"]), int(st["movement_counter"]), bool(st["wrote"])) == \
                        (rec["movement"], rec["counter"], rec["wrote"])


# (W, H, blur_scale) -> k = odd(int(W / blur_scale)); full-resolution mode (box_size = W)
GEOMETRIES = [
    (320, 240, 20),     # k = 17, 16-byte aligned BGR rows: gray fused into the staging
    (272, 33, 8),       # k = 35, one and a bit row groups, partial 256-column tile
    (256, 30, 3),       # k = 85: radius 42 > rows 30 (multiple reflections of rows)
    (64, 64, 1),        # k = 65: radius 32, mirror condition R16 < w holds narrowly
    (32, 48, 1),        # k = 33: radius 16 = w / 2, one column tile, slow border path
    (528, 20, 4),       # k = 133: radius 66 > rows 20, three column tiles
    (100, 75, 4),       # k = 25, rows not 16-byte aligned: gray plane + per-word staging
    (36, 28, 3),        # k = 13, tiny plane, w % 16 != 0
    (1040, 24, 10),     # k = 105, five 256-column tiles with a 16-pixel tail
]


@pytest.mark.parametrize("umma", [True, False])
@pytest.mark.parametrize("W,H,bs", GEOMETRIES)
def test_wide_blur_geometries(W, H, bs, umma):
    """umma=True: planes with w % 32 == 0 and k <= 97 take the tcgen05 one-pass kernel (k_umma.cu), the others the
    mma.sync two-pass kernels; umma=False: the library's default choice."""
    kw = dict(fps=6, box_size=W, blur_scale=bs, threshold=5, avg=0.2, min_time=0.3, cache_time=0.6,
              mask_areas=[((2, 1), (W // 3, H // 2)), ((W // 2, 0), (W - 1, H // 3), (W // 2, H - 1))])
    _run(W, H, 9, 4, kw, seed=500 + W, expect_front_end=1, umma=umma)


@pytest.mark.parametrize("umma", [True, False])
def test_wide_blur_two_streams_mixed_masks(umma):
    from find_motion_b200 import synth
    kw = dict(fps=10, box_size=640, blur_scale=20, threshold=8, avg=0.1, min_time=0.2, cache_time=0.4,
              mask_areas=synth.README_MASKS)                  # k = 33
    _run(640, 360, 10, 5, kw, seed=610, n_streams=2, expect_front_end=1, umma=umma)


# tcgen05 kernel: tile grid edges (partial 128 x 128 tiles), every kernel radius class, avg outside [0, 1], resize in front
UMMA_GEOMETRIES = [
    (128, 128, 2, None),                 # k = 65, exactly one tile
    (256, 130, 3, None),                 # k = 85, two tile rows, the second with 2 live rows
    (160, 100, 2, None),                 # k = 81 > plane height / 2: multiple reflections inside the apron
    (1280, 720, 256, None),              # k = 5 through the wide path (fused stencil switched off below)
    (640, 360, 7, None),                 # k = 91
    (96, 40, 1, None),                   # k = 97 = the largest radius the apron holds, plane smaller than a tile
    (32, 2, 4, None),                    # k = 9, two rows
]


@pytest.mark.parametrize("umma_apron", [False, True])
@pytest.mark.parametrize("W,H,bs,_", UMMA_GEOMETRIES)
def test_umma_blur_geometries(W, H, bs, _, umma_apron):
    """umma_apron=False: the BGR frames feed the tcgen05 kernel directly (TMA ring + gray conversion + mirroring inside the
    tile) where the geometry allows; True: through the gray plane with a materialised apron (the path of the resize modes)."""
    kw = dict(fps=6, box_size=W, blur_scale=bs, threshold=5, avg=0.2, min_time=0.3, cache_time=0.6,
              mask_areas=[((2, 1), (W // 3, H // 2)), ((W // 2, 0), (W - 1, H // 3), (W // 2, H - 1))])
    _run(W, H, 6, 4, kw, seed=900 + W, no_fused=True, umma=True, umma_apron=umma_apron)


@pytest.mark.parametrize("W,H,bs", [(1920, 1080, 20), (1920, 1080, 384), (1280, 720, 40), (640, 480, 64), (3840, 2160, 40)])
def test_umma_direct_full_frames(W, H, bs):
    """Full frames through the direct kernel, both apron classes (k <= 33 / k <= 97): every tile border case of real sizes."""
    kw = dict(fps=30, box_size=W, blur_scale=bs, threshold=10, avg=0.1, min_time=0.1, cache_time=0.2,
              mask_areas=[((0, 0), (100, 100)), ((0, 0), (0, 100), (100, 0)), ((W - 300, H - 200), (W - 1, H - 1))])
    _run(W, H, 3, 2, kw, seed=950 + W, no_fused=True, umma=True)


@pytest.mark.parametrize("umma_apron", [False, True])
def test_umma_blur_avg_outside_unit_range_and_k1(umma_apron):
    for avg, threshold in ((1.7, 6), (0.3, -1)):
        kw = dict(fps=6, box_size=128, blur_scale=9, threshold=threshold, avg=avg, min_time=0.3, cache_time=0.5)     # k = 15
        _run(128, 96, 8, 4, kw, seed=930, no_fused=True, umma=True, umma_apron=umma_apron)
    kw = dict(fps=6, box_size=128, blur_scale=128, threshold=6, avg=0.3, min_time=0.3, cache_time=0.5)   # k = 1: identity blur
    _run(128, 96, 8, 4, kw, seed=931, no_fused=True, umma=True, umma_apron=umma_apron)


def test_umma_blur_after_resize():
    """2x integer resize (960x540 -> 480x270 would not be % 32; 1280x720 -> 640x360 is), k = 33 on the resized plane."""
    kw = dict(fps=8, box_size=640, blur_scale=20, threshold=6, avg=0.15, min_time=0.3, cache_time=0.5)
    _run(1280, 720, 6, 3, kw, seed=940, expect_front_end=2, umma=True)


def test_wide_blur_after_resize():
    """Downscaled processing plane (resize front end) with a kernel the fused path does not take: k = 7."""
    kw = dict(fps=8, box_size=160, blur_scale=22, threshold=6, avg=0.15, min_time=0.3, cache_time=0.5)
    _run(640, 480, 10, 5, kw, seed=620, expect_front_end=2)
