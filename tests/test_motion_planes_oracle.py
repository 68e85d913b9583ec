"""CPU: the designed motion planes of tests/motion_planes.py are what they claim to be.

- R.external_components (through motion_planes.components) equals cv2.findContours + contourArea + boundingRect on every
  dilated plane the GPU contour-stage test uses, at the sizes it uses them.
- The encoders reproduce the designed raw planes through the whole per-frame chain (StreamOracle on small planes,
  oracle.cv2_chain.Cv2Stream at 1080p) for every encoder and every (threshold, avg) mode, with and without masks.
- Every scenario reaches the labelling path it claims: heavy frames hold more than CCL2_CAP runs of a polarity in their
  window, cached / uncached windows fit / exceed the shared-memory row cache, edge planes touch their edge."""
import numpy as np
import pytest

from tests import motion_planes as M

cv2 = pytest.importorskip("cv2")

SCENARIOS = M.scenarios()


def _cv2_components(dil):
    cnts = cv2.findContours(dil.copy(), cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_SIMPLE)[-2]
    return sorted((int(round(2 * cv2.contourArea(c))), tuple(int(v) for v in cv2.boundingRect(c))) for c in cnts)


def _distinct_raws(sc):
    h, w = sc.hw
    keep = ~sc.mask()
    seen = {}
    for c in sc.calls:
        for row in c.raws:
            for raw in row:
                if raw is not None and sc.threshold <= 254:
                    eff = raw & keep
                    seen[np.packbits(eff).tobytes()] = eff
    return list(seen.values())


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_components_equal_cv2_on_scenario_planes(name):
    sc = SCENARIOS[name]()
    raws = _distinct_raws(sc)
    assert raws or sc.threshold == 255
    for raw in raws:
        dil, comps = M.expected_plane(raw)
        assert (dil == cv2.dilate(raw.astype(np.uint8) * 255, None, iterations=2)).all(), name
        assert comps == _cv2_components(dil), name


@pytest.mark.parametrize("name", sorted(SCENARIOS))
def test_scenario_claims(name):
    sc = SCENARIOS[name]()
    M.check_claims(sc)
    paths = {M.contour_path(sc, c.T) for c in sc.calls}
    want = {"no_plan_4128x48": "k_dilate+global", "no_plan_64x7440": "k_dilate+global",
            "generic_200x75_masked": "k_dilate+smem", "nofused_256x147": "k_dilate+smem",
            "fused_256x146_threshold_255": "k_dilate+smem"}.get(name, "smem_dilate")
    assert paths == {want}, (name, paths)
    for c in sc.calls:                                  # frames past n_valid hold something the GPU must ignore
        nv = c.n_valid or (c.T,) * sc.S
        assert all(t >= nv[s] for s, t in c.fill), name


def test_claim_kinds_are_all_reached():
    """Across the scenarios: heavy, shared-memory cached and uncached windows, clamped and quiet frames."""
    kinds = set()
    for b in SCENARIOS.values():
        for c in b().calls:
            for cl in c.claims.values():
                kinds |= cl
    assert {"heavy", "cached", "uncached", "smem", "clamped", "quiet"} <= kinds, kinds


@pytest.mark.parametrize("h,w", [(75, 200), (146, 256), (147, 256), (121, 160), (38, 4096), (48, 4128), (7440, 64),
                                 (1080, 1920)])
def test_edge_planes_touch_their_edges(h, w):
    e = M.edge_planes(h, w)
    assert e["corner_tl"][0, 0] and e["corner_tr"][0, w - 1] and e["corner_bl"][h - 1, 0] and e["corner_br"][h - 1, w - 1]
    assert e["row_first"][0].any() and e["row_last"][h - 1].any()
    assert e["col_first"][:, 0].any() and e["col_last"][:, w - 1].any()
    (y0, x0), = np.argwhere(e["row_end"])
    (y1, x1), = np.argwhere(e["next_row_start"])
    assert x0 == w - 1 and (y1, x1) == (y0 + 1, 0)            # adjacent bits of the flat bit order
    if w < M.TILE_PX and "tile_end" in e:
        (y, x), = np.argwhere(e["tile_end"])
        i = y * w + x
        assert i % M.TILE_PX == M.TILE_PX - 1                 # the last pixel of its k_temporal tile ...
        if w < M.TILE_PX // 2:
            assert y - (i - M.TILE_PX + 1) // w >= 2          # ... which spans at least three rows
    if (h, w) == (75, 200):
        assert "tile_end" in e


def test_one_frame_planes_sit_in_the_last_row_of_a_warp_group():
    sc = SCENARIOS["fused_256x146_one_frame_index"]()
    for c, ts in ((sc.calls[1], (0, 15, 16, 31)), (sc.calls[2], (31, 32, 33, 39))):
        for s, t in enumerate(ts):
            assert [i for i, p in enumerate(c.raws[s]) if p is not None] == [t]
            ys = np.flatnonzero(c.raws[s][t].any(axis=1))
            assert ys[-1] % 4 == 3 and ys[-1] + 2 < sc.hw[0]


def _small_scenario(kind, threshold, avg, masks=None):
    """One stream of edges, window topology, random planes and a comb on a 160 x 122 plane (full resolution, or
    320 x 244 at ratio 2)."""
    from find_motion_b200 import synth
    h, w = 122, 160
    edg, top = list(M.edge_planes(h, w).values()), list(M.topology_planes(h, w).values())
    rnd = M.random_plane(h, w, 0.02, 21)
    raws = M._seq(24, edg[:10] + [rnd] + top + [rnd, None, rnd, M.comb(h, w, 20, 100)])
    W, H = (320, 244) if kind == "area" else (160, 122)
    return M.Scenario(f"{kind}_{threshold}_{avg}", W, H, kind, 1, 24, threshold, avg, [M.Call([raws])],
                      box_size=160, mask_areas=masks and synth.README_MASKS)


def _to_bgr(kind, frame):
    return cv2.cvtColor(frame, cv2.COLOR_YUV2BGR_NV12) if kind == "nv12" else frame


@pytest.mark.parametrize("kind", ["bgr", "nv12", "area"])
@pytest.mark.parametrize("threshold,avg,masks", [(0, 0, False), (0, 1, False), (254, 0, False), (254, 1, True),
                                                 (255, 0, False), (254, 1, False), (0, 0, True)])
def test_encoders_reproduce_the_designed_planes(kind, threshold, avg, masks):
    """StreamOracle on the encoded frames gives the replay's dilated plane, records and counters for every frame, and
    the replay's background after the last one."""
    from oracle import restated as R
    sc = _small_scenario(kind, threshold, avg, masks)
    (batch,) = list(M.frames(sc))
    (res, bgs), = M.replay(sc)
    orc = R.StreamOracle(sc.W, sc.H, **sc.tuning())
    assert orc.k == 1
    for t, fr in enumerate(res[0]):
        rec = orc.process(_to_bgr(kind, batch[0, t]), keep_planes=True)
        assert (rec["planes"]["thresh"] == fr.dil).all(), t
        assert rec["areas"] == sorted(a / 2.0 for a, _ in fr.comps) and rec["boxes"] == sorted(b for _, b in fr.comps)
        got = (int(rec["movement"]), rec["counter"], rec["decay"], rec["cache_len"], int(rec["wrote"]), rec["n_flush"])
        st = fr.stats
        assert got == (st["movement"], st["movement_counter"], st["movement_decay"], st["cache_len"], st["wrote"],
                       st["n_flush"]), t
    assert (orc.bg == bgs[0]).all()
    if threshold <= 254 and not masks:
        assert any(fr.comps for fr in res[0])


@pytest.mark.parametrize("name", ["fused_bgr_1080", "fused_nv12_1080"])
def test_cv2_chain_reproduces_the_1080p_planes(name):
    """The 1080p scenarios through the reference's cv2 calls: the first frames of each stream of the first call."""
    from oracle.cv2_chain import Cv2Stream
    sc = SCENARIOS[name]()
    sc.calls = sc.calls[:1]
    (batch,) = list(M.frames(sc))
    (res, _), = M.replay(sc)
    for s in range(sc.S):
        cs = Cv2Stream(sc.W, sc.H, **sc.tuning())
        for t in range(5):
            out = cs.step(_to_bgr(sc.kind, batch[s, t]))
            fr = res[s][t]
            assert (out["thresh"] == fr.dil).all(), (s, t)
            assert out["areas"] == sorted(a / 2.0 for a, _ in fr.comps), (s, t)
            assert (int(out["movement"]), out["counter"], out["decay"], out["cache_len"], int(out["wrote"]),
                    out["n_flush"]) == tuple(fr.stats[k] for k in ("movement", "movement_counter", "movement_decay",
                                                                    "cache_len", "wrote", "n_flush")), (s, t)
