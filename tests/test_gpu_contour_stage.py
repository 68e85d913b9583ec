"""GPU: the contour stage as fm_process runs it, on designed raw threshold planes (tests/motion_planes.py).

Each scenario feeds planes whose raw threshold bits are known exactly (k = 1, black first frame, frames painted 255 * P)
through a real front end (fused BGR and NV12, the generic k_gray + k_blur_identity + k_temporal, no_fused, default-mode
resize) and one of the contour paths of fm_launch_morph_ccl (F = S T >= 32 with the dilation inside k_ccl_frame_smem, at
8, 60 and 128 words per row, aligned and not; F < 32 with k_dilate; planes without a shared-memory plan), with heavy
frames for the global-memory fallback, cached and uncached windows, edges, window topology, motion in one frame index,
clamping and ragged calls.  For every valid frame: the exported dilated plane, the contour count, the records (a
sub-multiset of exactly max_components of them when clamped), the decision counters, the background after the call,
and a clean eng.check(); frames past n_valid produce nothing."""
from collections import Counter

import numpy as np
import pytest

from tests import motion_planes as M

pytestmark = pytest.mark.gpu

STATS = ("n_contours", "n_counted", "movement", "movement_counter", "movement_decay", "cache_len", "wrote", "n_flush")
DESIGNED = sorted(n for n in M.scenarios() if n != "chained_256x146")
FRONT_END = {"fused_bgr_1080": 0, "fused_nv12_1080": 0, "fused_256x146_one_frame_index": 0, "generic_200x75": 1,
             "generic_200x75_masked": 1, "nofused_256x147": 1, "area_320x242": 2, "fused_4096x38": 0,
             "no_plan_4128x48": 0, "no_plan_64x7440": 0, "fused_256x146_threshold_255": 0, "chained_256x146": 0}


def _engine(sc, **extra):
    from find_motion_b200.engine import MotionEngine
    eng = MotionEngine(sc.W, sc.H, n_streams=sc.S, max_frames=sc.Tmax, nv12=sc.kind == "nv12",
                       max_components=sc.max_components, **sc.tuning(), **sc.engine, **extra)
    assert (eng.h, eng.w) == sc.hw and eng.info["gaussian"] == 1 and eng.info["front_end"] == FRONT_END[sc.name]
    return eng


def _outputs(eng, sc, T):
    """What the test compares after a call besides the stats: (count, records) and the dilated plane of every frame,
    and the background of every stream."""
    comps = {(s, t): eng.components(s, t, max_n=sc.max_components) for s in range(sc.S) for t in range(T)}
    dil = {(s, t): eng.planes(s, t, gray=False, blur=False, bg=False)["thresh"] for s in range(sc.S) for t in range(T)}
    bg = [eng.planes(s, 0, gray=False, blur=False, thresh=False)["bg"] for s in range(sc.S)]
    return comps, dil, bg


def _where(sc, i, s, t, fr=None):
    lab = M.labelling(fr.dil) if fr is not None else None
    return f"{sc.name} call {i} stream {s} frame {t} path {M.contour_path(sc, sc.calls[i].T)} window {lab}"


def _check(sc, i, stats, out, exp):
    comps, dil, bg = out
    res, bgs = exp
    T = sc.calls[i].T
    for s in range(sc.S):
        for t in range(T):
            n, recs = comps[(s, t)]
            if t >= len(res[s]):           # past n_valid: nothing
                assert all(int(stats[s, t][k]) == 0 for k in STATS), _where(sc, i, s, t)
                assert n == 0 and not dil[(s, t)].any(), _where(sc, i, s, t)
                continue
            fr = res[s][t]
            got = {k: int(stats[s, t][k]) for k in STATS}
            assert got == fr.stats, (_where(sc, i, s, t, fr), got, fr.stats)
            assert n == len(fr.comps), _where(sc, i, s, t, fr)
            if n <= sc.max_components:
                assert sorted(recs) == fr.comps, _where(sc, i, s, t, fr)
            else:
                assert len(recs) == sc.max_components, _where(sc, i, s, t, fr)
                assert not Counter(recs) - Counter(fr.comps), _where(sc, i, s, t, fr)
            if not (dil[(s, t)] == fr.dil).all():
                bad = np.argwhere(dil[(s, t)] != fr.dil)
                raise AssertionError(f"{_where(sc, i, s, t, fr)}: dilated plane differs at {len(bad)} pixels, first {bad[:4]}")
        if bgs[s] is not None:
            assert (bg[s] == bgs[s]).all(), _where(sc, i, s, -1)


def _run_synchronised(sc, exp, **extra):
    import torch
    outs = []
    with _engine(sc, **extra) as eng:
        for i, (c, batch) in enumerate(zip(sc.calls, M.frames(sc))):
            for s in c.reset:
                eng.reset(s)
            stats = eng.process(torch.from_numpy(batch).cuda(), n_valid=c.n_valid)
            out = _outputs(eng, sc, c.T)
            _check(sc, i, stats, out, exp[i])
            outs.append((stats, out))
            eng.check()
    return outs


@pytest.mark.parametrize("name", DESIGNED)
def test_designed_planes(name):
    sc = M.scenarios()[name]()
    _run_synchronised(sc, M.replay(sc))


def test_chained_calls_equal_synchronised_calls():
    """Calls 0..k issued back to back with sync=False on the fused path (each call's front end starts under the previous
    call's contour stage) give the outputs of call k that the same calls give synchronised one by one, and both give
    the designed outputs."""
    import torch
    from find_motion_b200.engine import STATS_DTYPE
    sc = M.chained_scenario()
    exp = M.replay(sc)
    ref = _run_synchronised(sc, exp)
    batches = [torch.from_numpy(b).cuda() for b in M.frames(sc)]
    for k in range(len(sc.calls)):
        with _engine(sc) as eng:
            for i in range(k + 1):
                for s in sc.calls[i].reset:
                    eng.reset(s)
                st = eng.process(batches[i], sync=False, n_valid=sc.calls[i].n_valid)
            torch.cuda.synchronize()
            T = sc.calls[k].T
            stats = st.cpu().numpy().view(STATS_DTYPE).reshape(sc.S, T).copy()
            out = _outputs(eng, sc, T)
            eng.check()
        ref_stats, (ref_comps, ref_dil, ref_bg) = ref[k]
        assert (stats == ref_stats).all(), k
        assert out[0] == ref_comps, k
        assert all((out[1][key] == ref_dil[key]).all() for key in out[1]), k
        assert all((a == b).all() for a, b in zip(out[2], ref_bg)), k
        _check(sc, k, stats, out, exp[k])


@pytest.mark.parametrize("extra,front_end", [({}, 0), ({"no_fused": True}, 1), ({"no_fused": True, "umma": True}, 1)],
                         ids=["k_fused", "k_wide", "umma"])
def test_k3_front_ends_on_designed_frames(extra, front_end):
    """k = 3 on k_fused, on the mma.sync wide kernels (no_fused) and on tcgen05 (no_fused, umma): the raw plane is no
    longer designed, so every frame is checked against StreamOracle (dilated plane, records, counters, background)."""
    import torch
    from oracle import restated as R
    from find_motion_b200.engine import MotionEngine
    h, w, S, T = 96, 256, 2, 8
    kw = dict(fps=10, box_size=w, blur_scale=80, threshold=12, avg=0.5, min_time=0.3, cache_time=0.5)
    edg, top = list(M.edge_planes(h, w).values()), list(M.topology_planes(h, w).values())
    planes = [[None] + edg[:7] + top[:4] + [M.comb(h, w, 10, 80), None, M.random_plane(h, w, 0.01, 30), None],
              [None] + top + [M.random_plane(h, w, 0.02, 31)] + edg[4:11] + [None]]
    clips = np.stack([[M.encode_bgr(p if p is not None else np.zeros((h, w), bool)) for p in ps] for ps in planes])
    orcs = [R.StreamOracle(w, h, **kw) for _ in range(S)]
    dev = torch.from_numpy(clips).cuda()
    with MotionEngine(w, h, n_streams=S, max_frames=T, **kw, **extra) as eng:
        assert eng.info["gaussian"] == 3 and eng.info["front_end"] == front_end
        for t0 in range(0, clips.shape[1], T):
            stats = eng.process(dev[:, t0:t0 + T])
            for s in range(S):
                for t in range(T):
                    rec = orcs[s].process(clips[s, t0 + t], keep_planes=True)
                    st = stats[s, t]
                    assert (eng.planes(s, t, gray=False, blur=False, bg=False)["thresh"] == rec["planes"]["thresh"]).all()
                    n, comps = eng.components(s, t)
                    assert n == len(rec["areas"]) and sorted(a / 2.0 for a, _ in comps) == rec["areas"]
                    assert sorted(b for _, b in comps) == rec["boxes"]
                    assert (int(st["movement"]), int(st["movement_counter"]), int(st["movement_decay"]),
                            int(st["cache_len"]), int(st["wrote"]), int(st["n_flush"])) == \
                        (int(rec["movement"]), rec["counter"], rec["decay"], rec["cache_len"], int(rec["wrote"]),
                         rec["n_flush"]), (s, t0 + t)
                bg = eng.planes(s, 0, gray=False, blur=False, thresh=False)["bg"]
                assert (bg == orcs[s].bg).all()
            eng.check()
