"""GPU: the fused front end of a call starts under the contour stage of the previous one (programmatic dependent launch,
csrc/k_fused.cu fused_exit).  Calls issued back to back must give exactly what the same calls give with the device
synchronised after each one: per-call stats, every contour record and the float64 background."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# S * T = 32 frames per call: the contour stage runs the shared-memory labelling kernel that dilates the raw bits itself
# (the path of the 8 x 16 headline shape), and h * (w / 2 + 2) > 4096 keeps the global-memory fallback in the chain
W, H, S, T, R = 256, 192, 4, 8, 32


def _kw():
    return dict(fps=10, box_size=W, blur_scale=64, threshold=12, avg=0.1, min_time=0.3, cache_time=0.5,
                min_box_scale=50, max_components=8192)


def _frames():
    """moving: a walker in every frame; quiet: the same static background and noise only; heavy: quiet with vertical
    1-px lines 8 px apart changed by 110 in frame 2 of stream 1 (3 px above threshold, 7 px after the 5x5 dilation: ~28
    runs per row, more than the shared-memory tables hold, so k_ccl_frame labels that frame)."""
    import torch
    from find_motion_b200 import synth
    mov = np.stack([synth.make_clip(W, H, R, seed=500 + s, fps=10, script=[("walker", 0, R)]) for s in range(S)])
    qui = np.stack([synth.make_clip(W, H, R, seed=500 + s, fps=10, script=[]) for s in range(S)])
    hvy = qui[:, :T].copy()
    lines = hvy[1, 2, :, 3::8].astype(np.int16)
    hvy[1, 2, :, 3::8] = np.where(lines < 128, lines + 110, lines - 110).astype(np.uint8)
    return {k: torch.from_numpy(v).cuda() for k, v in (("mov", mov), ("qui", qui), ("hvy", hvy))}, (mov, qui)


# one call each: (clip, first frame, n_valid or None); motion alternates between a large window and none, n_valid
# changes between calls, and one call carries the heavy frame
CALLS = [("mov", 0, None), ("qui", 8, None), ("mov", 16, None), ("qui", 24, None), ("mov", 8, [8, 3, 0, 8]),
         ("qui", 16, [2, 8, 8, 0]), ("hvy", 0, None), ("mov", 0, None), ("qui", 8, None), ("mov", 24, [8, 8, 5, 8])]
RESET_BEFORE = {8: 2}      # reset(2) before call 8: stream 2 starts over (first frame = background) inside the chain


def _issue(eng, fr, i):
    if i in RESET_BEFORE:
        eng.reset(RESET_BEFORE[i])
    clip, a, nv = CALLS[i]
    return eng.process(fr[clip][:, a:a + T], sync=False, n_valid=nv)


def _outputs(eng, stats_dev):
    from find_motion_b200.engine import STATS_DTYPE
    stats = stats_dev.cpu().numpy().view(STATS_DTYPE).reshape(S, T).copy()
    comps = [eng.components(s, t) for s in range(S) for t in range(T)]
    bg = np.stack([eng.planes(s, 0, gray=False, blur=False, thresh=False)["bg"] for s in range(S)])
    return stats, comps, bg


def _assert_same(a, b, where):
    assert (a[0] == b[0]).all(), ("stats", where)
    assert a[1] == b[1], ("contours", where)
    assert (a[2] == b[2]).all(), ("background", where)


def _reference(fr):
    """Outputs after every call with the device synchronised after each one."""
    import torch
    from find_motion_b200.engine import MotionEngine
    out = []
    with MotionEngine(W, H, n_streams=S, max_frames=T, **_kw()) as eng:
        assert eng.info["front_end"] == 0, "fused front end expected"
        for i in range(len(CALLS)):
            st = _issue(eng, fr, i)
            torch.cuda.synchronize()
            out.append(_outputs(eng, st))
            if CALLS[i][0] == "hvy":     # more runs of set pixels than the shared-memory tables hold (4096)
                dil = eng.planes(1, 2, gray=False, blur=False, bg=False)["thresh"] > 0
                assert int((np.diff(dil.astype(np.int8), axis=1, prepend=0) == 1).sum()) > 4096
    return out


@pytest.mark.parametrize("timing", [False, True])
def test_back_to_back_calls_equal_synchronised_calls(timing):
    """For every k: calls 0..k issued back to back (no synchronisation between them), then the outputs of call k."""
    import torch
    from find_motion_b200.engine import MotionEngine
    fr, _ = _frames()
    ref = _reference(fr)
    assert all(int(r[0]["n_contours"].sum()) > 0 for r in ref[0::2][:3])
    for k in range(len(CALLS)):
        with MotionEngine(W, H, n_streams=S, max_frames=T, **_kw()) as eng:
            eng.timing(enable=timing)
            for i in range(k + 1):
                st = _issue(eng, fr, i)
            torch.cuda.synchronize()
            _assert_same(_outputs(eng, st), ref[k], k)
            eng.check()


def test_mixed_entry_points_in_a_chain():
    """process / process_clip / submit_host / wait_host / submit_reset / process_host, components() and plane exports
    between chained calls: what each read returns equals the same sequence run with a synchronisation after every
    call."""
    import torch
    from find_motion_b200.engine import MotionEngine, STATS_DTYPE
    fr, (mov, qui) = _frames()

    def run(sync_each):
        reads = []
        with MotionEngine(W, H, n_streams=S, max_frames=T, device_clips=True, **_kw()) as eng:
            def dev(i):
                st = _issue(eng, fr, i)
                if sync_each:
                    torch.cuda.synchronize()
                return st
            stats, clips = eng.process_clip(fr["mov"][:, 0:T])
            reads.append((stats.copy(), [c.cpu().numpy() for c in clips]))
            dev(1)
            dev(2)
            st = dev(3)
            reads.append(_outputs(eng, st))                 # components() and planes() right after chained calls
            dev(4)
            stats, clips = eng.process_clip(fr["qui"][:, 0:T])
            reads.append((stats.copy(), [c.cpu().numpy() for c in clips]))
            dev(6)
            st = dev(7)
            reads.append(_outputs(eng, st))
            torch.cuda.synchronize()                        # the host entry points run on the context's own stream
            eng.submit_host(0, mov[:, 8:16])
            eng.submit_host(1, qui[:, 16:24])
            reads.append(eng.wait_host(0))
            eng.submit_reset(1)
            eng.submit_host(0, mov[:, 24:32])
            reads.append(eng.wait_host(1))
            reads.append(eng.wait_host(0))
            reads.append(eng.process_host(qui[:, 0:8]))
            st = dev(9)
            reads.append(_outputs(eng, st))
        return reads

    a, b = run(False), run(True)
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        if isinstance(x, np.ndarray):
            assert x.dtype == STATS_DTYPE and (x == y).all(), i
        elif len(x) == 2:
            assert (x[0] == y[0]).all() and len(x[1]) == len(y[1]), i
            assert all((p == q).all() for p, q in zip(x[1], y[1])), i
        else:
            _assert_same(x, y, i)
