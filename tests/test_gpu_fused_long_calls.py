"""K1 (the fused front end) records which rows of each frame hold a threshold bit (`rawrange`, read by the contour stage)
in one of two ways: for calls of up to 32 frames per stream once after the frame loop, for longer calls frame by frame.
Both must give the stats and contour records of the generic multi-kernel front end, including ragged batches whose
streams end on either side of 32 frames."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("T,n_valid", [(32, (32, 7)), (40, (40, 33)), (40, (32, 31))])
def test_fused_rawrange_equals_generic_front_end(T, n_valid):
    import torch
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine
    W, H, S = 256, 144, 2
    kw = dict(fps=10, box_size=W, blur_scale=W // 5, threshold=10, avg=0.1, min_time=0.3, cache_time=0.6,
              mask_areas=synth.README_MASKS)
    clips = np.stack([synth.make_clip(W, H, 2 * T, seed=120 + s, fps=10) for s in range(S)])
    dev = torch.from_numpy(clips).cuda()
    with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as a, \
            MotionEngine(W, H, n_streams=S, max_frames=T, no_fused=True, **kw) as b:
        assert a.info["front_end"] == 0 and b.info["front_end"] == 1
        for t0 in (0, T):
            sa = a.process(dev[:, t0:t0 + T], n_valid=n_valid)
            sb = b.process(dev[:, t0:t0 + T], n_valid=n_valid)
            for s in range(S):
                assert (sa[s, :n_valid[s]] == sb[s, :n_valid[s]]).all(), (t0, s)
                for t in range(n_valid[s]):
                    assert a.components(s, t) == b.components(s, t), (t0, s, t)
