"""GPU: bench.py times exactly --steps steps, and --dump-outputs writes what the last of them computed (checked against
a replay of the same seeded steps on a fresh engine)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_steps_and_dump_outputs(tmp_path):
    import torch
    import bench
    from find_motion_b200 import synth
    from find_motion_b200.engine import STATS_DTYPE, MotionEngine

    W, H, S, T, R, steps, warmup = 640, 480, 2, 8, 16, 3, 2
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--size", f"{W}x{H}", "--streams", str(S), "--frames", str(T),
           "--ring", str(R), "--steps", str(steps), "--warmup", str(warmup), "--no-e2e", "--no-cpu-baseline",
           "--no-extras", "--dump-outputs", str(out)]
    res = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads(res.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["timed_steps"] == steps

    dumped = {f[:-4]: np.load(out / f) for f in os.listdir(out)}
    assert set(dumped) == set(STATS_DTYPE.names) | {"components", "background_sample"}
    assert all(a.dtype in (np.float32, np.float64) for a in dumped.values())
    assert sum(a.nbytes for a in dumped.values()) <= 64 << 20

    # replay: the priming passes and reset of bench.measure, the warm-up steps, then the timed steps
    kw = dict(bench.tuning("full", None), box_size=W)
    clips = np.stack([synth.make_clip(W, H, R, synth.stream_seed(2, s), script=bench.bench_script(R)) for s in range(S)])
    dev = torch.from_numpy(clips).cuda()
    with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as eng:
        for _ in range(2):
            eng.process(dev[:, :T])
        eng.reset()
        for i in range(warmup + steps):
            a = (i % (R // T)) * T
            stats = eng.process(dev[:, a:a + T])
        for name in STATS_DTYPE.names:
            assert (dumped[name] == stats[name]).all(), name
        assert dumped["n_contours"].sum() > 0, "the last step should see motion"
        rows = [(s, t, a2, *box) for s in range(S) for t in range(T) for a2, box in eng.components(s, t)[1]]
        assert (dumped["components"] == np.array(rows, np.float64).reshape(-1, 7)).all()
        n = eng.w * eng.h
        idx = np.sort(np.random.default_rng(0).choice(n, min(n, bench.DUMP_BG_VALUES // S), replace=False))
        for s in range(S):
            bg = eng.planes(s, T - 1, gray=False, blur=False, thresh=False)["bg"].ravel()
            assert (dumped["background_sample"][s] == bg[idx]).all(), s
