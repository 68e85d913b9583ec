"""Cost of the device-side look-back cache and motion-clip write-back (FM_FLAG_DEVICE_CLIPS, csrc/k_clips.cu).

One JSON line per regime, printed and appended to --out:
  * two scenes per regime: "moving" (every frame written: the gathers carry the copies) and "quiet" (every frame
    cached: the ring stores carry them);
  * frames/s of the whole per-frame path without the flag (fm_process), with it (fm_process_clip) and with it through
    plain fm_process (ring upkeep only), the three arms alternated window by window in the same run, CUDA events around
    each window of --steps calls after --warmup untimed ones; inputs come from an HBM ring larger than L2 (each call
    reads the next T frames of every stream), so no call re-reads cached input;
  * k_clip_plan / k_clip_gather / k_clip_store times from torch.profiler, in a separate run of --prof-steps calls;
  * the bytes the gather and store kernels move (read + write, counted from the stats of those calls) over their time;
  * as the copy ceiling, a cudaMemcpyAsync device-to-device copy of the same byte count per call in the same run
    (torch's copy_ of two contiguous uint8 tensors, source and destination rotating through buffers larger than L2);
  * the GPU's name and power limit, read in the same run.

    python tools/bench_clips.py [--out profiles/bench_clips.jsonl] [--steps 100] [--rounds 5]

Needs a CUDA device; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_upscale import L2_BYTES, gpu_facts, make_ring  # noqa: E402

# motion of the input ring: "moving" is bench_upscale's (a walker and a blob in every stream: every frame is written,
# the gathers carry the copies), "quiet" has no objects (every frame is cached: the ring stores carry them)
SCENES = ("moving", "quiet")

# name, W, H, box_size, blur_scale (bench.py's full-resolution k=5 and default-mode regimes)
REGIMES = [
    ("1080p_full_k5", 1920, 1080, 1920, 384),
    ("1080p_default_box100", 1920, 1080, 100, 20),
]
TUNING = dict(fps=30, min_box_scale=50, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)   # bench.py: C = 30


def quiet_ring(W, H, S, T, device):
    """[S][R][H][W][3] like make_ring, sensor noise over a static background only."""
    import math
    import torch
    from find_motion_b200 import synth
    R = max(2 * T, math.ceil(3 * L2_BYTES / (S * W * H * 3) / T) * T)
    ring = torch.empty((S, R, H, W, 3), dtype=torch.uint8, device=device)
    n = min(R, 16)
    for s in range(S):
        c = torch.from_numpy(synth.make_clip(W, H, n, seed=synth.stream_seed(9, s), script=[])).to(device)
        for r0 in range(0, R, n):
            ring[s, r0:r0 + min(n, R - r0)] = c[:min(n, R - r0)]
    return ring, R


def run_regime(name, W, H, box, bs, scene, args):
    import numpy as np
    import torch
    from torch.profiler import ProfilerActivity, profile
    from find_motion_b200 import _lib
    from find_motion_b200.engine import STATS_DTYPE, MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    ring, R = (make_ring if scene == "moving" else quiet_ring)(W, H, S, T, f"cuda:{dev}")
    fb = W * H * 3
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    res = {"regime": name, "scene": scene, "W": W, "H": H, "box_size": box, "blur_scale": bs, "streams": S, "frames_per_call": T,
           "ring_frames_per_stream": R, "ring_mb": round(S * R * fb / 1e6, 1)}
    calls = R // T
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as off, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, device_clips=True, **kw) as on:
        Cf = on.info["cache_frames"]
        res.update(cache_frames=Cf, min_movement_frames=on.info["min_movement_frames"], front_end=on.info["front_end"])
        out = torch.empty((S, Cf + T, H, W, 3), dtype=torch.uint8, device=f"cuda:{dev}")
        stats_all = torch.empty((max(args.prof_steps, 1), S * T * STATS_DTYPE.itemsize), dtype=torch.uint8,
                                device=f"cuda:{dev}")
        lib = on._lib

        def clip_call(i, stats_ptr=None):
            a = (i % calls) * T
            src = ring[:, a:a + T]
            st = torch.cuda.current_stream().cuda_stream
            _lib.check(lib.fm_process_clip(on._ctx, src.data_ptr(), src.stride(0), src.stride(1), T, None,
                                           C.c_void_p(st), stats_ptr, out.data_ptr(), out.stride(0), out.shape[1]))

        arms = {
            "off": lambda i: off.process(ring[:, (i % calls) * T:(i % calls) * T + T], sync=False),
            "on_clip": clip_call,
            "on_process": lambda i: on.process(ring[:, (i % calls) * T:(i % calls) * T + T], sync=False),
        }
        rates = {k: [] for k in arms}
        i = 0
        for k, fn in arms.items():                       # warm every arm
            for _ in range(args.warmup):
                fn(i)
                i += 1
        torch.cuda.synchronize()
        for _ in range(args.rounds):
            for k, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    fn(i)
                    i += 1
                e1.record()
                torch.cuda.synchronize()
                rates[k].append(args.steps * S * T / (e0.elapsed_time(e1) / 1e3))
        off.check()
        on.check()
        for k, v in rates.items():
            res[f"frames_per_s_{k}"] = round(statistics.median(v), 1)
            res[f"frames_per_s_{k}_all"] = [round(x, 1) for x in v]

        # kernel times, in a run of their own; the stats of every profiled call give the bytes the copies moved
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for j in range(args.prof_steps):
                clip_call(i, stats_all[j].data_ptr())
                i += 1
            torch.cuda.synchronize()
        st = stats_all.cpu().numpy().view(STATS_DTYPE).reshape(args.prof_steps, S, T)
        gather_frames = int(st["wrote"].sum() + st["n_flush"].sum())
        store_frames = int(np.minimum(st["cache_len"][:, :, T - 1], T).sum()) if Cf > 0 else 0
        kt = {}
        for evt in prof.key_averages():
            for kn in ("k_clip_plan", "k_clip_gather", "k_clip_store"):
                if kn in evt.key:
                    us = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
                    kt[kn] = (kt.get(kn, (0.0, 0))[0] + us, kt.get(kn, (0.0, 0))[1] + evt.count)
        for kn in ("k_clip_plan", "k_clip_gather", "k_clip_store"):
            if kn not in kt:
                raise RuntimeError(f"{kn} did not appear in the profile")
            res[f"{kn}_us"] = round(kt[kn][0] / kt[kn][1], 2)
        n = args.prof_steps
        gb = 2 * fb * gather_frames / n                 # read + write per call
        sb = 2 * fb * store_frames / n
        rate = lambda b, us: round(b / (us * 1e-6) / 1e9, 1) if b else None  # noqa: E731
        res.update(profiled_calls=n, gather_frames_per_call=round(gather_frames / n, 2),
                   store_frames_per_call=round(store_frames / n, 2),
                   gather_bytes_per_call=round(gb), store_bytes_per_call=round(sb),
                   gather_gb_per_s=rate(gb, res["k_clip_gather_us"]), store_gb_per_s=rate(sb, res["k_clip_store_us"]),
                   copies_gb_per_s=rate(gb + sb, res["k_clip_gather_us"] + res["k_clip_store_us"]))

        # copy ceiling: cudaMemcpyAsync of the same bytes per call (half of read + write), over buffers larger than L2
        nbytes = max(int((gb + sb) / 2), 1 << 20)
        nbuf = max(2, -(-3 * L2_BYTES // nbytes) + 1)
        del ring
        torch.cuda.empty_cache()
        bufs = [torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{dev}") for _ in range(nbuf)]
        for j in range(nbuf):
            bufs[(j + 1) % nbuf].copy_(bufs[j])
        torch.cuda.synchronize()
        reps = max(20, args.prof_steps)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for j in range(reps):
            bufs[(j + 1) % nbuf].copy_(bufs[j % nbuf])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        ceil = 2 * nbytes / (ms * 1e-3) / 1e9
        res.update(memcpy_bytes=nbytes, memcpy_us=round(ms * 1e3, 2), memcpy_gb_per_s=round(ceil, 1))
        for k in ("copies", "gather", "store"):
            v = res[f"{k}_gb_per_s"]
            res[f"{k}_share_of_memcpy"] = round(v / ceil, 3) if v else None
        del bufs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_clips.jsonl"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--prof-steps", type=int, default=50)
    ap.add_argument("--regimes", default=",".join(r[0] for r in REGIMES))
    ap.add_argument("--scenes", default=",".join(SCENES))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_clips.py needs a CUDA device (there is no CPU fallback)")
    from find_motion_b200 import build
    build.build()
    facts = gpu_facts(args.device)
    want = set(args.regimes.split(","))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for name, W, H, box, bs in REGIMES:
            if name not in want:
                continue
            for scene in args.scenes.split(","):
                res = run_regime(name, W, H, box, bs, scene, args)
                res.update(facts)
                line = json.dumps(res)
                print(line, flush=True)
                f.write(line + "\n")


if __name__ == "__main__":
    main()
