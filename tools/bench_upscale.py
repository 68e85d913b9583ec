"""Throughput of the upscaling front end (FM_FLAG_UPSCALE, csrc/k_upscale.cu): frames narrower than box_size.

One JSON line per regime, printed and appended to --out:
  * frames/s of the whole per-frame path (fm_process, S streams x T frames per call) over --steps timed calls after
    --warmup untimed ones, CUDA events around the timed window; the inputs come from an HBM ring larger than L2
    (each call reads the next T frames of every stream), so no call re-reads cached input;
  * the k_upscale_gray kernel time from torch.profiler, in a separate run of --prof-steps calls;
  * the bytes that kernel has to move, 3*W*H (BGR in) + w*h (gray out) per frame, over its time, beside the HBM3e
    bandwidth of NVIDIA's B200 data sheet (7.7 TB/s; a ratio to it is not a measured peak);
  * the GPU's name and power limit, read in the same run.

    python tools/bench_upscale.py [--out profiles/bench_upscale.jsonl] [--steps 200]

Needs a CUDA device; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

L2_BYTES = 126 * 2 ** 20
HBM_DATASHEET = 7.7e12

# name, W, H, box_size, blur_scale
REGIMES = [
    ("720p_to_1920_k5", 1280, 720, 1920, 384),
    ("720p_to_1920_k97", 1280, 720, 1920, 20),
    ("640x480_to_800", 640, 480, 800, 20),
    ("80x60_to_100", 80, 60, 100, 20),
]


def gpu_facts(device):
    import torch
    facts = {"gpu": torch.cuda.get_device_name(device), "power_limit_w": None, "sm_clock_max_mhz": None}
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30).stdout
        pl, clk = [v.strip() for v in out.strip().splitlines()[0].split(",")]
        facts["power_limit_w"], facts["sm_clock_max_mhz"] = float(pl), float(clk)
    except Exception as e:                      # reported, not guessed
        facts["power_limit_error"] = str(e)
    return facts


def make_ring(W, H, S, T, device):
    """[S][R][H][W][3] uint8 on the device, R a multiple of T and S*R frames > 3x L2: seeded synthetic clips (a walker
    and a masked blob over a textured background), a 64-frame clip per stream tiled along the ring."""
    import numpy as np
    import torch
    from find_motion_b200 import synth
    fb = W * H * 3
    R = max(2 * T, math.ceil(3 * L2_BYTES / (S * fb) / T) * T)
    n = min(R, 64)
    ring = torch.empty((S, R, H, W, 3), dtype=torch.uint8, device=device)
    for s in range(S):
        clip = synth.make_clip(W, H, n, seed=synth.stream_seed(7, s), script=[("walker", n // 4, n // 4 + max(4, n // 3)),
                                                                               ("hidden", 2, n // 2)])
        c = torch.from_numpy(np.ascontiguousarray(clip)).to(device)
        for r0 in range(0, R, n):
            m = min(n, R - r0)
            ring[s, r0:r0 + m] = c[:m]
    return ring, R


def run_regime(name, W, H, box, bs, args):
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    ring, R = make_ring(W, H, S, T, f"cuda:{dev}")
    kw = dict(fps=30, box_size=box, blur_scale=bs, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)
    res = {"regime": name, "W": W, "H": H, "box_size": box, "blur_scale": bs, "streams": S, "frames_per_call": T,
           "ring_frames_per_stream": R, "ring_mb": round(S * R * W * H * 3 / 1e6, 1)}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, upscale=True, **kw) as eng:
        w, h = eng.w, eng.h
        res.update(w=w, h=h, gaussian=eng.info["gaussian"], front_end=eng.info["front_end"])
        calls = R // T

        def step(i):
            a = (i % calls) * T
            eng.process(ring[:, a:a + T], sync=False)

        for i in range(args.warmup):
            step(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            step(args.warmup + i)
        e1.record()
        torch.cuda.synchronize()
        eng.check()
        ms = e0.elapsed_time(e1)
        res.update(timed_steps=args.steps, step_ms=round(ms / args.steps, 4),
                   frames_per_s=round(args.steps * S * T / (ms / 1e3), 1))
        # kernel time under the profiler, in a run of its own
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(args.prof_steps):
                step(i)
            torch.cuda.synchronize()
        tot_us, cnt = 0.0, 0
        for evt in prof.key_averages():
            if "k_upscale_gray" in evt.key:
                tot_us += getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
                cnt += evt.count
        if cnt == 0:
            raise RuntimeError("k_upscale_gray did not appear in the profile")
        kern_us = tot_us / cnt
        need = S * T * (3 * W * H + w * h)
        res.update(kernel="k_upscale_gray", kernel_us=round(kern_us, 2), kernel_calls_profiled=cnt,
                   kernel_bytes_per_call=need, kernel_bytes_per_frame=3 * W * H + w * h,
                   kernel_gb_per_s=round(need / (kern_us * 1e-6) / 1e9, 1),
                   kernel_share_of_datasheet_hbm=round(need / (kern_us * 1e-6) / HBM_DATASHEET, 3),
                   kernel_share_of_step=round(kern_us / 1e3 / (ms / args.steps), 3))
    del ring
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_upscale.jsonl"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--prof-steps", type=int, default=50)
    ap.add_argument("--regimes", default=",".join(r[0] for r in REGIMES))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_upscale.py needs a CUDA device (there is no CPU fallback)")
    from find_motion_b200 import build
    build.build()
    facts = gpu_facts(args.device)
    want = set(args.regimes.split(","))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for name, W, H, box, bs in REGIMES:
            if name not in want:
                continue
            res = run_regime(name, W, H, box, bs, args)
            res.update(facts)
            line = json.dumps(res)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
