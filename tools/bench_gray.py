"""Gray input (FM_FLAG_GRAY) against BGR input, per regime, and on the pipelined host path.

One JSON line per regime, printed and appended to --out:
  * the same synthetic scenes as gray frames (cv2 COLOR_BGR2GRAY of bench.py's ring) and as their COLOR_GRAY2BGR twins
    (both arms compute identical results), each in an HBM ring larger than L2 (each call reads the next T frames of every
    stream);
  * frames/s of fm_process on BGR input and on gray input, the two arms alternated window by window in the same run,
    CUDA events around each window of --steps calls after --warmup untimed ones; median of --rounds windows;
  * B_alg per frame, the bytes the algorithm must move: the frame (3 W H for BGR, W H for gray), the float64 background
    once per call (16 w h / T) and the threshold bit plane (w h / 8);
  * as the ceiling, a device-to-device cudaMemcpyAsync moving B_alg(gray) per frame (read + write) for a call's frames,
    over buffers larger than L2, in the same run, and each arm's share of it.
Then one line for the host path: fm_submit_host / fm_wait on two pinned slots, gray and BGR batches alternated window by
window, next to a copy-only host-to-device ceiling (pinned -> device copies of the gray batch bytes) measured in the same
run.  Every line carries the GPU's name, power limit and maximum SM clock, read in the same run.

    python tools/bench_gray.py [--out profiles/bench_gray.jsonl] [--steps 100] [--rounds 5]

Needs a CUDA device; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_upscale import L2_BYTES, gpu_facts, make_ring  # noqa: E402

# name, W, H, box_size, blur_scale: bench.py's full-resolution k=5, k=97 and default-mode regimes
REGIMES = [
    ("1080p_full_k5", 1920, 1080, 1920, 384),
    ("1080p_full_k97", 1920, 1080, 1920, 20),
    ("1080p_default_box100", 1920, 1080, 100, 20),
]
TUNING = dict(fps=30, min_box_scale=50, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)


def gray_rings(W, H, S, T, device):
    """-> (gray [S][R][H][W], bgr [S][R][H][W][3] = its COLOR_GRAY2BGR twin, R): the gray ring, too, holds more than 3x L2"""
    import math
    import cv2
    import numpy as np
    import torch
    ring, R0 = make_ring(W, H, S, T, device)
    host = ring.cpu().numpy()
    del ring
    R = max(R0, math.ceil(3 * L2_BYTES / (S * W * H) / T) * T)
    g = np.empty((S, R, H, W), np.uint8)
    for s in range(S):
        for r in range(R0):
            g[s, r] = cv2.cvtColor(host[s, r], cv2.COLOR_BGR2GRAY)
        for r in range(R0, R):
            g[s, r] = g[s, r % R0]
    del host
    gd = torch.from_numpy(g).to(device)
    return gd, gd.unsqueeze(-1).expand(S, R, H, W, 3).contiguous(), R


def alternate(arms, args, S, T):
    """{arm: median frames/s, arm_all: every window}: arms alternated window by window, CUDA events around each"""
    import torch
    rates = {k: [] for k in arms}
    i = 0
    for fn in arms.values():
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
    out = {}
    for k, v in rates.items():
        out[f"frames_per_s_{k}"] = round(statistics.median(v), 1)
        out[f"frames_per_s_{k}_all"] = [round(x, 1) for x in v]
    return out


def d2d_copy_ms(nbytes, dev):
    import torch
    nbuf = max(2, -(-3 * L2_BYTES // nbytes) + 1)
    bufs = [torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{dev}") for _ in range(nbuf)]
    for j in range(nbuf):
        bufs[(j + 1) % nbuf].copy_(bufs[j])
    torch.cuda.synchronize()
    reps = 100
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for j in range(reps):
        bufs[(j + 1) % nbuf].copy_(bufs[j % nbuf])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_regime(name, W, H, box, bs, args):
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    g_ring, bgr_ring, R = gray_rings(W, H, S, T, f"cuda:{dev}")
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    calls = R // T
    res = {"regime": name, "W": W, "H": H, "box_size": box, "blur_scale": bs, "streams": S, "frames_per_call": T,
           "ring_frames_per_stream": R, "ring_mb_gray": round(g_ring.numel() / 1e6, 1),
           "ring_mb_bgr": round(bgr_ring.numel() / 1e6, 1)}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as bgr, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, gray=True, **kw) as gray:
        w, h = bgr.w, bgr.h
        assert gray.info == bgr.info
        res.update(w=w, h=h, gaussian=bgr.info["gaussian"], front_end=gray.info["front_end"])
        first = (gray.process(g_ring[:, :T]), bgr.process(bgr_ring[:, :T]))
        assert (first[0] == first[1]).all(), "gray and BGR arms disagree"
        arms = {
            "bgr": lambda i: bgr.process(bgr_ring[:, (i % calls) * T:(i % calls) * T + T], sync=False),
            "gray": lambda i: gray.process(g_ring[:, (i % calls) * T:(i % calls) * T + T], sync=False),
        }
        res.update(alternate(arms, args, S, T))
        bgr.check()
        gray.check()
        res["gray_over_bgr"] = round(res["frames_per_s_gray"] / res["frames_per_s_bgr"], 3)
        b_gray = 1.0 * W * H + 16.0 / T * w * h + w * h / 8
        b_bgr = 3.0 * W * H + 16.0 / T * w * h + w * h / 8
        res.update(b_alg_gray_bytes_per_frame=round(b_gray), b_alg_bgr_bytes_per_frame=round(b_bgr))
        del g_ring, bgr_ring
        torch.cuda.empty_cache()
        nbytes = int(b_gray * S * T / 2)
        ms = d2d_copy_ms(nbytes, dev)
        ceil_fps = S * T / (ms * 1e-3)
        copy_bw = 2 * nbytes / (ms * 1e-3)
        res.update(memcpy_bytes_per_call=nbytes, memcpy_us=round(ms * 1e3, 2), memcpy_gb_per_s=round(copy_bw / 1e9, 1),
                   ceiling_frames_per_s_gray=round(ceil_fps, 1),
                   gray_share_of_copy_bw=round(res["frames_per_s_gray"] * b_gray / copy_bw, 3),
                   bgr_share_of_copy_bw=round(res["frames_per_s_bgr"] * b_bgr / copy_bw, 3))
    torch.cuda.empty_cache()
    return res


def run_host(args):
    """fm_submit_host / fm_wait on two pinned slots (bench.py's end-to-end pattern): gray against BGR, and the copy-only
    host-to-device rate of the gray batch bytes"""
    import numpy as np
    import torch
    from find_motion_b200.engine import MotionEngine, PinnedBatch
    name, W, H, box, bs = REGIMES[0]
    S, T, dev = args.streams, args.frames, args.device
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    g_ring, bgr_ring, _ = gray_rings(W, H, S, T, f"cuda:{dev}")
    pins = {"gray": [PinnedBatch((S, T, H, W), dev) for _ in range(2)],
            "bgr": [PinnedBatch((S, T, H, W, 3), dev) for _ in range(2)]}
    for j in range(2):
        pins["gray"][j].array[...] = g_ring[:, j * T:(j + 1) * T].cpu().numpy()
        pins["bgr"][j].array[...] = bgr_ring[:, j * T:(j + 1) * T].cpu().numpy()
    del g_ring, bgr_ring
    torch.cuda.empty_cache()
    res = {"regime": "host_path_" + name, "W": W, "H": H, "streams": S, "frames_per_call": T}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as bgr, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, gray=True, **kw) as gray:
        engs = {"gray": gray, "bgr": bgr}

        def window(k, n):
            e, p = engs[k], pins[k]
            t0 = time.perf_counter()
            for j in range(n):
                if j >= 2:
                    e.wait_host(j & 1)
                e.submit_host(j & 1, p[j & 1].array)
            for j in range(max(0, n - 2), n):
                e.wait_host(j & 1)
            return n * S * T / (time.perf_counter() - t0)
        for k in engs:
            window(k, 10)
        rates = {k: [] for k in engs}
        for _ in range(args.rounds):
            for k in engs:
                rates[k].append(window(k, args.host_steps))
        for k, v in rates.items():
            res[f"frames_per_s_{k}"] = round(statistics.median(v), 1)
            res[f"frames_per_s_{k}_all"] = [round(x, 1) for x in v]
        res["gray_over_bgr"] = round(res["frames_per_s_gray"] / res["frames_per_s_bgr"], 3)
    # copy-only ceiling: pinned host -> device copies of a gray batch
    nbytes = S * T * W * H
    src = torch.from_numpy(np.zeros(nbytes, np.uint8)).pin_memory()
    dst = torch.empty(nbytes, dtype=torch.uint8, device=f"cuda:{dev}")
    for _ in range(5):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    reps = args.host_steps
    t0 = time.perf_counter()
    for _ in range(reps):
        dst.copy_(src, non_blocking=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    h2d = reps * nbytes / dt
    res.update(h2d_copy_only_gb_per_s=round(h2d / 1e9, 2),
               ceiling_frames_per_s_gray=round(h2d / (W * H), 1), ceiling_frames_per_s_bgr=round(h2d / (3 * W * H), 1),
               gray_h2d_gb_per_s=round(res["frames_per_s_gray"] * W * H / 1e9, 2),
               bgr_h2d_gb_per_s=round(res["frames_per_s_bgr"] * 3 * W * H / 1e9, 2))
    for v in pins.values():
        for p in v:
            p.free()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_gray.jsonl"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--host-steps", type=int, default=40)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--regimes", default=",".join(r[0] for r in REGIMES) + ",host")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_gray.py needs a CUDA device (there is no CPU fallback)")
    from find_motion_b200 import build
    build.build()
    facts = gpu_facts(args.device)
    want = set(args.regimes.split(","))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        todo = [(n, lambda r=r: run_regime(*r, args)) for r in REGIMES for n in [r[0]] if n in want]
        if "host" in want:
            todo.append(("host", lambda: run_host(args)))
        for _, fn in todo:
            res = fn()
            res.update(facts)
            line = json.dumps(res)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
