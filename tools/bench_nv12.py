"""Cost of NV12 input (FM_FLAG_NV12) against BGR input, per regime.

One JSON line per regime, printed and appended to --out:
  * the same synthetic scenes as NV12 frames and as their cv2.cvtColor(COLOR_YUV2BGR_NV12) twins (both arms compute
    identical results), each in an HBM ring larger than L2 (each call reads the next T frames of every stream);
  * frames/s of fm_process on BGR input and on NV12 input, the two arms alternated window by window in the same run,
    CUDA events around each window of --steps calls after --warmup untimed ones; median of --rounds windows;
  * B_alg per frame, the bytes the algorithm must move: the frame (3 W H for BGR, 1.5 W H for NV12), the float64
    background once per call (16 w h / T) and the threshold bit plane (w h / 8);
  * as the ceiling, a cudaMemcpyAsync device-to-device copy moving B_alg(NV12) per frame (read + write) for a call's
    frames, over buffers larger than L2, in the same run, and each arm's share of it;
  * with --ab-staged, a third arm: NV12 through the staged path (k_nv12_bgr, then the BGR front end) on every regime,
    from a second copy of the library built with -DFM_NV12_STAGED into a temporary directory, alternated with the
    others in the same run; on the full-resolution k=5 regime this is the A/B of the fused NV12 front end of k_fused
    against staging (elsewhere both copies stage);
  * per-call kernel times of every arm from torch.profiler, in a separate run of --prof-steps calls;
  * the GPU's name, power limit and maximum SM clock, read in the same run.

    python tools/bench_nv12.py [--out profiles/bench_nv12.jsonl] [--steps 100] [--rounds 5]

Needs a CUDA device; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_upscale import L2_BYTES, gpu_facts, make_ring  # noqa: E402

# name, W, H, box_size, blur_scale: bench.py's full-resolution k=5, default-mode and k=97 regimes
REGIMES = [
    ("1080p_full_k5", 1920, 1080, 1920, 384),
    ("1080p_default_box100", 1920, 1080, 100, 20),
    ("1080p_full_k97", 1920, 1080, 1920, 20),
]
TUNING = dict(fps=30, min_box_scale=50, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)


def nv12_rings(W, H, S, T, device):
    """-> (nv12 [S][R][H*3/2][W], bgr [S][R][H][W][3] = cv2's conversion of it, R)"""
    import cv2
    import numpy as np
    import torch
    ring, R = make_ring(W, H, S, T, device)
    host = ring.cpu().numpy()
    del ring
    nv = np.empty((S, R, H * 3 // 2, W), np.uint8)
    for s in range(S):
        for r in range(R):
            yuv = cv2.cvtColor(host[s, r], cv2.COLOR_BGR2YUV_I420)
            nv[s, r, :H] = yuv[:H]
            c = yuv[H:].reshape(2, H // 2, W // 2)            # the U plane, then the V plane
            nv[s, r, H:] = np.stack([c[0], c[1]], -1).reshape(H // 2, W)
            host[s, r] = cv2.cvtColor(nv[s, r], cv2.COLOR_YUV2BGR_NV12)
    return torch.from_numpy(nv).to(device), torch.from_numpy(host).to(device), R


def staged_lib():
    """libfmgpu.so built with -DFM_NV12_STAGED (every NV12 configuration staged) into a temporary directory, loaded
    with every symbol bound."""
    import ctypes
    import subprocess
    import tempfile
    from find_motion_b200 import _lib, build
    path = os.path.join(tempfile.mkdtemp(prefix="fm_nv12_ab_"), "libfmgpu_staged.so")
    subprocess.run([build.find_nvcc()] + build.NVCC_FLAGS + ["-DFM_NV12_STAGED", "-o", path] + build.sources(),
                   check=True, cwd=build.CSRC)
    lib = ctypes.CDLL(path)
    for name, (res, argtypes) in _lib.SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, argtypes
    return lib


def engine_on(lib, *a, **kw):
    """MotionEngine bound to `lib` instead of the in-tree library"""
    from find_motion_b200 import _lib
    from find_motion_b200.engine import MotionEngine
    saved = _lib._lib
    _lib._lib = lib
    try:
        return MotionEngine(*a, **kw)
    finally:
        _lib._lib = saved


def run_regime(name, W, H, box, bs, args, alt_lib=None):
    import contextlib
    import torch
    from torch.profiler import ProfilerActivity, profile
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    nv_ring, bgr_ring, R = nv12_rings(W, H, S, T, f"cuda:{dev}")
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    calls = R // T
    res = {"regime": name, "W": W, "H": H, "box_size": box, "blur_scale": bs, "streams": S, "frames_per_call": T,
           "ring_frames_per_stream": R, "ring_mb_nv12": round(nv_ring.numel() / 1e6, 1),
           "ring_mb_bgr": round(bgr_ring.numel() / 1e6, 1)}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as bgr, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, nv12=True, **kw) as nv12, \
            (engine_on(alt_lib, W, H, n_streams=S, max_frames=T, device=dev, nv12=True, **kw) if alt_lib
             else contextlib.nullcontext()) as staged:
        w, h = bgr.w, bgr.h
        res.update(w=w, h=h, gaussian=bgr.info["gaussian"], front_end=nv12.info["front_end"])
        arms = {
            "bgr": lambda i: bgr.process(bgr_ring[:, (i % calls) * T:(i % calls) * T + T], sync=False),
            "nv12": lambda i: nv12.process(nv_ring[:, (i % calls) * T:(i % calls) * T + T], sync=False),
        }
        if staged is not None:
            arms["nv12_staged"] = lambda i: staged.process(nv_ring[:, (i % calls) * T:(i % calls) * T + T], sync=False)
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
        bgr.check()
        nv12.check()
        if staged is not None:
            staged.check()
        for k, v in rates.items():
            res[f"frames_per_s_{k}"] = round(statistics.median(v), 1)
            res[f"frames_per_s_{k}_all"] = [round(x, 1) for x in v]
        res["nv12_over_bgr"] = round(res["frames_per_s_nv12"] / res["frames_per_s_bgr"], 3)
        if staged is not None:
            res["nv12_over_nv12_staged"] = round(res["frames_per_s_nv12"] / res["frames_per_s_nv12_staged"], 3)

        # kernel times per call, in a run of their own per arm
        for k, fn in arms.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.prof_steps):
                    fn(i)
                    i += 1
                torch.cuda.synchronize()
            kt = {}
            for evt in prof.key_averages():
                us = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
                kname = evt.key.split("(")[0].split("<")[0].strip().split(" ")[-1]      # "void k_x<...>(...)" -> k_x
                if us and kname.startswith("k_"):
                    kt[kname] = kt.get(kname, 0.0) + us / args.prof_steps
            staged_arm = k == "nv12_staged" or (k == "nv12" and res["front_end"] != 0)
            if k != "bgr" and staged_arm != ("k_nv12_bgr" in kt):
                raise RuntimeError(f"arm {k}: k_nv12_bgr {'missing from' if staged_arm else 'in'} the profile")
            res[f"kernel_us_per_call_{k}"] = {n: round(v, 2) for n, v in sorted(kt.items())}

        # B_alg and the copy ceiling: cudaMemcpyAsync moving B_alg(NV12) per frame (read + write) for one call's frames
        b_nv12 = 1.5 * W * H + 16.0 / T * w * h + w * h / 8
        b_bgr = 3.0 * W * H + 16.0 / T * w * h + w * h / 8
        res.update(b_alg_nv12_bytes_per_frame=round(b_nv12), b_alg_bgr_bytes_per_frame=round(b_bgr))
        nbytes = int(b_nv12 * S * T / 2)
        nbuf = max(2, -(-3 * L2_BYTES // nbytes) + 1)
        del nv_ring, bgr_ring
        torch.cuda.empty_cache()
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
        ms = e0.elapsed_time(e1) / reps
        ceil_fps = S * T / (ms * 1e-3)
        res.update(memcpy_bytes_per_call=nbytes, memcpy_us=round(ms * 1e3, 2),
                   memcpy_gb_per_s=round(2 * nbytes / (ms * 1e-3) / 1e9, 1),
                   ceiling_frames_per_s_nv12=round(ceil_fps, 1),
                   nv12_share_of_ceiling=round(res["frames_per_s_nv12"] / ceil_fps, 3),
                   nv12_b_alg_gb_per_s=round(res["frames_per_s_nv12"] * b_nv12 / 1e9, 1),
                   bgr_b_alg_gb_per_s=round(res["frames_per_s_bgr"] * b_bgr / 1e9, 1))
        del bufs
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_nv12.jsonl"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--prof-steps", type=int, default=50)
    ap.add_argument("--regimes", default=",".join(r[0] for r in REGIMES))
    ap.add_argument("--ab-staged", action="store_true", help="add the staged-path arm (a -DFM_NV12_STAGED build)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_nv12.py needs a CUDA device (there is no CPU fallback)")
    from find_motion_b200 import build
    build.build()
    facts = gpu_facts(args.device)
    alt = staged_lib() if args.ab_staged else None
    want = set(args.regimes.split(","))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        for name, W, H, box, bs in REGIMES:
            if name not in want:
                continue
            res = run_regime(name, W, H, box, bs, args, alt)
            res.update(facts)
            line = json.dumps(res)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
