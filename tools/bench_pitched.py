"""Cost of pitched input (fm_process_frames) against packed input and against packing the frames first.

One JSON line per regime, printed and appended to --out:
  * --streams x --frames 1080p frames per call from HBM rings larger than L2 (each call reads the next T frames of every
    stream);
  * three arms over the same frames, alternated window by window in the same run:
      packed  - the frames packed, through fm_process_ragged;
      pitched - the same frames in a pitched ring (BGR rows 6144 bytes apart; NV12 decoder-like surfaces of pitch 2048
                and 1088 coded rows, chroma after them), passed directly through fm_process_frames;
      pack    - the pitched frames packed into a batch first, then processed as packed: the workaround without
                fm_process_frames (BGR: one cudaMemcpy2DAsync per stream; NV12: torch's strided copy, one per plane,
                because the rows of successive surfaces are not evenly spaced);
    frames/s from CUDA events around windows of --steps calls after --warmup untimed ones, median of --rounds windows;
  * kernel times per call of every arm from torch.profiler, in a separate run of --prof-steps calls;
  * the GPU's name, power limit and maximum SM clock, and the clock-throttle reasons, read in the same run.

    python tools/bench_pitched.py [--out profiles/bench_pitched.jsonl] [--steps 100] [--rounds 5]

Needs a CUDA device; there is no CPU fallback.
"""
from __future__ import annotations

import argparse
import ctypes as C
import glob
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_object_planes import kernel_us  # noqa: E402
from bench_upscale import gpu_facts, make_ring  # noqa: E402

# name, box_size, blur_scale, nv12
REGIMES = [("1080p_full_k5", 1920, 384, False), ("1080p_default_box100", 100, 20, False), ("1080p_full_k97", 1920, 20, False),
           ("1080p_nv12_fused_k5", 1920, 384, True), ("1080p_nv12_default_box100", 100, 20, True)]
TUNING = dict(fps=30, min_box_scale=50, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0)
BGR_PITCH, NV12_PITCH, NV12_CODED = 6144, 2048, 1088


def cudart():
    import torch
    cands = glob.glob(os.path.join(os.path.dirname(torch.__file__), "lib", "libcudart.so*"))
    cands += glob.glob(os.path.join(os.path.dirname(os.path.dirname(torch.__file__)), "nvidia", "cuda_runtime", "lib", "libcudart.so*"))
    cands += glob.glob("/usr/local/cuda/lib64/libcudart.so*")
    for p in cands:
        try:
            lib = C.CDLL(p)
            lib.cudaMemcpy2DAsync.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t,
                                              C.c_int, C.c_void_p]
            return lib
        except OSError:
            continue
    raise SystemExit("libcudart not found")


def throttle_reasons(device):
    try:
        return subprocess.run(["nvidia-smi", "-i", str(device), "--query-gpu=clocks.sm,clocks_throttle_reasons.active",
                               "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:
        return f"unavailable: {e}"


def run_regime(name, box, bs, nv12, ring, R, rt, args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, f"cuda:{args.device}"
    W, H = 1920, 1080
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    calls = R // T
    res = {"regime": name, "W": W, "H": H, "box_size": box, "blur_scale": bs, "nv12": nv12, "streams": S,
           "frames_per_call": T, "ring_frames_per_stream": R}
    # the packed ring and the same frames pitched
    if nv12:
        from tests import nv12_restated as N12
        n = min(R, 64)
        nvr = torch.from_numpy(N12.nv12_from_bgr(ring[:, :n].cpu().numpy())).to(dev)       # [S][n][3H/2][W]
        packed = torch.empty((S, R, H * 3 // 2, W), dtype=torch.uint8, device=dev)
        for r0 in range(0, R, n):
            packed[:, r0:r0 + min(n, R - r0)] = nvr[:, :min(n, R - r0)]
        surf = torch.zeros((S, R, NV12_CODED * 3 // 2, NV12_PITCH), dtype=torch.uint8, device=dev)
        surf[..., :H, :W] = packed[:, :, :H]
        surf[..., NV12_CODED:NV12_CODED + H // 2, :W] = packed[:, :, H:]
        luma, uv = surf[..., :H, :W], surf[..., NV12_CODED:NV12_CODED + H // 2, :W]
        res["row_pitch"], res["uv_offset"] = NV12_PITCH, NV12_PITCH * NV12_CODED
    else:
        packed = ring
        canvas = torch.zeros((S, R, H, BGR_PITCH // 3, 3), dtype=torch.uint8, device=dev)
        canvas[:, :, :, :W] = ring
        pitched = canvas[:, :, :, :W]
        res["row_pitch"] = BGR_PITCH
    res["ring_mb_packed"] = round(packed.numel() / 1e6, 1)
    staging = torch.empty((S, T) + tuple(packed.shape[2:]), dtype=torch.uint8, device=dev)
    with torch.cuda.device(args.device), MotionEngine(W, H, n_streams=S, max_frames=T, device=args.device, nv12=nv12, **kw) as e_p, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=args.device, nv12=nv12, **kw) as e_d, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=args.device, nv12=nv12, **kw) as e_c:
        res["front_end"] = e_p.info["front_end"]

        def sl(x, i):
            j = (i % calls) * T
            return x[:, j:j + T]

        def pack(i):
            if nv12:
                staging[:, :, :H].copy_(sl(luma, i))
                staging[:, :, H:].copy_(sl(uv, i))
            else:
                src = sl(pitched, i)
                st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
                for s in range(S):     # T frames of H rows each, evenly spaced: one 2-D copy per stream
                    rc = rt.cudaMemcpy2DAsync(staging[s].data_ptr(), W * 3, src[s].data_ptr(), BGR_PITCH, W * 3, T * H, 3, st)
                    assert rc == 0, rc
            return staging

        arms = {
            "packed": lambda i: e_p.process(sl(packed, i), sync=False),
            "pitched": (lambda i: e_d.process(sl(luma, i), chroma=sl(uv, i), sync=False)) if nv12 else
                       (lambda i: e_d.process(sl(pitched, i), sync=False)),
            "pack": lambda i: e_c.process(pack(i), sync=False),
        }
        # the three arms compute the same thing: checked on one call before timing
        outs = [fn(0).cpu() for fn in arms.values()]
        assert all(torch.equal(outs[0], o) for o in outs[1:]), "arms disagree"
        rates = {k: [] for k in arms}
        i = 1
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
        res["throttle_after_timing"] = throttle_reasons(args.device)
        for e in (e_p, e_d, e_c):
            e.check()
        for k, v in rates.items():
            res[f"frames_per_s_{k}"] = round(statistics.median(v), 1)
            res[f"frames_per_s_{k}_all"] = [round(x, 1) for x in v]
            res[f"ms_per_call_{k}"] = round(S * T / statistics.median(v) * 1e3, 4)
        res["pitched_over_packed"] = round(res["frames_per_s_pitched"] / res["frames_per_s_packed"], 4)
        res["pack_over_packed"] = round(res["frames_per_s_pack"] / res["frames_per_s_packed"], 4)
        for k, fn in arms.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.prof_steps):
                    fn(i)
                    i += 1
                torch.cuda.synchronize()
            kt = {}
            for evt in prof.key_averages():      # the 2-D copies are listed as Memcpy DtoD
                us = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
                if us and "Memcpy" in evt.key:
                    kt[evt.key] = round(us / args.prof_steps, 2)
            kt.update(kernel_us(prof, args.prof_steps))
            res[f"kernel_us_per_call_{k}"] = kt
    del packed, staging
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_pitched.jsonl"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--prof-steps", type=int, default=50)
    ap.add_argument("--regimes", default=",".join(r[0] for r in REGIMES))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_pitched.py needs a CUDA device (there is no CPU fallback)")
    from find_motion_b200 import build
    build.build()
    facts = gpu_facts(args.device)
    rt = cudart()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    ring, R = make_ring(1920, 1080, args.streams, args.frames, f"cuda:{args.device}")
    want = set(args.regimes.split(","))
    for name, box, bs, nv12 in REGIMES:
        if name not in want:
            continue
        res = run_regime(name, box, bs, nv12, ring, R, rt, args)
        res.update(facts)
        line = json.dumps(res)
        print(line, flush=True)
        with open(args.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
