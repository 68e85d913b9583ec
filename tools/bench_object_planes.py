"""Cost of the detector input planes (FM_FLAG_OBJECT_PLANES, fm_object_planes) on 1080p calls.

One JSON line per regime and scene, printed and appended to --out:
  * --streams x --frames 1080p frames per call from an HBM ring larger than L2 (each call reads the next T frames of
    every stream), at bench.py's full-resolution k=5 and default-mode tunings;
  * two scenes: "moving" (min_time 0: every frame is written) and "quiet" (min_time 1e6 s: no frame is);
  * three arms, alternated window by window in the same run: the flag off, the flag on without fm_object_planes, the
    flag on with fm_object_planes after every call; frames/s from CUDA events around windows of --steps calls after
    --warmup untimed ones, median of --rounds windows;
  * kernel times per call of every arm from torch.profiler, in a separate run of --prof-steps calls;
  * bytes per written frame 3 W H + 3 * 300 * oh (the frame read, the plane written) over the time of the plane kernels,
    against a same-run cudaMemcpyAsync device-to-device copy of those bytes for a call's frames;
  * an A/B of the resize of the planes: the rows kernel (k_resize_rows<true>) against the fallback (k_resize_gray, the
    library's FM_FLAG_NO_ROWS), fm_object_planes alone on the frames of one moving call, 1080p and 4K;
  * the GPU's name, power limit and maximum SM clock, read in the same run.

    python tools/bench_object_planes.py [--out profiles/bench_object_planes.jsonl] [--steps 100] [--rounds 5]

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

# name, box_size, blur_scale: bench.py's full-resolution k=5 and default-mode regimes
REGIMES = [("1080p_full_k5", 1920, 384), ("1080p_default_box100", 100, 20)]
SCENES = {"moving": 0.0, "quiet": 1e6}          # min_time: 0 -> every frame written, 1e6 s -> none
TUNING = dict(fps=30, min_box_scale=50, threshold=12, avg=0.1, cache_time=1.0)


def kernel_us(prof, steps):
    kt = {}
    for evt in prof.key_averages():
        us = getattr(evt, "device_time_total", None) or getattr(evt, "cuda_time_total", 0.0)
        name = evt.key.split("(")[0].strip().split(" ")[-1]          # "void k_x<true>(...)" -> k_x<true>
        if us and name.startswith("k_"):
            kt[name] = kt.get(name, 0.0) + us / steps
    return {n: round(v, 2) for n, v in sorted(kt.items())}


def memcpy_us(nbytes, dev):
    """cudaMemcpyAsync device to device of nbytes, over buffers that together exceed L2 (us per copy)"""
    import torch
    nbuf = max(2, -(-3 * L2_BYTES // nbytes) + 1)
    bufs = [torch.empty(nbytes, dtype=torch.uint8, device=dev) for _ in range(nbuf)]
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
    return e0.elapsed_time(e1) / reps * 1e3


def run_regime(name, box, bs, scene, ring, R, args):
    import torch
    from torch.profiler import ProfilerActivity, profile
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    W, H = 1920, 1080
    kw = dict(TUNING, box_size=box, blur_scale=bs, min_time=SCENES[scene])
    calls = R // T
    res = {"regime": name, "scene": scene, "W": W, "H": H, "box_size": box, "blur_scale": bs, "streams": S,
           "frames_per_call": T, "ring_frames_per_stream": R, "ring_mb": round(ring.numel() / 1e6, 1)}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as off, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, object_planes=True, **kw) as on:
        oh = on.object_shape[0]
        out = torch.empty((S, T) + on.object_shape, dtype=torch.uint8, device=f"cuda:{dev}")
        res.update(front_end=on.info["front_end"], object_h=oh)

        def batch(i):
            j = (i % calls) * T
            return ring[:, j:j + T]

        def planes():
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            rc = on._lib.fm_object_planes(on._ctx, st, out.data_ptr(), out.stride(0), T)
            assert rc == 0, rc

        arms = {
            "off": lambda i: off.process(batch(i), sync=False),
            "flag": lambda i: on.process(batch(i), sync=False),
            "planes": lambda i: (on.process(batch(i), sync=False), planes()),
        }
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
        off.check()
        on.check()
        for k, v in rates.items():
            res[f"frames_per_s_{k}"] = round(statistics.median(v), 1)
            res[f"frames_per_s_{k}_all"] = [round(x, 1) for x in v]
        res["planes_over_off"] = round(res["frames_per_s_planes"] / res["frames_per_s_off"], 3)
        res["flag_over_off"] = round(res["frames_per_s_flag"] / res["frames_per_s_off"], 3)
        stats = on.process(batch(i))
        i += 1
        written = int(stats["wrote"].sum())
        res["written_per_call"] = written
        for k, fn in arms.items():
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.prof_steps):
                    fn(i)
                    i += 1
                torch.cuda.synchronize()
            res[f"kernel_us_per_call_{k}"] = kernel_us(prof, args.prof_steps)
        kt = res["kernel_us_per_call_planes"]
        plane_us = sum(v for n, v in kt.items() if n.startswith(("k_object_plan", "k_resize_rows<true>", "k_resize_gray")))
        res["plane_kernels_us_per_call"] = round(plane_us, 2)
        bytes_per_frame = 3 * W * H + 3 * 300 * oh
        res["bytes_per_written_frame"] = bytes_per_frame
        if written:
            res["plane_gb_per_s"] = round(written * bytes_per_frame / (plane_us * 1e-6) / 1e9, 1)
            cp = memcpy_us(written * bytes_per_frame // 2, f"cuda:{dev}")      # reads half, writes half: the same traffic
            res["memcpy_us_same_bytes"] = round(cp, 2)
            res["memcpy_gb_per_s"] = round(written * bytes_per_frame / (cp * 1e-6) / 1e9, 1)
            res["plane_share_of_memcpy"] = round(cp / plane_us, 3)
    torch.cuda.empty_cache()
    return res


def rows_ab(W, H, args):
    """fm_object_planes alone on one moving call: the rows kernel against the fallback (FM_FLAG_NO_ROWS)"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    ring, R = make_ring(W, H, S, T, f"cuda:{dev}")
    kw = dict(TUNING, box_size=W, blur_scale=W // 5, min_time=0.0)
    res = {"regime": f"rows_ab_{W}x{H}", "W": W, "H": H, "streams": S, "frames_per_call": T,
           "call_mb": round(S * T * W * H * 3 / 1e6, 1)}
    with torch.cuda.device(dev), \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, object_planes=True, **kw) as rows, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, object_planes=True, no_rows=True, **kw) as k0:
        out = torch.empty((S, T) + rows.object_shape, dtype=torch.uint8, device=f"cuda:{dev}")
        engines = {"rows": rows, "resize_gray": k0}
        for e in engines.values():
            assert int(e.process(ring[:, :T])["wrote"].sum()) == S * T

        def planes(e):
            st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            assert e._lib.fm_object_planes(e._ctx, st, out.data_ptr(), out.stride(0), T) == 0

        got = {}
        for k, e in engines.items():
            planes(e)
            got[k] = out.clone()
        assert torch.equal(got["rows"], got["resize_gray"])
        times = {k: [] for k in engines}
        for k, e in engines.items():
            for _ in range(args.warmup):
                planes(e)
        for _ in range(args.rounds):
            for k, e in engines.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    planes(e)
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / args.steps * 1e3)
        for k, v in times.items():
            res[f"us_per_call_{k}"] = round(statistics.median(v), 2)
            res[f"us_per_call_{k}_all"] = [round(x, 2) for x in v]
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(args.prof_steps):
                    planes(engines[k])
                torch.cuda.synchronize()
            res[f"kernel_us_per_call_{k}"] = kernel_us(prof, args.prof_steps)
        res["rows_speedup"] = round(res["us_per_call_resize_gray"] / res["us_per_call_rows"], 3)
    del ring
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_object_planes.jsonl"))
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("--streams", type=int, default=8)
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--prof-steps", type=int, default=50)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_object_planes.py needs a CUDA device (there is no CPU fallback)")
    from find_motion_b200 import build
    build.build()
    facts = gpu_facts(args.device)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    lines = []
    ring, R = make_ring(1920, 1080, args.streams, args.frames, f"cuda:{args.device}")
    for name, box, bs in REGIMES:
        for scene in SCENES:
            lines.append(run_regime(name, box, bs, scene, ring, R, args))
    del ring
    for W, H in ((1920, 1080), (3840, 2160)):
        lines.append(rows_ab(W, H, args))
    with open(args.out, "a") as f:
        for res in lines:
            res.update(facts)
            line = json.dumps(res)
            print(line, flush=True)
            f.write(line + "\n")


if __name__ == "__main__":
    main()
