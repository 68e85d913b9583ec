"""RGB, BGRA and RGBA input (FM_FLAG_RGB, FM_FLAG_ALPHA) against BGR input and against converting to BGR first, per regime,
and on the pipelined host path.

One JSON line per regime, printed and appended to --out:
  * bench.py's synthetic scenes in an HBM ring larger than L2 as BGR, and the same ring as RGB (channels flipped), BGRA
    and RGBA (a seeded random alpha byte appended); every arm computes identical results; each call reads the next T
    frames of every stream;
  * frames/s of three arms, alternated window by window in the same run, CUDA events around each window of --steps calls
    after --warmup untimed ones, median of --rounds windows:
      bgr      the BGR ring into a BGR context;
      rgb      the RGB ring into an RGB context (read in place);
      convert  the RGB ring flipped by torch into one preallocated BGR batch per call (three strided channel copies),
               then the BGR context;
      convert_gather  the same flip as one torch.index_select over the channel dimension;
      bgra, rgba      the four-byte rings into BGRA / RGBA contexts (read in place);
      convert_bgra, convert_rgba  the four-byte rings compacted by torch into the BGR batch (one strided copy of the
               first three bytes; three strided channel copies), then the BGR context;
      bgra_no_fused   (full resolution k=5 only) the BGRA ring into a BGRA context without k_fused (FM_FLAG_NO_FUSED):
               the A/B of the four-byte k_fused at three CTAs per SM;
  * B_alg per frame, the bytes the algorithm must move (the frame, the float64 background once per call, the threshold
    bit plane), and a device-to-device cudaMemcpyAsync of B_alg per frame for a call's frames over buffers larger than
    L2, in the same run, with each arm's share of that copy bandwidth.
Then one line for the host path: fm_submit_host / fm_wait on two pinned slots, RGB and BGR batches alternated window by
window, next to a copy-only host-to-device ceiling measured in the same run.  Every line carries the GPU's name, power
limit and maximum SM clock, read in the same run.

    python tools/bench_pixfmt.py [--out profiles/bench_pixfmt.jsonl] [--steps 100] [--rounds 5]

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

from bench_gray import REGIMES, TUNING, alternate, d2d_copy_ms  # noqa: E402
from bench_upscale import gpu_facts, make_ring  # noqa: E402


def run_regime(name, W, H, box, bs, args):
    import torch
    from find_motion_b200.engine import MotionEngine
    S, T, dev = args.streams, args.frames, args.device
    bgr_ring, R = make_ring(W, H, S, T, f"cuda:{dev}")
    rgb_ring = bgr_ring.flip(-1).contiguous()
    g = torch.Generator(device=f"cuda:{dev}").manual_seed(5)
    alpha = torch.randint(0, 256, bgr_ring.shape[:-1] + (1,), generator=g, device=f"cuda:{dev}", dtype=torch.uint8)
    bgra_ring = torch.cat([bgr_ring, alpha], -1)
    rgba_ring = torch.cat([rgb_ring, alpha], -1)
    del alpha
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    calls = R // T
    res = {"regime": name, "W": W, "H": H, "box_size": box, "blur_scale": bs, "streams": S, "frames_per_call": T,
           "ring_frames_per_stream": R, "ring_mb": round(bgr_ring.numel() / 1e6, 1)}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as bgr, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as conv, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, rgb=True, **kw) as rgb, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, alpha=True, **kw) as bgra, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, alpha=True, no_fused=True, **kw) as bgra_nf, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, rgb=True, alpha=True, **kw) as rgba:
        w, h = bgr.w, bgr.h
        assert rgb.info == bgr.info
        res.update(w=w, h=h, gaussian=bgr.info["gaussian"], front_end=rgb.info["front_end"])
        scratch = torch.empty((S, T, H, W, 3), dtype=torch.uint8, device=f"cuda:{dev}")
        first = (rgb.process(rgb_ring[:, :T]), bgr.process(bgr_ring[:, :T]))
        assert (first[0] == first[1]).all(), "RGB and BGR arms disagree"
        assert (bgra.process(bgra_ring[:, :T]) == first[1]).all() and (rgba.process(rgba_ring[:, :T]) == first[1]).all()
        res["front_end_bgra"] = bgra.info["front_end"]
        sl = lambda i: slice((i % calls) * T, (i % calls) * T + T)       # noqa: E731

        order = torch.tensor([2, 1, 0], device=f"cuda:{dev}")

        def convert(i):
            j = (i % calls) * T
            for c in range(3):
                scratch[..., c].copy_(rgb_ring[:, j:j + T, ..., 2 - c])
            return conv.process(scratch, sync=False)

        def convert_gather(i):
            j = (i % calls) * T
            torch.index_select(rgb_ring[:, j:j + T], -1, order, out=scratch)
            return conv.process(scratch, sync=False)
        def convert_bgra(i):
            scratch.copy_(bgra_ring[:, sl(i), ..., :3])
            return conv.process(scratch, sync=False)

        def convert_rgba(i):
            for c in range(3):
                scratch[..., c].copy_(rgba_ring[:, sl(i), ..., 2 - c])
            return conv.process(scratch, sync=False)
        arms = {
            "bgr": lambda i: bgr.process(bgr_ring[:, sl(i)], sync=False),
            "rgb": lambda i: rgb.process(rgb_ring[:, sl(i)], sync=False),
            "convert": convert,
            "convert_gather": convert_gather,
            "bgra": lambda i: bgra.process(bgra_ring[:, sl(i)], sync=False),
            "rgba": lambda i: rgba.process(rgba_ring[:, sl(i)], sync=False),
            "convert_bgra": convert_bgra,
            "convert_rgba": convert_rgba,
        }
        if name == "1080p_full_k5":
            arms["bgra_no_fused"] = lambda i: bgra_nf.process(bgra_ring[:, sl(i)], sync=False)
        res.update(alternate(arms, args, S, T))
        for e in (bgr, conv, rgb, bgra, bgra_nf, rgba):
            e.check()
        res["rgb_over_bgr"] = round(res["frames_per_s_rgb"] / res["frames_per_s_bgr"], 3)
        res["rgb_over_convert"] = round(res["frames_per_s_rgb"] / res["frames_per_s_convert"], 3)
        for k in ("bgra", "rgba"):
            res[f"{k}_over_bgr"] = round(res[f"frames_per_s_{k}"] / res["frames_per_s_bgr"], 3)
            res[f"{k}_over_convert"] = round(res[f"frames_per_s_{k}"] / res[f"frames_per_s_convert_{k}"], 3)
        b_alg = 3.0 * W * H + 16.0 / T * w * h + w * h / 8
        b_alg4 = b_alg + 1.0 * W * H                # the fourth byte is read too
        res.update(b_alg_bytes_per_frame=round(b_alg), b_alg4_bytes_per_frame=round(b_alg4))
        del bgr_ring, rgb_ring, bgra_ring, rgba_ring, scratch
        torch.cuda.empty_cache()
        nbytes = int(b_alg * S * T / 2)
        ms = d2d_copy_ms(nbytes, dev)
        copy_bw = 2 * nbytes / (ms * 1e-3)
        res.update(memcpy_bytes_per_call=nbytes, memcpy_us=round(ms * 1e3, 2), memcpy_gb_per_s=round(copy_bw / 1e9, 1),
                   ceiling_frames_per_s=round(S * T / (ms * 1e-3), 1))
        for k in ("bgr", "rgb", "convert", "convert_gather"):
            res[f"{k}_share_of_copy_bw"] = round(res[f"frames_per_s_{k}"] * b_alg / copy_bw, 3)
        for k in ("bgra", "rgba"):
            res[f"{k}_share_of_copy_bw"] = round(res[f"frames_per_s_{k}"] * b_alg4 / copy_bw, 3)
    torch.cuda.empty_cache()
    return res


def run_host(args):
    """fm_submit_host / fm_wait on two pinned slots (bench.py's end-to-end pattern): RGB against BGR, and the copy-only
    host-to-device rate of the batch bytes"""
    import numpy as np
    import torch
    from find_motion_b200.engine import MotionEngine, PinnedBatch
    name, W, H, box, bs = REGIMES[0]
    S, T, dev = args.streams, args.frames, args.device
    kw = dict(TUNING, box_size=box, blur_scale=bs)
    ring, _ = make_ring(W, H, S, T, f"cuda:{dev}")
    pins = {k: [PinnedBatch((S, T, H, W, 4 if k == "bgra" else 3), dev) for _ in range(2)] for k in ("rgb", "bgr", "bgra")}
    for j in range(2):
        b = ring[:, j * T:(j + 1) * T].cpu().numpy()
        pins["bgr"][j].array[...] = b
        pins["rgb"][j].array[...] = b[..., ::-1]
        pins["bgra"][j].array[..., :3] = b
        pins["bgra"][j].array[..., 3] = 255
    del ring
    torch.cuda.empty_cache()
    res = {"regime": "host_path_" + name, "W": W, "H": H, "streams": S, "frames_per_call": T}
    with torch.cuda.device(dev), MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, **kw) as bgr, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, rgb=True, **kw) as rgb, \
            MotionEngine(W, H, n_streams=S, max_frames=T, device=dev, alpha=True, **kw) as bgra:
        engs = {"rgb": rgb, "bgr": bgr, "bgra": bgra}

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
        res["rgb_over_bgr"] = round(res["frames_per_s_rgb"] / res["frames_per_s_bgr"], 3)
        res["bgra_over_bgr"] = round(res["frames_per_s_bgra"] / res["frames_per_s_bgr"], 3)
    nbytes = S * T * W * H * 3
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
    h2d = reps * nbytes / (time.perf_counter() - t0)
    res.update(h2d_copy_only_gb_per_s=round(h2d / 1e9, 2), ceiling_frames_per_s=round(h2d / (3 * W * H), 1),
               ceiling_frames_per_s_four_byte=round(h2d / (4 * W * H), 1))
    for v in pins.values():
        for p in v:
            p.free()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_pixfmt.jsonl"))
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
        raise SystemExit("bench_pixfmt.py needs a CUDA device (there is no CPU fallback)")
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
