#!/usr/bin/env python
"""bench.py -- 1080p frames/s of the motion-detection hot path on N B200s (+ HBM roofline).

A step = one pass of the hot path (fm_process) over one batch of synthetic input: S streams x T
frames of 1920x1080 BGR per GPU, taken from an HBM-resident ring of R frames per stream (ring >
L2, so no step re-reads cached input).  Streams are independent, so ranks share nothing on the
data path (weak scaling: S streams per GPU); the only collective is the max-over-ranks of the
timed region.  `value` is whole-job frames/s with inputs resident in HBM; `e2e` is the same
through the host-buffer entry point (fm_process_host: pinned host frames -> H2D -> kernels ->
stats D2H, every step).  `--impl reference` times the reference's CPU path (the cv2 call chain
of find_motion.py:852-904 re-typed in oracle/cv2_chain.py, one process per stream over all host
cores, as run_pool does) on the same configuration.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

W, H = 1920, 1080
METRIC = "1080p frames/sec (whole box)"   # other --size values are characterisation runs


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="full", choices=["full", "default"],
                    help="full = --box-size 1920 (full-resolution stencil); default = reference default --box-size 100")
    ap.add_argument("--blur-scale", type=int, default=None,
                    help="reference --blur-scale; full mode default 384 (k=5, HBM-bound regime), 20 gives k=97")
    ap.add_argument("--streams", type=int, default=8, help="streams per GPU")
    ap.add_argument("--frames", type=int, default=16, help="T: frames per stream per step")
    ap.add_argument("--ring", type=int, default=32, help="frames per stream resident in HBM")
    ap.add_argument("--e2e-steps", type=int, default=32)
    ap.add_argument("--min-seconds", type=float, default=0.0,
                    help="repeat the K-step block until the timed region lasts at least this long (sustained clocks); "
                         "0 = exactly K timed steps")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (see dump_outputs)")
    ap.add_argument("--size", default="1920x1080", help="frame size WxH (the headline metric is 1080p)")
    ap.add_argument("--distinct", type=int, default=0, help="distinct synthetic clips (0 = one per stream); "
                    "streams reuse them round-robin (large-batch sweeps)")
    ap.add_argument("--front-end", default="auto", choices=["auto", "stencil", "umma", "umma-apron", "mma-sync", "warp-resize"],
                    help="A/B of the front-end kernels: stencil = k_fused (k <= 5), umma = tcgen05 kernel fed by the BGR frames, "
                         "umma-apron = tcgen05 kernel through the apron plane, mma-sync = the two-pass mma.sync Gaussian, "
                         "warp-resize = default mode with the warp-per-destination-row INTER_AREA kernels instead of the row-per-lane one")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary regimes (k=97, default mode)")
    return ap.parse_args()


def tuning(mode, blur_scale):
    from find_motion_b200 import synth
    kw = dict(fps=30, min_box_scale=50, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0,
              mask_areas=synth.CFG2_MASKS)
    if mode == "full":
        kw.update(box_size=W, blur_scale=blur_scale if blur_scale else 384)
    else:
        kw.update(box_size=100, blur_scale=blur_scale if blur_scale else 20)
    return kw


def bench_script(ring):
    # one walker episode per ring pass, the rest quiet: a mix of motion and idle frames
    return [("walker", ring // 4, ring // 4 + max(4, ring // 3)), ("hidden", 2, ring // 2)]


def alg_bytes_per_frame(w, h, T, m=1.0 / 8):
    """SURVEY.md 8(d): BGR in once + float64 background in/out once per T frames + m B/px mask out."""
    return 3.0 * W * H + (16.0 / T) * w * h + m * w * h


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._halt = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.01)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def cpu_baseline(kw, cores, target_s=2.5):
    """Reference CPU path on a bounded sample: one stream per process over all host cores."""
    from oracle import cv2_chain
    probe = cv2_chain.time_cpu_path(W, H, kw, 1, 4, 1, clip_len=4)
    per_frame = probe["seconds"] / 4
    frames = max(4, min(400, int(target_s / per_frame)))
    r = cv2_chain.time_cpu_path(W, H, kw, cores, frames, cores, clip_len=8)
    out = {"value": round(r["fps"], 2), "unit": "frames/s", "cores": r["processes"], "kind": "port",
           "sample": f"{cores} synthetic {W}x{H} streams x {frames} frames, one process per stream "
                     f"({r['engine']}, cv2 threads/process = {r['cv_threads']}), decode/encode excluded",
           "seconds": round(r["seconds"], 3)}
    # the two other variants SURVEY.md 8(d) asks for (bounded to a few seconds each)
    variants = {}
    try:
        v = cv2_chain.time_cpu_path(W, H, kw, cores, max(4, frames // 2), cores, clip_len=8, cv_threads=0)
        variants["cv2_threads_default_oversubscribed"] = {
            "value": round(v["fps"], 2), "unit": "frames/s",
            "sample": f"{cores} processes, cv2 threads = cores in each (the reference's implicit default), from memory"}
        nf = max(4, min(64, frames // 4))
        v = cv2_chain.time_cpu_path(W, H, kw, cores, nf, cores, clip_len=8, source="ffv1")
        variants["ffv1_decode_included"] = {
            "value": round(v["fps"], 2), "unit": "frames/s",
            "sample": f"{cores} processes x {nf} frames pulled through cv2.VideoCapture from a lossless FFV1 file each"}
    except Exception as e:
        variants["error"] = str(e)[:200]
    out["variants"] = variants
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kw = tuning(args.mode, args.blur_scale)
    cores = os.cpu_count() or 1
    from oracle import cv2_chain
    probe = cv2_chain.time_cpu_path(W, H, kw, 1, 4, 1, clip_len=4)
    per_frame = probe["seconds"] / 4
    # bounded sample: the whole warm-up + K steps loop of a worker lasts ~45 s at most
    frames = max(1, min(400, int(45.0 / per_frame / max(1, args.steps + args.warmup))))
    r = cv2_chain.time_cpu_path(W, H, kw, cores, frames, cores, clip_len=8, steps=args.steps, warmup=args.warmup)
    tot_f, tot_s = r["frames"], r["seconds"]
    fps = tot_f / tot_s
    info = probe_info(kw)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(fps, 2), "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * tot_s / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8+f64", "data": "synthetic",
        "config": workload_config(args, kw, info),
        "cpu_baseline": {"value": round(fps, 2), "unit": "frames/s", "cores": cores, "kind": "port",
                         "sample": f"{cores} synthetic 1080p streams x {frames} frames per step, one process per "
                                   f"stream ({r['engine']}, cv2 threads/process = 1), decode/encode excluded"},
        "e2e": {"value": round(fps, 2), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def probe_info(kw):
    from oracle import restated as R
    return R.derive_params(W, H, kw["fps"], kw["box_size"], kw["min_box_scale"], kw["cache_time"], kw["min_time"],
                           kw["blur_scale"])


def workload_config(args, kw, info):
    return {
        "workload": f"BASELINE configs[1]/[2]: {args.streams} x {W}x{H} synthetic streams per GPU "
                    f"({args.streams * args.gpus} in the job; 64 at 8 GPUs = configs[2]), CFG2 polygon masks "
                    f"(README square+triangle + translated pair), min-time/cache-time logic, "
                    f"{'full-resolution' if args.mode == 'full' else 'reference-default'} mode",
        "frame": f"{W}x{H} BGR u8", "proc": f"{info['w']}x{info['h']}", "gaussian": info["gaussian"],
        "box_size": kw["box_size"], "blur_scale": kw["blur_scale"], "threshold": kw["threshold"], "avg": kw["avg"],
        "min_time": kw["min_time"], "cache_time": kw["cache_time"], "fps": kw["fps"],
        "streams_per_gpu": args.streams, "frames_per_step_per_stream": args.frames, "ring_frames": args.ring,
        "front_end": args.front_end,
        "l2_policy": f"inputs larger than L2: ring of {args.ring} frames/stream = "
                     f"{args.streams * args.ring * W * H * 3 / 1e6:.0f} MB per GPU, each step reads the next T frames",
        "parallelism": f"streams sharded over {args.gpus} GPU(s), no data-path collective",
    }


def time_engine(eng, ring_dev, args, torch, dist, world):
    """warm-up, then EXACTLY K timed steps (a multiple of K with --min-seconds) between two CUDA events; returns ms (max
    over ranks), the step count, the launch count and the device stats of the last step."""
    R, T = args.ring, args.frames
    nslots = R // T

    def step(i):
        a = (i % nslots) * T
        return eng.process(ring_dev[:, a:a + T], sync=False)

    eng.timing(enable=False)                 # warm-up calls stay out of the kernel-group times
    for i in range(args.warmup):
        step(i)
    # how often the K-step block must repeat for the timed region to last --min-seconds (same count on every rank)
    reps = 1
    if getattr(args, "min_seconds", 0) > 0:
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(args.steps):
            step(args.warmup + i)
        c1.record()
        torch.cuda.synchronize()
        est = torch.tensor([c0.elapsed_time(c1) / 1e3], device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(est, op=dist.ReduceOp.MIN)
        reps = max(1, int(-(-args.min_seconds // max(float(est.item()), 1e-6))))
    eng.timing(enable=True, reset=True)      # no call is pending, so neither waits for the device
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    from find_motion_b200.engine import launch_count
    l0 = launch_count()
    # queued behind the warm-up steps still in flight: the K timed steps start on a busy device, as inside a long run,
    # rather than after an idle gap and the launch latency of their first step
    e0.record()
    for i in range(args.steps * reps):
        stats = step(args.warmup + i)
    e1.record()
    launches = launch_count() - l0
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    eng.check()
    return ms, args.steps * reps, launches, stats


def main():
    global W, H
    args = parse_args()
    W, H = (int(v) for v in args.size.lower().split("x"))
    if args.impl == "reference":
        return run_reference(args)
    # libraries (NCCL's version banner, ...) write to fd 1; keep stdout clean for the ONE JSON line
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    try:
        line = run_b200(args)
    finally:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        os.close(saved_stdout)
    if line is not None:
        print(json.dumps(line), flush=True)


def measure(eng, ring_dev, args, torch, dist, world, S, T, launch_count, local):
    """Timed region of one regime: throughput, per-kernel-group times (CUDA events on the launching stream, recorded
    inside the timed region), launch count and the clocks seen under load."""
    eng.timing(enable=True, reset=True)
    for i in range(2):                       # untimed priming pass
        eng.process(ring_dev[:, :T], sync=False)
    torch.cuda.synchronize()
    eng.reset()
    sampler = ClockSampler(local)
    sampler.start()
    ms, timed_steps, launches, stats = time_engine(eng, ring_dev, args, torch, dist, world)
    clocks = sampler.stop()
    groups = eng.timing()                    # reset at the start of the timed region: timed steps only
    fps = S * T * timed_steps * world / (ms / 1e3)
    per_call = {k: v[0] / max(1, v[1]) for k, v in groups.items()}
    eng.timing(enable=False)
    return {"fps": fps, "ms": ms, "timed_steps": timed_steps, "step_ms": ms / timed_steps, "per_call": per_call,
            "launches": int(launches), "clocks": clocks, "last_stats": stats}


def roofline_of(m, info, S, T, traffic=None):
    per_call = m["per_call"]
    dom = max(per_call, key=per_call.get)
    peak, peak_src = hbm_peak()
    balg = alg_bytes_per_frame(info["proc_width"], info["proc_height"], T)
    bytes_launch = balg * S * T
    achieved = bytes_launch / (per_call[dom] / 1e3) / 1e9
    r = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
         "frac": round(achieved / peak, 4), "traffic": None, "kernel": dom,
         "kernel_ms_per_launch": round(per_call[dom], 4), "peak_source": peak_src,
         "alg_bytes_per_frame": round(balg), "alg_formula": "3*W*H + (16/T)*w*h + m*w*h, m=1/8 (bit-packed mask)",
         "groups_ms_per_step": {k: round(v, 4) for k, v in per_call.items()},
         "whole_step_frac": round(bytes_launch / (m["step_ms"] / 1e3) / 1e9 / peak, 4)}
    if traffic:
        r["traffic"], r["traffic_source"] = traffic
    return r


def ncu_traffic_for(args, info, name):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel: NOT measured by this run (a
    number taken under a profiler is never a bench value) -- read from the committed `ncu --set full` capture of this
    same command line, and labelled with its file; null when the workload differs from the captured one."""
    try:
        if (W, H, args.streams, args.frames) != (1920, 1080, 8, 16):
            return None
        path = os.path.join("profiles", f"r2_{name}_ncu_full.json")
        with open(os.path.join(ROOT, path)) as f:
            return int(json.load(f)["traffic_bytes_per_launch"]), path + " (ncu --set full of the same command)"
    except Exception:
        return None


DUMP_BG_VALUES = 1 << 20       # background values kept over all streams (8 MB)
DUMP_COMPONENT_ROWS = 1 << 19  # contour records kept (28 MB); the whole dump stays under 64 MB


def dump_outputs(path, eng, stats_dev, S, T, prefix=""):
    """What the last timed step computed, as float64 DIR/<prefix><name>.npy, so that two builds run with the same
    arguments (hence the same seeded inputs) can be compared file by file:
      <stats field>      [S, T]  the per-frame stats fm_process returns, one file per field (n_contours, movement, ...)
      components         [n, 7]  every contour record of the step: stream, frame, area_x2, x, y, w, h (the library's
                                 sorted order; a fixed seeded sample of rows past DUMP_COMPONENT_ROWS)
      background_sample  [S, k]  the float64 background after the step at k fixed seeded pixels (row-major index)"""
    import numpy as np
    from find_motion_b200.engine import STATS_DTYPE
    out = {}
    stats = stats_dev.cpu().numpy().view(STATS_DTYPE).reshape(S, T)
    for name in STATS_DTYPE.names:
        out[name] = stats[name].astype(np.float64)
    rows = [(s, t, a2, *box) for s in range(S) for t in range(T) for a2, box in eng.components(s, t)[1]]
    comps = np.array(rows, np.float64).reshape(-1, 7)
    if len(comps) > DUMP_COMPONENT_ROWS:
        comps = comps[np.sort(np.random.default_rng(1).choice(len(comps), DUMP_COMPONENT_ROWS, replace=False))]
    out["components"] = comps
    n = eng.w * eng.h
    idx = np.sort(np.random.default_rng(0).choice(n, min(n, max(1, DUMP_BG_VALUES // S)), replace=False))
    out["background_sample"] = np.stack(
        [eng.planes(s, T - 1, gray=False, blur=False, thresh=False)["bg"].ravel()[idx] for s in range(S)])
    assert sum(a.nbytes for a in out.values()) <= 64 << 20, "dump larger than 64 MB"
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, prefix + name + ".npy"), a)


def run_b200(args):

    import numpy as np
    import torch
    import torch.distributed as dist

    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine, PinnedBatch, launch_count
    from find_motion_b200.sharding import gather_stats, shard_streams

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert args.ring % args.frames == 0 and args.ring >= args.frames
    assert args.steps >= 1, "--steps: at least one timed step"

    kw = tuning(args.mode, args.blur_scale)
    S, T, R = args.streams, args.frames, args.ring
    my_streams = shard_streams(S * world, world, rank)          # stream s of the job lives on rank s mod G

    # CPU baseline first (rank 0, N=1 only), before the GPU is busy
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline(kw, os.cpu_count() or 1)
        except Exception as e:   # never let the baseline kill the measurement
            cpu = {"error": str(e)[:200]}

    # synthetic streams: seed = 1000*cfg + global stream id (SURVEY.md 8d), resident in HBM; the host copy lives in
    # pinned memory allocated next to this rank's GPU (fm_host_alloc)
    nd = min(S, args.distinct) if args.distinct else S
    ring_pin = None
    if nd == S:
        ring_pin = PinnedBatch((S, R, H, W, 3), local)
        for i, s in enumerate(my_streams):
            ring_pin.array[i] = synth.make_clip(W, H, R, synth.stream_seed(2, s), script=bench_script(R))
        ring_host = torch.from_numpy(ring_pin.array)
        ring_dev = ring_host.cuda()
    else:
        ring_host = None
        ring_dev = torch.empty((S, R, H, W, 3), dtype=torch.uint8, device="cuda")
        for d in range(nd):
            clip = torch.from_numpy(synth.make_clip(W, H, R, synth.stream_seed(2, my_streams[d]), script=bench_script(R))).cuda()
            for s in range(d, S, nd):
                ring_dev[s] = clip
    torch.cuda.synchronize()

    fe = {"auto": {}, "stencil": {}, "umma": dict(no_fused=True, umma=True), "umma-apron": dict(no_fused=True, umma=True, umma_apron=True),
          "mma-sync": dict(no_fused=True, no_umma=True), "warp-resize": dict(no_rows=True)}[args.front_end]
    eng = MotionEngine(W, H, n_streams=S, max_frames=T, device=local, **fe, **kw)
    info = dict(eng.info, w=eng.w, h=eng.h)
    m = measure(eng, ring_dev, args, torch, dist, world, S, T, launch_count, local)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, eng, m["last_stats"], S, T, "" if world == 1 else f"rank{rank}_")
    name = "fused" if info["front_end"] == 0 else ("wide" if args.mode == "full" else "default")
    roofline = roofline_of(m, info, S, T, ncu_traffic_for(args, info, name))

    # NCCL is used only here: the per-frame stats of one more (untimed) step are gathered so that rank 0 can report
    # motion flags for the whole box
    last = eng.process(ring_dev[:, :T], sync=True)
    allstats = gather_stats(last, S * world, dist if world > 1 else None)
    gathered = {"streams": int(allstats.shape[0]), "frames": int(allstats.size),
                "motion_frames": int((allstats["movement"] != 0).sum()), "via": "nccl all_gather" if world > 1 else "local"}

    # end to end through the host-buffer entry points: pinned host frames -> H2D -> kernels -> stats D2H every step,
    # pipelined on two slots (fm_submit_host / fm_wait) exactly as the job driver does it
    eng.reset()
    e2e = None
    if not args.no_e2e and ring_host is not None:
        host_batch = [ring_pin.array[:, a:a + T] for a in range(0, R, T)]
        nb = len(host_batch)
        for i in range(2):
            eng.process_host(host_batch[i % nb])
        torch.cuda.synchronize()
        # ceiling: the same bytes through cudaMemcpyAsync alone, all ranks at once
        stage = torch.empty((S, T, H, W, 3), dtype=torch.uint8, device="cuda")
        src = [[torch.from_numpy(b[s]) for s in range(S)] for b in host_batch]      # [T, H, W, 3] each, contiguous, pinned
        for s in range(S):
            stage[s].copy_(src[0][s], non_blocking=True)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(8):
            for s in range(S):
                stage[s].copy_(src[i % nb][s], non_blocking=True)
        torch.cuda.synchronize()
        copy_s = time.perf_counter() - t0
        bytes_step = S * T * W * H * 3
        if world > 1:
            dist.barrier()
        t0 = time.perf_counter()
        for i in range(args.e2e_steps):
            eng.submit_host(i & 1, host_batch[i % nb])
            if i:
                eng.wait_host((i - 1) & 1)
        eng.wait_host((args.e2e_steps - 1) & 1)
        e2e_s = time.perf_counter() - t0
        mine = torch.tensor([e2e_s, copy_s], device="cuda", dtype=torch.float64)
        allr = [torch.empty_like(mine) for _ in range(world)]
        if world > 1:
            dist.all_gather(allr, mine)
        else:
            allr = [mine]
        e2e_all = [float(t[0]) for t in allr]
        copy_all = [float(t[1]) for t in allr]
        e2e_s = max(e2e_all)
        e2e = {"value": round(S * T * args.e2e_steps * world / e2e_s, 1), "unit": "frames/s",
               "h2d_bytes_per_step": bytes_step, "d2h_bytes_per_step": S * T * 32, "steps": args.e2e_steps,
               "seconds": round(e2e_s, 3),
               "h2d_gbs_per_rank": [round(bytes_step * args.e2e_steps / t / 1e9, 1) for t in e2e_all],
               "h2d_copy_only_gbs_per_rank": [round(bytes_step * 8 / t / 1e9, 1) for t in copy_all],
               "pinned_numa_node": ring_pin.numa_node,
               "api": "fm_submit_host / fm_wait (MotionEngine.submit_host / wait_host), two slots, pinned host frames "
                      "allocated with fm_host_alloc; h2d_copy_only = the same bytes through cudaMemcpyAsync alone on "
                      "all ranks at once (the platform's ceiling for this path)"}
        del stage

    extras = {}
    if rank == 0 and world == 1 and not args.no_extras:
        extras = secondary_regimes(args, ring_dev, torch, dist, launch_count, local)
    eng.close()
    line = None
    if rank == 0:
        clocks = dict(m["clocks"])
        line = {
            "metric": METRIC if (W, H) == (1920, 1080) else f"{W}x{H} frames/sec (whole box)", "value": round(m["fps"], 1),
            "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(m["step_ms"], 4), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8+f64", "data": "synthetic", "config": workload_config(args, kw, info),
            "timed_steps": m["timed_steps"], "timed_region_s": round(m["ms"] / 1e3, 3),
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": m["launches"], "clocks": clocks,
            "gathered_stats": gathered,
        }
        if extras:
            line["other_regimes"] = extras
    if world > 1:
        dist.destroy_process_group()
    if ring_pin is not None:
        del ring_host
        ring_pin.free()
    return line


def secondary_regimes(args, ring_dev, torch, dist, launch_count, local):
    """Same streams in the other two regimes SURVEY.md 8(d) asks for, each with its own roofline (the reference's own
    blur scale, k=97 at 1080p, runs on the tensor cores; the reference's CLI default, box 100, is bound by reading
    3*W*H)."""
    from find_motion_b200.engine import MotionEngine
    out = {}
    S, T = args.streams, args.frames
    for name, mode, bs, tag in (("full_k97_reference_blur_scale", "full", 20, "wide"), ("default_box100", "default", 20, "default")):
        if mode == args.mode and (args.blur_scale or (384 if mode == "full" else 20)) == bs:
            continue
        kw = tuning(mode, bs)
        try:
            with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as eng:
                info = dict(eng.info, w=eng.w, h=eng.h)
                m = measure(eng, ring_dev, args, torch, dist, 1, S, T, launch_count, local)
                out[name] = {"value": round(m["fps"], 1), "unit": "frames/s", "proc": f"{eng.w}x{eng.h}",
                             "gaussian": eng.info["gaussian"], "timed_steps": m["timed_steps"],
                             "ms_per_step": round(m["step_ms"], 4),
                             "roofline": roofline_of(m, info, S, T, ncu_traffic_for(args, info, tag)),
                             "clocks": m["clocks"]}
        except Exception as e:
            out[name] = {"error": str(e)[:200]}
    return out


if __name__ == "__main__":
    main()
