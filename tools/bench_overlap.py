"""How far the fused front end (K1, k_fused) of call i+1 runs under the contour stage of call i.

K1 is launched as a programmatic dependent of k_decide, the last kernel of the previous call's contour stage
(csrc/k_fused.cu, fused_exit), so on an idle GPU it starts before k_decide of the previous call ends.  This tool runs
bench.py's headline configuration (8 streams x 16 frames of 1920x1080 per call, full resolution, k = 5, the same seeded
HBM ring of 32 frames per stream) and writes:
  * a torch.profiler trace of --steps chained calls (sync=False, back to back) per timing mode, to
    <--trace-dir>/overlap_timing_{off,on}.pt.trace.json;
  * one JSON line, printed and appended to --out, with, per timing mode (fm_timing_enable off / on) and per pair of
    consecutive calls, head_start_us = end of k_decide(i) - start of k_fused(i+1) from the trace (> 0: K1 of call i+1
    ran that long before k_decide of call i finished), the gap between k_ccl_frame_smem(i)'s end and K1(i+1)'s start,
    and step_ms from CUDA events around --timed calls without the profiler (both modes alternated, --rounds times);
  * the GPU's name and power limit, read in the same run.

    python tools/bench_overlap.py [--out profiles/bench_overlap.jsonl] [--trace-dir profiles]

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

from bench_upscale import gpu_facts  # noqa: E402


def kernel_spans(trace_path):
    """{short name: [(start_us, end_us), ...] in start order} of the kernels in a chrome trace written by torch.profiler."""
    with open(trace_path) as f:
        ev = json.load(f)["traceEvents"]
    out = {}
    for e in ev:
        if e.get("cat") != "kernel":
            continue
        name = e["name"]
        for short in ("k_fused<", "k_decide(", "k_ccl_frame_smem(", "k_ccl_frame("):
            if short in name:
                out.setdefault(short.rstrip("<("), []).append((float(e["ts"]), float(e["ts"]) + float(e["dur"])))
    return {k: sorted(v) for k, v in out.items()}


def head_starts(spans):
    """Per pair of consecutive calls: how long K1(i+1) ran before k_decide(i) ended, and the gap labelling(i) -> K1(i+1)."""
    k1, dec, ccl = spans.get("k_fused", []), spans.get("k_decide", []), spans.get("k_ccl_frame_smem", [])
    rows = []
    for i in range(min(len(dec), len(ccl), len(k1) - 1)):       # the trace starts on an idle device: call i = i-th
        s = k1[i + 1][0]
        rows.append({"head_start_us": round(dec[i][1] - s, 2), "ccl_end_to_k1_start_us": round(s - ccl[i][1], 2)})
    return rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench_overlap.jsonl"))
    ap.add_argument("--trace-dir", default=os.path.join(ROOT, "profiles"))
    ap.add_argument("--steps", type=int, default=6, help="chained calls in each trace (steps - 1 pairs)")
    ap.add_argument("--timed", type=int, default=200, help="calls per timed window")
    ap.add_argument("--rounds", type=int, default=3)
    args = ap.parse_args()

    import torch
    from torch.profiler import ProfilerActivity, profile

    import bench
    from find_motion_b200 import synth
    from find_motion_b200.engine import MotionEngine

    assert torch.cuda.is_available(), "bench_overlap.py needs a CUDA device (no CPU fallback)"
    W, H, S, T, R = 1920, 1080, 8, 16, 32
    kw = bench.tuning("full", None)
    ring = torch.from_numpy(
        __import__("numpy").stack([synth.make_clip(W, H, R, synth.stream_seed(2, s), script=bench.bench_script(R))
                                   for s in range(S)])).cuda()
    eng = MotionEngine(W, H, n_streams=S, max_frames=T, **kw)
    assert eng.info["front_end"] == 0, "the headline configuration runs the fused front end"

    def step(i):
        a = (i % (R // T)) * T
        return eng.process(ring[:, a:a + T], sync=False)

    for i in range(8):
        step(i)
    torch.cuda.synchronize()

    modes = {}
    os.makedirs(args.trace_dir, exist_ok=True)
    for timing in (False, True):
        eng.timing(enable=timing, reset=True)
        for i in range(3):
            step(i)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(args.steps):
                step(i)
            torch.cuda.synchronize()
        path = os.path.join(args.trace_dir, f"overlap_timing_{'on' if timing else 'off'}.pt.trace.json")
        prof.export_chrome_trace(path)
        modes["timing_on" if timing else "timing_off"] = {"pairs": head_starts(kernel_spans(path)), "step_ms": []}
        eng.timing(enable=False)

    for _ in range(args.rounds):
        for timing in (False, True):
            eng.timing(enable=timing, reset=True)
            for i in range(4):
                step(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.timed):
                step(i)
            e1.record()
            torch.cuda.synchronize()
            modes["timing_on" if timing else "timing_off"]["step_ms"].append(round(e0.elapsed_time(e1) / args.timed, 4))
            eng.timing(enable=False)
    eng.check()
    for m in modes.values():
        m["step_ms_median"] = statistics.median(m["step_ms"])
        hs = [p["head_start_us"] for p in m["pairs"]]
        m["head_start_us_median"] = statistics.median(hs) if hs else None
    line = {"tool": "bench_overlap", **gpu_facts(0),
            "config": f"{S} streams x {T} frames of {W}x{H} per call, full resolution k=5 (bench.py defaults)",
            **modes}
    print(json.dumps(line), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "a") as f:
        f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
