"""Development aid: per-phase cycle counts of K1 (k_fused) on the benchmark's headline workload.

Builds the library with -DFM_K1_PROF into a temporary directory (the tree and its libfmgpu.so are not touched), runs
8 streams x 16 frames of 1080p at k = 5 (bench.py's headline regime) and prints, per phase of the frame loop, the cycles
thread 0 of a CTA spends per frame, averaged over all CTAs.  The instrumentation changes register allocation, so read
the phases against each other, not the total against an uninstrumented run.  Needs a GPU.
"""
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from find_motion_b200 import _lib, build as B, synth  # noqa: E402
from find_motion_b200.engine import MotionEngine  # noqa: E402

W, H, S, T = 1920, 1080, 8, 16
lib_path = os.path.join(tempfile.mkdtemp(prefix="k1_prof_"), "libfmgpu.so")
subprocess.run([B.find_nvcc()] + B.NVCC_FLAGS + ["-DFM_K1_PROF", "-o", lib_path] + B.sources(), check=True, cwd=B.CSRC)
_lib.LIB_PATH = lib_path
lib = _lib.load()
kw = dict(fps=30, box_size=W, blur_scale=384, min_box_scale=50, threshold=12, avg=0.1, min_time=0.5, cache_time=1.0,
          mask_areas=synth.CFG2_MASKS)
clip = torch.from_numpy(synth.make_clip(W, H, T, seed=1)).cuda()
frames = clip[None].expand(S, T, H, W, 3).contiguous()
with MotionEngine(W, H, n_streams=S, max_frames=T, **kw) as eng:
    print("gaussian k", eng.info["gaussian"], file=sys.stderr)
    for i in range(3):
        eng.process(frames, sync=False)
    torch.cuda.synchronize()
    lib.fm_k1_prof_dump()
    for i in range(20):
        eng.process(frames, sync=False)
    torch.cuda.synchronize()
    lib.fm_k1_prof_dump()
