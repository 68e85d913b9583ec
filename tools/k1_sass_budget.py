"""Static instruction budget of K1 (k_fused), per phase, from the sm_100a SASS.  Needs nvcc, no GPU.

Compiles csrc/k_fused.cu with build.py's flags plus `-Xptxas -v` into a cubin, disassembles the benchmarked
instantiation (KEEP off, SAFE on: `k_fused<false, true>`) with nvdisasm's inline line information, and attributes each
instruction to the line of the kernel body it comes from (for inlined code: the outermost call site).  The phases are
the marked sections of the frame loop in the source, so the table follows the code when lines move:

    loop top    `for (int t = 0; t < Ts; t++)` .. the `// ---- staged BGR -> gray` header
    gray        .. `if (border)`
    border      .. the `// ---- horizontal pass` header
    horizontal  .. the `// ---- vertical pass` header
    vertical    .. the `// ---- two bytes of the bit plane` header, itemised per fused_rows call site (variant)
    tail        .. the end of the frame loop, itemised per line (the per-frame rawrange path is taken only for T > 32)

Counts are static (every instruction of the section once, predicated or not): a per-thread budget of one frame for
the straight-line sections, and the sum over the variants for `vertical`, which is why each call site is listed too.

usage: python tools/k1_sass_budget.py [--keep-cubin DIR] [-D NAME[=VALUE] ...]
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from find_motion_b200 import build as B  # noqa: E402

SRC = os.path.join(B.CSRC, "k_fused.cu")
KERNEL = "_Z7k_fusedILb0ELb1EEv14CUtensorMap_st11FusedParams"
MARKERS = [  # (phase that starts at the first line containing the text, text)
    ("loop top", "for (int t = 0; t < Ts; t++)"),
    ("gray", "// ---- staged BGR -> gray"),
    ("border", "if (border)"),
    ("horizontal", "// ---- horizontal pass"),
    ("vertical", "// ---- vertical pass"),
    ("tail", "// ---- two bytes of the bit plane"),
]


def source_phases(lines):
    """line number -> phase, for the kernel body of k_fused."""
    start = next(i for i, l in enumerate(lines) if re.match(r"__global__ void .*k_fused\(", l)) + 1
    bounds = []
    i = start
    for name, text in MARKERS:
        i = next(j for j in range(i, len(lines)) if text in lines[j])
        bounds.append((i + 1, name))
    loop = bounds[0][0] - 1
    indent = len(lines[loop]) - len(lines[loop].lstrip())
    end = next(j for j in range(loop + 1, len(lines)) if lines[j].rstrip() == " " * indent + "}") + 1
    phase = {}
    for n in range(start + 1, len(lines) + 1):
        if n > end:
            phase[n] = "after the loop"
        elif n < bounds[0][0]:
            phase[n] = "before the loop"
        else:
            phase[n] = [name for b, name in bounds if b <= n][-1]
    return phase


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--keep-cubin", help="directory to keep the cubin and the annotated SASS in")
    ap.add_argument("-D", action="append", default=[], help="extra preprocessor definition, e.g. -D FM_K1_PROF")
    a = ap.parse_args()
    out = a.keep_cubin or tempfile.mkdtemp(prefix="k1_sass_")
    os.makedirs(out, exist_ok=True)
    cubin = os.path.join(out, "k_fused.cubin")
    flags = [f for f in B.NVCC_FLAGS if f not in ("-shared", "-Xcompiler", "-fPIC", "-O2")]
    cmd = [B.find_nvcc()] + flags + ["-cubin", "-Xptxas", "-v", "-I", B.CSRC] + ["-D" + d for d in a.D] + \
          ["-o", cubin, SRC]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode:
        raise SystemExit(r.stdout + r.stderr)
    ptxas = r.stderr.splitlines()
    nvdisasm = os.path.join(os.path.dirname(B.find_nvcc()), "nvdisasm")
    sass = subprocess.run([nvdisasm, "-gi", cubin], check=True, capture_output=True, text=True).stdout
    with open(os.path.join(out, "k_fused.sass"), "w") as f:
        f.write(sass)

    for i, l in enumerate(ptxas):
        if "Compiling entry function '%s'" % KERNEL in l:
            spill = ptxas[i + 2].strip()
            regs = ptxas[i + 3].split(":", 1)[1].strip()
            break
    else:
        raise SystemExit("ptxas output has no %s" % KERNEL)

    with open(SRC) as f:
        lines = f.read().splitlines()
    phase = source_phases(lines)
    body = sass.split(".text.%s:" % KERNEL, 1)[1].split("\n.text.", 1)[0]
    loc = None
    pending = None
    counts, sites = {}, {}
    for l in body.splitlines():
        m = re.match(r'\s*//## File "(.*)", line (\d+)(.*)', l)
        if m:
            if os.path.basename(m.group(1)) == "k_fused.cu" and "inlined at" not in m.group(3):
                pending = int(m.group(2))        # the last annotation of a group is the outermost location
            continue
        if not re.match(r"\s+/\*[0-9a-f]{4}\*/", l):
            continue
        if pending is not None:
            loc, pending = pending, None
        ph = phase.get(loc, "before the loop")
        counts[ph] = counts.get(ph, 0) + 1
        if ph in ("vertical", "tail"):
            sites[loc] = sites.get(loc, 0) + 1

    print("k_fused<false, true> (KEEP off, SAFE on): %s; %s" % (regs, spill))
    order = ["before the loop"] + [n for n, _ in MARKERS] + ["after the loop"]
    print("%-16s %6s" % ("phase", "SASS"))
    for n in order:
        print("%-16s %6d" % (n, counts.get(n, 0)))
        if n in ("vertical", "tail"):
            for ln in sorted(l for l in sites if phase[l] == n):
                print("    line %4d %6d   %s" % (ln, sites[ln], lines[ln - 1].strip()[:90]))
    print("%-16s %6d" % ("total", sum(counts.values())))


if __name__ == "__main__":
    main()
