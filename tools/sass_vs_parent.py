"""Per-function SASS comparison of two builds of libfmgpu.so (cuobjdump -sass), e.g. a parent commit's against a change's.

    python tools/sass_vs_parent.py PARENT.so CHANGE.so [--rename REGEX REPLACEMENT ...]

Instructions are compared without their addresses and encodings, with branch labels renumbered per function (label
numbers run across a module, so a kernel added in the same file shifts them).  --rename rewrites the change's demangled
names (re.sub) before they are matched with the parent's, so that a pre-existing instantiation whose kernel gained a
template parameter with a default value is compared with the instantiation it became.  Prints one line per function:
same / DIFFERENT / REMOVED / NEW with the instruction counts, and exits 1 if any pre-existing function differs or is gone.
"""
import argparse
import re
import subprocess
import sys

CUOBJDUMP = "/usr/local/cuda/bin/cuobjdump"
CUFILT = "/usr/local/cuda/bin/cu++filt"


def functions(lib):
    out = subprocess.run([CUOBJDUMP, "-sass", lib], check=True, capture_output=True, text=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = body
            name, body = m.group(1), []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;?\s*/\*", line)
        if name and m:
            body.append(m.group(1))
        elif name and re.match(r"\s*\.L_x_\d+:", line):
            body.append(line.strip())
    if name:
        funcs[name] = body
    return funcs


def normalise(body):
    labels = {}

    def lab(m):
        return labels.setdefault(m.group(0), ".L%d" % len(labels))
    return [re.sub(r"\.L_x_\d+", lab, ins) for ins in body]


def demangle(names):
    out = subprocess.run([CUFILT], input="\n".join(names), check=True, capture_output=True, text=True).stdout
    return dict(zip(names, out.splitlines()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("parent")
    ap.add_argument("change")
    ap.add_argument("--rename", nargs=2, action="append", default=[], metavar=("REGEX", "REPLACEMENT"))
    a = ap.parse_args()
    old, new = functions(a.parent), functions(a.change)
    dold, dnew = demangle(list(old)), demangle(list(new))

    def key(d):
        for pat, repl in a.rename:
            d = re.sub(pat, repl, d)
        return d
    by_key = {key(dnew[n]): n for n in new}
    bad, matched = 0, set()
    for n in sorted(old, key=lambda n: dold[n]):
        m = by_key.get(dold[n])
        if m is None:
            print("REMOVED   %6d        %s" % (len(old[n]), dold[n]))
            bad += 1
            continue
        matched.add(m)
        same = normalise(old[n]) == normalise(new[m])
        bad += not same
        print("%-9s %6d %6d %s%s" % ("same" if same else "DIFFERENT", len(old[n]), len(new[m]), dold[n],
                                     "" if dnew[m] == dold[n] else "  ->  " + dnew[m]))
    for m in sorted(set(new) - matched, key=lambda n: dnew[n]):
        print("NEW              %6d %s" % (len(new[m]), dnew[m]))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
