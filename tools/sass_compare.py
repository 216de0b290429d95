#!/usr/bin/env python
"""Compare the SASS of two builds of libfrg.so kernel by kernel: the opcode sequence (mnemonics with their
modifiers, operands dropped) of every kernel of the OLD library must be the same in the NEW one.  Runs without a GPU.
    python tools/sass_compare.py OLD/libfrg.so NEW/libfrg.so

Kernels are matched by demangled name.  The mangled names leave out defaulted trailing template flags, so a flag
appended with a default (tc_scan_kernel's GROUPED) renames existing instantiations: tc_scan_kernel's argument list
is padded with `false` to all five flags on both sides first.
Exit status 1 when a kernel of OLD is missing from NEW or its opcodes differ.
"""
import re
import subprocess
import sys


def kernels(lib):
    sass = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    per, cur = {}, None
    for line in sass.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            per[cur] = []
            continue
        m = re.search(r"/\*[0-9a-f]{4}\*/\s+((?:@!?U?P\w+\s+)?[A-Z0-9_.]+)", line)
        if cur and m:
            per[cur].append(m.group(1))
    names = subprocess.run(["c++filt"], input="\n".join(per), capture_output=True, text=True).stdout.splitlines()
    out = {}
    for (mangled, ops), name in zip(per.items(), names):
        m = re.match(r"^(void frg::tc_scan_kernel<)([^>]*)(>.*)$", name)
        if m:            # <MODE, MASKED, PAIR[, I8[, GROUPED]]>: defaulted flags spelled out
            args = [a.strip() for a in m.group(2).split(",")]
            name = m.group(1) + ", ".join(args + ["false"] * (5 - len(args))) + m.group(3)
        out[name] = ops
    return out


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    bad = 0
    for name, ops in old.items():
        if name not in new:
            print("MISSING  %s" % name)
            bad += 1
        elif new[name] != ops:
            print("CHANGED  %s (%d -> %d instructions)" % (name, len(ops), len(new[name])))
            bad += 1
        else:
            print("same     %s (%d instructions)" % (name, len(ops)))
    for name in new:
        if name not in old:
            print("NEW      %s (%d instructions)" % (name, len(new[name])))
    print("# %d kernels in the old library, %d changed or missing; %d in the new one" % (len(old), bad, len(new)))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
