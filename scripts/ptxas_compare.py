"""Compare two `-Xptxas -v` reports kernel by kernel: registers, barriers, shared memory, stack frame and spills.

    nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xptxas=-v \\
         -I include -I speaker_embedding_ge2e_loss_b200/csrc -c speaker_embedding_ge2e_loss_b200/csrc/ge2e_simt.cu \\
         -o /tmp/x.o 2> REPORT            # once on the parent tree, once on this one
    python scripts/ptxas_compare.py PARENT_REPORT NEW_REPORT

Kernels are matched by demangled name (c++filt).  ``--rename OLD=NEW`` (regular expression and replacement, applied to
the new report's names, repeatable) maps a kernel whose template arguments grew; the default maps the single-kernel
step's PART argument 0 back to the four-argument name it had before it was split into halves.  Prints every parent
kernel whose line changed or is missing, a count of the unchanged ones, and every new kernel with its line.
"""
from __future__ import annotations

import argparse
import re
import subprocess


def parse(path):
    """{demangled kernel name: 'Used ... | stack / spills'} of one report."""
    out, cur = {}, None
    with open(path) as f:
        for line in f:
            m = re.search(r"Compiling entry function '(\S+)'", line)
            if m:
                cur = m.group(1)
                out[cur] = []
            elif cur and ("Used" in line or "spill" in line or "stack frame" in line):
                out[cur].append(re.sub(r"^.*?: ", "", line.strip()))
    names = list(out)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True,
                         check=True).stdout.split("\n")
    return {d: " | ".join(out[n]) for n, d in zip(names, dem)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("parent")
    ap.add_argument("new")
    ap.add_argument("--rename", action="append",
                    default=[r"small_step_kernel<(.*), 0>\(=small_step_kernel<\1>("])
    args = ap.parse_args()
    old, new = parse(args.parent), parse(args.new)
    rules = [r.split("=", 1) for r in args.rename]

    def norm(name):
        for pat, rep in rules:
            name = re.sub(pat, rep, name)
        return name

    by_old_name = {}
    for k, v in new.items():
        by_old_name.setdefault(norm(k), v)
    same = 0
    for k, v in old.items():
        if k not in by_old_name:
            print("MISSING", k)
        elif by_old_name[k] != v:
            print("CHANGED", k, "\n  parent:", v, "\n  new   :", by_old_name[k])
        else:
            same += 1
    print(f"unchanged {same} of {len(old)}")
    added = [k for k in new if norm(k) not in old]
    print(f"new kernels {len(added)}")
    for k in added:
        print(k, "::", new[k])


if __name__ == "__main__":
    main()
