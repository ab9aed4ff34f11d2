#!/usr/bin/env python
"""Registers / stack / spills / shared memory of every kernel of libpcindex (nvcc -Xptxas -v, no GPU needed).
    python scripts/ptxas_report.py [filter-substring]
    python scripts/ptxas_report.py --sass-diff REV
The second form compiles pc_index.cu of this tree and of git revision REV with the build's NVCC flags (__graft_entry__.py),
disassembles both (cuobjdump -sass) and compares every function's instruction list, addresses and comments stripped."""
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def ptxas_report(flt):
    out = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xptxas", "-v", "-c", "-o", "/tmp/pc_ptxas.o",
                          os.path.join(ROOT, "pointcloudtraj_b200", "csrc", "pc_index.cu")], capture_output=True, text=True)
    txt = subprocess.run(["c++filt"], input=out.stderr + out.stdout, capture_output=True, text=True).stdout
    name, st = None, ("0", "0")
    for l in txt.split("\n"):
        m = re.search(r"Compiling entry function '(.*)' for", l)
        if m:
            name = m.group(1)[:64]
        m = re.search(r"(\d+) bytes stack frame, (\d+) bytes spill stores", l)
        if m:
            st = m.group(1), m.group(2)
        m = re.search(r"Used (\d+) registers", l)
        if m and name and flt in name:
            sm = re.search(r"(\d+) bytes smem", l)
            print(f"{name:66s} regs={m.group(1):>3s} stack={st[0]:>4s} spill={st[1]:>3s} smem={sm.group(1) if sm else 0}")


def sass_functions(tree, tmp):
    """{function: [instruction, ...]} of pc_index.cu under `tree`"""
    sys.path.insert(0, ROOT)
    from __graft_entry__ import NVCC_FLAGS
    obj = os.path.join(tmp, os.path.basename(tree) + ".o")
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    subprocess.run(["nvcc"] + flags + ["-c", "-o", obj, os.path.join(tree, "pointcloudtraj_b200", "csrc", "pc_index.cu")],
                   check=True, capture_output=True)
    sass = subprocess.run(["cuobjdump", "-sass", obj], check=True, capture_output=True, text=True).stdout
    funcs, name = {}, None
    for l in sass.split("\n"):
        m = re.match(r"\s*Function : (\S+)", l)
        if m:
            name = m.group(1)
            funcs[name] = []
            continue
        m = re.search(r"/\*[0-9a-f]{4,}\*/\s+(.*?);", l)
        if name is not None and m:
            funcs[name].append(re.sub(r"\s+", " ", m.group(1)))
    return funcs


def sass_diff(rev):
    with tempfile.TemporaryDirectory() as tmp:
        old = os.path.join(tmp, "parent")
        os.makedirs(old)
        archive = subprocess.run(["git", "-C", ROOT, "archive", rev, "pointcloudtraj_b200/csrc", "include"], check=True, capture_output=True).stdout
        subprocess.run(["tar", "-x", "-C", old], input=archive, check=True)
        a, b = sass_functions(old, tmp), sass_functions(ROOT, tmp)
    demangled = dict(zip(sorted(set(a) | set(b)), subprocess.run(["c++filt"], input="\n".join(sorted(set(a) | set(b))),
                                                                  capture_output=True, text=True).stdout.split("\n")))
    same = 0
    for f in sorted(set(a) | set(b), key=lambda f: demangled[f]):
        if f not in a or f not in b:
            what = "NEW    " if f not in a else "REMOVED"
        elif a[f] == b[f]:
            what = "same   "
            same += 1
        else:
            what = "DIFF   "
        print(f"{what} {len(a.get(f, [])):6d} {len(b.get(f, [])):6d}  {demangled[f][:110]}")
    print(f"# {same} of {len(set(a) | set(b))} functions have identical SASS ({rev}: {len(a)} functions, this tree: {len(b)})")


if __name__ == "__main__":
    if len(sys.argv) > 2 and sys.argv[1] == "--sass-diff":
        sass_diff(sys.argv[2])
    else:
        ptxas_report(sys.argv[1] if len(sys.argv) > 1 else "")
