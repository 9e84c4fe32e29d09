"""Compare the SASS of every kernel of two builds of libsfm_b200.so (instruction text without addresses or encodings).

usage: python tools/sass_check.py PARENT.so NEW.so [ptxas -v log of NEW] > profiles/<name>_sass_check.txt
A kernel of the parent is "identical" when its instruction stream is; kernels only in NEW are listed as "new", with
their registers, stack and spills from the ptxas log when one is given.  Exit status 1 when a parent kernel differs or
is missing."""
from __future__ import annotations

import re
import subprocess
import sys

CUDA_BIN = "/usr/local/cuda/bin"


def kernels(so: str) -> dict:
    text = subprocess.run([f"{CUDA_BIN}/cuobjdump", "-sass", so], check=True, capture_output=True, text=True).stdout
    out, name = {}, None
    for line in text.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4,}\*/\s+(.*?);", line)
        if name and m:
            out[name].append(m.group(1).strip())
    return out


def demangle(names):
    res = subprocess.run([f"{CUDA_BIN}/cu++filt"], input="\n".join(names), check=True, capture_output=True, text=True)
    return dict(zip(names, res.stdout.splitlines()))


def ptxas_props(log: str) -> dict:
    props, cur = {}, None
    for line in open(log):
        m = re.search(r"Function properties for (\S+)", line)
        if m:
            cur = m.group(1)
            continue
        if cur and ("stack frame" in line or "Used" in line):
            props[cur] = (props.get(cur, "") + "; " + line.split(":", 1)[-1].strip()).lstrip("; ")
    return props


def main(argv):
    parent, new = kernels(argv[1]), kernels(argv[2])
    props = ptxas_props(argv[3]) if len(argv) > 3 else {}
    dm = demangle(sorted(set(parent) | set(new)))
    same = 0
    for k in sorted(parent, key=lambda k: dm[k]):
        if k not in new:
            print(f"missing  {len(parent[k]):6d} instr  {dm[k]}")
        elif parent[k] == new[k]:
            same += 1
            print(f"identical{len(parent[k]):6d} instr  {dm[k]}")
        else:
            print(f"CHANGED  {len(parent[k]):6d} -> {len(new[k])} instr  {dm[k]}")
    added = sorted(set(new) - set(parent), key=lambda k: dm[k])
    for k in added:
        print(f"new      {len(new[k]):6d} instr  {dm[k]}")
    print(f"\nparent kernels: {len(parent)}, identical instruction streams: {same}")
    if props and added:
        print("\nptxas -v of the new kernels:")
        for k in added:
            print(f"  {dm[k]}: {props.get(k, 'not in the log')}")
    return 0 if same == len(parent) else 1


if __name__ == "__main__":
    sys.exit(main(sys.argv))
