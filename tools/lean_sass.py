"""SASS of the lean step-kernel instantiations (SpecLean<LAW>, step_device.cuh) of an object or library.

The lean kernels run cfg 2 / 3 / 4; a change that adds a general-path feature should leave them exactly
as they were.  `python tools/lean_sass.py OBJ` prints one line per lean kernel: the mangled name and the
SHA-256 of its SASS text (cuobjdump -sass, one function at a time).  `--diff A B` compares two builds.
"""
import argparse
import hashlib
import re
import subprocess
import sys


def lean_sass(path):
    out = subprocess.run(["cuobjdump", "-sass", path], check=True, capture_output=True, text=True).stdout
    funcs, name, body = {}, None, []
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            if name:
                funcs[name] = "\n".join(body)
            name, body = m.group(1), []
        elif name:
            body.append(line)
    if name:
        funcs[name] = "\n".join(body)
    # SpecLean<LAW> mangles as 8SpecLeanILi<LAW>EE
    return {k: hashlib.sha256(v.encode()).hexdigest() for k, v in funcs.items() if "SpecLean" in k}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("paths", nargs="+")
    ap.add_argument("--diff", action="store_true")
    a = ap.parse_args()
    if not a.diff:
        for k, v in sorted(lean_sass(a.paths[0]).items()):
            print(v, k)
        return 0
    x, y = lean_sass(a.paths[0]), lean_sass(a.paths[1])
    bad = sorted(k for k in set(x) | set(y) if x.get(k) != y.get(k))
    print(f"{len(x)} / {len(y)} lean kernels; {len(bad)} differ")
    for k in bad:
        print("  differs:", k)
    return 1 if bad or not x else 0


if __name__ == "__main__":
    sys.exit(main())
