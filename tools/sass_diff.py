#!/usr/bin/env python
"""Compare the kernels of two `cuobjdump -sass` dumps instruction by instruction.

    python tools/sass_diff.py old.sass new.sass [--map OLD_SUFFIX=NEW_SUFFIX] [-v]

Addresses, encodings and comments are ignored; a kernel is matched by its mangled name, after the optional
--map replacement of a name's suffix (e.g. a template parameter and a kernel parameter added).  Prints `same` / `DIFF` per kernel of the
first dump and exits non-zero if any differs or is missing.
"""
import argparse
import difflib
import re
import sys


def kernels(path):
    out, cur = {}, None
    for line in open(path):
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        if cur:
            ins = re.sub(r"/\*[^*]*\*/", "", line).strip()
            if ins and not ins.startswith("."):
                out[cur].append(re.sub(r"\s+", " ", ins))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--map", action="append", default=[])
    ap.add_argument("-v", action="store_true")
    args = ap.parse_args()
    a, b = kernels(args.old), kernels(args.new)
    bad = 0
    for name, ins in a.items():
        new = name
        for m in args.map:
            old_s, new_s = m.split("=", 1)
            if new.endswith(old_s):
                new = new[:len(new) - len(old_s)] + new_s
        if new not in b:
            print("MISSING", name)
            bad += 1
            continue
        same = ins == b[new]
        bad += not same
        print("same" if same else "DIFF", len(ins), name)
        if not same and args.v:
            print("\n".join(list(difflib.unified_diff(ins, b[new], lineterm=""))[:40]))
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
