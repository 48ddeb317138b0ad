#!/usr/bin/env python3
"""Compare the SASS of each kernel in two `cuobjdump -sass` listings, parameter offsets aside.

usage: sass_compare.py <before.sass> <after.sass>

A kernel of the first listing is matched with the kernel of the second that has the same name and template arguments
once a trailing `bool` template argument of value false (`Lb0E`) is dropped: the whole-image instantiation of a kernel
that gained a compile-time crop switch.  Constant-bank operands `c[0x0][...]` (kernel parameters) are compared as one
placeholder.  Prints one line per kernel, SAME or DIFF, and exits 1 when any differs or is missing."""
import re
import sys


def kernels(path):
    out, cur = {}, None
    for line in open(path):
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            out[cur] = []
            continue
        m = re.match(r"\s+/\*[0-9a-f]{4}\*/\s+(.*?);", line)
        if m and cur:
            out[cur].append(re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", m.group(1)))
    return out


def key(name):
    m = re.match(r"_ZN4kpeg(\d+)(\w+?)I((?:L[ib]\d+E)+)E", name)
    if not m:
        return name
    args = re.findall(r"L[ib]\d+E", m.group(3))
    if args and args[-1] == "Lb0E":
        args = args[:-1]
    return m.group(2) + "<" + ",".join(a[2:-1] for a in args) + ">"


def main():
    a, b = kernels(sys.argv[1]), kernels(sys.argv[2])
    bk = {key(k): v for k, v in b.items()}
    bad = 0
    for k, v in a.items():
        w = bk.get(key(k))
        if w is None:
            print(f"MISSING {key(k)}")
            bad += 1
            continue
        same = v == w
        bad += not same
        print(f"{'SAME' if same else 'DIFF'} {key(k)}: {len(v)} -> {len(w)} instructions")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
