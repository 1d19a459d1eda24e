#!/usr/bin/env python
"""Compare the SASS of every kernel in two builds of libmpb200.so, function by function (no GPU needed).

Addresses and instruction encodings are dropped and anonymous-namespace hashes normalised, so two builds of the same
source compare equal.  --pair OLD NEW additionally compares one renamed kernel (substrings of the mangled names).

  python scripts/sass_diff.py OLD.so NEW.so [--pair gmt_kernelENS0_7GmtArgsE GmtTableEdge]
"""
import argparse
import collections
import re
import subprocess


def functions(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    fs, cur = collections.OrderedDict(), None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = re.sub(r"_GLOBAL__N__\w+?_cu_[0-9a-f]+", "ANON", m.group(1))
            fs[cur] = []
            continue
        if cur is None or not re.match(r"\s*/\*[0-9a-f]{4}\*/", line):
            continue                                                   # instructions only
        line = re.sub(r"/\*[0-9a-f]{4,}\*/|/\* 0x[0-9a-f]+ \*/", "", line)
        fs[cur].append(re.sub(r"_GLOBAL__N__\w+?_cu_[0-9a-f]+", "ANON", line).strip())
    return fs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--pair", nargs=2, action="append", default=[])
    a = ap.parse_args()
    A, B = functions(a.old), functions(a.new)
    common = [k for k in A if k in B]
    differ = [k for k in common if A[k] != B[k]]
    print("kernels: %d before, %d after; %d in both, %d of them with identical SASS" % (
        len(A), len(B), len(common), len(common) - len(differ)))
    for k in differ:
        print("DIFFERS", k)
    for k in A:
        if k not in B:
            print("ONLY BEFORE", k)
    for k in B:
        if k not in A:
            print("ONLY AFTER", k)
    for old, new in a.pair:
        ko = [k for k in A if old in k]
        kn = [k for k in B if new in k]
        assert len(ko) == 1 and len(kn) == 1, (ko, kn)
        same = A[ko[0]] == B[kn[0]]
        print("%s (%d instructions) vs %s (%d instructions): %s" % (ko[0], len(A[ko[0]]), kn[0], len(B[kn[0]]),
                                                                   "identical SASS" if same else "SASS DIFFERS"))


if __name__ == "__main__":
    main()
