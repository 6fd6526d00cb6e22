#!/usr/bin/env python
"""Did a change leave existing kernels alone?  For every kernel of the OLD libmgym.so, is there a kernel of the NEW
one with the identical instruction stream (names ignored: a new template parameter renames a kernel without changing
its code)?  No GPU needed.

    python tools/sass_compare.py old/libmgym.so new/libmgym.so
"""
import collections
import hashlib
import re
import subprocess
import sys


def kernels(lib):
    out = subprocess.run(["cuobjdump", "-sass", lib], capture_output=True, text=True, check=True).stdout
    fs, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            fs[cur] = []
        elif cur is not None:
            m = re.match(r"\s*/\*[0-9a-f]{4}\*/\s*(.*?)\s*;", line)  # one instruction, without its address
            if m:
                fs[cur].append(m.group(1))
    return fs


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    digest = lambda ins: hashlib.sha1("\n".join(ins).encode()).hexdigest()
    have = collections.Counter(digest(v) for v in new.values())
    changed = sorted(k for k, v in old.items() if have[digest(v)] == 0)
    print(f"{len(old)} kernels before, {len(new)} after; {len(changed)} old kernels without an identical stream")
    for k in changed:
        print("  ", k)
    sys.exit(1 if changed else 0)


if __name__ == "__main__":
    main()
