#!/usr/bin/env python
"""Compare the machine code of every kernel of two builds of libgpd_b200.so (cuobjdump -sass, no GPU needed).

    python profiles/sass_compare.py OLD.so NEW.so

Kernels are matched by mangled name; instruction words (encodings included) are compared with the address comments and
column padding removed.  Exit status 1 if a kernel of OLD is missing from NEW or compiles to different code; kernels only in
NEW are listed.  Used to show that a change adding kernels or refactoring shared device functions leaves the existing
kernels' code untouched."""
import re
import subprocess
import sys

HEADER = re.compile(r"\s*(identifier|compressed|code version|host =|compile_size|code for|Fatbin|arch =|producer|\.\.\.|$)")


def kernels(path):
    out = subprocess.run(["cuobjdump", "-sass", path], capture_output=True, text=True, check=True).stdout
    res, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            res[cur] = []
        elif cur and not HEADER.match(line):
            res[cur].append(" ".join(re.sub(r"/\*[0-9a-f]{4,}\*/", "", line).split()))
    return res


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    bad = [k for k in old if old[k] != new.get(k)]
    for k in bad:
        print("differs or missing:", k)
    added = [k for k in new if k not in old]
    for k in added:
        print("new:", k)
    print(f"{len(old)} kernels in {sys.argv[1]}: {len(old) - len(bad)} identical, {len(bad)} differ; {len(added)} new")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
