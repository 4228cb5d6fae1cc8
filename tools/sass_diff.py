"""Per-kernel SASS comparison of two builds of the same object file, e.g. the parent commit's and this tree's.

Usage: python tools/sass_diff.py OLD.o NEW.o [name-filter]
Prints SAME / DIFF / NEW / GONE per kernel, keyed by its demangled name and template arguments, and exits 1 when a
kernel of OLD is missing from NEW or differs.  Only instruction lines are compared, so the two objects may be compiled
from different directories (e.g. a `git worktree` of the parent).  No GPU needed."""
import re
import subprocess
import sys


def kernels(obj: str) -> dict:
    out = subprocess.run(["cuobjdump", "-sass", obj], capture_output=True, text=True, check=True).stdout
    d, cur = {}, None
    for line in out.splitlines():
        m = re.match(r"\s+Function : (\S+)", line)
        if m:
            cur = m.group(1)
            d[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4,}\*/", line):   # instructions only
            d[cur].append(" ".join(line.split()))   # column widths depend on the whole dump
    names = list(d)
    pretty = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True).stdout.splitlines()
    # key: name and template arguments; the parameter list may spell a dependent type differently between builds
    return {re.sub(r"\(.*$", "", p.replace("(anonymous namespace)::", "")): d[n] for n, p in zip(names, pretty)}


def main():
    old, new = kernels(sys.argv[1]), kernels(sys.argv[2])
    filt = sys.argv[3] if len(sys.argv) > 3 else ""
    bad = 0
    for n in sorted(set(old) | set(new)):
        if filt not in n:
            continue
        tag = "NEW" if n not in old else "GONE" if n not in new else "SAME" if old[n] == new[n] else "DIFF"
        bad += tag in ("DIFF", "GONE")
        print(f"{tag:4}  {n}")
    sys.exit(1 if bad else 0)


if __name__ == "__main__":
    main()
