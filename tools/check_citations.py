#!/usr/bin/env python
"""Every `dir/file.py:LINE[-LINE]` citation of the reference tree in our sources and docs must name an existing reference file and a
line range inside it (a reviewer follows these to check parity).  Needs the reference tree (or build()'s copy under oracle/_ref);
the test suite checks against the line counts stored in tests/golden/reference_line_counts.json instead.
    python tools/check_citations.py            # prints the stale ones, exit code 1 if any"""
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
CITE = re.compile(r"(?<![\w/.])((?:search|train|latency|tools)/[\w/]+\.py):(\d+)(?:-(\d+))?")
BARE = re.compile(r"(?<![\w/.])([a-z_]+\.py):(\d+)(?:-(\d+))?")      # `model_search.py:361-475`: must fit a reference file of that name
SCAN = ("fasterseg_b200", "include", "oracle", "tests", "tools", "bench.py", "__graft_entry__.py", "DESIGN.md", "INTEGRATION.md", "README.md")
SKIP_DIRS = {"__pycache__", "_ref", "golden", "debug"}


def files():
    for top in SCAN:
        p = os.path.join(ROOT, top)
        if os.path.isfile(p):
            yield p
            continue
        for d, dirs, names in os.walk(p):
            dirs[:] = [x for x in dirs if x not in SKIP_DIRS]
            for n in names:
                if n.endswith((".py", ".cu", ".cuh", ".h", ".md", ".sh")):
                    yield os.path.join(d, n)


def line_counts(ref_root):
    """{path relative to the reference root: number of lines} of every reference .py file"""
    counts = {}
    for d, _, names in os.walk(ref_root):
        for n in names:
            if n.endswith(".py"):
                p = os.path.join(d, n)
                counts[os.path.relpath(p, ref_root).replace(os.sep, "/")] = sum(1 for _ in open(p, errors="replace"))
    return counts


def stale(counts):
    """citations that do not fit the reference files described by `counts` (see line_counts) -> (stale ones, number checked)"""
    bad, total = [], 0
    by_name = {}
    for path, n in counts.items():
        by_name.setdefault(os.path.basename(path), []).append(n)
    for f in files():
        try:
            text = open(f, errors="replace").read()
        except OSError:
            continue
        for m in CITE.finditer(text):
            path, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            total += 1
            n = counts.get(path, -1)
            if n < 0:
                bad.append((os.path.relpath(f, ROOT), m.group(0), "no such reference file"))
            elif not (1 <= lo <= hi <= n):
                bad.append((os.path.relpath(f, ROOT), m.group(0), "file has %d lines" % n))
        for m in BARE.finditer(text):
            name, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            if name not in by_name:
                continue                  # one of OUR files (graphed.py:12 ...), not a reference citation
            total += 1
            if not any(1 <= lo <= hi <= n for n in by_name[name]):
                bad.append((os.path.relpath(f, ROOT), m.group(0), "reference files of that name have %s lines" % by_name[name]))
    return bad, total


def main():
    from oracle import ref_harness
    if not ref_harness.reference_available():
        print("reference tree not available")
        return 0
    bad, total = stale(line_counts(ref_harness.REFERENCE_ROOT))
    for b in bad:
        print("%s: %s (%s)" % b)
    print("%d citations checked, %d stale" % (total, len(bad)))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
