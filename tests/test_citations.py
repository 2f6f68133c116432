"""Every `file:line` citation of the reference in the ABI header, the docs, the oracle and the CUDA sources must point at
an existing file of the reference tree with at least that many lines.  The reference tree is not part of this repository:
the check runs against tests/golden/reference_line_counts.json, the path and line count of every file of that tree.
Regenerate it from a checkout of the reference with  python tests/test_citations.py <reference-dir>"""
import json
import os
import re
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INDEX = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
PAT = re.compile(r"([A-Za-z0-9_/\.]+\.(?:h|cpp|yaml|md|txt)):(\d+)(?:-(\d+))?")


def _n_lines(p):
    with open(p, errors="ignore") as fh:
        return sum(1 for _ in fh)


def make_index(ref_dir):
    """{path relative to the reference root: number of lines} of every file of the reference tree."""
    out = {}
    for d, dirs, fs in os.walk(ref_dir):
        dirs[:] = sorted(x for x in dirs if x != ".git")
        for f in sorted(fs):
            p = os.path.join(d, f)
            out[os.path.relpath(p, ref_dir)] = _n_lines(p)
    return out


def _sources():
    out = [os.path.join(ROOT, p) for p in ("DESIGN.md", "INTEGRATION.md", "include/fls_b200.h", "funny_lidar_slam_b200/shim/b200_registration.h")]
    for d, exts in (("oracle", (".h", ".cpp", ".py")), ("funny_lidar_slam_b200/csrc", (".cu", ".cuh", ".h"))):
        out += [os.path.join(ROOT, d, f) for f in sorted(os.listdir(os.path.join(ROOT, d))) if f.endswith(exts)]
    return out


def test_reference_citations_resolve():
    with open(INDEX) as fh:
        index = json.load(fh)
    files = {}
    for rel, n in index.items():
        files.setdefault(os.path.basename(rel), []).append(("/" + rel, n))

    checked, bad = 0, []
    for src in _sources():
        for m in PAT.finditer(open(src, errors="ignore").read()):
            path, last = m.group(1), int(m.group(3) or m.group(2))
            base = os.path.basename(path)
            if base.startswith(("fls_", "orc_")) or base == "b200_registration.h":
                continue  # this repository's own files
            checked += 1
            cands = files.get(base, [])
            if "/" in path:
                cands = [c for c in cands if c[0].endswith(path)] or cands
            if not cands:
                bad.append((os.path.relpath(src, ROOT), m.group(0), "no such file in the reference"))
            elif max(n for _, n in cands) < last:
                bad.append((os.path.relpath(src, ROOT), m.group(0), "file is shorter than the cited line"))
    assert checked > 150
    assert not bad, bad


if __name__ == "__main__":
    with open(INDEX, "w") as fh:
        json.dump(make_index(sys.argv[1]), fh, indent=0, sort_keys=True)
        fh.write("\n")
