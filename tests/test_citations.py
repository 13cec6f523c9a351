"""Every `path:line[-line]` citation of the reference in the headers, kernels, oracle and docs points at an existing file and
line range of the reference tree (tests/golden/reference_files.json: every file of the reference and its line count)."""
import glob
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_FILES = os.path.join(ROOT, "tests", "golden", "reference_files.json")
OWN = ("lsd", "hostmath", "internal", "track", "depth", "frame", "perma", "sim3", "output")


def test_reference_citations_resolve():
    with open(REF_FILES) as f:
        lines = json.load(f)
    idx = {}
    for p in lines:
        idx.setdefault(os.path.basename(p), []).append(p)
    pat = re.compile(r"([A-Za-z0-9_/\.]+\.(?:cpp|h|hpp|msg|cfg|txt)):(\d+)(?:-(\d+))?")
    srcs = ["include/lsdgpu.h", "DESIGN.md", "INTEGRATION.md", "README.md", "BASELINE.md"]
    for g in ("lsd_slam_b200/csrc/*", "lsd_slam_b200/host/*", "lsd_slam_b200/*.py", "oracle/*.c", "oracle/*.inc", "oracle/*.h", "tests/*.py"):
        srcs += [os.path.relpath(p, ROOT) for p in glob.glob(os.path.join(ROOT, g))]
    checked, bad = 0, []
    for s in srcs:
        txt = open(os.path.join(ROOT, s), errors="ignore").read()
        for m in pat.finditer(txt):
            path, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            base = os.path.basename(path)
            if base not in idx:
                if base.endswith((".cpp", ".h", ".hpp")) and not base.startswith(OWN):
                    bad.append((s, path, a, "no such file in the reference"))
                continue
            cands = [p for p in idx[base] if p.endswith(path)] or idx[base]
            n_lines = max(lines[p] for p in cands)
            checked += 1
            if b > n_lines or a > b:
                bad.append((s, path, a, b, n_lines))
    assert not bad, bad[:20]
    assert checked > 300
