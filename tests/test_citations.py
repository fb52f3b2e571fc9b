"""Every `file.cc:line` / `file.h:from-to` citation of the reference in this repo's sources and documents must point at a file that
exists in the reference and is long enough (a citation that rotted is worse than none).  The reference's files and their line counts
are committed as tests/golden/reference_line_counts.json (tests/golden/make_reference_line_counts.py writes it from a reference tree)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINE_COUNTS = os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")
OWN = {"b200c.h", "kernels.h", "gp_rules.h", "bloom_rules.h", "sst_host.h", "sst_host.cc", "compaction_oracle.h", "compaction_oracle.c",
       "encode.cu", "merge.cu", "decode.cu", "api.cu", "common.cuh", "b200_compaction_executor.cc", "b200_compaction_executor.h",
       "ref_compact.cc", "ref_sst_check.cc"}
PAT = re.compile(r"([A-Za-z0-9_./]+\.(?:cc|h)):(\d+)(?:-(\d+))?")


def repo_files():
    """the repository's sources and documents, relative to ROOT (build output and hidden / private directories left out)"""
    out = []
    for dp, ds, fs in os.walk(ROOT):
        ds[:] = sorted(d for d in ds if not d.startswith((".", "_")) and d != "build")
        for f in sorted(fs):
            rel = os.path.relpath(os.path.join(dp, f), ROOT)
            if f.endswith((".h", ".cu", ".cuh", ".cc", ".c", ".py", ".md")) and rel not in ("SURVEY.md", "PAPERS.md", "SNIPPETS.md"):
                out.append(rel)
    return out


def citations():
    """(file, citation text, cited path, first line, last line) of every citation of a reference file"""
    for f in repo_files():
        txt = open(os.path.join(ROOT, f), errors="replace").read()
        for m in PAT.finditer(txt):
            path, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            if os.path.basename(path) not in OWN:
                yield f, m.group(0), path, a, b


def test_reference_citations_resolve():
    nlines = json.load(open(LINE_COUNTS))["files"]
    index = {}
    for p in nlines:
        index.setdefault(os.path.basename(p), []).append(p)
    checked, bad = 0, []
    for f, cite, path, a, b in citations():
        cands = index.get(os.path.basename(path), [])
        if "/" in path:
            cands = [c for c in cands if ("/" + c).endswith("/" + path)] or cands
        checked += 1
        if not cands:
            bad.append((f, cite, "no such file in the reference"))
        elif all(max(a, b) > nlines[c] for c in cands):
            bad.append((f, cite, "beyond the end of the file"))
    assert checked > 200
    assert not bad, bad[:20]
