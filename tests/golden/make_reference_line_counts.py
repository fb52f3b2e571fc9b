"""Writes tests/golden/reference_line_counts.json: the line count of every .cc / .h file of the reference whose base name a citation in
this repository names (all files of that name, wherever they lie), so that tests/test_citations.py checks the citations without the
reference.  Run again after adding a citation of a file not listed yet:
    python tests/golden/make_reference_line_counts.py <reference source tree>"""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from test_citations import LINE_COUNTS, citations  # noqa: E402

ref = sys.argv[1]
cited = {os.path.basename(path) for _, _, path, _, _ in citations()}
files = {}
for dp, _, fs in os.walk(ref):
    for f in fs:
        if f.endswith((".cc", ".h")) and f in cited:
            p = os.path.join(dp, f)
            with open(p, errors="replace") as fh:
                files[os.path.relpath(p, ref)] = sum(1 for _ in fh)
with open(LINE_COUNTS, "w") as fh:
    json.dump({"files": dict(sorted(files.items()))}, fh, indent=0)
    fh.write("\n")
print(len(files), "files of", len(cited), "cited names")
