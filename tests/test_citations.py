"""Every reference citation `path.py:line[-line]` in the C header, the oracle and the host layer must point into an existing file of
the reference tree, inside its length (CPU only).  The file lengths were recorded from the reference tree by
tests/golden/make_golden_reference_meta.py (tests/golden/reference_line_counts.json)."""
import json
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CITED_DIRS = ("coot", "nntrainer", "mart", "tests_nntrainer", "config")
PAT = re.compile(r"((?:" + "|".join(CITED_DIRS) + r")/[\w/.]+\.(?:py|yaml)):(\d+)(?:-(\d+))?")
SOURCES = ["include/coot_sm100.h", "oracle/coot_oracle.py", "oracle/retrieval_oracle.py", "oracle/optim_oracle.py", "oracle/ref_runner.py",
           "DESIGN.md", "INTEGRATION.md", "coot_videotext_b200/model_retrieval.py", "coot_videotext_b200/loss_fn.py",
           "coot_videotext_b200/retrieval.py", "coot_videotext_b200/optimization.py", "coot_videotext_b200/export.py",
           "coot_videotext_b200/data.py", "coot_videotext_b200/h5min.py", "coot_videotext_b200/synthetic.py"]


def test_reference_citations_resolve():
    lengths = json.load(open(os.path.join(ROOT, "tests", "golden", "reference_line_counts.json")))
    bad, total = [], 0
    for src in SOURCES:
        text = open(os.path.join(ROOT, src), encoding="utf8").read()
        for m in PAT.finditer(text):
            path, lo, hi = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            total += 1
            n = lengths.get(path, -1)
            if n < 0 or not (1 <= lo <= hi <= n):
                bad.append((src, m.group(0), n))
    assert total > 100, total
    assert not bad, bad
