"""Every `file.py:NN[-MM]` citation of a reference file in the product, the oracle, the tests and the docs points INSIDE that file
(VERDICT round 1 found citations of lines that do not exist).  Range check only - what the lines say is the reviewer's job.
The line counts of the reference's files are stored (tests/refgold.py)."""
import glob
import os
import re

from oracle import ref_dit
from tests import refgold

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAT = re.compile(r"([A-Za-z0-9_]+\.(?:py|yaml|txt|toml)):(\d+)(?:[-–](\d+))?((?:,\s*\d+(?:[-–]\d+)?)*)")


def _reference_file_lengths():
    """{file name: [line count of every reference file of that name]}"""
    lengths = {}
    for pat in ("**/*.py", "**/*.yaml", "*.txt", "*.toml"):
        for p in sorted(glob.glob(os.path.join(ref_dit.REFERENCE_ROOT, pat), recursive=True)):
            with open(p, errors="replace") as f:
                lengths.setdefault(os.path.basename(p), []).append(sum(1 for _ in f))
    return lengths


def test_reference_citations_are_inside_the_cited_files():
    lengths = refgold.want("citations/reference_file_lengths", _reference_file_lengths)
    files = [p for pat in ("easyanimate_b200/**/*.py", "easyanimate_b200/csrc/*.cu*", "easyanimate_b200/csrc/*.h", "include/*.h",
                           "oracle/**/*.py", "tests/**/*.py", "tools/*.py", "*.md", "bench.py", "__graft_entry__.py")
             for p in glob.glob(os.path.join(ROOT, pat), recursive=True)
             if os.path.basename(p) not in ("VERDICT.md", "SURVEY.md", "BASELINE.md", "PAPERS.md", "SNIPPETS.md", "ADVICE.md")]
    checked, bad = 0, []
    for path in files:
        with open(path, errors="replace") as f:
            text = f.read()
        for m in PAT.finditer(text):
            name = m.group(1)
            if name not in lengths:
                continue  # a file of this repository, not of the reference
            last = max(int(x) for x in re.findall(r"\d+", m.group(0)[len(name) + 1:]))
            checked += 1
            if all(last > n for n in lengths[name]):
                bad.append(f"{os.path.relpath(path, ROOT)}: {m.group(0)} (longest {name}: {max(lengths[name])} lines)")
    assert checked > 200 and not bad, bad
