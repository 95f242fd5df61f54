"""Every `[src/]<file>.f90:<line[-line]>` citation into the reference (headers, kernels, oracle, docs) must point at lines that
exist.  Runs where the CDFTOOLS sources are at hand ($CDFTOOLS_REF, a checkout of the reference); skipped without them."""
import os
import re
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
REF = Path(os.environ["CDFTOOLS_REF"]) if os.environ.get("CDFTOOLS_REF") else None
PAT = re.compile(r"\b(?:src/)?([A-Za-z0-9_]+\.[fF]90)\s*:\s*(\d+)(?:\s*-\s*(\d+))?")


def _sources():
    pats = ["include/*.h", "cdftools_b200/csrc/*.cu*", "cdftools_b200/csrc/*.inc", "cdftools_b200/csrc/host/*pp", "oracle/*.c", "oracle/*.py",
            "cdftools_b200/*.py", "cdftools_b200/fortran/*.f90", "DESIGN.md", "INTEGRATION.md", "tests/*.py", "tests/golden/*.json"]
    for p in pats:
        yield from ROOT.glob(p)


@pytest.mark.skipif(REF is None or not (REF / "src").exists(), reason="needs the CDFTOOLS sources ($CDFTOOLS_REF)")
def test_cited_reference_lines_exist():
    nlines = {}
    bad, total = [], 0
    for f in _sources():
        for m in PAT.finditer(f.read_text(errors="ignore")):
            rel, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            path = REF / "src" / rel
            if rel not in nlines:
                nlines[rel] = len(path.read_text(errors="ignore").splitlines()) if path.exists() else -1
            total += 1
            if nlines[rel] < 0 or not (1 <= a <= b <= nlines[rel]):
                bad.append((f.relative_to(ROOT).as_posix(), m.group(0), nlines[rel]))
    assert total > 200, total                      # the tree cites the reference a few hundred times
    assert not bad, bad[:20]
