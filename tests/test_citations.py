"""Reference citations (file:line) in the C ABI header, the kernels, the oracle and DESIGN.md point at real lines of the
reference tree. Needs a checkout of the original BaMMmotif2 (the tree oracle/Makefile builds the reference from), named by the
environment variable BAMM_REFERENCE; skipped without it."""
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("BAMM_REFERENCE", "")
CITE = re.compile(r"(?<![A-Za-z_/.])((?:src/[A-Za-z_/]+/)?[A-Za-z_]+\.(?:cpp|h)):(\d+)(?:-(\d+))?")


def cited_files():
    out = [os.path.join(ROOT, "include", "bamm_b200.h"), os.path.join(ROOT, "DESIGN.md"), os.path.join(ROOT, "INTEGRATION.md"),
           os.path.join(ROOT, "oracle", "bamm_oracle.c")]
    for d in ("bammmotif2_b200/csrc", "bammmotif2_b200/host"):
        for f in sorted(os.listdir(os.path.join(ROOT, d))):
            if f.endswith((".cuh", ".cu", ".inl", ".cpp", ".h")):
                out.append(os.path.join(ROOT, d, f))
    return out


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "src"))), reason="BAMM_REFERENCE does not name a BaMMmotif2 checkout")
def test_reference_citations_resolve():
    by_name = {}
    for d, _, files in os.walk(os.path.join(REF, "src")):
        for f in files:
            by_name.setdefault(f, []).append(os.path.relpath(os.path.join(d, f), REF))
    lengths, bad, n = {}, [], 0
    for path in cited_files():
        for m in CITE.finditer(open(path, errors="replace").read()):
            rel, a, b = m.group(1), int(m.group(2)), int(m.group(3) or m.group(2))
            if "/" not in rel:                                   # bare file name: must be a reference file (ours are not cited this way)
                cands = by_name.get(rel, [])
                if len(cands) != 1:
                    continue
                rel = cands[0]
            n += 1
            full = os.path.join(REF, rel)
            if rel not in lengths:
                lengths[rel] = sum(1 for _ in open(full, errors="replace")) if os.path.isfile(full) else -1
            if lengths[rel] < 0 or not (1 <= a <= b <= lengths[rel]):
                bad.append("%s cites %s:%d-%d (file has %d lines)" % (os.path.relpath(path, ROOT), rel, a, b, lengths[rel]))
    assert n > 100, "expected the sources to carry reference citations"
    assert not bad, "\n".join(bad[:20])
