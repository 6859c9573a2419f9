"""CPU: every ``src/<file>.py:<line>[-<line>]`` citation in the header, the docs, the oracle and the package points at
lines that exist in the reference.  Needs a checkout of the original project: point ``AVDN_REFERENCE_DIR`` at it (the
directory holding ``src/``); without one the test skips."""
import glob
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("AVDN_REFERENCE_DIR", "")
PAT = re.compile(r"(src/[\w/]+\.py):(\d+)(?:-(\d+))?")


@pytest.mark.skipif(not (REF and os.path.isdir(os.path.join(REF, "src"))),
                    reason="AVDN_REFERENCE_DIR does not name a checkout of the original project")
def test_reference_citations_exist():
    files = [os.path.join(ROOT, f) for f in ("include/avdn.h", "DESIGN.md", "INTEGRATION.md", "README.md")]
    files += glob.glob(os.path.join(ROOT, "oracle", "*.py"))
    files += glob.glob(os.path.join(ROOT, "aerial-vision-and-dialog-navigation_b200", "**", "*.py"), recursive=True)
    files += glob.glob(os.path.join(ROOT, "aerial-vision-and-dialog-navigation_b200", "csrc", "*.cu"))
    n_lines, bad, n = {}, [], 0
    for f in files:
        with open(f) as fh:
            text = fh.read()
        for m in PAT.finditer(text):
            n += 1
            path = os.path.join(REF, m.group(1))
            if path not in n_lines:
                n_lines[path] = len(open(path).read().splitlines()) if os.path.exists(path) else None
            lo, hi = int(m.group(2)), int(m.group(3) or m.group(2))
            if n_lines[path] is None or lo < 1 or hi < lo or hi > n_lines[path]:
                bad.append((os.path.relpath(f, ROOT), m.group(0)))
    assert n > 100, n                                   # the header alone cites dozens of call sites
    assert not bad, bad
