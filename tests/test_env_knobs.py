"""CPU: the ELECTOR_* environment variables the library reads are exactly those INTEGRATION.md's environment table lists:
getenv("ELECTOR_...") in elector_b200/csrc, os.environ...("ELECTOR_...") in the Python package."""
import glob
import os
import re

from conftest import ROOT


def names_read():
    names = set()
    for path in glob.glob(os.path.join(ROOT, "elector_b200", "csrc", "*")):
        names |= set(re.findall(r'\bgetenv\(\s*"(ELECTOR_[A-Z0-9_]+)"', open(path).read()))
    for path in glob.glob(os.path.join(ROOT, "elector_b200", "*.py")):
        names |= set(re.findall(r'\bos\.environ(?:\.\w+\(|\[)\s*["\'](ELECTOR_[A-Z0-9_]+)["\']', open(path).read()))
    return names


def names_documented():
    lines = open(os.path.join(ROOT, "INTEGRATION.md")).read().splitlines()
    start = next(i for i, line in enumerate(lines) if line.startswith("## Environment knobs"))
    rows = []
    for line in lines[start + 1:]:
        if line.startswith("|"):
            rows.append(line)
        elif rows or line.startswith("#"):
            break
    return set(re.findall(r"`(ELECTOR_[A-Z0-9_]+)`", "\n".join(rows)))


def test_environment_table_lists_exactly_what_the_library_reads():
    read, documented = names_read(), names_documented()
    assert "ELECTOR_TRACE" in read and "ELECTOR_DEVICE" in read
    assert read - documented == set(), "read but not in INTEGRATION.md's environment table"
    assert documented - read == set(), "in INTEGRATION.md's environment table but read nowhere"
