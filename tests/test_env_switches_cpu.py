"""The environment switches INTEGRATION.md documents are exactly the ones the library and the tools read."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def names_read_by_the_code():
    names = set()
    for d, _, files in os.walk(os.path.join(ROOT, "pacbio_b200", "csrc")):
        for f in files:
            if f.endswith((".cu", ".cuh", ".cpp", ".hpp", ".h")):
                names |= set(re.findall(r'getenv\(\s*"(MR_[A-Z0-9_]+)"', open(os.path.join(d, f)).read()))
    return names


def names_in_integration_md():
    status = set(re.findall(r"#define\s+(MR_[A-Z0-9_]+)", open(os.path.join(ROOT, "include", "mega_reads_b200.h")).read()))
    return set(re.findall(r"\b(MR_[A-Z0-9_]+)\b", open(os.path.join(ROOT, "INTEGRATION.md")).read())) - status


def test_integration_md_lists_every_switch_the_code_reads():
    code, doc = names_read_by_the_code(), names_in_integration_md()
    assert len(code) > 10
    assert sorted(code - doc) == [], "read by the code but not documented in INTEGRATION.md"
    assert sorted(doc - code) == [], "documented in INTEGRATION.md but read nowhere"
