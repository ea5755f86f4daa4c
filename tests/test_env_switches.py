"""CPU: the environment variables the library reads are exactly the ones INTEGRATION.md lists."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _read_by_code():
    names = set()
    for path in glob.glob(os.path.join(ROOT, "pinthememory_b200", "csrc", "*.cu")) + \
            glob.glob(os.path.join(ROOT, "pinthememory_b200", "csrc", "*.cuh")):
        names |= set(re.findall(r'getenv\(\s*"(\w+)"', open(path).read()))
    for path in glob.glob(os.path.join(ROOT, "pinthememory_b200", "*.py")):
        names |= set(re.findall(r'os\.environ\.get\(\s*"(\w+)"', open(path).read()))
    return names


def _documented():
    """First backticked name of every item of INTEGRATION.md's "Environment" list."""
    lines = open(os.path.join(ROOT, "INTEGRATION.md")).read().splitlines()
    start = next(i for i, line in enumerate(lines) if line.startswith("* Environment"))
    names = []
    for line in lines[start + 1:]:
        if not line.startswith("  "):
            break
        m = re.match(r"\s+- `(\w+)", line)
        if m:
            names.append(m.group(1))
    return names


def test_every_environment_variable_is_documented_and_nothing_else():
    code, doc = _read_by_code(), _documented()
    assert len(doc) == len(set(doc)), doc
    assert code, "no environment reads found: the scan is broken"
    assert sorted(code - set(doc)) == [], "read by the code, not listed in INTEGRATION.md"
    assert sorted(set(doc) - code) == [], "listed in INTEGRATION.md, not read by the code"
