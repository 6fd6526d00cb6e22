"""The library has one behaviour: no environment variable, overridable macro or Makefile define selects a second code
path or changes a tuned constant.  A variant worth comparing is built from its own commit (MGYM_LIB loads another
build of the library) instead of living on in the source behind a switch that no test sets."""
import glob
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "modurl_gym_b200", "csrc")


def sources():
    paths = sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cuh")))
    assert paths, "no CUDA sources found"
    return {os.path.basename(p): open(p).read() for p in paths}


def test_no_environment_overrides():
    found = [name for name, text in sources().items() if re.search(r"\bgetenv\s*\(", text)]
    assert not found, f"getenv() in {found}: the library reads no environment variables"


def test_no_overridable_macro_defaults():
    # `#ifndef X` directly followed by `#define X ...`: a default that a -DX=... build flag replaces
    pattern = re.compile(r"^[ \t]*#[ \t]*ifndef[ \t]+(\w+)[ \t]*\n[ \t]*#[ \t]*define[ \t]+\1\b", re.M)
    found = [(name, m.group(1)) for name, text in sources().items() for m in pattern.finditer(text)]
    assert not found, f"overridable build-time defaults: {found}"


def test_makefile_passes_no_defines():
    text = open(os.path.join(CSRC, "Makefile")).read()
    found = re.findall(r"(?<!\S)-D\S*", text)
    assert not found, f"the Makefile passes {found}"
