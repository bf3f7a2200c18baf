"""CPU test of the native library's configuration surface: the environment variables it reads."""
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "genpercept_b200", "csrc")

# GP_GN_FUSE: GroupNorm fusion into the patch-resident convolution (read at plan time).
# GP_MAX_PLANS: bound on the cached execution plans per engine (include/genpercept_b200.h).
EXPECTED = {"GP_GN_FUSE", "GP_MAX_PLANS"}


def test_native_library_reads_only_the_documented_environment_variables():
    names = set()
    for f in sorted(os.listdir(CSRC)):
        if not f.endswith((".cu", ".cuh", ".h")):
            continue
        src = open(os.path.join(CSRC, f)).read()
        names |= set(re.findall(r"\bgetenv\s*\(\s*\"([A-Za-z0-9_]+)\"\s*\)", src))
        assert len(re.findall(r"\bgetenv\s*\(\s*\"", src)) == len(re.findall(r"\bgetenv\s*\(", src)), \
            f"{f}: getenv with a non-literal name"
    assert names == EXPECTED, sorted(names ^ EXPECTED)
