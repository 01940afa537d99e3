"""Every kernel of the build is launched by an in-process test, or deliberately excluded.

profiles/kernel_census.json is written on a B200 by profiles/experiments/kernel_census.py: for each kernel symbol of
libdist_b200.so, the GPU tests that launched it.  tests/kernel_census_exclusions.json lists the kernels no test launches
on purpose, each with its reason.  Against the symbols `cuobjdump -elf` finds in the built library (no GPU needed):
  - a symbol in neither file is a kernel instantiation without a test (a new template argument, a new kernel);
  - a census or exclusion entry the build no longer has is stale (the census was not re-run after a change).
"""
import json
import os
import re
import shutil
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB = os.path.join(ROOT, "distributions_b200", "lib", "libdist_b200.so")
CENSUS = os.path.join(ROOT, "profiles", "kernel_census.json")
EXCLUSIONS = os.path.join(ROOT, "tests", "kernel_census_exclusions.json")


def _cuobjdump():
    for p in (os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump"), "/usr/local/cuda/bin/cuobjdump"):
        if os.path.exists(p):
            return p
    return shutil.which("cuobjdump")


@pytest.fixture(scope="module")
def symbols():
    tool = _cuobjdump()
    if tool is None:
        pytest.skip("cuobjdump not found")
    if not os.path.exists(LIB):
        pytest.skip("libdist_b200.so not built")
    out = subprocess.run([tool, "-elf", LIB], capture_output=True, text=True, check=True).stdout
    # nvcc names an anonymous namespace after a hash of the source file's path: left out, so that the census written from one
    # build matches a build in another directory (the same rule is in profiles/experiments/kernel_census.py)
    syms = {re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__@_", s) for s in re.findall(r"(?<![\w.])\.text\.(\S+)", out)}
    assert syms, "no kernel sections found in %s" % LIB
    return syms


def _load(path):
    with open(path) as fh:
        return json.load(fh)


def test_exclusions_have_reasons():
    ex = _load(EXCLUSIONS)
    for sym, reason in ex.items():
        assert isinstance(reason, str) and reason.strip(), sym


def test_every_kernel_is_launched_or_excluded(symbols):
    launched = set(_load(CENSUS)["kernels"])
    excluded = set(_load(EXCLUSIONS))
    missing = sorted(symbols - launched - excluded)
    assert not missing, "kernels no test launches (run profiles/experiments/kernel_census.py on a B200): %s" % missing


def test_census_names_only_built_kernels(symbols):
    census = _load(CENSUS)
    stale = sorted((set(census["kernels"]) | set(_load(EXCLUSIONS))) - symbols)
    assert not stale, "census / exclusion entries the build does not have: %s" % stale
