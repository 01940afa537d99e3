"""Kernel census: which test launches which kernel of libdist_b200.so.

Runs the in-process GPU suite (pytest -m gpu) with a plugin that wraps every test -- setup, call and teardown -- in
torch.profiler with CUDA activities.  CUPTI records every kernel of the process, the ctypes-loaded library's as well as
torch's own; the kernels of the library are recognised by their demangled names and written back under their mangled
symbols, the names `cuobjdump -elf` lists:

    profiles/kernel_census.json   {"kernels": {mangled symbol: {"tests": count, "launched_by": [test ids]}}, ...}

tests/test_kernel_census.py compares that file with the symbols of a fresh build: a kernel neither in the census nor in
tests/kernel_census_exclusions.json fails the suite on a machine without a GPU.

Not seen: kernels launched in a child process -- the C++ drivers under tests/cpp/ (test_cpp_api.py, test_dropin.py,
the C++ cases of test_gpu_score_logp.py) and the multi-process runs of test_multigpu.py.  A kernel reached only there
shows up as never launched: it needs an in-process test too.  Run on a B200:

    python profiles/experiments/kernel_census.py [--out=PATH] [extra pytest args]
"""
import json
import os
import re
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from distributions_b200 import build  # noqa: E402

OUT = os.path.join(ROOT, "profiles", "kernel_census.json")
MAX_IDS = 25  # test ids kept per kernel (the count is kept in full)
NOT_SEEN = ("kernels launched in child processes are not recorded: tests/cpp/* drivers (test_cpp_api.py, test_dropin.py, "
            "the C++ cases of test_gpu_score_logp.py) and the multi-process runs of test_multigpu.py")


def cuda_bin(name):
    for d in (os.environ.get("CUDA_HOME", ""), "/usr/local/cuda"):
        p = os.path.join(d, "bin", name)
        if d and os.path.exists(p):
            return p
    return name


def portable(sym):
    """a kernel symbol without the hash nvcc derives from the source file's path for an anonymous namespace, so that
    builds in different directories name a kernel alike (the same rule is in tests/test_kernel_census.py)"""
    return re.sub(r"_GLOBAL__N__[0-9a-f]+_", "_GLOBAL__N__@_", sym)


def kernel_symbols(lib=build.LIB):
    """mangled names of every kernel in the library's device code (one .text.<symbol> section each)"""
    out = subprocess.run([cuda_bin("cuobjdump"), "-elf", lib], capture_output=True, text=True, check=True).stdout
    return sorted(set(re.findall(r"(?<![\w.])\.text\.(\S+)", out)))


def _norm(name):
    return re.sub(r"\s+", "", name)


def demangled_map(symbols):
    """normalised demangled name -> mangled symbol, by both demanglers (their spellings of a template argument differ)"""
    m = {}
    for tool in (cuda_bin("cu++filt"), "c++filt"):
        try:
            out = subprocess.run([tool], input="\n".join(symbols), capture_output=True, text=True, check=True).stdout
        except (OSError, subprocess.CalledProcessError):
            continue
        for sym, dem in zip(symbols, out.splitlines()):
            m[_norm(dem)] = sym
            m[_norm(dem.split("(")[0])] = sym  # without the parameter list
    return m


class Census:
    def __init__(self, symbols):
        self.symbols = set(symbols)
        self.by_name = demangled_map(symbols)
        self.hits = {}        # mangled -> set of test ids
        self.foreign = set()  # kernels of other libraries (torch's own)

    def _resolve(self, name):
        if name in self.symbols:
            return name
        n = _norm(name)
        return self.by_name.get(n) or self.by_name.get(n.split("(")[0])

    @pytest.hookimpl(hookwrapper=True)
    def pytest_runtest_protocol(self, item, nextitem):
        prof = torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA])
        prof.__enter__()
        try:
            yield
        finally:
            if torch.cuda.is_available():
                torch.cuda.synchronize()
            prof.__exit__(None, None, None)
            for ev in prof.events():
                if ev.device_type != torch.autograd.DeviceType.CUDA:
                    continue
                sym = self._resolve(ev.name)
                if sym is None:
                    self.foreign.add(ev.name)
                else:
                    self.hits.setdefault(sym, set()).add(item.nodeid)


def main(argv):
    out = OUT
    if argv and argv[0].startswith("--out="):
        out, argv = argv[0][len("--out="):], argv[1:]
    assert torch.cuda.is_available(), "the census needs a CUDA device"
    lib = build.build()
    symbols = kernel_symbols(lib)
    census = Census(symbols)
    args = [os.path.join(ROOT, "tests"), "-m", "gpu", "-q", "-p", "no:cacheprovider"] + argv
    rc = pytest.main(args, plugins=[census])
    kernels = {portable(s): {"tests": len(ids), "launched_by": sorted(ids)[:MAX_IDS]} for s, ids in sorted(census.hits.items())}
    never = sorted(set(map(portable, symbols)) - set(kernels))
    with open(out, "w") as fh:
        json.dump({"pytest_args": ["tests", "-m", "gpu"] + argv, "pytest_exit": int(rc), "not_seen": NOT_SEEN,
                   "symbols_in_build": len(symbols), "kernels": kernels, "never_launched": never}, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print("[census] pytest exit %d; %d of %d kernel symbols launched in-process; %s" % (rc, len(kernels), len(symbols), NOT_SEEN))
    for s in never:
        print("[census] never launched: %s" % s)
    print("[census] other kernels seen (not in the library): %d" % len(census.foreign))
    for name in sorted(n for n in census.foreign if "distb200" in n):  # a name the demanglers spell differently
        print("[census] UNRESOLVED library kernel: %s" % name)
    # CUPTI sees the ctypes-loaded library: the numerics probe is launched by exactly this test
    probe = [s for s in kernels if "numerics_probe_kernel" in s]
    print("[census] numerics_probe_kernel launched by: %s" % [kernels[s]["launched_by"] for s in probe])
    return int(rc)


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
