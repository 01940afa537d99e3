"""Build distributions_b200/lib/libdist_b200.so (the C-ABI library + sm_100a kernels) in-tree with nvcc.

    python -m distributions_b200.build [--force] [--verbose]

nvcc cross-compiles for sm_100a without a GPU.  The .so is git-ignored but travels to the GPU box.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libdist_b200.so")
OBJ_DIR = os.path.join(LIB_DIR, "obj")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
COMMON = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
          "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
# per-file extra flags.  prep.cu keeps the reference's unfused multiply/add rounding; sample_values.cu shares its
# posterior code (posterior.cuh).
SOURCES = {
    "api.cu": [],
    "prep.cu": ["--fmad=false"],
    "score_rows.cu": [],
    "score_rows_cc32.cu": [],
    "score_rows_cc64.cu": [],
    "score_rows_masked.cu": [],
    "score_rows_masked_cc.cu": [],
    "missing.cu": [],
    "score_rows_nich.cu": [],
    "nich_rows.cu": [],
    "score_rows_gp.cu": [],
    "score_rows_bnb.cu": [],
    "score_rows_bb.cu": [],
    "score_rows_dd.cu": [],
    "gather_rows.cu": [],
    "table_rows.cu": [],
    "peer.cu": [],
    "niw.cu": [],
    "niw_tc.cu": [],
    "niw_tc_wide.cu": [],
    "niw_stats.cu": [],
    "microbench.cu": [],
    "stats.cu": [],
    "wire.cu": [],
    "sample_values.cu": ["--fmad=false"],
}


def _deps():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "dist_b200.h")]


def build(force=False, verbose=False):
    os.makedirs(OBJ_DIR, exist_ok=True)
    deps = _deps()
    newest = max(os.path.getmtime(d) for d in deps)
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= newest:
        return LIB
    hdr_time = max(os.path.getmtime(d) for d in deps if not d.endswith(".cu"))
    objs = []
    procs = []
    for src, extra in SOURCES.items():
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        if not force and os.path.exists(obj) and os.path.getmtime(obj) >= max(os.path.getmtime(path), hdr_time):
            continue
        cmd = [NVCC] + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write("---- %s\n%s\n" % (src, out))
        failed = failed or p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [NVCC, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
