"""Throughput of dist_b200_sample_values_batch (batched Group::sample_value) per model, at sizes larger than L2:
10^8 rows for the scalar models, 10^7 rows for niw at d = 32.  For each model it prints the time of one call (CUDA
events, median of 5 after a warm-up), draws per second, and the share of the HBM bound, with the bytes counted from
the shapes: 4 B of assign plus the output bytes per row and feature.  Where a model does not reach the HBM bound, the
line also gives the FP32-FMA lane-op slots one draw occupies at the measured rate (dist_b200_pipe_peak(1) over the
draw rate), the measure of how much arithmetic -- the Philox4x32-10 block(s) and the rejection samplers -- each
draw costs.  The device name and power limit are read in the same run.  Run on a B200:
    python profiles/experiments/sample_values.py > profiles/experiments/sample_values.txt
"""
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
from distributions_b200 import capi  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


def workloads(rng, G=256):
    sizes = rng.integers(0, 5000, G)
    yield "nich", dict(model="nich", shared=np.array([0, 1, 1, 1], np.float32), count=sizes.astype(np.int32),
                       mean=rng.normal(size=G).astype(np.float32), ctv=(sizes * rng.uniform(0.5, 2, G)).astype(np.float32)), 10**8
    yield "gp", dict(model="gp", shared=np.array([1, 1], np.float32), count=sizes.astype(np.uint32),
                     sum=(sizes * rng.uniform(0.5, 30, G)).astype(np.uint32)), 10**8
    yield "bnb", dict(model="bnb", shared=np.array([2, 2, 3], np.float32), count=sizes.astype(np.uint32),
                      sum=(sizes * rng.uniform(0.5, 30, G)).astype(np.uint32)), 10**8
    yield "bb", dict(model="bb", shared=np.array([0.5, 2], np.float32), heads=(sizes // 3).astype(np.int32),
                     tails=(sizes - sizes // 3).astype(np.int32)), 10**8
    yield "dd16", dict(model="dd", alphas=np.full(16, 0.5, np.float32), counts=rng.integers(0, 300, (G, 16)).astype(np.int32)), 10**8
    yield "dd256", dict(model="dd", alphas=np.full(256, 0.5, np.float32), counts=rng.integers(0, 30, (G, 256)).astype(np.int32)), 10**8
    V = 1024
    yield "dpd1024", dict(model="dpd", alpha=2.0, beta0=0.1, keys=np.arange(V, dtype=np.uint32) * 3,
                          betas=np.full(V, 0.9 / V, np.float32), counts=rng.integers(0, 10, (G, V)).astype(np.int32)), 10**8
    d, Gn = 32, 64
    x = rng.normal(size=(Gn, 50, d)).astype(np.float32)
    yield "niw32", dict(model="niw", mu=np.zeros(d, np.float32), kappa=1.0, psi=np.eye(d, dtype=np.float32), nu=d + 1.0,
                        count=np.full(Gn, 50, np.int32), sum_x=x.sum(1), sum_xxT=np.einsum("gni,gnj->gij", x, x)), 10**7


def main():
    ctx = capi.Context(0)
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    fma = ctx.pipe_peak(1)
    print("device: %s | power limit, max SM clock: %s | FP32 FMA lane-ops/s (measured): %.3g" % (name, q, fma))
    print("%-8s %11s %10s %12s %9s %10s %s" % ("model", "rows", "ms/call", "draws/s", "GB/s", "HBM share", "FMA lane-op slots / draw"))
    rng = np.random.default_rng(0)
    for label, w, N in workloads(rng):
        mid = {"nich": capi.NICH, "gp": capi.GP, "bnb": capi.BNB, "bb": capi.BB, "dd": capi.DD, "dpd": capi.DPD, "niw": capi.NIW}[w["model"]]
        f = ctx.feature(mid).update_all(w)
        G = f.groups
        assign = torch.randint(0, G, (N,), dtype=torch.int32, device="cuda")
        shape = (N, f.dim) if mid == capi.NIW else (N,)
        out = torch.empty(shape, dtype={capi.BB: torch.uint8, capi.NICH: torch.float32, capi.NIW: torch.float32}.get(mid, torch.int32),
                          device="cuda")
        ctx.sample_values_batch([f], assign, N, [out], seed=1)
        torch.cuda.synchronize()
        times = []
        for rep in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ctx.sample_values_batch([f], assign, N, [out], seed=2 + rep)
            b.record()
            b.synchronize()
            times.append(a.elapsed_time(b) / 1e3)
        t = float(np.median(times))
        nbytes = N * (4 + out.element_size() * (f.dim if mid == capi.NIW else 1))
        share = nbytes / t / HBM_BYTES_PER_S
        print("%-8s %11d %10.3f %12.4g %9.0f %9.1f%% %.0f" % (label, N, t * 1e3, N / t, nbytes / t / 1e9, 100 * share, fma / (N / t)))
        del assign, out
        f.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
