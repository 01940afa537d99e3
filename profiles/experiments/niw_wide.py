"""NormalInverseWishart at d in {64, 100, 128} (the tcgen05 route of niw_tc_wide.cu and the other wide entries).

For d in {64, 100, 128}, G in {64, 256} and N = 1M rows (512 MB of rows at d = 128: more than L2), with CUDA events
around each call, the L2 flushed (256 MB written) before each, median of 5 after 2 warm-ups:
  score_sample    score_sample_batch (materialise + the stand-alone sampler)
  score           score_batch into [N][G]
  logp            score_logp_batch
  add_rows        add_rows_batch of all N rows
  score_data      score_data_grid at one grid point
  sample_values   sample_values_batch, one value per row
  torch_fp32      the same scores in torch fp32 with TF32 off: X @ Wstack^T - b, squared and summed per group (row chunks
                  of 32768), the Student-t epilogue omitted -- a plain-GEMM yardstick
Counted flops: 2 d^2 + 2 d per cell.  Issued fp16 flops of the route: (3 DP + 16) 2 DP per cell over the padded groups.
Both against the 2,250 TFLOP/s dense fp16 data-sheet figure for one HGX B200 GPU.  The card name, power limit and max SM
clock are read in the same run.  Run on a B200:
    python profiles/experiments/niw_wide.py > profiles/experiments/niw_wide.txt
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from distributions_b200 import capi, synth  # noqa: E402

PEAK_FP16 = 2250e12
FLUSH = torch.empty(256 * 1024 * 1024 // 4, device="cuda", dtype=torch.float32)


def timed(step, reps=5, warm=2):
    for _ in range(warm):
        FLUSH.zero_()
        step()
    ts = []
    for _ in range(reps):
        FLUSH.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) * 1e-3)
    return float(np.median(ts))


def whitening(w):
    """per group W = L^-1 and b = W mu' in float64 (the posterior of niw_posterior_cholesky), as float32 tensors"""
    d, G = w["mu"].size, w["count"].size
    mu, psi, kap, nu = w["mu"].astype(np.float64), w["psi"].astype(np.float64), float(w["kappa"]), float(w["nu"])
    Ws, bs = np.zeros((G, d, d)), np.zeros((G, d))
    for g in range(G):
        n = float(w["count"][g])
        sx, sxx = w["sum_x"][g].astype(np.float64), w["sum_xxT"][g].astype(np.float64)
        xbar = sx / n if n else np.zeros(d)
        diff = xbar - mu
        pk, dof = kap + n, nu + n - d + 1.0
        c_n = sxx - np.outer(sx, xbar) - np.outer(xbar, sx) + n * np.outer(xbar, xbar)
        S = (psi + c_n + kap * n / (kap + n) * np.outer(diff, diff)) * (pk + 1.0) / (pk * dof)
        W = np.linalg.inv(np.linalg.cholesky(S))
        Ws[g], bs[g] = W, W @ (kap / pk * mu + n / pk * xbar)
    return torch.from_numpy(Ws.reshape(G * d, d).astype(np.float32)).cuda(), torch.from_numpy(bs.reshape(G * d).astype(np.float32)).cuda()


def main():
    torch.backends.cuda.matmul.allow_tf32 = False
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()[0]
    print("# card: %s (name, power limit, max SM clock), read in this run" % q)
    print("# N = 1M rows, median of 5 after 2 warm-ups, L2 flushed before each call; times in ms")
    ctx = capi.Context(0)
    N = 1 << 20
    hdr = ("d", "G", "score_sample", "score", "logp", "add_rows", "score_data", "sample_values", "torch_fp32",
           "counted_TF/s", "counted/peak", "issued_TF/s", "issued/peak", "torch_TF/s")
    print(" ".join("%13s" % h for h in hdr))
    for d in (64, 100, 128):
        for G in (64, 256):
            w = synth.niw(4000 + d + G, G, N, d=d)
            f = ctx.feature(capi.NIW).update_all(w)
            col = torch.from_numpy(w["values"]).cuda()
            u = torch.from_numpy(w["u"]).cuda()
            prior = torch.zeros(G, device="cuda")
            assign = torch.empty(N, device="cuda", dtype=torch.int32)
            scores = torch.empty((N, G), device="cuda")
            logp = torch.empty(N, device="cuda")
            rows_assign = torch.from_numpy(np.random.default_rng(d).integers(0, G, N).astype(np.int32)).cuda()
            out = torch.empty((N, d), device="cuda")
            shared = np.concatenate([[w["kappa"], w["nu"]], w["mu"], w["psi"].ravel()]).astype(np.float32)[None, :]
            t = {}
            t["score_sample"] = timed(lambda: ctx.score_sample_batch([f], [col], N, prior, u, assign))
            t["score"] = timed(lambda: ctx.score_batch([f], [col], N, None, scores))
            t["logp"] = timed(lambda: ctx.score_logp_batch([f], [col], N, prior, logp))

            def add_remove():
                ctx.add_rows_batch([f], [col], rows_assign, N)
                ctx.remove_rows_batch([f], [col], rows_assign, N)
            t["add_rows"] = timed(add_remove) / 2  # an add and the remove that restores the statistics, halved
            t["score_data"] = timed(lambda: f.score_data_grid(shared))
            t["sample_values"] = timed(lambda: ctx.sample_values_batch([f], rows_assign, N, [out], seed=1))
            Wst, bst = whitening(w)
            sc2 = torch.empty((N, G), device="cuda")

            def yard():
                for r0 in range(0, N, 32768):
                    y = col[r0:r0 + 32768] @ Wst.T - bst
                    sc2[r0:r0 + 32768] = (y * y).view(-1, G, d).sum(2)
            t["torch_fp32"] = timed(yard)
            dp = 64 if d <= 64 else 128
            gpad = (G + 128 // dp - 1) // (128 // dp) * (128 // dp)
            counted = N * G * (2.0 * d * d + 2 * d)
            issued = N * gpad * (3.0 * dp + 16) * 2 * dp
            row = [d, G] + ["%.3f" % (t[k] * 1e3) for k in hdr[2:9]]
            row += ["%.1f" % (counted / t["score"] / 1e12), "%.3f" % (counted / t["score"] / PEAK_FP16),
                    "%.1f" % (issued / t["score"] / 1e12), "%.3f" % (issued / t["score"] / PEAK_FP16),
                    "%.1f" % (counted / t["torch_fp32"] / 1e12)]
            print(" ".join("%13s" % x for x in row), flush=True)
            f.close()
            del scores, sc2, out, col
            torch.cuda.empty_cache()
    ctx.close()


if __name__ == "__main__":
    main()
