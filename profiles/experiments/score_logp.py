"""Row log-likelihood (dist_b200_score_logp_batch) at the bench shapes, against what a user has without it.

For each shape (bench.py's workloads: c1-steady dd16 G=100 x 5e7 rows, c2 nich 1M x 1024, c3 cross-cat 1M x 256 features x
128 groups, c4 dpd V=4096 G=512 x 1e7, c5 niw d=32 G=256 x 1M) it times, with the Pitman-Yor prior:
  logp       score_logp_batch with the default routes (c1 / c4: the per-value table; c2: nich_logp_kernel; c3: score_rows
             logp mode; c5: materialise + logp_scores_kernel)
  logp_cell  score_logp_batch with DIST_B200_OPT_VALUE_CDF = 1 (c1: score_rows logp mode; c4: materialise + reduce)
  sample     score_sample_batch on the same rows (its default route)
  baseline   score_batch into [N][G] followed by torch.logsumexp (what a caller has to do without the entry)
CUDA events around each call, the L2 flushed (256 MB written) before each, median of 7 after 2 warm-ups.  For the fused
routes the fraction of the MUFU roofline (cells x MUFU ops per cell over dist_b200_pipe_peak(0)); for the per-value route
the fraction of the HBM bound over the bytes it moves (value + logp per row, plus the table build).  The card name, power
limit and max SM clock are read in the same run.  Run on a B200:
    python profiles/experiments/score_logp.py > profiles/experiments/score_logp.txt
"""
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from distributions_b200 import capi  # noqa: E402

HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU
SHAPES = [("c1", "c1_dd_steady"), ("c2", "c2_nich"), ("c3", "c3_crosscat"), ("c4", "c4_dpd"), ("c5", "c5_niw")]
MID = {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW}
FLUSH = torch.empty(256 * 1024 * 1024 // 4, device="cuda", dtype=torch.float32)


def timed(step, reps=7, warm=2):
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
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ctx = capi.Context(0)
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    mufu = ctx.pipe_peak(0)
    print("device: %s | power limit, max SM clock: %s | MUFU lane-ops/s (measured): %.3g" % (name, q, mufu))
    print("%-4s %-10s %10s  %s" % ("shape", "route", "ms/call", "roofline"))
    for label, wname in SHAPES:
        wl = bench.make_workload(wname)
        G, N, ws = wl["G"], wl["N"], wl["feats"]
        feats = [ctx.feature(MID[w["model"]]).update_all(w) for w in ws]
        cols = [torch.from_numpy(np.ascontiguousarray(w["values"].astype(capi.COLUMN_DTYPE[MID[w["model"]]]))).cuda() for w in ws]
        prior = torch.from_numpy(ctx.prior_pitman_yor_host(1.0, 0.1, np.asarray(wl["sizes"], np.int32))).cuda()
        u = torch.from_numpy(wl["u"]).cuda()
        logp = torch.empty(N, device="cuda", dtype=torch.float32)
        assign = torch.empty(N, device="cuda", dtype=torch.int32)
        model = ws[0]["model"]
        cells = float(N) * G

        def roof_mufu(ms, per_cell):
            return "MUFU %.0f%% (%.1f MUFU ops / cell)" % (100 * cells * per_cell / mufu / (ms * 1e-3), per_cell)

        t = timed(lambda: ctx.score_logp_batch(feats, cols, N, prior, logp))
        if model in ("dd", "dpd"):
            R = ws[0]["counts"].shape[1] + (1 if model == "dpd" else 0)
            nbytes = N * (4 + 4) + 4 * R * G
            roof = "HBM %.1f%% (%.3g B moved)" % (100 * nbytes / HBM_BYTES_PER_S / (t * 1e-3), nbytes)
        elif model == "nich":
            roof = roof_mufu(t, 2.0)
        elif model == "niw":
            roof = "materialised [N][G] (not a fused route)"
        else:
            roof = roof_mufu(t, 1.0)
        print("%-4s %-10s %10.3f  %s" % (label, "logp", t, roof))
        if model in ("dd", "dpd"):
            ctx.set_option(0, 1)
            t = timed(lambda: ctx.score_logp_batch(feats, cols, N, prior, logp))
            ctx.set_option(0, 0)
            print("%-4s %-10s %10.3f  %s" % (label, "logp_cell", t, roof_mufu(t, 1.0) if model == "dd" else "materialised [N][G]"))
        t = timed(lambda: ctx.score_sample_batch(feats, cols, N, prior, u, assign))
        print("%-4s %-10s %10.3f" % (label, "sample", t))
        scores = torch.empty((N, G), device="cuda", dtype=torch.float32)

        def baseline():
            ctx.score_batch(feats, cols, N, prior, scores)
            torch.logsumexp(scores, dim=1, out=logp)

        t = timed(baseline)
        print("%-4s %-10s %10.3f" % (label, "baseline", t))
        del scores, logp, assign, cols, u, prior
        for f in feats:
            f.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
