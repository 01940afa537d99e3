"""Missing cells (the *_masked entries) at the bench shapes, against the unmasked entries on the same data.

Shapes (bench.py workloads): c3 cross-cat 1M rows x 256 features x 128 groups, the same list at G = 256 (the kSub kernel),
c2 nich 1M x 1024 (masked: the feature-list kernel with a list of one, unmasked: nich_rows2_kernel), c4 dpd (masked: the
generic route, one extra [N][G] pass), and an add + remove of the c3 rows.  Each masked shape runs with all-ones words
(masked, nothing missing) and at 10 % and 50 % missing cells per feature.  score_sample_batch unless noted; CUDA events,
the L2 flushed (256 MB written) before each call, median of 7 after 2 warm-ups.  The card name, power limit and max SM
clock are read in the same run.  Run on a B200:
    python profiles/experiments/missing_cells.py > profiles/experiments/missing_cells.txt
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

MID = {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW, "bnb": capi.BNB}
FLUSH = torch.empty(256 * 1024 * 1024 // 4, device="cuda", dtype=torch.float32)
HBM_BYTES_PER_S = 7.7e12  # HGX B200 data sheet, one GPU


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


def words(N, F, rate, seed):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(F):
        obs = np.ones(N, bool) if rate == 0 else rng.random(N) >= rate
        out.append(torch.from_numpy(capi.pack_observed(obs).view(np.int32)).cuda())
    return out


def main():
    ctx = capi.Context(0)
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    mufu = ctx.pipe_peak(0)
    print("device: %s | power limit, max SM clock: %s | MUFU lane-ops/s (measured): %.3g" % (name, q, mufu))
    print("%-12s %-22s %10s %8s  %s" % ("shape", "call", "ms/call", "x unmasked", "roofline"))
    for label, wname, G in [("c3", "c3_crosscat", None), ("c3 G=256", "c3_crosscat", 256), ("c2", "c2_nich", None),
                            ("c4", "c4_dpd", None)]:
        wl = bench.make_workload(wname)
        N, ws = wl["N"], wl["feats"]
        if G is not None:  # the same list with more groups: the caches stream, the sampler takes the kSub kernel
            from distributions_b200 import synth
            ws = [getattr(synth, w["model"])(500 + i, G, N, **({"dim": w["counts"].shape[1]} if w["model"] == "dd" else {}))
                  for i, w in enumerate(ws)]
            for w in ws[1:]:
                w["sizes"] = ws[0]["sizes"]
            sizes = ws[0]["sizes"]
        else:
            G, sizes = wl["G"], wl["sizes"]
        feats = [ctx.feature(MID[w["model"]]).update_all(w) for w in ws]
        cols = [torch.from_numpy(np.ascontiguousarray(w["values"].astype(capi.COLUMN_DTYPE[MID[w["model"]]]))).cuda() for w in ws]
        prior = torch.from_numpy(ctx.prior_pitman_yor_host(1.0, 0.1, np.asarray(sizes, np.int32))).cuda()
        u = torch.from_numpy(np.random.default_rng(1).random(N).astype(np.float32)).cuda()
        assign = torch.empty(N, device="cuda", dtype=torch.int32)
        cells = float(N) * G * len(ws)
        t0 = timed(lambda: ctx.score_sample_batch(feats, cols, N, prior, u, assign))
        ref = assign.clone()
        if label == "c4":  # the masked form materialises [N][G] three times: dpd scores, masked add, sampler read
            nbytes = 4.0 * N * G * 5
            roof = "masked: HBM bound %.2f ms (%.3g B: 2 [N][G] writes, 3 reads)" % (nbytes / HBM_BYTES_PER_S * 1e3, nbytes)
        elif label == "c2":
            roof = "MUFU %.0f%% at 1 op / cell" % (100 * cells / mufu / (t0 * 1e-3))
        else:
            roof = "not MUFU-bound: one cache gather per cell and feature"
        print("%-12s %-22s %10.3f %8s  %s" % (label, "unmasked", t0, "1.00", roof))
        for rate in (0.0, 0.1, 0.5):
            m = words(N, len(ws), rate, 7)
            t = timed(lambda: ctx.score_sample_batch(feats, cols, N, prior, u, assign, observed=m))
            extra = ""
            if rate == 0.0:
                extra = "draws equal to unmasked: %.5f" % (assign == ref).float().mean().item()
            print("%-12s %-22s %10.3f %8.2f  %s" % (label, "masked, %d%% missing" % int(100 * rate), t, t / t0, extra))
            del m
        if label == "c3":
            assign_rows = torch.from_numpy(np.random.default_rng(2).integers(0, G, N).astype(np.int32)).cuda()
            t0 = timed(lambda: (ctx.add_rows_batch(feats, cols, assign_rows, N), ctx.remove_rows_batch(feats, cols, assign_rows, N)))
            nbytes = 2 * sum(c.numel() * c.element_size() + 4 * N for c in cols)
            print("%-12s %-22s %10.3f %8s  HBM %.0f%% (%.3g B: columns + assign, twice)" %
                  (label, "add+remove unmasked", t0, "1.00", 100 * nbytes / HBM_BYTES_PER_S / (t0 * 1e-3), nbytes))
            for rate in (0.0, 0.1, 0.5):
                m = words(N, len(ws), rate, 8)
                t = timed(lambda: (ctx.add_rows_batch(feats, cols, assign_rows, N, observed=m),
                                   ctx.remove_rows_batch(feats, cols, assign_rows, N, observed=m)))
                print("%-12s %-22s %10.3f %8.2f" % (label, "add+remove %d%% missing" % int(100 * rate), t, t / t0))
                del m
        del cols, u, prior, assign
        for f in feats:
            f.close()
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
