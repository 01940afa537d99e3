"""Cost of dist_b200_regroup_batch (group births and deaths) at the bench shapes, and of a blocked Gibbs sweep that uses
it against the same sweep at fixed G.

Shapes: c2 nich 1M rows x 1024 groups; c3 256 features (128 gp + 128 bb) x 128 groups, 1M rows; c4 dpd V = 4096 x 512
groups, 1M rows; c5 niw d = 32 x 256 groups, 256K rows.  Every feature starts from zero statistics with its rows added on
the device, so statistics and assignments agree.  A regroup is timed in steady state: 10 % of the groups (fixed
positions) have size 0 and n_empty equals their number, so G stays the same from call to call and every call moves
the same bytes.

Per shape:
  - wall: host clock around the call, which returns after its one readback of K+ and with the copy-back and cache
    rebuild enqueued, plus a device synchronise (median of 20 after 3 warm-ups);
  - the device time of each kernel family from torch.profiler (CUDA activities, a separate run of 20 calls, per call):
    remap (one block), relabel, arrays (gathers + copy-backs), rebuild (the prep kernels of the fresh groups, the dpd
    table, the niw tensor-core images), and the 4-byte D2H copy;
  - host: wall minus the device time, i.e. launch overhead plus the readback round trip.
Sweep (c2): 8 blocks, one pass over all rows.  "fixed G": remove rows, count, Pitman-Yor prior, score + sample, add
rows per block (what the library could do before regroup_batch).  "regroup": the same with regroup_batch between the
count and the prior (distributions_b200.gibbs.BlockedGibbs).  The two alternate, median of 7 sweeps each after 2
warm-ups.  The card name, power limit and max SM clock are read in the same run.  Run on a B200:
    python profiles/experiments/regroup.py > profiles/experiments/regroup.txt
"""
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from distributions_b200 import capi, gibbs, models  # noqa: E402


def zero_workload(name, G, **kw):
    if name == "nich":
        return dict(shared=np.array([0, 1, 1, 1], np.float32), count=np.zeros(G, np.int32), mean=np.zeros(G, np.float32),
                    ctv=np.zeros(G, np.float32))
    if name == "gp":
        return dict(shared=np.array([1, 1], np.float32), count=np.zeros(G, np.uint32), sum=np.zeros(G, np.uint32))
    if name == "bb":
        return dict(shared=np.array([0.5, 2], np.float32), heads=np.zeros(G, np.int32), tails=np.zeros(G, np.int32))
    if name == "dpd":
        V = kw["V"]
        return dict(keys=np.arange(V, dtype=np.uint32), betas=np.full(V, 0.9 / V, np.float32), alpha=0.5, beta0=0.1,
                    counts=np.zeros((G, V), np.int32))
    d = kw["d"]
    return dict(mu=np.zeros(d, np.float32), kappa=1.0, psi=np.eye(d, dtype=np.float32), nu=float(d + 1), count=np.zeros(G, np.int32),
                sum_x=np.zeros((G, d), np.float32), sum_xxT=np.zeros((G, d, d), np.float32))


def column(name, rng, N, **kw):
    if name == "nich":
        return rng.standard_normal(N).astype(np.float32)
    if name == "gp":
        return rng.poisson(3.0, N).astype(np.uint32)
    if name == "bb":
        return (rng.random(N) < 0.3).astype(np.uint8)
    if name == "dpd":
        return rng.integers(0, kw["V"], N).astype(np.uint32)
    return rng.standard_normal((N, kw["d"])).astype(np.float32)


def build(ctx, specs, G, N, seed):
    rng = np.random.default_rng(seed)
    feats, cols = [], []
    for name, kw in specs:
        feats.append(ctx.feature(getattr(capi, name.upper())).update_all(zero_workload(name, G, **kw)))
        cols.append(torch.from_numpy(column(name, rng, N, **kw)).cuda())
    assign = torch.from_numpy(rng.integers(0, G, N).astype(np.int32)).cuda()
    ctx.add_rows_batch(feats, cols, assign, N)
    torch.cuda.synchronize()
    return feats, cols, assign


SHAPES = [("c2", [("nich", {})], 1024, 1 << 20),
          ("c3", [("gp", {})] * 128 + [("bb", {})] * 128, 128, 1 << 20),
          ("c4", [("dpd", dict(V=4096))], 512, 1 << 20),
          ("c5", [("niw", dict(d=32))], 256, 1 << 18)]
FAMILIES = ("regroup_remap", "regroup_relabel", "regroup_arrays")


def regroup_cost(ctx, tag, specs, G, N):
    feats, cols, assign = build(ctx, specs, G, N, 1)
    rng = np.random.default_rng(2)
    sizes = np.ones(G, np.int32)
    dead = rng.choice(G, G // 10, replace=False)
    sizes[dead] = 0
    counts = torch.from_numpy(sizes).cuda()
    n_empty = dead.size

    def call():
        assert ctx.regroup_batch(feats, counts, G, n_empty, assign, N) == G

    for _ in range(3):
        call()
    torch.cuda.synchronize()
    walls = []
    for _ in range(20):
        t0 = time.perf_counter()
        call()
        torch.cuda.synchronize()
        walls.append(time.perf_counter() - t0)
    wall = float(np.median(walls)) * 1e3
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(20):
            call()
        torch.cuda.synchronize()
    dev = {k: 0.0 for k in FAMILIES + ("rebuild", "readback")}
    for e in prof.key_averages():
        t = e.device_time_total if hasattr(e, "device_time_total") else e.cuda_time_total
        if t <= 0:
            continue
        key = next((k for k in FAMILIES if k in e.key), None)
        if key is None:
            key = "readback" if "DtoH" in e.key or "Device -> Pageable" in e.key or "Memcpy" in e.key else "rebuild"
        dev[key] += t / 20 / 1e3  # us -> ms per call
    total_dev = sum(dev.values())
    print("%-4s F=%-3d G=%-5d N=%-8d wall %7.3f ms | remap %.4f relabel %.4f arrays %.4f rebuild %.4f D2H %.4f | host %.3f ms"
          % (tag, len(specs), G, N, wall, dev["regroup_remap"], dev["regroup_relabel"], dev["regroup_arrays"], dev["rebuild"],
             dev["readback"], wall - total_dev))
    for f in feats:
        f.close()


def sweep_compare(ctx):
    G, N, n_blocks = 1024, 1 << 20, 8
    feats, cols, assign = build(ctx, [("nich", {})], G, N, 3)
    prior_model = models.PitmanYor(1.0, 0.1)
    kind = gibbs.BlockedGibbs(ctx, feats, cols, assign, prior_model, n_empty=1)
    gen = torch.Generator(device="cuda").manual_seed(0)
    counts = torch.zeros(4 * G, device="cuda", dtype=torch.int32)
    prior = torch.zeros(4 * G, device="cuda", dtype=torch.float32)

    def fixed():  # the same blocks at fixed G: no births, no deaths
        Gf = kind.G
        for r0, r1 in kind.blocks(n_blocks):
            n = r1 - r0
            ids = assign[r0:r1]
            ctx.remove_rows_batch(feats, [c[r0:r1] for c in cols], ids, n)
            ids.fill_(-1)
            ctx.count_assignments(assign, N, Gf, counts)
            ctx.prior_pitman_yor_dev(prior_model.alpha, prior_model.d, Gf, counts, prior)
            u = torch.rand(n, generator=gen, device="cuda")
            ctx.score_sample_batch(feats, [c[r0:r1] for c in cols], n, prior, u, ids)
            ctx.add_rows_batch(feats, [c[r0:r1] for c in cols], ids, n)

    def births():
        kind.sweep(n_blocks, gen)

    def timed(fn):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        return (time.perf_counter() - t0) * 1e3

    for _ in range(2):
        timed(fixed)
        timed(births)
    a, b = [], []
    for _ in range(7):
        a.append(timed(fixed))
        b.append(timed(births))
    print("sweep c2 (nich 1M rows, %d blocks): fixed G %.3f ms | regroup %.3f ms (G after: %d) | ratio %.3f"
          % (n_blocks, np.median(a), np.median(b), kind.G, np.median(b) / np.median(a)))
    feats[0].close()


def main():
    ctx = capi.Context(0)
    name = torch.cuda.get_device_name(0)
    q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True).stdout.strip()
    print("device: %s | power limit, max SM clock: %s" % (name, q))
    print("regroup_batch per call (steady state: 10 % of the groups die, as many are born)")
    for tag, specs, G, N in SHAPES:
        regroup_cost(ctx, tag, specs, G, N)
    sweep_compare(ctx)
    ctx.close()


if __name__ == "__main__":
    main()
