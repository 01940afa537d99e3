#!/usr/bin/env python
"""bench.py -- value-group scores/sec of the batched score_value + sample_from_scores hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload all|c2_nich|...] [--dump-outputs DIR]

A "step" is one pass of the hot path (prior + Mixture::score_value for every row x group +
sample_from_scores) over one batch of synthetic rows with frozen group statistics.

Headline (top-level keys of the ONE JSON line rank 0 prints): BASELINE.json configs[1], NormalInverseChiSq
1M rows x 1024 groups fp32; for N > 1 rows are sharded across ranks with no data-path collective (weak
scaling: every rank scores its own 1M-row shard).

`configs` (with --workload all, the default): one sub-record per remaining BASELINE shape, each with its own
ms_per_step / value / binding roofline / e2e --
  N = 1 : c1_dd (100k rows, launch-latency bound), c1_dd_steady (50M rows), c3_crosscat, c4_dpd, c5_niw
  N > 1 : c4_dpd row-sharded (weak) and c3_crosscat FEATURE-sharded (strong: the 1M x 256 x 128 table is fixed)
          in both implementations, "push" (partials stored into the owner's memory over NVLink from inside the
          score kernel) and "rs" (NCCL reduce-scatter), each with the same table timed on one GPU in the same run.
Single-feature table models (c1, c4) report the per-cell kernel as `value` (that is what the roofline measures)
and the per-value CDF shortcut (SURVEY.md 8d, the library's default for those calls) beside it, flagged.

--steps K is the step count of every timed loop: each configuration's event-timed steps and each e2e host-entry mode.
Warm-up runs max(W, 3) steps.

--dump-outputs DIR writes, after each configuration's timed steps, what its last step handed the caller (the sampled
group index of every row; with --materialise the scores, with --sweep the refreshed prior and group sizes) as
DIR/<workload>_<output>.npy in float32 (exact for the indices and sizes, which stay below 2^24).  Outputs longer than
DUMP_ROWS rows keep every (rows // DUMP_ROWS)-th row from a seeded offset; with N > 1, row-sharded outputs are rank 0's
shard.  The inputs are seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "value-group scores/sec (score_value+sample)"
UNIT = "value-group scores/s"

WORKLOADS = {
    "c1_dd": dict(model="dd", G=100, N=100_000, seed=20241, dim=16),
    "c1_dd_steady": dict(model="dd", G=100, N=50_000_000, seed=20241, dim=16),
    "c2_nich": dict(model="nich", G=1024, N=1_000_000, seed=20242),
    "c3_crosscat": dict(model="crosscat", G=128, N=1_000_000, seed=20243, n_gp=128, n_bb=128),
    "c4_dpd": dict(model="dpd", G=512, N=10_000_000, seed=20244, V=4096),
    "c5_niw": dict(model="niw", G=256, N=1_000_000, seed=20245, d=32),
    # beyond BASELINE.json (A/B harness only, --workload): the cross-cat kind with more groups than one register tile
    "x_crosscat_g256": dict(model="crosscat", G=256, N=200_000, seed=20246, n_gp=128, n_bb=128),
    "x_crosscat_g256_1m": dict(model="crosscat", G=256, N=1_000_000, seed=20246, n_gp=128, n_bb=128),
    "x_crosscat_g1024": dict(model="crosscat", G=1024, N=100_000, seed=20247, n_gp=128, n_bb=128),
}
HEADLINE = "c2_nich"
SUB_N1 = ["c1_dd", "c1_dd_steady", "c3_crosscat", "c4_dpd", "c5_niw"]

# --dump-outputs: at most 1M rows of a per-row output and 4096 rows of the [N][G] scores, 64 MB over all files
DUMP_ROWS = 1 << 20
DUMP_SCORE_ROWS = 4096
DUMP_SEED = 7
DUMP_MAX_BYTES = 64 << 20

# committed ncu --set full summaries: dram__bytes of one launch of the config's dominant kernel
NCU_SUMMARY = {
    "c2_nich": "r02_c2_nich_rows_v3_static_reference.txt",
    "c1_dd_steady": "r02_c1_dd_steady.txt",
    "c3_crosscat": "r02_c3_crosscat.txt",
    "c4_dpd": "r02_c4_dpd_table_rows_v2_staged_walk.txt",
    "c5_niw": "r02_c5_niw_fused.txt",
}


def ncu_traffic(summary):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from a committed ncu --set full summary"""
    path = os.path.join(ROOT, "profiles", summary or "")
    if not summary or not os.path.exists(path):
        return None, None
    total = 0.0
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
    for line in open(path):
        parts = line.split()
        if len(parts) >= 3 and parts[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
            total += float(parts[1]) * unit.get(parts[2], 1.0)
    return (total or None), "profiles/" + summary


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=float(p["hbm_gbs"]), bf16_tflops=float(p["bf16_tflops"]),
                    bf16_tflops_sustained=float(p.get("bf16_tflops_sustained", p["bf16_tflops"])),
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs"""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            time.sleep(0.3)  # first sample before the timed region starts
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1]))
                mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_workload(name, rank=0):
    from distributions_b200 import synth
    cfg = dict(WORKLOADS[name])
    model = cfg.pop("model")
    seed = cfg.pop("seed") + 1000 * rank
    G, N = cfg.pop("G"), cfg.pop("N")
    w = getattr(synth, model)(seed, G, N, **cfg)
    feats = w["features"] if model == "crosscat" else [w]
    return dict(name=name, G=G, N=N, feats=feats, sizes=w["sizes"], u=w["u"])


def write_outputs(outputs, out_dir):
    total = sum(a.nbytes for a in outputs.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in outputs.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def model_id(capi, name):
    return {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW}[name]


# ------------------------------------------------------------------------------------------------
def cpu_reference_arm(wl, seconds_target, threads=None):
    """The reference's own CPU path (oracle/_ref, unmodified reference code) on a bounded sample of the workload,
    all host threads; the C port where the reference cannot be compiled (NIW: Eigen is absent)."""
    from distributions_b200 import synth
    from oracle.pyoracle import Oracle, Ref
    threads = threads or os.cpu_count() or 1
    G = wl["G"]
    cols = [w["values"] for w in wl["feats"]]
    F = len(cols)
    model = wl["feats"][0]["model"]
    if model == "niw":
        o = Oracle()
        w = wl["feats"][0]
        prior = o.py_prior(synth.PY_ALPHA, synth.PY_D, wl["sizes"])

        def run_rows(rows):
            t0 = time.perf_counter()
            sc = np.tile(prior, (rows, 1)).astype(np.float32)
            o.niw_score_rows(w["mu"], w["kappa"], w["psi"], w["nu"], w["count"], w["sum_x"], w["sum_xxT"],
                             np.ascontiguousarray(w["values"][:rows]), sc)
            o.sample_rows(sc, wl["u"][:rows])
            return time.perf_counter() - t0
        probe = 256
        rate = probe / max(run_rows(probe), 1e-6)
        rows = int(min(wl["N"], max(probe, rate * seconds_target)))
        return (lambda: run_rows(rows)), rows, "port", 1
    if Ref.available():
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import cases
        r = Ref()
        k = r.kind(G, wl["sizes"], synth.PY_ALPHA, synth.PY_D)
        for w in wl["feats"]:
            cases.ref_add_feature(k, w)
        probe = min(wl["N"], max(threads * 64, 2000 // max(F, 1)))
        secs, _ = k.bench(cols, probe, threads)
        rate = probe / max(secs, 1e-6)
        rows = int(min(wl["N"], max(probe, rate * seconds_target)))
        run = lambda: k.bench(cols, rows, threads)[0]  # noqa: E731
        return run, rows, "reference", threads
    if F != 1 or model != "nich":
        raise RuntimeError("oracle/_ref is required for the CPU arm of this workload")
    o = Oracle()
    w = wl["feats"][0]
    cache = o.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])
    prior = o.py_prior(synth.PY_ALPHA, synth.PY_D, wl["sizes"])
    probe = min(wl["N"], 2000)
    secs, _ = o.bench_nich(cache, prior, w["values"][:probe], wl["u"][:probe], threads)
    rate = probe / max(secs, 1e-6)
    rows = int(min(wl["N"], max(probe, rate * seconds_target)))
    run = lambda: o.bench_nich(cache, prior, w["values"][:rows], wl["u"][:rows], threads)[0]  # noqa: E731
    return run, rows, "port", threads


def cpu_baseline_record(wl, seconds_target):
    F = len(wl["feats"])
    try:
        run, rows, kind, threads = cpu_reference_arm(wl, seconds_target=seconds_target)
        secs = run()
        return {"value": rows * F * wl["G"] / secs, "unit": UNIT, "cores": threads, "kind": kind,
                "sample": "first %d of %d rows, one pass, %d thread%s%s" % (rows, wl["N"], threads, "s" if threads > 1 else "",
                                                                           " (row shards)" if threads > 1 else "")}
    except Exception as exc:  # the baseline is a report, never a reason to lose the GPU number
        return {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": str(exc)[:200]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    name = HEADLINE if args.workload == "all" else args.workload
    wl = make_workload(name)
    F = len(wl["feats"])
    run, rows, kind, threads = cpu_reference_arm(wl, seconds_target=3.0)
    for _ in range(args.warmup):
        run()
    t = [run() for _ in range(args.steps)]
    per_step = float(np.mean(t))
    value = rows * F * wl["G"] / per_step
    sample = "first %d of %d rows per step, %d threads (row shards)" % (rows, wl["N"], threads)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": name, "rows_per_gpu": wl["N"], "groups": wl["G"], "features": F, "sample_rows_per_step": rows},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
class Peaks:
    """roofline denominators: HBM / bf16 from MEASURED_PEAKS.json, MUFU / FP32 / L2-gather measured here"""

    def __init__(self, ctx):
        self.m = measured_peaks()
        self.mufu = ctx.pipe_peak(0)
        self.fma = ctx.pipe_peak(1)
        self.l2_gather = ctx.pipe_peak(2)


def binding_roofline(name, wl, ms, peaks, cdf_shortcut=False, materialise=False):
    """SURVEY.md 8(d): t_roof = max over the resources the ALGORITHM needs per cell; frac = t_roof / t_measured."""
    G, N, F = wl["G"], wl["N"], len(wl["feats"])
    cells = float(N) * F * G
    t = ms * 1e-3
    cols_bytes = sum(w["values"].nbytes for w in wl["feats"])
    hbm_bytes = cols_bytes + 4 * N + 4 * N + (4 * N * G if materialise else 0)  # values + u in, assign out
    model = wl["feats"][0]["model"]
    if model == "dpd":
        hbm_bytes += 4 * (wl["feats"][0]["keys"].size + 1) * G
    hbm = {"bound": "hbm", "algorithmic_bytes_per_launch": int(hbm_bytes), "achieved": hbm_bytes / t / 1e9, "peak": peaks.m["hbm_gbs"],
           "unit": "GB/s", "frac": hbm_bytes / t / 1e9 / peaks.m["hbm_gbs"], "peak_source": peaks.m["source"]}
    traffic, traffic_src = ncu_traffic(NCU_SUMMARY.get(name))
    if cdf_shortcut or materialise:
        r = dict(hbm)
        r["kernel"] = ("value_guide_build_kernel + value_guide_sample_kernel (per-value CDF rows + guide tables, one thread per row)" if cdf_shortcut
                       else "score_rows_kernel (scores materialised)")
    elif model in ("dd", "nich", "dpd"):
        mufu_per_cell = 2.0 if model == "nich" else 1.0  # nich: lg2 + ex2; dd / dpd: ex2
        t_sfu = cells * mufu_per_cell / peaks.mufu
        r = {"bound": "sfu", "achieved": cells * mufu_per_cell / t / 1e9, "peak": peaks.mufu / 1e9, "unit": "G MUFU lane-ops/s",
             "frac": t_sfu / t, "mufu_per_cell": mufu_per_cell, "t_roof_ms": t_sfu * 1e3,
             "peak_source": "measured here (dist_b200_pipe_peak: register-only ex2 / lg2 chains)",
             "kernel": {"dd": "score_rows_kernel<112, dd scaled table, 128 threads>", "nich": "nich_rows2_kernel<5> (packed fp32x2, static softmax reference, four rows per thread, 5 of 16 exp2 pairs on the FMA pipe)", "dpd": "table_rows_kernel<4, staged walk, 1 of 4 quads on the FMA pipe>"}[model]}
        if model == "dpd":  # SURVEY 8(d): max(t_SFU, gathered bytes / measured L2 gather bandwidth)
            t_l2 = 4.0 * cells / peaks.l2_gather
            r["l2_gather"] = {"gathered_bytes": 4.0 * cells, "achieved_gbs": 4.0 * cells / t / 1e9, "peak_gbs": peaks.l2_gather / 1e9,
                              "t_roof_ms": t_l2 * 1e3, "frac": t_l2 / t,
                              "peak_source": "measured here (random 2 KB rows of an L2-resident 8 MB table, LDG.128)"}
            if t_l2 > t_sfu:
                r.update({"bound": "l2_gather", "achieved": 4.0 * cells / t / 1e9, "peak": peaks.l2_gather / 1e9, "unit": "GB/s",
                          "frac": t_l2 / t, "t_roof_ms": t_l2 * 1e3})
        r["hbm"] = hbm
    elif model == "niw":
        flops = cells * (2.0 * 32 * 32 + 2 * 32)  # 2 d^2 + 2 d per cell (random.hpp:182)
        peak = peaks.m["bf16_tflops"]
        r = {"bound": "tensor", "achieved": flops / t / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": flops / t / 1e12 / peak,
             "flop_per_cell": 2112, "t_roof_ms": flops / (peak * 1e12) * 1e3,
             "peak_source": peaks.m["source"] + ": dense bf16 burst; the kernel keeps fp32-level parity with split fp16 operands "
                            "(7 kind::f16 MMAs of K = 16 per 128 x 256 tile = 3.4 x the counted flops) and runs at the board's power cap "
                            "(profiles/r02_c5_power.txt)",
             "kernel": "niw_tc_fused_kernel (tcgen05 kind::f16, split fp16 operands, fused sampler)", "hbm": hbm}
        # what the tensor pipe actually executes: 5.5 MMA-equivalents of 128 x 256 x 16 per (128 rows, 8 groups) = 5 632 flop / cell
        issued = cells * 5.5 * 128 * 256 * 16 * 2 / (128.0 * 8)
        r["issued"] = {"flop_per_cell": 5632, "achieved": issued / t / 1e12, "unit": "TFLOP/s", "frac_of_peak": issued / t / 1e12 / peak,
                       "note": "fp16 MMA flops issued (hi x hi, lo x hi, hi x lo terms; the k-step over x[16..32) at N = 128); the "
                               "SURVEY 8(d) figure above counts 2 d^2 + 2 d"}
    else:  # cross-cat gp + bb: FP32 pipe per SURVEY 8(d): 10 FMA per gp cell, 1 per bb cell
        n_gp = sum(1 for w in wl["feats"] if w["model"] == "gp")
        fma_ops = float(N) * G * (10.0 * n_gp + 1.0 * (F - n_gp))
        t_fp = fma_ops / peaks.fma
        r = {"bound": "fp32", "achieved": fma_ops / t / 1e9, "peak": peaks.fma / 1e9, "unit": "G FMA lane-ops/s", "frac": t_fp / t,
             "t_roof_ms": t_fp * 1e3, "peak_source": "measured here (dist_b200_pipe_peak: register-only FFMA chains)",
             "kernel": "score_rows_kernel<128, cross-cat>",
             "kernel_limiter": "the kernel tabulates the GammaPoisson term per (group, value < 32), so a gp cell is one shared-memory "
                               "gather + FADD instead of the 10-FMA polynomial: its own limiter is one LDS wavefront per warp-cell "
                               "(N F G / 32 wavefronts at 1 / clk / SM)",
             "lds_wavefront_t_roof_ms": cells / 32.0 / (148 * 1.965e9) * 1e3, "hbm": hbm}
    r["traffic"] = traffic
    r["traffic_source"] = traffic_src
    return r


def launches_per_step(wl, cdf_shortcut=False):
    model = wl["feats"][0]["model"]
    if cdf_shortcut:
        return 2  # CDF build + per-row search
    if model == "niw":
        return 1
    return 1


class Bench:
    """one process = one GPU; times workloads through the device-pointer and the host-buffer C-ABI entries"""

    def __init__(self, args):
        import torch
        self.torch = torch
        from distributions_b200 import capi, synth
        self.capi, self.synth = capi, synth
        self.args = args
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.ctx = capi.Context(self.local_rank)
        for kv in getattr(args, "option", None) or []:  # A/B runs only: dist_b200_ctx_set_option
            k, v = kv.split("=")
            self.ctx.set_option(int(k), int(v))
        self.flush = torch.empty(256 * 1024 * 1024 // 4, device=self.dev, dtype=torch.float32)  # > 126 MB L2
        self.stream = torch.cuda.current_stream().cuda_stream
        self.peaks = Peaks(self.ctx)
        self.outputs = {}

    def keep_output(self, name, a):
        """--dump-outputs: a host copy of one output (device tensor or numpy array), rows sampled past the limit"""
        if not self.args.dump_outputs:
            return
        limit = DUMP_ROWS if a.ndim == 1 else DUMP_SCORE_ROWS
        if a.shape[0] > limit:
            stride = a.shape[0] // limit
            rows = int(np.random.default_rng(DUMP_SEED).integers(stride)) + stride * np.arange(limit)
            a = a[rows] if isinstance(a, np.ndarray) else a[self.torch.from_numpy(rows).to(a.device)]
        if not isinstance(a, np.ndarray):
            a = a.cpu().numpy()
        self.outputs[name] = a.astype(np.float32)

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.dist is not None:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([float(x)], device=self.dev, dtype=self.torch.float64)
        if self.dist is not None:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def timed(self, step, steps, warmup, flush=True, sampler=None):
        """W untimed steps, then K steps each bracketed by CUDA events on the launching stream, the L2 flushed between
        steps outside the event pairs; barrier + synchronize on both sides; ms per step = max over ranks"""
        torch = self.torch
        for _ in range(max(warmup, 3)):
            if flush:
                self.flush.zero_()
            step()
        self.barrier()
        if sampler is not None:
            sampler.start()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        self.barrier()
        t_wall = time.perf_counter()
        for s0, s1 in ev:
            if flush:
                self.flush.zero_()
            s0.record()
            step()
            s1.record()
        self.barrier()
        t_wall = time.perf_counter() - t_wall
        clocks = sampler.stop() if sampler is not None else None
        ms = self.max_over_ranks(sum(a.elapsed_time(b) for a, b in ev)) / steps
        return ms, t_wall, clocks

    def load(self, wl):
        torch, capi, ctx = self.torch, self.capi, self.ctx
        G, N = wl["G"], wl["N"]
        feats = [ctx.feature(model_id(capi, w["model"])).update_all(w) for w in wl["feats"]]
        cols_host = [np.ascontiguousarray(w["values"], dtype=capi.COLUMN_DTYPE[model_id(capi, w["model"])]) for w in wl["feats"]]
        cols = [torch.from_numpy(c).to(self.dev) for c in cols_host]
        u = torch.from_numpy(wl["u"]).to(self.dev)
        prior = torch.empty(G, device=self.dev, dtype=torch.float32)
        ctx.prior_pitman_yor(self.synth.PY_ALPHA, self.synth.PY_D, wl["sizes"], prior)
        assign = torch.empty(N, device=self.dev, dtype=torch.int32)
        return dict(feats=feats, cols_host=cols_host, cols=cols, u=u, prior=prior, assign=assign)

    def e2e(self, wl, st, steps):
        """the host-buffer C-ABI call a reference-side binding makes, H2D + D2H inside the timed region: once with the
        caller's buffers page-locked (copied from / to directly), once with plain pageable numpy arrays (staged by the
        library through its own pinned area)"""
        torch, ctx = self.torch, self.ctx
        G, N, F = wl["G"], wl["N"], len(wl["feats"])
        cells = float(N) * F * G * self.world
        prior_host = st["prior"].cpu().numpy()
        h2d = sum(c.nbytes for c in st["cols_host"]) + wl["u"].nbytes + 4 * G
        out = {}
        pins = None
        reg_ms = None
        for mode in ("pinned", "pageable", "registered"):
            if mode == "registered":
                # the same plain numpy arrays, page-locked IN PLACE once through dist_b200_host_register (what a caller
                # whose data columns live in ordinary memory does before its first sweep)
                aa = np.empty(N, np.int32)
                t0 = time.perf_counter()
                for arr in list(st["cols_host"]) + [wl["u"], aa]:
                    ctx.host_register(arr)
                reg_ms = (time.perf_counter() - t0) * 1e3
                cols, uu = st["cols_host"], wl["u"]
            elif mode == "pinned":
                pins = ([torch.from_numpy(c).pin_memory() for c in st["cols_host"]], torch.from_numpy(wl["u"]).pin_memory(),
                        torch.empty(N, dtype=torch.int32).pin_memory())
                cols, uu, aa = [c.numpy() for c in pins[0]], pins[1].numpy(), pins[2].numpy()
            else:
                pins = None
                cols, uu, aa = st["cols_host"], wl["u"], np.empty(N, np.int32)
            ctx.score_sample_batch_host(st["feats"], cols, prior_host, uu, assign_out=aa)  # warm (staging alloc)
            self.barrier()
            t0 = time.perf_counter()
            for _ in range(steps):
                a_host, _ = ctx.score_sample_batch_host(st["feats"], cols, prior_host, uu, assign_out=aa)
            self.barrier()
            dt = self.max_over_ranks((time.perf_counter() - t0) / steps)
            out[mode] = (cells / dt, np.array(a_host, copy=True))
            if mode == "registered":
                for arr in list(st["cols_host"]) + [wl["u"], aa]:
                    ctx.host_unregister(arr)
        e2e = {"value": out["pinned"][0], "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(4 * N),
               "buffers": "caller's buffers page-locked (torch pin_memory)",
               "pageable": {"value": out["pageable"][0], "unit": UNIT,
                            "buffers": "plain numpy arrays, staged through the library's pinned area (memcpy + H2D)"},
               "registered": {"value": out["registered"][0], "unit": UNIT, "register_ms_once": reg_ms,
                              "matches_pinned": bool(np.array_equal(out["registered"][1], out["pinned"][1])),
                              "buffers": "the same plain numpy arrays page-locked in place once (dist_b200_host_register), then zero-copy"}}
        return e2e, out["pinned"][1], out["pageable"][1]

    # ---- one configuration, rows sharded over the ranks (weak scaling; N = 1: the whole configuration) ----------
    def run_rows(self, name, steps, warmup, sampler=None, with_cpu=False, with_e2e=True):
        torch, ctx, capi = self.torch, self.ctx, self.capi
        args = self.args
        wl = make_workload(name, self.rank)
        G, N, F = wl["G"], wl["N"], len(wl["feats"])
        st = self.load(wl)
        model = wl["feats"][0]["model"]
        table_model = F == 1 and model in ("dd", "dpd")
        scores_buf = torch.empty((N, G), device=self.dev, dtype=torch.float32) if (args.materialise and name == HEADLINE) else None
        flush = N * 12 < 200e6  # inputs of the big configurations exceed the L2 on their own

        sweep = args.sweep and name == HEADLINE
        base_sizes = torch.from_numpy(wl["sizes"].astype(np.int32)).to(self.dev)
        sizes_dev = base_sizes.clone()
        in_groups = [False]

        def step():
            # --sweep: one blocked Gibbs pass over the rows, all on the device -- the rows leave their groups
            # (remove_value), are scored against the rest and resampled, join their new groups (add_value), and the
            # clustering prior is refreshed from the new group sizes
            if sweep and in_groups[0]:
                ctx.remove_rows_batch(st["feats"], st["cols"], st["assign"], N, stream=self.stream)
            ctx.score_sample_batch(st["feats"], st["cols"], N, st["prior"], st["u"], st["assign"], scores_buf, stream=self.stream)
            if sweep:
                ctx.add_rows_batch(st["feats"], st["cols"], st["assign"], N, stream=self.stream)
                sizes_dev.copy_(base_sizes)
                ctx.count_assignments(st["assign"], N, G, sizes_dev, accumulate=True, stream=self.stream)
                ctx.prior_pitman_yor_dev(self.synth.PY_ALPHA, self.synth.PY_D, G, sizes_dev, st["prior"], stream=self.stream)
                in_groups[0] = True

        cells = float(N) * F * G * self.world
        rec = {"workload": name, "rows_per_gpu": N, "groups": G, "features": F, "steps": steps,
               "l2": "flushed between timed steps (256 MB memset outside the event pairs)" if flush else
                     "inputs (%d MB per step) exceed the 126 MB L2" % ((sum(c.nbytes for c in st["cols_host"]) + 8 * N) >> 20)}
        if table_model:
            # per-cell kernel = the measured roofline; the library default (per-value CDF trees) beside it, flagged
            ctx.set_option(capi.OPT_VALUE_CDF, 1)
            ms, t_wall, clocks = self.timed(step, steps, warmup, flush, sampler)
            a_cell = st["assign"].cpu().numpy()
            self.keep_output(name + "_assign", a_cell)
            ctx.set_option(capi.OPT_VALUE_CDF, 0)
            ms_cdf, _, _ = self.timed(step, steps, warmup, flush)
            a_cdf = st["assign"].cpu().numpy()
            self.keep_output(name + "_cdf_assign", a_cdf)
            rec["value_cdf_shortcut"] = {
                "flag": "ALGORITHMIC SHORTCUT (SURVEY.md 8d): one table feature with frozen statistics -- the likelihood vector is "
                        "evaluated once per distinct VALUE, rows only search per-value CDF trees; N G / t is still reported. This is "
                        "the library's default for such calls (DIST_B200_OPT_VALUE_CDF)",
                "ms_per_step": ms_cdf, "value": cells / (ms_cdf * 1e-3),
                "roofline": binding_roofline(name, wl, ms_cdf, self.peaks, cdf_shortcut=True),
                "index_agreement_with_per_cell_kernel": float(np.mean(a_cell == a_cdf)), "gpu_launches_per_step": 2}
        else:
            ms, t_wall, clocks = self.timed(step, steps, warmup, flush, sampler)
            self.keep_output(name + "_assign", st["assign"])
            if scores_buf is not None:
                self.keep_output(name + "_scores", scores_buf)
            if sweep:
                self.keep_output(name + "_prior", st["prior"])
                self.keep_output(name + "_group_sizes", sizes_dev)
        rec.update({"ms_per_step": ms, "value": cells / (ms * 1e-3), "wall_s_timed_region": t_wall,
                    "roofline": binding_roofline(name, wl, ms, self.peaks, materialise=scores_buf is not None),
                    "gpu_launches_per_step": launches_per_step(wl)})
        if table_model:
            ctx.set_option(capi.OPT_VALUE_CDF, 1)  # e2e below through the same per-cell kernel as `value`
        if with_e2e and not sweep:
            a_dev = None
            step()
            torch.cuda.synchronize()
            a_dev = st["assign"].cpu().numpy()
            e2e, a_pin, a_page = self.e2e(wl, st, steps)
            rec["e2e"] = e2e
            rec["e2e_matches_device_assign"] = bool(np.array_equal(a_pin, a_dev) and np.array_equal(a_page, a_dev))
        if table_model:
            ctx.set_option(capi.OPT_VALUE_CDF, 0)
        if with_cpu and self.world == 1 and self.rank == 0:
            rec["cpu_baseline"] = cpu_baseline_record(wl, 12.0 if name == HEADLINE else 3.0)
        self.last_assign = st["assign"].cpu().numpy() if not sweep else None  # parity self-checks of the multi-GPU records
        del st, scores_buf
        torch.cuda.empty_cache()
        return rec, clocks

    # ---- c3 at N > 1: the features of one cross-cat kind sharded over the ranks (strong scaling) -----------------
    def run_feature_sharded(self, name, steps, warmup, mode, row_shards=1):
        """mode "push": NVLink peer push (row_shards > 1: the feature x row hybrid); "rs": NCCL reduce-scatter"""
        torch, ctx, capi = self.torch, self.ctx, self.capi
        from distributions_b200 import sharding
        wl = make_workload(name, 0)  # the same table on every rank; each rank keeps its (features, rows) block
        G, N, F = wl["G"], wl["N"], len(wl["feats"])
        peer = sharding.PeerFeatureShards(ctx, N, G, row_shards=row_shards) if mode == "push" else None
        mine = peer.features(F) if peer else sharding.feature_shard(F, self.rank, self.world)
        r0, r1 = peer.rows() if peer else (0, N)
        feats = [ctx.feature(model_id(capi, wl["feats"][f]["model"])).update_all(wl["feats"][f]) for f in mine]
        cols = [torch.from_numpy(np.ascontiguousarray(wl["feats"][f]["values"][r0:r1],
                                                      dtype=capi.COLUMN_DTYPE[model_id(capi, wl["feats"][f]["model"])])).to(self.dev)
                for f in mine]
        u = torch.from_numpy(wl["u"]).to(self.dev)
        prior = torch.empty(G, device=self.dev, dtype=torch.float32)
        ctx.prior_pitman_yor(self.synth.PY_ALPHA, self.synth.PY_D, wl["sizes"], prior)
        comm = torch.cuda.Stream(device=self.dev)
        launches = [0]

        def score_partial(lo, hi, out):
            ctx.score_batch(feats, [c[lo:hi] for c in cols], hi - lo, prior if self.rank == 0 else None, out, stream=self.stream)
            launches[0] += 1

        def sample_block(scores, ub, out):
            ctx.sample_from_scores(scores, scores.shape[0], G, ub, out, stream=self.stream)
            launches[0] += 1

        lo_own, hi_own = peer.owned() if peer else (0, 0)
        assign_own = torch.empty(max(hi_own - lo_own, 1), device=self.dev, dtype=torch.int32)
        u_own = u[lo_own:hi_own]

        def step():
            if peer is not None:
                launches[0] += peer.launches_per_step
                return peer.step(feats, cols, prior, u_own, assign_own, stream=self.stream)
            return sharding.feature_sharded_score_sample(score_partial, sample_block, N, G, u, self.dev, tile_rows=self.args.tile_rows,
                                                         comm_stream=comm)

        ms, t_wall, _ = self.timed(step, steps, warmup, flush=False)
        launches[0] = 0
        out = step()
        self.barrier()
        per_step = launches[0]
        # parity self-check (the driver's multi-GPU run executes it): the whole job's assignment vector, every rank's rows
        # filled in, all-reduced -- compared with the single-GPU result of the same table by the caller
        torch.cuda.synchronize()
        full = torch.full((N,), -1, device=self.dev, dtype=torch.int32)
        if peer is not None:
            lo, hi = out
            if hi > lo:
                full[lo:hi] = assign_own[:hi - lo]
        else:
            assigns, rows = out
            for a_t, (lo, hi) in zip(assigns, rows):
                full[lo:hi] = a_t
        torch.cuda.synchronize()
        self.dist.all_reduce(full, op=self.dist.ReduceOp.MAX)
        self.last_full_assign = full.cpu().numpy()
        fs = peer.fs if peer else self.world
        if peer is not None:
            peer.close()
        cells = float(N) * F * G
        rows_group = r1 - r0
        rec = {"workload": name, "rows": N, "groups": G, "features": F, "features_per_rank": len(mine), "rows_per_group": rows_group,
               "feature_shards": fs, "row_shards": self.world // fs, "steps": steps,
               "scaling": "strong", "ms_per_step": ms, "value": cells / (ms * 1e-3), "gpu_launches_per_step": per_step,
               "parallelism": ("feature shards" + (" x row shards (hybrid)" if fs != self.world else "") +
                               "; partial rows stored into the owning rank's memory over NVLink from inside the score kernel "
                               "(16-byte stores), device-side epoch flags instead of host barriers, the owner samples the "
                               "fixed-order sum of its slots" if mode == "push" else
                               "feature shards + NCCL reduce-scatter(sum) of [rows][G] partials, tiles of %d rows overlapped on a "
                               "second stream" % self.args.tile_rows),
               "nvlink_bytes_per_step_per_rank": int(4 * rows_group * G * (fs - 1) / fs),
               "l2": "inputs (640 MB of columns + 512 MB of partial scores per step over the ranks) exceed the 126 MB L2"}
        del feats, cols
        torch.cuda.empty_cache()
        return rec


def run_b200(args):
    b = Bench(args)
    torch = b.torch
    if args.feature_sharded and b.world > 1:
        r = b.run_feature_sharded("c3_crosscat", args.steps, args.warmup, "rs" if args.feature_sharded == "rs" else "push", args.row_shards)
        b.keep_output("c3_crosscat_feature_sharded_%s_assign" % args.feature_sharded, b.last_full_assign)
        if b.rank == 0:
            print(json.dumps(r))
            if args.dump_outputs:
                write_outputs(b.outputs, args.dump_outputs)
        b.dist.destroy_process_group()
        return 0
    headline = HEADLINE if args.workload == "all" else args.workload
    sampler = ClockSampler(b.local_rank) if b.rank == 0 else None
    rec, clocks = b.run_rows(headline, args.steps, args.warmup, sampler=sampler, with_cpu=not args.no_cpu)
    configs = {}
    if args.workload == "all":
        if b.world == 1:
            for name in SUB_N1:
                r, _ = b.run_rows(name, args.steps, args.warmup, with_cpu=not args.no_cpu)
                configs[name] = r
        else:
            r, _ = b.run_rows("c4_dpd", args.steps, args.warmup, with_e2e=False)
            r["scaling"] = "weak"
            r["parallelism"] = "row shards: caches and prior replicated, every rank scores its own 10M-row shard, no collective"
            configs["c4_dpd_row_sharded"] = r
            variants = [("push", "push", 1), ("rs", "rs", 1)]
            if b.world >= 4:  # feature x row hybrid: 2 feature shards, world / 2 row shards
                variants.append(("hybrid_2x%d" % (b.world // 2), "push", b.world // 2))
            full_assign = {}
            for label, mode, row_shards in variants:
                configs["c3_crosscat_feature_sharded_" + label] = b.run_feature_sharded("c3_crosscat", args.steps, args.warmup, mode, row_shards)
                full_assign[label] = b.last_full_assign
                b.keep_output("c3_crosscat_feature_sharded_%s_assign" % label, b.last_full_assign)
            # the same table on ONE GPU in the same run (rank 0 only, the others wait): the strong-scaling reference
            t1 = torch.zeros(1, device=b.dev, dtype=torch.float64)
            if b.rank == 0:
                world, b.world, dist, b.dist = b.world, 1, b.dist, None
                r1, _ = b.run_rows("c3_crosscat", args.steps, args.warmup, with_e2e=False)
                b.world, b.dist = world, dist
                t1[0] = r1["ms_per_step"]
                for label, _, _ in variants:
                    got = full_assign[label]
                    configs["c3_crosscat_feature_sharded_" + label]["parity_self_check"] = {
                        "rows_assigned": int((got >= 0).sum()), "rows": int(got.size),
                        "index_agreement_with_single_gpu": float(np.mean(got == b.last_assign)),
                        "note": "the partial sums are associated differently from the single-GPU sum: every mismatch is a "
                                "near-tie (tests/test_multigpu.py asserts that against the oracle at 2 / 4 / 8 GPUs)"}
            b.barrier()
            b.dist.broadcast(t1, 0)
            for label, _, _ in variants:
                r = configs["c3_crosscat_feature_sharded_" + label]
                r["single_gpu_ms_same_run"] = float(t1.item())
                r["strong_scaling_efficiency"] = float(t1.item()) / (b.world * r["ms_per_step"])
    if b.rank != 0:
        if b.dist is not None:
            b.dist.destroy_process_group()
        return 0

    roof = rec.pop("roofline")
    e2e = rec.pop("e2e", None)
    cpu = rec.pop("cpu_baseline", None)
    line = {
        "metric": METRIC, "value": rec["value"], "unit": UNIT, "n_gpus": b.world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": headline, "rows_per_gpu": rec["rows_per_gpu"], "groups": rec["groups"], "features": rec["features"],
                   "l2": rec["l2"],
                   "mode": ("score+prior+sample with the [N][G] scores also written to HBM" if args.materialise else
                            "fused score+prior+sample, scores not materialised") +
                           (" + batched remove_value / add_value, cache rebuild and prior refresh on the device "
                            "(one blocked Gibbs pass per step)" if args.sweep else ""),
                   "wall_s_timed_region": rec["wall_s_timed_region"], "e2e_matches_device_assign": rec.get("e2e_matches_device_assign")},
        "clocks": clocks, "e2e": e2e, "gpu_launches": args.steps * rec["gpu_launches_per_step"],
        "roofline": roof, "cpu_baseline": cpu,
    }
    if "value_cdf_shortcut" in rec:
        line["value_cdf_shortcut"] = rec["value_cdf_shortcut"]
    if configs:
        line["configs"] = configs
    print(json.dumps(line))
    if args.dump_outputs:
        write_outputs(b.outputs, args.dump_outputs)
    if b.dist is not None:
        b.dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all"] + sorted(WORKLOADS),
                    help="all (default): headline c2_nich + one sub-record per remaining BASELINE shape; or one shape alone")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--materialise", action="store_true", help="headline: also write the [N][G] log scores (HBM-write-bound mode)")
    ap.add_argument("--sweep", action="store_true",
                    help="headline: each step is a blocked Gibbs pass on the device: remove_value, score+sample, add_value, cache / prior refresh")
    ap.add_argument("--feature-sharded", default=None, choices=["push", "rs"],
                    help="N > 1 only: time just c3_crosscat feature-sharded in this mode (development runs)")
    ap.add_argument("--row-shards", type=int, default=1, help="with --feature-sharded push: feature x row hybrid")
    ap.add_argument("--tile-rows", type=int, default=65536, help="row tile of the feature-sharded reduce-scatter")
    ap.add_argument("--option", action="append", metavar="K=V", help="A/B runs: dist_b200_ctx_set_option(K, V) before anything runs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each configuration's last step computed as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
