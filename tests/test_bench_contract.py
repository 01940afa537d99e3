"""The JSON line bench.py prints is a contract with the driver: check the committed lines of the last GPU run
(profiles/r01_bench) and a live run of the CPU reference arm against it."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _line(name):
    with open(os.path.join(ROOT, "profiles", "r01_bench", name)) as fh:
        return json.loads(fh.read().strip().splitlines()[-1])


def test_headline_line_has_every_contract_key():
    d = _line("c2_nich.json")
    baseline = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert BASE_KEYS | {"roofline", "clocks"} <= set(d)
    assert d["config"]["workload"] == "c2_nich" and "model" not in d["config"]
    assert d["n_gpus"] == 1 and d["warmup"] >= 3 and d["higher_is_better"] is True and d["data"] == "synthetic"
    assert d["vs_baseline"] is None  # BASELINE.md publishes no number for this exact metric
    assert isinstance(baseline, dict)
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["unit"] == d["unit"]
    assert e["value"] < d["value"]  # the end-to-end number includes the copies
    c = d["cpu_baseline"]
    assert c["kind"] in ("reference", "port") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    assert d["gpu_launches"] >= d["steps"]
    clk = d["clocks"]
    assert not {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"} & set(clk["reasons"])


def test_committed_reference_arm_line():
    d = _line("c2_reference_arm.json")
    assert d["impl"] == "reference" and d["gpu_launches"] == 0
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]


def test_reference_arm_runs_here():
    from oracle.pyoracle import Ref
    if not Ref.available():
        pytest.skip("oracle/_ref not built and /root/reference absent")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "c1_dd", "--steps", "1",
                          "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads(out.stdout.strip().splitlines()[-1])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d) and d["value"] > 0
    assert d["config"]["workload"] == "c1_dd"


def test_steps_below_one_rejected():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


@pytest.mark.gpu
def test_timed_loop_runs_the_requested_steps():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import types
    import bench
    b = bench.Bench(types.SimpleNamespace(option=None, dump_outputs=None))
    calls = []
    for steps in (1, 7):
        del calls[:]
        ms, _, _ = b.timed(lambda: calls.append(1), steps, 0, flush=False)
        assert len(calls) == 3 + steps and ms >= 0  # at least three warm-up steps, then exactly the timed ones
    b.ctx.close()


@pytest.mark.gpu
def test_dump_outputs_are_the_sampled_indices(tmp_path, oracle):
    """--dump-outputs at c1: both timed paths' indices are what the oracle samples from the same scores and uniforms,
    up to near-ties"""
    import numpy as np
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import bench
    import cases
    from distributions_b200 import synth
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1_dd", "--steps", "2", "--warmup", "0",
                          "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["workload"] == "c1_dd"
    assert sorted(os.listdir(str(tmp_path))) == ["c1_dd_assign.npy", "c1_dd_cdf_assign.npy"]
    wl = bench.make_workload("c1_dd")
    scores = cases.oracle_scores(oracle, wl["feats"], prior=oracle.py_prior(synth.PY_ALPHA, synth.PY_D, wl["sizes"]))
    want = oracle.sample_rows(scores.copy(), wl["u"])
    for f in ("c1_dd_assign.npy", "c1_dd_cdf_assign.npy"):
        a = np.load(str(tmp_path / f))
        assert a.dtype == np.float32 and a.shape == (wl["N"],) and np.array_equal(a, np.round(a))
        got = a.astype(np.int32)
        assert cases.explained_mismatch(scores.astype(np.float64), wl["u"], got, want, 2e-5).all(), f
        assert np.mean(got == want) > 0.999, f
