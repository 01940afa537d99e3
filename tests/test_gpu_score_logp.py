"""Row log-likelihood on the device: dist_b200_score_logp_batch[_host] and dist_b200_logp_from_scores.

logp[n] = log sum_g exp(prior[g] + sum_f score_f(x[n][f]; g)) is checked against L = the float64 logsumexp of the [N][G]
scores that score_batch returns for the same features and prior:

    |logp - L| <= 2^-21 (1 + max_g |s_ng|) + (G + 8) 2^-24

(rounding of each exponent, ex2 at 2^-22 relative on MUFU or on the polynomial, an fp32 sum of G positive terms, the
final add).  Every route of score_dispatch is taken by at least one case:
  R1  score_rows_kernel logp mode (row-mapped features): nich G <= 128, gp / bnb every G, dd / bb with VALUE_CDF = 1,
      nich with NICH_PACKED = 1 / 2, ROW_TILE = 32 / 64, SMALL_TILE = 1 / 2 / 3, cross-cat lists (resident: the small list;
      streaming through the cp.async ring: 256 features at G = 128 and 256)
  R2  nich_logp_kernel: one nich feature, G > 128, default options
  R3  per-value table (value_logp_*): one dd / dpd / bb feature, default options, N >= 4 table rows
  R4  materialise + logp_scores_kernel: dpd with VALUE_CDF = 1 (or N < 4 table rows), niw, mixed lists with dpd / niw
"""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy import special

import cases
from distributions_b200 import capi, synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_score_logp.cc")
gpu = pytest.mark.gpu
MODEL_ID = {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW, "bnb": capi.BNB}
OPT_VALUE_CDF, OPT_ROW_TILE, OPT_SMALL_TILE, OPT_NICH_PACKED = 0, 1, 5, 6
GS = (1, 7, 32, 100, 128, 300, 1024)


@pytest.fixture(scope="module")
def ctx():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = capi.Context(0)
    yield c
    c.close()


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _column(w, n=None):
    v = w["values"] if n is None else w["values"][:n]
    return np.ascontiguousarray(v.astype(capi.COLUMN_DTYPE[MODEL_ID[w["model"]]]))


def _workload(model, G, N, seed):
    if model == "dd":
        return synth.dd(seed, G, N, dim=16)
    if model == "dpd":
        return synth.dpd(seed, G, N, V=100, other_frac=0.1)
    if model == "niw":
        return synth.niw(seed, G, N, d=3)
    return getattr(synth, model)(seed, G, N)


def _prior(ctx, sizes):
    return ctx.prior_pitman_yor_host(synth.PY_ALPHA, synth.PY_D, np.asarray(sizes, np.int32))


class _Opts:
    """context options for the duration of a block"""

    def __init__(self, ctx, opts):
        self.ctx, self.opts = ctx, opts

    def __enter__(self):
        for k, v in self.opts.items():
            self.ctx.set_option(k, v)

    def __exit__(self, *a):
        for k in self.opts:
            self.ctx.set_option(k, 0)


def _run(ctx, feats, ws, prior, n, opts=None):
    """(score_batch scores, score_logp_batch logp) of the first n rows, device-pointer entries"""
    import torch
    cols = [_dev(_column(w, n)) for w in ws]
    G = feats[0].groups
    prior_d = None if prior is None else _dev(np.asarray(prior, np.float32))
    scores = torch.empty((n, G), device="cuda", dtype=torch.float32)
    ctx.score_batch(feats, cols, n, prior_d, scores)
    logp = torch.full((n,), 777.0, device="cuda", dtype=torch.float32)
    with _Opts(ctx, opts or {}):
        ctx.score_logp_batch(feats, cols, n, prior_d, logp)
    torch.cuda.synchronize()
    return scores.cpu().numpy(), logp.cpu().numpy()


def _lse(scores):
    s = scores.astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        return special.logsumexp(s, axis=1)


def _check(scores, logp, what=""):
    """|logp - L| within the stated bound; rows whose every term is -inf must be -inf"""
    G = scores.shape[1]
    L = _lse(scores)
    fin = np.where(np.isfinite(scores), np.abs(scores), 0.0).max(axis=1)
    bound = 2.0 ** -21 * (1.0 + fin) + (G + 8) * 2.0 ** -24
    dead = np.isneginf(L)
    assert np.array_equal(np.isneginf(logp), dead), what
    err = np.abs(logp[~dead].astype(np.float64) - L[~dead])
    assert not np.isnan(logp).any(), what
    assert (err <= bound[~dead]).all(), "%s: worst %.3g (bound %.3g)" % (what, err.max(), bound[~dead][err.argmax()])
    return err


def _features(ctx, ws):
    return [ctx.feature(MODEL_ID[w["model"]]).update_all(w) for w in ws]


# ---- against the library's own scores ---------------------------------------------------------------------------
ROW_VARIANTS = {  # option sets whose route differs from the default for some G (comments: the route taken)
    "default": {},                                       # nich G > 128: R2; dd / bb: R3; the rest R1
    "value_cdf_off": {OPT_VALUE_CDF: 1},                 # dd / bb: R1
    "row_tile_32": {OPT_VALUE_CDF: 1, OPT_ROW_TILE: 32},  # G > 128: R1 with 32-group tiles
    "row_tile_64": {OPT_VALUE_CDF: 1, OPT_ROW_TILE: 64},  # G > 128: R1 with 64-group tiles
    "small_tile_256": {OPT_VALUE_CDF: 1, OPT_SMALL_TILE: 1},  # 64 < G <= 128: 256-thread blocks
    "small_tile_128x3": {OPT_VALUE_CDF: 1, OPT_SMALL_TILE: 2},
    "small_tile_4x32": {OPT_VALUE_CDF: 1, OPT_SMALL_TILE: 3},  # 64 < G <= 128: four 32-group tiles
    "nich_scalar": {OPT_NICH_PACKED: 1},                 # nich: R1 with the scalar loop (also G > 128)
    "nich_packed_one_row": {OPT_NICH_PACKED: 2},         # nich G > 128: R1 packed instead of R2
}


@gpu
@pytest.mark.parametrize("G", GS)
@pytest.mark.parametrize("model", ["nich", "gp", "bnb", "bb", "dd"])
def test_row_mapped_models(ctx, model, G):
    n = 3001
    w = _workload(model, G, n, 700 + G)
    prior = _prior(ctx, w["sizes"])
    feats = _features(ctx, [w])
    ref = None
    for name, opts in ROW_VARIANTS.items():
        if name.startswith("nich") and model != "nich":
            continue
        scores, logp = _run(ctx, feats, [w], prior, n, opts)
        _check(scores, logp, "%s G=%d %s" % (model, G, name))
        ref = scores if ref is None else ref
        assert np.array_equal(scores, ref)  # the options change no score


@gpu
@pytest.mark.parametrize("G", [19, 128, 512, 1100])
def test_dpd(ctx, G):
    """R3 (default), R4 (VALUE_CDF = 1, and a batch below 4 table rows); non-dense keys included"""
    n = 2000
    w = _workload("dpd", G, n, 900 + G)
    if G == 512:  # sorted-key search instead of the identity map
        keys = (np.arange(w["keys"].size, dtype=np.uint32) * 7 + 3)[::-1].copy()
        other = w["values"] == 0xFFFFFFFF
        w["values"] = np.where(other, 0xFFFFFFFF, keys[np.minimum(w["values"], keys.size - 1)]).astype(np.uint32)
        w["keys"] = keys
    prior = _prior(ctx, w["sizes"])
    feats = _features(ctx, [w])
    for opts in ({}, {OPT_VALUE_CDF: 1}):
        scores, logp = _run(ctx, feats, [w], prior, n, opts)
        _check(scores, logp, "dpd G=%d %s" % (G, opts))
    scores, logp = _run(ctx, feats, [w], prior, 50)  # 50 < 4 * 101 rows: per-cell route
    _check(scores, logp, "dpd short batch")


@gpu
@pytest.mark.parametrize("d,G", [(3, 40), (5, 130), (8, 7), (32, 256)])
def test_niw(ctx, d, G):
    n = 3000
    w = synth.niw(40 + d, G, n, d=d)
    scores, logp = _run(ctx, _features(ctx, [w]), [w], _prior(ctx, w["sizes"]), n)
    _check(scores, logp, "niw d=%d" % d)


def _small_list(G, n, seed):
    ws = [synth.nich(seed, G, n), synth.gp(seed + 1, G, n), synth.bb(seed + 2, G, n), synth.dd(seed + 3, G, n, dim=16),
          synth.bnb(seed + 4, G, n)]
    for w in ws[1:]:
        w["sizes"] = ws[0]["sizes"]
    return ws


@gpu
@pytest.mark.parametrize("G", [37, 300])
def test_crosscat_small_list(ctx, G):
    """five models in one list: caches resident (R1); G = 300 with ROW_TILE 32 / 64"""
    n = 4000
    ws = _small_list(G, n, 500 + G)
    feats = _features(ctx, ws)
    prior = _prior(ctx, ws[0]["sizes"])
    for opts in ({}, {OPT_ROW_TILE: 32}, {OPT_ROW_TILE: 64}):
        scores, logp = _run(ctx, feats, ws, prior, n, opts)
        _check(scores, logp, "small list G=%d %s" % (G, opts))


@gpu
@pytest.mark.parametrize("G", [128, 256])
def test_crosscat_streaming(ctx, G):
    """128 gp + 128 bb features: caches stream through the cp.async ring (R1)"""
    n = 2048
    kind = synth.crosscat(61, G, n)
    ws = kind["features"]
    feats = _features(ctx, ws)
    prior = _prior(ctx, kind["sizes"])
    scores, logp = _run(ctx, feats, ws, prior, n)
    _check(scores, logp, "streaming G=%d" % G)
    scores, logp = _run(ctx, feats, ws, np.full(G, -np.inf, np.float32), 300)
    assert np.isneginf(logp).all()


@gpu
def test_mixed_lists(ctx):
    """lists holding dpd / niw materialise the scores (R4)"""
    G, n = 40, 3000
    a = synth.nich(81, G, n)
    b = synth.dpd(82, G, n, V=50, other_frac=0.05)
    c = synth.niw(83, G, n, d=3)
    e = synth.gp(84, G, n)
    for w in (b, c, e):
        w["sizes"] = a["sizes"]
    prior = _prior(ctx, a["sizes"])
    for ws in ([a, b], [e, c], [b, c, a]):
        scores, logp = _run(ctx, _features(ctx, ws), ws, prior, n)
        _check(scores, logp, "+".join(w["model"] for w in ws))


# ---- against the oracle -------------------------------------------------------------------------------------------
def _envelope(oracle, w, n):
    """[n][G] per-cell score envelope of the parity tests (bnb: its cancellation envelope, test_gpu_bnb.py)"""
    if w["model"] == "bnb":
        from test_gpu_bnb import envelope
        return envelope(oracle.bnb_caches(w["shared"], w["count"], w["sum"]), w["values"][:n])
    from test_gpu_parity import envelope
    return np.broadcast_to(envelope(oracle, w)[None, :], (n, w["sizes"].size))


@gpu
@pytest.mark.parametrize("model", ["nich", "gp", "bb", "dd", "dpd", "bnb"])
@pytest.mark.parametrize("G", [7, 100, 300])
def test_against_oracle(ctx, oracle, model, G):
    n = 2000
    w = _workload(model, G, n, 1300 + G)
    if model == "bnb" and not hasattr(oracle, "bnb_caches"):
        pytest.skip("oracle without bnb")
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    _, logp = _run(ctx, _features(ctx, [w]), [w], prior, n)
    so = cases.oracle_scores(oracle, [w], n, prior).astype(np.float64)
    L = _lse(so)
    top = so.argmax(axis=1)
    s_top = so[np.arange(n), top]
    env = _envelope(oracle, w, n)[np.arange(n), top] + 3e-6 * (1 + np.abs(s_top))
    fin = np.abs(so).max(axis=1)
    bound = env + 2.0 ** -21 * (1.0 + fin) + (G + 8) * 2.0 ** -24
    err = np.abs(logp - L)
    assert (err <= bound).all(), "worst %.3g" % err.max()


# ---- meaning: the posterior predictive integrates to one --------------------------------------------------------
def _single_logp(ctx, w, values, prior):
    import torch
    f = _features(ctx, [w])
    col = _dev(np.ascontiguousarray(values.astype(capi.COLUMN_DTYPE[MODEL_ID[w["model"]]])))
    logp = torch.empty(values.shape[0], device="cuda", dtype=torch.float32)
    ctx.score_logp_batch(f, [col], values.shape[0], _dev(prior), logp)
    torch.cuda.synchronize()
    return logp.cpu().numpy().astype(np.float64)


@gpu
@pytest.mark.parametrize("G", [7, 300])
def test_predictive_sums_to_one(ctx, G):
    """with the Pitman-Yor prior (sizes include the empty group) sum_v exp(logp(v)) = 1 within 1e-3 (the reference's TOL)"""
    bb = synth.bb(31, G, 10)
    assert abs(np.exp(_single_logp(ctx, bb, np.array([0, 1]), _prior(ctx, bb["sizes"]))).sum() - 1) < 1e-3
    dd = synth.dd(32, G, 10, dim=16)
    assert abs(np.exp(_single_logp(ctx, dd, np.arange(16), _prior(ctx, dd["sizes"]))).sum() - 1) < 1e-3
    gp = synth.gp(33, G, 10)
    p = np.exp(_single_logp(ctx, gp, np.arange(20000), _prior(ctx, gp["sizes"])))
    assert p[-1000:].sum() < 1e-7 and abs(p.sum() - 1) < 1e-3
    ni = synth.nich(34, G, 10)
    ni["shared"] = np.array(ni["shared"], np.float32)
    ni["shared"][3] = max(float(ni["shared"][3]), 4.0)
    x = np.linspace(-400.0, 400.0, 800001)
    p = np.exp(_single_logp(ctx, ni, x.astype(np.float32), _prior(ctx, ni["sizes"])))
    # loosened beyond 1e-3 by the reference's own fast_log: its table truncates the mantissa (one step = LOG_STEP in
    # the log), so log(1 + precision d^2) is low by half a step on average, and the score, log_coeff = -(nu' + 1) / 2
    # times that log, is high by up to LOG_STEP / 2 * |log_coeff| -- a density inflated by ~1e-3 at 40-row groups
    log_step = 6.2e-5
    bias = 0.5 * log_step * (float(ni["shared"][3]) + float(ni["count"].max()) + 1) / 2
    assert abs(np.trapezoid(p, x) - 1) < 1e-3 + bias


# ---- outliers and -inf ----------------------------------------------------------------------------------------------
@gpu
def test_nich_outlier_rows(ctx):
    """nich G > 128 (R2), no broad group, every seventh row thousands of sigmas away: the rows re-evaluated with their own
    maximum agree with L"""
    n, G = 20_000, 300
    w = synth.nich(77, G, n)
    rng = np.random.default_rng(78)
    w["count"] = np.maximum(w["count"], 60).astype(w["count"].dtype)
    w["sizes"] = w["count"].astype(w["sizes"].dtype)
    w["mean"] = rng.normal(0.0, 5.0, G).astype(np.float32)
    w["ctv"] = (w["count"] * rng.uniform(0.5, 2.0, G)).astype(np.float32)
    far = np.arange(n) % 7 == 0
    w["values"] = rng.normal(0.0, 5.0, n).astype(np.float32)
    w["values"][far] = np.where(np.arange(far.sum()) % 2 == 0, 3e4, -7e5).astype(np.float32) + w["values"][far]
    prior = _prior(ctx, w["sizes"])
    scores, logp = _run(ctx, _features(ctx, [w]), [w], prior, n)
    assert scores[far].max(axis=1).max() < scores[~far].max(axis=1).min() - 100.0
    _check(scores, logp, "outliers")


@gpu
@pytest.mark.parametrize("case", ["nich50", "nich300", "dd", "dd_cells", "dpd", "dpd_cells", "niw", "bb", "gp"])
def test_prior_minus_inf(ctx, case):
    """a prior of -inf everywhere gives -inf on every route, never NaN"""
    model, G = {"nich50": ("nich", 50), "nich300": ("nich", 300), "dd": ("dd", 40), "dd_cells": ("dd", 40), "dpd": ("dpd", 40),
                "dpd_cells": ("dpd", 40), "niw": ("niw", 20), "bb": ("bb", 300), "gp": ("gp", 1024)}[case]
    n = 1000
    w = _workload(model, G, n, 5)
    opts = {OPT_VALUE_CDF: 1} if case.endswith("cells") else {}
    _, logp = _run(ctx, _features(ctx, [w]), [w], np.full(G, -np.inf, np.float32), n, opts)
    assert np.isneginf(logp).all()


# ---- ordering and forms ---------------------------------------------------------------------------------------------
@gpu
def test_sees_add_rows_on_another_stream(ctx):
    import torch
    G, n = 300, 200_000
    w = synth.nich(91, G, n)
    f = _features(ctx, [w])
    col = _dev(_column(w))
    assign = _dev(np.random.default_rng(1).integers(0, G, n).astype(np.int32))
    before = torch.empty(n, device="cuda", dtype=torch.float32)
    ctx.score_logp_batch(f, [col], n, None, before)
    torch.cuda.synchronize()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    after = torch.empty(n, device="cuda", dtype=torch.float32)
    ctx.add_rows_batch(f, [col], assign, n, stream=s1.cuda_stream)
    ctx.score_logp_batch(f, [col], n, None, after, stream=s2.cuda_stream)
    torch.cuda.synchronize()
    again = torch.empty(n, device="cuda", dtype=torch.float32)
    ctx.score_logp_batch(f, [col], n, None, again)
    torch.cuda.synchronize()
    assert not torch.equal(before, again)
    assert torch.equal(after, again)


@gpu
@pytest.mark.parametrize("case", ["nich300", "dd", "dpd", "small_list", "niw"])
def test_host_form_bit_identical(ctx, case):
    """pageable, cudaHostAlloc (torch pin_memory) and registered buffers give the device form's bits"""
    import torch
    n = 200_001
    if case == "small_list":
        ws = _small_list(37, n, 17)
    else:
        ws = [{"nich300": lambda: synth.nich(18, 300, n), "dd": lambda: synth.dd(19, 100, n, dim=16),
               "dpd": lambda: synth.dpd(21, 200, n, V=100, other_frac=0.1), "niw": lambda: synth.niw(20, 50, n, d=5)}[case]()]
    feats = _features(ctx, ws)
    prior = _prior(ctx, ws[0]["sizes"])
    _, ref = _run(ctx, feats, ws, prior, n)
    cols = [_column(w) for w in ws]
    assert np.array_equal(ctx.score_logp_batch_host(feats, cols, prior), ref)
    pinned = [torch.from_numpy(c).pin_memory().numpy() for c in cols]
    out = torch.empty(n, dtype=torch.float32).pin_memory().numpy()
    assert np.array_equal(ctx.score_logp_batch_host(feats, pinned, prior, logp_out=out), ref)
    reg = [c.copy() for c in cols]
    out2 = np.empty(n, np.float32)
    for a in reg + [out2]:
        ctx.host_register(a)
    try:
        assert np.array_equal(ctx.score_logp_batch_host(feats, reg, prior, logp_out=out2), ref)
    finally:
        for a in reg + [out2]:
            ctx.host_unregister(a)


@gpu
def test_logp_from_scores(ctx):
    import torch
    G, n = 300, 5000
    w = synth.gp(71, G, n)
    scores, _ = _run(ctx, _features(ctx, [w]), [w], _prior(ctx, w["sizes"]), n)
    logp = torch.empty(n, device="cuda", dtype=torch.float32)
    ctx.logp_from_scores(_dev(scores), n, G, logp)
    torch.cuda.synchronize()
    _check(scores, logp.cpu().numpy(), "logp_from_scores")


# ---- error codes ----------------------------------------------------------------------------------------------------
@gpu
def test_errors(ctx):
    import torch
    L = ctx.L
    G, n = 20, 100
    w = synth.nich(1, G, n)
    f = _features(ctx, [w])[0]
    col = _dev(_column(w))
    out = torch.empty(n, device="cuda", dtype=torch.float32)
    fa = (ctypes.c_void_p * 1)(f.h)
    ca = (ctypes.c_void_p * 1)(col.data_ptr())
    assert L.dist_b200_score_logp_batch(ctx.h, fa, 1, ca, n, None, None, None) == 1  # ERR_INVALID: null logp
    assert L.dist_b200_score_logp_batch_host(ctx.h, fa, 1, ca, n, None, None) == 1
    g2 = _features(ctx, [synth.gp(2, G + 1, n)])[0]
    gcol = _dev(_column(synth.gp(2, G + 1, n)))
    fa2 = (ctypes.c_void_p * 2)(f.h, g2.h)
    ca2 = (ctypes.c_void_p * 2)(col.data_ptr(), gcol.data_ptr())
    assert L.dist_b200_score_logp_batch(ctx.h, fa2, 2, ca2, n, None, out.data_ptr(), None) == 4  # ERR_STATE: G mismatch
    fresh = ctx.feature(capi.NICH)
    fa3 = (ctypes.c_void_p * 1)(fresh.h)
    assert L.dist_b200_score_logp_batch(ctx.h, fa3, 1, ca, n, None, out.data_ptr(), None) == 4  # before update_all
    assert L.dist_b200_logp_from_scores(ctx.h, out.data_ptr(), n, 0, out.data_ptr(), None) == 1
    torch.cuda.synchronize()


# ---- mirrors --------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["nich", "gp", "bnb", "bb", "dd", "dpd", "niw"])
def test_models_score_logp(ctx, name):
    """models.<name>.Mixture.score_logp after add_value choreography equals the C entry on the same feature"""
    from distributions_b200 import models
    model = models.MODELS[name]
    shared = model.Shared(r=3) if name == "bnb" else model.Shared()
    mixture = model.Mixture(ctx)
    rng = np.random.default_rng(len(name) + 11)
    for _ in range(3):
        g = model.Group()
        g.init(shared)
        mixture.append(g)
    mixture.init(shared)
    vals = {"nich": lambda: float(rng.normal(2.0, 1.0)), "gp": lambda: int(rng.poisson(4)), "bnb": lambda: int(rng.poisson(4)),
            "bb": lambda: bool(rng.random() < 0.8), "dd": lambda: int(rng.integers(0, 3)),
            "dpd": lambda: int(rng.integers(0, 3)), "niw": lambda: rng.normal(2.0, 1.0, shared.dim).astype(np.float32)}[name]
    for i in range(300):
        mixture.add_value(shared, 1 + i % 2, vals())
    values = [vals() for _ in range(500)]
    prior = np.log(np.array([0.2, 0.5, 0.3], np.float32))
    got = mixture.score_logp(shared, values, prior)
    assert got.shape == (500,) and got.dtype == np.float32
    col = np.ascontiguousarray(np.asarray(values, capi.COLUMN_DTYPE[mixture.model_id]))
    if name == "niw":
        col = col.reshape(-1, shared.dim)
    ref = ctx.score_logp_batch_host([mixture.feature], [col], prior)
    assert np.array_equal(got, ref)
    scores = np.zeros((500, 3), np.float32)
    for i, v in enumerate(values[:20]):  # and the per-value scores agree with it
        s = prior.copy()
        mixture.score_value(shared, v, s)
        scores[i] = s
    assert np.allclose(got[:20], _lse(scores[:20]), atol=1e-5, rtol=1e-6)


def _compile_cpp(out):
    from distributions_b200 import build
    build.build()
    lib_dir = os.path.join(ROOT, "distributions_b200", "lib")
    cmd = ["g++", "-std=c++14", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), CPP_SRC, "-o", out,
           "-L" + lib_dir, "-ldist_b200", "-Wl,-rpath," + lib_dir]
    subprocess.run(cmd, check=True)
    return out


def test_cpp_score_logp_compiles(tmp_path):
    _compile_cpp(str(tmp_path / "test_score_logp"))


@gpu
def test_cpp_score_logp_matches_capi(ctx, tmp_path):
    exe = _compile_cpp(str(tmp_path / "test_score_logp"))
    lines = dict(l.split(" ", 1) for l in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.strip().splitlines())
    got = {k: np.array(v.split(), np.uint32).view(np.float32) for k, v in lines.items()}
    gpf = ctx.feature(capi.GP).update_all(dict(model="gp", shared=np.array([2, 0.5], np.float32), count=np.array([0, 20, 5], np.uint32),
                                               sum=np.array([0, 190, 510], np.uint32)))
    bbf = ctx.feature(capi.BB).update_all(dict(model="bb", shared=np.array([0.5, 2], np.float32), heads=np.array([0, 10, 0], np.int32),
                                               tails=np.array([0, 0, 10], np.int32)))
    prior = np.array([-0.5, -1.25, -2.0], np.float32)
    gv = np.array([0, 3, 9, 17, 40, 101, 250, 1], np.uint32)
    bv = np.array([1, 0, 1, 1, 0, 0, 1, 0], np.uint8)
    assert np.array_equal(got["gp"], ctx.score_logp_batch_host([gpf], [gv], prior))
    assert np.array_equal(got["bb"], ctx.score_logp_batch_host([bbf], [bv]))
    assert np.array_equal(got["kind"], ctx.score_logp_batch_host([gpf, bbf], [gv, bv], prior))
