"""Batched Group::sample_value (dist_b200_sample_values_batch): posterior-predictive draws on the device.

Every statistical test draws 2^20 values per group with a fixed seed, so it passes or fails the same way on every run.
The expected distributions are exact float64 formulas from scipy (t, nbinom, betanbinom, multivariate t through its
univariate projections); discrete models are checked with Pearson's chi-square (cells of expected count < 5 pooled),
continuous ones with Kolmogorov-Smirnov.  All tests share one p-value floor, P_FLOOR.  The power tests show that the
same statistics reject draws tested against a posterior off by 1 % or against the neighbouring group, and
test_parametrisation_matches_score_value ties each scipy distribution to the library's own score_value (which the
parity tests pin to the reference)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest
from scipy import special, stats

from distributions_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP_SRC = os.path.join(ROOT, "tests", "cpp", "test_sample_values.cc")
P_FLOOR = 1e-6  # one floor for every distribution test: a correct sampler fails it with probability 1e-6 per test
DRAWS = 1 << 20
gpu = pytest.mark.gpu


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


# ---- workloads: statistics of the test groups and the exact predictive of each (float64) -------------------------
def _nich():
    sh = np.array([0.5, 2.0, 1.5, 1.0], np.float32)  # nu = 1: the empty group's chi-square shape 1/2 takes the boost
    count = np.array([0, 5, 1_000_000], np.int32)
    mean = np.array([0.0, -1.0, 0.3], np.float32)
    ctv = np.array([0.0, 3.0, 2.0e6], np.float32)
    w = dict(model="nich", shared=sh, count=count, mean=mean, ctv=ctv)
    mu, kappa, sigmasq, nu = sh.astype(np.float64)
    dists = []
    for n, m, c in zip(count.astype(np.float64), mean.astype(np.float64), ctv.astype(np.float64)):
        pk, pn = kappa + n, nu + n
        pm = (kappa * mu + m * n) / pk
        ps = (nu * sigmasq + c + n * kappa * (mu - m) ** 2 / pk) / pn
        dists.append(stats.t(df=pn, loc=pm, scale=np.sqrt(ps * (pk + 1) / pk)))
    return w, dists


def _gp():
    sh = np.array([0.5, 0.5], np.float32)  # alpha < 1: the empty group's gamma shape takes the boost
    count = np.array([0, 3, 1000], np.uint32)
    sm = np.array([0, 7, 1_000_000], np.uint32)  # large group: shape 10^6, lambda ~ 10^3
    w = dict(model="gp", shared=sh, count=count, sum=sm)
    return w, [_gp_dist(sh[0] + s, sh[1] + c) for c, s in zip(count.astype(np.float64), sm.astype(np.float64))]


def _gp_dist(shape, rate):
    return stats.nbinom(n=float(shape), p=float(rate) / (1.0 + float(rate)))


def _bnb():
    r = 1000
    sh = np.array([2.5, 2.0, r], np.float32)
    count = np.array([0, 4, 1000], np.uint32)   # large group: alpha' = 10^6, beta' ~ 10^6, mean ~ 10^3
    sm = np.array([0, 9000, 1_000_000], np.uint32)
    w = dict(model="bnb", shared=sh, count=count, sum=sm)
    return w, [_bnb_dist(r, sh[0] + r * c, sh[1] + s) for c, s in zip(count.astype(np.float64), sm.astype(np.float64))]


def _bnb_dist(r, a, b):
    return stats.betanbinom(n=r, a=float(a), b=float(b))


def _bb():
    sh = np.array([0.5, 2.0], np.float32)
    heads = np.array([0, 3, 400_000], np.int32)
    tails = np.array([0, 1, 600_000], np.int32)
    w = dict(model="bb", shared=sh, heads=heads, tails=tails)
    p = (sh[0] + heads.astype(np.float64)) / (sh[0] + sh[1] + heads.astype(np.float64) + tails.astype(np.float64))
    return w, [np.array([1 - q, q]) for q in p]


def _dd(dim):
    rng = np.random.default_rng(dim)
    alphas = rng.uniform(0.05, 2.0, dim).astype(np.float32)
    counts = np.zeros((3, dim), np.int32)
    counts[1, rng.integers(0, dim, 10)] += 1
    counts[2] = rng.integers(0, 5000, dim)
    w = dict(model="dd", alphas=alphas, counts=counts)
    wt = alphas.astype(np.float64)[None, :] + counts
    return w, list(wt / wt.sum(1, keepdims=True))


def _dpd(beta0):
    rng = np.random.default_rng(11 if beta0 else 12)
    V = 40
    keys = np.sort(rng.choice(100_000, V, replace=False)).astype(np.uint32)[rng.permutation(V)]  # non-contiguous, unsorted
    betas = rng.uniform(0.1, 1.0, V)
    betas = (betas / betas.sum() * (1.0 - beta0)).astype(np.float32)
    beta0 = max(0.0, 1.0 - float(betas.astype(np.float64).sum())) if beta0 else 0.0
    alpha = 3.0
    counts = np.zeros((3, V), np.int32)
    counts[1, :4] = [2, 0, 5, 1]
    counts[2] = rng.integers(0, 3000, V)
    w = dict(model="dpd", alpha=alpha, beta0=beta0, keys=keys, betas=betas, counts=counts)
    wt = np.concatenate([alpha * betas.astype(np.float64)[None, :] + counts, np.full((3, 1), alpha * np.float64(np.float32(beta0)))], 1)
    return w, list(wt / wt.sum(1, keepdims=True))


def _niw(d):
    rng = np.random.default_rng(100 + d)
    mu = rng.normal(size=d).astype(np.float32)
    A = rng.normal(size=(d, d))
    psi = (A @ A.T / d + np.eye(d)).astype(np.float32)
    kappa, nu = 1.5, d + 2.0
    x = rng.normal(size=(60, d)) * 2 + 1
    count = np.array([0, 60], np.int32)
    sum_x = np.stack([np.zeros(d), x.sum(0)]).astype(np.float32)
    sum_xxT = np.stack([np.zeros((d, d)), x.T @ x]).astype(np.float32)
    w = dict(model="niw", mu=mu, kappa=kappa, psi=psi, nu=nu, count=count, sum_x=sum_x, sum_xxT=sum_xxT)
    dists = []
    for g in range(2):
        n = float(count[g])
        sx, sxx = sum_x[g].astype(np.float64), sum_xxT[g].astype(np.float64)
        xbar = sx / n if n else np.zeros(d)
        diff = xbar - mu
        C = sxx - np.outer(sx, xbar) - np.outer(xbar, sx) + n * np.outer(xbar, xbar)
        pk, pn = kappa + n, nu + n
        ppsi = psi.astype(np.float64) + C + kappa * n / (kappa + n) * np.outer(diff, diff)
        dof = pn - d + 1
        dists.append(dict(loc=(kappa * mu + n * xbar) / pk, shape=ppsi * (pk + 1) / (pk * dof), df=dof))
    return w, dists


MODEL_ID = {"nich": capi.NICH, "gp": capi.GP, "bnb": capi.BNB, "bb": capi.BB, "dd": capi.DD, "dpd": capi.DPD, "niw": capi.NIW}
CASES = {"nich": _nich, "gp": _gp, "bnb": _bnb, "bb": _bb, "dd16": lambda: _dd(16), "dd256": lambda: _dd(256),
         "dpd_beta0": lambda: _dpd(0.2), "dpd_no_beta0": lambda: _dpd(0.0),
         "niw1": lambda: _niw(1), "niw3": lambda: _niw(3), "niw8": lambda: _niw(8), "niw32": lambda: _niw(32)}


def _feature(ctx, w):
    return ctx.feature(MODEL_ID[w["model"]]).update_all(w)


def _draw(ctx, f, G, seed=1):
    """2^20 draws of every group, rows group-major"""
    assign = np.repeat(np.arange(G, dtype=np.int32), DRAWS)
    x = ctx.sample_values_batch_host([f], assign, seed)[0]
    return x.reshape(G, DRAWS, -1) if f.model == capi.NIW else x.reshape(G, DRAWS)


# ---- tests of fit ------------------------------------------------------------------------------------------------
def _pool(obs, exp):
    """merge adjacent cells until every expected count is >= 5"""
    o_out, e_out, o_acc, e_acc = [], [], 0.0, 0.0
    for o, e in zip(obs, exp):
        o_acc += o
        e_acc += e
        if e_acc >= 5:
            o_out.append(o_acc)
            e_out.append(e_acc)
            o_acc = e_acc = 0.0
    if e_acc > 0 or o_acc > 0:
        o_out[-1] += o_acc
        e_out[-1] += e_acc
    return np.array(o_out), np.array(e_out)


def chi2_categorical(cats, probs):
    obs = np.bincount(cats, minlength=len(probs)).astype(np.float64)
    assert obs.size == len(probs), "draw outside the support"
    o, e = _pool(obs, cats.size * np.asarray(probs, np.float64))
    return stats.chi2.sf(((o - e) ** 2 / e).sum(), len(o) - 1)


def chi2_count(x, dist):
    """Pearson chi-square of integer draws against a scipy distribution on 0, 1, 2, ...: one cell per value up to the
    largest draw (at most 200k cells; heavy tails beyond go into the last cell, which also takes the mass above)"""
    x = x.astype(np.int64)
    hi = int(min(x.max(), 200_000))
    p = np.exp(dist.logpmf(np.arange(hi + 1)))
    p[-1] += max(0.0, 1.0 - p.sum())
    obs = np.bincount(np.minimum(x, hi), minlength=hi + 1).astype(np.float64)
    o, e = _pool(obs, x.size * p)
    return stats.chi2.sf(((o - e) ** 2 / e).sum(), len(o) - 1)


def _dpd_cats(w, x):
    keys = list(map(int, w["keys"])) + [0xFFFFFFFF]
    lut = {k: i for i, k in enumerate(keys)}
    return np.array([lut[int(v)] for v in np.unique(x)]), np.unique(x, return_inverse=True)[1]


def _fit_p(case, w, dists, g, x):
    m = w["model"]
    if m == "nich":
        return stats.kstest(x.astype(np.float64), dists[g].cdf).pvalue
    if m in ("gp", "bnb"):
        return chi2_count(x, dists[g])
    if m == "bb":
        return chi2_categorical(x.astype(np.int64), dists[g])
    if m == "dd":
        return chi2_categorical(x.astype(np.int64), dists[g])
    if m == "dpd":
        ids, inv = _dpd_cats(w, x)
        return chi2_categorical(ids[inv], dists[g])
    raise ValueError(m)


def _niw_ps(x, dist, rng, n_proj=4):
    """KS p-values of random unit projections a^T x ~ t(df, a^T loc, sqrt(a^T shape a)), and the mean's z-score"""
    x = x.astype(np.float64)
    d = x.shape[1]
    ps = []
    for _ in range(n_proj):
        a = rng.normal(size=d)
        a /= np.linalg.norm(a)
        ps.append(stats.kstest(x @ a, stats.t(df=dist["df"], loc=a @ dist["loc"], scale=np.sqrt(a @ dist["shape"] @ a)).cdf).pvalue)
    cov = dist["shape"] * dist["df"] / (dist["df"] - 2)
    z = np.abs(x.mean(0) - dist["loc"]) / np.sqrt(np.diag(cov) / x.shape[0])
    return ps, float(z.max())


@gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_distribution(ctx, case):
    w, dists = CASES[case]()
    f = _feature(ctx, w)
    G = len(dists)
    x = _draw(ctx, f, G)
    if w["model"] == "niw":
        rng = np.random.default_rng(5)
        for g in range(G):
            ps, z = _niw_ps(x[g], dists[g], rng)
            assert min(ps) > P_FLOOR, (case, g, ps)
            assert z < stats.norm.isf(P_FLOOR / (2 * x.shape[-1])), (case, g, z)  # the floor, two-sided, over the d means
        return
    for g in range(G):
        p = _fit_p(case, w, dists, g, x[g])
        assert p > P_FLOOR, (case, g, p)


@gpu
def test_power_off_by_one_percent(ctx):
    """the chi-square rejects draws tested against a posterior parameter 1 % off"""
    w, dists = _gp()
    x = _draw(ctx, _feature(ctx, w), 3)
    shape, rate = 0.5 + 1_000_000, 0.5 + 1000
    assert chi2_count(x[2], dists[2]) > P_FLOOR
    assert chi2_count(x[2], _gp_dist(shape * 1.01, rate)) < P_FLOOR
    w, dists = _bnb()
    x = _draw(ctx, _feature(ctx, w), 3)
    assert chi2_count(x[2], dists[2]) > P_FLOOR
    assert chi2_count(x[2], _bnb_dist(1000, 2.5 + 1000 * 1000, (2.0 + 1_000_000) * 1.01)) < P_FLOOR
    w, dists = _bb()
    x = _draw(ctx, _feature(ctx, w), 3)
    q = dists[2][1] * 1.01
    assert chi2_categorical(x[2].astype(np.int64), [1 - q, q]) < P_FLOOR


@gpu
@pytest.mark.parametrize("case", ["nich", "dd16", "dpd_beta0", "niw3"])
def test_power_neighbouring_group(ctx, case):
    """the same statistics reject draws of group 1 tested against group 0's predictive"""
    w, dists = CASES[case]()
    x = _draw(ctx, _feature(ctx, w), len(dists))
    if w["model"] == "niw":
        ps, z = _niw_ps(x[1], dists[0], np.random.default_rng(5))
        assert min(ps) < P_FLOOR or z > 10
    else:
        assert _fit_p(case, w, dists, 0, x[1]) < P_FLOOR


# ---- the scipy parametrisation against the library's score_value ------------------------------------------------
@gpu
@pytest.mark.parametrize("case", ["nich", "gp", "bnb", "bb", "dd16", "dpd_beta0", "niw3"])
def test_parametrisation_matches_score_value(ctx, case):
    """log pmf / pdf of the expected distribution == score_value (bnb: plus log C(v + r - 1, v), which the reference's
    score omits), on the empty and the small group.  The tolerance is the envelope of the reference's fp32 score:
    fast_lgamma_nu's approximation at nu ~ 1 is ~1e-2 (nich's empty group), fast_log / fast_lgamma a few 1e-3; a
    wrong parameter (scale, dof, shape, rate off) moves the log density by far more.  The large groups are left out:
    there the reference's fp32 score itself cancels terms of 10^6..10^7 and is off by up to ~0.5."""
    w, dists = CASES[case]()
    f = _feature(ctx, w)
    m, G = w["model"], len(dists)
    rng = np.random.default_rng(3)
    for g in range(min(G, 2)):
        if m == "nich":
            vals = dists[g].ppf(rng.uniform(0.02, 0.98, 5)).astype(np.float32)
        elif m in ("gp", "bnb"):
            vals = dists[g].ppf(rng.uniform(0.05, 0.95, 5)).astype(np.uint32)
        elif m == "bb":
            vals = np.array([0, 1], np.uint8)
        elif m == "dd":
            vals = rng.integers(0, len(dists[g]), 5).astype(np.int32)
        elif m == "dpd":
            vals = np.concatenate([w["keys"][rng.integers(0, len(w["keys"]), 4)], [0xFFFFFFFF]]).astype(np.uint32)
        else:
            vals = stats.multivariate_t(loc=dists[g]["loc"], shape=dists[g]["shape"], df=dists[g]["df"]).rvs(3, random_state=rng)
            vals = np.atleast_2d(vals).astype(np.float32)
        for v in vals:
            slack = 0.0
            acc = np.zeros(G, np.float32)
            ctx.score_value_host(f, v, acc)
            got = float(acc[g])
            if m == "nich":
                want = dists[g].logpdf(float(v))
            elif m == "gp":
                want = dists[g].logpmf(int(v))
            elif m == "bnb":
                want = dists[g].logpmf(int(v))
                got += special.gammaln(int(v) + 1000) - special.gammaln(int(v) + 1) - special.gammaln(1000)
                a, b = dists[g].kwds["a"], dists[g].kwds["b"]
                terms = special.gammaln([a + b, a, b, a + 1000, b + int(v), a + b + 1000 + int(v)])
                slack = 4e-7 * np.abs(terms).sum()  # the fp32 score sums lgamma terms of up to ~10^5: its rounding
            elif m in ("bb", "dd"):
                want = np.log(dists[g][int(v)])
            elif m == "dpd":
                k = len(w["keys"]) if int(v) == 0xFFFFFFFF else list(map(int, w["keys"])).index(int(v))
                want = np.log(dists[g][k])
            else:
                want = stats.multivariate_t(loc=dists[g]["loc"], shape=dists[g]["shape"], df=dists[g]["df"]).logpdf(v.astype(np.float64))
            assert abs(got - want) <= 2e-2 + 2e-3 * abs(want) + slack, (case, g, v, got, want)


# ---- the random-number contract ---------------------------------------------------------------------------------
def _mixed(ctx, N=200_000):
    w, _ = _nich()
    f = _feature(ctx, w)
    assign = np.random.default_rng(0).integers(0, 3, N).astype(np.int32)
    return f, assign


@gpu
def test_same_call_twice_is_bit_identical(ctx):
    for case in ("nich", "gp", "bnb", "bb", "dd16", "dpd_beta0", "niw8"):
        w, dists = CASES[case]()
        f = _feature(ctx, w)
        assign = np.random.default_rng(1).integers(0, len(dists), 50_000).astype(np.int32)
        a = ctx.sample_values_batch_host([f], assign, 9)[0]
        b = ctx.sample_values_batch_host([f], assign, 9)[0]
        assert np.array_equal(a.view(np.uint8), b.view(np.uint8)), case


@gpu
def test_row_shards_reproduce_one_call(ctx):
    for case in ("nich", "dpd_beta0", "niw3"):
        w, dists = CASES[case]()
        f = _feature(ctx, w)
        N, k = 100_003, 37_171
        assign = np.random.default_rng(2).integers(0, len(dists), N).astype(np.int32)
        whole = ctx.sample_values_batch_host([f], assign, 5, row0=0)[0]
        head = ctx.sample_values_batch_host([f], assign[:k], 5, row0=0)[0]
        tail = ctx.sample_values_batch_host([f], assign[k:], 5, row0=k)[0]
        assert np.array_equal(np.concatenate([head, tail]), whole), case


@gpu
def test_seed_changes_draws(ctx):
    f, assign = _mixed(ctx)
    a = ctx.sample_values_batch_host([f], assign, 1)[0]
    b = ctx.sample_values_batch_host([f], assign, 2)[0]
    assert np.mean(a == b) < 1e-3


@gpu
def test_identical_features_in_one_call_are_uncorrelated(ctx):
    w, _ = _nich()
    f1, f2 = _feature(ctx, w), _feature(ctx, w)
    assign = np.ones(DRAWS, np.int32)  # the small group: one common distribution
    a, b = ctx.sample_values_batch_host([f1, f2], assign, 3)
    r = np.corrcoef(a.astype(np.float64), b.astype(np.float64))[0, 1]
    assert abs(r) < stats.norm.isf(P_FLOOR / 2) / np.sqrt(DRAWS), r
    p = stats.ks_2samp(a, b).pvalue  # and the same distribution
    assert p > P_FLOOR


# ---- semantics --------------------------------------------------------------------------------------------------
@gpu
def test_out_of_range_rows_keep_their_values(ctx):
    for case in ("nich", "bb", "dd16", "niw3"):
        w, dists = CASES[case]()
        f = _feature(ctx, w)
        G = len(dists)
        assign = np.array([0, -1, G, 1, -7, G + 5, 1, 0] * 100, np.int32)
        bad = (assign < 0) | (assign >= G)
        dtype = capi.COLUMN_DTYPE[f.model]
        shape = (assign.size, f.dim) if f.model == capi.NIW else assign.size
        out = np.full(shape, 77, dtype)
        ctx.sample_values_batch_host([f], assign, 4, out=[out])
        assert np.all(out[bad] == 77), case
        dev_out = _dev(np.full(shape, 77, dtype))
        ctx.sample_values_batch([f], _dev(assign), assign.size, [dev_out], seed=4)
        import torch
        torch.cuda.synchronize()
        assert np.array_equal(dev_out.cpu().numpy(), out), case  # host form == device form, bit for bit


@gpu
def test_host_form_equals_device_form(ctx):
    import torch
    for case in sorted(CASES):
        w, dists = CASES[case]()
        f = _feature(ctx, w)
        assign = np.random.default_rng(6).integers(0, len(dists), 30_000).astype(np.int32)
        host = ctx.sample_values_batch_host([f], assign, 8, row0=1000)[0]
        dev_out = _dev(np.zeros_like(host))
        ctx.sample_values_batch([f], _dev(assign), assign.size, [dev_out], seed=8, row0=1000)
        torch.cuda.synchronize()
        assert np.array_equal(dev_out.cpu().numpy().view(np.uint8), host.view(np.uint8)), case


@gpu
def test_draws_follow_add_rows_on_the_same_stream(ctx):
    """add_rows_batch then sample_values on one stream, no host synchronise between: the draws see the new counts"""
    import torch
    dim = 16
    w = dict(model="dd", alphas=np.ones(dim, np.float32), counts=np.zeros((2, dim), np.int32))
    f = _feature(ctx, w)
    s = torch.cuda.Stream()
    n_add, N = 100_000, 200_000
    col = _dev(np.full(n_add, 3, np.int32))
    add_assign = _dev(np.zeros(n_add, np.int32))
    assign = _dev(np.zeros(N, np.int32))
    out = _dev(np.zeros(N, np.int32))
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ctx.add_rows_batch([f], [col], add_assign, n_add, stream=s.cuda_stream)
        ctx.sample_values_batch([f], assign, N, [out], seed=1, stream=s.cuda_stream)
    s.synchronize()
    frac = float((out.cpu().numpy() == 3).mean())
    want = (1 + n_add) / (dim + n_add)
    assert abs(frac - want) < 6 * np.sqrt(want * (1 - want) / N), (frac, want)


@gpu
def test_sampled_columns_feed_score_and_add(ctx):
    """the output columns have the exact types score_sample_batch and add_rows_batch read"""
    import torch
    feats, G = [], 3
    for case in ("nich", "gp", "bnb", "bb", "dd16", "dpd_beta0"):
        w, _ = CASES[case]()
        feats.append(_feature(ctx, w))
    N = 50_000
    assign = _dev(np.random.default_rng(7).integers(0, G, N).astype(np.int32))
    cols = [_dev(np.zeros(N, capi.COLUMN_DTYPE[f.model])) for f in feats]
    ctx.sample_values_batch(feats, assign, N, cols, seed=2)
    u = _dev(np.random.default_rng(8).random(N).astype(np.float32))
    for f, c in zip(feats, cols):
        out = _dev(np.full(N, -1, np.int32))
        ctx.score_sample_batch([f], [c], N, None, u, out)
        torch.cuda.synchronize()
        got = out.cpu().numpy()
        assert got.min() >= 0 and got.max() < G
    ctx.add_rows_batch(feats, cols, assign, N)
    torch.cuda.synchronize()
    for f in feats:
        assert f.groups == G


# ---- errors -----------------------------------------------------------------------------------------------------
@gpu
def test_errors(ctx):
    L = ctx.L
    w, _ = _nich()
    f = _feature(ctx, w)
    assign = np.zeros(4, np.int32)
    col = np.zeros(4, np.float32)
    fa = (ctypes.c_void_p * 2)(f.h.value, f.h.value)
    ca = (ctypes.c_void_p * 2)(col.ctypes.data, col.ctypes.data)
    a = assign.ctypes.data
    host = L.dist_b200_sample_values_batch_host
    assert host(None, fa, 1, a, 4, 0, 0, ca) == 1
    assert host(ctx.h, None, 1, a, 4, 0, 0, ca) == 1
    assert host(ctx.h, fa, 1, None, 4, 0, 0, ca) == 1
    assert host(ctx.h, fa, 1, a, 4, 0, 0, None) == 1
    assert host(ctx.h, fa, 0, a, 4, 0, 0, ca) == 1
    assert host(ctx.h, fa, 2, a, 4, 0, 0, (ctypes.c_void_p * 2)(col.ctypes.data, None)) == 1
    assert L.dist_b200_sample_values_batch(ctx.h, fa, 0, a, 4, 0, 0, ca, None) == 1
    g2 = _feature(ctx, dict(w, count=w["count"][:2], mean=w["mean"][:2], ctv=w["ctv"][:2]))
    assert host(ctx.h, (ctypes.c_void_p * 2)(f.h.value, g2.h.value), 2, a, 4, 0, 0, ca) == 4
    fresh = ctx.feature(capi.GP)
    out = np.zeros(4, np.uint32)
    assert host(ctx.h, (ctypes.c_void_p * 1)(fresh.h.value), 1, a, 4, 0, 0, (ctypes.c_void_p * 1)(out.ctypes.data)) == 4


# ---- mirrors ----------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["nich", "gp", "bnb", "bb", "dd", "dpd", "niw"])
def test_models_sample_values(ctx, name):
    """models.<name>.Mixture.sample_values / sample_value after add_value choreography: Value type, shape, and the
    draws of a well-filled group centre on its posterior-predictive mean"""
    from distributions_b200 import models
    model = models.MODELS[name]
    shared = model.Shared(r=3) if name == "bnb" else model.Shared()
    mixture = model.Mixture(ctx)
    rng = np.random.default_rng(len(name))
    for _ in range(2):
        g = model.Group()
        g.init(shared)
        mixture.append(g)
    mixture.init(shared)
    vals = {"nich": lambda: float(rng.normal(2.0, 1.0)), "gp": lambda: int(rng.poisson(4)), "bnb": lambda: int(rng.poisson(4)),
            "bb": lambda: bool(rng.random() < 0.8), "dd": lambda: int(rng.integers(0, 3)),
            "dpd": lambda: int(rng.integers(0, 3)), "niw": lambda: rng.normal(2.0, 1.0, shared.dim).astype(np.float32)}[name]
    added = [vals() for _ in range(400)]
    for v in added:
        mixture.add_value(shared, 1, v)
    x = mixture.sample_values(shared, np.ones(20_000, np.int32), seed=3)
    if name == "niw":
        assert x.shape == (20_000, shared.dim) and x.dtype == np.float32
        assert np.all(np.abs(x.mean(0) - np.mean(added, 0)) < 0.1)
        assert mixture.sample_value(shared, 0, seed=1).shape == (shared.dim,)
        return
    assert x.shape == (20_000,)
    assert x.dtype == {"bb": np.bool_, "nich": np.float32}.get(name, capi.COLUMN_DTYPE[mixture.model_id])
    if name in ("dd", "dpd"):
        assert set(np.unique(x)) <= {0, 1, 2} | set(range(100)) | {0xFFFFFFFF}
        assert np.mean(x < 3) > 0.9
    else:
        assert abs(float(np.mean(x.astype(np.float64))) - float(np.mean(np.asarray(added, np.float64)))) < 0.15 * (1 + abs(np.mean(added)))
    v = mixture.sample_value(shared, 0, seed=1)
    assert isinstance(v, model.Value if name != "nich" else float)


def _compile_cpp(out):
    from distributions_b200 import build
    build.build()
    lib_dir = os.path.join(ROOT, "distributions_b200", "lib")
    cmd = ["g++", "-std=c++14", "-O1", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), CPP_SRC, "-o", out,
           "-L" + lib_dir, "-ldist_b200", "-Wl,-rpath," + lib_dir]
    subprocess.run(cmd, check=True)
    return out


def test_cpp_sample_values_compiles(tmp_path):
    _compile_cpp(str(tmp_path / "test_sample_values"))


@gpu
def test_cpp_sample_values_matches_capi(ctx, tmp_path):
    exe = _compile_cpp(str(tmp_path / "test_sample_values"))
    lines = dict(l.split(" ", 1) for l in subprocess.run([exe], check=True, capture_output=True, text=True).stdout.strip().splitlines())
    got = {k: np.array(v.split(), np.int64) for k, v in lines.items()}
    gpf = _feature(ctx, dict(model="gp", shared=np.array([2, 0.5], np.float32), count=np.array([0, 20, 5], np.uint32),
                             sum=np.array([0, 190, 510], np.uint32)))
    bbf = _feature(ctx, dict(model="bb", shared=np.array([0.5, 2], np.float32), heads=np.array([0, 10, 0], np.int32),
                             tails=np.array([0, 0, 10], np.int32)))
    ids = np.array([0, 1, 2, 1, -1, 0, 3, 2], np.int32)
    gp_out = ctx.sample_values_batch_host([gpf], ids, 7, 100, out=[np.full(8, 12345, np.uint32)])[0]
    bb_out = ctx.sample_values_batch_host([bbf], ids, 7, 100, out=[np.ones(8, np.uint8)])[0]
    kind = ctx.sample_values_batch_host([gpf, bbf], ids, 7, 100, out=[np.full(8, 12345, np.uint32), np.full(8, 7, np.uint8)])
    assert np.array_equal(got["gp"], gp_out)
    assert np.array_equal(got["bb"], bb_out)
    assert np.array_equal(got["kind0"], kind[0]) and np.array_equal(got["kind1"], kind[1])
