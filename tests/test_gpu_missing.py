"""Missing cells: the *_masked entries with per-feature observed masks (dist_b200.h, "missing cells").

The rules are checked against the library's unmasked entries, which the parity suites hold to the oracle:
  - scores[n][g] = prior[g] + sum_f bit_f[n] * score_f(x_f[n]; g), with score_f from an unmasked score_batch of feature f
    alone; a missing cell holds NaN / an out-of-range value and is never read for arithmetic;
  - a masked draw is the stand-alone sampler's draw on those scores, near-ties excepted; logp is their logsumexp;
  - masked add / remove = the unmasked entries applied per feature to that feature's observed rows only;
  - imputation = where(observed, input column, the unmasked call's draws), bit for bit;
  - and against the oracle: masked scores = prior + sum_f bit_f * oracle.score_rows (single dd / bb / dpd features
    bit-exact), draws against the oracle sampler, N = 1 / 31 / 33 (partial warps and mask words), and one masked Gibbs
    step (remove, score + sample, add, sizes, prior) against the same steps on the oracle / numpy side;
  - with every mask NULL the entries are the unmasked ones (bit-identical), with all-ones words the same within the
    parity tolerance.
CPU tests (no mark): pack_observed against a direct bit loop.
"""
import numpy as np
import pytest
from scipy import special

import cases
from distributions_b200 import capi, synth

gpu = pytest.mark.gpu
MODEL_ID = {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW, "bnb": capi.BNB}
# a value no kernel may use: NaN for the continuous models, far out of range for the discrete ones
JUNK = {"nich": np.float32(np.nan), "niw": np.float32(np.nan), "gp": np.uint32(0xFFFFFFF0), "bnb": np.uint32(0xFFFFFFF0),
        "dd": np.int32(1 << 30), "dpd": np.uint32(0x7FFFFFFF), "bb": np.uint8(255)}


def _bits(mask):
    words = np.zeros((mask.size + 31) // 32, dtype=np.uint32)
    for n, b in enumerate(mask):
        if b:
            words[n // 32] |= np.uint32(1) << np.uint32(n % 32)
    return words


@pytest.mark.parametrize("n", [1, 31, 32, 33, 64, 1000, 1025])
def test_pack_observed_layout(n):
    m = np.random.default_rng(n).random(n) < 0.6
    assert np.array_equal(capi.pack_observed(m), _bits(m))
    assert capi.pack_observed(m).dtype == np.uint32


def test_pack_observed_torch():
    torch = pytest.importorskip("torch")
    m = np.random.default_rng(5).random(77) < 0.5
    t = capi.pack_observed(torch.from_numpy(m))
    assert isinstance(t, torch.Tensor)
    assert np.array_equal(t.numpy().view(np.uint32), _bits(m))


MASKED_ENTRIES = ["dist_b200_score_batch_masked", "dist_b200_score_sample_batch_masked", "dist_b200_score_logp_batch_masked",
                  "dist_b200_add_rows_batch_masked", "dist_b200_remove_rows_batch_masked", "dist_b200_rows_accumulate_masked",
                  "dist_b200_sample_values_batch_masked"]


def test_masked_symbols_exported():
    """the library exports every masked entry, and the binding declares each with one argument more than its unmasked
    form (the observed-mask array)"""
    import ctypes
    from distributions_b200 import build
    lib = ctypes.CDLL(build.build())
    for name in MASKED_ENTRIES:
        assert hasattr(lib, name), name
        plain = name[:-len("_masked")]
        assert len(capi.SIGNATURES[name][1]) == len(capi.SIGNATURES[plain][1]) + 1, name


# ---- on the device -------------------------------------------------------------------------------------------------
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
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a).cuda()


def _workload(model, G, N, seed, d=3):
    if model == "dd":
        return synth.dd(seed, G, N, dim=16)
    if model == "dpd":
        return synth.dpd(seed, G, N, V=100, other_frac=0.1)
    if model == "niw":
        return synth.niw(seed, G, N, d=d)
    return getattr(synth, model)(seed, G, N)


def _list(models, G, N, seed):
    ws = [_workload(m, G, N, seed + i) for i, m in enumerate(models)]
    for w in ws[1:]:
        w["sizes"] = ws[0]["sizes"]
    return ws


def _column(w):
    return np.ascontiguousarray(w["values"].astype(capi.COLUMN_DTYPE[MODEL_ID[w["model"]]]))


def _masks(ws, N, rate, seed, all_missing_rows=()):
    """bool [F][N] observed masks at missing rate `rate` (per feature), rows in all_missing_rows missing everywhere"""
    rng = np.random.default_rng(seed)
    obs = rng.random((len(ws), N)) >= rate
    obs[:, list(all_missing_rows)] = False
    return obs


def _junked(w, obs):
    c = _column(w).copy()
    c[~obs] = JUNK[w["model"]]
    return c


def _features(ctx, ws):
    return [ctx.feature(MODEL_ID[w["model"]]).update_all(w) for w in ws]


def _prior(ctx, sizes):
    return ctx.prior_pitman_yor_host(synth.PY_ALPHA, synth.PY_D, np.asarray(sizes, np.int32))


def _feature_scores(ctx, feats, ws, N):
    """unmasked score_batch of every feature alone, no prior: [F][N][G] float32"""
    import torch
    G = feats[0].groups
    out = []
    for f, w in zip(feats, ws):
        s = torch.empty((N, G), device="cuda", dtype=torch.float32)
        ctx.score_batch([f], [_dev(_column(w))], N, None, s)
        out.append(s.cpu().numpy())
    return np.stack(out)


def _expected(prior, fs, obs):
    return prior.astype(np.float64)[None, :] + (fs.astype(np.float64) * obs[:, :, None]).sum(axis=0)


def _tol(fs, obs, prior):
    """fp32 accumulation of F + 1 terms, each already within the parity tolerance of its own entry"""
    mag = np.abs(prior.astype(np.float64))[None, :] + (np.abs(fs.astype(np.float64)) * obs[:, :, None]).sum(axis=0)
    return 4e-6 * (1.0 + mag)


def _run_masked(ctx, feats, cols, obs_words, N, prior, u):
    import torch
    G = feats[0].groups
    prior_d = _dev(prior)
    scores = torch.empty((N, G), device="cuda", dtype=torch.float32)
    ctx.score_batch(feats, cols, N, prior_d, scores, observed=obs_words)
    assign = torch.full((N,), -7, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch(feats, cols, N, prior_d, _dev(u), assign, observed=obs_words)
    logp = torch.empty((N,), device="cuda", dtype=torch.float32)
    ctx.score_logp_batch(feats, cols, N, prior_d, logp, observed=obs_words)
    torch.cuda.synchronize()
    return scores.cpu().numpy(), assign.cpu().numpy(), logp.cpu().numpy()


def _lse_bound(expected):
    G = expected.shape[1]
    fin = np.where(np.isfinite(expected), np.abs(expected), 0.0).max(axis=1)
    return 2.0 ** -21 * (1.0 + fin) + (G + 8) * 2.0 ** -24


ROUTES = [  # (feature models, G): fused lists at every tile tier and kSub, single features, dpd / niw, mixed lists
    (["nich"], 20), (["gp"], 100), (["bnb"], 300), (["bb"], 64), (["dd"], 1024),
    (["nich", "gp", "bb", "dd", "bnb"], 20), (["nich", "gp", "bb", "dd", "bnb"], 100),
    (["nich", "gp", "bb", "dd", "bnb"] * 3, 256), (["nich", "gp", "bb", "dd"] * 40, 256), (["nich", "gp", "bb", "dd"] * 40, 1024),
    (["dpd"], 37), (["niw"], 20), (["nich", "dpd", "gp", "niw"], 100), (["dpd", "niw", "dd"], 256),
]


def _route_id(r):
    return "%s-G%d" % ("+".join(sorted(set(r[0]))) + ("x%d" % len(r[0]) if len(r[0]) > 1 else ""), r[1])


@gpu
@pytest.mark.parametrize("route", ROUTES, ids=_route_id)
@pytest.mark.parametrize("rate", [0.0, 0.3, 1.0])
def test_masked_against_per_feature_scores(ctx, route, rate):
    """every route, including niw (which the oracle scores apart), against the library's unmasked per-feature scores"""
    import torch
    models, G = route
    N = 1000 if len(models) > 20 else 2333  # (not a multiple of any row tile)
    ws = _list(models, G, N, 4000 + G)
    feats = _features(ctx, ws)
    prior = _prior(ctx, ws[0]["sizes"])
    obs = _masks(ws, N, rate, 11 + G, all_missing_rows=(0, 5, N - 1))
    cols = [_dev(_junked(w, o)) for w, o in zip(ws, obs)]
    words = [_dev(capi.pack_observed(o)) for o in obs]
    u = np.random.default_rng(G).random(N).astype(np.float32)
    fs = _feature_scores(ctx, feats, ws, N)
    exp = _expected(prior, fs, obs)
    scores, assign, logp = _run_masked(ctx, feats, cols, words, N, prior, u)
    what = "%s G=%d rate=%.1f" % (_route_id(route), G, rate)
    err = np.abs(scores.astype(np.float64) - exp)
    tol = _tol(fs, obs, prior)
    assert (err <= tol).all(), "%s: scores worst %.3g" % (what, (err - tol).max())
    # rows with every feature missing score the prior alone, exactly
    for r in (0, 5, N - 1):
        assert np.array_equal(scores[r], prior), what
    # draws: the stand-alone sampler on the float64 expectation, near-ties excepted
    ref = torch.empty(N, device="cuda", dtype=torch.int32)
    ctx.sample_from_scores(_dev(exp.astype(np.float32)), N, G, _dev(u), ref)
    ref = ref.cpu().numpy()
    assert ((assign >= 0) & (assign < G)).all(), what
    ok = cases.explained_mismatch(exp, u, assign, ref, 1e-4)
    assert ok.all(), "%s: %d unexplained draws" % (what, (~ok).sum())
    # logp: logsumexp of the expected scores; an all-missing row gives logsumexp(prior)
    L = special.logsumexp(exp, axis=1)
    bound = _lse_bound(exp) + 2.0 ** -20 * (1.0 + np.abs(L))
    assert (np.abs(logp.astype(np.float64) - L) <= bound).all(), what
    lp = special.logsumexp(prior.astype(np.float64))
    assert abs(float(logp[0]) - lp) <= 1e-5 * (1 + abs(lp)), what


@gpu
@pytest.mark.parametrize("route", ROUTES, ids=_route_id)
def test_null_and_all_ones_masks(ctx, route):
    """NULL masks: the unmasked entries, bit for bit.  All-ones words: the masked kernels, same scores within tolerance"""
    import torch
    models, G = route
    N = 1000 if len(models) > 20 else 3001
    ws = _list(models, G, N, 5000 + G)
    feats = _features(ctx, ws)
    prior = _prior(ctx, ws[0]["sizes"])
    cols = [_dev(_column(w)) for w in ws]
    u = np.random.default_rng(G + 1).random(N).astype(np.float32)
    prior_d, u_d = _dev(prior), _dev(u)
    s0 = torch.empty((N, G), device="cuda", dtype=torch.float32)
    a0 = torch.empty(N, device="cuda", dtype=torch.int32)
    l0 = torch.empty(N, device="cuda", dtype=torch.float32)
    ctx.score_batch(feats, cols, N, prior_d, s0)
    ctx.score_sample_batch(feats, cols, N, prior_d, u_d, a0)
    ctx.score_logp_batch(feats, cols, N, prior_d, l0)
    s0, a0, l0 = s0.cpu().numpy(), a0.cpu().numpy(), l0.cpu().numpy()
    s, a, lp = _run_masked(ctx, feats, cols, [None] * len(ws), N, prior, u)
    assert np.array_equal(s, s0) and np.array_equal(a, a0) and np.array_equal(lp, l0)
    ones = [_dev(capi.pack_observed(np.ones(N, bool))) for _ in ws]
    s, a, lp = _run_masked(ctx, feats, cols, ones, N, prior, u)
    assert np.allclose(s, s0, rtol=1e-6, atol=1e-5)
    ok = cases.explained_mismatch(s0.astype(np.float64), u, a, a0, 1e-4)
    assert ok.all(), "%d unexplained draws" % (~ok).sum()
    assert np.allclose(lp, l0, rtol=1e-6, atol=1e-5)


@gpu
@pytest.mark.parametrize("d", [3, 32, 64])
def test_niw_masked(ctx, d):
    """niw alone and beside a nich feature at d = 3 / 32 / 64 (generic route: one masked [N][G] pass per feature)"""
    import torch
    N, G = 1500, 40
    ws = [synth.niw(70 + d, G, N, d=d), synth.nich(71 + d, G, N)]
    ws[1]["sizes"] = ws[0]["sizes"]
    feats = _features(ctx, ws)
    prior = _prior(ctx, ws[0]["sizes"])
    obs = _masks(ws, N, 0.3, d, all_missing_rows=(3,))
    cols = [_dev(_junked(w, o)) for w, o in zip(ws, obs)]
    words = [_dev(capi.pack_observed(o)) for o in obs]
    fs = _feature_scores(ctx, feats, ws, N)
    for k in (1, 2):
        exp = _expected(prior, fs[:k], obs[:k])
        s = torch.empty((N, G), device="cuda", dtype=torch.float32)
        ctx.score_batch(feats[:k], cols[:k], N, _dev(prior), s, observed=words[:k])
        err = np.abs(s.cpu().numpy().astype(np.float64) - exp)
        assert (err <= _tol(fs[:k], obs[:k], prior) * 10).all(), "niw d=%d k=%d worst %.3g" % (d, k, err.max())


@gpu
def test_feature_missing_everywhere_is_left_out(ctx):
    """a feature missing in every row: the logp of the list without it"""
    import torch
    N, G = 2000, 70
    ws = _list(["nich", "gp", "dd"], G, N, 77)
    feats = _features(ctx, ws)
    prior = _prior(ctx, ws[0]["sizes"])
    obs = np.ones((3, N), bool)
    obs[1] = False
    cols = [_dev(_junked(w, o)) for w, o in zip(ws, obs)]
    lp = torch.empty(N, device="cuda", dtype=torch.float32)
    ctx.score_logp_batch(feats, cols, N, _dev(prior), lp, observed=[None, _dev(capi.pack_observed(obs[1])), None])
    ref = torch.empty(N, device="cuda", dtype=torch.float32)
    ctx.score_logp_batch([feats[0], feats[2]], [cols[0], cols[2]], N, _dev(prior), ref)
    assert np.allclose(lp.cpu().numpy(), ref.cpu().numpy(), rtol=2e-6, atol=2e-6)


def _stats(f):
    return f.download_stats(1 << 24)


def _same_stats(a, b, model, rtol=1e-5, atol=1e-4):
    """integer statistics exact; float ones (nich / niw sums) within tolerance.  Words that are not normal floats (the
    integer counts) must match exactly."""
    if model not in ("nich", "niw"):
        return np.array_equal(a, b)
    fa, fb = a.view(np.float32), b.view(np.float32)
    ints = np.abs(fa) < 1e-30
    return np.array_equal(a.view(np.uint32)[ints], b.view(np.uint32)[ints]) and np.allclose(fa, fb, rtol=rtol, atol=atol)


@gpu
@pytest.mark.parametrize("models", [["nich", "gp", "bnb", "bb", "dd", "dpd"], ["niw"], ["nich", "niw", "dd", "nich"]])
def test_add_remove_masked(ctx, models):
    """masked add = per feature the unmasked add of its observed rows; masked remove restores the statistics"""
    N, G = 5000, 30
    ws = _list(models, G, N, 900)
    obs = _masks(ws, N, 0.4, 3)
    assign = np.random.default_rng(4).integers(-1, G, N).astype(np.int32)
    feats = _features(ctx, ws)
    before = [_stats(f) for f in feats]
    cols = [_dev(_junked(w, o)) for w, o in zip(ws, obs)]
    words = [_dev(capi.pack_observed(o)) if i % 3 != 2 else None for i, o in enumerate(obs)]
    obs_eff = [o if wd is not None else np.ones(N, bool) for o, wd in zip(obs, words)]
    ctx.add_rows_batch(feats, [c if wd is not None else _dev(_column(w)) for c, w, wd in zip(cols, ws, words)],
                       _dev(assign), N, observed=words)
    got = [_stats(f) for f in feats]
    refs = _features(ctx, ws)
    for f, w, o in zip(refs, ws, obs_eff):
        ctx.add_rows_batch([f], [_dev(_column(w)[o])], _dev(assign[o]), int(o.sum()))
    for i, (g, f) in enumerate(zip(got, refs)):
        assert _same_stats(g, _stats(f), models[i]), models[i]  # (float sums: same rows, maybe another order)
    ctx.remove_rows_batch(feats, [c if wd is not None else _dev(_column(w)) for c, w, wd in zip(cols, ws, words)],
                          _dev(assign), N, observed=words)
    for i, (f, b) in enumerate(zip(feats, before)):
        assert _same_stats(_stats(f), b, models[i], rtol=1e-4, atol=1e-3), models[i]


@gpu
def test_rows_exchange_masked(ctx):
    """two row shards accumulated with masks, summed and merged = one masked add"""
    import torch
    N, G = 4000, 25
    ws = _list(["nich", "dd", "gp", "niw", "bb"], G, N, 31)
    obs = _masks(ws, N, 0.35, 8)
    assign = np.random.default_rng(9).integers(0, G, N).astype(np.int32)
    cols = [_junked(w, o) for w, o in zip(ws, obs)]
    half = 1700
    one = _features(ctx, ws)
    ctx.add_rows_batch(one, [_dev(c) for c in cols], _dev(assign), N, observed=[_dev(capi.pack_observed(o)) for o in obs])
    two = _features(ctx, ws)
    n_x = ctx.rows_xchg_doubles(two)
    total = torch.zeros(n_x, device="cuda", dtype=torch.float64)
    for lo, hi in ((0, half), (half, N)):
        x = torch.zeros(n_x, device="cuda", dtype=torch.float64)
        ctx.rows_accumulate(two, [_dev(c[lo:hi]) for c in cols], _dev(assign[lo:hi]), hi - lo, x,
                            observed=[_dev(capi.pack_observed(o[lo:hi])) for o in obs])
        torch.cuda.synchronize()
        total += x
    ctx.rows_merge(two, total)
    for i, (a, b) in enumerate(zip(one, two)):
        assert _same_stats(_stats(a), _stats(b), ws[i]["model"]), ws[i]["model"]


@gpu
@pytest.mark.parametrize("d", [3, 32, 100])
def test_imputation_where_identity(ctx, d):
    """masked output = where(observed, input, unmasked draws) bit for bit, for all seven models"""
    import torch
    N, G = 3000, 17
    models = ["nich", "gp", "bnb", "bb", "dd", "dpd", "niw"]
    ws = [_workload(m, G, N, 60 + i, d=d) for i, m in enumerate(models)]
    for w in ws[1:]:
        w["sizes"] = ws[0]["sizes"]
    feats = _features(ctx, ws)
    obs = _masks(ws, N, 0.3, 21)
    assign = np.random.default_rng(3).integers(-2, G + 2, N).astype(np.int32)  # invalid ids included
    inputs = [_column(w) for w in ws]
    ref = [_dev(np.zeros_like(c)) for c in inputs]
    ctx.sample_values_batch(feats, _dev(assign), N, ref, seed=99, row0=12345)
    out = [_dev(c.copy()) for c in inputs]
    ctx.sample_values_batch(feats, _dev(assign), N, out, seed=99, row0=12345,
                            observed=[_dev(capi.pack_observed(o)) for o in obs])
    torch.cuda.synchronize()
    valid = (assign >= 0) & (assign < G)
    for m, c, r, o, ob in zip(models, inputs, ref, out, obs):
        r, o = r.cpu().numpy().view(c.dtype), o.cpu().numpy().view(c.dtype)
        write = (~ob) & valid
        if c.ndim == 2:
            write = write[:, None]
        expect = np.where(write, r, c)
        assert np.array_equal(expect.view(np.uint8), o.view(np.uint8)), m


# ---- against the oracle ------------------------------------------------------------------------------------------
EPS_TIE = 2e-5


def _envelope(oracle, w, values):
    """[n][G] fast_log / lgamma slack of the parity suites (test_gpu_parity.envelope, test_gpu_bnb.envelope)"""
    n, G = values.shape[0], w["sizes"].size
    if w["model"] == "nich":
        e = 1e-6 * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])
    elif w["model"] == "gp":
        e = 6e-7 * (1.0 + np.abs(oracle.gp_caches(w["shared"], w["count"], w["sum"])[0]))
    elif w["model"] == "bnb":
        score, post_beta, alpha = oracle.bnb_caches(w["shared"], w["count"], w["sum"])
        beta = post_beta[None, :] + values[:, None].astype(np.float64)
        return 6e-7 * (1 + np.abs(score)[None, :] + np.abs(special.gammaln(beta)) + np.abs(special.gammaln(beta + alpha[None, :])))
    else:
        e = np.zeros(G)
    return np.broadcast_to(e[None, :], (n, G))


def _oracle_masked(oracle, ws, obs, prior):
    """the oracle's scores of the masked rows in the kernel's order: prior, then every feature left to right on its
    observed rows only (float32, as the oracle adds); plus the float64 sum of |terms| for the tolerance"""
    N, G = obs.shape[1], prior.size
    s32 = np.repeat(prior[None, :].astype(np.float32), N, axis=0)
    mag = np.repeat(np.abs(prior[None, :]).astype(np.float64), N, axis=0)
    env = np.zeros((N, G))
    for w, o in zip(ws, obs):
        if not o.any():
            continue
        vals = w["values"][o]
        if w["model"] == "dpd":
            vals = cases.dpd_rows(w, vals)
        t = np.zeros((int(o.sum()), G), np.float32)
        oracle.score_rows(cases.MODEL_ID[w["model"]], cases.oracle_caches(oracle, w), vals, t)
        s32[o] += t
        mag[o] += np.abs(t)
        env[o] += _envelope(oracle, w, w["values"][o])
    return s32, mag, env


ORACLE_ROUTES = [  # row-mapped features and dpd (the oracle scores niw apart; niw is covered against the library above)
    (["dd"], 29), (["bb"], 100), (["dpd"], 37), (["nich"], 64), (["gp"], 300), (["bnb"], 20),
    (["nich", "gp", "bb", "dd", "bnb"], 45), (["nich", "gp", "bb", "dd"] * 40, 256), (["nich", "dpd", "gp", "dd"], 130),
]


@gpu
@pytest.mark.parametrize("route", ORACLE_ROUTES, ids=_route_id)
@pytest.mark.parametrize("N", [1, 31, 33, 2333])
@pytest.mark.parametrize("rate", [0.0, 0.3, 1.0])
def test_masked_against_oracle(ctx, oracle, route, N, rate):
    """expected score = prior + sum_f bit_f * oracle.score_rows(model_f, ...); single dd / bb / dpd features bit-exact,
    the rest within the parity tolerance; draws against the oracle sampler, logp against float64 logsumexp"""
    models, G = route
    ws = _list(models, G, max(N, 64), 7000 + G)
    for w in ws:
        w["values"] = w["values"][:N]
    feats = _features(ctx, ws)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, ws[0]["sizes"]).astype(np.float32)
    obs = _masks(ws, N, rate, 31 + N + G, all_missing_rows=(0, N - 1) if N > 2 else ())
    cols = [_dev(_junked(w, o)) for w, o in zip(ws, obs)]
    words = [_dev(capi.pack_observed(o)) for o in obs]
    u = np.random.default_rng(N + G).random(N).astype(np.float32)
    scores, assign, logp = _run_masked(ctx, feats, cols, words, N, prior, u)
    want, mag, env = _oracle_masked(oracle, ws, obs, prior)
    what = "%s N=%d rate=%.1f" % (_route_id(route), N, rate)
    if len(models) == 1 and models[0] in ("dd", "bb", "dpd"):
        assert np.array_equal(scores, want), what  # table gathers: bit-exact, as unmasked
    else:
        err = np.abs(scores.astype(np.float64) - want)
        tol = 5e-6 * (1.0 + mag) + env
        assert (err <= tol).all(), "%s: worst excess %.3g" % (what, (err - tol).max())
    if N > 2:
        assert np.array_equal(scores[0], prior) and np.array_equal(scores[N - 1], prior), what
    a_orc = oracle.sample_rows(scores.copy(), u)  # the oracle's sampler on the kernel's scores: near-ties only
    assert cases.explained_mismatch(scores.astype(np.float64), u, assign, a_orc, EPS_TIE).all(), what
    L = special.logsumexp(want.astype(np.float64), axis=1)
    bound = _lse_bound(want.astype(np.float64)) + (5e-6 * (1.0 + mag) + env).max(axis=1)
    assert (np.abs(logp.astype(np.float64) - L) <= bound).all(), what


def _np_update(w, vals, a, o, sign):
    """Group::add_value / remove_value of the observed rows in numpy (integer statistics: exact)"""
    def add_at(arr, idx, v):  # (modular for unsigned statistics, as the device's integer atomics)
        np.add.at(arr, idx, np.broadcast_to(np.asarray(v, np.int64), g.shape).astype(arr.dtype))

    G = w["sizes"].size
    ok = o & (a >= 0) & (a < G)
    g, x = a[ok], vals[ok].astype(np.int64)
    if w["model"] == "dd":
        add_at(w["counts"], (g, x), sign)
    elif w["model"] == "bb":
        add_at(w["heads"], g, sign * x)
        add_at(w["tails"], g, sign * (1 - x))
    else:  # gp
        add_at(w["count"], g, sign)
        add_at(w["sum"], g, sign * x)


@gpu
def test_masked_gibbs_step_against_oracle(ctx, oracle):
    """one masked Gibbs step on the device -- remove, score + sample, add, group sizes, prior -- against the same steps
    on the oracle / numpy side on the same masked data (the numpy side follows the device's draws, so a near-tie does
    not make the two chains diverge)"""
    import copy
    import torch
    N, G = 4001, 24
    ws = _list(["dd", "bb", "gp", "dd", "bb"], G, N, 321)
    obs = _masks(ws, N, 0.3, 17, all_missing_rows=(9,))
    cols = [_dev(_junked(w, o)) for w, o in zip(ws, obs)]
    words = [_dev(capi.pack_observed(o)) for o in obs]
    feats = _features(ctx, ws)
    ref = copy.deepcopy(ws)
    a0 = np.random.default_rng(5).integers(0, G, N).astype(np.int32)
    ctx.add_rows_batch(feats, cols, _dev(a0), N, observed=words)  # the rows' current assignment
    for w, o in zip(ref, obs):
        _np_update(w, w["values"], a0, o, +1)
    # remove
    ctx.remove_rows_batch(feats, cols, _dev(a0), N, observed=words)
    for w, o in zip(ref, obs):
        _np_update(w, w["values"], a0, o, -1)
    # score + sample under the prior of the remaining sizes (the synthetic sizes)
    sizes = np.asarray(ws[0]["sizes"], np.int32)
    prior_d = torch.empty(G, device="cuda", dtype=torch.float32)
    ctx.prior_pitman_yor_dev(synth.PY_ALPHA, synth.PY_D, G, _dev(sizes), prior_d)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, sizes).astype(np.float32)
    assert np.allclose(prior_d.cpu().numpy(), prior, rtol=1e-6, atol=1e-6)
    u = np.random.default_rng(6).random(N).astype(np.float32)
    a1 = torch.empty(N, device="cuda", dtype=torch.int32)
    sc = torch.empty((N, G), device="cuda", dtype=torch.float32)
    ctx.score_sample_batch(feats, cols, N, _dev(prior), _dev(u), a1, scores=sc, observed=words)
    a1, sc = a1.cpu().numpy(), sc.cpu().numpy()
    want, mag, env = _oracle_masked(oracle, ref, obs, prior)
    assert (np.abs(sc.astype(np.float64) - want) <= 5e-6 * (1.0 + mag) + env).all()
    a_orc = oracle.sample_rows(want.copy(), u)
    assert cases.explained_mismatch(want.astype(np.float64), u, a1, a_orc, 1e-4).all()
    # add under the new assignment
    ctx.add_rows_batch(feats, cols, _dev(a1), N, observed=words)
    for w, o in zip(ref, obs):
        _np_update(w, w["values"], a1, o, +1)
    # sizes, prior
    counts = torch.empty(G, device="cuda", dtype=torch.int32)
    ctx.count_assignments(_dev(a1), N, G, counts)
    sizes1 = np.bincount(a1, minlength=G).astype(np.int32)
    assert np.array_equal(counts.cpu().numpy(), sizes1)
    ctx.prior_pitman_yor_dev(synth.PY_ALPHA, synth.PY_D, G, counts, prior_d)
    prior1 = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, sizes1).astype(np.float32)
    assert np.allclose(prior_d.cpu().numpy(), prior1, rtol=1e-6, atol=1e-6)
    # the statistics after the step: every feature's scores of all rows against the oracle on the numpy statistics
    full = np.ones((len(ws), N), bool)
    for i, (f, w) in enumerate(zip(feats, ref)):
        s = torch.empty((N, G), device="cuda", dtype=torch.float32)
        ctx.score_batch([f], [_dev(_column(ws[i]))], N, None, s)
        s = s.cpu().numpy()
        want, mag, env = _oracle_masked(oracle, [w], full[:1], np.zeros(G, np.float32))
        if w["model"] in ("dd", "bb"):
            assert np.array_equal(s, want), w["model"]
        else:
            assert (np.abs(s.astype(np.float64) - want) <= 5e-6 * (1.0 + mag) + env).all(), w["model"]
