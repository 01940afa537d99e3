"""Routes the rest of the suite does not reach, each against a plain high-precision reference of the same operation.

profiles/kernel_census.json (profiles/experiments/kernel_census.py) records which test launches which kernel; the cases
here launch the instantiations nothing else did, and both sides of the runtime fallbacks a symbol census cannot see
(a fallback lands on a kernel some other shape also launches).  The standards are the suite's:
  scores  against cases.oracle_scores within the envelopes of the test_gpu_parity.py docstring; table models bit-exact
  logp    against the float64 logsumexp L of the kernel's own materialised scores:
          |logp - L| <= 2^-21 (1 + max_g |s_ng|) + (G + 8) 2^-24   (test_gpu_score_logp.py)
  draws   identical to oracle.sample_rows on the materialised scores except proven near-ties (EPS_TIE)
  add / remove rows: integer statistics exact; nich (count, mean, ctv) against float64 sums of the rows merged with the
          stored float32 statistics by Group::merge (and its inverse): the device merges in double (merge_prep_batch_kernel)
          and rounds once to float, so |got - ref| <= 2^-24 |ref| + 2^-44 S, S the magnitude of the double terms that cancel
"""
import contextlib

import numpy as np
import pytest
from scipy import special
from scipy.special import gammaln

import cases
from distributions_b200 import synth

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

EPS_TIE = 2e-5
OPT_VALUE_CDF = 0
F32_HALF_ULP = 2.0 ** -24  # float32 rounding of a double, relative
DOUBLE_NOISE = 2.0 ** -44  # a few dozen double roundings, relative to the terms that cancel


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from distributions_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def mid(name):
    from distributions_b200 import capi
    return {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "bnb": capi.BNB}[name]


def col_dtype(name):
    from distributions_b200 import capi
    return capi.COLUMN_DTYPE[mid(name)]


def workload(name, G, n, seed, **kw):
    defaults = {"dd": dict(dim=16), "dpd": dict(V=100, other_frac=0.05), "bnb": dict(r=3)}
    return getattr(synth, name)(seed, G, n, **(kw or defaults.get(name, {})))


@contextlib.contextmanager
def options(ctx, opts):
    for k, v in opts.items():
        ctx.set_option(k, v)
    try:
        yield
    finally:
        for k in opts:
            ctx.set_option(k, 0)


def envelope(oracle, w, n):
    """per-cell model envelope of test_gpu_parity.py / test_gpu_bnb.py, [n][G] or broadcastable"""
    m = w["model"]
    if m == "nich":
        return 1e-6 * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])[None, :]
    if m == "gp":
        return 6e-7 * (1.0 + np.abs(oracle.gp_caches(w["shared"], w["count"], w["sum"])[0]))[None, :]
    if m == "bnb":
        score, post_beta, alpha = oracle.bnb_caches(w["shared"], w["count"], w["sum"])
        beta = post_beta[None, :] + w["values"][:n, None].astype(np.float64)
        return 6e-7 * (1 + np.abs(score)[None, :] + np.abs(gammaln(beta)) + np.abs(gammaln(beta + alpha[None, :])))
    return 0.0


def check_scores(oracle, ws, prior, scores, observed=None):
    """observed: per feature a bool row mask; a missing cell contributes nothing"""
    n = scores.shape[0]
    if observed is None:
        want = cases.oracle_scores(oracle, ws, n=n, prior=prior)
    else:
        want = np.tile(prior.astype(np.float32), (n, 1))
        for w, m in zip(ws, observed):
            want += np.where(m[:n, None], cases.oracle_scores(oracle, [w], n=n), np.float32(0))
    if all(w["model"] in ("dd", "dpd", "bb") for w in ws):
        assert np.array_equal(scores, want)
    else:
        env = sum(envelope(oracle, w, n) for w in ws)
        err = np.abs(scores - want) - (3e-6 * (1 + np.abs(want)) + env)
        assert np.all(err <= 0), err.max()


def check_draws(scores, u, assign, oracle):
    """draws against the oracle's sampler on the kernel's own scores: identical except proven near-ties"""
    G = scores.shape[1]
    assert assign.min() >= 0 and assign.max() < G
    a_orc = oracle.sample_rows(scores.copy(), u)
    assert cases.explained_mismatch(scores.astype(np.float64), u, assign, a_orc, EPS_TIE).all()
    # and rare, at the group counts where a rate says something: beyond ~1000 groups the near-tie bands of EPS_TIE around
    # the G - 1 CDF boundaries cover a sizeable share of the unit interval, and the per-row proof above is the check
    if G <= 1024:
        assert np.mean(assign != a_orc) <= 2e-3


def check_logp(scores, logp):
    s = scores.astype(np.float64)
    L = special.logsumexp(s, axis=1)
    bound = 2.0 ** -21 * (1.0 + np.abs(s).max(axis=1)) + (scores.shape[1] + 8) * 2.0 ** -24
    err = np.abs(logp.astype(np.float64) - L)
    assert np.all(err <= bound), (err.max(), bound[err.argmax()])


def run(ctx, ws, n, prior, u, mode, opts=None, observed=None):
    """mode 'scores': (assign, scores) of the materialising score + sample launch; 'score_only': (None, scores) of
    score_batch; 'sample': fused draws (no scores); 'logp': the row log-likelihoods.  observed: None or one bool row
    mask per feature (the *_masked entries)"""
    from distributions_b200 import capi
    feats = [ctx.feature(mid(w["model"])).update_all(w) for w in ws]
    cols = [dev(w["values"][:n].astype(col_dtype(w["model"]))) for w in ws]
    obs = None if observed is None else [capi.pack_observed(torch.from_numpy(m[:n]).cuda()) for m in observed]
    G = ws[0]["sizes"].size
    prior_d = dev(prior.astype(np.float32))
    with options(ctx, opts or {}):
        if mode == "logp":
            logp = torch.full((n,), 777.0, device="cuda")
            ctx.score_logp_batch(feats, cols, n, prior_d, logp, observed=obs)
            torch.cuda.synchronize()
            return logp.cpu().numpy()
        scores = torch.full((n, G), 777.0, device="cuda") if mode != "sample" else None
        if mode == "score_only":
            ctx.score_batch(feats, cols, n, prior_d, scores, observed=obs)
            torch.cuda.synchronize()
            return None, scores.cpu().numpy()
        assign = torch.full((n,), -5, device="cuda", dtype=torch.int32)
        ctx.score_sample_batch(feats, cols, n, prior_d, dev(u[:n].astype(np.float32)), assign, scores, observed=obs)
        torch.cuda.synchronize()
        return assign.cpu().numpy(), (scores.cpu().numpy() if scores is not None else None)


def full_check(ctx, oracle, ws, n, sample_opts=None, logp_opts=None, u=None, opts=None, observed=None):
    """scores (materialising launches: with draws and alone) against the oracle, the draws and the fused draws against
    the oracle's sampler on those scores, logp against their float64 logsumexp.  opts: options of every launch;
    sample_opts / logp_opts: added for the fused draws / the logp launch"""
    opts = opts or {}
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, ws[0]["sizes"])
    u = ws[0]["u"] if u is None else u
    assign, scores = run(ctx, ws, n, prior, u, "scores", opts, observed)
    check_scores(oracle, ws, prior, scores, observed)
    check_draws(scores, u[:n], assign, oracle)
    check_scores(oracle, ws, prior, run(ctx, ws, n, prior, u, "score_only", opts, observed)[1], observed)
    a_fused, _ = run(ctx, ws, n, prior, u, "sample", {**opts, **(sample_opts or {})}, observed)
    check_draws(scores, u[:n], a_fused, oracle)
    check_logp(scores, run(ctx, ws, n, prior, u, "logp", {**opts, **(logp_opts or {})}, observed))
    return scores


# ---- register tiles of the single-feature kernels ------------------------------------------------------------------
# logp of a row-mapped feature at 32 < G <= 64 runs score_rows_kernel<64, KIND, logp>, which the logp tests' group counts
# (1, 7, 32, 100, ...) skip; bnb takes every tier here (test_group_count_tiers covers the other models); dd / bb logp and
# sampling need VALUE_CDF = 1 to stay on the row-mapped kernel
TILE_CASES = [(m, G) for m in ("nich", "gp", "bnb", "bb", "dd") for G in (33, 50, 64)] + \
             [("bnb", G) for G in (1, 7, 32, 65, 80, 81, 96, 97, 112, 113, 128, 129, 300)]


@pytest.mark.parametrize("name,G", TILE_CASES)
def test_single_feature_tiles(ctx, oracle, name, G):
    n = 2053
    w = workload(name, G, n, 8800 + G)
    cell = {OPT_VALUE_CDF: 1} if name in ("dd", "bb") else {}
    full_check(ctx, oracle, [w], n, sample_opts=cell, logp_opts=cell)
    if name in ("dd", "bb"):  # and the defaults: the per-value tables (dd: the scaled register kernel for sampling)
        full_check(ctx, oracle, [w], n)


@pytest.mark.parametrize("G", [70, 90, 110, 128])
def test_dd_scaled_runtime_dim(ctx, oracle, G):
    """dd sampling at 64 < G <= 128 with dim != 16 (VALUE_CDF = 1 keeps it off the per-value tables): the scaled-table
    kernel with a runtime dim at every 16-group tile"""
    n = 2053
    full_check(ctx, oracle, [workload("dd", G, n, 8700 + G, dim=8)], n, opts={OPT_VALUE_CDF: 1})


OPT_SMALL_TILE, OPT_NICH_PACKED, OPT_EXP_OFFLOAD = 5, 6, 9
# the documented A/B options with scores materialised and logp as well as sampling (FUSED_VARIANTS in test_gpu_parity.py
# runs them for sampling only)
OPTION_CASES = [(m, 100, {OPT_SMALL_TILE: 1}) for m in ("nich", "gp", "bnb", "bb", "dd")] + \
               [("dd", 100, {OPT_SMALL_TILE: 2}), ("nich", 100, {OPT_NICH_PACKED: 1, OPT_SMALL_TILE: 1})] + \
               [("nich", G, {OPT_NICH_PACKED: 1}) for G in (20, 50, 100, 300)] + \
               [("nich", 300, {OPT_NICH_PACKED: 3, OPT_EXP_OFFLOAD: 5}), ("nich", 300, {OPT_NICH_PACKED: 3, OPT_EXP_OFFLOAD: 9}),
                ("nich", 300, {OPT_EXP_OFFLOAD: 7})]


OPTION_NAMES = {OPT_SMALL_TILE: "small_tile", OPT_NICH_PACKED: "nich_packed", OPT_EXP_OFFLOAD: "exp_offload"}


@pytest.mark.parametrize("case", range(len(OPTION_CASES)),
                         ids=["%s-G%d-%s" % (m, G, "-".join("%s=%d" % (OPTION_NAMES[k], v) for k, v in o.items()))
                              for m, G, o in OPTION_CASES])
def test_option_variants(ctx, oracle, case):
    name, G, opts = OPTION_CASES[case]
    n = 2053
    cell = {OPT_VALUE_CDF: 1} if name in ("dd", "bb") else {}
    full_check(ctx, oracle, [workload(name, G, n, 8600 + G + case)], n, opts={**opts, **cell})


@pytest.mark.parametrize("G", [50, 100])
def test_masked_list_tiles(ctx, oracle, G):
    """a feature list with missing cells, scores materialised: the masked 64- and 128-group tiles"""
    n = 2053
    ws = [workload("nich", G, n, 8500 + G), workload("gp", G, n, 8510 + G), workload("bb", G, n, 8520 + G)]
    for w in ws[1:]:
        w["sizes"] = ws[0]["sizes"]
    rng = np.random.default_rng(G)
    observed = [rng.random(n) < p for p in (0.7, 0.9, 0.5)]
    full_check(ctx, oracle, ws, n, observed=observed)


# ---- runtime fallbacks: both sides of every threshold ---------------------------------------------------------------
# The group counts below straddle shared-memory limits of the launchers.  The *_fits functions restate those limits from
# the library's constants, named here as in the C++ source: when one of them changes, change it here too, or the cases
# stop straddling the threshold they are named after.
NR_CHUNK, NR_THREADS, N2_ROWS = 32, 256, 4                  # nich_rows.cu: kNrChunk, kNrThreads, kN2Rows
SLOTS, SUB_GROUPS, STAGES, LGAMMA_ROW = 16, 16, 3, 8        # score_rows.cuh: kSlots, kSubGroups, kStages; numerics.cuh: kLgammaRowStride
NICH_SMEM_LIMIT, SCORE_ROWS_SMEM_LIMIT = 220 * 1024, 227 * 1024  # nich_rows.cu launch_nich_rows / launch_nich_logp; launch_variant


def nich_parameter_bytes(G):
    """nich_rows.cu: float4 parameters of every 32-group chunk + one float4 per slot of chunks"""
    nchunks = -(-G // NR_CHUNK)
    cps = -(-nchunks // SLOTS)
    return 16 * (nchunks * NR_CHUNK + -(-nchunks // cps))


def nich_rows2_fits(G):
    """launch_nich_rows (smem2): parameters + per-row slot sums of kN2Rows rows per thread"""
    return nich_parameter_bytes(G) + 4 * N2_ROWS * SLOTS * NR_THREADS <= NICH_SMEM_LIMIT


def nich_logp_fits(G):
    """launch_nich_logp: parameters and slot maxima only"""
    return nich_parameter_bytes(G) <= NICH_SMEM_LIMIT


def ksub_fits(G):
    """score_rows.cuh launch_variant<128, -1, kSub> for a list of stride-4 features at 128 threads: lgamma table rows, prior,
    sub-slot sums of every 128-group tile per thread (fixed), plus the cp.async ring of streamed caches"""
    nchunks = -(-G // 128)
    fixed = 4 * (33 * LGAMMA_ROW + 64 + 128 * nchunks) + 4 * nchunks * (128 // SUB_GROUPS + 1) * 128
    return fixed + 4 * STAGES * (128 * 4 + 128) <= SCORE_ROWS_SMEM_LIMIT


@pytest.mark.parametrize("G", [9952, 9953])
def test_nich_sampling_beyond_nich_rows2(ctx, oracle, G):
    """one nich feature, sampling only: nich_rows2_kernel up to 9952 groups; beyond, its shared memory does not fit and
    the feature-list kernel (too wide for the kSub sums too: 32-group streaming tiles) takes over"""
    assert nich_rows2_fits(G) == (G <= 9952)
    n = 1500
    full_check(ctx, oracle, [workload("nich", G, n, 8900 + G)], n)


@pytest.mark.parametrize("G", [14048, 14049])
def test_nich_logp_beyond_shared_memory(ctx, oracle, G):
    """one nich feature, logp: nich_logp_kernel up to 14048 groups, the score_rows logp tiles beyond"""
    assert nich_logp_fits(G) == (G <= 14048)
    n = 700
    w = workload("nich", G, n, 9000 + G)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    _, scores = run(ctx, [w], n, prior, w["u"], "scores")
    check_scores(oracle, [w], prior, scores)
    check_logp(scores, run(ctx, [w], n, prior, w["u"], "logp"))


@pytest.mark.parametrize("G", [5504, 5505])
def test_ksub_beyond_shared_memory(ctx, oracle, G):
    """a feature list too wide to keep resident, sampling only: the kSub kernel up to 5504 groups (43 sub-slot tiles);
    beyond, its launcher returns ERR_UNSUPPORTED and the 32-group streaming tiles take over"""
    assert ksub_fits(G) == (G <= 5504)
    n = 1200
    ws = [workload("nich", G, n, 9100 + G), workload("bb", G, n, 9200 + G)]
    ws[1]["sizes"] = ws[0]["sizes"]
    full_check(ctx, oracle, ws, n)


@pytest.mark.parametrize("cdf", [0, 1])
@pytest.mark.parametrize("G,n", [(40, 403), (40, 404), (1024, 600), (1025, 600), (4096, 600), (4097, 600)])
def test_dpd_sampling_thresholds(ctx, oracle, cdf, G, n):
    """one dpd feature (V = 100, R = 101 table rows), sampling only.  Default (cdf = 0): below 4 R rows the gather
    kernel, else the per-value guide tables (G <= 1024) or 8-ary CDF trees (G <= 4096), beyond that the gather kernel.
    VALUE_CDF = 1: table_rows_kernel for 4 R <= n and G <= 1024, the gather kernel otherwise"""
    w = workload("dpd", G, n, 9300 + G + n)
    full_check(ctx, oracle, [w], n, sample_opts={OPT_VALUE_CDF: 1} if cdf else None)


@pytest.mark.parametrize("G", [100, 200, 300, 600, 700, 800, 1000])
def test_dpd_table_rows_tiers(ctx, oracle, G):
    """VALUE_CDF = 1, sampling only: table_rows_kernel at every lane-segment width (one per 128 groups)"""
    n = 600
    full_check(ctx, oracle, [workload("dpd", G, n, 9350 + G)], n, sample_opts={OPT_VALUE_CDF: 1})


@pytest.mark.parametrize("name,n", [("dd", 63), ("dd", 64), ("bb", 7), ("bb", 8), ("dpd", 403), ("dpd", 404)])
def test_value_logp_threshold(ctx, oracle, name, n):
    """one table feature, logp: the per-value log-normaliser from 4 R rows on (dd R = dim = 16, bb R = 2, dpd R = V + 1),
    below it the row-mapped logp kernel (dd / bb) or materialise + reduce (dpd)"""
    full_check(ctx, oracle, [workload(name, 90, n, 9400 + n)], n)


# ---- add / remove rows: the global-memory and scalar-load kernels of stats.cu ---------------------------------------
# kSmem = false: more cells than the shared-memory histogram holds (dd / dpd G x dim > 12288, pooled G > 2048, counted
# groups > 12288).  kVec = false: an assign or column pointer that is not 16-byte aligned -- views offset by 1..3
# elements; the row counts are not multiples of 4, so the vector kernels' scalar tails run too.
def offset_view(a, offset):
    """a device copy of numpy array `a` that starts `offset` elements into its allocation"""
    buf = torch.empty(a.size + 3, dtype={np.int32: torch.int32, np.uint32: torch.int32, np.uint8: torch.uint8,
                                         np.float32: torch.float32}[a.dtype.type], device="cuda")
    v = buf[offset:offset + a.size]
    v.copy_(torch.from_numpy(a.view(np.int32) if a.dtype == np.uint32 else a).cuda())
    assert (v.data_ptr() % 16 == 0) == (offset == 0)
    return v


def row_setup(G, n, seed, skew=True):
    rng = np.random.default_rng(seed)
    assign = rng.integers(0, G, n).astype(np.int32)
    if skew:  # most rows in a few groups: many lanes of a warp share one
        assign = np.where(rng.random(n) < 0.6, rng.integers(0, 3, n), assign).astype(np.int32)
    assign[::11] = -1  # rows left unassigned are skipped
    observed = rng.random(n) < 0.8
    return assign, observed


def nich_merge_ref(count, mean, ctv, assign, values, sign):
    """(count, mean, ctv) after adding (sign = +1) or removing (-1) the rows, from the stored float32 statistics and
    float64 sums of the rows, by Group::merge / its inverse; and the magnitude of the double terms behind each result"""
    G = count.size
    c0, m0, v0 = count.astype(np.float64), mean.astype(np.float64), ctv.astype(np.float64)
    keep = (assign >= 0) & (assign < G)
    a, x = assign[keep], values[keep].astype(np.float64)
    m = np.bincount(a, minlength=G).astype(np.float64)
    sx = np.bincount(a, weights=x, minlength=G)
    with np.errstate(invalid="ignore", divide="ignore"):
        mb = np.where(m > 0, sx / np.maximum(m, 1), 0.0)
        vb = np.bincount(a, weights=(x - mb[a]) ** 2, minlength=G)  # two-pass: no cancellation in the reference
        sxx = np.bincount(a, weights=x * x, minlength=G)
        if sign > 0:
            tot = c0 + m
            d = mb - m0
            mean_r = np.where(m > 0, m0 + m / tot * d, m0)
            ctv_r = np.where(m > 0, v0 + vb + c0 * m / np.maximum(tot, 1) * d * d, v0)
            cnt = tot
            s_mean = np.abs(m0) + np.abs(mb)
            s_ctv = v0 + sxx + c0 * m / np.maximum(tot, 1) * d * d
        else:
            rest = c0 - m
            mean_r = np.where(rest > 0, (c0 * m0 - m * mb) / np.maximum(rest, 1), 0.0)
            d = mb - mean_r
            ctv_r = np.where(rest > 1, np.maximum(v0 - vb - rest * m / np.maximum(c0, 1) * d * d, 0.0), 0.0)
            mean_r = np.where(m > 0, mean_r, m0)
            ctv_r = np.where(m > 0, ctv_r, v0)
            cnt = np.maximum(rest, 0)
            s_mean = (c0 * np.abs(m0) + m * np.abs(mb)) / np.maximum(rest, 1)
            s_ctv = v0 + sxx + rest * m / np.maximum(c0, 1) * d * d
    return cnt.astype(np.int64), mean_r, ctv_r, s_mean, s_ctv


def download(f, name, G, dim=None):
    if name == "nich":
        raw = f.download_stats(12 * G)
        return raw[:4 * G].view(np.int32).copy(), raw[4 * G:8 * G].view(np.float32).copy(), raw[8 * G:].view(np.float32).copy()
    if name in ("gp", "bnb"):
        raw = f.download_stats(8 * G).view(np.uint32)
        return raw[:G].copy(), raw[G:].copy()
    if name == "bb":
        raw = f.download_stats(8 * G).view(np.int32)
        return raw[:G].copy(), raw[G:].copy()
    return f.download_stats(4 * G * dim).view(np.int32).reshape(G, dim).copy()


def expected_pooled(name, before, assign, values, sign):
    G = before[0].size
    keep = (assign >= 0) & (assign < G)
    a, x = assign[keep], values[keep]
    if name in ("gp", "bnb"):
        m = np.bincount(a, minlength=G).astype(np.uint32)
        s = (np.bincount(a, weights=x.astype(np.float64), minlength=G).astype(np.uint64) & 0xFFFFFFFF).astype(np.uint32)
        return (before[0] + m, before[1] + s) if sign > 0 else (before[0] - m, before[1] - s)
    heads = np.bincount(a[x != 0], minlength=G).astype(np.int32)
    tails = np.bincount(a[x == 0], minlength=G).astype(np.int32)
    return before[0] + sign * heads, before[1] + sign * tails


def check_nich(got, before, assign, values, sign):
    cnt, mean, ctv, s_mean, s_ctv = nich_merge_ref(*before, assign, values, sign)
    assert np.array_equal(got[0], cnt)
    assert np.all(np.abs(got[1] - mean) <= F32_HALF_ULP * np.abs(mean) + DOUBLE_NOISE * s_mean), np.abs(got[1] - mean).max()
    assert np.all(np.abs(got[2] - ctv) <= F32_HALF_ULP * np.abs(ctv) + DOUBLE_NOISE * s_ctv), np.abs(got[2] - ctv).max()


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("offset", [0, 1, 2, 3])
@pytest.mark.parametrize("G", [2048, 2049])
@pytest.mark.parametrize("name", ["nich", "gp", "bnb", "bb"])
def test_pooled_add_remove(ctx, oracle, name, G, offset, masked):
    """add_rows_pooled[_masked]_kernel: shared-memory accumulators up to 2048 groups, global beyond; vector and scalar
    row loads; the rows are added and then removed again"""
    from distributions_b200 import capi
    n = 4001 + offset
    w = workload(name, G, n, 9500 + G + 7 * offset)
    assign, observed = row_setup(G, n, G + offset)
    values = w["values"].astype(col_dtype(name))
    f = ctx.feature(mid(name)).update_all(w)
    a_d, c_d = offset_view(assign, offset), offset_view(values, offset)
    obs = [capi.pack_observed(torch.from_numpy(observed).cuda())] if masked else None
    eff = np.where(observed, assign, -1).astype(np.int32) if masked else assign  # a missing cell is neither added nor removed
    before = download(f, name, G)
    ctx.add_rows_batch([f], [c_d], a_d, n, observed=obs)
    torch.cuda.synchronize()
    added = download(f, name, G)
    if name == "nich":
        check_nich(added, before, eff, values, +1)
        np.testing.assert_allclose(f.download_caches(4), oracle.nich_caches(w["shared"], *added), rtol=2e-6, atol=2e-6)
    else:
        want = expected_pooled(name, before, eff, values, +1)
        assert np.array_equal(added[0], want[0]) and np.array_equal(added[1], want[1])
    ctx.remove_rows_batch([f], [c_d], a_d, n, observed=obs)
    torch.cuda.synchronize()
    removed = download(f, name, G)
    if name == "nich":
        check_nich(removed, added, eff, values, -1)
    else:
        assert np.array_equal(removed[0], before[0]) and np.array_equal(removed[1], before[1])


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("offset", [0, 1, 2, 3])
@pytest.mark.parametrize("name,G,dim", [("dd", 192, 64), ("dd", 193, 64), ("dpd", 122, 100), ("dpd", 123, 100)])
def test_count_tables_add_remove(ctx, oracle, name, G, dim, offset, masked):
    """add_rows_counts[_masked]_kernel: a shared-memory histogram up to 12288 cells of the G x dim table (dd 192 x 64,
    dpd 122 x 100 keys), global atomics beyond; counts exact"""
    from distributions_b200 import capi
    n = 3001 + offset
    kw = dict(dim=dim) if name == "dd" else dict(V=dim, other_frac=0.05)
    w = workload(name, G, n, 9600 + G + 7 * offset, **kw)
    assign, observed = row_setup(G, n, 3 * G + offset)
    values = w["values"].astype(col_dtype(name))
    f = ctx.feature(mid(name)).update_all(w)
    a_d, c_d = offset_view(assign, offset), offset_view(values, offset)
    obs = [capi.pack_observed(torch.from_numpy(observed).cuda())] if masked else None
    eff = np.where(observed, assign, -1) if masked else assign
    before = download(f, name, G, dim)
    ctx.add_rows_batch([f], [c_d], a_d, n, observed=obs)
    torch.cuda.synchronize()
    keep = eff >= 0
    rows = values[keep].astype(np.int64)
    ok = rows < dim  # dpd: OTHER (no key) is not counted; dd values are < dim
    want = before.copy()
    np.add.at(want, (eff[keep][ok], rows[ok]), 1)
    assert np.array_equal(download(f, name, G, dim), want)
    ctx.remove_rows_batch([f], [c_d], a_d, n, observed=obs)
    torch.cuda.synchronize()
    assert np.array_equal(download(f, name, G, dim), before)


@pytest.mark.parametrize("offset", [0, 1, 2, 3])
@pytest.mark.parametrize("G", [12288, 12289])
def test_count_assignments_wide(ctx, G, offset):
    """count_assignments_kernel: a shared-memory histogram up to 12288 groups, global atomics beyond; exact counts,
    overwrite and accumulate"""
    n = 5001 + offset
    assign, _ = row_setup(G, n, G + offset)
    assign[5::97] = G + 3  # out of range: not counted
    a_d = offset_view(assign, offset)
    counts = torch.full((G,), 99, device="cuda", dtype=torch.int32)
    ctx.count_assignments(a_d, n, G, counts)
    torch.cuda.synchronize()
    ok = (assign >= 0) & (assign < G)
    want = np.bincount(assign[ok], minlength=G).astype(np.int32)
    assert np.array_equal(counts.cpu().numpy(), want)
    ctx.count_assignments(a_d, n, G, counts, accumulate=True)
    torch.cuda.synchronize()
    assert np.array_equal(counts.cpu().numpy(), 2 * want)


# ---- the masked niw group histogram and the regroup relabel beyond their shared-memory tables ----------------------
# count_observed_kernel<kSmem, kVec> (stats.cu) counts the observed rows per group for the masked niw add / remove: a
# shared-memory histogram up to 12288 groups, global atomics beyond; kVec needs a 16-byte aligned assign pointer
@pytest.mark.parametrize("offset", [0, 1, 2, 3])
@pytest.mark.parametrize("G", [12288, 12289])
def test_niw_masked_add_remove_wide(ctx, G, offset):
    """masked niw add_rows / remove_rows: counts exact against np.bincount of the observed rows; sum_x and sum_xxT against
    float64 sums (the device accumulates in double and rounds once onto the float statistics: niw_apply_kernel)"""
    from distributions_b200 import capi
    d, n = 2, 5001 + offset
    w = synth.niw(9700 + G + offset, G, n, d=d)
    assign, observed = row_setup(G, n, 5 * G + offset)
    assign[7::101] = G + 2  # out of range: skipped
    f = ctx.feature(capi.NIW).update_all(w)
    vals = dev(np.ascontiguousarray(w["values"], dtype=np.float32))
    a_d = offset_view(assign, offset)
    obs = [capi.pack_observed(torch.from_numpy(observed).cuda())]

    def stats():
        raw = f.download_stats(4 * G * (1 + d + d * d))
        return (raw[:4 * G].view(np.int32).copy(), raw[4 * G:4 * G * (1 + d)].view(np.float32).reshape(G, d).astype(np.float64),
                raw[4 * G * (1 + d):].view(np.float32).reshape(G, d, d).astype(np.float64))

    def check(got, base, sign):
        keep = observed & (assign >= 0) & (assign < G)
        a, x = assign[keep], w["values"][keep].astype(np.float64)
        cnt = base[0] + sign * np.bincount(a, minlength=G).astype(np.int32)
        assert np.array_equal(got[0], cnt)
        for k, term in ((1, x), (2, x[:, :, None] * x[:, None, :])):
            want, mag = base[k].copy(), np.abs(base[k])
            np.add.at(want, a, sign * term)
            np.add.at(mag, a, np.abs(term))
            want = np.where((cnt == 0).reshape((G,) + (1,) * (want.ndim - 1)), 0.0, want)  # an emptied group is reset
            assert np.all(np.abs(got[k] - want) <= F32_HALF_ULP * np.abs(want) + DOUBLE_NOISE * mag), k

    before = stats()
    ctx.add_rows_batch([f], [vals], a_d, n, observed=obs)
    torch.cuda.synchronize()
    added = stats()
    check(added, before, +1)
    ctx.remove_rows_batch([f], [vals], a_d, n, observed=obs)
    torch.cuda.synchronize()
    check(stats(), added, -1)


@pytest.mark.parametrize("G", [12288, 12289])
def test_regroup_relabel_wide(ctx, G):
    """clustering-only regroup (regroup.cu launch_regroup_relabel): the old -> new table in shared memory up to 12288
    groups (48 KB), read from global memory beyond; against the numpy reference of tests/regroup_ref.py"""
    import regroup_ref as ref
    rng = np.random.default_rng(G)
    sizes = rng.integers(1, 60, G).astype(np.int32)
    sizes[rng.random(G) < 0.3] = 0
    assign = rng.integers(-1, G + 1, 40_003).astype(np.int32)
    rm, counts, G_want = ref.remap(sizes, 2)
    a_dev, co = dev(assign), torch.zeros(G + 2, device="cuda", dtype=torch.int32)
    assert ctx.regroup_batch([], dev(sizes), G, 2, a_dev, assign.size, co) == G_want
    assert np.array_equal(a_dev.cpu().numpy(), ref.relabel(assign, rm))
    assert np.array_equal(co.cpu().numpy()[:G_want], counts)
