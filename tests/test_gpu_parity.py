"""GPU parity tests proper: the CUDA path (through the C-ABI) against the oracle restatement on the
same seeded inputs, against the committed golden vectors of the compiled reference, and -- where
oracle/_ref travelled to the box -- against the live unmodified reference.

Stated tolerances (see tests/test_oracle.py for the measured origins):
  scores  |cuda - oracle| <= 3e-6 * (1 + |ref|) + model envelope, where the envelope is
          nich: 1e-6 * |log_coeff[g]|  (MUFU.LG2 vs the table entry: <= 2^-22 in log2)
          gp  : 6e-7 * (1 + |score[g]|) (fp32 cancellation of score[g] + lgamma(post_alpha+v))
          dd / dpd / bb: none (table gathers are bit-exact: tolerance 0)
  vs the compiled reference add LOG_STEP * |log_coeff[g]| for nich (fast_log is a step function; the
  -ffast-math build may evaluate its argument one ulp away).
  assignments: identical to the oracle's for the same uniforms except near-ties, i.e. rows where
          u * total lies within eps * total of a CDF boundary between the two indices, eps = 2e-5
          (fast_exp's build envelope 5e-6 + summation order); the mismatch rate is also bounded.
"""
import numpy as np
import pytest

import cases
from distributions_b200 import synth

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

LOG_STEP = 6.2e-5
EPS_TIE = 2e-5


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


def model_id(name):
    from distributions_b200 import capi
    return {"dd": capi.DD, "dpd": capi.DPD, "bb": capi.BB, "gp": capi.GP, "nich": capi.NICH, "niw": capi.NIW, "bnb": capi.BNB}[name]


def envelope(oracle, w):
    G = w["sizes"].size
    if w["model"] == "nich":
        return 1e-6 * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])
    if w["model"] == "gp":
        return 6e-7 * (1.0 + np.abs(oracle.gp_caches(w["shared"], w["count"], w["sum"])[0]))
    return np.zeros(G)


# every kernel variant behind the fused (sampling-only) entry: dist_b200_option settings
FUSED_VARIANTS = {
    "default": {},                                  # per-value CDF trees for single dpd / dd / bb, packed nich, ...
    "value_cdf_tree": {0: 2},                       # per-value CDFs searched as 8-ary trees (default: guide-table walk)
    "row_tile_32": {1: 32},                         # G > 128: 32-group tiles + slots everywhere (also instead of the kSub streaming kernel)
    "no_value_cdf": {0: 1},                         # per-cell kernels: table_rows (dpd), score_rows (dd / bb)
    "table_rows_walk_in_loop": {0: 1, 4: 2},        # dpd G in (384, 512]: every lane walks inside the row loop (default: the owner's walk staged)
    "table_rows_all_mufu": {0: 1, 9: 1},            # dpd G in (384, 512]: every exp2 on the MUFU pipe
    "round1_gather": {0: 1, 4: 1},                  # dpd: round-1 warp-per-row gather kernel
    "small_tile_256": {0: 1, 5: 1},                 # 64 < G <= 128: one 256-thread block / SM
    "small_tile_4x32": {0: 1, 5: 3},                # 64 < G <= 128: four 32-group tiles
    "nich_scalar": {6: 1},                          # nich: scalar loop instead of packed fp32x2
    "nich_packed_one_row": {6: 2},                  # nich: packed loop, one row per thread (default: two rows for G > 128)
    "nich_online_max_two_rows": {6: 3},             # nich G > 128: the two-row kernel with per-tile maxima (default: static reference, four rows)
    "nich_online_max_mufu": {6: 3, 9: 1},           # ... every exp2 on the MUFU pipe
    "nich_exp_all_mufu": {9: 1},                    # nich G > 128: every softmax exp2 on the MUFU pipe
    "nich_exp_offload_4": {9: 5},                   # ... 4 of 16 pairs on the FMA pipe (polynomial)
    "nich_exp_offload_8": {9: 9},                   # ... 8 of 16
}


def check_fused_variants(ctx, feats_w, prior, u, n, scores, assign):
    """the sampling-only launches (scores never materialised) must agree with the materialising launch on the same
    rows: every index identical or a proven near-tie on the kernel's own scores, and rare"""
    for name, opts in FUSED_VARIANTS.items():
        for k, v in opts.items():
            ctx.set_option(k, v)
        try:
            a2, _ = run_cuda(ctx, feats_w, prior, u, n, want_scores=False)
        finally:
            for k in opts:
                ctx.set_option(k, 0)
        assert a2.min() >= 0 and a2.max() < scores.shape[1], name
        diff = np.nonzero(a2 != assign)[0]
        assert diff.size <= max(2, 2e-3 * n), (name, diff.size)
        if diff.size:
            assert cases.explained_mismatch(scores[diff].astype(np.float64), u[:n][diff], assign[diff], a2[diff], EPS_TIE).all(), name


def run_cuda(ctx, feats_w, prior, u, n, want_scores=True, sample=True):
    """score (+sample) the first n rows of the workloads through the device-pointer C-ABI."""
    feats = [ctx.feature(model_id(w["model"])).update_all(w) for w in feats_w]
    cols = [dev(w["values"][:n].astype(__import__("distributions_b200.capi", fromlist=["x"]).COLUMN_DTYPE[model_id(w["model"])])) for w in feats_w]
    G = feats_w[0]["sizes"].size
    prior_d = dev(prior.astype(np.float32)) if prior is not None else None
    scores_d = torch.full((n, G), 777.0, device="cuda", dtype=torch.float32) if want_scores else None
    if sample:
        u_d = dev(u[:n].astype(np.float32))
        assign_d = torch.full((n,), -5, device="cuda", dtype=torch.int32)
        ctx.score_sample_batch(feats, cols, n, prior_d, u_d, assign_d, scores_d)
        torch.cuda.synchronize()
        return assign_d.cpu().numpy(), (scores_d.cpu().numpy() if want_scores else None)
    ctx.score_batch(feats, cols, n, prior_d, scores_d)
    torch.cuda.synchronize()
    return None, scores_d.cpu().numpy()


# ------------------------------------------------------------------------------------ numerics
def test_numerics_device_functions(ctx, oracle):
    sweeps = {
        0: np.concatenate([np.logspace(-37, 38, 200001), -np.logspace(-5, 5, 1001), [0.0, np.inf]]),
        2: np.logspace(-3, 9.6, 200001),
        3: np.logspace(-3, 9.6, 200001),
        5: np.concatenate([np.logspace(0, 30, 200001), 1 + np.logspace(-7, 0, 50001), [np.finfo(np.float32).max]]),
        6: np.logspace(-3, 9.6, 200001),
    }
    tol = {0: 0.0, 2: 1e-6, 3: 2e-6, 5: 5e-7, 6: 1e-6}
    orc_fn = {0: 0, 2: 2, 3: 3, 5: 0, 6: 2}
    for fn, x in sweeps.items():
        x = x.astype(np.float32)
        xd = dev(x)
        out = torch.empty_like(xd)
        ctx.numerics_probe(fn, xd, out, x.size)
        torch.cuda.synchronize()
        got = out.cpu().numpy().astype(np.float64)
        want = oracle.vec(orc_fn[fn], x).astype(np.float64)
        err = np.abs(got - want) / (1 + np.abs(want))
        err = np.where(got == want, 0.0, err)
        assert err.max() <= tol[fn], (fn, err.max(), x[np.argmax(err)])
    # the per-cell log needs a finite argument (DESIGN §4): at inf it gives inf, where the table gives 128 ln 2
    xd = dev(np.array([np.inf], np.float32))
    out = torch.empty_like(xd)
    ctx.numerics_probe(5, xd, out, 1)
    assert out.cpu().numpy()[0] == np.inf
    # fast_exp on the sampler's domain: relative to the restated fmath::exp
    x = np.linspace(-87.0, 0.0, 200001).astype(np.float32)
    xd = dev(x)
    out = torch.empty_like(xd)
    ctx.numerics_probe(1, xd, out, x.size)
    got = out.cpu().numpy().astype(np.float64)
    want = oracle.fast_exp(x).astype(np.float64)
    # x * log2(e) is rounded once at magnitude |x| * 1.44: the relative error grows with |x| (the
    # reference's own (x + 1) - r*b re-association has the same shape, 5e-6 at x = -87)
    assert np.all(np.abs(got - want) / want <= 5e-7 + 1.2e-7 * np.abs(x))
    # log factorial
    n = np.concatenate([np.arange(0, 300), [1000, 65535, 1 << 20]]).astype(np.uint32)
    xd = dev(n.view(np.float32))
    out = torch.empty_like(xd)
    ctx.numerics_probe(4, xd, out, n.size)
    np.testing.assert_allclose(out.cpu().numpy(), oracle.fast_log_factorial(n), rtol=1e-6)


def test_numerics_poly_ex2(ctx):
    """fn 7, poly_ex2_pair (the sampling kernels' exp2 on the FMA pipe) against float64 exp2: relative 2.21e-7 over every
    fp32 in [-1, -2^-30] (every fractional part x - round(x) the range reduction can produce, at full resolution; below
    2^-30 the polynomial is 1 to within an ulp) and on a grid of [-125, 0], exact powers of two at integers, exactly 2^-125
    below the clamp"""
    bits = torch.arange(0xB0800000 - 2 ** 32, 0xBF800000 - 2 ** 32 + 1, device="cuda", dtype=torch.int64).to(torch.int32)
    xe = bits.view(torch.float32)
    ye = torch.empty_like(xe)
    ctx.numerics_probe(7, xe, ye, xe.numel())
    torch.cuda.synchronize()
    err = (ye.double() / torch.exp2(xe.double()) - 1).abs()
    assert float(err.max()) <= 2.21e-7, (float(err.max()), float(xe[int(torch.argmax(err))]))
    del bits, xe, ye, err
    x = np.concatenate([np.linspace(-125.0, 0.0, 2000001), -np.logspace(-30, 0, 10001), [0.0, -0.5, 0.5 - 1.0]]).astype(np.float32)
    ints = np.arange(-125, 1).astype(np.float32)
    below = np.array([-125.5, -126.0, -150.0, -1e30, -np.inf], np.float32)
    xa = np.concatenate([x, ints, below])
    xd = dev(xa)
    out = torch.empty_like(xd)
    ctx.numerics_probe(7, xd, out, xa.size)
    torch.cuda.synchronize()
    got = out.cpu().numpy().astype(np.float64)
    g_x, g_i, g_b = got[:x.size], got[x.size:x.size + ints.size], got[x.size + ints.size:]
    err = np.abs(g_x / np.exp2(x.astype(np.float64)) - 1)
    assert err.max() <= 2.21e-7, (err.max(), x[np.argmax(err)])
    assert np.array_equal(g_i, np.exp2(ints.astype(np.float64)))
    assert np.all(g_b == 2.0 ** -125)


def test_prior(ctx, oracle, golden):
    for j in range(5):
        for empties in (1, 10):
            key = "prior_%d_%d" % (j, empties)
            sizes = golden[key + "_sizes"]
            alpha, d = [float(v) for v in golden[key + "_alpha_d"]]
            out = torch.zeros(sizes.size, device="cuda")
            ctx.prior_pitman_yor(alpha, d, sizes, out)
            torch.cuda.synchronize()
            got = out.cpu().numpy()
            assert np.array_equal(got, oracle.py_prior(alpha, d, sizes))  # same table, same op order
            np.testing.assert_allclose(got, golden[key + "_out"], atol=2e-6, rtol=0)


CACHE_ROWS = {"nich": 4, "gp": 3, "bb": 2}


@pytest.mark.parametrize("name", list(cases.SMALL))
def test_caches(ctx, oracle, golden, name):
    w = cases.make(name, **cases.SMALL[name])
    f = ctx.feature(model_id(name)).update_all(w)
    want = cases.oracle_caches(oracle, w)
    if name in CACHE_ROWS:
        got = f.download_caches(CACHE_ROWS[name])
        np.testing.assert_allclose(got, want, rtol=2e-6, atol=2e-6)
        np.testing.assert_allclose(got, golden["%s_caches" % name], rtol=3e-6, atol=3e-6)
    elif name == "dd":
        got = f.download_caches(w["alphas"].size)          # score_value_group table [dim][G]
        assert np.array_equal(got, want[:-1] - want[-1][None, :])
    else:
        got = f.download_caches(w["keys"].size + 1)        # [V+1][G], last row = OTHER
        assert np.array_equal(got, want[:-1] - want[-1][None, :])


# ------------------------------------------------------------------------------ single features
@pytest.mark.parametrize("name", list(cases.SMALL))
def test_single_feature_golden_and_oracle(ctx, oracle, golden, name):
    cfg = cases.SMALL[name]
    w = cases.make(name, **cfg)
    n = cfg["N"]
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    u = golden["%s_u" % name]
    assign, scores = run_cuda(ctx, [w], prior, u, n)
    want = cases.oracle_scores(oracle, [w], prior=prior)
    env = envelope(oracle, w)[None, :]
    if name in ("dd", "dpd", "bb"):
        assert np.array_equal(scores, want)
    else:
        assert np.all(np.abs(scores - want) <= 3e-6 * (1 + np.abs(want)) + env)
    # against the compiled reference's outputs
    ref_scores = golden["%s_scores" % name]
    step = LOG_STEP * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])[None, :] if name == "nich" else 0.0
    assert np.all(np.abs(scores - ref_scores) <= 4e-6 * (1 + np.abs(ref_scores)) + env + step)
    # assignments: vs the oracle sampler on the CUDA scores, and vs the reference's indices
    a_orc = oracle.sample_rows(scores.copy(), u)
    assert cases.explained_mismatch(scores.astype(np.float64), u, assign, a_orc, EPS_TIE).all()
    a_ref = golden["%s_assign" % name]
    ok = cases.explained_mismatch(ref_scores.astype(np.float64), u, assign, a_ref, 2e-3 if name == "nich" else EPS_TIE)
    assert ok.all()
    assert np.mean(assign == a_ref) > 0.95
    # fused (no materialised scores) gives the same indices as the materialising launch
    check_fused_variants(ctx, [w], prior, u, n, scores, assign)


@pytest.mark.parametrize("name", list(cases.SMALL))
def test_accumulate_semantic(ctx, oracle, golden, name):
    """Mixture.score_value ADDS into the buffer (reference test_models.py:552-557)."""
    from distributions_b200 import capi
    w = cases.make(name, **cases.SMALL[name])
    noise = golden["%s_noise" % name]
    f = ctx.feature(model_id(name)).update_all(w)
    col = dev(w["values"][:8].astype(capi.COLUMN_DTYPE[model_id(name)]))
    sc = dev(noise)
    ctx.score_batch([f], [col], 8, None, sc, accumulate=True)
    torch.cuda.synchronize()
    got = sc.cpu().numpy()
    want = golden["%s_accum" % name]
    env = envelope(oracle, w)[None, :]
    step = LOG_STEP * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])[None, :] if name == "nich" else 0.0
    assert np.all(np.abs(got - want) <= 4e-6 * (1 + np.abs(want)) + env + step)
    # == per-group Group::score_value at the reference's own tolerance
    row0 = got[0] - noise[0]
    gs = golden["%s_group_scores" % name]
    assert np.all(np.abs(row0 - gs) <= 1e-3 * (1 + np.abs(row0) + np.abs(gs)))
    # per-value host entry (MixtureSlave::score_value drop-in)
    acc = noise[0].copy()
    ctx.score_value_host(f, w["values"][:1], acc)
    np.testing.assert_array_equal(acc, got[0])


@pytest.mark.parametrize("G", [1, 2, 31, 32, 33, 64, 70, 90, 100, 110, 128, 129, 257, 1000])
@pytest.mark.parametrize("name", ["nich", "gp", "bb", "dd"])
def test_group_count_tiers(ctx, oracle, name, G):
    """ragged group counts across every register-tile / multi-chunk tier, ragged row counts"""
    n = 517
    w = cases.make(name, seed=1000 + G, G=G, N=n)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = run_cuda(ctx, [w], prior, w["u"], n)
    want = cases.oracle_scores(oracle, [w], prior=prior)
    env = envelope(oracle, w)[None, :]
    assert np.all(np.abs(scores - want) <= 3e-6 * (1 + np.abs(want)) + env)
    a_orc = oracle.sample_rows(scores.copy(), w["u"])
    assert cases.explained_mismatch(scores.astype(np.float64), w["u"], assign, a_orc, EPS_TIE).all()
    assert np.mean(assign == a_orc) > 0.98
    check_fused_variants(ctx, [w], prior, w["u"], n, scores, assign)
    assert assign.min() >= 0 and assign.max() < G


@pytest.mark.parametrize("G,V", [(19, 100), (512, 4096), (77, 1000)])
def test_dpd_tiers(ctx, oracle, G, V):
    n = 1031
    w = synth.dpd(2000 + G, G, n, V=V, other_frac=0.05)
    if V == 1000:  # sparse, shuffled keys: device-side key search
        rng = np.random.default_rng(1)
        keys = rng.choice(1 << 20, V, replace=False).astype(np.uint32)
        known = w["values"] != 0xFFFFFFFF
        w["values"][known] = keys[w["values"][known]]
        w["keys"] = keys
        w["values"][:5] = [3, 5, 7, 11, 13][:5]  # (almost surely) unknown values -> the OTHER row
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = run_cuda(ctx, [w], prior, w["u"], n)
    want = cases.oracle_scores(oracle, [w], prior=prior)
    assert np.array_equal(scores, want)
    a_orc = oracle.sample_rows(scores.copy(), w["u"])
    assert cases.explained_mismatch(scores.astype(np.float64), w["u"], assign, a_orc, EPS_TIE).all()
    check_fused_variants(ctx, [w], prior, w["u"], n, scores, assign)


@pytest.mark.parametrize("name,G,kw", [("dpd", 512, dict(V=4096, other_frac=0.02)), ("dpd", 100, dict(V=37, other_frac=0.3)),
                                       ("dd", 100, dict(dim=16)), ("dd", 600, dict(dim=40)), ("bb", 128, {}), ("bb", 5, {})])
def test_table_features_at_scale(ctx, oracle, name, G, kw):
    """single table features (dpd at the c4 shape, dd at the c1 shape, bb) over enough rows that every warp of
    the register kernel / the per-value CDF search runs many iterations incl. a ragged last one: scores bit-exact
    against the oracle on a block, every fused variant against the materialised scores of ALL rows"""
    n = 100_003
    w = getattr(synth, name)(3100 + G, G, n, **kw)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = run_cuda(ctx, [w], prior, w["u"], n)
    blk = slice(n - 3000, n)
    wb = dict(w)
    wb["values"] = w["values"][blk]
    want = cases.oracle_scores(oracle, [wb], prior=prior)
    assert np.array_equal(scores[blk], want)
    a_orc = oracle.sample_rows(scores[blk].copy(), w["u"][blk])
    assert cases.explained_mismatch(scores[blk].astype(np.float64), w["u"][blk], assign[blk], a_orc, EPS_TIE).all()
    check_fused_variants(ctx, [w], prior, w["u"], n, scores, assign)
    # u = 0 and u -> 1 pick the first / last group carrying mass on every path
    u_edge = np.where(np.arange(n) % 2 == 0, 0.0, np.nextafter(np.float32(1), np.float32(0))).astype(np.float32)
    a_e, s_e = run_cuda(ctx, [w], prior, u_edge, n)
    check_fused_variants(ctx, [w], prior, u_edge, n, s_e, a_e)


# ------------------------------------------------------------------------------------ cross-cat
def _crosscat_small():
    G, N = 17, 64
    cc = synth.crosscat(201, G, N, n_gp=3, n_bb=3)
    extra = []
    for f in range(2):
        w = synth.nich(300 + f, G, N)
        w["count"] = cc["sizes"].copy()
        w["mean"][cc["sizes"] == 0] = 0
        w["ctv"][cc["sizes"] == 0] = 0
        extra.append(w)
    return cc, cc["features"] + extra


def test_crosscat_golden(ctx, oracle, golden):
    cc, feats = _crosscat_small()
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, cc["sizes"])
    u = golden["crosscat_u"]
    assign, scores = run_cuda(ctx, feats, prior, u, 64)
    want = cases.oracle_scores(oracle, feats, prior=prior)
    env = sum(envelope(oracle, w) for w in feats)[None, :]
    assert np.all(np.abs(scores - want) <= 4e-6 * (1 + np.abs(want)) + env)
    ref_scores = golden["crosscat_scores"]
    step = sum(LOG_STEP * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1]) for w in feats[-2:])[None, :]
    assert np.all(np.abs(scores - ref_scores) <= 5e-6 * (1 + np.abs(ref_scores)) + env + step)
    a_orc = oracle.sample_rows(scores.copy(), u)
    assert cases.explained_mismatch(scores.astype(np.float64), u, assign, a_orc, EPS_TIE).all()


@pytest.mark.parametrize("G,F", [(128, 24), (200, 10), (300, 12), (1000, 8)])
def test_crosscat_streaming(ctx, oracle, G, F):
    """enough features that the group caches do not fit in shared memory (double-buffered staging)"""
    n = 700
    cc = synth.crosscat(500 + G, G, n, n_gp=F // 2, n_bb=F // 2)
    feats = cc["features"]
    # widen the caches with dd features so the resident budget is exceeded
    for k in range(6):
        w = synth.dd(900 + k, G, n, dim=32)
        feats.append(w)
    if G > 128:  # a nich member: the generic per-cell branch of the sub-slot re-score (G > 128: kSub kernel)
        w = synth.nich(950, G, n)
        w["count"] = cc["sizes"].astype(w["count"].dtype)
        w["mean"][cc["sizes"] == 0] = 0
        w["ctv"][cc["sizes"] == 0] = 0
        feats.append(w)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, cc["sizes"])
    assign, scores = run_cuda(ctx, feats, prior, cc["u"], n)
    want = cases.oracle_scores(oracle, feats, prior=prior)
    env = sum(envelope(oracle, w) for w in feats)[None, :]
    assert np.all(np.abs(scores - want) <= 5e-6 * (1 + np.abs(want)) + env)
    a_orc = oracle.sample_rows(scores.copy(), cc["u"])
    assert cases.explained_mismatch(scores.astype(np.float64), cc["u"], assign, a_orc, EPS_TIE).all()
    check_fused_variants(ctx, feats, prior, cc["u"], n, scores, assign)


def test_mixed_dpd_and_rows(ctx, oracle):
    """a dpd feature next to row-mapped features: materialise + accumulate + stand-alone sampler"""
    G, n = 40, 333
    w1 = synth.nich(71, G, n)
    w2 = synth.dpd(72, G, n, V=64, other_frac=0.1)
    w2["sizes"] = w1["sizes"]
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w1["sizes"])
    assign, scores = run_cuda(ctx, [w1, w2], prior, w1["u"], n)
    want = cases.oracle_scores(oracle, [w1, w2], prior=prior)
    assert np.all(np.abs(scores - want) <= 4e-6 * (1 + np.abs(want)) + envelope(oracle, w1)[None, :])
    a_orc = oracle.sample_rows(scores.copy(), w1["u"])
    assert cases.explained_mismatch(scores.astype(np.float64), w1["u"], assign, a_orc, EPS_TIE).all()


# -------------------------------------------------------------------------------------- sampler
@pytest.mark.parametrize("G", [1, 2, 5, 100, 1024])
def test_sampler_golden(ctx, golden, G):
    s = golden["sampler_%d_scores" % G]
    u = golden["sampler_%d_u" % G]
    want = golden["sampler_%d_assign" % G]
    out = torch.full((s.shape[0],), -1, device="cuda", dtype=torch.int32)
    ctx.sample_from_scores(dev(s), s.shape[0], G, dev(u), out)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    assert cases.explained_mismatch(s.astype(np.float64), u, got, want, EPS_TIE).all()
    assert np.mean(got == want) >= 0.95


def test_sampler_large_vs_oracle_and_distribution(ctx, oracle):
    rng = np.random.default_rng(9)
    n, G = 200000, 333
    base = (rng.standard_normal((1000, G)) * 2).astype(np.float32)
    s = np.ascontiguousarray(base.repeat(200, axis=0))  # 1000 distinct rows x 200 draws each
    u = rng.random(n, dtype=np.float32)
    out = torch.empty(n, device="cuda", dtype=torch.int32)
    ctx.sample_from_scores(dev(s), n, G, dev(u), out)
    torch.cuda.synchronize()
    got = out.cpu().numpy()
    want = oracle.sample_rows(s.copy(), u)
    assert cases.explained_mismatch(s.astype(np.float64), u, got, want, EPS_TIE).all()
    assert np.mean(got != want) < 2e-4
    # the draws follow softmax(scores): chi-square style check on one row's 200 draws pooled over rows
    p = np.exp(base.astype(np.float64) - base.max(1, keepdims=True))
    p /= p.sum(1, keepdims=True)
    hits = np.zeros(1000)
    for r in range(1000):
        hits[r] = p[r, got[r * 200:(r + 1) * 200]].mean()
    assert abs(hits.mean() - (p ** 2).sum(1).mean()) < 5e-3


# ----------------------------------------------------------------------------------- properties
def test_full_size_properties_nich(ctx, oracle):
    """BASELINE config 2 at full size (1M rows x 1024 groups): size-independent properties --
    indices in range; a shifted prior (+c on every group) leaves every index unchanged; rows with a
    dominant group pick it; a spot-check block against the oracle."""
    from distributions_b200 import capi
    G, n = 1024, 1_000_000
    w = synth.nich(20242, G, n)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    f = ctx.feature(capi.NICH).update_all(w)
    col, u_d = dev(w["values"]), dev(w["u"])
    a1 = torch.empty(n, device="cuda", dtype=torch.int32)
    a2 = torch.empty(n, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch([f], [col], n, dev(prior), u_d, a1)
    ctx.score_sample_batch([f], [col], n, dev(prior + np.float32(0.5)), u_d, a2)
    torch.cuda.synchronize()
    a1, a2 = a1.cpu().numpy(), a2.cpu().numpy()
    assert a1.min() >= 0 and a1.max() < G
    assert np.mean(a1 != a2) < 1e-4  # softmax shift invariance (up to rounding near-ties)
    blk = slice(500000, 500000 + 2048)
    sc = cases.oracle_scores(oracle, [dict(w, values=w["values"][blk])], prior=prior)
    want = oracle.sample_rows(sc.copy(), w["u"][blk])
    ok = cases.explained_mismatch(sc.astype(np.float64), w["u"][blk], a1[blk], want, 1e-4)
    assert ok.all()
    assert np.mean(a1[blk] == want) > 0.99


def test_host_entry(ctx, oracle):
    n, G = 3000, 50
    w = synth.nich(5, G, n)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    from distributions_b200 import capi
    f = ctx.feature(capi.NICH).update_all(w)
    assign, scores = ctx.score_sample_batch_host([f], [w["values"]], prior, w["u"], want_scores=True)
    a_dev, s_dev = run_cuda(ctx, [w], prior, w["u"], n)
    assert np.array_equal(assign, a_dev) and np.array_equal(scores, s_dev)


def test_update_group_add_remove_group(ctx, oracle):
    """update_group / add_group / remove_group keep the device caches equal to a fresh update_all
    (MixtureSlave::add_value / add_group / remove_group choreography, mixture.hpp:361-398)."""
    from distributions_b200 import capi
    G = 9
    w = synth.nich(11, G, 10)
    f = ctx.feature(capi.NICH).update_all(w)
    # mutate group 3 on the host (Group::add_value restated in the oracle), refresh just that group
    c, m, v = oracle.nich_group_update(+1, int(w["count"][3]), float(w["mean"][3]), float(w["ctv"][3]), [1.25, -0.5])
    rec = np.zeros(1, dtype=[("c", np.int32), ("m", np.float32), ("v", np.float32)])
    rec[0] = (c, m, v)
    f.update_group(3, rec)
    w2 = dict(w, count=w["count"].copy(), mean=w["mean"].copy(), ctv=w["ctv"].copy())
    w2["count"][3], w2["mean"][3], w2["ctv"][3] = c, m, v
    want = oracle.nich_caches(w2["shared"], w2["count"], w2["mean"], w2["ctv"])
    np.testing.assert_allclose(f.download_caches(4), want, rtol=2e-6, atol=2e-6)
    # add an empty group, then remove group 2 (swap-with-last)
    f.add_group()
    assert f.groups == G + 1
    w3 = dict(w2, count=np.append(w2["count"], 0).astype(np.int32), mean=np.append(w2["mean"], 0).astype(np.float32),
              ctv=np.append(w2["ctv"], 0).astype(np.float32))
    np.testing.assert_allclose(f.download_caches(4), oracle.nich_caches(w3["shared"], w3["count"], w3["mean"], w3["ctv"]), rtol=2e-6, atol=2e-6)
    f.remove_group(2)
    assert f.groups == G
    for k in ("count", "mean", "ctv"):
        a = w3[k].copy()
        a[2] = a[-1]
        w3[k] = a[:-1]
    np.testing.assert_allclose(f.download_caches(4), oracle.nich_caches(w3["shared"], w3["count"], w3["mean"], w3["ctv"]), rtol=2e-6, atol=2e-6)


def test_error_codes(ctx):
    from distributions_b200 import capi
    f = ctx.feature(capi.NICH)
    with pytest.raises(capi.DistB200Error):  # no update_all yet -> ERR_STATE, not a crash
        ctx.score_batch([f], [torch.zeros(4, device="cuda")], 4, None, torch.zeros(4, device="cuda"))
    w1, w2 = synth.nich(1, 5, 4), synth.nich(2, 6, 4)
    f1, f2 = ctx.feature(capi.NICH).update_all(w1), ctx.feature(capi.NICH).update_all(w2)
    with pytest.raises(capi.DistB200Error):  # features disagree on G
        ctx.score_batch([f1, f2], [dev(w1["values"]), dev(w2["values"])], 4, None, torch.zeros(4 * 5, device="cuda"))


# ------------------------------------------------------------------------------------------ NIW
def _niw_cuda(ctx, w, n, prior, sample=True, extra=None):
    from distributions_b200 import capi
    f = ctx.feature(capi.NIW).update_all(w)
    feats, cols = [f], [dev(np.ascontiguousarray(w["values"][:n], dtype=np.float32))]
    if extra is not None:
        feats.append(ctx.feature(model_id(extra["model"])).update_all(extra))
        cols.append(dev(extra["values"][:n].astype(capi.COLUMN_DTYPE[model_id(extra["model"])])))
    G = w["sizes"].size
    scores = torch.full((n, G), 555.0, device="cuda")
    assign = torch.full((n,), -3, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch(feats, cols, n, dev(prior), dev(w["u"][:n]), assign, scores)
    torch.cuda.synchronize()
    return assign.cpu().numpy(), scores.cpu().numpy()


def _niw_tol(w, want):
    d = w["mu"].size
    dof = w["nu"] + w["count"].astype(np.float64) - d + 1.0
    coef3 = 0.5 * (dof + d)
    # fast_log step envelope (the argument 1 + q/dof is built from a whitened sum of squares here, from
    # sigma^-1 in the oracle: last-bit differences move it across table steps) + fp32 accumulation
    return 2e-5 * (1 + np.abs(want)) + LOG_STEP * coef3[None, :]


@pytest.mark.parametrize("d,G", [(2, 9), (3, 40), (8, 33), (32, 9), (32, 70)])
def test_niw_vs_oracle(ctx, oracle, d, G):
    n = 301
    w = synth.niw(600 + d + G, G, n, d=d)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = _niw_cuda(ctx, w, n, prior)
    want = np.tile(prior, (n, 1)).astype(np.float32)
    oracle.niw_score_rows(w["mu"], w["kappa"], w["psi"], w["nu"], w["count"], w["sum_x"], w["sum_xxT"], w["values"][:n], want)
    assert np.all(np.abs(scores - want) <= _niw_tol(w, want))
    assert np.mean(np.abs(scores - want) <= 2e-5 * (1 + np.abs(want))) > 0.9
    a_orc = oracle.sample_rows(scores.copy(), w["u"][:n])
    assert cases.explained_mismatch(scores.astype(np.float64), w["u"][:n], assign, a_orc, EPS_TIE).all()
    assert assign.min() >= 0 and assign.max() < G


@pytest.mark.parametrize("d,G", [(1, 40), (2, 9), (3, 64), (4, 300), (5, 33), (8, 256)])
def test_niw_small_d_fused(ctx, oracle, d, G):
    """d <= 8, sampling only: niw_rows_kernel (scores never materialised, static softmax reference) against the oracle's
    sampler on the materialising route's scores -- every mismatch a near-tie -- incl. a ragged last tile, rows far
    from every group (re-evaluated with their own maximum) and the materialising route selected by option"""
    from distributions_b200 import capi
    n = 20_011
    w = synth.niw(700 + d + G, G, n, d=d)
    w["values"] = w["values"].copy()
    w["values"][::7] *= 300.0  # outliers to every group
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = _niw_cuda(ctx, w, n, prior)
    a_orc = oracle.sample_rows(scores.copy(), w["u"][:n])
    assert cases.explained_mismatch(scores.astype(np.float64), w["u"][:n], assign, a_orc, EPS_TIE).all()
    f = ctx.feature(capi.NIW).update_all(w)
    col, u_d, prior_d = dev(np.ascontiguousarray(w["values"], dtype=np.float32)), dev(w["u"]), dev(prior)
    for path in (0, 1):
        ctx.set_option(capi.OPT_NIW_PATH, path)
        try:
            a_f = torch.full((n,), -3, device="cuda", dtype=torch.int32)
            ctx.score_sample_batch([f], [col], n, prior_d, u_d, a_f, None)
            torch.cuda.synchronize()
        finally:
            ctx.set_option(capi.OPT_NIW_PATH, 0)
        a_f = a_f.cpu().numpy()
        assert a_f.min() >= 0 and a_f.max() < G
        diff = np.nonzero(a_f != assign)[0]
        assert diff.size <= max(2, 2e-3 * n), (path, diff.size)
        if diff.size:
            assert cases.explained_mismatch(scores[diff].astype(np.float64), w["u"][:n][diff], assign[diff], a_f[diff], EPS_TIE).all(), path


@pytest.fixture(scope="module")
def golden_niw():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "niw_golden.npz"))


@pytest.mark.parametrize("name", cases.NIW_GOLDEN_CASES)
def test_niw_golden_reference_python(ctx, oracle, golden_niw, name):
    """CUDA NIW against fixtures produced by the reference's own exact-math Python (dbg/models/niw.py +
    dbg/random.py, imported by tests/golden/make_golden_niw.py): EXAMPLES of dims 2 / 3 / 4 on the FP32 kernel,
    d = 32 on the tcgen05 kernel.  Same three checks that pin the oracle (cases.check_niw_golden)."""
    from distributions_b200 import capi
    c = cases.niw_golden_case(golden_niw, name)
    f = ctx.feature(capi.NIW).update_all(c)

    def score(c, values):
        n = values.shape[0]
        sc = torch.full((n, c["count"].size), 321.0, device="cuda")
        ctx.score_batch([f], [dev(np.ascontiguousarray(values, np.float32))], n, None, sc)
        torch.cuda.synchronize()
        return sc.cpu().numpy()

    cases.check_niw_golden(score, oracle, c)


def test_niw_c5_scale(ctx, oracle):
    """The c5 shape (d = 32, G = 256) at N = 320 000: every CTA of the tensor-core kernel runs many work items,
    the operand rings and TMEM buffers wrap hundreds of times.  A 2 048-row block from the middle of the batch is
    compared with the oracle, every assignment of the batch against the sampler run on the kernel's own scores,
    and the fused (scores not materialised) launch against the materialising one."""
    from distributions_b200 import capi
    d, G, n = 32, 256, 320_000
    w = synth.niw(20245, G, n, d=d)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    f = ctx.feature(capi.NIW).update_all(w)
    col, u_d, prior_d = dev(w["values"]), dev(w["u"]), dev(prior)
    scores = torch.full((n, G), 555.0, device="cuda")
    assign = torch.full((n,), -3, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch([f], [col], n, prior_d, u_d, assign, scores)
    assign_fused = torch.full((n,), -3, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch([f], [col], n, prior_d, u_d, assign_fused, None)
    torch.cuda.synchronize()
    a, a_fused, sc = assign.cpu().numpy(), assign_fused.cpu().numpy(), scores.cpu().numpy()
    assert a.min() >= 0 and a.max() < G and a_fused.min() >= 0 and a_fused.max() < G
    for lo in (0, 163_840 - 1024, n - 2048):  # first rows, a block straddling row-chunk boundaries, the ragged tail
        blk = slice(lo, lo + 2048)
        want = np.tile(prior, (2048, 1)).astype(np.float32)
        oracle.niw_score_rows(w["mu"], w["kappa"], w["psi"], w["nu"], w["count"], w["sum_x"], w["sum_xxT"],
                              np.ascontiguousarray(w["values"][blk]), want)
        assert np.all(np.abs(sc[blk] - want) <= _niw_tol(w, want)), lo
        assert np.mean(np.abs(sc[blk] - want) <= 2e-5 * (1 + np.abs(want))) > 0.9
        a_orc = oracle.sample_rows(sc[blk].copy(), w["u"][blk])
        assert cases.explained_mismatch(sc[blk].astype(np.float64), w["u"][blk], a[blk], a_orc, EPS_TIE).all(), lo
    # the whole batch: fused vs materialising launch -- every mismatch a proven near-tie on the kernel's scores
    diff = np.nonzero(a != a_fused)[0]
    assert diff.size <= 2e-4 * n, diff.size
    if diff.size:
        assert cases.explained_mismatch(sc[diff].astype(np.float64), w["u"][diff], a[diff], a_fused[diff], EPS_TIE).all()
    # and the materialised scores are finite everywhere with plausible assignments (no stale tiles)
    assert np.isfinite(sc).all() and not np.any(sc == 555.0)
    sel = np.take_along_axis(sc, a[:, None].astype(np.int64), axis=1)[:, 0]
    assert np.all(sel >= sc.max(axis=1) - 90.0)


def test_niw_1d_reference_kat(ctx, ref):
    """reference KAT test_normal_models.py:34-84: NIW(d=1) == NICH(sigmasq = psi/nu), vs the REFERENCE's
    nich output at the reference's tolerance 1e-3"""
    from distributions_b200 import capi
    data = np.array([4.0, 3.0, 7.0, 10.0])
    vals = np.array([32.0, -0.1], np.float32)
    k = ref.kind(1, None)
    k.add_nich([30.0, 0.3, 2.0 / 3.0, 3.0], [len(data)], [np.float32(data.mean())], [np.float32(((data - data.mean()) ** 2).sum())])
    want = k.score_rows([vals], 2, with_prior=False)
    w = dict(mu=[30.0], kappa=0.3, psi=[[2.0]], nu=3.0, count=[len(data)], sum_x=np.float32([[data.sum()]]),
             sum_xxT=np.float32([[[(data ** 2).sum()]]]))
    f = ctx.feature(capi.NIW).update_all(w)
    sc = torch.zeros((2, 1), device="cuda")
    ctx.score_batch([f], [dev(vals.reshape(2, 1))], 2, None, sc)
    torch.cuda.synchronize()
    got = sc.cpu().numpy()
    assert np.all(np.abs(got - want) <= 1e-3 * (1 + np.abs(got) + np.abs(want)))


def test_niw_mixed_with_nich(ctx, oracle):
    G, n, d = 21, 200, 8
    w = synth.niw(77, G, n, d=d)
    w2 = synth.nich(78, G, n)
    w2["sizes"] = w["sizes"]
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = _niw_cuda(ctx, w, n, prior, extra=w2)
    want = cases.oracle_scores(oracle, [w2], prior=prior)
    oracle.niw_score_rows(w["mu"], w["kappa"], w["psi"], w["nu"], w["count"], w["sum_x"], w["sum_xxT"], w["values"][:n], want)
    assert np.all(np.abs(scores - want) <= _niw_tol(w, want) + envelope(oracle, w2)[None, :])
    a_orc = oracle.sample_rows(scores.copy(), w["u"][:n])
    assert cases.explained_mismatch(scores.astype(np.float64), w["u"][:n], assign, a_orc, EPS_TIE).all()


def test_host_entry_pinned_and_chunked(ctx, oracle):
    """host-buffer entry with page-locked caller buffers (direct copies) and enough rows to exercise
    the two-stream chunk pipeline: identical to the device-pointer path"""
    from distributions_b200 import capi
    n, G = 300_000, 70
    w = synth.nich(15, G, n)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    f = ctx.feature(capi.NICH).update_all(w)
    a_dev, _ = run_cuda(ctx, [w], prior, w["u"], n, want_scores=False)
    pv = torch.from_numpy(w["values"]).pin_memory()
    pu = torch.from_numpy(w["u"]).pin_memory()
    pa = torch.empty(n, dtype=torch.int32).pin_memory()
    assign, _ = ctx.score_sample_batch_host([f], [pv.numpy()], prior, pu.numpy(), assign_out=pa.numpy())
    assert np.array_equal(assign, a_dev)
    assign2, _ = ctx.score_sample_batch_host([f], [w["values"]], prior, w["u"])  # pageable: staged
    assert np.array_equal(assign2, a_dev)


def test_nich_outlier_rows(ctx, oracle):
    """rows far from every group (no broad empty group to catch them): every score lies hundreds of nats below the best
    group constant, the regime where a static softmax reference would underflow -- the sampling kernels must still agree
    with the oracle's sampler on the materialised scores (nich_rows2: rows re-evaluated with their own maximum)"""
    n, G = 40_000, 300
    w = synth.nich(77, G, n)
    # every group well populated (steep Student-t tails, no empty group), a third of the rows thousands of sigmas away
    rng = np.random.default_rng(78)
    w["count"] = np.maximum(w["count"], 60).astype(w["count"].dtype)
    w["sizes"] = w["count"].astype(w["sizes"].dtype)
    w["mean"] = rng.normal(0.0, 5.0, G).astype(np.float32)
    w["ctv"] = (w["count"] * rng.uniform(0.5, 2.0, G)).astype(np.float32)
    far = np.arange(n) % 3 == 0
    w["values"] = rng.normal(0.0, 5.0, n).astype(np.float32)
    w["values"][far] = np.where(np.arange(far.sum()) % 2 == 0, 3e4, -7e5).astype(np.float32) + w["values"][far]
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    assign, scores = run_cuda(ctx, [w], prior, w["u"], n)
    assert scores[far].max(axis=1).max() < scores[~far].max(axis=1).min() - 100.0  # they really are outliers
    a_orc = oracle.sample_rows(scores.copy(), w["u"])
    assert cases.explained_mismatch(scores.astype(np.float64), w["u"], assign, a_orc, EPS_TIE).all()
    check_fused_variants(ctx, [w], prior, w["u"], n, scores, assign)


def test_host_register(ctx, oracle):
    """dist_b200_host_register: plain numpy arrays page-locked in place take the zero-copy route; same draws as the
    device-pointer path; registering twice is fine, unregistering an unknown pointer is an error, not a crash"""
    from distributions_b200 import capi
    n, G = 120_001, 300
    w = synth.nich(18, G, n)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    f = ctx.feature(capi.NICH).update_all(w)
    a_dev, _ = run_cuda(ctx, [w], prior, w["u"], n, want_scores=False)
    vals, uu, out = w["values"].copy(), w["u"].copy(), np.full(n, -7, np.int32)
    for arr in (vals, uu, out, vals):
        ctx.host_register(arr)
    try:
        assign, _ = ctx.score_sample_batch_host([f], [vals], prior, uu, assign_out=out)
        assert assign is out and np.array_equal(out, a_dev)
    finally:
        for arr in (vals, uu, out):
            ctx.host_unregister(arr)
    with pytest.raises(capi.DistB200Error):
        ctx.host_unregister(np.zeros(16, np.float32))
    assign2, _ = ctx.score_sample_batch_host([f], [vals], prior, uu)  # pageable again
    assert np.array_equal(assign2, a_dev)


def test_host_entry_niw_chunked(ctx, oracle):
    """niw through the host-buffer entry: the H2D copies of later row chunks run ahead on the second stream while the
    kernels stay on one (they share the context's packed-row buffer) -- pinned and pageable buffers, staged option too;
    identical to the device-pointer path"""
    from distributions_b200 import capi
    n, G = 200_000, 24
    w = synth.niw(16, G, n, d=32)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    f = ctx.feature(capi.NIW).update_all(w)
    a_dev, _ = run_cuda(ctx, [w], prior, w["u"], n, want_scores=False)
    pv = torch.from_numpy(w["values"]).pin_memory()
    pu = torch.from_numpy(w["u"]).pin_memory()
    pa = torch.empty(n, dtype=torch.int32).pin_memory()
    assign, _ = ctx.score_sample_batch_host([f], [pv.numpy()], prior, pu.numpy(), assign_out=pa.numpy())
    assert np.array_equal(assign, a_dev)
    assign2, _ = ctx.score_sample_batch_host([f], [w["values"]], prior, w["u"])
    assert np.array_equal(assign2, a_dev)


def test_host_entry_staged_option(ctx, oracle):
    """DIST_B200_OPT_HOST_ZEROCOPY = 1 (A/B runs): page-locked caller buffers through the staged chunk pipeline == zero-copy"""
    from distributions_b200 import capi
    n, G = 150_000, 200
    w = synth.nich(17, G, n)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    f = ctx.feature(capi.NICH).update_all(w)
    pv = torch.from_numpy(w["values"]).pin_memory()
    pu = torch.from_numpy(w["u"]).pin_memory()
    pa = torch.empty(n, dtype=torch.int32).pin_memory()
    zc, _ = ctx.score_sample_batch_host([f], [pv.numpy()], prior, pu.numpy(), assign_out=pa.numpy())
    zc = zc.copy()
    ctx.set_option(capi.OPT_HOST_ZEROCOPY, 1)
    try:
        staged, _ = ctx.score_sample_batch_host([f], [pv.numpy()], prior, pu.numpy(), assign_out=pa.numpy())
    finally:
        ctx.set_option(capi.OPT_HOST_ZEROCOPY, 0)
    assert np.array_equal(zc, staged)


def test_crosscat_gp_table_and_fallback(ctx, oracle):
    """multi-feature lists score GammaPoisson through the per-(group, value) table; counts beyond the
    table (>= 32, >= 64) take the direct formula -- both must equal the oracle"""
    G, n = 45, 400
    cc = synth.crosscat(640, G, n, n_gp=5, n_bb=2)
    feats = cc["features"]
    for k, w in enumerate(feats[:5]):
        w["values"][k::7] = [31, 32, 33, 63, 64, 65, 200, 5000][k % 8]
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, cc["sizes"])
    assign, scores = run_cuda(ctx, feats, prior, cc["u"], n)
    want = cases.oracle_scores(oracle, feats, prior=prior)
    env = sum(envelope(oracle, w) for w in feats)[None, :]
    assert np.all(np.abs(scores - want) <= 5e-6 * (1 + np.abs(want)) + env)
    a_orc = oracle.sample_rows(scores.copy(), cc["u"])
    assert cases.explained_mismatch(scores.astype(np.float64), cc["u"], assign, a_orc, EPS_TIE).all()
    # the single-feature (direct) kernel and the table path agree bit for bit on one feature
    _, s_direct = run_cuda(ctx, [feats[0]], None, cc["u"], n, sample=False)
    _, s_both = run_cuda(ctx, [feats[0], feats[5]], None, cc["u"], n, sample=False)
    _, s_bb = run_cuda(ctx, [feats[5]], None, cc["u"], n, sample=False)
    assert np.array_equal(s_both, s_direct + s_bb)


def test_c2_shape_vs_live_reference(ctx, oracle, ref):
    """BASELINE config 2's shape (nich, 1024 groups) against the UNMODIFIED reference run here
    (oracle/_ref): same statistics, same uniforms (captured from the reference's rng).  Scores within
    the stated envelope; indices identical except near-ties, whose rate is reported and bounded."""
    G, n = 1024, 20000
    w = synth.nich(20242, G, n)
    k = ref.kind(G, w["sizes"], synth.PY_ALPHA, synth.PY_D)
    cases.ref_add_feature(k, w)
    u, a_ref, s_ref = k.score_sample_rows([w["values"][:n]], n, seed=314)
    prior = k.prior()
    assign, scores = run_cuda(ctx, [w], prior, u, n)
    coeff = np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])[None, :]
    tol = 4e-6 * (1 + np.abs(s_ref)) + (1e-6 + LOG_STEP) * coeff
    assert np.all(np.abs(scores - s_ref) <= tol)
    # table-step flips (an argument one ulp away landing on the neighbouring fast_log entry) are rare
    assert np.mean(np.abs(scores - s_ref) <= 4e-6 * (1 + np.abs(s_ref)) + 1e-6 * coeff) > 0.99
    mism = assign != a_ref
    # every mismatch must be explained by the difference between the two score rows: u*total lies
    # between the CDF boundaries computed from the reference's scores and from ours
    ok_ref = cases.explained_mismatch(s_ref.astype(np.float64), u, assign, a_ref, 2e-3)
    assert ok_ref.all()
    assert mism.mean() < 2e-3, mism.mean()
    # with OUR scores the reference's own sampler reproduces our indices up to fp32 near-ties
    lik = scores.copy()
    a_ref_on_ours = oracle.sample_rows(lik, u)
    assert cases.explained_mismatch(scores.astype(np.float64), u, assign, a_ref_on_ours, EPS_TIE).all()
