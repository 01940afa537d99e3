"""The float64 reference of tests/gibbs_exact_ref.py on its own (no GPU): the Gibbs-invariance identity, order-free
chain-rule marginals, parity of the predictives with the oracle's fp32 scores, and the calibration and power of the
chain test that tests/test_gpu_gibbs_exact.py applies to the device chain."""
import numpy as np
import pytest
from scipy import special, stats

import gibbs_exact_ref as ref
from test_gpu_gibbs_exact import CASES, Exact, feature

MODELS = ["nich", "gp", "bnb", "bb", "dd", "dpd", "niw"]


def table(models_, N, seed=0, masked=False):
    rng = np.random.default_rng(seed)
    feats = []
    for k, m in enumerate(models_):
        p, x = feature(m, N, seed * 10 + k)
        feats.append(ref.Feature(m, p, x, (rng.random(N) < 0.7) if masked else None))
    return ref.Table(feats)


@pytest.mark.parametrize("n_empty", [1, 3])
@pytest.mark.parametrize("d", [0.0, 0.4])
@pytest.mark.parametrize("models_,masked", [(["nich"], False), (["nich", "gp", "bb", "dd"], True), (["dpd", "niw"], False)],
                         ids=["nich", "list_masked", "dpd_niw"])
def test_single_row_sweep_leaves_the_posterior_invariant(models_, masked, d, n_empty):
    """single-row blocks: pi_P == EPPF x marginal likelihoods, over every partition of 5 rows"""
    t = table(models_, 5, seed=len(models_) + int(10 * d), masked=masked)
    prior = ref.PitmanYorPrior(1.3, d)
    pi = ref.stationary(ref.sweep_matrix(t, prior, ref.single_rows(5), n_empty))
    post = ref.posterior(t, prior, ref.partitions(5))
    assert np.abs(pi - post).max() <= 1e-10
    assert post.max() < 0.5  # the identity is not checked at a point mass


def test_partitions_are_canonical():
    for N, bell in [(1, 1), (2, 2), (3, 5), (4, 15), (5, 52), (6, 203)]:
        states = ref.partitions(N)
        assert len(states) == len(set(states)) == bell
        assert all(ref.canonical(s) == s for s in states)
    assert ref.canonical([5, 5, 2, 9, 2]) == (0, 0, 1, 2, 1)


@pytest.mark.parametrize("model", MODELS)
def test_marginal_does_not_depend_on_row_order(model):
    t = table([model], 6, seed=3)
    rows = list(range(6))
    base = t.log_marginal(rows)
    rng = np.random.default_rng(4)
    for _ in range(5):
        perm = list(rng.permutation(rows))
        assert abs(t.log_marginal(perm) - base) <= 1e-12 * (1 + abs(base)), model


def test_block_rows_are_drawn_independently():
    """a block of all rows draws each among the fresh groups alone: uniform over labellings, whatever the data"""
    t = table(["nich"], 3, seed=1)
    states = ref.partitions(3)
    n_empty = 2
    P = ref.block_matrix(t, ref.PitmanYorPrior(1.0, 0.2), states, 0, 3, n_empty)
    want = np.zeros(len(states))
    for labels in np.ndindex(*(n_empty,) * 3):
        want[states.index(ref.canonical(labels))] += 1.0 / n_empty ** 3
    assert np.allclose(P, want[None, :], atol=1e-15)


@pytest.mark.parametrize("model", ["nich", "gp", "bnb", "bb", "dd"])
def test_predictives_match_oracle_scores(oracle, model):
    """the float64 predictive of every row against groups holding 0, 2 and 4 rows == the oracle's fp32 score_rows on
    the same statistics, within the envelope of the fp32 score (test_gpu_sample_values.py's tolerance)"""
    from oracle.pyoracle import BB, BNB, DD, GP, NICH
    p, x = feature(model, 6, 5)
    groups = [[], [0, 1], [2, 3, 4, 5]]
    xs = [x[g] for g in groups]
    n = np.array([len(g) for g in groups])
    if model == "nich":
        mean = np.array([v.astype(np.float64).mean() if v.size else 0.0 for v in xs])
        ctv = np.array([((v - m) ** 2).sum() for v, m in zip(xs, mean)])
        cache, mid = oracle.nich_caches(p["shared"], n, mean, ctv), NICH
    elif model in ("gp", "bnb"):
        s = np.array([v.astype(np.int64).sum() for v in xs])
        cache = (oracle.gp_caches if model == "gp" else oracle.bnb_caches)(p["shared"], n, s)
        mid = GP if model == "gp" else BNB
    elif model == "bb":
        heads = np.array([int(v.sum()) for v in xs])
        cache, mid = oracle.bb_caches(p["shared"], heads, n - heads), BB
    else:
        counts = np.stack([np.bincount(v, minlength=p["alphas"].size) for v in xs])
        cache, mid = oracle.dd_caches(p["alphas"], counts), DD
    got = oracle.score_rows(mid, cache, x, np.zeros((x.size, len(groups)), np.float32)).astype(np.float64)
    for r in range(x.size):
        for g, rows in enumerate(groups):
            want = ref.log_predictive(model, p, xs[g], x[r])
            if model == "bnb":  # the reference's score omits log C(v + r - 1, v)
                rr, v = float(p["shared"][2]), int(x[r])
                got[r, g] += special.gammaln(v + rr) - special.gammaln(v + 1) - special.gammaln(rr)
            assert abs(got[r, g] - want) <= 2e-2 + 2e-3 * abs(want), (model, r, g, got[r, g], want)


# ---- the chain test -------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def exact():
    """the sized exact chain of one GPU case"""
    case = next(c for c in CASES if c.name == "nich")
    return case, Exact(case)


def test_chain_test_is_calibrated(exact):
    """1000 numpy chains from P at the GPU case's S: the fraction with p < 0.01 is within binomial noise of 0.01"""
    case, ex = exact
    start = ex.states.index(ref.canonical(np.random.default_rng(case.seed).integers(0, 3, case.N)))
    burn = ref.burn_in(ex.P, ex.pi, start)
    n = 1000
    ps = np.array([ex.test.pvalue(h) for h in ref.simulate(ex.P, start, n, ex.S, burn, seed=1)])
    k = int((ps < 0.01).sum())
    assert stats.binom.cdf(k, n, 0.01) > ref.P_FLOOR and stats.binom.sf(k - 1, n, 0.01) > ref.P_FLOOR, k
    assert ps.min() > ref.P_FLOOR * 1e-2  # no chain from P comes near the floor's far tail


def test_chain_test_rejects_every_perturbed_kernel(exact):
    """200 numpy chains from each perturbed P' at the same S: >= 95 % rejected at P_FLOOR (the exact power is >= 0.99)"""
    case, ex = exact
    start = ex.states.index(ref.canonical(np.random.default_rng(case.seed).integers(0, 3, case.N)))
    sched = case.schedule()
    for k, alt in ex.alts.items():
        assert ex.test.power(alt) >= 0.99, k
        P_alt = ref.sweep_matrix(ex.table, ex.prior, sched, case.n_empty, k)
        burn = ref.burn_in(P_alt, alt, start)
        ps = np.array([ex.test.pvalue(h) for h in ref.simulate(P_alt, start, 200, ex.S, burn, seed=2)])
        assert np.mean(ps < ref.P_FLOOR) >= 0.95, (k, np.mean(ps < ref.P_FLOOR))


def test_pooling_keeps_every_state_in_one_cell():
    pi = np.array([0.5, 0.3, 0.1, 0.05, 0.03, 0.02])
    A = ref.pooling(pi, 100)
    assert np.array_equal(A.sum(0), np.ones(6)) and np.all(100 * (A @ pi) >= 5)
