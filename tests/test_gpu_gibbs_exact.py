"""The device Gibbs chain against exact float64 distributions over every partition of a tiny table.

Each case loads a table of 4 - 6 rows into one kind, runs S sweeps of gibbs.BlockedGibbs.block over a fixed schedule
of row blocks, and records the partition after every sweep.  tests/gibbs_exact_ref.py builds the exact transition
matrix P of that schedule in float64 (every partition, every draw), and the histogram of the sweeps is tested against
P's stationary distribution through the Markov-chain central limit theorem at the suite's p-value floor.  For blocks of
one row that distribution is the Pitman-Yor posterior (EPPF x marginal likelihoods; test_gibbs_exact_ref.py checks the
identity).  Blocks of several rows draw their rows independently given the rest: their stationary distribution is not
the posterior, and the assertion messages give how far it is (total variation).

The test is sized from the exact kernel: S is the number of sweeps at which the test rejects, with probability >= 0.99,
the stationary distribution of each perturbed kernel of gibbs_exact_ref.perturbations (the row scored against its own
statistics, the prior counting the row, the discount dropped, the empty mass not split, alpha off, one group index
over-weighted), and every case must be informative (>= 6 pooled cells, no partition above 0.6).  Large-G routes are
reached with many empty groups: they change G, not the posterior over partitions.  The first sweep of every case runs
under torch.profiler and must launch the kernel the case is meant to reach.

Not reached here: the one-table-feature sampling shortcuts (value-CDF guide tables and trees, table_rows) need at
least 4 R rows in one call (R table rows; test_gpu_routes.py::test_dpd_sampling_thresholds), and no block of an
enumerable table has that many.  The index-for-index route tests remain their check."""
import re
import time

import numpy as np
import pytest

import gibbs_exact_ref as ref
from distributions_b200 import capi, gibbs, models
from test_gpu_regroup import download, host_stats

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

MODEL_ID = {"nich": capi.NICH, "gp": capi.GP, "bnb": capi.BNB, "bb": capi.BB, "dd": capi.DD, "dpd": capi.DPD, "niw": capi.NIW}
DPD_KEYS = np.array([7, 3, 1000, 42], np.uint32)


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = capi.Context(0)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ---- the tables -----------------------------------------------------------------------------------------------------
def feature(model, N, seed, d=3):
    """(update_all parameters without statistics, N values): parameters and data chosen so that the posterior over
    partitions is spread and still depends on the data"""
    rng = np.random.default_rng(seed)
    if model == "nich":
        return dict(shared=np.array([0.0, 1.0, 1.0, 3.0], np.float32)), rng.normal(0, 1.5, N).astype(np.float32)
    if model == "gp":
        return dict(shared=np.array([2.0, 1.0], np.float32)), rng.choice([0, 1, 3, 6], N).astype(np.uint32)
    if model == "bnb":
        return dict(shared=np.array([3.0, 2.0, 2.0], np.float32)), rng.choice([0, 1, 4, 9], N).astype(np.uint32)
    if model == "bb":
        return dict(shared=np.array([0.5, 0.5], np.float32)), (np.arange(N) % 2).astype(np.uint8)[rng.permutation(N)]
    if model == "dd":
        return dict(alphas=np.full(4, 0.5, np.float32)), rng.integers(0, 4, N).astype(np.int32)
    if model == "dpd":
        p = dict(alpha=2.0, beta0=0.2, gamma=1.0, keys=DPD_KEYS, betas=np.array([0.3, 0.2, 0.2, 0.1], np.float32))
        return p, DPD_KEYS[rng.integers(0, DPD_KEYS.size, N)]
    # niw: a strong prior (kappa, nu large) keeps d dimensions from pinning the partition
    p = dict(mu=np.zeros(d, np.float32), kappa=float(d), psi=np.eye(d, dtype=np.float32) * (d + 30.0), nu=float(2 * d + 30))
    return p, rng.normal(0, 1.0, (N, d)).astype(np.float32)


def zero_stats(model, p, G):
    """update_all arguments: the parameters and G empty groups"""
    z = {"nich": lambda: dict(count=np.zeros(G, np.int32), mean=np.zeros(G, np.float32), ctv=np.zeros(G, np.float32)),
         "gp": lambda: dict(count=np.zeros(G, np.uint32), sum=np.zeros(G, np.uint32)),
         "bnb": lambda: dict(count=np.zeros(G, np.uint32), sum=np.zeros(G, np.uint32)),
         "bb": lambda: dict(heads=np.zeros(G, np.int32), tails=np.zeros(G, np.int32)),
         "dd": lambda: dict(counts=np.zeros((G, p.get("alphas", np.zeros(1)).size), np.int32)),
         "dpd": lambda: dict(counts=np.zeros((G, DPD_KEYS.size), np.int32)),
         "niw": lambda: dict(count=np.zeros(G, np.int32), sum_x=np.zeros((G, p.get("mu", np.zeros(1)).size), np.float32),
                             sum_xxT=np.zeros((G,) + (p.get("mu", np.zeros(1)).size,) * 2, np.float32))}[model]()
    return dict(p, model=model, **z)


class Case:
    def __init__(self, name, models_, N, expect, prior=("py", 1.0, 0.3), n_empty=1, block=1, masked=False, seed=0,
                 alpha=1.25, slot0=1.25, d=3):
        self.name, self.models, self.N, self.expect = name, models_, N, expect
        self.prior_spec, self.n_empty, self.block, self.masked, self.seed, self.d = prior, n_empty, block, masked, seed, d
        self.alpha, self.slot0 = alpha, slot0

    def __repr__(self):
        return self.name

    def prior(self):
        kind, *args = self.prior_spec
        return ref.PitmanYorPrior(*args) if kind == "py" else ref.LowEntropyPrior(*args)

    def device_prior(self):
        kind, *args = self.prior_spec
        return models.PitmanYor(*args) if kind == "py" else models.LowEntropy(*args)

    def schedule(self):
        """single rows, or blocks of self.block rows (the last one takes what is left)"""
        return [(r, min(self.N, r + self.block)) for r in range(0, self.N, self.block)]

    def table(self):
        feats = []
        rng = np.random.default_rng(100 + self.seed)
        for k, m in enumerate(self.models):
            p, x = feature(m, self.N, self.seed * 10 + k, self.d)
            obs = None
            if self.masked:
                obs = rng.random(self.N) < 0.7
                obs[k % self.N] = False  # every feature misses at least one cell
            feats.append(ref.Feature(m, p, x, obs))
        return ref.Table(feats)


SINGLE = [Case("nich", ["nich"], 5, r"score_rows_kernel<32, ", seed=1),
          Case("gp", ["gp"], 5, r"score_rows_kernel<32, ", seed=2),
          Case("bnb", ["bnb"], 5, r"score_rows_kernel<32, ", seed=3),
          Case("bb", ["bb"], 5, r"score_rows_kernel<32, ", seed=4),
          Case("dd", ["dd"], 5, r"score_rows_kernel<32, ", seed=5),
          Case("dpd", ["dpd"], 5, r"gather_rows", seed=6),
          Case("niw3", ["niw"], 5, r"niw_rows_kernel", seed=7),
          Case("nich_G1024", ["nich"], 5, r"nich_rows2_kernel", n_empty=1020, seed=8),
          Case("gp_G1100", ["gp"], 5, r"score_rows_kernel<32, ", n_empty=1100, seed=9),
          Case("dd_G1100", ["dd"], 5, r"score_rows_kernel<32, ", n_empty=1100, seed=10),
          Case("dpd_G1100", ["dpd"], 5, r"gather_rows", n_empty=1100, seed=11),
          Case("niw32", ["niw"], 4, r"niw_tc_fused_kernel", d=32, seed=12),
          Case("niw96", ["niw"], 4, r"niw_tc_wide_kernel", d=96, seed=13),
          Case("list", ["nich", "gp", "bb", "dd"], 5, r"score_rows_kernel<32, -1, ", seed=14),
          Case("list_ksub", ["nich", "gp", "bb", "dd"], 5, r"score_rows_kernel<128, -1, true, false, 128, true>",
               n_empty=1100, seed=15),
          Case("list_masked", ["nich", "gp", "bb", "dd"], 5, r"score_rows_kernel<32, -1, .*MaskList", masked=True, seed=16),
          Case("list_masked_ksub", ["nich", "gp", "bb", "dd"], 5,
               r"score_rows_kernel<128, -1, true, false, 128, true, distb200::MaskList>", n_empty=1100, masked=True, seed=17),
          Case("nich_crp", ["nich"], 5, r"prior_prep_kernel", prior=("py", 1.0, 0.0), n_empty=3, seed=18),
          Case("nich_low_entropy", ["nich"], 5, r"low_entropy_prep_kernel", prior=("le", 5), seed=19),
          Case("nich_power", ["nich"], 4, r"score_rows_kernel<32, ", prior=("py", 2.0, 0.3), seed=20, alpha=1.1, slot0=1.05)]
BLOCKS = [Case("nich_blocks2", ["nich"], 5, r"score_rows_kernel<32, ", n_empty=2, block=2, seed=21),
          Case("dd_blocks3", ["dd"], 6, r"score_rows_kernel<32, ", n_empty=3, block=3, seed=22)]
CASES = SINGLE + BLOCKS


class Exact:
    """the exact chain of a case: P, pi, the test at S sweeps, and the alternatives it must reject"""

    def __init__(self, case):
        self.table, self.prior = case.table(), case.prior()
        self.states = ref.partitions(case.N)
        sched = case.schedule()
        self.P = ref.sweep_matrix(self.table, self.prior, sched, case.n_empty)
        self.pi = ref.stationary(self.P)
        self.alts = {k: ref.stationary(ref.sweep_matrix(self.table, self.prior, sched, case.n_empty, k))
                     for k in ref.perturbations(self.prior, case.n_empty, case.alpha, case.slot0)}
        self.S = ref.sweeps_for_power(self.P, self.pi, list(self.alts.values()))
        self.test = ref.ChainTest(self.P, self.pi, self.S)


# ---- running the device chain ---------------------------------------------------------------------------------------
def load(ctx, case, table, start):
    """the table's features at the start partition: update_all with empty groups, then add_rows_batch"""
    G0 = max(start) + 1
    feats, cols, obs = [], [], []
    for f in table.features:
        feats.append(ctx.feature(MODEL_ID[f.model]).update_all(zero_stats(f.model, f.params, G0)))
        cols.append(dev(f.values.astype(capi.COLUMN_DTYPE[MODEL_ID[f.model]])))
        obs.append(None if f.observed is None else dev(capi.pack_observed(f.observed).view(np.int32)))
    observed = obs if case.masked else None
    assign = dev(np.asarray(start, np.int32))
    ctx.add_rows_batch(feats, cols, assign, case.N, observed=observed)
    return feats, cols, observed, assign


def launched(fn):
    """names of the CUDA kernels fn() launches"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def recount_matches(f, fe, assign, G):
    """the device statistics equal a float64 recount of the final assignment (integers exactly; floats within the
    tolerances of test_gpu_regroup.py::test_sweep_invariants)"""
    m, x, obs = fe.model, fe.values, fe.observed
    ok = (assign >= 0) if obs is None else (assign >= 0) & obs
    if m == "dpd":
        got = download("dpd", dict(counts=np.zeros((1, DPD_KEYS.size))), f, G)[0]
        idx = np.array([list(DPD_KEYS).index(int(v)) for v in x])
        want = np.zeros((G, DPD_KEYS.size), np.int64)
        np.add.at(want, (assign[ok], idx[ok]), 1)
        assert np.array_equal(got.astype(np.int64), want)
        return
    if m == "niw":
        d = x.shape[1]
        got = download("niw", dict(mu=np.zeros(d)), f, G)
        a = assign[ok]
        assert np.array_equal(got[0].ravel().view(np.int32), np.bincount(a, minlength=G))
        sx = np.zeros((G, d))
        sxx = np.zeros((G, d, d))
        np.add.at(sx, a, x[ok].astype(np.float64))
        np.add.at(sxx, a, np.einsum("ni,nj->nij", x[ok].astype(np.float64), x[ok].astype(np.float64)))
        np.testing.assert_allclose(got[1].view(np.float32).reshape(G, d), sx, rtol=1e-5, atol=1e-4)
        np.testing.assert_allclose(got[2].view(np.float32).reshape(G, d, d), sxx, rtol=1e-5, atol=1e-4)
        return
    name = "gp" if m == "bnb" else m
    w = dict(counts=np.zeros((1, fe.params["alphas"].size))) if m == "dd" else {}
    got = download(m, w, f, G)
    want = host_stats(name, x, assign, G, obs, fe.params["alphas"].size if m == "dd" else None)
    if m == "nich":
        assert np.array_equal(got[0].ravel().view(np.int32), want[0])
        np.testing.assert_allclose(got[1].ravel().view(np.float32), want[1], rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(got[2].ravel().view(np.float32), want[2], rtol=2e-4, atol=1e-3)
    else:
        for g_, w_ in zip(got, want):
            assert np.array_equal(g_.reshape(w_.shape).astype(np.int64), w_), m


@pytest.mark.parametrize("case", CASES, ids=repr)
def test_chain_matches_exact_distribution(ctx, case):
    ex = Exact(case)
    cells = ex.test.cells
    assert cells >= 6 and ex.pi.max() <= 0.6, (case, cells, ex.pi.max())  # the data are informative
    for k, a in ex.alts.items():
        assert ex.test.power(a) >= 0.99, (case, k, ex.test.power(a))
    rng = np.random.default_rng(case.seed)
    start = ref.canonical(rng.integers(0, 3, case.N))
    s0 = ex.states.index(start)
    burn = ref.burn_in(ex.P, ex.pi, s0)
    feats, cols, observed, assign = load(ctx, case, ex.table, start)
    kind = gibbs.BlockedGibbs(ctx, feats, cols, assign, case.device_prior(), n_empty=case.n_empty, observed=observed)
    gen = torch.Generator(device="cuda").manual_seed(1000 + case.seed)
    sched = case.schedule()

    def sweep():
        for r0, r1 in sched:
            kind.block(r0, r1, gen)

    names = launched(sweep)  # the first sweep: the route the case is for
    assert any(re.search(case.expect, n) for n in names), (case, case.expect, sorted(set(n.split("(")[0] for n in names)))
    for _ in range(burn):
        sweep()
    hist = torch.empty((ex.S, case.N), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for s in range(ex.S):
        sweep()
        hist[s].copy_(assign)
    torch.cuda.synchronize()
    per_sweep = (time.perf_counter() - t0) / ex.S
    index = {st: i for i, st in enumerate(ex.states)}
    visits = np.bincount([index[ref.canonical(h)] for h in hist.cpu().numpy()], minlength=len(ex.states))
    p_hat = visits / ex.S
    p = ex.test.pvalue(p_hat)
    msg = "%s: S %d, burn-in %d, %d cells, p %.3g, %.3f ms per sweep" % (case, ex.S, burn, cells, p, 1e3 * per_sweep)
    if isinstance(ex.prior, ref.PitmanYorPrior):
        msg += ", TV(pi_P, posterior) %.4f" % ref.tv(ex.pi, ref.posterior(ex.table, ex.prior, ex.states))
    print(msg)
    assert p > ref.P_FLOOR, msg
    a = assign.cpu().numpy()
    assert a.min() >= 0 and a.max() < kind.G and int((np.bincount(a) > 0).sum()) >= kind.G - case.n_empty
    for f, fe in zip(feats, ex.table.features):
        recount_matches(f, fe, a, kind.G)
        f.close()


@pytest.mark.parametrize("r0", [1, 5, 31, 33])
def test_masked_block_at_unaligned_rows(ctx, r0):
    """block(r0, r1) with observed masks and r0 % 32 != 0: the statistics equal a float64 recount of the assignment
    with the masks of the block's own rows"""
    N, n = 100, 7
    case = Case("unaligned", ["nich", "gp", "bb", "dd"], N, "", masked=True, seed=30 + r0)
    table = case.table()
    rng = np.random.default_rng(r0)
    for fe in table.features:
        fe.observed = rng.random(N) < 0.5
    start = ref.canonical(rng.integers(0, 4, N))
    feats, cols, observed, assign = load(ctx, case, table, start)
    kind = gibbs.BlockedGibbs(ctx, feats, cols, assign, models.PitmanYor(1.0, 0.2), n_empty=2, observed=observed)
    gen = torch.Generator(device="cuda").manual_seed(r0)
    for k in range(3):
        kind.block(r0 + k * n, r0 + (k + 1) * n, gen)
        a = assign.cpu().numpy()
        for f, fe in zip(feats, table.features):
            recount_matches(f, fe, a, kind.G)
    for f in feats:
        f.close()
