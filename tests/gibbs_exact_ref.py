"""float64 reference of the blocked collapsed-Gibbs chain of distributions_b200.gibbs over every partition of a tiny table.

    table = Table([Feature("nich", dict(shared=...), values), ...])
    states = partitions(N)                             # restricted growth strings, regroup's stable order
    P = sweep_matrix(table, PitmanYorPrior(1.0, 0.2), single_rows(N), n_empty=1)
    pi = stationary(P)                                 # == posterior(table, prior, states) for single-row schedules

The posterior predictives are the library's parametrisations (tests/test_gpu_sample_values.py ties each of them to the
library's score_value).  ChainTest compares a histogram of sweeps with pi through the Markov-chain central limit
theorem; ChainTest.power is the probability that it rejects the stationary distribution of a perturbed kernel."""
import itertools
import math

import numpy as np
from scipy import stats

P_FLOOR = 1e-6  # one p-value floor for every test of fit (test_gpu_sample_values.py uses the same)
OTHER = 0xFFFFFFFF  # DirichletProcessDiscrete's "any other value" key


# ---- posterior predictives of one value given a group's statistics (float64) ---------------------------------------
def nich_predictive(shared, n, mean, ctv):
    """NormalInverseChiSq: Student t; shared = (mu, kappa, sigmasq, nu), (n, mean, ctv) the group's statistics"""
    mu, kappa, sigmasq, nu = np.asarray(shared, np.float64)
    pk, pn = kappa + n, nu + n
    pm = (kappa * mu + mean * n) / pk
    ps = (nu * sigmasq + ctv + n * kappa * (mu - mean) ** 2 / pk) / pn
    return stats.t(df=pn, loc=pm, scale=np.sqrt(ps * (pk + 1) / pk))


def gp_predictive(shape, rate):
    """GammaPoisson: negative binomial; shape = alpha + sum, rate = beta + count"""
    return stats.nbinom(n=float(shape), p=float(rate) / (1.0 + float(rate)))


def bnb_predictive(r, a, b):
    """BetaNegativeBinomial: beta-negative-binomial; a = alpha + r * count, b = beta + sum"""
    return stats.betanbinom(n=r, a=float(a), b=float(b))


def bb_predictive(alpha, beta, heads, tails):
    """BetaBernoulli: [P(0), P(1)]"""
    q = (alpha + heads) / (alpha + beta + heads + tails)
    return np.array([1.0 - q, q])


def dd_predictive(alphas, counts):
    """DirichletDiscrete: the probability of each value"""
    wt = np.asarray(alphas, np.float64) + counts
    return wt / wt.sum(-1, keepdims=True)


def dpd_predictive(alpha, betas, beta0, counts):
    """DirichletProcessDiscrete: the probability of each key in order, then of OTHER"""
    wt = np.concatenate([alpha * np.asarray(betas, np.float64) + counts, [alpha * np.float64(beta0)]])
    return wt / wt.sum()


def niw_predictive(mu, kappa, psi, nu, n, sum_x, sum_xxT):
    """NormalInverseWishart: multivariate t as dict(loc, shape, df)"""
    mu, psi = np.asarray(mu, np.float64), np.asarray(psi, np.float64)
    d = mu.size
    xbar = sum_x / n if n else np.zeros(d)
    diff = xbar - mu
    C = sum_xxT - np.outer(sum_x, xbar) - np.outer(xbar, sum_x) + n * np.outer(xbar, xbar)
    pk, pn = kappa + n, nu + n
    ppsi = psi + C + kappa * n / (kappa + n) * np.outer(diff, diff)
    dof = pn - d + 1
    return dict(loc=(kappa * mu + n * xbar) / pk, shape=ppsi * (pk + 1) / (pk * dof), df=dof)


def log_predictive(model, p, xs, x):
    """log p(x | the values xs of one group), float64.  p: the feature's parameters as update_all takes them"""
    xs = np.asarray(xs)
    n = float(len(xs))
    if model == "nich":
        v = xs.astype(np.float64)
        mean = v.mean() if n else 0.0
        return float(nich_predictive(p["shared"], n, mean, ((v - mean) ** 2).sum()).logpdf(float(x)))
    if model == "gp":
        a, b = np.asarray(p["shared"], np.float64)
        return float(gp_predictive(a + xs.astype(np.float64).sum(), b + n).logpmf(int(x)))
    if model == "bnb":
        a, b, r = np.asarray(p["shared"], np.float64)
        return float(bnb_predictive(r, a + r * n, b + xs.astype(np.float64).sum()).logpmf(int(x)))
    if model == "bb":
        a, b = np.asarray(p["shared"], np.float64)
        heads = float(np.count_nonzero(xs))
        return float(np.log(bb_predictive(a, b, heads, n - heads)[int(bool(x))]))
    if model == "dd":
        dim = np.asarray(p["alphas"]).size
        return float(np.log(dd_predictive(p["alphas"], np.bincount(xs.astype(np.int64), minlength=dim))[int(x)]))
    if model == "dpd":
        keys = [int(k) for k in p["keys"]]
        idx = lambda v: len(keys) if int(v) == OTHER else keys.index(int(v))  # noqa: E731
        counts = np.zeros(len(keys))
        for v in xs:
            if int(v) != OTHER:
                counts[idx(v)] += 1
        return float(np.log(dpd_predictive(float(p["alpha"]), p["betas"], float(np.float32(p["beta0"])), counts)[idx(x)]))
    if model == "niw":
        v = xs.astype(np.float64).reshape(-1, np.asarray(p["mu"]).size)
        t = niw_predictive(p["mu"], float(p["kappa"]), p["psi"], float(p["nu"]), n, v.sum(0), v.T @ v)
        return float(stats.multivariate_t(loc=t["loc"], shape=t["shape"], df=t["df"]).logpdf(np.asarray(x, np.float64)))
    raise ValueError(model)


class Feature:
    """one column of the table: model name, update_all parameters, N values, and an optional observed mask"""

    def __init__(self, model, params, values, observed=None):
        self.model, self.params, self.values = model, params, np.asarray(values)
        self.observed = None if observed is None else np.asarray(observed, bool)

    def seen(self, r):
        return self.observed is None or bool(self.observed[r])


class Table:
    """the rows of a kind: log p(row r | a group's rows) summed over the features where r is observed, memoised"""

    def __init__(self, features):
        self.features = list(features)
        self.N = len(self.features[0].values)
        self._memo = {}

    def log_like(self, r, rows):
        key = (r, tuple(sorted(rows)))
        if key not in self._memo:
            total = 0.0
            for f in self.features:
                if f.seen(r):
                    total += log_predictive(f.model, f.params, [f.values[i] for i in key[1] if f.seen(i)], f.values[r])
            self._memo[key] = total
        return self._memo[key]

    def log_marginal(self, rows):
        """log p(x_rows) of one group by the chain rule, in the given order"""
        return sum(self.log_like(r, rows[:i]) for i, r in enumerate(rows))


# ---- set partitions -------------------------------------------------------------------------------------------------
def canonical(assign):
    """the restricted growth string of a labelling: groups numbered in order of first appearance (regroup's order)"""
    lut = {}
    return tuple(lut.setdefault(int(a), len(lut)) for a in assign)


def partitions(N):
    """every set partition of N rows as a restricted growth string, in lexicographic order (Bell(N) of them)"""
    out = [()]
    for _ in range(N):
        out = [s + (k,) for s in out for k in range((max(s) + 2) if s else 1)]
    return out


def groups_of(state):
    """the rows of each group, in group order"""
    g = [[] for _ in range(max(state) + 1)]
    for r, a in enumerate(state):
        g[a].append(r)
    return g


# ---- clustering priors: the weights prior_prep_kernel / low_entropy_prep_kernel give one draw ------------------------
class PitmanYorPrior:
    """a live group: (n_g - d) / (n + alpha); each of K0 empty groups: (alpha + d K+) / (K0 (n + alpha))"""

    def __init__(self, alpha, d):
        self.alpha, self.d = float(alpha), float(d)

    def log_weights(self, sizes, n_empty, full_empty=False):
        """log weight of each live group, and of each empty group; the shared 1 / (n + alpha) is left out"""
        sizes = np.asarray(sizes, np.float64)
        empty = self.alpha + self.d * sizes.size
        return np.log(sizes - self.d), math.log(empty if full_empty else empty / n_empty)

    def log_eppf(self, sizes):
        """log of the exchangeable partition probability function of PY(alpha, d)"""
        a, d, K, n = self.alpha, self.d, len(sizes), sum(sizes)
        out = sum(math.log(a + i * d) for i in range(1, K)) - sum(math.log(a + i) for i in range(1, n))
        return out + sum(math.log(j - d) for s in sizes for j in range(1, s))


class LowEntropyPrior:
    """Clustering::LowEntropy as low_entropy_prep_kernel evaluates it (clustering.hpp:265-293, :318-327)"""

    def __init__(self, dataset_size):
        self.dataset_size = int(dataset_size)

    def log_weights(self, sizes, n_empty, full_empty=False):
        sizes = np.asarray(sizes, np.float64)
        n_total = int(sizes.sum())
        empty = 0.0 if full_empty else -math.log(n_empty)
        if n_total + 1 < self.dataset_size:
            n = float(n_total + 1)
            empty += math.log(self.dataset_size / n) * (0.45 - 0.1 / n - 0.1 / self.dataset_size)
        big = sizes > 10000
        live = np.where(big, 1.0 + np.log1p(sizes), np.log((sizes + 1) / sizes) * sizes + np.log1p(sizes))
        return live, empty


# ---- the exact transition matrix of a sweep -------------------------------------------------------------------------
def perturbations(prior, n_empty, alpha=1.1, slot0=1.05):
    """the perturbed kernels that apply to a case, each a plausible device bug:
      stale_stats   the row is scored against statistics that still hold it (its own group's)
      stale_prior   the prior counts the row in its own group
      d_zero        the Pitman-Yor discount is dropped (cases with d > 0)
      full_empty    each empty group gets the whole alpha + d K+ (cases with n_empty > 1)
      alpha*<f>     alpha scaled by f (Pitman-Yor)
      slot0*<f>     the sampler weighs group index 0 by f"""
    out = ["stale_stats", "stale_prior", "slot0*%g" % slot0]
    if isinstance(prior, PitmanYorPrior):
        out.append("alpha*%g" % alpha)
        if prior.d > 0:
            out.append("d_zero")
    if n_empty > 1:
        out.append("full_empty")
    return out


def _factor(perturb, name):
    return float(perturb.split("*")[1]) if perturb and perturb.startswith(name + "*") else None


def single_rows(N):
    return [(r, r + 1) for r in range(N)]


def block_matrix(table, prior, states, r0, r1, n_empty, perturb=None):
    """one block over rows [r0, r1): the block's rows are removed, then each draws independently from its conditional
    against the remaining rows, over the K+ live groups and n_empty labelled empty groups; rows drawing the same empty
    group form one new group.  A single row draws "any empty group" as one outcome (its mass does not depend on how it
    is split).  perturb: None or one of perturbations()."""
    index = {s: i for i, s in enumerate(states)}
    block = list(range(r0, r1))
    if perturb == "d_zero":
        prior = PitmanYorPrior(prior.alpha, 0.0)
    elif _factor(perturb, "alpha"):
        prior = PitmanYorPrior(prior.alpha * _factor(perturb, "alpha"), prior.d)
    merge = len(block) == 1
    assert merge or n_empty <= 3, "blocks of several rows are enumerated over at most 3 labelled empty groups"
    P = np.zeros((len(states), len(states)))
    for i, s in enumerate(states):
        rest = [r for r in range(table.N) if r < r0 or r >= r1]
        live = canonical([s[r] for r in rest]) if rest else ()
        K = max(live) + 1 if rest else 0
        members = [[r for r, a in zip(rest, live) if a == g] for g in range(K)]
        log_live, log_empty = prior.log_weights([len(m) for m in members], n_empty, full_empty=perturb == "full_empty")
        fresh = 1 if merge else n_empty
        if merge:
            log_empty += math.log(n_empty)
        probs = []
        for r in block:
            own = [g for g in range(K) if any(s[m] == s[r] for m in members[g])]
            lw = np.empty(K + fresh)
            for g in range(K):
                rows, w = members[g], log_live[g]
                if g in own and perturb == "stale_stats":
                    rows = rows + [r]
                if g in own and perturb == "stale_prior":
                    w = prior.log_weights([len(m) + (h == g) for h, m in enumerate(members)], n_empty)[0][g]
                lw[g] = w + table.log_like(r, rows)
            lw[K:] = log_empty + table.log_like(r, [])
            if _factor(perturb, "slot0"):
                lw[0] += math.log(_factor(perturb, "slot0"))
            p = np.exp(lw - lw.max())
            probs.append(p / p.sum())
        for combo in itertools.product(*[range(K + fresh) for _ in block]):
            w = np.prod([probs[k][c] for k, c in enumerate(combo)])
            a = list(s)
            for r in rest:
                a[r] = live[rest.index(r)]
            for r, c in zip(block, combo):
                a[r] = c
            P[i, index[canonical(a)]] += w
    return P


def sweep_matrix(table, prior, schedule, n_empty, perturb=None):
    """the transition matrix of one sweep: the blocks of the schedule (row ranges) in order"""
    states = partitions(table.N)
    P = np.eye(len(states))
    for r0, r1 in schedule:
        P = P @ block_matrix(table, prior, states, r0, r1, n_empty, perturb)
    return P


def stationary(P):
    """the stationary distribution: pi P = pi, sum(pi) = 1"""
    n = P.shape[0]
    A = np.vstack([P.T - np.eye(n), np.ones((1, n))])
    b = np.zeros(n + 1)
    b[-1] = 1.0
    pi = np.linalg.lstsq(A, b, rcond=None)[0]
    return np.clip(pi, 0.0, None) / np.clip(pi, 0.0, None).sum()


def posterior(table, prior, states):
    """Pitman-Yor: EPPF(sizes) x prod_groups marginal(x_group), normalised over the states"""
    lp = np.array([prior.log_eppf([len(g) for g in groups_of(s)]) + sum(table.log_marginal(g) for g in groups_of(s))
                   for s in states])
    p = np.exp(lp - lp.max())
    return p / p.sum()


def tv(p, q):
    return 0.5 * float(np.abs(np.asarray(p) - np.asarray(q)).sum())


def burn_in(P, pi, start, tol=1e-3):
    """the smallest B with TV(delta_start P^B, pi) <= tol"""
    x = np.zeros(P.shape[0])
    x[start] = 1.0
    for B in range(100_000):
        if tv(x, pi) <= tol:
            return B
        x = x @ P
    raise AssertionError("the chain does not mix")


# ---- the test of a chain's histogram -------------------------------------------------------------------------------
def clt_covariance(P, pi):
    """asymptotic covariance of the histogram of a stationary chain: diag(pi) Z + Z^T diag(pi) - diag(pi) - pi pi^T"""
    n = P.shape[0]
    Z = np.linalg.inv(np.eye(n) - P + np.outer(np.ones(n), pi))
    D = np.diag(pi)
    return D @ Z + Z.T @ D - D - np.outer(pi, pi)


def pooling(pi, S):
    """cell of each state: states with S pi >= 5 keep a cell each (largest first); the others share one cell, which
    joins the smallest kept cell when its own S pi is below 5"""
    order = np.argsort(-pi, kind="stable")
    cell = np.full(pi.size, -1)
    big = [s for s in order if S * pi[s] >= 5]
    for k, s in enumerate(big):
        cell[s] = k
    small = cell < 0
    if small.any():
        if S * pi[small].sum() >= 5 or not big:
            cell[small] = len(big)
        else:
            cell[small] = len(big) - 1
    A = np.zeros((cell.max() + 1, pi.size))
    A[cell, np.arange(pi.size)] = 1.0
    return A


class ChainTest:
    """T = S (p - pi)^T Sigma^+ (p - pi) over the pooled cells, against chi2(cells - 1).  Sigma's null direction is
    the all-ones vector (the histogram sums to 1), so the last cell is dropped and the rest inverted."""

    def __init__(self, P, pi, S):
        self.P, self.pi, self.S = P, pi, int(S)
        self.A = pooling(pi, S)
        self.cells = self.A.shape[0]
        sig = self.A @ clt_covariance(P, pi) @ self.A.T
        self.inv = np.linalg.inv(sig[:-1, :-1])
        self.df = self.cells - 1
        self.critical = stats.chi2.isf(P_FLOOR, self.df)

    def statistic(self, p_hat):
        d = self.A @ (np.asarray(p_hat, np.float64) - self.pi)
        return self.S * float(d[:-1] @ self.inv @ d[:-1])

    def pvalue(self, p_hat):
        return float(stats.chi2.sf(self.statistic(p_hat), self.df))

    def power(self, pi_alt):
        """probability that the test at P_FLOOR rejects a chain whose stationary distribution is pi_alt"""
        return float(stats.ncx2.sf(self.critical, self.df, self.statistic(pi_alt)))


def sweeps_for_power(P, pi, alts, target=0.99, s_min=1000):
    """the smallest S (to 5 %) at which the test rejects every alternative stationary distribution with >= target"""
    S = s_min
    while min(ChainTest(P, pi, S).power(a) for a in alts) < target:
        S = int(S * 1.05) + 1
        assert S < 10_000_000, "the alternatives are indistinguishable"
    return S


def simulate(P, start, n_chains, S, burn, seed):
    """n_chains histograms of S sweeps after burn sweeps, every chain from state start (numpy, vectorised over chains)"""
    rng = np.random.default_rng(seed)
    cum = np.cumsum(P, 1)
    cum[:, -1] = 1.0
    x = np.full(n_chains, start)
    hist = np.zeros((n_chains, P.shape[0]))
    rows = np.arange(n_chains)
    for t in range(burn + S):
        x = np.minimum((rng.random(n_chains)[:, None] > cum[x]).sum(1), P.shape[0] - 1)
        if t >= burn:
            hist[rows, x] += 1
    return hist / S
