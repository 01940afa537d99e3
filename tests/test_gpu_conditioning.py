"""nich and NIW scores against float64 references on rescaled, shifted and mixed-magnitude data.

Every other continuous-valued test runs on data shaped like synth.py (unit spread, centres near 0, NIW psi = I) and
compares with the fp32 oracle under a blanket fast_log-table-step slack.  Here the data, the prior and the group
statistics are rescaled, shifted and mixed with far outliers, and every score is compared with a float64 evaluation of
the same operation under a STEP-AWARE rule instead:

  The per-cell log of the kernels is log2(trunc9(a)) (numerics.cuh fast_log2_cell: the low 9 mantissa bits of the fp32
  argument a are cleared, then MUFU.LG2), the reference's table fast_log(a) / ln 2 is the same step function.  The exact
  argument a64 is computed in float64; a route evaluates it to within a derived bound delta_a (below), so its log lies in
  [log2(trunc9(a64 - delta_a)), log2(trunc9(a64 + delta_a))] -- one value except for cells within delta_a of a table step,
  the only cells where the neighbouring step is allowed.  Then
      score  in  C + coef * ln 2 * [that interval]  +-  tol_round,
      tol_round = |coef ln 2| (2^-22 max(1, |L|) + 2^-23 |L|) + 2^-23 (|C| + |score|) + tol_C,
  where 2^-22 max(1, |L|) is MUFU.LG2's error (absolute on [1, 2), relative elsewhere), 2^-23 |L| the rounding of the
  folded coefficient coef ln 2 and of the fma, 2^-23 (|C| + |score|) the final additions, and tol_C the constant's own
  bound (nich: 0, the constant is the kernel's cache score_; NIW: below).  An argument whose fp32 evaluation overflows
  has the reference's table value fast_log(inf) = 128 ln 2.

nich (argument 1 + precision (x - mean)^2 from the cache rows of download_caches(4), prep.cu row order):
  fp32 evaluation: x - mean, its square, times precision, plus 1: four roundings, so
      delta_a = 4 u (a - 1) + u a,  u = 2^-24.

NIW (argument 1 + q / dof, q = |W (x - mu')|^2):
  The reference recomputes each group's posterior as niw_posterior_cholesky does, in float64 from the float32 statistics,
  rounds mu' to float32 as niw_prep_kernel does, takes W = L^-1 from the float64 Cholesky factor and evaluates q in
  float64.  The constant is term1 + term2 of score_mv_student_t with the oracle's fast_lgamma / fast_log(dof) and the
  log-determinant policy of niw_log_det: fast_log(float(det)) while det is a normal float, else the exact log det.
    FP32 route (niw_score_kernel, niw_rows_kernel): z = fl(x - mu') (u |z|) and W rounded to fp32 (u |W|) give
      2 u sum_j |W_ij| |z_j|; the fmaf chain over j = 0..i in ascending order rounds each partial sum s_ik = sum_{j <= k}
      W_ij z_j once (u |s_ik|): |dy_i| <= e_i = 2 u sum_j |W_ij| |z_j| + 1.01 u sum_k |s_ik| (1.01: the rounded partial
      sums' own drift).  The sum of squares, fmaf in ascending i, adds u sum_k Q_k (Q_k its partial sums); 1/dof and the
      product add 2 u q / dof, the final add u a:
      delta_a = (sum_i (2 |y_i| e_i + e_i^2) + u sum_k Q_k + 2 u q) / dof + u a.
    Tensor-core route (niw_tc.cu, d = 32): x 2^ex and W 2^ew are split in two fp16 terms each.  Per element the split
      keeps |v - hi - lo| <= 2^-22 |v| + 2^-25 (half of fp16's subnormal quantum, in the scaled units), the dropped
      lo x lo product is <= 2^-22 |x| |W|, and the tensor core accumulates 112 products in fp32 -- hi hi at K = 48, lo hi
      and hi lo at K = 32 each -- (<= 2^-23 per step,
      truncation allowed).  b = W mu' is formed in double and rounded to fp32.  With A_i = sum_j |W_ij| |x_j| and
      B_i = sum_j |W_ij| |mu'_j| (>= |b_i|):
      e_i = (3 2^-22 + u + 112 2^-23) A_i + (2^-22 + 2 u + 112 2^-23) B_i + 2^-25 (sum_j |W_ij| / sx + (sum_j |x_j| + 1) / sw),
      and delta_a as above with (d + 3) u q in place of u sum_k Q_k (the epilogue sums pairs in its own order).  The error scales with |W x| and |W mu'|, not with |W (x - mu')|: the route is exact to
      about 2^-20 relative of |W x|, so its log argument degrades with the data's offset from the origin in whitened units
      (DESIGN §6).  Measured on a B200 it meets the FP32 bound on data within a few standard deviations of the origin and
      misses it at 1e2 - 1e3 sigma and beside far-larger rows in its tile; the tests hold it to the FP32 bound in that
      domain and to its derived bound outside it.  The FP32 route on the same feature (DIST_B200_OPT_NIW_PATH = 1) must
      meet the FP32 bound everywhere.
    Constant: term1 and term2 are rounded to fp32 from double and added once: tol_C = 2^-22 (|lgamma terms| + |term2|).

Other routes: the sampling-only (fused) launches are compared with the materialising launch on the same rows by the
near-tie rule of test_gpu_parity; score_logp_batch with the float64 logsumexp of the reference interval, within the
route's own bound 2^-21 (1 + max |s|) + (G + 8) 2^-24 (test_gpu_score_logp).

Overflow: the per-cell log needs a finite argument.  When 1 + precision (x - mean)^2 or 1 + q / dof overflows fp32 the
kernels return log2(inf) = inf, i.e. a score of -inf, where the reference's table gives the finite 128 ln 2 (DESIGN §4,
dist_b200.h).  The tests pin that documented behaviour: exactly the overflowing cells are -inf, every other cell of the
row is checked as usual, and no other row of the batch is affected -- except, on the d = 32 tensor-core route, the other
rows of its 128-row tile, which lose their bits to the tile's scale and score NaN (DESIGN §6).
"""
import numpy as np
import pytest

import cases
from distributions_b200 import synth

U = 2.0 ** -24
LN2 = np.log(2.0)
LOG_PI_F = float(np.float32(1.1447298858494002))
FLT_MAX = float(np.finfo(np.float32).max)
EPS_TIE = 2e-5

# the nich-relevant option sets of the sampling-only entry (dist_b200_option settings, as in test_gpu_parity)
NICH_FUSED = {
    "default": {},
    "row_tile_32": {1: 32},
    "small_tile_256": {0: 1, 5: 1},
    "small_tile_4x32": {0: 1, 5: 3},
    "nich_scalar": {6: 1},
    "nich_packed_one_row": {6: 2},
    "nich_online_max_two_rows": {6: 3},
    "nich_online_max_mufu": {6: 3, 9: 1},
    "nich_exp_all_mufu": {9: 1},
    "nich_exp_offload_4": {9: 5},
    "nich_exp_offload_8": {9: 9},
}


# ----------------------------------------------------------------------------------------- the step-aware checker
def _log2_step(a):
    """log2 of the table step of float64 arguments a (rounded to fp32, low 9 mantissa bits cleared); fp32 overflow ->
    128, the reference's fast_log(inf) / ln 2"""
    a32 = np.asarray(a, np.float64).astype(np.float32)
    t = (a32.view(np.uint32) & np.uint32(0xFFFFFE00)).view(np.float32).astype(np.float64)
    with np.errstate(divide="ignore"):
        return np.where(np.isinf(t), 128.0, np.log2(t))


def log2_interval(a, delta):
    """[lo, hi] of log2(trunc9(a')) over a' in [a - delta, a + delta]; the ends are rounded outwards to fp32"""
    lo = np.maximum(np.asarray(a, np.float64) - delta, 1.0)
    hi = np.asarray(a, np.float64) + delta
    with np.errstate(over="ignore"):
        lo32 = lo.astype(np.float32)
    lo32 = np.where(lo32.astype(np.float64) > lo, np.nextafter(lo32, np.float32(0)), lo32)
    with np.errstate(over="ignore"):
        hi32 = hi.astype(np.float32)
    return _log2_step(lo32), _log2_step(hi32)


def overflows(a, delta):
    """cells whose fp32 argument overflows for every evaluation within delta"""
    return np.asarray(a, np.float64) - delta > FLT_MAX * (1 + U)


def check_step_aware(got, C, coef, a, delta, tol_C=0.0, what=""):
    """got[n][G] against C[g] + coef[g] ln 2 log2(trunc9(a[n][g])) (see the module docstring); returns the cells' bounds"""
    got = np.asarray(got, np.float64)
    C, coef = np.asarray(C, np.float64)[None, :], np.asarray(coef, np.float64)[None, :]
    L_lo, L_hi = log2_interval(a, delta)
    s1, s2 = C + coef * LN2 * L_lo, C + coef * LN2 * L_hi
    lo, hi = np.minimum(s1, s2), np.maximum(s1, s2)
    L = np.maximum(np.abs(L_lo), np.abs(L_hi))
    tol = np.abs(coef * LN2) * (2.0 ** -22 * np.maximum(1.0, L) + 2.0 ** -23 * L) + 2.0 ** -23 * (np.abs(C) + np.abs(hi) + np.abs(lo)) + tol_C
    bad = ~((got >= lo - tol) & (got <= hi + tol))
    if bad.any():
        i = np.argwhere(bad)[0]
        raise AssertionError("%s: %d of %d cells outside the step-aware bound; first %s: got %.9g, want [%.9g, %.9g] +- %.3g, a = %.9g +- %.3g"
                             % (what, bad.sum(), bad.size, tuple(i), got[tuple(i)], lo[tuple(i)], hi[tuple(i)], tol[tuple(i)],
                                np.asarray(a)[tuple(i)], np.broadcast_to(delta, bad.shape)[tuple(i)]))
    return lo - tol, hi + tol


# ----------------------------------------------------------------------------------------------------- nich
def nich_workload(seed, G, N, scale, offset, outliers=True, overflow=False):
    """synth.nich's shape with data, mean and sqrt(sigmasq) scaled by `scale` and data + prior mean shifted by `offset`
    standard deviations; statistics formed in float64 and rounded once.  Rows 3::17 sit at 1e3 sigma, rows 5::17 at 1e6
    sigma; with overflow, rows 7::97 at 1e22 sigma (|x - mean| sqrt(precision) > 1.8e19: the argument overflows fp32)."""
    rng = np.random.default_rng(seed)
    sizes = synth._sizes(rng, G)
    centres = rng.normal(0.0, 3.0, G)
    mean, ctv = np.zeros(G, np.float32), np.zeros(G, np.float32)
    for g in range(G):
        if sizes[g]:
            x = scale * (rng.normal(centres[g], 1.0, sizes[g]) + offset)
            mean[g] = x.mean()
            ctv[g] = ((x - x.mean()) ** 2).sum()
    v = 3.0 * rng.standard_normal(N)
    if outliers:
        v[3::17] += 1e3
        v[5::17] -= 1e6
    if overflow:
        v[7::97] = 1e22
    return dict(model="nich", shared=np.array([scale * offset, 1.0, scale * scale, 1.0], np.float32), sizes=sizes,
                count=sizes.copy(), mean=mean, ctv=ctv, values=(scale * (v + offset)).astype(np.float32),
                u=rng.random(N, dtype=np.float32))


def nich_reference(caches, values):
    """(C, coef, a, delta_a) of the module docstring from cache rows (score_, log_coeff_, precision_, mean_)"""
    score_, log_coeff, precision, mean = (np.asarray(r, np.float64) for r in caches)
    x = np.asarray(values, np.float32).astype(np.float64)[:, None]
    with np.errstate(over="ignore"):
        a = 1.0 + precision[None, :] * (x - mean[None, :]) ** 2
    return score_, log_coeff, a, 4 * U * (a - 1.0) + U * a


NICH_SCALES = (1e-6, 1e-3, 1.0, 1e3, 1e6)
NICH_OFFSETS = (0.0, 1e2, 1e4)


def nich_sweep():
    for i, scale in enumerate(NICH_SCALES):
        for j, offset in enumerate(NICH_OFFSETS):
            yield scale, offset, (50, 100, 300)[(i + j) % 3]


# ------------------------------------------------------------------------------------------------------ NIW
def niw_workload(seed, G, N, d, std, offset):
    """synth.niw's shape with per-dimension standard deviation `std` (psi = std^2 I, group spread std, centres 3 std N(0, I))
    and data, prior mu and group sums shifted by `offset` standard deviations along the first axis; statistics formed in
    float64 and rounded once.  Sigma_g of every group is asserted SPD in float64 (niw_groups).  The shift is along one axis
    because fp32 sum_xxT keeps 2^-24 of |shift|^2: spread over all d axes at 1e3 sigma, that rounding alone outweighs the
    groups' covariance and Sigma_g is no longer SPD -- the statistics, not the scorer, have lost the data."""
    rng = np.random.default_rng(seed)
    sizes = synth._sizes(rng, G)
    shift = offset * std * (np.arange(d) == 0)
    centres = 3.0 * std * rng.standard_normal((G, d))
    sum_x, sum_xxT = np.zeros((G, d)), np.zeros((G, d, d))
    for g in range(G):
        if sizes[g]:
            x = centres[g] + shift + std * rng.standard_normal((sizes[g], d))
            sum_x[g], sum_xxT[g] = x.sum(0), x.T @ x
    which = rng.integers(0, G, N)
    values = centres[which] + shift + std * rng.standard_normal((N, d))
    return dict(model="niw", mu=shift.astype(np.float32), kappa=1.0, psi=(std * std * np.eye(d)).astype(np.float32), nu=float(d + 2),
                sizes=sizes, count=sizes.copy(), sum_x=sum_x.astype(np.float32), sum_xxT=sum_xxT.astype(np.float32),
                values=values.astype(np.float32), u=rng.random(N, dtype=np.float32))


def niw_groups(w, o, clamp_det=False):
    """per group, in float64 as niw_posterior_cholesky / niw_prep_kernel: mu' (rounded to fp32), W = L^-1, the constant C,
    coef = -0.5 (dof + d), dof, log det, det, tol_C.  clamp_det: take fast_log(float(det)) whatever det is (the old,
    clamped constant)."""
    from scipy.linalg import solve_triangular
    d = w["mu"].size
    mu, psi = w["mu"].astype(np.float64), w["psi"].astype(np.float64)
    kap, nu = float(np.float32(w["kappa"])), float(np.float32(w["nu"]))
    out = []
    for g in range(w["count"].size):
        n = float(w["count"][g])
        sx, sxx = w["sum_x"][g].astype(np.float64), w["sum_xxT"][g].astype(np.float64)
        pk, dof = kap + n, nu + n - d + 1.0
        xbar = sx / n if n else np.zeros(d)
        diff = xbar - mu
        c_n = sxx - np.outer(sx, xbar) - np.outer(xbar, sx) + n * np.outer(xbar, xbar)
        S = (psi + c_n + kap * n / (kap + n) * np.outer(diff, diff)) * (pk + 1.0) / (pk * dof)
        Lc = np.linalg.cholesky(S)  # raises unless SPD
        mu_p = (kap / (kap + n) * mu + n / (kap + n) * xbar).astype(np.float32).astype(np.float64)
        W = solve_triangular(Lc, np.eye(d), lower=True)
        diag = np.diag(Lc)
        logdet, det = 2.0 * np.log(diag).sum(), np.prod(diag * diag)
        dof_f = np.float32(dof)
        lg = o.fast_lgamma(np.array([dof_f / 2.0 + d / 2.0, dof_f / 2.0], np.float64).astype(np.float32)).astype(np.float64)
        det_f = np.float32(det) if np.isfinite(det) and det < FLT_MAX else np.float32(np.inf)
        normal = np.isfinite(det_f) and det_f >= np.finfo(np.float32).tiny
        ld = float(o.fast_log(np.array([det_f]))[0]) if (normal or clamp_det) else logdet
        term2 = -0.5 * ld - d / 2.0 * (float(o.fast_log(np.array([dof_f]))[0]) + LOG_PI_F)
        out.append(dict(mu_p=mu_p, W=W, C=lg[0] - lg[1] + term2, coef=-0.5 * (float(dof_f) + d), dof=float(dof_f), logdet=logdet,
                        det=det, normal=normal, S=S, tol_C=2.0 ** -22 * (abs(lg[0]) + abs(lg[1]) + abs(term2)) + 2.0 ** -23 * abs(ld)))
    return out


def _tile_scales(X):
    """the power-of-two scale 2^ex of each row's 128-row tile (niw_tc_pack_x_kernel: split_scale(max(max |x|, 1)))"""
    n = X.shape[0]
    sx = np.empty(n)
    for t0 in range(0, n, 128):
        m = max(float(np.abs(X[t0:t0 + 128]).max()), 1.0)
        sx[t0:t0 + 128] = 2.0 ** (13 - np.frexp(m)[1])
    return sx


def _group_scale(gr):
    """2^ew of a group (niw_tc_prep_kernel: split_scale of the largest |W| and |b|, fp32)"""
    W32 = gr["W"].astype(np.float32).astype(np.float64)
    b = np.tril(W32) @ gr["mu_p"]
    m = float(max(np.abs(W32).max(), np.abs(b.astype(np.float32)).max()))
    return 2.0 ** (13 - np.frexp(m)[1]), W32, b


def niw_reference(w, groups, values, route="fp32"):
    """(C, coef, a, delta_a, tol_C) for values[n][d] under `route` ("fp32" or "tc"); see the module docstring"""
    X = np.asarray(values, np.float32).astype(np.float64)
    n, d, G = X.shape[0], X.shape[1], len(groups)
    a, delta = np.empty((n, G)), np.empty((n, G))
    sx = _tile_scales(X) if route == "tc" else None
    absX = np.abs(X)
    for g, gr in enumerate(groups):
        Z = X - gr["mu_p"][None, :]
        Y = Z @ gr["W"].T
        q = (Y * Y).sum(1)
        absW = np.abs(gr["W"])
        if route == "fp32":
            # y_i = sum_{j <= i} W_ij z_j by fmaf in ascending j: each step rounds its partial sum s_ij
            P = np.cumsum(Z[:, None, :] * gr["W"][None, :, :], axis=2)
            e = 2 * U * (np.abs(Z) @ absW.T) + 1.01 * U * np.abs(np.tril(np.ones((d, d)))[None] * P).sum(2)
            Qp = U * np.abs(np.cumsum(Y * Y, axis=1)).sum(1)
        else:
            sw, _, _ = _group_scale(gr)
            A = absX @ absW.T
            B = (absW @ np.abs(gr["mu_p"]))[None, :]
            e = ((3 * 2.0 ** -22 + U + 112 * 2.0 ** -23) * A + (2.0 ** -22 + 2 * U + 112 * 2.0 ** -23) * B
                 + 2.0 ** -25 * (absW.sum(1)[None, :] / sx[:, None] + (absX.sum(1)[:, None] + 1.0) / sw))
            Qp = (d + 3) * U * q
        dq = (2 * np.abs(Y) * e + e * e).sum(1) + Qp
        with np.errstate(over="ignore"):
            a[:, g] = 1.0 + q / gr["dof"]
        delta[:, g] = (dq + 2 * U * q) / gr["dof"] + U * a[:, g]
    C = np.array([gr["C"] for gr in groups])
    coef = np.array([gr["coef"] for gr in groups])
    tol_C = np.array([gr["tol_C"] for gr in groups])[None, :]
    return C, coef, a, delta, tol_C


NIW_DIMS = (3, 8, 16, 32)
NIW_STDS = (1e-3, 0.1, 1.0, 10.0, 1e3)
NIW_OFFSETS = (0.0, 1e2, 1e3)


def niw_sweep():
    """every (d, std, offset); G rotates through 9, 70, 256 -- except at 1e3 sigma, where a few of 256 groups' fp32
    sum_xxT have lost their covariance to rounding (Sigma_g not SPD, niw_workload), so G rotates through 9, 70"""
    k = 0
    for d in NIW_DIMS:
        for std in NIW_STDS:
            for offset in NIW_OFFSETS:
                yield d, std, offset, (9, 70)[k % 2] if offset >= 1e3 else (9, 70, 256)[k % 3]
                k += 1


def _seed(*xs):
    return int(abs(hash(tuple(round(np.log10(x), 3) if x > 0 else -9 for x in xs))) % 100000) + 17


# ================================================================================ CPU self-tests of the checkers
def test_nich_checker_accepts_oracle(oracle):
    """non-vacuous: the fp32 oracle restatement (the reference's arithmetic, fast_log(inf) = 128 ln 2 included) passes the
    nich checker on every nich sweep case, overflowing rows included"""
    for scale, offset, G in nich_sweep():
        w = nich_workload(_seed(scale, offset + 1, G), G, 600, scale, offset, overflow=True)
        caches = oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])
        got = oracle.score_rows(cases.MODEL_ID["nich"], caches, w["values"], np.zeros((600, G), np.float32))
        C, coef, a, delta = nich_reference(caches, w["values"])
        assert overflows(a, delta).any()
        check_step_aware(got, C, coef, a, delta, what="oracle nich scale %g offset %g" % (scale, offset))


def oracle_niw_slack(w, groups, values, oracle):
    """what the oracle's own arithmetic adds to the FP32 bound: orc_niw_score_rows forms the posterior in fp32 (niw.hpp's
    float expressions), so its sigma differs from the float64 one by at most, entrywise,
        E_S = 8 u (|psi| + |sxx| + 2 |sx xbar^T| + n |xbar xbar^T| + kappa n / (kappa + n) |diff diff^T|) (k' + 1) / (k' dof)
    (each term's fp32 rounding, the sums and the scaling).  To first order, with P = Sigma^-1:
        log det:  |d logdet| <= sum |P| E_S                      -> tol_C += 0.5 x 1.1 x that, plus the table steps
                                                                    between fast_log(det e^-+dlogdet) and fast_log(det);
        q:        |dq| <= 1.1 |P z|^T E_S |P z| + (d + 3) u |z|^T |P| |z|   (fp32 Sigma^-1, its float quadratic form,
                  fl(x - mu')) + 2 |P z| . dmu' + dmu'^T |P| dmu',  dmu' = 4 u (|kappa mu| + |n xbar|) / (kappa + n)
    Returns (extra delta_a [n][G], extra tol_C [G], first-order size max_g sum |P| E_S); the first-order argument holds
    while that size is small (<= 0.05)."""
    d = w["mu"].size
    X = np.asarray(values, np.float32).astype(np.float64)
    mu, psi, kap, nu = w["mu"].astype(np.float64), w["psi"].astype(np.float64), float(w["kappa"]), float(w["nu"])
    dA, dC, size = np.empty((X.shape[0], len(groups))), np.empty(len(groups)), 0.0
    for g, gr in enumerate(groups):
        n = float(w["count"][g])
        sx, sxx = w["sum_x"][g].astype(np.float64), w["sum_xxT"][g].astype(np.float64)
        pk, dof = kap + n, nu + n - d + 1.0
        xbar = sx / n if n else np.zeros(d)
        diff = xbar - mu
        E = 8 * U * (np.abs(psi) + np.abs(sxx) + 2 * np.abs(np.outer(sx, xbar)) + n * np.abs(np.outer(xbar, xbar))
                     + kap * n / (kap + n) * np.abs(np.outer(diff, diff))) * (pk + 1.0) / (pk * dof)
        P = gr["W"].T @ gr["W"]
        dlog = float((np.abs(P) * E).sum())
        size = max(size, dlog)
        ld = lambda det: float(oracle.fast_log(np.array([det], np.float32))[0]) if gr["normal"] else np.log(det)  # noqa: E731
        steps = max(abs(ld(gr["det"] * np.exp(s * 1.1 * dlog)) - ld(gr["det"])) for s in (-1.0, 1.0)) if gr["normal"] else 0.0
        dC[g] = 0.5 * (1.1 * dlog + steps)
        Z = X - gr["mu_p"][None, :]
        PZ = Z @ P
        dmu = 4 * U * (np.abs(kap * mu) + np.abs(n * xbar)) / (kap + n)
        dq = (1.1 * ((np.abs(PZ) @ E) * np.abs(PZ)).sum(1) + (d + 3) * U * ((np.abs(Z) @ np.abs(P)) * np.abs(Z)).sum(1)
              + 2 * np.abs(PZ) @ dmu + dmu @ np.abs(P) @ dmu)
        dA[:, g] = dq / gr["dof"]
    return dA, dC, size


def test_niw_checker_accepts_oracle(oracle):
    """non-vacuous: orc_niw_score_rows (fp32 restatement of Scorer::eval, now with the niw_log_det policy) passes the NIW
    checker -- FP32 bound plus the derived slack of its fp32 posterior (oracle_niw_slack) -- on every sweep case where
    that slack is first-order small: every unshifted case (both sides of every d's det window) and most at 1e2 sigma.  At
    1e3 sigma the oracle's fp32 c_n = sxx - ... cancels about |shift|^2 / std^2 u = 6 % of sigma: not a small perturbation."""
    seen_clamped, seen = 0, []
    for d, std, offset, G in niw_sweep():
        w = niw_workload(_seed(d, std, offset + 1, G), G, 200, d, std, offset)
        groups = niw_groups(w, oracle)
        dA, dC, size = oracle_niw_slack(w, groups, w["values"], oracle)
        if size > 0.05:
            assert offset > 0, (d, std, size)
            continue
        seen.append(offset)
        seen_clamped += sum(not gr["normal"] for gr in groups)
        got = oracle.niw_score_rows(w["mu"], w["kappa"], w["psi"], w["nu"], w["count"], w["sum_x"], w["sum_xxT"], w["values"],
                                    np.zeros((200, G), np.float32))
        C, coef, a, delta, tol_C = niw_reference(w, groups, w["values"])
        check_step_aware(got, C, coef, a, delta + dA, tol_C + dC[None, :], what="oracle niw d %d std %g offset %g" % (d, std, offset))
    assert seen.count(0.0) == len(NIW_DIMS) * len(NIW_STDS) and seen.count(1e2) > 0 and seen_clamped > 0  # the sweep reaches past the normal-float det window


def _split16(v):
    hi = v.astype(np.float16).astype(np.float64)
    return hi, (v - hi).astype(np.float16).astype(np.float64)


def split_fp16_scores(w, groups, values):
    """numpy emulation of the tensor-core route: niw_tc_pack_x_kernel's per-tile split of [x | 1] 2^ex and
    niw_tc_prep_kernel's per-group split of [W | -b] 2^ew (fp16, round to nearest), the three products hi hi + lo hi + hi lo
    and the augmented column, accumulated in float64; the log as the kernels take it"""
    X = np.asarray(values, np.float32).astype(np.float64)
    sx = _tile_scales(X)
    xh, xl = _split16(X * sx[:, None])
    out = np.empty((X.shape[0], len(groups)))
    for g, gr in enumerate(groups):
        sw, W32, b = _group_scale(gr)
        wh, wl = _split16(W32 * sw)
        nb = -b.astype(np.float32).astype(np.float64) * sw
        bh, bl = _split16(nb)
        acc = xh @ wh.T + xl @ wh.T + xh @ wl.T + sx[:, None] * (bh + bl)[None, :]
        q = ((acc / (sx[:, None] * sw)) ** 2).sum(1).astype(np.float32)
        arg = (np.float32(1) + np.float32(1.0 / np.float32(gr["dof"])) * q).astype(np.float32)
        out[:, g] = gr["C"] + gr["coef"] * LN2 * _log2_step(arg)
    return out


def test_niw_checker_rejects_split_fp16_at_offset(oracle):
    """has power: the split-fp16 form at 1000 sigma offset misses the FP32 bound (its error follows |W x|, not |W (x - mu')|),
    while its own derived bound holds -- on the same data at offset 0 it meets the FP32 bound too"""
    w = niw_workload(4242, 9, 256, 32, 1.0, 1e3)
    groups = niw_groups(w, oracle)
    got = split_fp16_scores(w, groups, w["values"])
    C, coef, a, delta, tol_C = niw_reference(w, groups, w["values"])
    with pytest.raises(AssertionError):
        check_step_aware(got, C, coef, a, delta, tol_C, what="split fp16, fp32 bound")
    C, coef, a, delta, tol_C = niw_reference(w, groups, w["values"], route="tc")
    check_step_aware(got, C, coef, a, delta, tol_C, what="split fp16, tc bound")
    w0 = niw_workload(4242, 9, 256, 32, 1.0, 0.0)
    g0 = niw_groups(w0, oracle)
    check_step_aware(split_fp16_scores(w0, g0, w0["values"]), *niw_reference(w0, g0, w0["values"])[:4], tol_C=niw_reference(w0, g0, w0["values"])[4],
                     what="split fp16 at offset 0, fp32 bound")


def test_niw_checker_rejects_clamped_det(oracle):
    """has power: at d = 32, std 10 the determinant overflows fp32; the old constant -0.5 fast_log(float(det)) sticks at
    -0.5 * 128 ln 2 and fails the checker"""
    w = niw_workload(4343, 9, 64, 32, 10.0, 0.0)
    groups = niw_groups(w, oracle)
    assert not any(gr["normal"] for gr in groups)
    clamped = niw_groups(w, oracle, clamp_det=True)
    C, coef, a, delta, tol_C = niw_reference(w, groups, w["values"])
    got = np.array([gr["C"] for gr in clamped])[None, :] + coef[None, :] * LN2 * _log2_step(a)
    with pytest.raises(AssertionError):
        check_step_aware(got, C, coef, a, delta, tol_C, what="clamped det")
    want = np.array([gr["C"] for gr in groups])[None, :] + coef[None, :] * LN2 * _log2_step(a)
    check_step_aware(want, C, coef, a, delta, tol_C, what="exact log det")


# ============================================================================================== GPU sweep
torch = pytest.importorskip("torch")


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


def _feature(ctx, w):
    from distributions_b200 import capi
    return ctx.feature({"nich": capi.NICH, "niw": capi.NIW, "gp": capi.GP, "bb": capi.BB}[w["model"]]).update_all(w)


def _col(w, n=None):
    from distributions_b200 import capi
    m = {"nich": capi.NICH, "niw": capi.NIW, "gp": capi.GP, "bb": capi.BB}[w["model"]]
    v = w["values"] if n is None else w["values"][:n]
    return dev(np.ascontiguousarray(v, dtype=capi.COLUMN_DTYPE[m]))


def _score(ctx, feats, cols, n, G, prior=None, opts=None):
    opts = opts or {}
    for k, v in opts.items():
        ctx.set_option(k, v)
    try:
        sc = torch.full((n, G), 777.0, device="cuda")
        ctx.score_batch(feats, cols, n, None if prior is None else dev(prior), sc)
        torch.cuda.synchronize()
    finally:
        for k in opts:
            ctx.set_option(k, 0)
    return sc.cpu().numpy()


def _sample(ctx, feats, cols, n, G, prior, u, want_scores, opts=None):
    opts = opts or {}
    for k, v in opts.items():
        ctx.set_option(k, v)
    try:
        sc = torch.full((n, G), 777.0, device="cuda") if want_scores else None
        assign = torch.full((n,), -5, device="cuda", dtype=torch.int32)
        ctx.score_sample_batch(feats, cols, n, dev(prior), dev(u), assign, sc)
        torch.cuda.synchronize()
    finally:
        for k in opts:
            ctx.set_option(k, 0)
    return assign.cpu().numpy(), (sc.cpu().numpy() if want_scores else None)


def _logp(ctx, feats, cols, n, prior):
    out = torch.full((n,), 777.0, device="cuda")
    ctx.score_logp_batch(feats, cols, n, dev(prior), out)
    torch.cuda.synchronize()
    return out.cpu().numpy().astype(np.float64)


def _lse(s):
    m = np.max(s, axis=1, keepdims=True)
    return (m + np.log(np.exp(s - m).sum(1, keepdims=True)))[:, 0]


def check_logp(got, lo, hi, prior):
    """logp against the float64 logsumexp of the reference interval shifted by the prior"""
    lo, hi = lo + prior[None, :], hi + prior[None, :]
    tol = 2.0 ** -21 * (1 + np.abs(hi).max(1)) + (lo.shape[1] + 8) * 2.0 ** -24
    assert np.all(got >= _lse(lo) - tol) and np.all(got <= _lse(hi) + tol), np.max(np.maximum(_lse(lo) - tol - got, got - _lse(hi) - tol))


def check_fused(name, a_fused, a_mat, scores, u):
    """the sampling-only launch against the materialising launch: identical or a proven near-tie, and rare"""
    assert a_fused.min() >= 0 and a_fused.max() < scores.shape[1], name
    diff = np.nonzero(a_fused != a_mat)[0]
    assert diff.size <= max(2, 2e-3 * a_mat.size), (name, diff.size)
    if diff.size:
        assert cases.explained_mismatch(scores[diff].astype(np.float64), u[diff], a_mat[diff], a_fused[diff], EPS_TIE).all(), name


@pytest.mark.gpu
@pytest.mark.parametrize("scale,offset,G", list(nich_sweep()))
def test_nich_conditioning(ctx, oracle, scale, offset, G):
    """score_batch step-aware against float64, every nich sampling-only option set against the materialising launch,
    score_logp_batch against the float64 logsumexp; scales 1e-6 .. 1e6, offsets to 1e4 sigma, outliers at 1e3 / 1e6 sigma"""
    n = 2048
    w = nich_workload(_seed(scale, offset + 1, G), G, n, scale, offset)
    f = _feature(ctx, w)
    caches = f.download_caches(4)
    for got_row, want_row in zip(caches, oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])):
        np.testing.assert_allclose(got_row, want_row, rtol=2e-6, atol=2e-6 * np.abs(want_row).max())
    col = _col(w)
    got = _score(ctx, [f], [col], n, G)
    C, coef, a, delta = nich_reference(caches, w["values"])
    lo, hi = check_step_aware(got, C, coef, a, delta, what="nich score_batch scale %g offset %g G %d" % (scale, offset, G))
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    a_mat, s_mat = _sample(ctx, [f], [col], n, G, prior, w["u"], True)
    for name, opts in NICH_FUSED.items():
        a_f, _ = _sample(ctx, [f], [col], n, G, prior, w["u"], False, opts)
        check_fused(name, a_f, a_mat, s_mat, w["u"])
    check_logp(_logp(ctx, [f], [col], n, prior), lo, hi, prior.astype(np.float64))


@pytest.mark.gpu
@pytest.mark.parametrize("G", [100, 300])
def test_nich_conditioning_crosscat(ctx, G):
    """one cross-cat list nich + gp + bb at offset 1e4 sigma, scale 1e3: the list's score is the nich reference interval
    plus the library's gp and bb scores, within the list's fp32 accumulation (2^-23 per term)"""
    n = 1024
    w = nich_workload(900 + G, G, n, 1e3, 1e4)
    wg, wb = synth.gp(901 + G, G, n), synth.bb(902 + G, G, n)
    wg["sizes"] = wb["sizes"] = w["sizes"]
    fs = [_feature(ctx, x) for x in (w, wg, wb)]
    cols = [_col(x) for x in (w, wg, wb)]
    got = _score(ctx, fs, cols, n, G).astype(np.float64)
    other = _score(ctx, fs[1:2], cols[1:2], n, G).astype(np.float64) + _score(ctx, fs[2:], cols[2:], n, G).astype(np.float64)
    C, coef, a, delta = nich_reference(fs[0].download_caches(4), w["values"])
    # the nich part: got - other, whose rounding is 2^-23 (|got| + |other|) on top of the nich bound
    slack = 2.0 ** -23 * (np.abs(got) + 2 * np.abs(other))
    lo, hi = log2_interval(a, delta)
    s1, s2 = C[None, :] + coef[None, :] * LN2 * lo, C[None, :] + coef[None, :] * LN2 * hi
    L = np.maximum(np.abs(lo), np.abs(hi))
    tol = np.abs(coef[None, :] * LN2) * (2.0 ** -22 * np.maximum(1.0, L) + 2.0 ** -23 * L) + 2.0 ** -23 * (np.abs(C)[None, :] + np.abs(s1)) + slack
    part = got - other
    assert np.all(part >= np.minimum(s1, s2) - tol) and np.all(part <= np.maximum(s1, s2) + tol)


def _niw_routes(ctx, oracle, w, n, what, tc_domain=None):
    """score_batch on the default route (tensor cores at d = 32) and, at d = 32, the FP32 kernel on the same feature; the
    sampling-only launch against the materialising one.  At d = 32 the tensor-core route is held to its own derived bound
    on every row and to the FP32 bound on the rows of tc_domain (a row mask: rows inside the route's stated domain,
    DESIGN §6 -- data and prior mean within a few standard deviations of the origin, no far-larger row in the tile)."""
    d, G = w["mu"].size, w["count"].size
    groups = niw_groups(w, oracle)
    f = _feature(ctx, w)
    col = _col(w, n)
    vals = w["values"][:n]
    got = _score(ctx, [f], [col], n, G)
    ref = niw_reference(w, groups, vals, route="tc" if d == 32 else "fp32")
    lo, hi = check_step_aware(got, *ref[:4], tol_C=ref[4], what=what + (" tc" if d == 32 else " fp32"))
    if d == 32:
        got32 = _score(ctx, [f], [col], n, G, opts={3: 1})
        ref32 = niw_reference(w, groups, vals, route="fp32")
        check_step_aware(got32, *ref32[:4], tol_C=ref32[4], what=what + " fp32 kernel")
        if tc_domain is not None:
            check_step_aware(got[tc_domain], ref32[0], ref32[1], ref32[2][tc_domain], ref32[3][tc_domain], tol_C=ref32[4],
                             what=what + " tc inside its domain, fp32 bound")
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    u = w["u"][:n]
    a_mat, s_mat = _sample(ctx, [f], [col], n, G, prior, u, True)
    a_f, _ = _sample(ctx, [f], [col], n, G, prior, u, False)
    check_fused(what + " fused", a_f, a_mat, s_mat, u)
    return f, col, groups, lo, hi, prior


@pytest.mark.gpu
@pytest.mark.parametrize("d,std,offset,G", list(niw_sweep()))
def test_niw_conditioning(ctx, oracle, d, std, offset, G):
    """NIW d in {3, 8, 16, 32} (niw_rows_kernel, niw_score_kernel dp 4 / 8 / 16 / 32, tensor cores), std 1e-3 .. 1e3 (both
    sides of every d's det window), offsets to 1e3 sigma, G in {9, 70, 256}"""
    n = 512
    w = niw_workload(_seed(d, std, offset + 1, G), G, n, d, std, offset)
    _niw_routes(ctx, oracle, w, n, "niw d %d std %g offset %g G %d" % (d, std, offset, G),
                tc_domain=np.ones(n, bool) if offset == 0 else None)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [127, 128, 129, 511, 512, 513, 4097])
def test_niw_tc_tile_edges(ctx, oracle, n):
    """d = 32 on the tensor cores at row counts around the 128-row tile and the 512-row chunk"""
    w = niw_workload(5000 + n, 70, n, 32, 1.0, 0.0)
    _niw_routes(ctx, oracle, w, n, "niw tc n %d" % n, tc_domain=np.ones(n, bool))


@pytest.mark.gpu
def test_niw_tc_mixed_tiles(ctx, oracle):
    """d = 32: one 128-row tile holding a row x1e4 and a row x1e6 (the tile scale follows them: its other rows keep the
    derived bound only; the other tiles, the FP32 bound),
    a tile of exact zeros and a tile of rows placed exactly at mu'_g; score_logp_batch; a mixed nich + NIW(32) list
    (materialising tensor-core route with accumulate)"""
    G, n = 70, 640
    w = niw_workload(5151, G, n, 32, 1.0, 0.0)
    groups = niw_groups(w, oracle)
    v = w["values"].copy()
    v[5] *= 1e4
    v[70] *= 1e6
    v[256:384] = 0.0
    for r in range(384, 512):
        v[r] = groups[r % G]["mu_p"].astype(np.float32)
    w["values"] = v
    f, col, groups, lo, hi, prior = _niw_routes(ctx, oracle, w, n, "niw tc mixed tiles", tc_domain=np.arange(n) >= 128)
    check_logp(_logp(ctx, [f], [col], n, prior), lo, hi, prior.astype(np.float64))
    wn = nich_workload(5152, G, n, 1.0, 0.0)
    wn["sizes"] = w["sizes"]
    fn = _feature(ctx, wn)
    coln = _col(wn)
    both = _score(ctx, [fn, f], [coln, col], n, G).astype(np.float64)
    alone = _score(ctx, [fn], [coln], n, G).astype(np.float64)
    part = both - alone
    tol = 2.0 ** -23 * (np.abs(both) + 2 * np.abs(alone))
    assert np.all(part >= lo - tol) and np.all(part <= hi + tol)


@pytest.mark.gpu
def test_overflowing_argument_is_minus_inf(ctx, oracle):
    """the documented precondition (DESIGN §4): a cell whose log argument overflows fp32 scores -inf on every route --
    the reference's table would give 128 ln 2 -- every other cell meets its bound, score_logp_batch gives -inf for a row
    that overflows in every group, and the other rows' draws are those of a batch without the overflowing rows"""
    G, n = 100, 1024
    w = nich_workload(6060, G, n, 1.0, 0.0, outliers=False, overflow=True)
    f = _feature(ctx, w)
    col = _col(w)
    caches = f.download_caches(4)
    C, coef, a, delta = nich_reference(caches, w["values"])
    ovf = overflows(a, delta)
    rows = ovf.all(1)
    assert rows.sum() == len(range(7, n, 97))
    got = _score(ctx, [f], [col], n, G)
    assert np.all(got[ovf] == -np.inf)
    check_step_aware(got[~rows], C, coef, a[~rows], delta[~rows], what="nich rows beside overflowing ones")
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    logp = _logp(ctx, [f], [col], n, prior)
    assert np.all(logp[rows] == -np.inf) and np.all(np.isfinite(logp[~rows]))
    keep = np.nonzero(~rows)[0]
    colk = _col(dict(w, values=w["values"][keep]))
    ref_a, ref_s = _sample(ctx, [f], [colk], keep.size, G, prior, w["u"][keep], True)
    a_m, s_m = _sample(ctx, [f], [col], n, G, prior, w["u"], True)  # the materialising route
    assert np.all(s_m[ovf] == -np.inf) and np.array_equal(s_m[keep], ref_s) and np.array_equal(a_m[keep], ref_a)
    for name, opts in NICH_FUSED.items():
        a_f, _ = _sample(ctx, [f], [col], n, G, prior, w["u"], False, opts)
        check_fused("nich overflow " + name, a_f[keep], ref_a, ref_s, w["u"][keep])

    # NIW d = 32: overflowing rows in the first 128-row tile only.  The tensor-core route scales each tile by the power
    # of two of its largest |x| (DESIGN §6): the other rows of that tile lose their bits to that scale and score NaN, so
    # on that route the rows of the other tiles are held to the bound; the FP32 kernel is held to it on every other row.
    d, n = 32, 512
    wn = niw_workload(6161, 9, n, d, 1.0, 0.0)
    groups = niw_groups(wn, oracle)
    vn = wn["values"].copy()
    rows = np.zeros(n, bool)
    rows[3:128:50] = True
    vn[rows] = 1e30
    wn["values"] = vn
    fw = _feature(ctx, wn)
    cw = _col(wn)
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, wn["sizes"])
    tile0 = (np.arange(n) < 128) & ~rows
    for opts, keep in (({}, np.arange(n) >= 128), ({3: 1}, ~rows)):
        got = _score(ctx, [fw], [cw], n, 9, opts=opts)
        assert np.all(got[rows] == -np.inf), opts
        ref = niw_reference(wn, groups, vn[keep], route="fp32" if opts else "tc")
        check_step_aware(got[keep], *ref[:4], tol_C=ref[4], what="niw rows beside overflowing ones %s" % opts)
        if not opts:  # the tile's unscale^2 overflows fp32 (DESIGN §6): its other rows are NaN
            assert np.all(np.isnan(got[tile0]))
        ki = np.nonzero(keep)[0]
        colk = _col(dict(wn, values=vn[ki]))
        ref_a, ref_s = _sample(ctx, [fw], [colk], ki.size, 9, prior, wn["u"][ki], True, opts)
        a_m, s_m = _sample(ctx, [fw], [cw], n, 9, prior, wn["u"], True, opts)
        assert np.all(s_m[rows] == -np.inf) and np.array_equal(s_m[ki], ref_s) and np.array_equal(a_m[ki], ref_a), opts
        a_f, _ = _sample(ctx, [fw], [cw], n, 9, prior, wn["u"], False, opts)
        check_fused("niw overflow fused %s" % opts, a_f[ki], ref_a, ref_s, wn["u"][ki])
    logp = _logp(ctx, [fw], [cw], n, prior)
    assert np.all(logp[rows] == -np.inf) and np.all(np.isfinite(logp[128:]))
