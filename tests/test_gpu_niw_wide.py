"""NormalInverseWishart at 32 < d <= 128: the tensor-core route of niw_tc_wide.cu and every other NIW entry at those d.

The wide route scores x - mu0 (mu0 = Shared.mu) against b_g = W_g (mu'_g - mu0), both operands split in two fp16 terms:
    x' = fl(x - mu0),  x' 2^ex = x_hi + x_lo (per 128-row tile),  [W_g | -b_g] 2^ew = hi + lo (per group),
    acc = x_hi W_hi + x_lo W_hi + x_hi W_lo + [1 1] [-b_hi -b_lo],  q = |acc|^2 2^-2(ex + ew).
Derived bound of one element y_i = (W x')_i - b_i (DESIGN.md section 6, "d > 32").  With A_i = sum_j |W_ij| |x'_j|,
B_i = sum_j |W_ij| |mu'_j - mu0_j| (>= |b_i|), DP the padded dimension and n = 3 DP + 16 the products the accumulator sums:
    e_i = (3 2^-22 + 2 u + n 2^-23) A_i + (2^-22 + 2 u + n 2^-23) B_i + 2^-25 (sum_j |W_ij| / sx + (sum_j |x'_j| + 1) / sw)
(the x split, the W split and the dropped lo lo term 2^-22 A each; fl(x - mu0) and W's fp32 rounding u A each; b's fp32
rounding and its split; one rounding of at most 2^-23 of the running sum per accumulated product; fp16's subnormal
quantum in the scaled units), and delta_a as test_gpu_conditioning's FP32 route with (DP / 2 + 3) u q for the epilogue's
paired sums of squares.  The error follows |W (x - mu0)| + |W (mu' - mu0)|: the spread of the data around the prior mean,
not its offset from the origin.
"""
import numpy as np
import pytest

from distributions_b200 import capi, synth
from test_gpu_niw_stats import expected_after, stats_of
from test_gpu_conditioning import LN2, U, _log2_step, _tile_scales, check_step_aware, niw_groups, niw_reference, niw_workload

torch = pytest.importorskip("torch")

DIST_B200_ERR_UNSUPPORTED = 3  # include/dist_b200.h


def _padded(d):
    return 64 if d <= 64 else 128


def wide_groups(w, o):
    """niw_groups with mu' kept in float64, as niw_prep_wide_kernel forms b from it"""
    groups = niw_groups(w, o)
    mu, kap = w["mu"].astype(np.float64), float(np.float32(w["kappa"]))
    for g, gr in enumerate(groups):
        n = float(w["count"][g])
        xbar = w["sum_x"][g].astype(np.float64) / n if n else np.zeros(mu.size)
        gr["mu_p"] = kap / (kap + n) * mu + n / (kap + n) * xbar
    return groups


def spd_workload(o, seed, G, n, d, std, offset):
    """niw_workload at the first seed from `seed` on whose groups' Sigma_g stay SPD in float64 -- at 1e3 sigma and d >= 64
    the fp32 sum_xxT of some draws have lost their covariance to rounding (niw_workload)"""
    for s in range(seed, seed + 200):
        w = niw_workload(s, G, n, d, std, offset)
        try:
            return w, wide_groups(w, o)
        except np.linalg.LinAlgError:
            continue
    raise AssertionError("no SPD workload")


def _centred(w, values):
    return (np.asarray(values, np.float32) - np.asarray(w["mu"], np.float32)).astype(np.float64)


def _wide_group_scale(gr, m):
    W32 = gr["W"].astype(np.float32).astype(np.float64)
    b = gr["W"] @ m
    mm = float(max(np.abs(W32).max(), np.abs(b.astype(np.float32)).max()))
    return 2.0 ** (13 - np.frexp(mm)[1]), W32, b


def wide_reference(w, groups, values):
    """(C, coef, a, delta_a, tol_C) of the wide route's derived bound (module docstring)"""
    X = np.asarray(values, np.float32).astype(np.float64)
    Xc = _centred(w, values)
    n, d, G = X.shape[0], X.shape[1], len(groups)
    dp = _padded(d)
    nacc = 3 * dp + 16
    sx = _tile_scales(Xc)
    absX = np.abs(Xc)
    mu0 = w["mu"].astype(np.float64)
    a, delta = np.empty((n, G)), np.empty((n, G))
    for g, gr in enumerate(groups):
        m = gr["mu_p"] - mu0
        sw, _, _ = _wide_group_scale(gr, m)
        Y = (X - gr["mu_p"][None, :]) @ gr["W"].T
        q = (Y * Y).sum(1)
        absW = np.abs(gr["W"])
        A = absX @ absW.T
        B = (absW @ np.abs(m))[None, :]
        e = ((3 * 2.0 ** -22 + 2 * U + nacc * 2.0 ** -23) * A + (2.0 ** -22 + 2 * U + nacc * 2.0 ** -23) * B
             + 2.0 ** -25 * (absW.sum(1)[None, :] / sx[:, None] + (absX.sum(1)[:, None] + 1.0) / sw))
        dq = (2 * np.abs(Y) * e + e * e).sum(1) + (dp / 2 + 3) * U * q
        with np.errstate(over="ignore"):
            a[:, g] = 1.0 + q / gr["dof"]
        delta[:, g] = (dq + 2 * U * q) / gr["dof"] + U * a[:, g]
    C = np.array([gr["C"] for gr in groups])
    coef = np.array([gr["coef"] for gr in groups])
    tol_C = np.array([gr["tol_C"] for gr in groups])[None, :]
    return C, coef, a, delta, tol_C


def _split16(v):
    hi = v.astype(np.float16).astype(np.float64)
    return hi, (v - hi).astype(np.float16).astype(np.float64)


def emulate_wide(w, groups, values, centre=True):
    """numpy emulation of the wide route: the (centred) per-tile split of [x' | 1 | 1], the per-group split of [W | -b],
    the three products and the augmented column accumulated in fp32, the log as the kernels take it.  centre=False: the
    same with mu0 = 0 (b = W mu')"""
    mu0 = w["mu"].astype(np.float32) if centre else np.zeros(w["mu"].size, np.float32)
    Xc = (np.asarray(values, np.float32) - mu0).astype(np.float64)
    sx = _tile_scales(Xc)
    xh, xl = _split16(Xc * sx[:, None])
    out = np.empty((Xc.shape[0], len(groups)))
    f32 = np.float32
    for g, gr in enumerate(groups):
        sw, W32, b = _wide_group_scale(gr, gr["mu_p"] - mu0.astype(np.float64))
        wh, wl = _split16(W32 * sw)
        bh, bl = _split16(-b.astype(np.float32).astype(np.float64) * sw)
        acc = (xh.astype(f32) @ wh.T.astype(f32)) + (xl.astype(f32) @ wh.T.astype(f32)) + (xh.astype(f32) @ wl.T.astype(f32))
        acc = acc + (sx[:, None] * bh[None, :]).astype(f32) + (sx[:, None] * bl[None, :]).astype(f32)
        q = ((acc.astype(np.float64) / (sx[:, None] * sw)) ** 2).sum(1).astype(f32)
        arg = (f32(1) + f32(1.0 / f32(gr["dof"])) * q).astype(f32)
        out[:, g] = gr["C"] + gr["coef"] * LN2 * _log2_step(arg)
    return out


# ======================================================================================================= CPU
@pytest.mark.parametrize("offset", [0.0, 1e2, 1e3])
def test_emulation_meets_derived_bound(oracle, offset):
    """the centred split-fp16 emulation passes the checker with the derived bound at 0, 1e2 and 1e3 sigma"""
    d = 100
    w, groups = spd_workload(oracle, 7100 + int(offset), 9, 256, d, 1.0, offset)
    got = emulate_wide(w, groups, w["values"])
    C, coef, a, delta, tol_C = wide_reference(w, groups, w["values"])
    check_step_aware(got, C, coef, a, delta, tol_C, what="wide emulation, derived bound, offset %g" % offset)


def test_uncentred_emulation_fails_fp32_bound(oracle):
    """has power: without centring, at 1e3 sigma the split error follows |W x| and misses the FP32 bound"""
    w, groups = spd_workload(oracle, 7200, 9, 256, 100, 1.0, 1e3)
    got = emulate_wide(w, groups, w["values"], centre=False)
    ref32 = niw_reference(w, groups, w["values"], route="fp32")
    with pytest.raises(AssertionError):
        check_step_aware(got, *ref32[:4], tol_C=ref32[4], what="uncentred emulation, fp32 bound")


def test_wire_round_trip_d100():
    d, G = 100, 5
    rng = np.random.default_rng(11)
    A = rng.normal(size=(d, d))
    psi = (A @ A.T / d + np.eye(d)).astype(np.float32)
    shared = np.concatenate([[1.5, d + 3.0], rng.normal(size=d), psi.ravel()]).astype(np.float32)
    msg = capi.wire_encode_shared(capi.NIW, shared)
    sxx = rng.normal(size=(G, d, d))
    sxx = (sxx + sxx.transpose(0, 2, 1)).astype(np.float32)
    stats = np.concatenate([np.arange(G, dtype=np.uint32), rng.normal(size=G * d).astype(np.float32).view(np.uint32),
                            sxx.ravel().view(np.uint32)])
    groups = capi.wire_encode_groups(capi.NIW, G, d, None, stats)
    sh, _, st = capi.wire_decode(capi.NIW, msg, groups)
    assert np.array_equal(sh.view(np.uint32), shared.view(np.uint32)) and np.array_equal(st, stats)


def test_wire_rejects_d129():
    """dim above 128: the Shared writer refuses it and the decoder returns DIST_B200_ERR_UNSUPPORTED"""
    import struct
    d = 129
    shared = np.concatenate([[1.0, d + 2.0], np.zeros(d), np.eye(d).ravel()]).astype(np.float32)
    with pytest.raises(ValueError):
        capi.wire_encode_shared(capi.NIW, shared)
    # mu (field 1), kappa (2), psi (3), nu (4), every value a fixed32
    body = b"".join(b"\x0d" + struct.pack("<f", 0.0) for _ in range(d)) + b"\x15" + struct.pack("<f", 1.0)
    body += b"".join(b"\x1d" + struct.pack("<f", v) for v in np.eye(d).ravel()) + b"\x25" + struct.pack("<f", d + 2.0)
    with pytest.raises(ValueError, match="status %d" % DIST_B200_ERR_UNSUPPORTED):
        capi.wire_decode(capi.NIW, body, [])


def test_oracle_niw_scorer_d128(oracle):
    """the oracle's fp32 NIW scorer agrees with float64 at d = 128 (within the fp32 posterior's slack)"""
    d, G, n = 128, 3, 64
    w = niw_workload(7300, G, n, d, 1.0, 0.0)
    groups = niw_groups(w, oracle)
    got = oracle.niw_score_rows(w["mu"], w["kappa"], w["psi"], w["nu"], w["count"], w["sum_x"], w["sum_xxT"], w["values"],
                                np.zeros((n, G), np.float32)).astype(np.float64)
    X = w["values"].astype(np.float64)
    want = np.empty((n, G))
    for g, gr in enumerate(groups):
        Y = (X - gr["mu_p"]) @ gr["W"].T
        want[:, g] = gr["C"] + gr["coef"] * np.log1p((Y * Y).sum(1) / gr["dof"])
    assert np.abs(got - want).max() <= 2e-3 * (1 + np.abs(want).max())


# ======================================================================================================= GPU
@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = capi.Context(0)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _score(ctx, feats, cols, n, G, prior=None):
    sc = torch.full((n, G), 777.0, device="cuda")
    ctx.score_batch(feats, cols, n, None if prior is None else dev(prior), sc)
    torch.cuda.synchronize()
    return sc.cpu().numpy()


def _lse(s):
    m = np.max(s, axis=1, keepdims=True)
    return (m + np.log(np.exp(s - m).sum(1, keepdims=True)))[:, 0]


def _check_routes(ctx, oracle, w, n, what, groups=None):
    """score_batch against the derived bound (at DP >= 64 it counts 3 DP + 16 accumulated products and is wider than the
    FP32 route's bound on every cell, so it is the bound that applies); the
    sampler's draws against sample_from_scores on the materialised scores; logp against the scores' float64 logsumexp"""
    G = w["count"].size
    groups = groups or wide_groups(w, oracle)
    f = ctx.feature(capi.NIW).update_all(w)
    vals = w["values"][:n]
    col = dev(vals)
    got = _score(ctx, [f], [col], n, G)
    C, coef, a, delta, tol_C = wide_reference(w, groups, vals)
    check_step_aware(got, C, coef, a, delta, tol_C, what=what + " derived bound")
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    u = w["u"][:n]
    sc = torch.full((n, G), 777.0, device="cuda")
    assign = torch.full((n,), -5, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch([f], [col], n, dev(prior), dev(u), assign, sc)
    a2 = torch.full((n,), -7, device="cuda", dtype=torch.int32)
    ctx.sample_from_scores(sc, n, G, dev(u), a2)
    a3 = torch.full((n,), -9, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch([f], [col], n, dev(prior), dev(u), a3)
    torch.cuda.synchronize()
    s = sc.cpu().numpy()
    assert np.array_equal(s, got + prior[None, :].astype(np.float32)) or np.allclose(s, got + prior[None, :], rtol=0, atol=2.0 ** -20 * (1 + np.abs(got).max()))
    assert np.array_equal(assign.cpu().numpy(), a2.cpu().numpy()) and np.array_equal(a3.cpu().numpy(), a2.cpu().numpy())
    logp = torch.full((n,), 777.0, device="cuda")
    ctx.score_logp_batch([f], [col], n, dev(prior), logp)
    torch.cuda.synchronize()
    want = _lse(s.astype(np.float64))
    tol = 2.0 ** -21 * (1 + np.abs(s).max(1)) + (G + 8) * 2.0 ** -24
    assert np.all(np.abs(logp.cpu().numpy() - want) <= tol)
    return f, col, got, prior


WIDE_DIMS = (33, 64, 100, 128)
WIDE_STDS = (1e-3, 1.0, 1e3)
WIDE_OFFSETS = (0.0, 1e2, 1e3)


def wide_sweep():
    k = 0
    for d in WIDE_DIMS:
        for std in WIDE_STDS:
            for offset in WIDE_OFFSETS:
                # at 1e3 sigma the fp32 statistics of many groups are no longer SPD (spd_workload): 9 groups there
                yield d, std, offset, 9 if offset >= 1e3 else (70 if k % 4 else 256)
                k += 1


@pytest.mark.gpu
@pytest.mark.parametrize("d,std,offset,G", list(wide_sweep()))
def test_wide_conditioning(ctx, oracle, d, std, offset, G):
    n = 256
    w, groups = spd_workload(oracle, 8000 + 7 * d + int(np.log10(std) * 3) + int(offset) % 97 + G, G, n, d, std, offset)
    _check_routes(ctx, oracle, w, n, "wide d %d std %g offset %g G %d" % (d, std, offset, G), groups)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [127, 128, 129, 1000])
def test_wide_tile_edges(ctx, oracle, n):
    """row counts around the 128-row tile (and the three-tile chunk at DP = 64), with a zero row"""
    for d in (64, 100):
        w = niw_workload(8500 + n + d, 70, n, d, 1.0, 0.0)
        w["values"][n // 2] = 0.0
        _check_routes(ctx, oracle, w, n, "wide tile edges d %d n %d" % (d, n))


@pytest.mark.gpu
def test_wide_mixed_tiles(ctx, oracle):
    """one tile holds a row x1e4 and a row x1e6 from the centre: its rows keep the derived bound"""
    d, G, n = 100, 9, 384
    w = niw_workload(8600, G, n, d, 1.0, 1e2)
    v = w["values"].copy()
    mu = w["mu"].astype(np.float32)
    v[5] = mu + (v[5] - mu) * 1e4
    v[70] = mu + (v[70] - mu) * 1e6
    w["values"] = v
    _check_routes(ctx, oracle, w, n, "wide mixed tiles")


@pytest.mark.gpu
def test_wide_mixed_list_and_host_entries(ctx, oracle):
    """niw d = 100 with nich and bb in one list: score_batch is the sum of the parts, sampling and logp follow the
    materialised scores; the host entries are bit-equal to the device ones"""
    G, n = 40, 700
    w = niw_workload(8700, G, n, 100, 1.0, 0.0)
    wn, wb = synth.nich(8701, G, n), synth.bb(8702, G, n)
    wn["sizes"] = wb["sizes"] = w["sizes"]
    fs = [ctx.feature(capi.NIW).update_all(w), ctx.feature(capi.NICH).update_all(wn), ctx.feature(capi.BB).update_all(wb)]
    cols_h = [np.ascontiguousarray(x["values"], capi.COLUMN_DTYPE[m]) for x, m in ((w, capi.NIW), (wn, capi.NICH), (wb, capi.BB))]
    cols = [dev(c) for c in cols_h]
    both = _score(ctx, fs, cols, n, G).astype(np.float64)
    parts = sum(_score(ctx, [f], [c], n, G).astype(np.float64) for f, c in zip(fs, cols))
    assert np.all(np.abs(both - parts) <= 2.0 ** -22 * (np.abs(both) + np.abs(parts) + 1))
    prior = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, w["sizes"])
    sc = torch.empty((n, G), device="cuda")
    assign = torch.empty((n,), device="cuda", dtype=torch.int32)
    ctx.score_sample_batch(fs, cols, n, dev(prior), dev(w["u"]), assign, sc)
    a2 = torch.empty((n,), device="cuda", dtype=torch.int32)
    ctx.sample_from_scores(sc, n, G, dev(w["u"]), a2)
    logp = torch.empty((n,), device="cuda")
    ctx.score_logp_batch(fs, cols, n, dev(prior), logp)
    torch.cuda.synchronize()
    assert np.array_equal(assign.cpu().numpy(), a2.cpu().numpy())
    s = sc.cpu().numpy().astype(np.float64)
    assert np.all(np.abs(logp.cpu().numpy() - _lse(s)) <= 2.0 ** -21 * (1 + np.abs(s).max(1)) + (G + 8) * 2.0 ** -24)
    ah, sh = ctx.score_sample_batch_host(fs, cols_h, prior, w["u"], want_scores=True)
    assert np.array_equal(ah, assign.cpu().numpy()) and np.array_equal(sh, sc.cpu().numpy())
    lh = ctx.score_logp_batch_host(fs, cols_h, prior)
    assert np.array_equal(lh, logp.cpu().numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 128])
def test_wide_add_remove_rows(ctx, oracle, d):
    """add_rows_batch / remove_rows_batch against the reference's sequential add_value / remove_value, an emptied group and
    negative ids; scoring after the update sees the new records"""
    G, n = 7, 3000
    w = synth.niw(8800 + d, G, n, d=d)
    w["count"][3], w["sum_x"][3], w["sum_xxT"][3] = 0, 0.0, 0.0  # group 3 holds only this batch's rows
    rng = np.random.default_rng(d)
    assign = rng.integers(0, G, n).astype(np.int32)
    assign[::13] = -1
    f = ctx.feature(capi.NIW).update_all(w)
    ctx.add_rows_batch([f], [dev(w["values"])], dev(assign), n)
    count, sx, sxx = stats_of(f, G, d)
    ec, esx, esxx = expected_after(oracle, w, w["values"], assign, +1)
    assert np.array_equal(count, ec)
    s = np.array([1.0 + np.abs(w["values"][assign == g]).max() ** 2 * (ec[g] + 1) for g in range(G)])
    assert np.all(np.abs(sxx - esxx).reshape(G, -1).max(1) <= (ec + 8.0) * 6e-8 * s)
    assert np.all(np.abs(sx - esx).max(1) <= (ec + 8.0) * 6e-8 * s)
    twin = ctx.feature(capi.NIW).update_all(dict(w, count=count, sum_x=sx.copy(), sum_xxT=sxx.copy()))
    m = 256
    vals = dev(w["values"][:m])
    assert np.array_equal(_score(ctx, [f], [vals], m, G), _score(ctx, [twin], [vals], m, G))
    # remove every row of group 3 and some of the others: group 3 comes back to exact zeros
    g3 = assign == 3
    rem = np.where(g3 | (rng.random(n) < 0.3), assign, -1).astype(np.int32)
    ctx.remove_rows_batch([f], [dev(w["values"])], dev(rem), n)
    count2, sx2, sxx2 = stats_of(f, G, d)
    ec2, _, _ = expected_after(oracle, dict(w, count=count, sum_x=sx.copy(), sum_xxT=sxx.copy()), w["values"], rem, -1)
    assert np.array_equal(count2, ec2)
    assert count2[3] == 0 and not sx2[3].any() and not sxx2[3].any()


@pytest.mark.gpu
def test_wide_row_shard_exchange(ctx):
    d, G, n = 128, 5, 2001
    w = synth.niw(8900, G, n, d=d)
    assign = np.random.default_rng(3).integers(0, G, n).astype(np.int32)
    single = ctx.feature(capi.NIW).update_all(w)
    ctx.add_rows_batch([single], [dev(w["values"])], dev(assign), n)
    shard = ctx.feature(capi.NIW).update_all(w)
    nd = ctx.rows_xchg_doubles([shard])
    assert nd == G * (1 + d + d * d)
    total = torch.zeros(nd, dtype=torch.float64, device="cuda")
    for lo, hi in ((0, n // 3), (n // 3, n)):
        x = torch.full((nd,), 123.0, dtype=torch.float64, device="cuda")
        ctx.rows_accumulate([shard], [dev(w["values"][lo:hi])], dev(assign[lo:hi]), hi - lo, x)
        total += x
    ctx.rows_merge([shard], total, +1)
    nb = 4 * G * (1 + d + d * d)
    assert np.array_equal(shard.download_stats(nb), single.download_stats(nb))
    ctx.rows_merge([shard], total, -1)
    orig = ctx.feature(capi.NIW).update_all(w)
    got, want = shard.download_stats(nb), orig.download_stats(nb)
    assert np.array_equal(got[:4 * G], want[:4 * G])


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 128])
def test_wide_score_data(ctx, oracle, d):
    """score_data_grid against the oracle, with grid points whose psi scale puts det outside the float range"""
    G = 6
    w = synth.niw(9000 + d, G, 400, d=d)
    f = ctx.feature(capi.NIW).update_all(w)
    shareds = []
    for scale in (1.0, 1e-2, 1e2):
        shareds.append(np.concatenate([[w["kappa"], w["nu"]], w["mu"], (w["psi"] * scale).ravel()]).astype(np.float32))
    got = f.score_data_grid(np.stack(shareds))
    for i, scale in enumerate((1.0, 1e-2, 1e2)):
        want = oracle.niw_score_data(w["mu"], w["kappa"], w["psi"] * np.float32(scale), w["nu"], w["count"], w["sum_x"], w["sum_xxT"])
        assert abs(float(got[i]) - float(want)) <= 2e-4 * (1 + abs(float(want))), (scale, got[i], want)


def _draws(ctx, f, G, d, reps, seed=1, row0=0):
    assign = np.repeat(np.arange(G, dtype=np.int32), reps)
    out = torch.empty((assign.size, d), device="cuda")
    ctx.sample_values_batch([f], dev(assign), assign.size, [out], seed=seed, row0=row0)
    torch.cuda.synchronize()
    return out.cpu().numpy().reshape(G, reps, d)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 128])
def test_wide_sample_values(ctx, d):
    from scipy import stats
    from test_gpu_sample_values import P_FLOOR, _niw_ps
    rng = np.random.default_rng(200 + d)
    mu = rng.normal(size=d).astype(np.float32)
    A = rng.normal(size=(d, d))
    psi = (A @ A.T / d + np.eye(d)).astype(np.float32)
    kappa, nu = 1.5, d + 6.0
    x = rng.normal(size=(300, d)) * 2 + 1
    count = np.array([0, 300], np.int32)
    sum_x = np.stack([np.zeros(d), x.sum(0)]).astype(np.float32)
    sum_xxT = np.stack([np.zeros((d, d)), x.T @ x]).astype(np.float32)
    w = dict(model="niw", mu=mu, kappa=kappa, psi=psi, nu=nu, count=count, sum_x=sum_x, sum_xxT=sum_xxT)
    f = ctx.feature(capi.NIW).update_all(w)
    reps = 20000
    xs = _draws(ctx, f, 2, d, reps)
    prng = np.random.default_rng(5)
    for g in range(2):
        n = float(count[g])
        sx, sxx = sum_x[g].astype(np.float64), sum_xxT[g].astype(np.float64)
        xbar = sx / n if n else np.zeros(d)
        diff = xbar - mu
        C = sxx - np.outer(sx, xbar) - np.outer(xbar, sx) + n * np.outer(xbar, xbar)
        pk, pn = kappa + n, nu + n
        ppsi = psi.astype(np.float64) + C + kappa * n / (kappa + n) * np.outer(diff, diff)
        dof = pn - d + 1
        dist = dict(df=dof, loc=(kappa * mu + n * xbar) / pk, shape=ppsi * (pk + 1) / (pk * dof))
        ps, z = _niw_ps(xs[g], dist, prng)
        assert min(ps) > P_FLOOR, (g, ps)
        assert z < stats.norm.isf(P_FLOOR / (2 * d)), (g, z)
    # row shards: rows [100, 200) drawn with row0 = 100 equal the same rows of the whole batch
    assign = np.repeat(np.arange(2, dtype=np.int32), 150)
    full = torch.empty((300, d), device="cuda")
    ctx.sample_values_batch([f], dev(assign), 300, [full], seed=9)
    part = torch.empty((100, d), device="cuda")
    ctx.sample_values_batch([f], dev(assign[100:200]), 100, [part], seed=9, row0=100)
    torch.cuda.synchronize()
    assert np.array_equal(full.cpu().numpy()[100:200], part.cpu().numpy())
    # distinct coordinates draw from distinct blocks: the whitened draws of the empty group have no repeated or
    # correlated coordinates (a reused block would repeat a standard normal exactly)
    L = np.linalg.cholesky(psi.astype(np.float64) * (kappa + 1) / (kappa * (nu - d + 1)))
    z = np.linalg.solve(L, (xs[0] - mu).T).T
    zr = np.round(z[:2000], 6)
    for i in range(d):
        for j in range(i + 1, d):
            assert not np.array_equal(zr[:, i], zr[:, j])
    cc = np.corrcoef(z[:5000].T)
    assert np.abs(cc - np.eye(d)).max() < 0.08


@pytest.mark.gpu
def test_wide_lifecycle(ctx, oracle):
    """a seeded add / update / remove-group and add / remove-rows script at d = 100: download_stats follows a host mirror,
    and a twin built by update_all from the mirror is bit-equal in scores and draws"""
    d, G = 100, 6
    w = synth.niw(9100, G, 600, d=d)
    rng = np.random.default_rng(91)
    f = ctx.feature(capi.NIW).update_all(w)
    count, sx, sxx = w["count"].astype(np.int32).copy(), w["sum_x"].copy(), w["sum_xxT"].copy()
    for step in range(6):
        op = step % 3
        if op == 0:
            f.add_group()
            count, sx, sxx = np.append(count, 0).astype(np.int32), np.vstack([sx, np.zeros((1, d), np.float32)]), np.concatenate([sxx, np.zeros((1, d, d), np.float32)])
        elif op == 1:
            g = int(rng.integers(0, count.size))
            x = rng.normal(size=(40, d))
            c, a_, b_ = np.int32(40), x.sum(0).astype(np.float32), (x.T @ x).astype(np.float32)
            f.update_group(g, np.concatenate([np.array([c], np.int32).view(np.float32), a_, b_.ravel()]))
            count[g], sx[g], sxx[g] = c, a_, b_
        else:
            g = int(rng.integers(0, count.size))
            f.remove_group(g)
            last = count.size - 1
            count[g], sx[g], sxx[g] = count[last], sx[last], sxx[last]
            count, sx, sxx = count[:last], sx[:last], sxx[:last]
        n = 300
        vals = rng.normal(size=(n, d)).astype(np.float32)
        Gc = count.size
        assign = rng.integers(-1, Gc, n).astype(np.int32)
        ctx.add_rows_batch([f], [dev(vals)], dev(assign), n)
        count, sx, sxx = expected_after(oracle, dict(mu=w["mu"], count=count, sum_x=sx, sum_xxT=sxx), vals, assign, +1)
        gc, gsx, gsxx = stats_of(f, Gc, d)
        assert np.array_equal(gc, count)
        np.testing.assert_allclose(gsx, sx, rtol=0, atol=1e-3 * (1 + np.abs(sx).max()))
        np.testing.assert_allclose(gsxx, sxx, rtol=0, atol=1e-3 * (1 + np.abs(sxx).max()))
        count, sx, sxx = gc.copy(), gsx.copy(), gsxx.copy()
    twin = ctx.feature(capi.NIW).update_all(dict(w, count=count, sum_x=sx, sum_xxT=sxx))
    m = 300
    vals = dev(rng.normal(size=(m, d)).astype(np.float32))
    assert np.array_equal(_score(ctx, [f], [vals], m, count.size), _score(ctx, [twin], [vals], m, count.size))
    assert np.array_equal(_draws(ctx, f, count.size, d, 50, seed=4), _draws(ctx, twin, count.size, d, 50, seed=4))


@pytest.mark.gpu
def test_wide_models_mirror(ctx):
    """models.py's niw namespace at d = 64: Mixture.score_value is the device score of the same statistics"""
    from distributions_b200 import models
    d = 64
    rng = np.random.default_rng(64)
    shared = models.niw.Shared(dim=d)
    shared.nu = np.float32(d + 2)
    mix = models.niw.Mixture(ctx)
    mix.init(shared)
    for _ in range(4):
        mix.add_group(shared)
    for i in range(200):
        mix.add_value(shared, i % 4, rng.normal(size=d).astype(np.float32))
    value = rng.normal(size=d).astype(np.float32)
    got = np.zeros(4, np.float32)
    mix.score_value(shared, value, got)
    w = dict(model="niw", mu=shared.mu, kappa=shared.kappa, psi=shared.psi, nu=shared.nu,
             count=np.array([g.count for g in mix.groups], np.int32), sum_x=np.array([g.sum_x for g in mix.groups], np.float32),
             sum_xxT=np.array([g.sum_xxT for g in mix.groups], np.float32))
    f = ctx.feature(capi.NIW).update_all(w)
    want = _score(ctx, [f], [dev(value[None, :])], 1, 4)[0]
    assert np.array_equal(got, want)


@pytest.mark.gpu
def test_wide_errors(ctx):
    d = 129
    w = dict(model="niw", mu=np.zeros(d, np.float32), kappa=1.0, psi=np.eye(d, dtype=np.float32), nu=d + 2.0,
             count=np.zeros(1, np.int32), sum_x=np.zeros((1, d), np.float32), sum_xxT=np.zeros((1, d, d), np.float32))
    with pytest.raises(capi.DistB200Error, match="status %d" % DIST_B200_ERR_UNSUPPORTED):
        ctx.feature(capi.NIW).update_all(w)
