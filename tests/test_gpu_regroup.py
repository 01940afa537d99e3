"""dist_b200_regroup_batch: group births and deaths in one batch, and the blocked Gibbs sweep built on it.

Every regroup is checked against the numpy reference of tests/regroup_ref.py (remap, compacted counts, new G, the
relabelled assignments, the compacted statistics, exactly), and every regrouped feature against a twin loaded by
update_all from the compacted statistics: caches, scores, fused samples and posterior-predictive draws bit for bit."""
import numpy as np
import pytest

import regroup_ref as ref
from distributions_b200 import capi, gibbs, models, synth

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ARRAYS = {"nich": ("count", "mean", "ctv"), "gp": ("count", "sum"), "bnb": ("count", "sum"), "bb": ("heads", "tails"),
          "dd": ("counts",), "dpd": ("counts",), "niw": ("count", "sum_x", "sum_xxT")}
CACHE_ROWS = {"nich": lambda w: 4, "gp": lambda w: 3, "bnb": lambda w: 3, "bb": lambda w: 2,
              "dd": lambda w: w["alphas"].size, "dpd": lambda w: w["keys"].size + 1}
CASES = [("nich", {}), ("gp", {}), ("bnb", {}), ("bb", {}), ("dd", dict(dim=16)), ("dpd", dict(V=40)), ("dpd", dict(V=4096)),
         ("niw", dict(d=3)), ("niw", dict(d=32)), ("niw", dict(d=96))]
CASE_IDS = [n + "".join("_%s%d" % kv for kv in k.items()) for n, k in CASES]


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = capi.Context(0)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def workload(name, kw, G, seed=41, log_prod=True):
    """synth statistics at G groups; gp's Group::log_prod is dropped (left invalid) unless log_prod"""
    w = getattr(synth, name)(seed, G, 8, **kw)
    if name == "gp" and not log_prod:
        w["log_prod"] = None
    return w


def elems(name, w):
    if name in ("dd", "dpd"):
        return (w["counts"].shape[1],)
    if name == "niw":
        d = w["mu"].size
        return (1, d, d * d)
    return (1,) * len(ARRAYS[name])


def download(name, w, f, G):
    """download_stats -> one [G][e] uint32 array per statistics array"""
    words = np.frombuffer(f.download_stats(4 * G * sum(elems(name, w))).tobytes(), dtype=np.uint32)
    out, off = [], 0
    for e in elems(name, w):
        out.append(words[off:off + G * e].reshape(G, e).copy())
        off += G * e
    assert off == words.size
    return out


def as_workload(name, w, stats, log_prod=None):
    """update_all arguments carrying the given statistics ([G][e] uint32 arrays)"""
    t = dict(w)
    for key, a in zip(ARRAYS[name], stats):
        dtype = np.asarray(w[key]).dtype
        t[key] = a.view(dtype).reshape((a.shape[0],) + np.asarray(w[key]).shape[1:])
    if name == "gp":
        t["log_prod"] = log_prod
    return t


def column(name, w, rng, n):
    if name == "nich":
        return (3 * rng.standard_normal(n)).astype(np.float32)
    if name in ("gp", "bnb"):
        return rng.poisson(5.0, n).astype(np.uint32)
    if name == "bb":
        return (rng.random(n) < 0.3).astype(np.uint8)
    if name == "dd":
        return rng.integers(0, w["counts"].shape[1], n).astype(np.int32)
    if name == "dpd":
        return rng.integers(0, w["counts"].shape[1], n).astype(np.uint32)
    return (3 * rng.standard_normal((n, w["mu"].size))).astype(np.float32)


def observe(ctx, name, w, f, G, seed):
    """what a user of the feature sees: caches, scores, fused samples and posterior-predictive draws"""
    rng = np.random.default_rng(seed)
    out = {}
    if name in CACHE_ROWS:
        out["caches"] = f.download_caches(CACHE_ROWS[name](w))
    n = 257
    prior = dev(rng.standard_normal(G).astype(np.float32))
    col = dev(column(name, w, rng, n))
    scores = torch.empty((n, G), device="cuda", dtype=torch.float32)
    ctx.score_batch([f], [col], n, prior, scores)
    assign = torch.empty(n, device="cuda", dtype=torch.int32)
    ctx.score_sample_batch([f], [col], n, prior, dev(rng.random(n, dtype=np.float32)), assign)
    n_draw = 513
    shape = (n_draw, w["mu"].size) if name == "niw" else (n_draw,)
    draws = torch.zeros(shape, device="cuda", dtype=torch.uint8 if name == "bb" else torch.int32)  # compared as bits
    ctx.sample_values_batch([f], dev(rng.integers(0, G, n_draw).astype(np.int32)), n_draw, [draws], seed=1234)
    torch.cuda.synchronize()
    out["scores"] = scores.cpu().numpy()
    out["assign"] = assign.cpu().numpy()
    out["draws"] = draws.cpu().numpy()
    return out


def assert_same(got, want, what):
    """bit patterns equal (NaN == NaN, -0 != +0)"""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got.view(np.uint8), want.view(np.uint8)):
        bad = np.argwhere(got != want)
        raise AssertionError("%s differs in %d of %d entries (first at %s)" % (what, bad.shape[0], got.size, bad[:3].tolist()))


def regroup_and_check(ctx, items, sizes, n_empty, assign=None, seed=0, twins=True):
    """items: [(name, w, feature)] all at G = sizes.size.  Regroups them, checks the clustering outputs and every
    feature's statistics against the numpy reference and (twins) against an update_all twin.  Returns G_new."""
    G = sizes.size
    want_rm, want_counts, want_G = ref.remap(sizes, n_empty)
    before = [download(name, w, f, G) for name, w, f in items]
    if assign is None:
        assign = np.random.default_rng(seed).integers(-2, G + 3, 4000).astype(np.int32)
    a_dev = dev(assign)
    rm_dev = torch.full((max(G, 1),), 77, device="cuda", dtype=torch.int32)
    co_dev = torch.full((G + n_empty,), 77, device="cuda", dtype=torch.int32)
    G_new = ctx.regroup_batch([f for _, _, f in items], dev(sizes.astype(np.int32)), G, n_empty, a_dev, assign.size, co_dev, rm_dev)
    assert G_new == want_G
    assert np.array_equal(rm_dev.cpu().numpy()[:G], want_rm)
    assert np.array_equal(co_dev.cpu().numpy()[:G_new], want_counts)
    assert np.array_equal(a_dev.cpu().numpy(), ref.relabel(assign, want_rm))
    for (name, w, f), old in zip(items, before):
        assert f.groups == G_new
        got = download(name, w, f, G_new)
        want = [ref.compact(a, sizes, n_empty) for a in old]
        for k, (x, y) in enumerate(zip(got, want)):
            assert np.array_equal(x, y), "%s: statistics array %d differs from the compaction" % (name, k)
        if twins:
            lp = None
            if name == "gp" and w.get("log_prod") is not None:
                lp = ref.compact(np.asarray(w["log_prod"], np.float32), sizes, n_empty)
            twin = ctx.feature(f.model).update_all(as_workload(name, w, want, lp))
            obs_t, obs_f = observe(ctx, name, w, twin, G_new, seed + 1), observe(ctx, name, w, f, G_new, seed + 1)
            for key in obs_t:
                assert_same(obs_f[key], obs_t[key], "%s G %d -> %d: %s" % (name, G, G_new, key))
            if lp is not None:
                shared = np.asarray(w["shared"], np.float32)
                assert_same(f.score_data_grid(shared), twin.score_data_grid(shared), "gp score_data_grid")
            twin.close()
    return G_new


def random_sizes(rng, G, zero_frac=0.3):
    sizes = rng.integers(1, 60, G).astype(np.int32)
    sizes[rng.random(G) < zero_frac] = 0
    return sizes


@pytest.mark.parametrize("n_empty", [1, 3])
@pytest.mark.parametrize("name,kw", CASES, ids=CASE_IDS)
def test_parity_per_model(ctx, name, kw, n_empty):
    rng = np.random.default_rng(CASES.index((name, kw)) * 10 + n_empty)
    G = 40 if kw.get("d", 0) > 32 else 150
    w = workload(name, kw, G)
    f = ctx.feature(getattr(capi, name.upper())).update_all(w)
    regroup_and_check(ctx, [(name, w, f)], random_sizes(rng, G), n_empty, seed=n_empty)
    f.close()


@pytest.mark.parametrize("case", ["no_deaths", "all_empty", "G1_live", "G1_dead"])
def test_edges(ctx, case):
    rng = np.random.default_rng(7)
    G = {"no_deaths": 90, "all_empty": 90, "G1_live": 1, "G1_dead": 1}[case]
    sizes = {"no_deaths": rng.integers(1, 9, G), "all_empty": np.zeros(G), "G1_live": np.array([5]),
             "G1_dead": np.array([0])}[case].astype(np.int32)
    items = []
    for name, kw in [("nich", {}), ("gp", {}), ("dd", dict(dim=16)), ("dpd", dict(V=40)), ("niw", dict(d=3)), ("niw", dict(d=32))]:
        w = workload(name, kw, G, seed=5, log_prod=False)
        items.append((name, w, ctx.feature(getattr(capi, name.upper())).update_all(w)))
    for n_empty in (1, 3):
        G_new = regroup_and_check(ctx, items, sizes, n_empty, seed=11)
        assert G_new == int((sizes > 0).sum()) + n_empty
        if case == "no_deaths":  # identity plus appended empties
            break
        sizes = np.concatenate([sizes[sizes > 0], np.zeros(n_empty, np.int32)])
    for _, _, f in items:
        f.close()


def test_clustering_only(ctx):
    rng = np.random.default_rng(3)
    G = 2500
    sizes = random_sizes(rng, G)
    assign = rng.integers(-1, G + 1, 100_000).astype(np.int32)
    rm, counts, G_want = ref.remap(sizes, 2)
    a_dev, co = dev(assign), torch.zeros(G + 2, device="cuda", dtype=torch.int32)
    assert ctx.regroup_batch([], dev(sizes), G, 2, a_dev, assign.size, co) == G_want
    assert np.array_equal(a_dev.cpu().numpy(), ref.relabel(assign, rm))
    assert np.array_equal(co.cpu().numpy()[:G_want], counts)


def test_growth_then_shrink(ctx):
    """127 live + 400 fresh groups cross the pooled caches' 128-group steps and the dpd / niw growth; then 600 -> 5"""
    rng = np.random.default_rng(9)
    G = 140
    items = []
    for name, kw in [("nich", {}), ("gp", {}), ("bb", {}), ("dd", dict(dim=16)), ("dpd", dict(V=40)), ("niw", dict(d=3)),
                     ("niw", dict(d=96))]:
        w = workload(name, kw, G, seed=6, log_prod=False)
        items.append((name, w, ctx.feature(getattr(capi, name.upper())).update_all(w)))
    sizes = np.zeros(G, np.int32)
    sizes[rng.choice(G, 127, replace=False)] = rng.integers(1, 30, 127)
    G_new = regroup_and_check(ctx, items, sizes, 400, seed=1)
    assert G_new == 527
    sizes = np.zeros(G_new, np.int32)  # 527 -> 600 -> 5
    sizes[:127] = 1
    G_new = regroup_and_check(ctx, items, sizes, 600 - 127, seed=2, twins=False)
    assert G_new == 600
    sizes = np.zeros(600, np.int32)
    sizes[rng.choice(600, 4, replace=False)] = 3
    assert regroup_and_check(ctx, items, sizes, 1, seed=3) == 5
    for _, _, f in items:
        f.close()


def test_mixed_list_crosses_launch_batch(ctx):
    rng = np.random.default_rng(4)
    G = 40
    items = []
    for i in range(135):
        name = ("nich", "gp", "bb", "bnb")[i % 4]
        w = workload(name, {}, G, seed=100 + i, log_prod=False)
        items.append((name, w, ctx.feature(getattr(capi, name.upper())).update_all(w)))
    for name, kw in [("dd", dict(dim=16)), ("dpd", dict(V=40)), ("niw", dict(d=3)), ("niw", dict(d=32))]:
        w = workload(name, kw, G, seed=7)
        items.append((name, w, ctx.feature(getattr(capi, name.upper())).update_all(w)))
    regroup_and_check(ctx, items, random_sizes(rng, G), 3, seed=4)
    for _, _, f in items:
        f.close()


def test_errors_leave_state_unchanged(ctx):
    G = 30
    wa, wb = workload("nich", {}, G), workload("nich", {}, G + 1)
    fa, fb = ctx.feature(capi.NICH).update_all(wa), ctx.feature(capi.NICH).update_all(wb)
    sizes = dev(np.arange(G + 1, dtype=np.int32))
    before = download("nich", wa, fa, G)
    L, g_out = ctx.L, capi.c_i(0)
    fl = (capi.c_p * 2)(fa.h, fb.h)
    assert L.dist_b200_regroup_batch(ctx.h, fl, 2, sizes.data_ptr(), G, 1, None, 0, None, None, capi.ctypes.byref(g_out), None) == 4
    fl1 = (capi.c_p * 1)(fa.h)
    assert L.dist_b200_regroup_batch(ctx.h, fl1, 1, sizes.data_ptr(), G, 0, None, 0, None, None, capi.ctypes.byref(g_out), None) == 1
    assert L.dist_b200_regroup_batch(ctx.h, fl1, 1, sizes.data_ptr(), G, 1, None, 0, None, None, None, None) == 1
    assert L.dist_b200_regroup_batch(ctx.h, fl1, 1, None, G, 1, None, 0, None, None, capi.ctypes.byref(g_out), None) == 1
    fresh = ctx.feature(capi.NICH)
    fl2 = (capi.c_p * 1)(fresh.h)
    assert L.dist_b200_regroup_batch(ctx.h, fl2, 1, sizes.data_ptr(), G, 1, None, 0, None, None, capi.ctypes.byref(g_out), None) == 4
    assert fa.groups == G and fb.groups == G + 1
    for x, y in zip(download("nich", wa, fa, G), before):
        assert np.array_equal(x, y)
    for f in (fa, fb, fresh):
        f.close()


def test_gp_log_prod(ctx):
    rng = np.random.default_rng(12)
    G = 60
    w = workload("gp", {}, G)
    f = ctx.feature(capi.GP).update_all(w)  # synth's gp carries log_prod: valid
    regroup_and_check(ctx, [("gp", w, f)], random_sizes(rng, G), 2, seed=5)  # compares score_data_grid with the twin
    w2 = dict(w, log_prod=None)
    f2 = ctx.feature(capi.GP).update_all(w2)
    ctx.regroup_batch([f2], dev(random_sizes(rng, G)), G, 1)
    with pytest.raises(capi.DistB200Error, match="status 4"):
        f2.score_data_grid(np.asarray(w["shared"], np.float32))
    f.close()
    f2.close()


def test_row_shards_on_one_device(ctx):
    """two replicas with half the rows each and the global counts end bit-identical to one replica with all rows"""
    rng = np.random.default_rng(21)
    G, N = 120, 6000
    specs = [("nich", {}), ("dd", dict(dim=16)), ("dpd", dict(V=40)), ("niw", dict(d=3))]
    reps = []
    for _ in range(3):
        reps.append([(name, workload(name, kw, G, seed=8), None) for name, kw in specs])
        reps[-1] = [(n, w, ctx.feature(getattr(capi, n.upper())).update_all(w)) for n, w, _ in reps[-1]]
    assign = rng.integers(0, G, N).astype(np.int32)
    assign[np.isin(assign, rng.choice(G, 40, replace=False))] = -1  # 40 groups lose all their rows
    sizes = np.bincount(assign[assign >= 0], minlength=G).astype(np.int32)
    halves = [assign[:N // 2].copy(), assign[N // 2:].copy()]
    outs = []
    for rep, rows in zip(reps, halves + [assign.copy()]):
        a = dev(rows)
        G_new = ctx.regroup_batch([f for _, _, f in rep], dev(sizes), G, 2, a, rows.size)
        outs.append((G_new, a.cpu().numpy(), [download(n, w, f, G_new) for n, w, f in rep]))
    assert outs[0][0] == outs[1][0] == outs[2][0]
    assert np.array_equal(np.concatenate([outs[0][1], outs[1][1]]), outs[2][1])
    for k in range(len(specs)):
        for x, y, z in zip(outs[0][2][k], outs[1][2][k], outs[2][2][k]):
            assert np.array_equal(x, z) and np.array_equal(y, z)
    for rep in reps:
        for _, _, f in rep:
            f.close()


# ---- the blocked Gibbs sweep ------------------------------------------------------------------------------------------
def host_stats(name, col, assign, G, obs, dim=None):
    """sufficient statistics recomputed on the host from (column, observed mask, assignments)"""
    ok = (assign >= 0) if obs is None else (assign >= 0) & obs
    a, x = assign[ok], col[ok]
    if name == "nich":
        cnt = np.bincount(a, minlength=G)
        s = np.bincount(a, weights=x.astype(np.float64), minlength=G)
        mean = np.divide(s, cnt, out=np.zeros(G), where=cnt > 0)
        ctv = np.bincount(a, weights=(x - mean[a]) ** 2, minlength=G)
        return cnt, mean, ctv
    if name == "gp":
        return np.bincount(a, minlength=G), np.bincount(a, weights=x.astype(np.float64), minlength=G).astype(np.int64)
    if name == "bb":
        return np.bincount(a[x != 0], minlength=G), np.bincount(a[x == 0], minlength=G)
    out = np.zeros((G, dim), np.int64)
    np.add.at(out, (a, x), 1)
    return (out,)


@pytest.mark.parametrize("masked", [False, True])
def test_sweep_invariants(ctx, masked):
    rng = np.random.default_rng(31 + masked)
    N, G0, n_empty, dim = 4096, 6, 2, 8
    truth = rng.integers(0, 4, N)
    cols = {"nich": (truth * 4.0 + rng.standard_normal(N)).astype(np.float32),
            "gp": rng.poisson(1.0 + 3 * truth).astype(np.uint32),
            "bb": (rng.random(N) < 0.2 + 0.2 * truth).astype(np.uint8),
            "dd": ((truth * 2 + rng.integers(0, 2, N)) % dim).astype(np.int32)}
    names = list(cols)
    obs = {n: (rng.random(N) < 0.85) if masked else None for n in names}
    zero = {"nich": dict(shared=np.array([0, 1, 1, 1], np.float32), count=np.zeros(G0, np.int32), mean=np.zeros(G0, np.float32),
                         ctv=np.zeros(G0, np.float32)),
            "gp": dict(shared=np.array([1, 1], np.float32), count=np.zeros(G0, np.uint32), sum=np.zeros(G0, np.uint32)),
            "bb": dict(shared=np.array([0.5, 2], np.float32), heads=np.zeros(G0, np.int32), tails=np.zeros(G0, np.int32)),
            "dd": dict(alphas=np.full(dim, 0.5, np.float32), counts=np.zeros((G0, dim), np.int32))}
    feats = [ctx.feature(getattr(capi, n.upper())).update_all(zero[n]) for n in names]
    cdev = [dev(cols[n]) for n in names]
    observed = [dev(capi.pack_observed(obs[n]).view(np.int32)) for n in names] if masked else None
    assign = dev(rng.integers(0, G0, N).astype(np.int32))
    ctx.add_rows_batch(feats, cdev, assign, N, observed=observed)
    kind = gibbs.BlockedGibbs(ctx, feats, cdev, assign, models.PitmanYor(1.0, 0.1), n_empty=n_empty, observed=observed)
    seen = []
    events = dict(live=G0, births=0, deaths=0)  # live groups after the previous block

    def check(k, r0, r1, K):
        G = k.G
        torch.cuda.synchronize()
        at_regroup = k.counts_out[:G].cpu().numpy()
        assert G == K + n_empty and np.all(at_regroup[:K] > 0) and np.all(at_regroup[K:] == 0)
        a = assign.cpu().numpy()
        assert a.min() >= 0 and a.max() < G
        ctx.count_assignments(assign, N, G, k.counts)
        assert np.array_equal(k.counts[:G].cpu().numpy(), np.bincount(a, minlength=G))
        live = int((np.bincount(a, minlength=G) > 0).sum())
        events["deaths"] += K < events["live"]  # a group the block emptied was dropped at the regroup
        events["births"] += live > K  # a fresh group received rows of the block
        events["live"] = live
        for name, f in zip(names, feats):
            w = zero[name]
            got = download(name, w, f, G)
            want = host_stats(name, cols[name], a, G, obs[name], dim)
            if name == "nich":
                assert np.array_equal(got[0].ravel().view(np.int32), want[0])
                np.testing.assert_allclose(got[1].ravel().view(np.float32), want[1], rtol=1e-5, atol=1e-5)
                np.testing.assert_allclose(got[2].ravel().view(np.float32), want[2], rtol=2e-4, atol=1e-3)
            else:
                for x, y in zip(got, want):
                    assert np.array_equal(x.reshape(y.shape).astype(np.int64), y), name
        seen.append(G)

    gen = torch.Generator(device="cuda").manual_seed(5)
    for _ in range(3):
        kind.sweep(8, gen, on_block=check)
    assert len(seen) == 24
    assert events["births"] > 0 and events["deaths"] > 0, events  # the number of groups really changed
    for f in feats:
        f.close()


# ---- host mirrors following a device regroup --------------------------------------------------------------------------
MIRRORS = ["nich", "gp", "bb", "dd", "niw"]


@pytest.mark.parametrize("name", MIRRORS)
def test_python_feature_mirror_follows_regroup(ctx, name):
    """models.<model>.Mixture.regroup re-reads its host Groups after regroup_batch moved its feature's groups"""
    model = models.MODELS[name]
    rng = np.random.default_rng(MIRRORS.index(name))
    shared = model.Shared()
    mixture = model.Mixture(ctx)
    G, n_empty = 9, 2
    for g in range(G):
        grp = model.Group()
        grp.init(shared)
        for _ in range(int(rng.integers(0, 6))):
            v = {"nich": lambda: float(np.float32(rng.normal(0, 3))), "gp": lambda: int(rng.poisson(6)),
                 "bb": lambda: bool(rng.random() < 0.4), "dd": lambda: int(rng.integers(0, 16)),
                 "niw": lambda: rng.normal(0, 2, 2).astype(np.float32)}[name]()
            grp.add_value(shared, v)
        mixture.append(grp)
    mixture.init(shared)
    before = [mixture._stats(shared, g) for g in mixture.groups]
    sizes = rng.integers(1, 5, G).astype(np.int32)
    sizes[[1, 4, 5]] = 0
    rm_dev = torch.zeros(G, device="cuda", dtype=torch.int32)
    G_new = ctx.regroup_batch([mixture.feature], dev(sizes), G, n_empty, remap_out=rm_dev)
    remap = rm_dev.cpu().numpy()
    assert G_new == G - 3 + n_empty and np.array_equal(remap, ref.remap(sizes, n_empty)[0])
    mixture.regroup(shared, remap, n_empty)
    fresh = model.Group()
    fresh.init(shared)
    want = [before[g] for g in np.flatnonzero(sizes > 0)] + [mixture._stats(shared, fresh)] * n_empty
    assert len(mixture.groups) == G_new
    for i, (g, w) in enumerate(zip(mixture.groups, want)):
        got = mixture._stats(shared, g)
        assert np.asarray(got).tobytes() == np.asarray(w).tobytes(), (name, i)


def test_cpp_feature_mirror_follows_regroup(tmp_path):
    """Mixture<NormalInverseChiSq>::regroup (include/distributions_b200/mixture.hpp) after a device regroup"""
    import subprocess
    from test_regroup_host import compile_regroup_api
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    exe = compile_regroup_api(str(tmp_path / "test_regroup_api"))
    out = subprocess.run([exe, "gpu"], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip() == "ok", out.stderr


def test_caller_buffers_written_within_their_sizes(ctx):
    """remap_out[G], counts_out[G + n_empty] and assign[n_rows] are written up to their documented sizes and no
    further: each sits in a larger buffer whose tail keeps a sentinel"""
    rng = np.random.default_rng(17)
    G, n_empty, N, pad = 300, 3, 1000, 64
    w = workload("nich", {}, G)
    f = ctx.feature(capi.NICH).update_all(w)
    sizes = random_sizes(rng, G)
    sentinel = 0x5A5A5A5A
    rm = torch.full((G + pad,), sentinel, device="cuda", dtype=torch.int32)
    co = torch.full((G + n_empty + pad,), sentinel, device="cuda", dtype=torch.int32)
    assign = np.full(N + pad, sentinel, np.int32)
    assign[:N] = rng.integers(-1, G, N)
    a_dev = dev(assign)
    G_new = ctx.regroup_batch([f], dev(sizes), G, n_empty, a_dev, N, counts_out=co, remap_out=rm)
    want_rm, want_co, want_G = ref.remap(sizes, n_empty)
    assert G_new == want_G
    rm_h, co_h, a_h = rm.cpu().numpy(), co.cpu().numpy(), a_dev.cpu().numpy()
    assert np.array_equal(rm_h[:G], want_rm) and np.all(rm_h[G:] == sentinel)
    assert np.array_equal(co_h[:G_new], want_co) and np.all(co_h[G + n_empty:] == sentinel)
    assert np.array_equal(a_h[:N], ref.relabel(assign[:N], want_rm)) and np.all(a_h[N:] == sentinel)
    f.close()


# ---- recovery --------------------------------------------------------------------------------------------------------
def adjusted_rand_index(a, b):
    """ARI of two labelings (Hubert and Arabie), from the contingency table"""
    _, ai = np.unique(a, return_inverse=True)
    _, bi = np.unique(b, return_inverse=True)
    table = np.zeros((ai.max() + 1, bi.max() + 1), np.int64)
    np.add.at(table, (ai, bi), 1)
    comb = lambda x: x * (x - 1) / 2.0  # noqa: E731
    index = comb(table).sum()
    rows, cols = comb(table.sum(1)).sum(), comb(table.sum(0)).sum()
    expected = rows * cols / comb(a.size)
    return (index - expected) / (0.5 * (rows + cols) - expected)


def test_recovery_from_one_group(ctx):
    """12 000 rows from 6 well-separated 1-D clusters (means -50 .. 50 in steps of 20, unit variance), all rows starting
    in ONE group, 40 sweeps of 8 blocks with one empty group per block: exactly 6 groups hold >= 1 % of the rows and the
    adjusted Rand index against the truth is >= 0.95.

    The Shared is the known-variance regime of the model the data come from: nu = 3e4 pins every group's variance near
    sigmasq = 1 (the clusters' true variance), and kappa = 1e-3 leaves the mean nearly free.  With a weak variance prior
    (nu ~ 1) no correct collapsed sampler leaves the one-group start: that group's predictive is broad enough to hold
    every row, and a row moves to the empty group only when alpha * p_empty(x) beats (n - 1) * p_group(x), which needs
    alpha of the order of n.  Pinning the variance makes a mixed group a poor fit, so births follow the data."""
    rng = np.random.default_rng(2026)
    N = 12_000
    means = np.array([-50.0, -30.0, -10.0, 10.0, 30.0, 50.0])
    truth = rng.integers(0, means.size, N)
    col = dev((means[truth] + rng.standard_normal(N)).astype(np.float32))
    f = ctx.feature(capi.NICH).update_all(dict(shared=np.array([0.0, 1e-3, 1.0, 3e4], np.float32), count=np.zeros(1, np.int32),
                                               mean=np.zeros(1, np.float32), ctv=np.zeros(1, np.float32)))
    assign = torch.zeros(N, device="cuda", dtype=torch.int32)
    ctx.add_rows_batch([f], [col], assign, N)
    kind = gibbs.BlockedGibbs(ctx, [f], [col], assign, models.PitmanYor(0.1, 0.0), n_empty=1)
    gen = torch.Generator(device="cuda").manual_seed(7)
    for _ in range(40):
        kind.sweep(8, gen)
    a = assign.cpu().numpy()
    sizes = np.bincount(a, minlength=kind.G)
    big = int((sizes >= 0.01 * N).sum())
    ari = adjusted_rand_index(truth, a)
    assert big == 6 and ari >= 0.95, (big, ari, sorted(sizes[sizes > 0].tolist()))
    f.close()
