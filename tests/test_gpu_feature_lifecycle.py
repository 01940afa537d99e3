"""One feature under churn, for every model: update_all at G = 5, then a seeded script of add_group, update_group,
remove_group (middle and last ids) and batched add / remove of rows that drives G past 300.  That crosses every
growth of the device-resident statistics and caches with groups present (the pooled caches start at 256 groups; dpd
and niw statistics grow many times on the way).

After every group operation download_stats must equal a host mirror of the statistics (append a zero group,
swap-with-last, set a record) exactly; after a batched rows operation the mirror is re-read from the device.  At
checkpoints a twin feature is built by update_all from the downloaded statistics, and the churned feature must give
the same download_caches, score_batch and sample_values_batch output as the twin, bit for bit."""
import numpy as np
import pytest

from distributions_b200 import capi, synth

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

N_OPS = 440
SCRIPT_SEED = 3  # reaches G = 332
CHECKPOINTS = (110, 220, 330, N_OPS)
# update_all argument names of each model's statistics arrays, in update_all (= download_stats) order
ARRAYS = {"nich": ("count", "mean", "ctv"), "gp": ("count", "sum"), "bnb": ("count", "sum"), "bb": ("heads", "tails"),
          "dd": ("counts",), "dpd": ("counts",), "niw": ("count", "sum_x", "sum_xxT")}
CACHE_ROWS = {"nich": lambda w: 4, "gp": lambda w: 3, "bnb": lambda w: 3, "bb": lambda w: 2,
              "dd": lambda w: w["alphas"].size, "dpd": lambda w: w["keys"].size + 1}
CASES = [("nich", {}), ("gp", {}), ("bnb", {}), ("bb", {}), ("dd", dict(dim=16)), ("dpd", dict(V=40)),
         ("niw", dict(d=3)), ("niw", dict(d=32))]


@pytest.fixture(scope="module")
def ctx():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = capi.Context(0)
    yield c
    c.close()


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def script(seed, G=5):
    """the operation sequence; it depends on the seed alone, so the group count it reaches is fixed"""
    rng = np.random.default_rng(seed)
    ops, pending = [], 0
    for _ in range(N_OPS):
        r = rng.random()
        if r < 0.78:
            ops.append(("add_group",))
            G += 1
        elif r < 0.86:
            ops.append(("update_group", int(rng.integers(G))))
        elif r < 0.93 and G > 1:
            ops.append(("remove_group", G - 1 if rng.random() < 0.3 else int(rng.integers(G - 1))))
            G -= 1
        elif r < 0.97 or pending == 0:
            ops.append(("add_rows",))
            pending += 1
        else:
            ops.append(("remove_rows",))
            pending -= 1
    return ops


def workload(name, kw):
    if name == "niw":
        return synth.niw(41, 5, 8, d=kw["d"])
    w = getattr(synth, name)(41, 5, 8, **kw)
    if name == "gp":
        w["log_prod"] = None
    return w


def elems(name, w):
    """4-byte elements per group of each statistics array"""
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


def as_workload(name, w, mirror):
    """update_all arguments carrying the mirrored statistics"""
    t = dict(w)
    for key, a in zip(ARRAYS[name], mirror):
        dtype = np.asarray(w[key]).dtype
        t[key] = a.view(dtype).reshape((a.shape[0],) + np.asarray(w[key]).shape[1:])
    return t


def random_record(name, w, rng):
    """one group's statistics (valid for the model) as the per-array slices, 4-byte words"""
    if name == "nich":
        n = int(rng.integers(0, 40))
        rec = [np.int32(n), np.float32(3 * rng.standard_normal()), np.float32(rng.gamma(2.0, 1.0) * n)]
    elif name in ("gp", "bnb"):
        n = int(rng.integers(0, 40))
        rec = [np.uint32(n), np.uint32(rng.integers(0, 8 * n + 1))]
    elif name == "bb":
        rec = [np.int32(rng.integers(0, 30)), np.int32(rng.integers(0, 30))]
    elif name in ("dd", "dpd"):
        rec = [rng.integers(0, 5, w["counts"].shape[1]).astype(np.int32)]
    else:
        d = w["mu"].size
        n = int(rng.integers(0, 20))
        x = (3 * rng.standard_normal(d) + rng.standard_normal((n, d))).astype(np.float32).astype(np.float64)
        rec = [np.int32(n), x.sum(0).astype(np.float32), (x.T @ x).astype(np.float32).ravel()]
    return [np.atleast_1d(np.asarray(r)).view(np.uint32) for r in rec]


def random_rows(name, w, rng, G):
    n = int(rng.integers(1, 160))
    assign = rng.integers(0, G, n).astype(np.int32)
    if name == "nich":
        vals = (3 * rng.standard_normal(n)).astype(np.float32)
    elif name in ("gp", "bnb"):
        vals = rng.poisson(5.0, n).astype(np.uint32)
    elif name == "bb":
        vals = (rng.random(n) < 0.3).astype(np.uint8)
    elif name in ("dd", "dpd"):
        vals = rng.integers(0, w["counts"].shape[1], n).astype(capi.COLUMN_DTYPE[capi.DD if name == "dd" else capi.DPD])
    else:
        vals = (3 * rng.standard_normal((n, w["mu"].size))).astype(np.float32)
    return vals, assign


def column(name, w, rng, n):
    vals, _ = random_rows(name, w, rng, 1)
    while vals.shape[0] < n:
        vals = np.concatenate([vals, random_rows(name, w, rng, 1)[0]])
    return vals[:n]


def observe(ctx, name, w, f, G, rng_seed):
    """what a user of the feature sees: its caches, its scores and its posterior-predictive draws"""
    rng = np.random.default_rng(rng_seed)
    out = {}
    if name in CACHE_ROWS:
        out["caches"] = f.download_caches(CACHE_ROWS[name](w))
    n = 257
    prior = dev(rng.standard_normal(G).astype(np.float32))
    scores = torch.empty((n, G), device="cuda", dtype=torch.float32)
    ctx.score_batch([f], [dev(column(name, w, rng, n))], n, prior, scores)
    n_draw = 513
    shape = (n_draw, w["mu"].size) if name == "niw" else (n_draw,)
    draws = torch.zeros(shape, device="cuda", dtype=torch.uint8 if name == "bb" else torch.int32)  # compared as bits
    ctx.sample_values_batch([f], dev(rng.integers(0, G, n_draw).astype(np.int32)), n_draw, [draws], seed=1234)
    torch.cuda.synchronize()
    out["scores"] = scores.cpu().numpy()
    out["draws"] = draws.cpu().numpy()
    return out


def assert_same(got, want, what):
    """bit patterns equal (NaN == NaN, -0 != +0)"""
    assert got.shape == want.shape, (what, got.shape, want.shape)
    if not np.array_equal(got.view(np.uint8), want.view(np.uint8)):
        a, b = got.astype(np.float64), want.astype(np.float64)
        bad = np.argwhere(got != want)
        raise AssertionError("%s differs in %d of %d entries, max |diff| %g, max rel %g (first at %s)"
                             % (what, bad.shape[0], got.size, float(np.nanmax(np.abs(a - b))),
                                float(np.nanmax(np.abs(a - b) / (1e-30 + np.abs(b)))), bad[:3].tolist()))


@pytest.mark.parametrize("name,kw", CASES, ids=[n + "".join("_%s%d" % kv for kv in k.items()) for n, k in CASES])
def test_lifecycle_matches_update_all(ctx, name, kw):
    seed = CASES.index((name, kw))
    model = getattr(capi, name.upper())
    w = workload(name, kw)
    f = ctx.feature(model).update_all(w)
    G = 5
    mirror = [a.copy() for a in download(name, w, f, G)]
    rng = np.random.default_rng(1000 + seed)
    pending = []  # rows added by add_rows_batch and still in their groups: [values, assign]
    peak = G
    for i, op in enumerate(script(SCRIPT_SEED), 1):
        kind = op[0]
        if kind == "add_group":
            f.add_group()
            mirror = [np.concatenate([a, np.zeros((1, a.shape[1]), np.uint32)]) for a in mirror]
            G += 1
        elif kind == "update_group":
            g = op[1]
            rec = random_record(name, w, rng)
            f.update_group(g, np.concatenate(rec))
            for a, r in zip(mirror, rec):
                a[g] = r
            for p in pending:  # the group's rows are replaced by the record
                keep = p[1] != g
                p[0], p[1] = p[0][keep], p[1][keep]
        elif kind == "remove_group":
            g, last = op[1], G - 1
            f.remove_group(g)
            for a in mirror:
                a[g] = a[last]
            mirror = [a[:last] for a in mirror]
            for p in pending:
                keep = p[1] != g
                p[0], p[1] = p[0][keep], p[1][keep]
                p[1][p[1] == last] = g
            G -= 1
        elif kind == "add_rows":
            vals, assign = random_rows(name, w, rng, G)
            ctx.add_rows_batch([f], [dev(vals)], dev(assign), assign.size)
            pending.append([vals, assign])
        else:
            vals, assign = pending.pop(0)
            if assign.size:
                ctx.remove_rows_batch([f], [dev(vals)], dev(assign), assign.size)
        assert f.groups == G
        got = download(name, w, f, G)
        if kind in ("add_rows", "remove_rows"):
            mirror = got
        else:
            for k, (a, b) in enumerate(zip(got, mirror)):
                assert np.array_equal(a, b), "op %d %s: statistics array %d differs from the mirror" % (i, op, k)
        peak = max(peak, G)
        if i in CHECKPOINTS:
            twin = ctx.feature(model).update_all(as_workload(name, w, mirror))
            assert all(np.array_equal(a, b) for a, b in zip(download(name, w, twin, G), mirror))
            want = observe(ctx, name, w, twin, G, i)
            got_obs = observe(ctx, name, w, f, G, i)
            for key in want:
                assert_same(got_obs[key], want[key], "op %d (G = %d): %s" % (i, G, key))
            twin.close()
    assert peak > 300
    f.close()
