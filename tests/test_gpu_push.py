"""The feature-shard push path (dist_b200_score_push_batch, peer_signal / peer_wait, sample_from_slots and the
sharding.PeerFeatureShards layout) on ONE GPU: K owners are simulated in one process, with every owner's slots in one
allocation and a guard band behind every slot.

Stated tolerances:
  slot rows   each row of owner o, slot j is shard j's partial score [prior] + sum_{f in shard j} score_f.  Reference:
              the per-feature oracle scores summed in float64.  Per feature test_gpu_parity's 3e-6 * (1 + |ref_f|) plus
              the model envelope (nich 1e-6 * |log_coeff|, gp 6e-7 * (1 + |score|), bnb 6e-7 * (1 + |score| + |lgamma(beta)|
              + |lgamma(beta + alpha)|) as in test_gpu_bnb, table models 0), plus 2^-23 of every
              running partial sum of the shard's terms (the fp32 additions, prior first, features in list order).
  bits        every slot row equals ctx.score_batch of the same shard on the same rows bit for bit (the push runs the
              same kernels with other store addresses) -- except a shard that is one GammaPoisson feature, which the
              push scores through the value table and score_batch directly: held to the float64 bound only.
  guards      every float the push must not write (guard bands, rows outside [row0, row0 + n_rows), slots of ranks
              without features) keeps the sentinel bits.
  sampler     sample_from_slots == sample_from_scores on the fp32 slot sum formed in slot order, index for index;
              against the oracle sampler on the float64 full scores every mismatch is a near-tie: within
              (2e-5 + 2 * the row's largest score bound) of the row total.
"""
import contextlib

import numpy as np
import pytest
from scipy.special import gammaln

import cases
from distributions_b200 import sharding, synth

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

SENTINEL = 0x7FC0DEAD  # a quiet NaN: an unwritten float never passes a tolerance check by accident
GUARD_ROWS = 32        # a warp tile is 32 rows: no store of one can reach past a 32-row guard band
EPS_TIE = 2e-5
MIX = ["nich", "gp", "bb", "dd16", "bnb", "gp_big", "dd40", "bb"]

OPT_ROW_TILE, OPT_SMALL_TILE, OPT_NICH_PACKED = 1, 5, 6


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


def column(w, values=None):
    from distributions_b200 import capi
    v = w["values"] if values is None else values
    return dev(v.astype(capi.COLUMN_DTYPE[model_id(w["model"])]))


def envelope(oracle, w):
    """[1][G] or [n][G]: the model envelopes of test_gpu_parity and, for bnb, of test_gpu_bnb (score[g], lgamma(beta) and
    lgamma(beta + alpha[g]) are each rounded at their own magnitude before they cancel)"""
    if w["model"] == "nich":
        return 1e-6 * np.abs(oracle.nich_caches(w["shared"], w["count"], w["mean"], w["ctv"])[1])[None, :]
    if w["model"] == "gp":
        return 6e-7 * (1.0 + np.abs(oracle.gp_caches(w["shared"], w["count"], w["sum"])[0]))[None, :]
    if w["model"] == "bnb":
        score, post_beta, alpha = oracle.bnb_caches(w["shared"], w["count"], w["sum"])
        beta = post_beta[None, :] + w["values"][:, None].astype(np.float64)
        return 6e-7 * (1 + np.abs(score)[None, :] + np.abs(gammaln(beta)) + np.abs(gammaln(beta + alpha[None, :])))
    return np.zeros((1, w["sizes"].size))


def workload(spec, G, n, seed):
    if spec == "nich":
        return synth.nich(seed, G, n)
    if spec == "gp":
        return synth.gp(seed, G, n)
    if spec == "gp_big":  # counts mostly above the 32-entry value table (kGpTableX): the direct fallback
        return synth.gp(seed, G, n, lam=40.0)
    if spec == "bnb":
        return synth.bnb(seed, G, n, r=3)
    if spec == "bb":
        return synth.bb(seed, G, n)
    if spec == "dd16":
        return synth.dd(seed, G, n, dim=16)
    if spec == "dd40":
        return synth.dd(seed, G, n, dim=40)
    raise ValueError(spec)


class Kind:
    """one feature list of G groups over n rows: device features and columns, the prior, per-feature oracle scores"""

    def __init__(self, ctx, oracle, specs, G, n, seed):
        self.G, self.n = G, n
        self.ws = [workload(s, G, n, seed + 7 * i) for i, s in enumerate(specs)]
        self.feats = [ctx.feature(model_id(w["model"])).update_all(w) for w in self.ws]
        self.cols = [column(w) for w in self.ws]
        self.prior_np = oracle.py_prior(synth.PY_ALPHA, synth.PY_D, self.ws[0]["sizes"])
        self.prior = dev(self.prior_np)
        self.refs = [cases.oracle_scores(oracle, [w]).astype(np.float64) for w in self.ws]
        self.envs = [envelope(oracle, w) for w in self.ws]

    def lone_gp(self, shard):
        return len(shard) == 1 and self.ws[shard[0]]["model"] == "gp"

    def partial_ref(self, shard, with_prior):
        """float64 partial score of a shard over the n rows and its tolerance"""
        s = np.zeros((self.n, self.G))
        if with_prior:
            s += self.prior_np.astype(np.float64)[None, :]
        tol = np.zeros_like(s)
        run = np.zeros_like(s)
        for f in shard:
            s = s + self.refs[f]
            tol += 3e-6 * (1 + np.abs(self.refs[f])) + self.envs[f]
            run += np.abs(s)
        return s, tol + 2.0 ** -23 * run


def shards(F, K):
    return [sharding.feature_shard(F, j, K) for j in range(K)]


class Slots:
    """K owners' slot areas in ONE allocation: owner o holds K slots [block][G], each followed by a guard band of at
    least GUARD_ROWS x G floats; slot strides are multiples of 64 floats, so every slot base is 256-byte aligned"""

    def __init__(self, K, block, G):
        self.K, self.block, self.G = K, block, G
        self.stride = ((block + GUARD_ROWS) * G + 63) // 64 * 64
        self.buf = torch.empty(K * K * self.stride, dtype=torch.int32, device="cuda")
        self.fill()

    def fill(self):
        self.buf.fill_(SENTINEL)

    @property
    def base(self):
        return self.buf.data_ptr()

    def owner_base(self, o):
        return self.base + 4 * o * self.K * self.stride

    def slot_ptrs(self, j):
        """rank j's slot in every owner's area"""
        return [self.owner_base(o) + 4 * j * self.stride for o in range(self.K)]

    def read(self):
        """int32 [K owners][K slots][stride]"""
        torch.cuda.synchronize()
        return self.buf.cpu().numpy().reshape(self.K, self.K, self.stride)

    def slot_rows(self, area, j):
        """slot j of every owner as [K * block][G] global rows (owner o holds rows [o * block, (o + 1) * block))"""
        return area[:, j, :self.block * self.G].reshape(self.K * self.block, self.G)


def push_all(ctx, kind, slots, parts, row0, n=None, cols=None):
    n = kind.n if n is None else n
    cols = kind.cols if cols is None else cols
    for j, shard in enumerate(parts):
        if shard:
            ctx.score_push_batch([kind.feats[f] for f in shard], [cols[f] for f in shard], n, row0,
                                 kind.prior if j == 0 else None, slots.slot_ptrs(j), slots.block)


def local_scores(ctx, kind, shard, with_prior, cols=None, n=None):
    """the same shard through ctx.score_batch (accumulate = 0): [n][G] float32 on the device"""
    n = kind.n if n is None else n
    cols = kind.cols if cols is None else cols
    out = torch.empty((n, kind.G), dtype=torch.float32, device="cuda")
    ctx.score_batch([kind.feats[f] for f in shard], [cols[f] for f in shard], n, kind.prior if with_prior else None, out)
    return out


def check_slots(ctx, kind, slots, parts, row0, label, gp_bits=None):
    """(a) every written row against float64, (b) bit-identity with score_batch, (c) sentinel everywhere else"""
    area = slots.read()
    n, G, K, block = kind.n, kind.G, slots.K, slots.block
    glob = np.arange(K * block)
    written = (glob >= row0) & (glob < row0 + n)
    assert np.all(area[:, :, block * G:] == SENTINEL), "%s: a guard band was written" % label
    for j, shard in enumerate(parts):
        rows = slots.slot_rows(area, j)
        if not shard:
            assert np.all(rows == SENTINEL), "%s: slot %d has no pusher but was written" % (label, j)
            continue
        assert np.all(rows[~written] == SENTINEL), "%s: slot %d: a row outside [row0, row0 + n) was written" % (label, j)
        got = rows[written]
        ref, tol = kind.partial_ref(shard, j == 0)
        err = np.abs(got.view(np.float32).astype(np.float64) - ref)
        bad = ~(err <= tol)
        assert not bad.any(), "%s: slot %d: %d of %d cells outside the float64 bound (first row %d, err %g, tol %g)" % (
            label, j, int(bad.sum()), bad.size, int(np.nonzero(bad)[0][0]), float(err[bad][0]), float(tol[bad][0]))
        want = local_scores(ctx, kind, shard, j == 0).cpu().numpy().view(np.int32)
        same = np.array_equal(got, want)
        if kind.lone_gp(shard):
            if gp_bits is not None:
                gp_bits.append(same)
        else:
            assert same, "%s: slot %d differs from score_batch in %d cells" % (label, j, int((got != want).sum()))


@contextlib.contextmanager
def options(ctx, opts):
    """dist_b200_option settings for the duration of a block, reset to the defaults in a finally"""
    try:
        for k, v in opts.items():
            ctx.set_option(k, v)
        yield
    finally:
        for k in opts:
            ctx.set_option(k, 0)


# (feature list, G, K, block_rows, row0, options).  n_rows = K * block - row0 - block // 3: the last block is partial.
def _cases():
    out = []
    # small and large row blocks at G = 40 (G % 4 == 0: the 16-byte store path of the first 32-group sub-tile)
    for block in (1, 5, 13, 16, 30, 31, 32, 33, 300):
        for row0 in (0, 8, 29):
            K = 16 if block <= 33 else 3
            if K * block - row0 - block // 3 <= 0:
                continue
            out.append(("mix", 40, K, block, row0, {}))
    # every register-tile tier, both sides of G % 4, and the slot sampler's generic kernel (G > 1024)
    for G, K, block, row0 in ((1, 16, 5, 8), (7, 8, 13, 0), (32, 16, 13, 29), (64, 16, 5, 0), (100, 3, 33, 8), (128, 8, 16, 8),
                              (129, 2, 300, 0), (200, 3, 31, 29), (256, 8, 13, 8), (1000, 2, 30, 0), (1100, 3, 33, 29)):
        out.append(("mix", G, K, block, row0, {}))
    # one feature of each row-mapped model (the single-feature kernels; ranks 1.. have nothing to push)
    for spec, G, K, block, row0 in (("nich", 40, 16, 5, 8), ("nich", 100, 3, 33, 0), ("nich", 256, 2, 300, 29),
                                    ("gp_big", 40, 16, 13, 0), ("gp_big", 128, 8, 16, 8), ("gp_big", 1000, 2, 31, 0),
                                    ("bnb", 64, 8, 16, 8), ("bnb", 200, 3, 32, 29), ("bb", 32, 16, 1, 0), ("bb", 129, 2, 300, 8),
                                    ("dd16", 100, 16, 5, 0), ("dd16", 40, 8, 30, 29), ("dd40", 256, 3, 13, 8), ("dd40", 64, 16, 31, 0)):
        out.append((spec, G, K, block, row0, {}))
    # shards of exactly one feature inside a mixed kind (F = K: single-feature kernels, prior NULL on ranks 1..)
    for G, K, block, row0 in ((40, 3, 13, 0), (100, 8, 16, 8), (64, 16, 5, 29), (256, 8, 33, 0)):
        out.append(("one_each", G, K, block, row0, {}))
    # a list whose caches exceed the 96 KB resident budget: the streaming kernel
    for G, K, block, row0, opts in ((256, 4, 13, 8, {}), (256, 2, 100, 0, {}), (256, 4, 13, 0, {OPT_ROW_TILE: 32})):
        out.append(("stream", G, K, block, row0, opts))
    # kernel variants behind options (the push goes through the same launchers)
    for tile in (32, 64):
        out.append(("mix", 200, 4, 13, 8, {OPT_ROW_TILE: tile}))
        out.append(("nich", 256, 3, 31, 0, {OPT_ROW_TILE: tile}))
    for v in (1, 3):
        for spec in ("nich", "gp_big", "bb", "dd16", "bnb"):
            out.append((spec, 100, 8, 13, 8, {OPT_SMALL_TILE: v}))
        out.append(("nich", 128, 3, 33, 0, {OPT_SMALL_TILE: v}))
    for v in (1, 2):
        out.append(("nich", 40, 16, 5, 29, {OPT_NICH_PACKED: v}))
        out.append(("nich", 256, 2, 300, 8, {OPT_NICH_PACKED: v}))
        out.append(("one_each", 100, 8, 16, 0, {OPT_NICH_PACKED: v}))
    return out


def _specs(name, K):
    if name == "mix":
        return [MIX[i % len(MIX)] for i in range(max(K, len(MIX)))]
    if name == "one_each":
        return [MIX[i % len(MIX)] for i in range(K)]
    if name == "stream":  # 32 GammaPoisson (32-float value tables per group) + 32 BetaBernoulli features
        return ["gp"] * 32 + ["bb"] * 32
    return [name]


def _case_id(c):
    name, G, K, block, row0, opts = c
    return "%s-G%d-K%d-b%d-r%d%s" % (name, G, K, block, row0, "".join("-o%d=%d" % kv for kv in opts.items()))


_GP_BITS = []  # lone GammaPoisson shards: did the value-table route come out bit-identical to score_batch?


@pytest.mark.parametrize("case", _cases(), ids=_case_id)
def test_push_slots(ctx, oracle, case):
    name, G, K, block, row0, opts = case
    n = K * block - row0 - block // 3
    specs = _specs(name, K)
    kind = Kind(ctx, oracle, specs, G, n, seed=5000 + 13 * G + block)
    parts = shards(len(specs), K)
    slots = Slots(K, block, G)
    # the bound of (a) is tight enough that a dropped or doubled prior falls outside it on nearly every cell of shard 0
    _, tol = kind.partial_ref(parts[0], True)
    assert np.mean(np.abs(kind.prior_np)[None, :] > tol) > 0.9
    with options(ctx, opts):
        push_all(ctx, kind, slots, parts, row0)
        check_slots(ctx, kind, slots, parts, row0, _case_id(case), gp_bits=_GP_BITS)


def test_push_lone_gp_bits(ctx, oracle):
    """a single GammaPoisson feature (values inside and beyond the value table): the push scores it through the table
    and the feature-list kernel, score_batch directly; reports whether both give the same bits (prints the result)"""
    kind = Kind(ctx, oracle, ["gp"], 40, 300, seed=77)
    slots = Slots(2, 150, 40)
    push_all(ctx, kind, slots, shards(1, 2), 0)
    check_slots(ctx, kind, slots, shards(1, 2), 0, "lone gp", gp_bits=_GP_BITS)
    print("lone GammaPoisson shards bit-identical to score_batch: %d of %d" % (sum(_GP_BITS), len(_GP_BITS)))


@pytest.mark.parametrize("G,K,block,a", [(40, 3, 50, 45), (7, 8, 5, 13), (128, 16, 13, 100), (256, 4, 40, 77)])
def test_push_split_launch(ctx, oracle, G, K, block, a):
    """one launch over [0, n) == two launches over [0, a) and [a, n) with row0 = a and the columns offset, bit for bit"""
    n = K * block - block // 3
    kind = Kind(ctx, oracle, MIX, G, n, seed=6100 + G)
    parts = shards(len(MIX), K)
    one, two = Slots(K, block, G), Slots(K, block, G)
    push_all(ctx, kind, one, parts, 0)
    push_all(ctx, kind, two, parts, 0, n=a)
    push_all(ctx, kind, two, parts, a, n=n - a, cols=[c[a:] for c in kind.cols])
    assert np.array_equal(one.read(), two.read())
    check_slots(ctx, kind, two, parts, 0, "split")


def test_push_zero_rows(ctx, oracle):
    kind = Kind(ctx, oracle, MIX, 40, 20, seed=61)
    slots = Slots(4, 5, 40)
    parts = shards(len(MIX), 4)
    for row0 in (0, 5, 20):
        for j, shard in enumerate(parts):
            ctx.score_push_batch([kind.feats[f] for f in shard], [kind.cols[f] for f in shard], 0, row0,
                                 kind.prior if j == 0 else None, slots.slot_ptrs(j), slots.block)
    assert np.all(slots.read() == SENTINEL)


# ------------------------------------------------------------------------------ flags, wait, slot sampler
class _DevWords:
    """a raw device pointer as a torch view (__cuda_array_interface__)"""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "strides": None,
                                         "version": 2}


def test_peer_flags(ctx):
    K, words = 5, 16  # owner o's flags: 16 words at base + 64 o
    base, handle = ctx.peer_alloc(4 * K * words)
    try:
        assert len(handle) == 64
        flags = torch.as_tensor(_DevWords(base, K * words), device="cuda")
        flag_ptrs = [base + 4 * words * o for o in range(K)]

        def read():
            torch.cuda.synchronize()
            return flags.cpu().numpy().reshape(K, words)

        want = np.zeros((K, words), np.int32)
        assert np.array_equal(read(), want)  # fresh peer_alloc memory reads zero
        for j, e in ((2, 7), (0, 3), (4, 9), (2, 8)):
            ctx.peer_signal(flag_ptrs, j, e)
            want[:, j] = e
            assert np.array_equal(read(), want), (j, e)
        ctx.peer_signal(flag_ptrs[:1], 15, 11)  # one peer, the last word
        want[0, 15] = 11
        assert np.array_equal(read(), want)
        # every pusher signals epoch 12 first; only then the waits (all satisfied) are enqueued
        for j in range(K):
            ctx.peer_signal(flag_ptrs, j, 12)
        for o in range(K):
            ctx.peer_wait(flag_ptrs[o], K, 12)
            ctx.peer_wait(flag_ptrs[o], K, 5)  # an epoch already passed
        want[:, :K] = 12
        assert np.array_equal(read(), want)
    finally:
        ctx.peer_free(base)


def owner_rows(K, block, n):
    return [(o * block, min(n, (o + 1) * block)) for o in range(K)]


def sample_slots(ctx, slots, K, n, G, u_d, assign_d):
    for o, (lo, hi) in enumerate(owner_rows(K, slots.block, n)):
        if hi > lo:
            ctx.sample_from_slots(slots.owner_base(o), K, slots.stride, hi - lo, G, u_d[lo:], assign_d[lo:])


def slot_sum(slots, area, K, n):
    """fp32 sum of the K slots of every row, in slot order (the sampler's order): [n][G]"""
    s = slots.slot_rows(area, 0)[:n].view(np.float32).copy()
    for j in range(1, K):
        s = s + slots.slot_rows(area, j)[:n].view(np.float32)
    return np.ascontiguousarray(s, dtype=np.float32)


def exact_from_sum(ctx, s, u_d):
    out = torch.full((s.shape[0],), -1, dtype=torch.int32, device="cuda")
    ctx.sample_from_scores(dev(s), s.shape[0], s.shape[1], u_d, out)
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("G,K,block", [(7, 8, 13), (40, 16, 5), (100, 3, 300), (256, 4, 31), (1000, 2, 33), (1100, 3, 40)])
def test_slot_sampler(ctx, oracle, G, K, block):
    n = K * block - block // 3
    specs = _specs("mix", K)
    kind = Kind(ctx, oracle, specs, G, n, seed=7100 + G)
    parts = shards(len(specs), K)
    slots = Slots(K, block, G)
    u = np.random.default_rng(G).random(n, dtype=np.float32)
    u_d = dev(u)
    assign_d = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    push_all(ctx, kind, slots, parts, 0)
    torch.cuda.synchronize()
    sample_slots(ctx, slots, K, n, G, u_d, assign_d)
    got = assign_d.cpu().numpy()
    area = slots.read()
    # exact: the stand-alone sampler on the slot sum formed in numpy
    assert np.array_equal(got, exact_from_sum(ctx, slot_sum(slots, area, K, n), u_d))
    # against float64: the oracle sampler on the full scores; every mismatch a near-tie, and rare
    full = kind.prior_np.astype(np.float64)[None, :] + sum(kind.refs)
    want = oracle.sample_rows(full.astype(np.float32), u)
    # score bound of the full row: the shards' bounds plus the rounding of the fp32 slot sum
    bound = np.zeros_like(full)
    run = np.zeros_like(full)
    for j, shard in enumerate(parts):
        ref, tol = kind.partial_ref(shard, j == 0)
        bound += tol
        run = run + ref if j else ref
        bound += 2.0 ** -23 * np.abs(run) if j else 0.0
    eps = EPS_TIE + 2 * bound.max(axis=1)  # a score error d moves every CDF boundary by at most ~2 d of the total
    diff = np.nonzero(got != want)[0]
    ok = [cases.explained_mismatch(full[i:i + 1], u[i:i + 1], got[i:i + 1], want[i:i + 1], eps[i])[0] for i in diff]
    assert all(ok), "%d of %d mismatches are not near-ties" % (len(ok) - sum(ok), len(ok))
    assert np.sum(got != want) <= max(2, 5e-3 * n)


@pytest.mark.parametrize("G,K,block", [(40, 4, 13), (100, 3, 300)])
def test_three_steps_alternating(ctx, oracle, G, K, block):
    """three steps as PeerFeatureShards runs them (slot buffers alternate by epoch, flags advance), all enqueued on one
    stream before the host looks: the uniforms and the row order of the columns change every step, so a stale slot or a
    wait that passes early gives a wrong assignment"""
    n = K * block - block // 3
    kind = Kind(ctx, oracle, MIX, G, n, seed=8100 + G)
    parts = shards(len(MIX), K)
    bufs = [Slots(K, block, G), Slots(K, block, G)]
    flags = torch.zeros(K * 16, dtype=torch.int32, device="cuda")
    flag_ptrs = [flags.data_ptr() + 64 * o for o in range(K)]
    rng = np.random.default_rng(G + K)
    steps = []
    for e in (1, 2, 3):
        perm = rng.permutation(n)
        cols = [column(w, w["values"][perm]) for w in kind.ws]
        u_d = dev(rng.random(n, dtype=np.float32))
        assign_d = torch.full((n,), -1, dtype=torch.int32, device="cuda")
        slots = bufs[e & 1]
        for j, shard in enumerate(parts):  # every rank: push, then signal
            ctx.score_push_batch([kind.feats[f] for f in shard], [cols[f] for f in shard], n, 0, kind.prior if j == 0 else None,
                                 slots.slot_ptrs(j), block)
            ctx.peer_signal(flag_ptrs, j, e)
        for o, (lo, hi) in enumerate(owner_rows(K, block, n)):  # then every owner: wait, sample
            ctx.peer_wait(flag_ptrs[o], K, e)
            if hi > lo:
                ctx.sample_from_slots(slots.owner_base(o), K, slots.stride, hi - lo, G, u_d[lo:], assign_d[lo:])
        steps.append((cols, u_d, assign_d))
    torch.cuda.synchronize()
    assert np.all(flags.cpu().numpy().reshape(K, 16)[:, :K] == 3)
    for e, (cols, u_d, assign_d) in enumerate(steps, 1):
        parts_d = [local_scores(ctx, kind, shard, j == 0, cols=cols) for j, shard in enumerate(parts)]
        s = parts_d[0].cpu().numpy()
        for p in parts_d[1:]:
            s = s + p.cpu().numpy()
        assert np.array_equal(assign_d.cpu().numpy(), exact_from_sum(ctx, s, u_d)), "step %d" % e
    for slots in bufs:
        area = slots.read()
        assert np.all(area[:, :, block * G:] == SENTINEL)


# ------------------------------------------------------------------------------ PeerFeatureShards on one GPU
class _StubDist:
    """the torch.distributed calls PeerFeatureShards makes, for W ranks in one process"""

    def __init__(self, world, handles):
        self.world, self.handles, self.rank = world, handles, 0

    def get_world_size(self, group=None):
        return self.world

    def get_rank(self, group=None):
        return self.rank

    def all_gather_object(self, out, obj, group=None):
        assert obj == self.handles[self.rank]
        out[:] = self.handles

    def barrier(self, group=None):
        pass


class _RankCtx:
    """rank r's context: peer memory from buffers made up front, the four launches of a step recorded"""

    def __init__(self, rank, bufs, handles, log):
        self.rank, self.bufs, self.handles, self.log = rank, bufs, handles, log

    def peer_alloc(self, nbytes):
        assert nbytes <= 4 * self.bufs[self.rank].numel()
        return self.bufs[self.rank].data_ptr(), self.handles[self.rank]

    def peer_open(self, handle):
        return self.bufs[self.handles.index(handle)].data_ptr()

    def peer_close(self, ptr):
        pass

    def peer_free(self, ptr):
        pass

    def __getattr__(self, name):
        if name in ("score_push_batch", "peer_signal", "peer_wait", "sample_from_slots"):
            return lambda *a, **k: self.log.append((self.rank, name, a, k))
        raise AttributeError(name)


# GammaPoisson features at 0, 1, 16, 17 only: with 18 features no GammaPoisson shard is ever alone
PFS_SPECS = ["gp", "gp_big", "nich", "bb", "dd16", "bnb", "nich", "bb", "dd40", "bnb", "nich", "bb", "dd16", "nich", "bb", "bnb",
             "gp_big", "gp"]


@pytest.mark.parametrize("n", [100, 5003])
@pytest.mark.parametrize("world,row_shards", [(w, r) for w in (2, 4, 8, 16) for r in (1, 2, 4, 8, 16) if r <= w])
def test_peer_feature_shards_replay(ctx, oracle, monkeypatch, world, row_shards, n):
    G, F = 40, len(PFS_SPECS)
    kind = Kind(ctx, oracle, PFS_SPECS, G, n, seed=9100)
    fs = world // row_shards
    handles = [("rank%d" % r).encode().ljust(64, b"\0") for r in range(world)]
    bufs = []
    for r in range(world):
        lo, hi = sharding.row_shard(n, r // fs, row_shards)
        bufs.append(torch.zeros((4 * 2 * fs * sharding.block_rows(hi - lo, fs) * G + 256) // 4, dtype=torch.int32, device="cuda"))
    stub = _StubDist(world, handles)
    monkeypatch.setattr(sharding, "dist", stub)
    log = []
    ranks = []
    for r in range(world):
        stub.rank = r
        ranks.append(sharding.PeerFeatureShards(_RankCtx(r, bufs, handles, log), n, G, row_shards=row_shards))

    # host-side layout: owned ranges partition the rows; slots of one owner's buffer are disjoint; flags past both buffers
    owned = sorted(s.owned() for s in ranks)
    covered = np.zeros(n, np.int32)
    for lo, hi in owned:
        covered[lo:hi] += 1
    assert np.all(covered == 1)
    for s in ranks:
        base = bufs[s.rank].data_ptr()
        assert s.bases[s.index] == base and s.flag_ptrs[s.index] == base + 4 * 2 * s.buf_floats
        assert s.flag_ptrs[s.index] + 4 * s.fs <= base + 4 * bufs[s.rank].numel()
        for k in (0, 1):
            spans = sorted((t.slot_ptrs[k][s.index], t.slot_ptrs[k][s.index] + 4 * t.slot_floats)
                           for t in ranks if t.rs_index == s.rs_index)
            assert len(spans) == s.fs and spans[0][0] >= base and spans[-1][1] <= base + 4 * 2 * s.buf_floats
            assert all(a[1] <= b[0] for a, b in zip(spans, spans[1:]))
            assert all(a % 16 == 0 for a, _ in spans)

    rng = np.random.default_rng(world * 100 + row_shards)
    steps = []
    for _ in range(2):  # two steps: both slot buffers, epochs 1 and 2
        u = rng.random(n, dtype=np.float32)
        u_d = dev(u)
        outs = []
        for s in ranks:
            r0, r1 = s.rows()
            lo, hi = s.owned()
            idx = s.features(F)
            out = torch.full((hi - lo,), -1, dtype=torch.int32, device="cuda")
            assert s.step([kind.feats[f] for f in idx], [kind.cols[f][r0:r1] for f in idx], kind.prior, u_d[lo:hi], out) == (lo, hi)
            outs.append(out)
        steps.append((u_d, outs))
    # replay in the phase order of a step: every rank's push and signal, then every rank's wait and sampler
    calls = [(r, name, a, k) for r, name, a, k in log]
    per_step = len(calls) // 2
    real = {"score_push_batch": ctx.score_push_batch, "peer_signal": ctx.peer_signal, "peer_wait": ctx.peer_wait,
            "sample_from_slots": ctx.sample_from_slots}
    for st in range(2):
        chunk = calls[st * per_step:(st + 1) * per_step]
        assert {r for r, *_ in chunk} == set(range(world))
        for phase in (("score_push_batch", "peer_signal"), ("peer_wait", "sample_from_slots")):
            for r, name, a, k in chunk:
                if name in phase:
                    real[name](*a, **k)
    torch.cuda.synchronize()

    # exact reference: every group's partials through score_batch, summed in fp32 in slot order, stand-alone sampler
    for u_d, outs in steps:
        for s, out in zip(ranks, outs):
            lo, hi = s.owned()
            if hi == lo:
                continue
            total = None
            for j in range(s.fs):
                idx = sharding.feature_shard(F, j, s.fs)
                p = local_scores(ctx, kind, idx, j == 0, cols=[c[lo:hi] for c in kind.cols], n=hi - lo).cpu().numpy()
                total = p if total is None else total + p
            assert np.array_equal(out.cpu().numpy(), exact_from_sum(ctx, total, u_d[lo:hi])), (s.rank, lo, hi)


# ------------------------------------------------------------------------------ argument checks
def test_push_argument_checks(ctx, oracle):
    """each bad request returns its status before anything launches and leaves the slots untouched"""
    from distributions_b200 import capi
    G, K, block = 40, 2, 16
    kind = Kind(ctx, oracle, ["nich", "bb"], G, 24, seed=31)
    slots = Slots(K, block, G)
    ptrs = slots.slot_ptrs(0)
    dpd = synth.dpd(32, G, 24, V=50)
    niw = synth.niw(33, G, 24, d=4)
    f_dpd = ctx.feature(capi.DPD).update_all(dpd)
    f_niw = ctx.feature(capi.NIW).update_all(niw)
    other = synth.bb(34, G + 1, 24)
    f_other = ctx.feature(capi.BB).update_all(other)
    f, c = kind.feats, kind.cols
    bad = [
        (capi.DistB200Error, "status 3", lambda: ctx.score_push_batch(f, c, 24, 0, kind.prior, ptrs * 8 + ptrs[:1], 2)),  # 17 owners
        (capi.DistB200Error, "status 1", lambda: ctx.score_push_batch(f, c, 24, 9, None, ptrs, block)),  # 33 rows > 2 x 16
        (capi.DistB200Error, "status 1", lambda: ctx.score_push_batch(f, c, 24, 0, None, ptrs[:1], block)),
        (capi.DistB200Error, "status 3", lambda: ctx.score_push_batch([f[0], f_dpd], [c[0], column(dpd)], 24, 0, None, ptrs, block)),
        (capi.DistB200Error, "status 3", lambda: ctx.score_push_batch([f_niw], [column(niw)], 24, 0, None, ptrs, block)),
        (capi.DistB200Error, "status 1", lambda: ctx.score_push_batch([f[0], f_other], [c[0], column(other)], 24, 0, None, ptrs, block)),
        (capi.DistB200Error, "status 1", lambda: ctx.score_push_batch(f, c, 24, 0, None, ptrs, 0)),  # block_rows = 0
        (capi.DistB200Error, "status 3", lambda: ctx.peer_signal([ptrs[0]] * 17, 0, 1)),
        (capi.DistB200Error, "status 3", lambda: ctx.peer_wait(ptrs[0], 33, 1)),
    ]
    for i, (exc, status, call) in enumerate(bad):
        with pytest.raises(exc, match=status):
            call()
        assert np.all(slots.read() == SENTINEL), i
