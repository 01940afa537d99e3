"""Python-3 mirror of the reference's `distributions.lp.models.*` classes for the mixture-scoring path
(SURVEY.md §8f rank 4; reference: distributions/lp/models/_nich.pyx:85-138 and siblings, doc/overview.rst:130-202).

    model = models.nich;  shared = model.Shared(mu=0, kappa=1, sigmasq=1, nu=1)
    mixture = model.Mixture(ctx)
    mixture.append(group) ...;  mixture.init(shared)
    mixture.add_value(shared, groupid, value);  mixture.score_value(shared, value, scores_accum)

Same names, argument meaning and accumulate semantics as the reference.  Group bookkeeping (add_value /
remove_value on the sufficient statistics) is host arithmetic in the reference's types (float32 Welford
updates for nich, nich.hpp:125-165; integer counts elsewhere); every score comes from the CUDA library through
the C-ABI -- there is no CPU scoring path here.  Two batched entries are added: score_values (score + sample
many rows) and add_values (batched Group::add_value on the device, groups read back).
"""
import numpy as np

from . import capi

_f32 = np.float32


class _Shared:
    FIELDS = ()

    def __init__(self, **kw):
        for k, default in self.FIELDS:
            setattr(self, k, kw.pop(k, default))
        if kw:
            raise TypeError("unknown Shared fields: %s" % sorted(kw))

    def dump(self):
        return {k: getattr(self, k) for k, _ in self.FIELDS}

    def load(self, raw):
        for k, _ in self.FIELDS:
            setattr(self, k, raw[k])
        return self


class _Group:
    FIELDS = ()

    def __init__(self):
        for k, default in self.FIELDS:
            setattr(self, k, default)

    def init(self, shared):
        for k, default in self.FIELDS:
            setattr(self, k, default)

    def dump(self):
        return {k: getattr(self, k) for k, _ in self.FIELDS}

    def load(self, raw):
        for k, _ in self.FIELDS:
            setattr(self, k, raw[k])
        return self


class _Mixture:
    """MixtureSlave (mixture.hpp:340-458) over a device-side value scorer."""
    model_id = None
    Group = None

    def __init__(self, ctx):
        self.ctx = ctx
        self.feature = ctx.feature(self.model_id)
        self.groups = []

    # container protocol of the lp Mixture (_nich.pyx:93-106)
    def __len__(self):
        return len(self.groups)

    def __getitem__(self, groupid):
        return self.groups[groupid]

    def append(self, group):
        self.groups.append(group)

    def clear(self):
        self.groups = []

    # mixture.hpp:354-359
    def init(self, shared):
        self.feature.update_all(self._workload(shared))

    # mixture.hpp:361-369
    def add_group(self, shared):
        g = self.Group()
        g.init(shared)
        self.groups.append(g)
        self.feature.add_group()

    # mixture.hpp:371-375: packed_remove = move the last group into the hole
    def remove_group(self, shared, groupid):
        self.groups[groupid] = self.groups[-1]
        self.groups.pop()
        self.feature.remove_group(groupid)

    # after dist_b200_regroup_batch moved this feature's groups: survivors in order, then n_empty fresh groups
    def regroup(self, shared, remap, n_empty):
        """follow a regroup of self.feature (capi.Context.regroup_batch): remap[g] = new id of old group g or -1; the
        host Groups are reordered the same way, fresh ones appended, and all of them re-read from the device"""
        remap = np.asarray(remap).ravel()
        assert remap.size == len(self.groups), "remap must have one entry per group"
        keep = [self.groups[g] for g in np.flatnonzero(remap >= 0)]
        assert all(remap[g] == i for i, g in enumerate(np.flatnonzero(remap >= 0))), "remap is not the stable compaction"
        fresh = []
        for _ in range(n_empty):
            grp = self.Group()
            grp.init(shared)
            fresh.append(grp)
        self.groups = keep + fresh
        assert self.feature.groups == len(self.groups), "the device feature was not regrouped to this G"
        self._pull_groups(shared)

    # mixture.hpp:377-398
    def add_value(self, shared, groupid, value):
        self.groups[groupid].add_value(shared, value)
        self.feature.update_group(groupid, self._stats(shared, self.groups[groupid]))

    def remove_value(self, shared, groupid, value):
        self.groups[groupid].remove_value(shared, value)
        self.feature.update_group(groupid, self._stats(shared, self.groups[groupid]))

    # mixture.hpp:416-425: ACCUMULATES into scores_accum
    def score_value(self, shared, value, scores_accum):
        assert len(scores_accum) == len(self.groups), "scores_accum != len(mixture)"
        assert scores_accum.dtype == np.float32
        self.ctx.score_value_host(self.feature, value, scores_accum)

    # mixture.hpp:400-414
    def score_value_group(self, shared, groupid, value):
        tmp = np.zeros(len(self.groups), np.float32)
        self.score_value(shared, value, tmp)
        return float(tmp[groupid])

    # mixture.hpp:427-438
    def score_data(self, shared):
        return float(self.score_data_grid([shared])[0])

    def score_data_grid(self, shareds):
        return self.feature.score_data_grid(np.array([self._pack_shared(s) for s in shareds], np.float32))

    # ---- batched entries (new) --------------------------------------------------------------------------
    def score_values(self, shared, values, prior, u, want_scores=False):
        """prior[G] (the clustering's vector, or None), u[n] uniforms: (assign[n], scores[n][G] or None)"""
        vals = np.ascontiguousarray(values, dtype=capi.COLUMN_DTYPE[self.model_id])
        return self.ctx.score_sample_batch_host([self.feature], [vals], prior, np.ascontiguousarray(u, np.float32), want_scores)

    def score_logp(self, shared, values, prior=None):
        """float32 logp[n] = log sum_g exp(prior[g] + score_value_group(g, values[n])) on the device, without the [n][G]
        scores.  With the clustering's Pitman-Yor vector as `prior` this is the log posterior-predictive density of each
        value under the mixture (niw: values is [n][d])."""
        vals = np.ascontiguousarray(values, dtype=capi.COLUMN_DTYPE[self.model_id])
        if self.model_id == capi.NIW:
            vals = vals.reshape(-1, shared.dim)
        return self.ctx.score_logp_batch_host([self.feature], [vals], prior)

    def add_values(self, shared, values, groupids):
        """batched add_value: one segmented reduction on the device, then the Groups are read back"""
        self.ctx.add_rows_batch_host([self.feature], [values], groupids)
        self._pull_groups(shared)

    def sample_values(self, shared, groupids, seed=0, row0=0):
        """batched Group::sample_value: one draw from the posterior predictive of group groupids[n] per row, with fresh
        parameters per value (Sampler::init + eval), on the device.  A draw depends on (seed, row0 + n) and the group
        only.  Returns an array of the model's Value type (bool for bb, [n][d] for niw)."""
        gid = np.ascontiguousarray(groupids, np.int32).ravel()
        assert gid.size == 0 or (gid.min() >= 0 and gid.max() < len(self.groups)), "bad group id"
        out = self.ctx.sample_values_batch_host([self.feature], gid, seed, row0)[0]
        return out.astype(bool) if self.model_id == capi.BB else out

    def sample_value(self, shared, groupid, seed=0):
        """Group::sample_value of one group"""
        v = self.sample_values(shared, [groupid], seed)[0]
        return v if self.model_id == capi.NIW else v.item()


# ------------------------------------------------------------------------------------------------------
class _NichShared(_Shared):
    FIELDS = (("mu", 0.0), ("kappa", 1.0), ("sigmasq", 1.0), ("nu", 1.0))  # EXAMPLE(), nich.hpp:71-78


class _NichGroup(_Group):
    FIELDS = (("count", 0), ("mean", _f32(0)), ("count_times_variance", _f32(0)))

    def add_value(self, shared, value):  # nich.hpp:125-133, fp32
        value = _f32(value)
        self.count += 1
        delta = _f32(value - _f32(self.mean))
        self.mean = _f32(_f32(self.mean) + _f32(delta / _f32(self.count)))
        self.count_times_variance = _f32(_f32(self.count_times_variance) + _f32(delta * _f32(value - self.mean)))

    def remove_value(self, shared, value):  # nich.hpp:146-165
        value = _f32(value)
        total = _f32(_f32(self.mean) * _f32(self.count))
        delta = _f32(value - _f32(self.mean))
        self.count -= 1
        if self.count == 0:
            self.mean = _f32(0)
        else:
            self.mean = _f32(_f32(total - value) / _f32(self.count))
        if self.count <= 1:
            self.count_times_variance = _f32(0)
        else:
            self.count_times_variance = _f32(_f32(self.count_times_variance) - _f32(delta * _f32(value - self.mean)))


class _NichMixture(_Mixture):
    model_id = capi.NICH
    Group = _NichGroup

    def _pack_shared(self, s):
        return [s.mu, s.kappa, s.sigmasq, s.nu]

    def _workload(self, s):
        return dict(model="nich", shared=np.array(self._pack_shared(s), np.float32),
                    count=np.array([g.count for g in self.groups], np.int32),
                    mean=np.array([g.mean for g in self.groups], np.float32),
                    ctv=np.array([g.count_times_variance for g in self.groups], np.float32))

    def _stats(self, s, g):
        return np.array([(g.count, g.mean, g.count_times_variance)], dtype=[("c", np.int32), ("m", np.float32), ("v", np.float32)])

    def _pull_groups(self, s):
        G = len(self.groups)
        raw = self.feature.download_stats(12 * G)
        c, m, v = raw[:4 * G].view(np.int32), raw[4 * G:8 * G].view(np.float32), raw[8 * G:].view(np.float32)
        for i, g in enumerate(self.groups):
            g.count, g.mean, g.count_times_variance = int(c[i]), _f32(m[i]), _f32(v[i])


class _CountSumGroup(_Group):
    FIELDS = (("count", 0), ("sum", 0))

    def add_value(self, shared, value):  # gp.hpp:109-116 / bnb.hpp:107-113 (uint32 arithmetic)
        self.count = (self.count + 1) & 0xFFFFFFFF
        self.sum = (self.sum + int(value)) & 0xFFFFFFFF

    def remove_value(self, shared, value):
        self.count = (self.count - 1) & 0xFFFFFFFF
        self.sum = (self.sum - int(value)) & 0xFFFFFFFF


class _CountSumMixture(_Mixture):
    def _stats(self, s, g):
        return np.array([g.count, g.sum], np.uint32)

    def _pull_groups(self, s):
        G = len(self.groups)
        raw = self.feature.download_stats(8 * G).view(np.uint32)
        for i, g in enumerate(self.groups):
            g.count, g.sum = int(raw[i]), int(raw[G + i])


class _GpShared(_Shared):
    FIELDS = (("alpha", 1.0), ("inv_beta", 1.0))  # gp.hpp:75-80


class _GpMixture(_CountSumMixture):
    model_id = capi.GP
    Group = _CountSumGroup

    def _pack_shared(self, s):
        return [s.alpha, s.inv_beta]

    def _workload(self, s):
        return dict(model="gp", shared=np.array(self._pack_shared(s), np.float32),
                    count=np.array([g.count for g in self.groups], np.uint32), sum=np.array([g.sum for g in self.groups], np.uint32))


class _BnbShared(_Shared):
    FIELDS = (("alpha", 1.0), ("beta", 1.0), ("r", 1))  # bnb.hpp:79-85


class _BnbMixture(_CountSumMixture):
    model_id = capi.BNB
    Group = _CountSumGroup

    def _pack_shared(self, s):
        return [s.alpha, s.beta]

    def _workload(self, s):
        return dict(model="bnb", shared=np.array([s.alpha, s.beta, s.r], np.float32),
                    count=np.array([g.count for g in self.groups], np.uint32), sum=np.array([g.sum for g in self.groups], np.uint32))


class _BbShared(_Shared):
    FIELDS = (("alpha", 0.5), ("beta", 2.0))  # bb.hpp:66-71


class _BbGroup(_Group):
    FIELDS = (("heads", 0), ("tails", 0))

    def add_value(self, shared, value):  # bb.hpp:102-107
        if value:
            self.heads += 1
        else:
            self.tails += 1

    def remove_value(self, shared, value):  # bb.hpp:117-122
        if value:
            self.heads -= 1
        else:
            self.tails -= 1


class _BbMixture(_Mixture):
    model_id = capi.BB
    Group = _BbGroup

    def _pack_shared(self, s):
        return [s.alpha, s.beta]

    def _workload(self, s):
        return dict(model="bb", shared=np.array(self._pack_shared(s), np.float32),
                    heads=np.array([g.heads for g in self.groups], np.int32), tails=np.array([g.tails for g in self.groups], np.int32))

    def _stats(self, s, g):
        return np.array([g.heads, g.tails], np.int32)

    def _pull_groups(self, s):
        G = len(self.groups)
        raw = self.feature.download_stats(8 * G).view(np.int32)
        for i, g in enumerate(self.groups):
            g.heads, g.tails = int(raw[i]), int(raw[G + i])


class _DdShared(_Shared):
    FIELDS = (("alphas", None),)

    def __init__(self, alphas=None, dim=16):
        self.alphas = np.asarray(alphas if alphas is not None else np.full(dim, 0.5), np.float32)  # dd.hpp:78-85

    @property
    def dim(self):
        return self.alphas.size


class _DdGroup(_Group):
    FIELDS = (("counts", None),)

    def init(self, shared):  # dd.hpp:113-121
        self.counts = np.zeros(shared.dim, np.int32)

    def add_value(self, shared, value):  # dd.hpp:123-130
        self.counts[int(value)] += 1

    def remove_value(self, shared, value):  # dd.hpp:142-149
        self.counts[int(value)] -= 1


class _DdMixture(_Mixture):
    model_id = capi.DD
    Group = _DdGroup

    def _pack_shared(self, s):
        return list(s.alphas)

    def _workload(self, s):
        return dict(model="dd", alphas=s.alphas, counts=np.array([g.counts for g in self.groups], np.int32).reshape(len(self.groups), s.dim))

    def _stats(self, s, g):
        return np.ascontiguousarray(g.counts, np.int32)

    def _pull_groups(self, s):
        G = len(self.groups)
        raw = self.feature.download_stats(4 * G * s.dim).view(np.int32).reshape(G, s.dim)
        for i, g in enumerate(self.groups):
            g.counts = raw[i].copy()


class _DpdShared(_Shared):
    """DirichletProcessDiscrete::Shared (dpd.hpp:59-152) with a FIXED set of known values: `values` (the keys of
    betas), `betas`, beta0 = max(0, 1 - sum betas) as Shared::protobuf_load computes it (dpd.hpp:104-125).  The
    Hierarchical-DP part that invents values (Shared::add_value / realize, dpd.hpp:66-100) is off the scoring path:
    change the value set with a new Shared and Mixture.init."""
    FIELDS = (("gamma", 1.0), ("alpha", 0.5), ("values", None), ("betas", None))
    OTHER = 0xFFFFFFFF  # dpd.hpp:55

    def __init__(self, gamma=1.0, alpha=0.5, values=None, betas=None, dim=100):
        self.gamma, self.alpha = float(gamma), float(alpha)
        if values is None:  # EXAMPLE(): dim 100, betas 1 / dim, beta0 = 0 (dpd.hpp:141-152)
            values, betas = np.arange(dim), np.full(dim, 1.0 / dim)
        self.values = np.asarray(values, np.uint32)
        self.betas = np.asarray(betas, np.float32)
        assert self.values.size == self.betas.size and np.unique(self.values).size == self.values.size
        self.beta0 = float(max(0.0, 1.0 - float(self.betas.astype(np.float64).sum())))
        self.index = {int(v): i for i, v in enumerate(self.values)}


class _DpdGroup(_Group):
    """SparseCounter<Value, count_t> (dpd.hpp:157-215): value -> count, absent = 0"""
    FIELDS = (("counts", None),)

    def __init__(self):
        self.counts = {}

    def init(self, shared):
        self.counts = {}

    def add_value(self, shared, value):  # dpd.hpp:188-196
        value = int(value)
        assert value != shared.OTHER, "cannot add OTHER"
        assert value in shared.index, "unknown value: %d" % value
        self.counts[value] = self.counts.get(value, 0) + 1

    def remove_value(self, shared, value):  # dpd.hpp:207-215
        value = int(value)
        assert value != shared.OTHER, "cannot remove OTHER"
        assert value in shared.index, "unknown value: %d" % value
        c = self.counts.get(value, 0) - 1
        if c:
            self.counts[value] = c
        else:
            self.counts.pop(value, None)

    def dense(self, shared):
        row = np.zeros(shared.values.size, np.int32)
        for v, c in self.counts.items():
            row[shared.index[v]] = c
        return row


class _DpdMixture(_Mixture):
    model_id = capi.DPD
    Group = _DpdGroup

    def _pack_shared(self, s):
        return [s.alpha]

    def _workload(self, s):
        counts = np.array([g.dense(s) for g in self.groups], np.int32).reshape(len(self.groups), s.values.size)
        return dict(model="dpd", alpha=s.alpha, beta0=s.beta0, keys=s.values, betas=s.betas, counts=counts)

    def _stats(self, s, g):
        return g.dense(s)

    def _pull_groups(self, s):
        G, V = len(self.groups), s.values.size
        raw = self.feature.download_stats(4 * G * V).view(np.int32).reshape(G, V)
        for i, g in enumerate(self.groups):
            g.counts = {int(s.values[v]): int(raw[i, v]) for v in np.nonzero(raw[i])[0]}


class _NiwShared(_Shared):
    """NormalInverseWishart::Shared (niw.hpp:52-170): mu[d], kappa, psi[d][d], nu"""
    FIELDS = (("mu", None), ("kappa", 1.0), ("psi", None), ("nu", None))

    def __init__(self, mu=None, kappa=1.0, psi=None, nu=None, dim=2):
        self.mu = np.asarray(mu if mu is not None else np.zeros(dim), np.float32)  # EXAMPLE(): niw.hpp:160-170
        d = self.mu.size
        self.kappa = float(kappa)
        self.psi = np.asarray(psi if psi is not None else np.eye(d), np.float32).reshape(d, d)
        self.nu = float(nu if nu is not None else d + 1)

    @property
    def dim(self):
        return self.mu.size


class _NiwGroup(_Group):
    """{count, sum_x, sum_xxT} (niw.hpp:187-190), float32 like the reference's Eigen Matrix<float>"""
    FIELDS = (("count", 0), ("sum_x", None), ("sum_xxT", None))

    def init(self, shared):  # niw.hpp:236-245
        self.count = 0
        self.sum_x = np.zeros(shared.dim, np.float32)
        self.sum_xxT = np.zeros((shared.dim, shared.dim), np.float32)

    def add_value(self, shared, value):  # niw.hpp:247-255: rank-1 updates
        x = np.asarray(value, np.float32)
        self.count += 1
        self.sum_x += x
        self.sum_xxT += np.outer(x, x)

    def remove_value(self, shared, value):  # niw.hpp:267-276
        x = np.asarray(value, np.float32)
        self.count -= 1
        self.sum_x -= x
        self.sum_xxT -= np.outer(x, x)


class _NiwMixture(_Mixture):
    """The reference has no NIW Mixture (niw.hpp has Group / Scorer only); this is the batched form of looping
    Group::score_value over the groups (mixture.hpp:321-337 semantics)."""
    model_id = capi.NIW
    Group = _NiwGroup

    def _workload(self, s):
        G, d = len(self.groups), s.dim
        return dict(model="niw", mu=s.mu, kappa=s.kappa, psi=s.psi, nu=s.nu,
                    count=np.array([g.count for g in self.groups], np.int32),
                    sum_x=np.array([g.sum_x for g in self.groups], np.float32).reshape(G, d),
                    sum_xxT=np.array([g.sum_xxT for g in self.groups], np.float32).reshape(G, d, d))

    def _stats(self, s, g):
        return np.concatenate([np.array([g.count], np.int32).view(np.float32), g.sum_x.ravel(), g.sum_xxT.ravel()]).astype(np.float32)

    def score_value(self, shared, value, scores_accum):
        assert len(scores_accum) == len(self.groups) and scores_accum.dtype == np.float32
        self.ctx.score_value_host(self.feature, np.asarray(value, np.float32).reshape(1, -1), scores_accum)

    def score_values(self, shared, values, prior, u, want_scores=False):
        vals = np.ascontiguousarray(values, np.float32).reshape(-1, shared.dim)
        return self.ctx.score_sample_batch_host([self.feature], [vals], prior, np.ascontiguousarray(u, np.float32), want_scores)

    def _pack_shared(self, s):  # kappa, nu, mu[d], psi[d][d]
        return np.concatenate([[s.kappa, s.nu], np.asarray(s.mu, np.float32).ravel(), np.asarray(s.psi, np.float32).ravel()]).astype(np.float32)

    def add_values(self, shared, values, groupids):
        """batched add_value (niw.hpp:247-255) as a per-group SYRK on the device, then the Groups are read back"""
        vals = np.ascontiguousarray(values, np.float32).reshape(-1, shared.dim)
        self.ctx.add_rows_batch_host([self.feature], [vals], groupids)
        self._pull_groups(shared)

    def _pull_groups(self, s):
        G, d = len(self.groups), s.dim
        raw = self.feature.download_stats(4 * G * (1 + d + d * d))
        cnt = raw[:4 * G].view(np.int32)
        sx = raw[4 * G:4 * G * (1 + d)].view(np.float32).reshape(G, d)
        sxx = raw[4 * G * (1 + d):].view(np.float32).reshape(G, d, d)
        for i, g in enumerate(self.groups):
            g.count, g.sum_x, g.sum_xxT = int(cnt[i]), sx[i].copy(), sxx[i].copy()


class MixtureIdTracker:
    """mixture.hpp:460-521: packed (contiguous, unstable under remove_group's swap-with-last) <-> global (fixed) group ids"""

    def __init__(self, group_count=0):
        self.init(group_count)

    def init(self, group_count=0):
        self.packed_to_global_ = []
        self.global_to_packed_ = {}
        self.global_size_ = 0
        for _ in range(group_count):
            self.add_group()

    def add_group(self):
        packed, glob = len(self.packed_to_global_), self.global_size_
        self.global_size_ += 1
        self.packed_to_global_.append(glob)
        self.global_to_packed_[glob] = packed

    def remove_group(self, packed):
        assert packed < self.packed_size(), "bad packed id: %d" % packed
        del self.global_to_packed_[self.packed_to_global_[packed]]
        last = self.packed_to_global_.pop()
        if packed != len(self.packed_to_global_):  # the last group moved into the hole
            self.packed_to_global_[packed] = last
            self.global_to_packed_[last] = packed

    def regroup(self, remap, n_empty):
        """follow dist_b200_regroup_batch: remap[p] = new packed id of packed group p, or -1 (dropped: its global id is
        retired); survivors keep their global ids, and n_empty fresh groups get new global ids at the end"""
        remap = np.asarray(remap).ravel()
        assert remap.size == self.packed_size(), "remap must have one entry per packed group"
        survivors = [self.packed_to_global_[p] for p in np.flatnonzero(remap >= 0)]
        for p in np.flatnonzero(remap < 0):
            del self.global_to_packed_[self.packed_to_global_[p]]
        self.packed_to_global_ = survivors
        self.global_to_packed_ = {glob: packed for packed, glob in enumerate(survivors)}
        for _ in range(n_empty):
            self.add_group()

    def packed_to_global(self, packed):
        assert packed < self.packed_size(), "bad packed id: %d" % packed
        return self.packed_to_global_[packed]

    def global_to_packed(self, glob):
        assert glob in self.global_to_packed_, "stale global id: %d" % glob
        return self.global_to_packed_[glob]

    def packed_size(self):
        return len(self.packed_to_global_)

    def global_size(self):
        return self.global_size_


class _Namespace:
    def __init__(self, name, Value, Shared, Group, Mixture):
        self.__name__, self.Value, self.Shared, self.Group, self.Mixture = name, Value, Shared, Group, Mixture


nich = _Namespace("nich", float, _NichShared, _NichGroup, _NichMixture)
gp = _Namespace("gp", int, _GpShared, _CountSumGroup, _GpMixture)
bnb = _Namespace("bnb", int, _BnbShared, _CountSumGroup, _BnbMixture)
bb = _Namespace("bb", bool, _BbShared, _BbGroup, _BbMixture)
dd = _Namespace("dd", int, _DdShared, _DdGroup, _DdMixture)
dpd = _Namespace("dpd", int, _DpdShared, _DpdGroup, _DpdMixture)
niw = _Namespace("niw", np.ndarray, _NiwShared, _NiwGroup, _NiwMixture)
MODELS = {m.__name__: m for m in (nich, gp, bnb, bb, dd, dpd, niw)}


# ------------------------------------------------------------------------------------------------------
# Clustering<int>::{PitmanYor, LowEntropy} and their Mixture drivers (clustering.hpp:45-331, mixture.hpp:48-163;
# Python reference: distributions/lp/clustering.pyx:120-257)
class _ClusteringMixture:
    """MixtureDriver bookkeeping (mixture.hpp:59-122): group sizes, the set of empty groups, the sample size;
    add_value / remove_value report whether a group was added / removed so that the feature mixtures follow
    (doc/overview.rst:185-202).  score_value OVERWRITES scores with the prior vector, evaluated on the device."""

    def __init__(self, ctx):
        self.ctx = ctx
        self.counts = []
        self.empty_groupids = set()
        self.sample_size = 0

    def __len__(self):
        return len(self.counts)

    def init(self, model, counts=None):
        if counts is not None:
            self.counts = [int(c) for c in counts]
        self.empty_groupids = {i for i, c in enumerate(self.counts) if c == 0}
        self.sample_size = sum(self.counts)
        assert self.empty_groupids, "missing empty groups"  # mixture.hpp:150

    def add_value(self, model, groupid, count=1):  # mixture.hpp:77-93
        assert count, "cannot add zero values"
        add_group = self.counts[groupid] == 0
        self.counts[groupid] += count
        self.sample_size += count
        if add_group:
            self.empty_groupids.discard(groupid)
            self.empty_groupids.add(len(self.counts))
            self.counts.append(0)
        return add_group

    def remove_value(self, model, groupid, count=1):  # mixture.hpp:95-122
        assert count and 0 < count <= self.counts[groupid], "cannot remove more values than are in group"
        self.counts[groupid] -= count
        self.sample_size -= count
        remove_group = self.counts[groupid] == 0
        if remove_group:
            last = len(self.counts) - 1
            if groupid != last:
                self.counts[groupid] = self.counts[-1]
                if self.counts[-1] == 0:
                    self.empty_groupids.discard(last)
                    self.empty_groupids.add(groupid)
            self.counts.pop()
        return remove_group

    def regroup(self, n_empty=1, counts=None):
        """the batched form of the bookkeeping above (dist_b200_regroup_batch): groups of size 0 are dropped, the live
        ones keep their order, and n_empty fresh empty groups follow.  counts (optional) replaces the group sizes first,
        e.g. the device's count_assignments.  Returns remap[g] = new id of old group g, -1 when dropped."""
        assert n_empty >= 1, "a mixture keeps at least one empty group"  # mixture.hpp:150
        if counts is not None:
            self.counts = [int(c) for c in counts]
        c = np.asarray(self.counts, dtype=np.int64)
        live = c > 0
        remap = np.where(live, np.cumsum(live) - 1, -1).astype(np.int32)
        K = int(live.sum())
        self.counts = [int(v) for v in c[live]] + [0] * n_empty
        self.empty_groupids = set(range(K, K + n_empty))
        self.sample_size = int(c[live].sum())
        return remap

    def score_value(self, model, scores):
        assert len(scores) == len(self.counts) and scores.dtype == np.float32
        scores[:] = self._prior(model)
        return scores


class PitmanYor:
    """Clustering<int>::PitmanYor (clustering.hpp:45-240); EXAMPLES as lp/clustering.pyx:211-217"""

    def __init__(self, alpha=1.0, d=0.0):
        self.alpha, self.d = float(alpha), float(d)

    class Mixture(_ClusteringMixture):
        def _prior(self, model):
            return self.ctx.prior_pitman_yor_host(model.alpha, model.d, self.counts)


class LowEntropy:
    """Clustering<int>::LowEntropy (clustering.hpp:245-331)"""

    def __init__(self, dataset_size):
        self.dataset_size = int(dataset_size)

    class Mixture(_ClusteringMixture):
        def _prior(self, model):
            return self.ctx.prior_low_entropy_host(model.dataset_size, self.counts)
