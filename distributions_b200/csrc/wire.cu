// wire.cu -- the reference's protobuf wire format (distributions/io/schema.proto:36-158) decoded straight
// into the packed SoA arrays update_all takes: Shared + G serialized Group messages -> statistics on the
// device, without materialising host object graphs (SURVEY.md 8f rank 4).  Host code only.
//
// Only what the schema uses is implemented: varint (wire type 0), 64-bit (1), length-delimited (2, also
// packed repeated scalars), 32-bit (5).  proto2 repeated scalars may arrive packed or unpacked; both are
// accepted.  Unknown fields are skipped, as protobuf readers do.  Counts are uint64 on the wire and 32-bit
// in the reference's Groups (e.g. nich.hpp:98-101, gp.hpp:84-87): a value that does not fit is an error.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "common.cuh"

namespace distb200 {
namespace {

struct Reader {
    const uint8_t *p, *end;
    bool ok = true;

    bool done() const { return p >= end || !ok; }
    uint64_t varint() {
        uint64_t v = 0;
        for (int shift = 0; shift < 64; shift += 7) {
            if (p >= end) {
                ok = false;
                return 0;
            }
            const uint8_t b = *p++;
            v |= static_cast<uint64_t>(b & 0x7f) << shift;
            if (!(b & 0x80)) return v;
        }
        ok = false;  // more than 10 bytes
        return 0;
    }
    float fixed32() {
        if (end - p < 4) {
            ok = false;
            return 0.f;
        }
        float f;
        std::memcpy(&f, p, 4);  // little-endian host (x86-64 / aarch64)
        p += 4;
        return f;
    }
    Reader sub() {  // length-delimited payload
        const uint64_t n = varint();
        if (!ok || n > static_cast<uint64_t>(end - p)) {
            ok = false;
            return Reader{p, p};
        }
        Reader r{p, p + n};
        p += n;
        return r;
    }
    void skip(int wire_type) {
        switch (wire_type) {
            case 0: varint(); break;
            case 1: if (end - p < 8) ok = false; else p += 8; break;
            case 2: sub(); break;
            case 5: if (end - p < 4) ok = false; else p += 4; break;
            default: ok = false;
        }
    }
};

// one field occurrence of a float / varint scalar, packed or not, appended to `out`
void read_floats(Reader &r, int wire_type, std::vector<float> &out) {
    if (wire_type == 5) out.push_back(r.fixed32());
    else if (wire_type == 2) {
        Reader s = r.sub();
        while (!s.done()) out.push_back(s.fixed32());
        if (!s.ok) r.ok = false;
    } else r.ok = false;
}
void read_varints(Reader &r, int wire_type, std::vector<uint64_t> &out) {
    if (wire_type == 0) out.push_back(r.varint());
    else if (wire_type == 2) {
        Reader s = r.sub();
        while (!s.done()) out.push_back(s.varint());
        if (!s.ok) r.ok = false;
    } else r.ok = false;
}

struct Fields {  // up to 5 numbered fields of one message, everything the schema's model messages need
    std::vector<float> f[6];
    std::vector<uint64_t> v[6];
};

// kinds: 'f' float field, 'v' varint field, 0 = not present in this message (skipped)
bool parse(const void *msg, size_t len, const char kinds[6], Fields &out) {
    Reader r{static_cast<const uint8_t *>(msg), static_cast<const uint8_t *>(msg) + len};
    while (!r.done()) {
        const uint64_t key = r.varint();
        if (!r.ok) break;
        const int wt = static_cast<int>(key & 7);
        const uint64_t num = key >> 3;
        if (num >= 1 && num <= 5 && kinds[num] == 'f') read_floats(r, wt, out.f[num]);
        else if (num >= 1 && num <= 5 && kinds[num] == 'v') read_varints(r, wt, out.v[num]);
        else r.skip(wt);
    }
    return r.ok;
}

bool fits32(uint64_t v) { return v <= 0xFFFFFFFFull; }

}  // namespace

// Eigen's isApprox(m, m^T) (niw.hpp:45-50): |m - m^T|_F <= 1e-5 min(|m|_F, |m^T|_F)
static bool symmetric(const float *m, size_t d) {
    double diff = 0, norm = 0;
    for (size_t i = 0; i < d; ++i)
        for (size_t j = 0; j < d; ++j) {
            const double a = m[i * d + j], b = m[j * d + i];
            diff += (a - b) * (a - b);
            norm += a * a;
        }
    return diff <= 1e-10 * norm;
}
// LDLT with a positive diagonal (niw.hpp:52-61), as a Cholesky factorisation in double
static bool positive_definite(const float *m, size_t d) {
    std::vector<double> L(d * d, 0.0);
    for (size_t j = 0; j < d; ++j) {
        double s = m[j * d + j];
        for (size_t k = 0; k < j; ++k) s -= L[j * d + k] * L[j * d + k];
        if (!(s > 0.0)) return false;
        L[j * d + j] = std::sqrt(s);
        for (size_t i = j + 1; i < d; ++i) {
            double t = m[i * d + j];
            for (size_t k = 0; k < j; ++k) t -= L[i * d + k] * L[j * d + k];
            L[i * d + j] = t / L[j * d + j];
        }
    }
    return true;
}

static uint32_t fbits(float f) {
    uint32_t u;
    std::memcpy(&u, &f, 4);
    return u;
}

int wire_decode(dist_b200_ctx *ctx, int model, const void *shared_msg, size_t shared_len, const void *const *group_msgs,
                const size_t *group_lens, int G, WireFeature &out) {
    auto bad = [&](const char *what) { return fail(ctx, DIST_B200_ERR_INVALID, std::string("wire: ") + what); };
    if (!shared_msg && shared_len) return bad("null Shared message");
    if (G < 0 || (G && (!group_msgs || !group_lens))) return bad("null Group messages");
    for (int i = 0; i < G; ++i)
        if (!group_msgs[i] && group_lens[i]) return bad("null Group message with a non-zero length");
    // non-repeated fields: a field that occurs more than once takes its LAST value, as protobuf readers
    // (the reference's included) do -- hence .empty() / .back() below
    Fields sh;
    const size_t g = static_cast<size_t>(G);
    switch (model) {
        case DIST_B200_NICH: {  // schema.proto:131-145
            if (!parse(shared_msg, shared_len, "\0ffff", sh)) return bad("malformed NormalInverseChiSq.Shared");
            for (int k = 1; k <= 4; ++k)
                if (sh.f[k].empty()) return bad("NormalInverseChiSq.Shared: missing required field");
            out.shared = {sh.f[1].back(), sh.f[2].back(), sh.f[3].back(), sh.f[4].back()};
            out.stats.assign(3 * g, 0);
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0vff\0", m)) return bad("malformed NormalInverseChiSq.Group");
                if (m.v[1].empty() || m.f[2].empty() || m.f[3].empty()) return bad("NormalInverseChiSq.Group: missing required field");
                if (m.v[1].back() > 0x7FFFFFFFull) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: count exceeds 32 bits");
                out.stats[i] = static_cast<uint32_t>(m.v[1].back());
                out.stats[g + i] = fbits(m.f[2].back());
                out.stats[2 * g + i] = fbits(m.f[3].back());
            }
        } break;
        case DIST_B200_GP: {  // schema.proto:105-116: count, sum, log_prod
            if (!parse(shared_msg, shared_len, "\0ff\0\0", sh)) return bad("malformed GammaPoisson.Shared");
            if (sh.f[1].empty() || sh.f[2].empty()) return bad("GammaPoisson.Shared: missing required field");
            out.shared = {sh.f[1].back(), sh.f[2].back()};
            out.stats.assign(3 * g, 0);
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0vvf\0", m)) return bad("malformed GammaPoisson.Group");
                if (m.v[1].empty() || m.v[2].empty() || m.f[3].empty()) return bad("GammaPoisson.Group: missing required field");
                if (!fits32(m.v[1].back()) || !fits32(m.v[2].back())) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: count exceeds 32 bits");
                out.stats[i] = static_cast<uint32_t>(m.v[1].back());
                out.stats[g + i] = static_cast<uint32_t>(m.v[2].back());
                out.stats[2 * g + i] = fbits(m.f[3].back());
            }
        } break;
        case DIST_B200_BNB: {  // schema.proto:118-129
            if (!parse(shared_msg, shared_len, "\0ffv\0", sh)) return bad("malformed BetaNegativeBinomial.Shared");
            if (sh.f[1].empty() || sh.f[2].empty() || sh.v[3].empty()) return bad("BetaNegativeBinomial.Shared: missing required field");
            if (!fits32(sh.v[3].back())) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: r exceeds 32 bits");
            out.shared = {sh.f[1].back(), sh.f[2].back(), static_cast<float>(sh.v[3].back())};
            out.keys = {static_cast<uint32_t>(sh.v[3].back())};  // r, exact
            out.stats.assign(2 * g, 0);
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0vv\0\0", m)) return bad("malformed BetaNegativeBinomial.Group");
                if (m.v[1].empty() || m.v[2].empty()) return bad("BetaNegativeBinomial.Group: missing required field");
                if (!fits32(m.v[1].back()) || !fits32(m.v[2].back())) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: count exceeds 32 bits");
                out.stats[i] = static_cast<uint32_t>(m.v[1].back());
                out.stats[g + i] = static_cast<uint32_t>(m.v[2].back());
            }
        } break;
        case DIST_B200_BB: {  // schema.proto:55-65
            if (!parse(shared_msg, shared_len, "\0ff\0\0", sh)) return bad("malformed BetaBernoulli.Shared");
            if (sh.f[1].empty() || sh.f[2].empty()) return bad("BetaBernoulli.Shared: missing required field");
            out.shared = {sh.f[1].back(), sh.f[2].back()};
            out.stats.assign(2 * g, 0);
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0vv\0\0", m)) return bad("malformed BetaBernoulli.Group");
                if (m.v[1].empty() || m.v[2].empty()) return bad("BetaBernoulli.Group: missing required field");
                if (m.v[1].back() > 0x7FFFFFFFull || m.v[2].back() > 0x7FFFFFFFull) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: count exceeds 32 bits");
                out.stats[i] = static_cast<uint32_t>(m.v[1].back());
                out.stats[g + i] = static_cast<uint32_t>(m.v[2].back());
            }
        } break;
        case DIST_B200_DD: {  // schema.proto:67-75: repeated alphas / repeated counts
            if (!parse(shared_msg, shared_len, "\0f\0\0\0", sh)) return bad("malformed DirichletDiscrete.Shared");
            const size_t dim = sh.f[1].size();
            if (dim < 1 || dim > 256) return bad("DirichletDiscrete.Shared: dim must be 1..256");
            out.shared = sh.f[1];
            out.dim = static_cast<int>(dim);
            out.stats.assign(g * dim, 0);
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0v\0\0\0", m)) return bad("malformed DirichletDiscrete.Group");
                if (m.v[1].size() != dim) return bad("DirichletDiscrete.Group: counts length differs from Shared.alphas (dd.hpp:104-111)");
                for (size_t v = 0; v < dim; ++v) {
                    if (m.v[1][v] > 0x7FFFFFFFull) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: count exceeds 32 bits");
                    out.stats[i * dim + v] = static_cast<uint32_t>(m.v[1][v]);
                }
            }
        } break;
        case DIST_B200_DPD: {  // schema.proto:77-90; Shared::protobuf_load dpd.hpp:104-125
            if (!parse(shared_msg, shared_len, "\0ffvfv", sh)) return bad("malformed DirichletProcessDiscrete.Shared");
            if (sh.f[1].empty() || sh.f[2].empty()) return bad("DirichletProcessDiscrete.Shared: missing required field");
            const size_t V = sh.v[3].size();
            if (V < 1 || sh.f[4].size() != V || sh.v[5].size() != V) return bad("DirichletProcessDiscrete.Shared: values / betas / counts lengths differ");
            double beta_sum = 0;  // dpd.hpp:114-124
            out.shared = {sh.f[1].back(), sh.f[2].back(), 0.f};
            for (size_t v = 0; v < V; ++v) {
                if (!fits32(sh.v[3][v])) return bad("DirichletProcessDiscrete.Shared: value exceeds 32 bits");
                if (!(sh.f[4][v] > 0.f)) return bad("DirichletProcessDiscrete.Shared: beta must be positive");
                out.keys.push_back(static_cast<uint32_t>(sh.v[3][v]));
                out.shared.push_back(sh.f[4][v]);
                beta_sum += sh.f[4][v];
            }
            if (beta_sum > 1 + 1e-4) return bad("DirichletProcessDiscrete.Shared: betas sum to more than 1");
            out.shared[2] = static_cast<float>(std::max(0.0, 1.0 - beta_sum));
            out.dim = static_cast<int>(V);
            out.stats.assign(g * V, 0);
            // key -> column of the dense [G][V] table, Shared's order
            std::vector<std::pair<uint32_t, uint32_t>> index(V);
            for (size_t v = 0; v < V; ++v) index[v] = {out.keys[v], static_cast<uint32_t>(v)};
            std::sort(index.begin(), index.end());
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0vv\0\0", m)) return bad("malformed DirichletProcessDiscrete.Group");
                if (m.v[1].size() != m.v[2].size()) return bad("DirichletProcessDiscrete.Group: keys / values lengths differ");
                for (size_t k = 0; k < m.v[1].size(); ++k) {
                    if (!fits32(m.v[1][k]) || m.v[2][k] > 0x7FFFFFFFull) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: count exceeds 32 bits");
                    const uint32_t key = static_cast<uint32_t>(m.v[1][k]);
                    auto it = std::lower_bound(index.begin(), index.end(), std::make_pair(key, 0u));
                    if (it == index.end() || it->first != key) return bad("DirichletProcessDiscrete.Group: key absent from Shared.values");
                    out.stats[i * V + it->second] += static_cast<uint32_t>(m.v[2][k]);
                }
            }
        } break;
        case DIST_B200_NIW: {  // schema.proto:147-161; Shared::protobuf_load niw.hpp:105-134, Group::protobuf_load :192-216
            if (!parse(shared_msg, shared_len, "\0ffff", sh)) return bad("malformed NormalInverseWishart.Shared");
            const size_t d = sh.f[1].size();
            if (d < 1) return bad("NormalInverseWishart.Shared: dim must be at least 1");
            if (d > 128) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: NormalInverseWishart.Shared: dim above 128 is not supported");
            if (sh.f[2].empty() || sh.f[4].empty()) return bad("NormalInverseWishart.Shared: missing required field");
            if (sh.f[3].size() != d * d) return bad("NormalInverseWishart.Shared: psi is not dim x dim (niw.hpp:92-94)");
            const float kappa = sh.f[2].back(), nu = sh.f[4].back();
            if (!(kappa > 0.f)) return bad("NormalInverseWishart.Shared: kappa must be positive (niw.hpp:115)");
            if (!(nu > static_cast<float>(d) - 1.f)) return bad("NormalInverseWishart.Shared: nu must exceed dim - 1 (niw.hpp:132)");
            if (!symmetric(sh.f[3].data(), d) || !positive_definite(sh.f[3].data(), d))
                return bad("NormalInverseWishart.Shared: psi is not symmetric positive definite (niw.hpp:127)");
            // packed Shared: kappa, nu, mu[d], psi[d][d]
            out.shared = {kappa, nu};
            out.shared.insert(out.shared.end(), sh.f[1].begin(), sh.f[1].end());
            out.shared.insert(out.shared.end(), sh.f[3].begin(), sh.f[3].end());
            out.dim = static_cast<int>(d);
            // statistics: count[G] | sum_x[G][d] | sum_xxT[G][d][d]
            out.stats.assign(g * (1 + d + d * d), 0);
            for (size_t i = 0; i < g; ++i) {
                Fields m;
                if (!parse(group_msgs[i], group_lens[i], "\0vff\0", m)) return bad("malformed NormalInverseWishart.Group");
                if (m.v[1].empty()) return bad("NormalInverseWishart.Group: missing required field");
                if (m.v[1].back() > 0x7FFFFFFFull) return bad("NormalInverseWishart.Group: count is negative or exceeds 31 bits");
                if (m.f[2].size() != d || m.f[3].size() != d * d) return bad("NormalInverseWishart.Group: sum_x / sum_xxT sizes differ from Shared's dim");
                if (!symmetric(m.f[3].data(), d)) return bad("NormalInverseWishart.Group: sum_xxT is not symmetric (niw.hpp:214)");
                out.stats[i] = static_cast<uint32_t>(m.v[1].back());
                for (size_t k = 0; k < d; ++k) out.stats[g + i * d + k] = fbits(m.f[2][k]);
                for (size_t k = 0; k < d * d; ++k) out.stats[g + g * d + i * d * d + k] = fbits(m.f[3][k]);
            }
        } break;
        default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: model has no wire loader");
    }
    return DIST_B200_OK;
}

// Clustering message (schema.proto:36-53): which = 1 PitmanYor {alpha, d}, 2 LowEntropy {dataset_size}
int wire_decode_clustering(dist_b200_ctx *ctx, const void *msg, size_t len, int *which, float *alpha, float *d,
                           uint64_t *dataset_size) {
    Reader r{static_cast<const uint8_t *>(msg), static_cast<const uint8_t *>(msg) + len};
    *which = 0;
    while (!r.done()) {
        const uint64_t key = r.varint();
        if (!r.ok) break;
        const int wt = static_cast<int>(key & 7);
        const uint64_t num = key >> 3;
        if (wt == 2 && (num == 1 || num == 2)) {
            Reader s = r.sub();
            if (!r.ok) break;
            Fields m;
            if (num == 1) {
                if (!parse(s.p, static_cast<size_t>(s.end - s.p), "\0ff\0\0", m) || m.f[1].empty() || m.f[2].empty())
                    return fail(ctx, DIST_B200_ERR_INVALID, "wire: malformed Clustering.PitmanYor");
                *alpha = m.f[1].back();
                *d = m.f[2].back();
            } else {
                if (!parse(s.p, static_cast<size_t>(s.end - s.p), "\0v\0\0\0", m) || m.v[1].empty())
                    return fail(ctx, DIST_B200_ERR_INVALID, "wire: malformed Clustering.LowEntropy");
                *dataset_size = m.v[1].back();
            }
            *which = static_cast<int>(num);
        } else {
            r.skip(wt);
        }
    }
    if (!r.ok || *which == 0) return fail(ctx, DIST_B200_ERR_INVALID, "wire: malformed Clustering message");
    return DIST_B200_OK;
}

// ---- encoder: SoA statistics -> Group messages, canonical proto2 output (fields in number order,
// repeated scalars unpacked), i.e. byte-identical to what the reference's writer produces
namespace {
void put_varint(std::vector<uint8_t> &o, uint64_t v) {
    while (v >= 0x80) {
        o.push_back(static_cast<uint8_t>(v) | 0x80);
        v >>= 7;
    }
    o.push_back(static_cast<uint8_t>(v));
}
void put_u(std::vector<uint8_t> &o, int field, uint64_t v) {
    put_varint(o, static_cast<uint64_t>(field) << 3);
    put_varint(o, v);
}
void put_f(std::vector<uint8_t> &o, int field, uint32_t bits) {
    put_varint(o, (static_cast<uint64_t>(field) << 3) | 5);
    for (int k = 0; k < 4; ++k) o.push_back(static_cast<uint8_t>(bits >> (8 * k)));
}
}  // namespace

int wire_encode_groups(dist_b200_ctx *ctx, int model, int G, int dim, const uint32_t *keys, const uint32_t *stats,
                       size_t stats_words, std::vector<uint8_t> &out, std::vector<size_t> &lens) {
    const size_t g = static_cast<size_t>(G);
    size_t need = 0;
    switch (model) {
        case DIST_B200_NICH: case DIST_B200_GP: need = 3 * g; break;
        case DIST_B200_BNB: case DIST_B200_BB: need = 2 * g; break;
        case DIST_B200_DD: case DIST_B200_DPD: need = g * static_cast<size_t>(dim); break;
        case DIST_B200_NIW: need = g * (1 + static_cast<size_t>(dim) + static_cast<size_t>(dim) * dim); break;
        default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: model has no Group writer");
    }
    if (G < 0 || stats_words < need || (G && !stats) || (model == DIST_B200_DPD && G && !keys))
        return fail(ctx, DIST_B200_ERR_INVALID, "wire_encode: statistics array too short");
    out.clear();
    lens.assign(g, 0);
    for (size_t i = 0; i < g; ++i) {
        const size_t start = out.size();
        switch (model) {
            case DIST_B200_NICH:  // count, mean, count_times_variance
                put_u(out, 1, stats[i]);
                put_f(out, 2, stats[g + i]);
                put_f(out, 3, stats[2 * g + i]);
                break;
            case DIST_B200_GP:  // count, sum, log_prod
                put_u(out, 1, stats[i]);
                put_u(out, 2, stats[g + i]);
                put_f(out, 3, stats[2 * g + i]);
                break;
            case DIST_B200_BNB:
            case DIST_B200_BB:
                put_u(out, 1, stats[i]);
                put_u(out, 2, stats[g + i]);
                break;
            case DIST_B200_DD:
                for (int v = 0; v < dim; ++v) put_u(out, 1, stats[i * dim + v]);
                break;
            case DIST_B200_NIW: {  // count (int32: negative values sign-extend to 64 bits), sum_x, sum_xxT row-major
                const size_t d = static_cast<size_t>(dim);
                put_u(out, 1, static_cast<uint64_t>(static_cast<int64_t>(static_cast<int32_t>(stats[i]))));
                for (size_t k = 0; k < d; ++k) put_f(out, 2, stats[g + i * d + k]);
                for (size_t k = 0; k < d * d; ++k) put_f(out, 3, stats[g + g * d + i * d * d + k]);
            } break;
            default:  // dpd: sparse (keys, values), non-zero counts in Shared order
                for (int v = 0; v < dim; ++v)
                    if (stats[i * dim + v]) put_u(out, 1, keys[v]);
                for (int v = 0; v < dim; ++v)
                    if (stats[i * dim + v]) put_u(out, 2, stats[i * dim + v]);
                break;
        }
        lens[i] = out.size() - start;
    }
    return DIST_B200_OK;
}

// Shared message of a model from the packed floats wire_decode returns.  dpd: keys = values[V] followed by the
// per-value totals Shared::counts[V] (dpd.hpp:64, :126-138 -- the sum of the groups' counts of the value when every
// add_value went through both, as the mixture drivers do); niw: kappa, nu, mu[d], psi[d][d].
int wire_encode_shared(dist_b200_ctx *ctx, int model, const float *shared, size_t n_shared, const uint32_t *keys,
                       size_t n_keys, std::vector<uint8_t> &out) {
    auto need = [&](size_t n) { return n_shared == n && shared; };
    out.clear();
    auto put_float = [&](int field, float f) {
        uint32_t u;
        std::memcpy(&u, &f, 4);
        put_f(out, field, u);
    };
    switch (model) {
        case DIST_B200_NICH:
            if (!need(4)) break;
            for (int k = 0; k < 4; ++k) put_float(k + 1, shared[k]);
            return DIST_B200_OK;
        case DIST_B200_GP:
        case DIST_B200_BB:
            if (!need(2)) break;
            put_float(1, shared[0]);
            put_float(2, shared[1]);
            return DIST_B200_OK;
        case DIST_B200_BNB:
            if (!need(3) || n_keys != 1 || !keys) break;
            put_float(1, shared[0]);
            put_float(2, shared[1]);
            put_u(out, 3, keys[0]);
            return DIST_B200_OK;
        case DIST_B200_DD:
            if (!shared || n_shared < 1 || n_shared > 256) break;
            for (size_t v = 0; v < n_shared; ++v) put_float(1, shared[v]);
            return DIST_B200_OK;
        case DIST_B200_DPD: {  // gamma, alpha, values, betas, counts (dpd.hpp:126-138)
            if (!shared || n_shared < 4 || !keys) break;
            const size_t V = n_shared - 3;
            if (n_keys != 2 * V) break;
            put_float(1, shared[0]);
            put_float(2, shared[1]);
            for (size_t v = 0; v < V; ++v) put_u(out, 3, keys[v]);
            for (size_t v = 0; v < V; ++v) put_float(4, shared[3 + v]);
            for (size_t v = 0; v < V; ++v) put_u(out, 5, keys[V + v]);
            return DIST_B200_OK;
        }
        case DIST_B200_NIW: {  // mu, kappa, psi, nu (niw.hpp:136-156)
            size_t d = 1;
            while (d <= 128 && 2 + d + d * d != n_shared) ++d;
            if (!shared || d > 128) break;
            for (size_t k = 0; k < d; ++k) put_float(1, shared[2 + k]);
            put_float(2, shared[0]);
            for (size_t k = 0; k < d * d; ++k) put_float(3, shared[2 + d + k]);
            put_float(4, shared[1]);
            return DIST_B200_OK;
        }
        default:
            return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: model has no Shared writer");
    }
    return fail(ctx, DIST_B200_ERR_INVALID, "wire_encode_shared: wrong number of Shared values for the model");
}

}  // namespace distb200
