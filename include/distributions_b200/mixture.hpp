// distributions_b200/mixture.hpp -- host-side C++ mirror of the reference's Shared / Group / Mixture
// interface for the mixture-scoring hot path, on top of the C-ABI (dist_b200.h).
//
// What is mirrored (paths relative to /root/reference):
//   MixtureSlave<Model, DataScorer, ValueScorer>            include/distributions/mixture.hpp:340-450
//     groups(), init, add_group, remove_group, add_value, remove_value, score_value (ACCUMULATES into
//     the caller's buffer), score_value_group                (same names, argument meaning, order)
//   Model::Shared / Model::Group {init, add_value, remove_value}
//     NormalInverseChiSq  models/nich.hpp:52-165      GammaPoisson   models/gp.hpp:52-135
//     BetaBernoulli       models/bb.hpp:52-122        DirichletDiscrete<max_dim>  models/dd.hpp:55-149
//     DirichletProcessDiscrete  models/dpd.hpp:55-215 (fixed value set)    NormalInverseWishart<dim>  models/niw.hpp:52-276
//   MixtureIdTracker                                        include/distributions/mixture.hpp:460-521
//   Clustering<int>::PitmanYor::Mixture (CachedMixture over MixtureDriver)
//                                                            clustering.hpp:126-234, mixture.hpp:48-163
//     counts(), empty_groupids(), sample_size(), init, add_value / remove_value (return whether a group
//     was added / removed), score_value (OVERWRITES the caller's buffer)
// What is new: Mixture::score_values / CrossCat::score_sample_values -- the batched entry that scores
// N rows against frozen statistics and samples a group per row (SURVEY.md §3.3); Mixture::score_logp_values /
// CrossCat::score_logp_values -- the log-likelihood of each row under the mixture; Mixture::sample_values /
// CrossCat::sample_values -- batched Group::sample_value, one posterior-predictive draw per row on the device
// (Sampler::init + Sampler::eval with fresh parameters per value), seeded explicitly instead of through rng_t.
//
// Group statistics live and mutate on the host exactly as in the reference (integer / float
// bookkeeping, SURVEY §8 a20); every score -- per value or batched -- is computed by the sm_100a
// kernels behind the C-ABI.  There is no CPU scoring path here: a failed C-ABI call throws
// std::runtime_error (the reference's DIST_THROW_ON_ERROR behaviour, common.hpp:49-67).
// Not mirrored (off the path): the per-group Sampler (one parameter draw shared by many values), protobuf,
// Group::merge, gp log_prod.
#pragma once

#include <dist_b200.h>

#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <utility>
#include <vector>

namespace distributions_b200 {

// borrowed (pointer, size) view, the reference's AlignedFloats (vector.hpp:63-90) without the
// 32-byte alignment requirement
struct Floats {
    float * ptr;
    size_t n;
    Floats(float * p, size_t size) : ptr(p), n(size) {}
    Floats(std::vector<float> & v) : ptr(v.data()), n(v.size()) {}  // NOLINT(runtime/explicit)
    float * data() { return ptr; }
    size_t size() const { return n; }
    float & operator[](size_t i) { return ptr[i]; }
};

namespace detail {
// value type as it travels in a column (dist_b200_model): bool -> uint8
template <class V> struct WireValue { typedef V type; };
template <> struct WireValue<bool> { typedef uint8_t type; };
}  // namespace detail

struct rng_t {};  // scoring never draws (doc/overview.rst:213-220) and sample_values takes a seed; kept so signatures match

class Context {
  public:
    explicit Context(int device = 0) {
        if (dist_b200_ctx_create(device, &ctx_) != DIST_B200_OK)
            throw std::runtime_error("dist_b200_ctx_create failed: no usable CUDA device (there is no CPU fallback)");
    }
    ~Context() { dist_b200_ctx_destroy(ctx_); }
    Context(const Context &) = delete;
    Context & operator=(const Context &) = delete;
    dist_b200_ctx * get() const { return ctx_; }
    void check(int rc, const char * what) const {
        if (rc != DIST_B200_OK)
            throw std::runtime_error(std::string(what) + ": " + dist_b200_last_error(ctx_));
    }
    // page-lock a caller-owned array once (e.g. the std::vector<Value> a sampler keeps its column in): every later
    // host-buffer call on it is zero-copy.  Unregister before the storage is freed or reallocated.
    template <class T>
    void host_register(std::vector<T> & v) const {
        if (!v.empty()) check(dist_b200_host_register(ctx_, v.data(), v.size() * sizeof(T)), "host_register");
    }
    template <class T>
    void host_unregister(std::vector<T> & v) const {
        if (!v.empty()) check(dist_b200_host_unregister(ctx_, v.data()), "host_unregister");
    }

  private:
    dist_b200_ctx * ctx_ = nullptr;
};

// ---------------------------------------------------------------------------------------------
// component models: Shared, Group and how a group list is uploaded

struct NormalInverseChiSq {
    typedef float Value;
    enum { model_id = DIST_B200_NICH };
    struct Shared {
        float mu, kappa, sigmasq, nu;
        static Shared EXAMPLE() { return Shared{0.f, 1.f, 1.f, 1.f}; }  // nich.hpp:87-94
    };
    struct Group {
        int32_t count;
        float mean;
        float count_times_variance;
        void init(const Shared &, rng_t &) { count = 0; mean = 0.f; count_times_variance = 0.f; }
        void add_value(const Shared &, const Value & value, rng_t &) {  // nich.hpp:125-133
            ++count;
            float delta = value - mean;
            mean += delta / count;
            count_times_variance += delta * (value - mean);
        }
        void remove_value(const Shared &, const Value & value, rng_t &) {  // nich.hpp:146-165
            float total = mean * count;
            float delta = value - mean;
            --count;
            mean = (count == 0) ? 0.f : (total - value) / count;
            if (count <= 1) count_times_variance = 0.f;
            else count_times_variance -= delta * (value - mean);
        }
    };
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size();
        std::vector<int32_t> count(G);
        std::vector<float> mean(G), ctv(G);
        for (size_t g = 0; g < G; ++g) {
            count[g] = groups[g].count; mean[g] = groups[g].mean; ctv[g] = groups[g].count_times_variance;
        }
        const float sh[4] = {s.mu, s.kappa, s.sigmasq, s.nu};
        return dist_b200_nich_update_all(f, sh, static_cast<int>(G), count.data(), mean.data(), ctv.data(), nullptr);
    }
    // arrays as dist_b200_feature_download_stats returns them: count | mean | count_times_variance
    static void load_groups(const unsigned char * raw, const Shared &, std::vector<Group> & groups) {
        const size_t G = groups.size();
        const int32_t * c = reinterpret_cast<const int32_t *>(raw);
        const float * m = reinterpret_cast<const float *>(raw + 4 * G);
        const float * v = reinterpret_cast<const float *>(raw + 8 * G);
        for (size_t g = 0; g < G; ++g) { groups[g].count = c[g]; groups[g].mean = m[g]; groups[g].count_times_variance = v[g]; }
    }
    static size_t stats_bytes(const Shared &, size_t G) { return 12 * G; }
    static void pack_shared(const Shared & s, std::vector<float> & out) {  // score_data_grid layout
        out.push_back(s.mu); out.push_back(s.kappa); out.push_back(s.sigmasq); out.push_back(s.nu);
    }
    static int update_group(dist_b200_feature * f, const Shared &, size_t groupid, const Group & g) {
        struct { int32_t count; float mean; float ctv; } st = {g.count, g.mean, g.count_times_variance};
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), &st, nullptr);
    }
};

struct GammaPoisson {
    typedef uint32_t Value;
    enum { model_id = DIST_B200_GP };
    struct Shared {
        float alpha, inv_beta;
        static Shared EXAMPLE() { return Shared{1.f, 1.f}; }  // gp.hpp:75-80
    };
    struct Group {
        uint32_t count;
        uint32_t sum;
        void init(const Shared &, rng_t &) { count = 0; sum = 0; }
        void add_value(const Shared &, const Value & value, rng_t &) { ++count; sum += value; }     // gp.hpp:109-116
        void remove_value(const Shared &, const Value & value, rng_t &) { --count; sum -= value; }  // gp.hpp:128-135
    };
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size();
        std::vector<uint32_t> count(G), sum(G);
        for (size_t g = 0; g < G; ++g) { count[g] = groups[g].count; sum[g] = groups[g].sum; }
        const float sh[2] = {s.alpha, s.inv_beta};
        return dist_b200_gp_update_all(f, sh, static_cast<int>(G), count.data(), sum.data(), nullptr);
    }
    static void load_groups(const unsigned char * raw, const Shared &, std::vector<Group> & groups) {  // count | sum
        const size_t G = groups.size();
        const uint32_t * c = reinterpret_cast<const uint32_t *>(raw);
        for (size_t g = 0; g < G; ++g) { groups[g].count = c[g]; groups[g].sum = c[G + g]; }
    }
    static size_t stats_bytes(const Shared &, size_t G) { return 8 * G; }
    static void pack_shared(const Shared & s, std::vector<float> & out) { out.push_back(s.alpha); out.push_back(s.inv_beta); }
    static int update_group(dist_b200_feature * f, const Shared &, size_t groupid, const Group & g) {
        const uint32_t st[2] = {g.count, g.sum};
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), st, nullptr);
    }
};

struct BetaNegativeBinomial {
    typedef uint32_t Value;
    enum { model_id = DIST_B200_BNB };
    struct Shared {
        float alpha, beta;
        uint32_t r;
        static Shared EXAMPLE() { return Shared{1.f, 1.f, 1u}; }  // bnb.hpp:79-85
    };
    struct Group {
        uint32_t count;
        uint32_t sum;
        void init(const Shared &, rng_t &) { count = 0; sum = 0; }
        void add_value(const Shared &, const Value & value, rng_t &) { ++count; sum += value; }     // bnb.hpp:107-113
        void remove_value(const Shared &, const Value & value, rng_t &) { --count; sum -= value; }  // bnb.hpp:124-130
    };
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size();
        std::vector<uint32_t> count(G), sum(G);
        for (size_t g = 0; g < G; ++g) { count[g] = groups[g].count; sum[g] = groups[g].sum; }
        const float sh[2] = {s.alpha, s.beta};
        return dist_b200_bnb_update_all(f, sh, s.r, static_cast<int>(G), count.data(), sum.data(), nullptr);
    }
    static void load_groups(const unsigned char * raw, const Shared &, std::vector<Group> & groups) {  // count | sum
        const size_t G = groups.size();
        const uint32_t * c = reinterpret_cast<const uint32_t *>(raw);
        for (size_t g = 0; g < G; ++g) { groups[g].count = c[g]; groups[g].sum = c[G + g]; }
    }
    static size_t stats_bytes(const Shared &, size_t G) { return 8 * G; }
    static void pack_shared(const Shared & s, std::vector<float> & out) { out.push_back(s.alpha); out.push_back(s.beta); }
    static int update_group(dist_b200_feature * f, const Shared &, size_t groupid, const Group & g) {
        const uint32_t st[2] = {g.count, g.sum};
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), st, nullptr);
    }
};

struct BetaBernoulli {
    typedef bool Value;
    enum { model_id = DIST_B200_BB };
    struct Shared {
        float alpha, beta;
        static Shared EXAMPLE() { return Shared{0.5f, 2.f}; }  // bb.hpp:70-75
    };
    struct Group {
        int32_t heads, tails;
        void init(const Shared &, rng_t &) { heads = 0; tails = 0; }
        void add_value(const Shared &, const Value & value, rng_t &) { (value ? heads : tails) += 1; }     // bb.hpp:102-107
        void remove_value(const Shared &, const Value & value, rng_t &) { (value ? heads : tails) -= 1; }  // bb.hpp:117-122
    };
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size();
        std::vector<int32_t> h(G), t(G);
        for (size_t g = 0; g < G; ++g) { h[g] = groups[g].heads; t[g] = groups[g].tails; }
        const float sh[2] = {s.alpha, s.beta};
        return dist_b200_bb_update_all(f, sh, static_cast<int>(G), h.data(), t.data(), nullptr);
    }
    static void load_groups(const unsigned char * raw, const Shared &, std::vector<Group> & groups) {  // heads | tails
        const size_t G = groups.size();
        const int32_t * c = reinterpret_cast<const int32_t *>(raw);
        for (size_t g = 0; g < G; ++g) { groups[g].heads = c[g]; groups[g].tails = c[G + g]; }
    }
    static size_t stats_bytes(const Shared &, size_t G) { return 8 * G; }
    static void pack_shared(const Shared & s, std::vector<float> & out) { out.push_back(s.alpha); out.push_back(s.beta); }
    static int update_group(dist_b200_feature * f, const Shared &, size_t groupid, const Group & g) {
        const int32_t st[2] = {g.heads, g.tails};
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), st, nullptr);
    }
};

template <int max_dim_>
struct DirichletDiscrete {
    typedef int Value;
    enum { model_id = DIST_B200_DD, max_dim = max_dim_ };
    struct Shared {
        int dim;
        float alphas[max_dim_];
        static Shared EXAMPLE() {  // dd.hpp:78-85
            Shared s;
            s.dim = max_dim_;
            for (int i = 0; i < max_dim_; ++i) s.alphas[i] = 0.5f;
            return s;
        }
    };
    struct Group {
        int dim;
        int count_sum;
        int counts[max_dim_];
        void init(const Shared & shared, rng_t &) {
            dim = shared.dim;
            count_sum = 0;
            for (int v = 0; v < dim; ++v) counts[v] = 0;
        }
        void add_value(const Shared &, const Value & value, rng_t &) { count_sum += 1; counts[value] += 1; }     // dd.hpp:123-130
        void remove_value(const Shared &, const Value & value, rng_t &) { count_sum -= 1; counts[value] -= 1; }  // dd.hpp:142-149
    };
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size();
        std::vector<int32_t> counts(G * s.dim);
        for (size_t g = 0; g < G; ++g)
            for (int v = 0; v < s.dim; ++v) counts[g * s.dim + v] = groups[g].counts[v];
        return dist_b200_dd_update_all(f, s.dim, s.alphas, static_cast<int>(G), counts.data(), nullptr);
    }
    static void load_groups(const unsigned char * raw, const Shared & s, std::vector<Group> & groups) {  // counts[G][dim]
        const int32_t * c = reinterpret_cast<const int32_t *>(raw);
        for (size_t g = 0; g < groups.size(); ++g) {
            groups[g].count_sum = 0;
            for (int v = 0; v < s.dim; ++v) { groups[g].counts[v] = c[g * s.dim + v]; groups[g].count_sum += c[g * s.dim + v]; }
        }
    }
    static size_t stats_bytes(const Shared & s, size_t G) { return 4 * G * s.dim; }
    static void pack_shared(const Shared & s, std::vector<float> & out) {
        for (int v = 0; v < s.dim; ++v) out.push_back(s.alphas[v]);
    }
    static int update_group(dist_b200_feature * f, const Shared &, size_t groupid, const Group & g) {
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), g.counts, nullptr);
    }
};

// DirichletProcessDiscrete (models/dpd.hpp:55-215) over a FIXED set of known values: Shared carries values / betas /
// beta0 as Shared::protobuf_load leaves them (dpd.hpp:104-125); the Hierarchical-DP part that invents values
// (Shared::add_value / realize, dpd.hpp:66-100) is off the scoring path -- change the value set with a new init().
// Group = SparseCounter<Value, count_t> (dpd.hpp:157-158); unknown values are an error as in dpd.hpp:193.
struct DirichletProcessDiscrete {
    typedef uint32_t Value;
    enum { model_id = DIST_B200_DPD };
    static constexpr Value OTHER() { return 0xFFFFFFFFu; }  // dpd.hpp:55
    struct Shared {
        float gamma, alpha, beta0;
        std::vector<Value> values;
        std::vector<float> betas;
        static Shared EXAMPLE() {  // dpd.hpp:141-152: dim 100, betas 1 / dim, beta0 = 0
            Shared s;
            s.gamma = 1.f; s.alpha = 0.5f; s.beta0 = 0.f;
            for (Value v = 0; v < 100; ++v) { s.values.push_back(v); s.betas.push_back(0.01f); }
            return s;
        }
        int index(Value v) const {
            for (size_t i = 0; i < values.size(); ++i) if (values[i] == v) return static_cast<int>(i);
            return -1;
        }
    };
    struct Group {
        std::unordered_map<Value, int32_t> counts;
        void init(const Shared &, rng_t &) { counts.clear(); }
        void add_value(const Shared & shared, const Value & value, rng_t &) {  // dpd.hpp:188-196
            if (value == OTHER() || shared.index(value) < 0) throw std::runtime_error("dpd: unknown value");
            counts[value] += 1;
        }
        void remove_value(const Shared & shared, const Value & value, rng_t &) {  // dpd.hpp:207-215
            if (value == OTHER() || shared.index(value) < 0) throw std::runtime_error("dpd: unknown value");
            if (--counts[value] == 0) counts.erase(value);
        }
        void dense(const Shared & shared, int32_t * row) const {
            for (size_t v = 0; v < shared.values.size(); ++v) row[v] = 0;
            for (const auto & kv : counts) row[shared.index(kv.first)] = kv.second;
        }
    };
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size(), V = s.values.size();
        std::vector<int32_t> counts(G * V);
        for (size_t g = 0; g < G; ++g) groups[g].dense(s, counts.data() + g * V);
        return dist_b200_dpd_update_all(f, s.alpha, s.beta0, static_cast<int>(V), s.values.data(), s.betas.data(),
                                        static_cast<int>(G), counts.data(), nullptr);
    }
    static void load_groups(const unsigned char * raw, const Shared & s, std::vector<Group> & groups) {  // counts[G][V]
        const int32_t * c = reinterpret_cast<const int32_t *>(raw);
        const size_t V = s.values.size();
        for (size_t g = 0; g < groups.size(); ++g) {
            groups[g].counts.clear();
            for (size_t v = 0; v < V; ++v) if (c[g * V + v]) groups[g].counts[s.values[v]] = c[g * V + v];
        }
    }
    static size_t stats_bytes(const Shared & s, size_t G) { return 4 * G * s.values.size(); }
    static void pack_shared(const Shared & s, std::vector<float> & out) { out.push_back(s.alpha); }
    static int update_group(dist_b200_feature * f, const Shared & s, size_t groupid, const Group & g) {
        std::vector<int32_t> row(s.values.size());
        g.dense(s, row.data());
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), row.data(), nullptr);
    }
};

// NormalInverseWishart<dim> (models/niw.hpp:52-276).  The reference has no NIW Mixture typedef; Mixture<NormalInverseWishart>
// is the batched form of looping Group::score_value over the groups (mixture.hpp:321-337 semantics).  Group statistics
// are the reference's {count, sum_x, sum_xxT} (niw.hpp:187-190) with its rank-1 updates (niw.hpp:247-276).
template <int dim_>
struct NormalInverseWishart {
    enum { model_id = DIST_B200_NIW, dim = dim_ };
    struct Value { float x[dim_]; };
    struct Shared {
        float mu[dim_];
        float kappa;
        float psi[dim_ * dim_];
        float nu;
        static Shared EXAMPLE() {  // niw.hpp:160-170
            Shared s;
            for (int i = 0; i < dim_; ++i) { s.mu[i] = 0.f; for (int j = 0; j < dim_; ++j) s.psi[i * dim_ + j] = i == j ? 1.f : 0.f; }
            s.kappa = 1.f;
            s.nu = dim_ + 1.f;
            return s;
        }
    };
    struct Group {  // also the packed layout dist_b200_feature_update_group takes for niw
        int32_t count;
        float sum_x[dim_];
        float sum_xxT[dim_ * dim_];
        void init(const Shared &, rng_t &) {
            count = 0;
            for (int i = 0; i < dim_; ++i) sum_x[i] = 0.f;
            for (int i = 0; i < dim_ * dim_; ++i) sum_xxT[i] = 0.f;
        }
        void add_value(const Shared &, const Value & v, rng_t &) {  // niw.hpp:247-255
            ++count;
            for (int i = 0; i < dim_; ++i) { sum_x[i] += v.x[i]; for (int j = 0; j < dim_; ++j) sum_xxT[i * dim_ + j] += v.x[i] * v.x[j]; }
        }
        void remove_value(const Shared &, const Value & v, rng_t &) {  // niw.hpp:267-276
            --count;
            for (int i = 0; i < dim_; ++i) { sum_x[i] -= v.x[i]; for (int j = 0; j < dim_; ++j) sum_xxT[i * dim_ + j] -= v.x[i] * v.x[j]; }
        }
    };
    static_assert(sizeof(Group) == 4 + 4 * dim_ + 4 * dim_ * dim_, "Group must be packed: it is passed to update_group as is");
    static int update_all(dist_b200_feature * f, const Shared & s, const std::vector<Group> & groups) {
        const size_t G = groups.size();
        std::vector<int32_t> count(G);
        std::vector<float> sx(G * dim_), sxx(G * dim_ * dim_);
        for (size_t g = 0; g < G; ++g) {
            count[g] = groups[g].count;
            for (int i = 0; i < dim_; ++i) sx[g * dim_ + i] = groups[g].sum_x[i];
            for (int i = 0; i < dim_ * dim_; ++i) sxx[g * dim_ * dim_ + i] = groups[g].sum_xxT[i];
        }
        return dist_b200_niw_update_all(f, dim_, s.mu, s.kappa, s.psi, s.nu, static_cast<int>(G), count.data(), sx.data(), sxx.data(), nullptr);
    }
    static int update_group(dist_b200_feature * f, const Shared &, size_t groupid, const Group & g) {
        return dist_b200_feature_update_group(f, static_cast<int>(groupid), &g, nullptr);
    }
    static void pack_shared(const Shared & s, std::vector<float> & out) {  // score_data_grid layout: kappa, nu, mu[d], psi[d][d]
        out.push_back(s.kappa);
        out.push_back(s.nu);
        out.insert(out.end(), s.mu, s.mu + dim_);
        out.insert(out.end(), s.psi, s.psi + dim_ * dim_);
    }
    // device-resident statistics: count[G] | sum_x[G][d] | sum_xxT[G][d][d]
    static size_t stats_bytes(const Shared &, size_t G) { return 4 * G * (1 + dim_ + dim_ * dim_); }
    static void load_groups(const unsigned char * raw, const Shared &, std::vector<Group> & groups) {
        const size_t G = groups.size();
        const int32_t * cnt = reinterpret_cast<const int32_t *>(raw);
        const float * sx = reinterpret_cast<const float *>(raw) + G;
        const float * sxx = sx + G * dim_;
        for (size_t g = 0; g < G; ++g) {
            groups[g].count = cnt[g];
            for (int i = 0; i < dim_; ++i) groups[g].sum_x[i] = sx[g * dim_ + i];
            for (int i = 0; i < dim_ * dim_; ++i) groups[g].sum_xxT[i] = sxx[g * dim_ * dim_ + i];
        }
    }
};
// ---------------------------------------------------------------------------------------------
// MixtureIdTracker (mixture.hpp:460-521): packed (contiguous; they move under remove_group's swap-with-last) <-> global
// (fixed, never reused) group ids
struct MixtureIdTracker {
    typedef uint32_t Id;
    void init(size_t group_count = 0) {
        packed_to_global_.clear();
        global_to_packed_.clear();
        global_size_ = 0;
        for (size_t i = 0; i < group_count; ++i) add_group();
    }
    void add_group() {
        const Id packed = static_cast<Id>(packed_to_global_.size()), global = static_cast<Id>(global_size_++);
        packed_to_global_.push_back(global);
        global_to_packed_[global] = packed;
    }
    void remove_group(Id packed) {
        if (packed >= packed_size()) throw std::runtime_error("bad packed id");
        global_to_packed_.erase(packed_to_global_[packed]);
        const Id last = packed_to_global_.back();
        packed_to_global_.pop_back();
        if (packed != packed_to_global_.size()) {  // the last group moved into the hole
            packed_to_global_[packed] = last;
            global_to_packed_[last] = packed;
        }
    }
    Id packed_to_global(Id packed) const {
        if (packed >= packed_size()) throw std::runtime_error("bad packed id");
        return packed_to_global_[packed];
    }
    Id global_to_packed(Id global) const {
        auto i = global_to_packed_.find(global);
        if (i == global_to_packed_.end()) throw std::runtime_error("stale global id");
        return i->second;
    }
    size_t packed_size() const { return packed_to_global_.size(); }
    size_t global_size() const { return global_size_; }
    // NEW: follow dist_b200_regroup_batch.  remap[p] = new packed id of packed group p or -1 (dropped: its global id is
    // retired); survivors keep their global ids and their order, and n_empty fresh groups get new global ids at the end.
    void regroup(const std::vector<int32_t> & remap, size_t n_empty) {
        if (remap.size() != packed_size()) throw std::runtime_error("regroup: remap size != packed size");
        std::vector<Id> survivors;
        for (size_t p = 0; p < remap.size(); ++p) {
            if (remap[p] >= 0) survivors.push_back(packed_to_global_[p]);
            else global_to_packed_.erase(packed_to_global_[p]);
        }
        packed_to_global_ = survivors;
        for (size_t p = 0; p < survivors.size(); ++p) global_to_packed_[survivors[p]] = static_cast<Id>(p);
        for (size_t i = 0; i < n_empty; ++i) add_group();
    }

  private:
    std::vector<Id> packed_to_global_;
    std::unordered_map<Id, Id> global_to_packed_;
    size_t global_size_ = 0;
};

// ---------------------------------------------------------------------------------------------
// Mixture: MixtureSlave with the device-side value scorer

template <class Model>
class Mixture {
  public:
    typedef typename Model::Value Value;
    typedef typename Model::Shared Shared;
    typedef typename Model::Group Group;

    explicit Mixture(std::shared_ptr<Context> ctx) : ctx_(std::move(ctx)) {
        ctx_->check(dist_b200_feature_create(ctx_->get(), Model::model_id, &f_), "feature_create");
    }
    ~Mixture() { dist_b200_feature_destroy(f_); }
    Mixture(const Mixture &) = delete;
    Mixture & operator=(const Mixture &) = delete;

    std::vector<Group> & groups() { return groups_; }
    const std::vector<Group> & groups() const { return groups_; }
    Group & groups(size_t i) { return groups_[i]; }
    const Group & groups(size_t i) const { return groups_[i]; }
    const dist_b200_feature * feature() const { return f_; }
    dist_b200_feature * feature() { return f_; }  // for dist_b200_regroup_batch over the features of a kind

    // mixture.hpp:354-359: value_scorer_.resize + update_all
    void init(const Shared & shared, rng_t &) {
        ctx_->check(Model::update_all(f_, shared, groups_), "update_all");
    }
    // mixture.hpp:361-369
    void add_group(const Shared & shared, rng_t & rng) {
        groups_.emplace_back();
        groups_.back().init(shared, rng);
        ctx_->check(dist_b200_feature_add_group(f_, nullptr), "add_group");
    }
    // mixture.hpp:371-375: packed_remove = swap with last (vector.hpp:47-51)
    void remove_group(const Shared &, size_t groupid) {
        groups_[groupid] = std::move(groups_.back());
        groups_.pop_back();
        ctx_->check(dist_b200_feature_remove_group(f_, static_cast<int>(groupid), nullptr), "remove_group");
    }
    // mixture.hpp:377-398
    void add_value(const Shared & shared, size_t groupid, const Value & value, rng_t & rng) {
        groups_[groupid].add_value(shared, value, rng);
        ctx_->check(Model::update_group(f_, shared, groupid, groups_[groupid]), "update_group");
    }
    void remove_value(const Shared & shared, size_t groupid, const Value & value, rng_t & rng) {
        groups_[groupid].remove_value(shared, value, rng);
        ctx_->check(Model::update_group(f_, shared, groupid, groups_[groupid]), "update_group");
    }
    // mixture.hpp:416-425: scores_accum[g] += score of `value` under group g
    void score_value(const Shared &, const Value & value, Floats scores_accum, rng_t &) const {
        if (scores_accum.size() != groups_.size()) throw std::runtime_error("score_value: size mismatch");
        const typename detail::WireValue<Value>::type wire = static_cast<typename detail::WireValue<Value>::type>(value);
        ctx_->check(dist_b200_score_value_host(ctx_->get(), f_, &wire, scores_accum.data()), "score_value");
    }
    // mixture.hpp:400-414
    float score_value_group(const Shared & shared, size_t groupid, const Value & value, rng_t & rng) const {
        std::vector<float> tmp(groups_.size(), 0.f);
        score_value(shared, value, Floats(tmp), rng);
        return tmp[groupid];
    }

    // mixture.hpp:427-438: log marginal likelihood of all groups under `shared` / under each of `shareds`,
    // evaluated on the device-resident statistics (fp32 terms of the reference, summed in double).
    // GammaPoisson needs Group::log_prod, which this mirror's Group does not carry: set it first with
    // dist_b200_gp_set_log_prod(feature(), ...).
    float score_data(const Shared & shared, rng_t & rng) const {
        std::vector<Shared> one(1, shared);
        float out = 0.f;
        score_data_grid(one, Floats(&out, 1), rng);
        return out;
    }
    void score_data_grid(const std::vector<Shared> & shareds, Floats scores_out, rng_t &) const {
        if (shareds.size() != scores_out.size()) throw std::runtime_error("score_data_grid: size mismatch");
        if (shareds.empty()) return;
        std::vector<float> packed;
        for (const Shared & s : shareds) Model::pack_shared(s, packed);
        ctx_->check(dist_b200_score_data_grid_host(f_, packed.data(), shareds.size(), packed.size() / shareds.size(),
                                                   scores_out.data()),
                    "score_data_grid");
    }

    // NEW: batched add_value.  values[n] join groups assign[n] (packed ids, negative = skip): one segmented
    // reduction on the device replaces n add_value calls (n cache refreshes); the host Groups are read back
    // so that groups() stays the source of truth for dump / remove_value.  nich statistics come from the
    // pairwise merge (nich.hpp:167-179), ~1e-6 relative from n sequential Welford steps.
    template <class T>
    void add_values(const Shared & shared, const T * values, const int32_t * assign, size_t n) {
        std::vector<typename detail::WireValue<Value>::type> wire(values, values + n);
        dist_b200_feature * feats[1] = {f_};
        const void * cols[1] = {wire.data()};
        ctx_->check(dist_b200_add_rows_batch_host(ctx_->get(), feats, 1, cols, assign, n), "add_values");
        std::vector<unsigned char> raw(Model::stats_bytes(shared, groups_.size()));
        size_t got = 0;
        ctx_->check(dist_b200_feature_download_stats(f_, raw.data(), raw.size(), &got, nullptr), "download_stats");
        if (got != raw.size()) throw std::runtime_error("add_values: statistics size mismatch");
        Model::load_groups(raw.data(), shared, groups_);
    }

    // NEW: follow dist_b200_regroup_batch on feature() (remap[g] = new id of old group g, or -1): the host Groups are
    // reordered the same way, n_empty fresh Groups (Group::init) appended, and all of them re-read from the device, as
    // add_values does.
    void regroup(const Shared & shared, const std::vector<int32_t> & remap, size_t n_empty, rng_t & rng) {
        if (remap.size() != groups_.size()) throw std::runtime_error("regroup: remap size != group count");
        std::vector<Group> kept;
        for (size_t g = 0; g < remap.size(); ++g)
            if (remap[g] >= 0) kept.push_back(std::move(groups_[g]));
        for (size_t i = 0; i < n_empty; ++i) {
            kept.emplace_back();
            kept.back().init(shared, rng);
        }
        groups_ = std::move(kept);
        if (static_cast<size_t>(dist_b200_feature_groups(f_)) != groups_.size())
            throw std::runtime_error("regroup: the device feature holds another group count");
        std::vector<unsigned char> raw(Model::stats_bytes(shared, groups_.size()));
        size_t got = 0;
        ctx_->check(dist_b200_feature_download_stats(f_, raw.data(), raw.size(), &got, nullptr), "download_stats");
        if (got != raw.size()) throw std::runtime_error("regroup: statistics size mismatch");
        Model::load_groups(raw.data(), shared, groups_);
    }

    // NEW: batched score (+ sample).  values[n] are rows of this feature, prior[G] the clustering
    // prior vector (or null), u[n] uniforms in [0,1); assign[n] receives the sampled packed group ids,
    // scores (optional) the [n][G] log scores.  Host buffers.
    template <class T>
    void score_values(const Shared &, const T * values, size_t n, const float * prior, const float * u,
                      int32_t * assign, float * scores = nullptr) const {
        std::vector<typename detail::WireValue<Value>::type> wire(values, values + n);
        const dist_b200_feature * feats[1] = {f_};
        const void * cols[1] = {wire.data()};
        ctx_->check(dist_b200_score_sample_batch_host(ctx_->get(), feats, 1, cols, n, prior, u, assign, scores),
                    "score_values");
    }

    // NEW: row log-likelihood.  logp[n] = log sum_g exp(prior[g] + score_value_group(g, values[n])), computed on the device
    // without the [n][G] scores; with the Pitman-Yor prior vector the log posterior-predictive density of values[n].
    template <class T>
    void score_logp_values(const Shared &, const T * values, size_t n, const float * prior, float * logp) const {
        std::vector<typename detail::WireValue<Value>::type> wire(values, values + n);
        const dist_b200_feature * feats[1] = {f_};
        const void * cols[1] = {wire.data()};
        ctx_->check(dist_b200_score_logp_batch_host(ctx_->get(), feats, 1, cols, n, prior, logp), "score_logp_values");
    }

    // NEW: batched Group::sample_value.  out[n] receives one draw from the posterior predictive of group groupids[n]
    // (fresh parameters per value, as Sampler::init + eval), computed on the device from its statistics.  A draw depends
    // on (seed, row0 + n) and that group only; an id outside [0, G) leaves out[n] as it is.
    void sample_values(const Shared &, const int32_t * groupids, size_t n, uint64_t seed, uint64_t row0, Value * out) const {
        std::vector<typename detail::WireValue<Value>::type> wire(out, out + n);
        const dist_b200_feature * feats[1] = {f_};
        void * cols[1] = {wire.data()};
        ctx_->check(dist_b200_sample_values_batch_host(ctx_->get(), feats, 1, groupids, n, seed, row0, cols), "sample_values");
        for (size_t i = 0; i < n; ++i) out[i] = static_cast<Value>(wire[i]);
    }

  private:
    std::shared_ptr<Context> ctx_;
    dist_b200_feature * f_ = nullptr;
    std::vector<Group> groups_;
};

// ---------------------------------------------------------------------------------------------
namespace detail {
// the batched driver bookkeeping of dist_b200_regroup_batch on host counts: groups of size 0 are dropped, the live
// ones keep their order and n_empty empty groups follow.  Returns remap[g] = new id of old group g, or -1.
inline std::vector<int32_t> regroup_counts(std::vector<int32_t> & counts, size_t n_empty) {
    if (n_empty < 1) throw std::runtime_error("regroup: a mixture keeps at least one empty group");  // mixture.hpp:150
    std::vector<int32_t> remap(counts.size(), -1), kept;
    for (size_t g = 0; g < counts.size(); ++g)
        if (counts[g] > 0) {
            remap[g] = static_cast<int32_t>(kept.size());
            kept.push_back(counts[g]);
        }
    kept.resize(kept.size() + n_empty, 0);
    counts = std::move(kept);
    return remap;
}
}  // namespace detail

// ---------------------------------------------------------------------------------------------
// Clustering<int>::PitmanYor and its Mixture (CachedMixture over MixtureDriver)

struct PitmanYor {
    float alpha;
    float d;

    class Mixture {
      public:
        typedef std::unordered_set<size_t> IdSet;
        explicit Mixture(std::shared_ptr<Context> ctx) : ctx_(std::move(ctx)) {}

        std::vector<int32_t> & counts() { return counts_; }
        const std::vector<int32_t> & counts() const { return counts_; }
        int32_t counts(size_t groupid) const { return counts_[groupid]; }
        const IdSet & empty_groupids() const { return empty_groupids_; }
        size_t sample_size() const { return sample_size_; }

        void init(const PitmanYor &) {  // mixture.hpp:63-75
            empty_groupids_.clear();
            sample_size_ = 0;
            for (size_t i = 0; i < counts_.size(); ++i) {
                sample_size_ += counts_[i];
                if (counts_[i] == 0) empty_groupids_.insert(i);
            }
        }
        bool add_value(const PitmanYor &, size_t groupid, int32_t count = 1) {  // mixture.hpp:77-93
            const bool add_group = (counts_[groupid] == 0);
            counts_[groupid] += count;
            sample_size_ += count;
            if (add_group) {
                empty_groupids_.erase(groupid);
                empty_groupids_.insert(counts_.size());
                counts_.push_back(0);
            }
            return add_group;
        }
        bool remove_value(const PitmanYor &, size_t groupid, int32_t count = 1) {  // mixture.hpp:95-122
            counts_[groupid] -= count;
            sample_size_ -= count;
            const bool remove_group = (counts_[groupid] == 0);
            if (remove_group) {
                const size_t last = counts_.size() - 1;
                if (groupid != last) {
                    counts_[groupid] = counts_.back();
                    if (counts_.back() == 0) {
                        empty_groupids_.erase(last);
                        empty_groupids_.insert(groupid);
                    }
                }
                counts_.pop_back();
            }
            return remove_group;
        }
        // NEW: the batched form of add_value / remove_value's group bookkeeping (dist_b200_regroup_batch on host counts;
        // counts() may first be overwritten with the device's group sizes).  Returns the remap the features follow.
        std::vector<int32_t> regroup(const PitmanYor &, size_t n_empty) {
            std::vector<int32_t> remap = detail::regroup_counts(counts_, n_empty);
            empty_groupids_.clear();
            sample_size_ = 0;
            for (size_t i = 0; i < counts_.size(); ++i) {
                sample_size_ += counts_[i];
                if (counts_[i] == 0) empty_groupids_.insert(i);
            }
            return remap;
        }
        // clustering.hpp:195-208: OVERWRITES scores with the prior vector
        void score_value(const PitmanYor & model, Floats scores) const {
            if (scores.size() != counts_.size()) throw std::runtime_error("score_value: size mismatch");
            ctx_->check(dist_b200_prior_pitman_yor_host(ctx_->get(), model.alpha, model.d, static_cast<int>(counts_.size()),
                                                        counts_.data(), scores.data()),
                        "prior_pitman_yor");
        }

      private:
        std::shared_ptr<Context> ctx_;
        std::vector<int32_t> counts_;
        IdSet empty_groupids_;
        size_t sample_size_ = 0;
    };
};

// ---------------------------------------------------------------------------------------------
// Clustering<int>::LowEntropy and its Mixture (the uncached MixtureDriver, clustering.hpp:245-303)

struct LowEntropy {
    int32_t dataset_size;

    class Mixture {
      public:
        explicit Mixture(std::shared_ptr<Context> ctx) : ctx_(std::move(ctx)) {}
        std::vector<int32_t> & counts() { return counts_; }
        const std::vector<int32_t> & counts() const { return counts_; }
        void init(const LowEntropy &) {}
        // mixture.hpp:77-93 / 95-122: same bookkeeping as the Pitman-Yor driver
        bool add_value(const LowEntropy &, size_t groupid, int32_t count = 1) {
            const bool add_group = (counts_[groupid] == 0);
            counts_[groupid] += count;
            if (add_group) counts_.push_back(0);
            return add_group;
        }
        bool remove_value(const LowEntropy &, size_t groupid, int32_t count = 1) {
            counts_[groupid] -= count;
            const bool remove_group = (counts_[groupid] == 0);
            if (remove_group) {
                counts_[groupid] = counts_.back();
                counts_.pop_back();
            }
            return remove_group;
        }
        // NEW: as PitmanYor::Mixture::regroup
        std::vector<int32_t> regroup(const LowEntropy &, size_t n_empty) { return detail::regroup_counts(counts_, n_empty); }
        // mixture.hpp:123-141: OVERWRITES scores with score_add_value of every group
        void score_value(const LowEntropy & model, Floats scores) const {
            if (scores.size() != counts_.size()) throw std::runtime_error("score_value: size mismatch");
            ctx_->check(dist_b200_prior_low_entropy_host(ctx_->get(), model.dataset_size, static_cast<int>(counts_.size()),
                                                         counts_.data(), scores.data()),
                        "prior_low_entropy");
        }

      private:
        std::shared_ptr<Context> ctx_;
        std::vector<int32_t> counts_;
    };
};

// ---------------------------------------------------------------------------------------------
// One cross-cat kind: a clustering mixture plus feature mixtures sharing its partition
// (examples/mixture/main.py:59-123 in C++), with the batched row step.
class CrossCat {
  public:
    explicit CrossCat(std::shared_ptr<Context> ctx) : ctx_(std::move(ctx)) {}
    void add_feature(const dist_b200_feature * f, const void * column_host) {
        feats_.push_back(f);
        cols_.push_back(column_host);
    }
    // prior -> every feature -> sample, for n rows (the fused path of SURVEY.md §3.3)
    void score_sample_values(size_t n, const float * prior, const float * u, int32_t * assign, float * scores = nullptr) {
        ctx_->check(dist_b200_score_sample_batch_host(ctx_->get(), feats_.data(), static_cast<int>(feats_.size()), cols_.data(), n,
                                                      prior, u, assign, scores),
                    "score_sample_values");
    }

    // logp[n] = log sum_g exp(prior[g] + sum_f score_f(row n; g)) for n rows of the kind's features (conditional densities:
    // the difference of two calls over nested feature lists)
    void score_logp_values(size_t n, const float * prior, float * logp) {
        ctx_->check(dist_b200_score_logp_batch_host(ctx_->get(), feats_.data(), static_cast<int>(feats_.size()), cols_.data(), n, prior,
                                                    logp),
                    "score_logp_values");
    }

    // batched Group::sample_value for every feature of the kind: columns_out[i] (host, the column type of feature i)
    // receives, for every row n with 0 <= assign[n] < G, a posterior-predictive draw of group assign[n]
    void sample_values(size_t n, const int32_t * assign, uint64_t seed, uint64_t row0, void * const * columns_out) {
        ctx_->check(dist_b200_sample_values_batch_host(ctx_->get(), feats_.data(), static_cast<int>(feats_.size()), assign, n, seed,
                                                       row0, columns_out),
                    "sample_values");
    }

  private:
    std::shared_ptr<Context> ctx_;
    std::vector<const dist_b200_feature *> feats_;
    std::vector<const void *> cols_;
};

}  // namespace distributions_b200
