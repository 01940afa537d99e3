// api.cu -- the C-ABI of include/dist_b200.h: contexts, feature (MixtureValueScorer) lifecycle,
// dispatch of the hot-path entry points onto the sm_100a kernels.  No CPU compute path exists here:
// every scoring / sampling call ends in a kernel launch or an error code.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <initializer_list>
#include <new>
#include <numeric>

#include "common.cuh"
#include "ref_tables.inc"

using namespace distb200;

namespace {

cudaStream_t as_stream(void *s) { return static_cast<cudaStream_t>(s); }

int ensure_scratch(dist_b200_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->scratch_bytes) return DIST_B200_OK;
    return grow(ctx, ctx->scratch_dev, ctx->scratch_bytes, std::max<size_t>(bytes + bytes / 4, 1 << 20));
}

int ensure_pinned(dist_b200_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->pinned_bytes) return DIST_B200_OK;
    if (ctx->pinned) {
        DISTB200_CUDA(ctx, cudaDeviceSynchronize());
        DISTB200_CUDA(ctx, cudaFreeHost(ctx->pinned));
        ctx->pinned = nullptr;
        ctx->pinned_bytes = 0;
    }
    const size_t want = std::max<size_t>(bytes + bytes / 4, 1 << 20);
    DISTB200_CUDA(ctx, cudaMallocHost(&ctx->pinned, want));
    ctx->pinned_bytes = want;
    return DIST_B200_OK;
}

// Host arrays staged through the context scratch: region() lays out 256-byte aligned regions, reserve() grows the
// device scratch (and the page-locked mirror ctx->pinned over the first `mirror` bytes, same offsets), put / get copy
// between host arrays and regions, through the mirror when asked.  Every stream it was handed is drained when it leaves
// scope, on every return path: no copy into the caller's buffers or out of the mirror is still queued when an entry
// returns, and the next host entry may overwrite the scratch.
struct Staging {
    dist_b200_ctx *ctx;
    cudaStream_t streams[2];
    int n_streams;
    size_t bytes = 0;
    Staging(dist_b200_ctx *c, cudaStream_t s) : ctx(c), streams{s, s}, n_streams(1) {}
    Staging(dist_b200_ctx *c, cudaStream_t s0, cudaStream_t s1) : ctx(c), streams{s0, s1}, n_streams(2) {}
    ~Staging() {
        for (int i = 0; i < n_streams; ++i) cudaStreamSynchronize(streams[i]);
    }
    size_t region(size_t n) {
        const size_t off = bytes;
        bytes += round_up(n, 256);
        return off;
    }
    int reserve(size_t mirror = 0) {
        if (int rc = ensure_pinned(ctx, mirror)) return rc;
        return ensure_scratch(ctx, bytes + 256);
    }
    template <class T = char>
    T *dev(size_t off) const { return reinterpret_cast<T *>(static_cast<char *>(ctx->scratch_dev) + off); }
    char *pin(size_t off) const { return static_cast<char *>(ctx->pinned) + off; }
    int put(size_t off, const void *host, size_t n, cudaStream_t s, bool via_mirror = false) {
        if (via_mirror) host = std::memcpy(pin(off), host, n);
        DISTB200_CUDA(ctx, cudaMemcpyAsync(dev(off), host, n, cudaMemcpyHostToDevice, s));
        return DIST_B200_OK;
    }
    // via the mirror the bytes land at pin(off): the caller copies them out after drain()
    int get(void *host, size_t off, size_t n, cudaStream_t s, bool via_mirror = false) {
        DISTB200_CUDA(ctx, cudaMemcpyAsync(via_mirror ? pin(off) : host, dev(off), n, cudaMemcpyDeviceToHost, s));
        return DIST_B200_OK;
    }
    int drain() {
        for (int i = 0; i < n_streams; ++i) DISTB200_CUDA(ctx, cudaStreamSynchronize(streams[i]));
        n_streams = 0;  // drained: nothing left for the destructor
        return DIST_B200_OK;
    }
};

// a clustering prior over G host group sizes on `s`: launch(sizes_dev, prior, s) writes prior_dev or, with prior_host,
// the scratch that is copied out to the host array
template <class Launch>
int prior_from_host_sizes(dist_b200_ctx *ctx, int G, const int32_t *group_sizes, float *prior_dev, float *prior_host,
                          cudaStream_t s, Launch launch) {
    Staging stage(ctx, s);
    const size_t sizes_off = stage.region(sizeof(int32_t) * G), out_off = stage.region(sizeof(float) * G);
    int rc;
    if ((rc = stage.reserve()) || (rc = stage.put(sizes_off, group_sizes, sizeof(int32_t) * G, s)) ||
        (rc = launch(stage.dev<const int32_t>(sizes_off), prior_host ? stage.dev<float>(out_off) : prior_dev, s)) ||
        (prior_host && (rc = stage.get(prior_host, out_off, sizeof(float) * G, s))))
        return rc;
    return stage.drain();
}


// per-group floats of the hot layout
size_t group_floats(const dist_b200_feature *f) {
    switch (f->model) {
        case DIST_B200_DD: return static_cast<size_t>(f->dim);
        default: return 4;
    }
}

// floats of one niw record (niw.cu)
size_t niw_rec_floats(int d) { return static_cast<size_t>(niw_padded_dim(d)) * (niw_padded_dim(d) + 1) + 4; }

// device-side raw statistics: number of arrays, 4-byte elements per group of array a, and of all arrays
int stat_arrays(const dist_b200_feature *f) {
    switch (f->model) {
        case DIST_B200_NICH: case DIST_B200_NIW: return 3;
        case DIST_B200_GP: case DIST_B200_BB: case DIST_B200_BNB: return 2;
        default: return 1;
    }
}
size_t stat_elems(const dist_b200_feature *f, int a) {
    const size_t d = static_cast<size_t>(f->dim);
    switch (f->model) {
        case DIST_B200_DD: case DIST_B200_DPD: return d;
        case DIST_B200_NIW: return a == 0 ? 1 : a == 1 ? d : d * d;
        default: return 1;
    }
}
size_t group_words(const dist_b200_feature *f) {
    size_t n = 0;
    for (int a = 0; a < stat_arrays(f); ++a) n += stat_elems(f, a);
    return n;
}
bool stats_resident(const dist_b200_feature *f) { return f->stats[0] != nullptr; }

// (re)allocate the statistics arrays for G groups, keeping the first G groups of the feature when `keep`.  Each model
// keeps its growth slack: pooled and dd as their hot caches, dpd a quarter, niw a quarter + 8 groups.
int reserve_stats(dist_b200_feature *f, int G, bool keep) {
    const int na = stat_arrays(f), need = std::max(G, 1);
    bool fits = need <= f->stats_cap;
    for (int a = 0; a < na; ++a) fits = fits && 4 * stat_elems(f, a) * f->stats_cap <= f->stats_bytes[a];
    if (fits) return DIST_B200_OK;
    int cap;
    if (f->model == DIST_B200_DPD) {
        cap = static_cast<int>(round_up(static_cast<size_t>(need) + need / 4, 8));
    } else if (f->model == DIST_B200_NIW) {
        cap = need + need / 4 + 8;
    } else {
        const size_t c = round_up(static_cast<size_t>(need), 128);
        cap = static_cast<int>(round_up(c + c / 2, 128));
    }
    for (int a = 0; a < na; ++a) {
        const size_t e = 4 * stat_elems(f, a);
        if (int rc = grow(f->ctx, f->stats[a], f->stats_bytes[a], e * cap, keep ? e * std::min(f->G, cap) : 0)) return rc;
    }
    f->stats_cap = cap;
    return DIST_B200_OK;
}

// (re)allocate the hot caches for G groups, keeping the first G groups of the feature when `keep`.  Pooled models and
// dd: params (nich also aux), padded to 128 groups so that the score kernel may stage whole register tiles, and
// zero-filled past the kept part.  dpd: the table, (V + 2) rows of G floats (every caller rebuilds it whole).  niw: the
// records and, at d = 32 and d > 32, the tensor-core images (sized by d).
int ensure_params(dist_b200_feature *f, int G, bool keep) {
    dist_b200_ctx *ctx = f->ctx;
    const size_t need = static_cast<size_t>(std::max(G, 1));
    int rc = DIST_B200_OK;
    if (f->model == DIST_B200_NIW) {
        const size_t rec = sizeof(float) * niw_rec_floats(f->dim), tc = sizeof(float) * niw_tc_floats(static_cast<int>(need));
        if (rec * need > f->niw_bytes)
            rc = grow(ctx, f->niw_buf, f->niw_bytes, rec * need + rec * need / 4, keep ? rec * f->G : 0);
        if (!rc && f->dim == 32 && tc > f->niw_tc_bytes) rc = grow(ctx, f->niw_tc, f->niw_tc_bytes, tc + tc / 4);
        if (!rc && f->dim > 32) {
            const size_t wide = sizeof(float) * niw_tc_wide_floats(static_cast<int>(need), f->dim);
            if (wide > f->niw_tc_bytes) rc = grow(ctx, f->niw_tc, f->niw_tc_bytes, wide + wide / 4);
        }
        return rc;
    }
    if (f->model == DIST_B200_DPD) {  // table rows + OTHER row + shift row
        const size_t row = sizeof(float) * (f->dim + 2);
        if (row * need > f->params_bytes) rc = grow(ctx, f->params, f->params_bytes, row * round_up(need + need / 4, 8));
        f->capacity = static_cast<int>(f->params_bytes / row);
        return rc;
    }
    const size_t gb = sizeof(float) * group_floats(f), cap = round_up(need, 128);
    if (gb * cap > f->params_bytes) {
        const size_t fresh = round_up(cap + cap / 2, 128);
        if ((rc = grow(ctx, f->params, f->params_bytes, gb * fresh, keep ? f->params_bytes : 0, true))) return rc;
        if (f->model == DIST_B200_NICH && (rc = grow(ctx, f->aux, f->aux_bytes, sizeof(float) * fresh, keep ? f->aux_bytes : 0, true)))
            return rc;
    }
    f->capacity = static_cast<int>(f->params_bytes / gb);
    return DIST_B200_OK;
}

// recompute the caches of groups [g0, g0 + n) from the resident statistics.  The prep launchers read group i of their
// inputs from the pointers given and write cache g0 + i.
int rebuild(dist_b200_feature *f, int g0, int n, cudaStream_t s) {
    dist_b200_ctx *ctx = f->ctx;
    auto u32 = [&](int a) { return f->stats[a] + stat_elems(f, a) * g0; };
    auto i32 = [&](int a) { return reinterpret_cast<const int32_t *>(u32(a)); };
    auto f32 = [&](int a) { return reinterpret_cast<const float *>(u32(a)); };
    float4 *params = static_cast<float4 *>(f->params);
    switch (f->model) {
        case DIST_B200_NICH: return launch_nich_prep(ctx, f->shared, f->G, g0, n, i32(0), f32(1), f32(2), params, f->aux, s);
        case DIST_B200_GP:
            f->gp_table_dirty = true;
            f->log_prod_valid = false;
            return launch_gp_prep(ctx, f->shared, g0, n, u32(0), u32(1), params, s);
        case DIST_B200_BNB: return launch_bnb_prep(ctx, f->shared, g0, n, u32(0), u32(1), params, s);
        case DIST_B200_BB: return launch_bb_prep(ctx, f->shared, g0, n, i32(0), i32(1), params, s);
        case DIST_B200_DD:
            return launch_dd_prep(ctx, f->dim, f->alphas_dev, f->alpha_sum, g0, n, i32(0), static_cast<float *>(f->params), s);
        case DIST_B200_DPD: {  // the canonical value-major table (dpd.hpp:471-497), its stride is G
            float *table = static_cast<float *>(f->params);
            if (n == 1 && f->G > 1)
                return launch_dpd_update_group(ctx, f->shared[0], f->shared[1], f->dim, f->alphas_dev, f->G, g0, i32(0), table, s);
            int rc = launch_dpd_prep(ctx, f->shared[0], f->shared[1], f->dim, f->alphas_dev, f->G, i32(0), table, s);
            if (rc || f->G < 1) return rc;
            // + the scratch table_rows.cu re-lays the table out into per call
            return grow(ctx, f->dpd_hot, f->dpd_hot_bytes, sizeof(float) * table_hot_floats(f->dim + 1, f->G));
        }
        case DIST_B200_NIW: {  // records, then the tensor-core images of all groups
            const int d = f->dim;
            int rc = launch_niw_prep(ctx, d, f->alphas_dev, f->shared[0], f->alphas_dev + d, f->shared[1], n, i32(0), f32(1), f32(2),
                                     f->niw_buf + niw_rec_floats(d) * g0, s);
            if (rc == DIST_B200_OK && d == 32 && f->niw_tc && f->G > 0) rc = launch_niw_tc_prep(ctx, f->G, f->niw_buf, f->niw_tc, s);
            if (rc == DIST_B200_OK && d > 32 && f->G > 0) rc = launch_niw_tc_wide_prep(ctx, f->G, d, f->niw_buf, f->niw_tc, s);
            return rc;
        }
        default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "unknown model");
    }
}

bool check_feature(const dist_b200_feature *f, int model) { return f && f->ctx && f->model == model; }

// cache mutations are asynchronous on the caller's stream: mark their completion ...
int mark_ready(dist_b200_feature *f, int rc, cudaStream_t s) {
    if (rc != DIST_B200_OK) return rc;
    DISTB200_CUDA(f->ctx, cudaEventRecord(f->ready, s));
    // the update entries copy from the caller's host arrays asynchronously: drain the stream, so that every update
    // returns with its work complete and the caller may reuse or free those arrays at once
    DISTB200_CUDA(f->ctx, cudaStreamSynchronize(s));
    return DIST_B200_OK;
}
// ... and make a scoring stream wait for them (no-op when it is the same stream)
int wait_ready(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F, cudaStream_t s) {
    for (int f = 0; f < F; ++f)
        if (features[f] && features[f]->ready) DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, features[f]->ready, 0));
    return DIST_B200_OK;
}

}  // namespace

extern "C" {

int dist_b200_abi_version(void) { return DIST_B200_ABI_VERSION; }

int dist_b200_ctx_create(int device, dist_b200_ctx **out) {
    if (!out) return DIST_B200_ERR_INVALID;
    *out = nullptr;
    dist_b200_ctx *ctx = new (std::nothrow) dist_b200_ctx();
    if (!ctx) return DIST_B200_ERR_CUDA;
    ctx->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (e != cudaSuccess) {
        delete ctx;
        return DIST_B200_ERR_CUDA;
    }
    // numerics tables.  fast_log's table is rebuilt the way the reference builds it
    // (special.cc:35-44: log2 of 1 + i / 2^14, float argument); the polynomial / factorial tables are
    // the reference's data (ref_tables.inc, generated by oracle/gen_tables.py).
    const size_t n_log = 1 << 14, n_lg = 33 * kLgammaRowStride, n_nu = 18 * 4, n_lf = 64;
    std::vector<float> host(n_log + n_lg + n_nu + n_lf, 0.f);
    for (size_t i = 0; i < n_log; ++i) {
        const float scaled = static_cast<float>(i) * static_cast<float>(1 << 9);
        const float v = static_cast<float>(1.0 + static_cast<double>(scaled / static_cast<float>(1 << 23)));
        host[i] = log2f(v);
    }
    for (int c = 0; c < 33; ++c)
        for (int k = 0; k < 6; ++k) std::memcpy(&host[n_log + c * kLgammaRowStride + k], &kLgammaCoeff5Bits[c * 6 + k], 4);
    std::memcpy(&host[n_log + n_lg], kLgammaNuCoeff3Bits, sizeof(float) * n_nu);
    std::memcpy(&host[n_log + n_lg + n_nu], kLogFactorialBits, sizeof(float) * n_lf);
    e = cudaMalloc(&ctx->tables_storage, host.size() * sizeof(float));
    if (e == cudaSuccess) e = cudaMemcpy(ctx->tables_storage, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->own_stream2, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ctx->ev, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        if (ctx->tables_storage) cudaFree(ctx->tables_storage);
        delete ctx;
        return DIST_B200_ERR_CUDA;
    }
    ctx->tables.log2_table = ctx->tables_storage;
    ctx->tables.lgamma5 = ctx->tables_storage + n_log;
    ctx->tables.lgamma_nu3 = ctx->tables_storage + n_log + n_lg;
    ctx->tables.log_factorial = ctx->tables_storage + n_log + n_lg + n_nu;
    *out = ctx;
    return DIST_B200_OK;
}

void dist_b200_ctx_destroy(dist_b200_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->tables_storage) cudaFree(ctx->tables_storage);
    if (ctx->scratch_dev) cudaFree(ctx->scratch_dev);
    if (ctx->add_acc) cudaFree(ctx->add_acc);
    if (ctx->add_done) cudaEventDestroy(ctx->add_done);
    if (ctx->regroup_buf) cudaFree(ctx->regroup_buf);
    if (ctx->regroup_k_host) cudaFreeHost(ctx->regroup_k_host);
    if (ctx->regroup_done) cudaEventDestroy(ctx->regroup_done);
    if (ctx->scores_scratch) cudaFree(ctx->scores_scratch);
    if (ctx->missing_scratch) cudaFree(ctx->missing_scratch);
    if (ctx->xpack) cudaFree(ctx->xpack);
    if (ctx->bbt) cudaFree(ctx->bbt);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->own_stream2) cudaStreamDestroy(ctx->own_stream2);
    if (ctx->ev) cudaEventDestroy(ctx->ev);
    delete ctx;
}

int dist_b200_ctx_set_option(dist_b200_ctx *ctx, int option, int value) {
    if (!ctx || option < 0 || option >= DIST_B200_OPT_COUNT_) return DIST_B200_ERR_INVALID;
    ctx->opt[option] = value;
    return DIST_B200_OK;
}

const char *dist_b200_last_error(const dist_b200_ctx *ctx) { return ctx ? ctx->last_error.c_str() : "null context"; }
int dist_b200_sm_count(const dist_b200_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

int dist_b200_feature_create(dist_b200_ctx *ctx, int model, dist_b200_feature **out) {
    if (!ctx || !out) return DIST_B200_ERR_INVALID;
    *out = nullptr;
    if (model < DIST_B200_DD || model > DIST_B200_BNB) return fail(ctx, DIST_B200_ERR_INVALID, "unknown model");
    dist_b200_feature *f = new (std::nothrow) dist_b200_feature();
    if (!f) return fail(ctx, DIST_B200_ERR_CUDA, "out of host memory");
    f->ctx = ctx;
    f->model = model;
    if (cudaEventCreateWithFlags(&f->ready, cudaEventDisableTiming) != cudaSuccess) {
        delete f;
        return fail(ctx, DIST_B200_ERR_CUDA, "cudaEventCreate failed");
    }
    *out = f;
    return DIST_B200_OK;
}

void dist_b200_feature_destroy(dist_b200_feature *f) {
    if (!f) return;
    cudaDeviceSynchronize();
    if (f->params) cudaFree(f->params);
    if (f->aux) cudaFree(f->aux);
    if (f->gp_table) cudaFree(f->gp_table);
    if (f->keys_dev) cudaFree(f->keys_dev);
    if (f->key_rows_dev) cudaFree(f->key_rows_dev);
    if (f->dpd_hot) cudaFree(f->dpd_hot);
    if (f->cdf_buf) cudaFree(f->cdf_buf);
    if (f->niw_buf) cudaFree(f->niw_buf);
    if (f->niw_tc) cudaFree(f->niw_tc);
    if (f->sample_buf) cudaFree(f->sample_buf);
    for (uint32_t *st : f->stats)
        if (st) cudaFree(st);
    if (f->alphas_dev) cudaFree(f->alphas_dev);
    if (f->log_prod_dev) cudaFree(f->log_prod_dev);
    if (f->ready) cudaEventDestroy(f->ready);
    delete f;
}

int dist_b200_feature_model(const dist_b200_feature *f) { return f ? f->model : -1; }
int dist_b200_feature_groups(const dist_b200_feature *f) { return f ? f->G : 0; }

// update_all after the model's validation (f->dim, f->shared and f->alphas set): the Shared vector and the statistics
// arrays (G groups each, in stats order) go straight into the resident buffers, then every cache is rebuilt
static int write_all(dist_b200_feature *f, int G, std::initializer_list<const void *> arrays, void *stream) {
    dist_b200_ctx *ctx = f->ctx;
    cudaStream_t s = as_stream(stream);
    int rc;
    if ((rc = grow(ctx, f->alphas_dev, f->alphas_bytes, sizeof(float) * f->alphas.size())) || (rc = ensure_params(f, G, false)) ||
        (rc = reserve_stats(f, G, false)))
        return rc;
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
    if (!f->alphas.empty())
        DISTB200_CUDA(ctx, cudaMemcpyAsync(f->alphas_dev, f->alphas.data(), sizeof(float) * f->alphas.size(), cudaMemcpyHostToDevice, s));
    int a = 0;
    for (const void *src : arrays) {
        if (G) DISTB200_CUDA(ctx, cudaMemcpyAsync(f->stats[a], src, 4 * stat_elems(f, a) * G, cudaMemcpyHostToDevice, s));
        ++a;
    }
    f->G = G;
    return mark_ready(f, rebuild(f, 0, G, s), s);
}

int dist_b200_nich_update_all(dist_b200_feature *f, const float shared[4], int G, const int32_t *count,
                              const float *mean, const float *ctv, void *stream) {
    if (!check_feature(f, DIST_B200_NICH) || !shared || G < 0 || (G && (!count || !mean || !ctv))) return DIST_B200_ERR_INVALID;
    std::memcpy(f->shared, shared, sizeof(float) * 4);
    return write_all(f, G, {count, mean, ctv}, stream);
}

int dist_b200_gp_update_all(dist_b200_feature *f, const float shared[2], int G, const uint32_t *count,
                            const uint32_t *sum, void *stream) {
    if (!check_feature(f, DIST_B200_GP) || !shared || G < 0 || (G && (!count || !sum))) return DIST_B200_ERR_INVALID;
    f->shared[0] = shared[0];
    f->shared[1] = shared[1];
    return write_all(f, G, {count, sum}, stream);
}

int dist_b200_bnb_update_all(dist_b200_feature *f, const float shared[2], uint32_t r, int G, const uint32_t *count,
                             const uint32_t *sum, void *stream) {
    if (!check_feature(f, DIST_B200_BNB) || !shared || G < 0 || (G && (!count || !sum))) return DIST_B200_ERR_INVALID;
    f->shared[0] = shared[0];
    f->shared[1] = shared[1];
    f->shared[2] = static_cast<float>(r);  // the reference converts r to float wherever it enters (bnb.hpp:59,208)
    return write_all(f, G, {count, sum}, stream);
}

int dist_b200_bb_update_all(dist_b200_feature *f, const float shared[2], int G, const int32_t *heads,
                            const int32_t *tails, void *stream) {
    if (!check_feature(f, DIST_B200_BB) || !shared || G < 0 || (G && (!heads || !tails))) return DIST_B200_ERR_INVALID;
    f->shared[0] = shared[0];
    f->shared[1] = shared[1];
    return write_all(f, G, {heads, tails}, stream);
}

int dist_b200_dd_update_all(dist_b200_feature *f, int dim, const float *alphas, int G, const int32_t *counts,
                            void *stream) {
    if (!check_feature(f, DIST_B200_DD) || dim < 1 || !alphas || G < 0 || (G && !counts)) return DIST_B200_ERR_INVALID;
    if (dim > 256) return fail(f->ctx, DIST_B200_ERR_UNSUPPORTED, "dd: dim > 256");
    f->dim = dim;
    f->alphas.assign(alphas, alphas + dim);
    float alpha_sum = 0;  // dd.hpp:404-407, sequential float sum
    for (int v = 0; v < dim; ++v) alpha_sum += alphas[v];
    f->alpha_sum = alpha_sum;
    return write_all(f, G, {counts}, stream);
}

int dist_b200_dpd_update_all(dist_b200_feature *f, float alpha, float beta0, int V, const uint32_t *keys,
                             const float *betas, int G, const int32_t *counts, void *stream) {
    if (!check_feature(f, DIST_B200_DPD) || V < 1 || !keys || !betas || G < 0 || (G && !counts)) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    // value -> table row: identity when keys are 0..V-1, else sorted keys + binary search on device
    bool dense = true;
    for (int v = 0; v < V; ++v) dense = dense && keys[v] == static_cast<uint32_t>(v);
    if (V != f->dim || !f->keys_dev || !std::equal(keys, keys + V, f->keys.begin()) ) {
        std::vector<int> order(V);
        std::iota(order.begin(), order.end(), 0);
        std::sort(order.begin(), order.end(), [&](int x, int y) { return keys[x] < keys[y]; });
        std::vector<uint32_t> sorted(V);
        for (int i = 0; i < V; ++i) sorted[i] = keys[order[i]];
        for (int i = 1; i < V; ++i)
            if (sorted[i] == sorted[i - 1]) return fail(ctx, DIST_B200_ERR_INVALID, "dpd: duplicate key");
        int rc;
        if ((rc = grow(ctx, f->keys_dev, f->keys_bytes, sizeof(uint32_t) * V)) || (rc = grow(ctx, f->key_rows_dev, f->key_rows_bytes, sizeof(int) * V)))
            return rc;
        cudaStream_t s = as_stream(stream);
        DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
        DISTB200_CUDA(ctx, cudaMemcpyAsync(f->keys_dev, sorted.data(), sizeof(uint32_t) * V, cudaMemcpyHostToDevice, s));
        DISTB200_CUDA(ctx, cudaMemcpyAsync(f->key_rows_dev, order.data(), sizeof(int) * V, cudaMemcpyHostToDevice, s));
        DISTB200_CUDA(ctx, cudaStreamSynchronize(s));  // the host vectors go out of scope
        f->keys.assign(keys, keys + V);
    }
    f->keys_dense = dense;
    f->dim = V;
    f->shared[0] = alpha;
    f->shared[1] = beta0;
    f->alphas.assign(betas, betas + V);
    return write_all(f, G, {counts}, stream);
}

int dist_b200_niw_update_all(dist_b200_feature *f, int d, const float *mu, float kappa, const float *psi,
                             float nu, int G, const int32_t *count, const float *sum_x, const float *sum_xxT,
                             void *stream) {
    if (!check_feature(f, DIST_B200_NIW) || d < 1 || !mu || !psi || G < 0 || (G && (!count || !sum_x || !sum_xxT)))
        return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (d > 128) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "niw: d > 128 (the group prep holds a d x d double Cholesky factor in shared memory)");
    if (!(kappa > 0.f) || !(nu > static_cast<float>(d) - 1.f))
        return fail(ctx, DIST_B200_ERR_INVALID, "niw: need kappa > 0 and nu > d - 1 (niw.hpp:121,132)");
    f->dim = d;
    f->shared[0] = kappa;
    f->shared[1] = nu;
    f->alphas.assign(mu, mu + d);
    f->alphas.insert(f->alphas.end(), psi, psi + static_cast<size_t>(d) * d);
    return write_all(f, G, {count, sum_x, sum_xxT}, stream);
}

// the record of one group is its slice of each statistics array, in update_all's order (dist_b200.h)
int dist_b200_feature_update_group(dist_b200_feature *f, int groupid, const void *stats, void *stream) {
    if (!f || !f->ctx || !stats) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (groupid < 0 || groupid >= f->G) return fail(ctx, DIST_B200_ERR_INVALID, "update_group: bad groupid");
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
    const char *rec = static_cast<const char *>(stats);
    for (int a = 0; a < stat_arrays(f); ++a) {
        const size_t e = stat_elems(f, a);
        DISTB200_CUDA(ctx, cudaMemcpyAsync(f->stats[a] + e * groupid, rec, 4 * e, cudaMemcpyHostToDevice, s));
        rec += 4 * e;
    }
    return mark_ready(f, rebuild(f, groupid, 1, s), s);
}

// a fresh group is Group::init (all-zero statistics) followed by update_group (mixture.hpp:361-369)
int dist_b200_feature_add_group(dist_b200_feature *f, void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (!stats_resident(f)) return fail(ctx, DIST_B200_ERR_STATE, "add_group: call update_all first");
    const int g = f->G;
    int rc;
    if ((rc = ensure_params(f, g + 1, true)) || (rc = reserve_stats(f, g + 1, true))) return rc;
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
    for (int a = 0; a < stat_arrays(f); ++a)
        DISTB200_CUDA(ctx, cudaMemsetAsync(f->stats[a] + stat_elems(f, a) * g, 0, 4 * stat_elems(f, a), s));
    f->G = g + 1;
    // the dpd table's stride is G: it is rebuilt whole (O(V G))
    return mark_ready(f, f->model == DIST_B200_DPD ? rebuild(f, 0, f->G, s) : rebuild(f, g, 1, s), s);
}

// packed_remove: the last group moves into the hole (vector.hpp:47-51)
int dist_b200_feature_remove_group(dist_b200_feature *f, int groupid, void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (groupid < 0 || groupid >= f->G) return fail(ctx, DIST_B200_ERR_INVALID, "remove_group: bad groupid");
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
    const int last = f->G - 1;
    for (int a = 0; a < stat_arrays(f) && groupid != last; ++a) {
        const size_t e = stat_elems(f, a);
        DISTB200_CUDA(ctx, cudaMemcpyAsync(f->stats[a] + e * groupid, f->stats[a] + e * last, 4 * e, cudaMemcpyDeviceToDevice, s));
    }
    f->G = last;
    if (f->model == DIST_B200_DPD) return mark_ready(f, rebuild(f, 0, last, s), s);  // stride G again
    int rc = DIST_B200_OK;
    if (f->model == DIST_B200_NIW) {
        const size_t rec = niw_rec_floats(f->dim);
        if (groupid != last)
            DISTB200_CUDA(ctx, cudaMemcpyAsync(f->niw_buf + rec * groupid, f->niw_buf + rec * last, sizeof(float) * rec, cudaMemcpyDeviceToDevice, s));
        if (f->dim == 32 && f->niw_tc && last > 0) rc = launch_niw_tc_prep(ctx, last, f->niw_buf, f->niw_tc, s);
        if (f->dim > 32 && last > 0) rc = launch_niw_tc_wide_prep(ctx, last, f->dim, f->niw_buf, f->niw_tc, s);
        return mark_ready(f, rc, s);
    }
    const size_t gb = sizeof(float) * group_floats(f);
    char *base = static_cast<char *>(f->params);
    if (groupid != last) DISTB200_CUDA(ctx, cudaMemcpyAsync(base + gb * groupid, base + gb * last, gb, cudaMemcpyDeviceToDevice, s));
    DISTB200_CUDA(ctx, cudaMemsetAsync(base + gb * last, 0, gb, s));
    if (f->aux && groupid != last)
        DISTB200_CUDA(ctx, cudaMemcpyAsync(f->aux + groupid, f->aux + last, sizeof(float), cudaMemcpyDeviceToDevice, s));
    f->gp_table_dirty = true;
    f->log_prod_valid = false;
    return mark_ready(f, rc, s);
}

static bool pooled_model(int model);

// the per-group device arrays regroup_batch moves with their group: the statistics, and the caches a gather keeps
// (pooled and dd params, nich aux, a valid gp log_prod, niw records).  dpd's table is rebuilt instead.
static void regroup_arrays(dist_b200_feature *f, bool log_prod, std::vector<RegroupArray> &out) {
    for (int a = 0; a < stat_arrays(f); ++a) out.push_back({f->stats[a], f->stats[a], stat_elems(f, a)});
    uint32_t *params = static_cast<uint32_t *>(f->params);
    if (pooled_model(f->model) || f->model == DIST_B200_DD) out.push_back({params, params, group_floats(f)});
    if (f->model == DIST_B200_NICH) out.push_back({reinterpret_cast<uint32_t *>(f->aux), reinterpret_cast<uint32_t *>(f->aux), 1});
    if (log_prod) out.push_back({reinterpret_cast<uint32_t *>(f->log_prod_dev), reinterpret_cast<uint32_t *>(f->log_prod_dev), 1});
    if (f->model == DIST_B200_NIW) {
        uint32_t *recs = reinterpret_cast<uint32_t *>(f->niw_buf);
        out.push_back({recs, recs, niw_rec_floats(f->dim)});
    }
}

// one launch per kRegroupBatch arrays
static int regroup_launch(dist_b200_ctx *ctx, const std::vector<RegroupArray> &arrays, int rows, const int32_t *inv,
                          const int32_t *k, cudaStream_t s) {
    RegroupBatch b;
    b.rows = rows;
    b.inv = inv;
    b.k = k;
    for (size_t i0 = 0; i0 < arrays.size(); i0 += kRegroupBatch) {
        b.n = static_cast<int>(std::min<size_t>(kRegroupBatch, arrays.size() - i0));
        for (int i = 0; i < b.n; ++i) b.a[i] = arrays[i0 + i];
        if (int rc = launch_regroup_arrays(ctx, b, s)) return rc;
    }
    return DIST_B200_OK;
}

int dist_b200_regroup_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features, const int32_t *counts_dev,
                            int G, int n_empty, int32_t *assign_dev, size_t n_rows, int32_t *counts_out_dev,
                            int32_t *remap_out_dev, int *G_out, void *stream) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    if (!G_out || G < 0 || n_features < 0 || (n_features && !features) || (G && !counts_dev) || (n_rows && !assign_dev))
        return fail(ctx, DIST_B200_ERR_INVALID, "regroup_batch: null or negative argument");
    if (n_empty < 1 || n_empty > INT32_MAX - G)
        return fail(ctx, DIST_B200_ERR_INVALID, "regroup_batch: need n_empty >= 1 (a mixture always keeps an empty group)");
    for (int i = 0; i < n_features; ++i) {
        const dist_b200_feature *f = features[i];
        if (!f || f->ctx != ctx) return fail(ctx, DIST_B200_ERR_INVALID, "regroup_batch: null feature or one of another context");
        if (!stats_resident(f)) return fail(ctx, DIST_B200_ERR_STATE, "regroup_batch: call update_all first");
        if (f->G != G) return fail(ctx, DIST_B200_ERR_STATE, "regroup_batch: a feature's G differs from the G given");
    }
    cudaStream_t s = as_stream(stream);
    const int rows = G + n_empty;  // K+ <= G: an upper bound of the new G, so the gather needs no readback

    // the source arrays and the layout of the context buffer: remap | inv | K+ | one gathered copy per array
    std::vector<RegroupArray> src;
    std::vector<bool> log_prod(n_features);
    for (int i = 0; i < n_features; ++i) {
        log_prod[i] = features[i]->model == DIST_B200_GP && features[i]->log_prod_valid;
        regroup_arrays(features[i], log_prod[i], src);
    }
    size_t bytes = 0;
    auto region = [&](size_t n) { const size_t off = bytes; bytes += round_up(n, 256); return off; };
    const size_t remap_off = region(sizeof(int32_t) * G), inv_off = region(sizeof(int32_t) * rows), k_off = region(sizeof(int32_t));
    std::vector<size_t> arr_off(src.size());
    for (size_t i = 0; i < src.size(); ++i) arr_off[i] = region(4 * src[i].words * rows);
    int rc;
    if (bytes > ctx->regroup_bytes && (rc = grow(ctx, ctx->regroup_buf, ctx->regroup_bytes, bytes + bytes / 4))) return rc;
    if (!ctx->regroup_k_host) DISTB200_CUDA(ctx, cudaMallocHost(&ctx->regroup_k_host, sizeof(int32_t)));
    if (!ctx->regroup_done) DISTB200_CUDA(ctx, cudaEventCreateWithFlags(&ctx->regroup_done, cudaEventDisableTiming));
    char *buf = static_cast<char *>(ctx->regroup_buf);
    int32_t *remap = remap_out_dev ? remap_out_dev : reinterpret_cast<int32_t *>(buf + remap_off);
    int32_t *inv = reinterpret_cast<int32_t *>(buf + inv_off), *k_dev = reinterpret_cast<int32_t *>(buf + k_off);

    // phase 1, before K+ is known: the remap, the relabel and every gather into the context buffer.  The buffer is
    // ordered behind the last regroup's copy-back by the context's regroup_done event.
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, ctx->regroup_done, 0));
    if ((rc = wait_ready(ctx, features, n_features, s)) ||
        (rc = launch_regroup_remap(ctx, counts_dev, G, n_empty, remap, inv, counts_out_dev, k_dev, s)) ||
        (rc = launch_regroup_relabel(ctx, assign_dev, n_rows, remap, G, s)))
        return rc;
    std::vector<RegroupArray> gather(src);
    for (size_t i = 0; i < src.size(); ++i) gather[i].dst = reinterpret_cast<uint32_t *>(buf + arr_off[i]);
    if ((rc = regroup_launch(ctx, gather, rows, inv, k_dev, s))) return rc;
    // the one host round trip: the new G sets grid sizes and f->G
    DISTB200_CUDA(ctx, cudaMemcpyAsync(ctx->regroup_k_host, k_dev, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    DISTB200_CUDA(ctx, cudaStreamSynchronize(s));
    const int K = *ctx->regroup_k_host, G_new = K + n_empty;

    // phase 2: capacity for G_new (the old contents are in the context buffer, so nothing is kept), then the copy back
    // of rows [0, max(G, G_new)): survivors, zeroed fresh groups, and zeros over the dropped tail
    for (int i = 0; i < n_features; ++i) {
        dist_b200_feature *f = features[i];
        if ((rc = reserve_stats(f, G_new, false)) || (rc = ensure_params(f, G_new, false)) ||
            (log_prod[i] && (rc = grow(ctx, f->log_prod_dev, f->log_prod_bytes, sizeof(float) * f->capacity))))
            return rc;
    }
    std::vector<RegroupArray> back;
    for (int i = 0; i < n_features; ++i) regroup_arrays(features[i], log_prod[i], back);
    for (size_t i = 0; i < back.size(); ++i) back[i].src = reinterpret_cast<const uint32_t *>(buf + arr_off[i]);
    if ((rc = regroup_launch(ctx, back, std::max(G, G_new), nullptr, nullptr, s))) return rc;

    // caches of the fresh groups (dpd: the whole table at the new stride; niw: also the tensor-core images, once)
    for (int i = 0; i < n_features; ++i) {
        dist_b200_feature *f = features[i];
        f->G = G_new;
        rc = f->model == DIST_B200_DPD ? rebuild(f, 0, G_new, s) : rebuild(f, K, n_empty, s);
        if (rc) return rc;
        f->gp_table_dirty = true;
        f->log_prod_valid = log_prod[i];
        DISTB200_CUDA(ctx, cudaEventRecord(f->ready, s));
    }
    DISTB200_CUDA(ctx, cudaEventRecord(ctx->regroup_done, s));
    *G_out = G_new;
    return DIST_B200_OK;
}

// batched Group::add_value over many features of one kind.  Everything is enqueued on `stream`: the
// accumulators live in a dedicated context buffer guarded by an event (not the upload scratch), so the
// call returns without draining the stream; later scoring calls order themselves behind the features'
// `ready` events.
// phase: kRowsBoth = accumulate + merge (single GPU); kRowsAccumulate = accumulate and pack into `xchg`
// ([n_features][4][G] doubles) for an all-reduce; kRowsMerge = merge from the (all-reduced) `xchg`
enum { kRowsBoth = 0, kRowsAccumulate = 1, kRowsMerge = 2 };

static bool pooled_model(int model) {
    return model == DIST_B200_NICH || model == DIST_B200_GP || model == DIST_B200_BB || model == DIST_B200_BNB;
}

// observed (accumulating phases): per feature NULL or a mask (dist_b200.h).  The pooled, count-table and niw kernels skip
// a missing cell themselves (their masked instantiations); pooled batches keep up to kAddBatch features whatever the masks
static int rows_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                      const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, int sign, void *stream,
                      int phase = kRowsBoth, double *xchg = nullptr, const uint32_t *const *observed = nullptr) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    if (n_features < 0 || (n_features && !features) || (phase != kRowsMerge && ((n_features && !columns_dev) || !assign_dev)))
        return fail(ctx, DIST_B200_ERR_INVALID, "add_rows: null argument");
    if (phase != kRowsBoth) {
        if (!xchg) return fail(ctx, DIST_B200_ERR_INVALID, "rows exchange: null exchange buffer");
        for (int i = 0; i < n_features; ++i) {
            const dist_b200_feature *f = features[i];
            if (!f) return fail(ctx, DIST_B200_ERR_INVALID, "rows exchange: null feature");
            if (f->G != features[0]->G) return fail(ctx, DIST_B200_ERR_INVALID, "rows exchange: features disagree on the number of groups");
        }
    }
    cudaStream_t s = as_stream(stream);
    size_t acc_need = 0, table_tmp = 0, niw_tmp = 0;  // pooled accumulators | (exchange) one count table of delta counts | niw work area
    int n_pooled = 0;
    for (int i = 0; i < n_features; ++i) {
        dist_b200_feature *f = features[i];
        if (!f || f->ctx != ctx || (phase != kRowsMerge && !columns_dev[i])) return fail(ctx, DIST_B200_ERR_INVALID, "add_rows: bad feature / column");
        if (f->G < 1 || !stats_resident(f)) return fail(ctx, DIST_B200_ERR_STATE, "add_rows: call update_all first");
        if (pooled_model(f->model)) {
            acc_need = std::max(acc_need, add_rows_acc_bytes(f->G) * std::min(n_features, kAddBatch));
            ++n_pooled;
        } else if (f->model == DIST_B200_NIW) {
            if (phase != kRowsMerge) niw_tmp = std::max(niw_tmp, niw_add_rows_bytes(f->G, f->dim, n_rows));
        } else if (phase == kRowsAccumulate) {
            table_tmp = std::max(table_tmp, round_up(sizeof(int32_t) * static_cast<size_t>(f->G) * f->dim, 256));
        }
    }
    acc_need = round_up(acc_need, 256);
    const size_t pooled_bytes = acc_need;
    acc_need += table_tmp + niw_tmp;
    // exchange layout: the pooled features' [4][G] blocks first (list order), then the count tables (list order)
    size_t table_off = phase == kRowsBoth ? 0 : static_cast<size_t>(n_pooled) * 4 * features[0]->G;
    int rc = grow(ctx, ctx->add_acc, ctx->add_acc_bytes, acc_need);
    if (rc) return rc;
    if (!ctx->add_done) DISTB200_CUDA(ctx, cudaEventCreateWithFlags(&ctx->add_done, cudaEventDisableTiming));
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, ctx->add_done, 0));  // the previous batch may have run on another stream
    if ((rc = wait_ready(ctx, features, n_features, s))) return rc;

    AddBatch b{};
    b.sign = sign;
    b.N = n_rows;
    b.assign = assign_dev;
    b.acc = static_cast<char *>(ctx->add_acc);
    AddMasks bm{};  // the pending pooled batch's observed masks (bm.m[k] for b.d[k])
    auto mask_of = [&](int i) -> const uint32_t * { return observed && phase != kRowsMerge ? observed[i] : nullptr; };
    int flushed = 0;  // pooled features already processed = index of b.d[0] in the exchange buffer
    auto flush = [&]() -> int {
        if (b.n == 0) return DIST_B200_OK;
        b.acc_stride = add_rows_acc_bytes(b.G);
        b.xchg = phase == kRowsMerge ? xchg : nullptr;
        b.xchg_first = flushed;
        int r = DIST_B200_OK;
        if (phase != kRowsMerge) r = launch_add_rows_pooled(ctx, b, s, &bm);
        if (!r && phase == kRowsAccumulate) r = launch_pack_accumulators(ctx, b, xchg, s);
        if (!r && phase != kRowsAccumulate) r = launch_merge_prep_batch(ctx, b, s);
        flushed += b.n;
        b.n = 0;
        bm = AddMasks{};
        return r;
    };
    // count tables (dd / dpd).  Single GPU: the rows go straight into the feature's table.  Exchange: accumulate = this
    // rank's delta counts as doubles into the feature's block of xchg, merge = the summed deltas into the table.
    auto table_counts = [&](dist_b200_feature *f, int i) -> int {
        const size_t cells = static_cast<size_t>(f->G) * f->dim;
        int r = DIST_B200_OK;
        if (phase == kRowsBoth) {
            r = launch_add_rows_counts(ctx, f, columns_dev[i], assign_dev, n_rows, sign, s, nullptr, mask_of(i));
        } else if (phase == kRowsAccumulate) {
            int32_t *tmp = reinterpret_cast<int32_t *>(static_cast<char *>(ctx->add_acc) + pooled_bytes);
            DISTB200_CUDA(ctx, cudaMemsetAsync(tmp, 0, sizeof(int32_t) * cells, s));
            r = launch_add_rows_counts(ctx, f, columns_dev[i], assign_dev, n_rows, +1, s, tmp, mask_of(i));
            if (!r) r = launch_counts_to_doubles(ctx, tmp, xchg + table_off, cells, s);
        } else {
            r = launch_merge_counts(ctx, reinterpret_cast<int32_t *>(f->stats[0]), xchg + table_off, cells, sign, s);
        }
        table_off += cells;
        return r;
    };
    for (int i = 0; i < n_features; ++i) {
        dist_b200_feature *f = features[i];
        const int G = f->G;
        switch (f->model) {
            case DIST_B200_NICH:
            case DIST_B200_GP:
            case DIST_B200_BB:
            case DIST_B200_BNB: {
                if (b.n == kAddBatch || (b.n && b.G != G))
                    if ((rc = flush())) return rc;
                b.G = G;
                bm.m[b.n] = mask_of(i);
                AddDesc &d = b.d[b.n++];
                d.column = columns_dev ? columns_dev[i] : nullptr;
                d.st0 = f->stats[0];
                d.st1 = f->stats[1];
                d.st2 = f->stats[2];
                d.params = static_cast<float4 *>(f->params);
                d.aux = f->aux;
                for (int k = 0; k < 4; ++k) d.shared[k] = f->shared[k];
                d.model = f->model;
                if (f->model == DIST_B200_GP && phase != kRowsAccumulate) {
                    f->gp_table_dirty = true;
                    f->log_prod_valid = false;  // Group::log_prod is not maintained by the batched update
                }
            } break;
            case DIST_B200_DD:
            case DIST_B200_DPD:
                if ((rc = table_counts(f, i))) return rc;
                if (phase == kRowsAccumulate) break;
                if ((rc = rebuild(f, 0, G, s))) return rc;
                break;
            case DIST_B200_NIW: {  // per-group SYRK into a [G][1 + d + d^2] double block (niw_stats.cu), then the records again
                const int d = f->dim;
                const size_t per = group_words(f);
                char *area = static_cast<char *>(ctx->add_acc) + pooled_bytes + table_tmp;
                double *acc = phase == kRowsBoth ? reinterpret_cast<double *>(area) : xchg + table_off;
                void *work = area + round_up(sizeof(double) * G * per, 256);
                if (phase != kRowsMerge &&
                    (rc = launch_niw_accumulate(ctx, G, d, columns_dev[i], assign_dev, n_rows, acc, work, s, mask_of(i))))
                    return rc;
                table_off += G * per;
                if (phase == kRowsAccumulate) break;
                if ((rc = launch_niw_apply(ctx, G, d, sign, acc, reinterpret_cast<int32_t *>(f->stats[0]), reinterpret_cast<float *>(f->stats[1]),
                                           reinterpret_cast<float *>(f->stats[2]), s)))
                    return rc;
                if ((rc = rebuild(f, 0, G, s))) return rc;
            } break;
            default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "add_rows: unsupported model");
        }
    }
    if ((rc = flush())) return rc;
    if (phase != kRowsAccumulate)
        for (int i = 0; i < n_features; ++i) DISTB200_CUDA(ctx, cudaEventRecord(features[i]->ready, s));
    DISTB200_CUDA(ctx, cudaEventRecord(ctx->add_done, s));
    return DIST_B200_OK;
}

// Row-sharded update (one process per GPU): every rank accumulates its own rows, the [n_features][4][G] double
// buffers are summed over the ranks (NCCL all-reduce by the caller), every rank merges the global sums into
// its replica of the statistics -- all replicas stay identical.
int dist_b200_rows_accumulate(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                              const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, double *xchg_dev,
                              void *stream) {
    return rows_batch(ctx, features, n_features, columns_dev, assign_dev, n_rows, +1, stream, kRowsAccumulate, xchg_dev);
}

int dist_b200_rows_xchg_doubles(dist_b200_feature *const *features, int n_features, size_t *n_doubles) {
    if (n_features < 0 || (n_features && !features) || !n_doubles) return DIST_B200_ERR_INVALID;
    size_t n = 0;
    for (int i = 0; i < n_features; ++i) {
        const dist_b200_feature *f = features[i];
        if (!f) return DIST_B200_ERR_INVALID;
        n += static_cast<size_t>(f->G) * (pooled_model(f->model) ? 4 : group_words(f));
    }
    *n_doubles = n;
    return DIST_B200_OK;
}

int dist_b200_rows_merge(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features, const double *xchg_dev,
                         int sign, void *stream) {
    if (sign != 1 && sign != -1) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "rows_merge: sign must be +1 or -1") : DIST_B200_ERR_INVALID;
    return rows_batch(ctx, features, n_features, nullptr, nullptr, 0, sign, stream, kRowsMerge, const_cast<double *>(xchg_dev));
}

int dist_b200_add_rows_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                             const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, void *stream) {
    return rows_batch(ctx, features, n_features, columns_dev, assign_dev, n_rows, +1, stream);
}

int dist_b200_remove_rows_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, void *stream) {
    return rows_batch(ctx, features, n_features, columns_dev, assign_dev, n_rows, -1, stream);
}

int dist_b200_rows_accumulate_masked(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                     const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, double *xchg_dev,
                                     const uint32_t *const *observed_dev, void *stream) {
    return rows_batch(ctx, features, n_features, columns_dev, assign_dev, n_rows, +1, stream, kRowsAccumulate, xchg_dev,
                      observed_dev);
}

int dist_b200_add_rows_batch_masked(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                    const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows,
                                    const uint32_t *const *observed_dev, void *stream) {
    return rows_batch(ctx, features, n_features, columns_dev, assign_dev, n_rows, +1, stream, kRowsBoth, nullptr, observed_dev);
}

int dist_b200_remove_rows_batch_masked(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                       const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows,
                                       const uint32_t *const *observed_dev, void *stream) {
    return rows_batch(ctx, features, n_features, columns_dev, assign_dev, n_rows, -1, stream, kRowsBoth, nullptr, observed_dev);
}

// bytes of one value of the feature's column: bool as uint8, niw a row of d floats, everything else 4 bytes
static size_t value_bytes(const dist_b200_feature *f) {
    return f->model == DIST_B200_BB ? 1 : f->model == DIST_B200_NIW ? 4 * static_cast<size_t>(f->dim) : 4;
}

// host buffers: stage columns + assignments through the context scratch, run the device batch, drain
static int rows_batch_host(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                           const void *const *columns_host, const int32_t *assign_host, size_t n_rows, int sign) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    if (n_features < 1 || !features || !columns_host || !assign_host) return fail(ctx, DIST_B200_ERR_INVALID, "add_rows_host: null argument");
    if (n_rows == 0) return DIST_B200_OK;
    for (int i = 0; i < n_features; ++i)
        if (!features[i] || !columns_host[i]) return fail(ctx, DIST_B200_ERR_INVALID, "add_rows_host: null feature / column");
    cudaStream_t s = ctx->own_stream;
    Staging stage(ctx, s);
    std::vector<size_t> off(n_features);
    for (int i = 0; i < n_features; ++i) off[i] = stage.region(value_bytes(features[i]) * n_rows);
    const size_t assign_off = stage.region(sizeof(int32_t) * n_rows);
    int rc = stage.reserve();
    if (rc) return rc;
    std::vector<const void *> cols(n_features);
    for (int i = 0; i < n_features; ++i) {
        if ((rc = stage.put(off[i], columns_host[i], value_bytes(features[i]) * n_rows, s))) return rc;
        cols[i] = stage.dev(off[i]);
    }
    if ((rc = stage.put(assign_off, assign_host, sizeof(int32_t) * n_rows, s)) ||
        (rc = rows_batch(ctx, features, n_features, cols.data(), stage.dev<const int32_t>(assign_off), n_rows, sign, s)))
        return rc;
    return stage.drain();
}

int dist_b200_add_rows_batch_host(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                  const void *const *columns_host, const int32_t *assign_host, size_t n_rows) {
    return rows_batch_host(ctx, features, n_features, columns_host, assign_host, n_rows, +1);
}

int dist_b200_remove_rows_batch_host(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                     const void *const *columns_host, const int32_t *assign_host, size_t n_rows) {
    return rows_batch_host(ctx, features, n_features, columns_host, assign_host, n_rows, -1);
}

// ---- batched Group::sample_value (sample_values.cu) ----------------------------------------------------------------
// arguments shared by the device and host forms; ERR_STATE for a feature without statistics or a G mismatch
static int check_sample_args(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features, const int32_t *assign,
                             void *const *columns_out) {
    if (n_features < 1 || !features || !assign || !columns_out) return fail(ctx, DIST_B200_ERR_INVALID, "sample_values: null argument");
    for (int i = 0; i < n_features; ++i) {
        const dist_b200_feature *f = features[i];
        if (!f || f->ctx != ctx || !columns_out[i]) return fail(ctx, DIST_B200_ERR_INVALID, "sample_values: bad feature / output column");
        if (f->G < 1 || !stats_resident(f)) return fail(ctx, DIST_B200_ERR_STATE, "sample_values: call update_all first");
        if (f->G != features[0]->G) return fail(ctx, DIST_B200_ERR_STATE, "sample_values: features disagree on the number of groups");
    }
    return DIST_B200_OK;
}

static SampleSrc sample_src(const dist_b200_feature *f) {
    SampleSrc src{};
    src.model = f->model;
    src.G = f->G;
    src.dim = f->dim;
    for (int k = 0; k < 4; ++k) src.shared[k] = f->shared[k];
    src.st0 = f->stats[0];
    src.st1 = f->stats[1];
    src.st2 = f->stats[2];
    src.alphas = f->alphas_dev;
    src.keys_sorted = f->keys_dev;
    src.key_rows = f->key_rows_dev;
    return src;
}

int dist_b200_sample_values_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                  const int32_t *assign_dev, size_t n_rows, uint64_t seed, uint64_t row0,
                                  void *const *columns_out_dev, void *stream) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    dist_b200_feature *const *fs = const_cast<dist_b200_feature *const *>(features);
    int rc = check_sample_args(ctx, fs, n_features, assign_dev, columns_out_dev);
    if (rc || n_rows == 0) return rc;
    cudaStream_t s = as_stream(stream);
    if ((rc = wait_ready(ctx, features, n_features, s))) return rc;  // a preceding add / remove / update on another stream
    for (int i = 0; i < n_features; ++i)
        if ((rc = launch_sample_values(ctx, fs[i], sample_src(fs[i]), static_cast<uint32_t>(i), assign_dev, n_rows, seed, row0,
                                       columns_out_dev[i], s)))
            return rc;
    return DIST_B200_OK;
}

// imputation: the unmasked kernels over an assignment vector that keeps only the missing cells' rows (mask_assign, keep = 0),
// so every drawn cell is the unmasked call's draw for the same (seed, row, position) and every other cell is untouched
int dist_b200_sample_values_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                         const int32_t *assign_dev, size_t n_rows, uint64_t seed, uint64_t row0,
                                         void *const *columns_out_dev, const uint32_t *const *observed_dev, void *stream) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    dist_b200_feature *const *fs = const_cast<dist_b200_feature *const *>(features);
    int rc = check_sample_args(ctx, fs, n_features, assign_dev, columns_out_dev);
    if (rc || n_rows == 0 || !observed_dev) return rc;
    cudaStream_t s = as_stream(stream);
    if ((rc = wait_ready(ctx, features, n_features, s))) return rc;
    if ((rc = grow(ctx, ctx->missing_scratch, ctx->missing_scratch_bytes, sizeof(int32_t) * n_rows))) return rc;
    int32_t *missing_assign = static_cast<int32_t *>(ctx->missing_scratch);
    for (int i = 0; i < n_features; ++i) {
        if (!observed_dev[i]) continue;  // fully observed: nothing to impute
        if ((rc = launch_mask_assign(ctx, assign_dev, observed_dev[i], n_rows, 0, missing_assign, s)) ||
            (rc = launch_sample_values(ctx, fs[i], sample_src(fs[i]), static_cast<uint32_t>(i), missing_assign, n_rows, seed, row0,
                                       columns_out_dev[i], s)))
            return rc;
    }
    return DIST_B200_OK;
}

// host buffers: the assignments and the output columns go up (rows the call skips keep their values), the columns come back
int dist_b200_sample_values_batch_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                       const int32_t *assign_host, size_t n_rows, uint64_t seed, uint64_t row0,
                                       void *const *columns_out_host) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    int rc = check_sample_args(ctx, const_cast<dist_b200_feature *const *>(features), n_features, assign_host, columns_out_host);
    if (rc || n_rows == 0) return rc;
    cudaStream_t s = ctx->own_stream;
    Staging stage(ctx, s);
    std::vector<size_t> off(n_features);
    for (int i = 0; i < n_features; ++i) off[i] = stage.region(value_bytes(features[i]) * n_rows);
    const size_t assign_off = stage.region(sizeof(int32_t) * n_rows);
    if ((rc = stage.reserve())) return rc;
    std::vector<void *> cols(n_features);
    for (int i = 0; i < n_features; ++i) {
        cols[i] = stage.dev(off[i]);
        if ((rc = stage.put(off[i], columns_out_host[i], value_bytes(features[i]) * n_rows, s))) return rc;
    }
    if ((rc = stage.put(assign_off, assign_host, sizeof(int32_t) * n_rows, s)) ||
        (rc = dist_b200_sample_values_batch(ctx, features, n_features, stage.dev<const int32_t>(assign_off), n_rows, seed, row0,
                                            cols.data(), s)))
        return rc;
    for (int i = 0; i < n_features; ++i)
        if ((rc = stage.get(columns_out_host[i], off[i], value_bytes(features[i]) * n_rows, s))) return rc;
    return stage.drain();
}

int dist_b200_feature_add_rows(dist_b200_feature *f, const void *column_dev, const int32_t *assign_dev, size_t n_rows,
                               void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    return dist_b200_add_rows_batch(f->ctx, &f, 1, &column_dev, assign_dev, n_rows, stream);
}

// ---- score_data_grid (next row: hyper-parameter inference over the same device-resident statistics) ----
static size_t shared_stride(const dist_b200_feature *f) {
    switch (f->model) {
        case DIST_B200_NICH: return 4;
        case DIST_B200_GP: case DIST_B200_BB: case DIST_B200_BNB: return 2;
        case DIST_B200_DD: return static_cast<size_t>(f->dim);
        case DIST_B200_DPD: return 1;
        case DIST_B200_NIW: return 2 + static_cast<size_t>(f->dim) + static_cast<size_t>(f->dim) * f->dim;  // kappa, nu, mu[d], psi[d][d]
        default: return 0;
    }
}

int dist_b200_gp_set_log_prod(dist_b200_feature *f, const float *log_prod_host, void *stream) {
    if (!check_feature(f, DIST_B200_GP) || !log_prod_host) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (f->G < 1) return fail(ctx, DIST_B200_ERR_STATE, "gp_set_log_prod: call update_all first");
    if (int rc = grow(ctx, f->log_prod_dev, f->log_prod_bytes, sizeof(float) * f->capacity)) return rc;
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaMemcpyAsync(f->log_prod_dev, log_prod_host, sizeof(float) * f->G, cudaMemcpyHostToDevice, s));
    DISTB200_CUDA(ctx, cudaStreamSynchronize(s));  // pageable source
    f->log_prod_valid = true;
    return DIST_B200_OK;
}

int dist_b200_score_data_grid(dist_b200_feature *f, const float *shareds_dev, size_t n_grid, size_t stride,
                              float *out_dev, void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (!shareds_dev || !out_dev) return fail(ctx, DIST_B200_ERR_INVALID, "score_data_grid: null argument");
    if (f->G < 1 || !stats_resident(f)) return fail(ctx, DIST_B200_ERR_STATE, "score_data_grid: call update_all first");
    if (stride < shared_stride(f)) return fail(ctx, DIST_B200_ERR_INVALID, "score_data_grid: stride shorter than the model's packed Shared");
    if (f->model == DIST_B200_GP && !f->log_prod_valid)
        return fail(ctx, DIST_B200_ERR_STATE, "score_data_grid: gp needs Group::log_prod (dist_b200_gp_set_log_prod) after the last statistics change");
    if (n_grid == 0) return DIST_B200_OK;
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
    // the double accumulators live next to the add_value accumulators (same event guards both)
    int rc = grow(ctx, ctx->add_acc, ctx->add_acc_bytes, sizeof(double) * n_grid);
    if (rc) return rc;
    if (!ctx->add_done) DISTB200_CUDA(ctx, cudaEventCreateWithFlags(&ctx->add_done, cudaEventDisableTiming));
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, ctx->add_done, 0));
    double *acc = static_cast<double *>(ctx->add_acc);
    if (f->model == DIST_B200_NIW) {
        DISTB200_CUDA(ctx, cudaMemsetAsync(acc, 0, sizeof(double) * n_grid, s));
        rc = launch_niw_score_data(ctx, f->G, f->dim, reinterpret_cast<const int32_t *>(f->stats[0]), reinterpret_cast<const float *>(f->stats[1]),
                                   reinterpret_cast<const float *>(f->stats[2]), shareds_dev, n_grid, stride, acc, s);
        if (!rc) rc = launch_score_data_finish(ctx, n_grid, acc, out_dev, s);
    } else {
        rc = launch_score_data(ctx, f, f->stats[0], f->stats[1], f->stats[2], f->alphas_dev, f->log_prod_dev, shareds_dev, n_grid, stride,
                               acc, out_dev, s);
    }
    if (rc) return rc;
    DISTB200_CUDA(ctx, cudaEventRecord(ctx->add_done, s));
    return DIST_B200_OK;
}

int dist_b200_score_data_grid_host(dist_b200_feature *f, const float *shareds_host, size_t n_grid, size_t stride,
                                   float *out_host) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (!shareds_host || !out_host) return fail(ctx, DIST_B200_ERR_INVALID, "score_data_grid: null argument");
    if (n_grid == 0) return DIST_B200_OK;
    cudaStream_t s = ctx->own_stream;
    Staging stage(ctx, s);
    const size_t in_off = stage.region(sizeof(float) * n_grid * stride), out_off = stage.region(sizeof(float) * n_grid);
    int rc;
    if ((rc = stage.reserve()) || (rc = stage.put(in_off, shareds_host, sizeof(float) * n_grid * stride, s)) ||
        (rc = dist_b200_score_data_grid(f, stage.dev<const float>(in_off), n_grid, stride, stage.dev<float>(out_off), s)) ||
        (rc = stage.get(out_host, out_off, sizeof(float) * n_grid, s)))
        return rc;
    return stage.drain();
}

// ---- protobuf wire format (schema.proto) -> update_all (SURVEY 8f rank 4) --------------------------
int dist_b200_wire_decode(dist_b200_ctx *ctx, int model, const void *shared_msg, size_t shared_len,
                          const void *const *group_msgs, const size_t *group_lens, int G, float *shared_out,
                          size_t shared_cap, uint32_t *keys_out, size_t keys_cap, uint32_t *stats_out, size_t stats_cap,
                          size_t counts_out[3]) {
    if (!counts_out) return DIST_B200_ERR_INVALID;  // ctx may be null: decoding needs no device
    WireFeature w;
    int rc = wire_decode(ctx, model, shared_msg, shared_len, group_msgs, group_lens, G, w);
    if (rc) return rc;
    counts_out[0] = w.shared.size();
    counts_out[1] = w.keys.size();
    counts_out[2] = w.stats.size();
    if (w.shared.size() > shared_cap || w.keys.size() > keys_cap || w.stats.size() > stats_cap)
        return fail(ctx, DIST_B200_ERR_INVALID, "wire_decode: output buffer too small (sizes returned in counts_out)");
    if (shared_out && !w.shared.empty()) std::memcpy(shared_out, w.shared.data(), sizeof(float) * w.shared.size());
    if (keys_out && !w.keys.empty()) std::memcpy(keys_out, w.keys.data(), sizeof(uint32_t) * w.keys.size());
    if (stats_out && !w.stats.empty()) std::memcpy(stats_out, w.stats.data(), sizeof(uint32_t) * w.stats.size());
    return DIST_B200_OK;
}

int dist_b200_update_all_wire(dist_b200_feature *f, const void *shared_msg, size_t shared_len,
                              const void *const *group_msgs, const size_t *group_lens, int G, void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    WireFeature w;
    int rc = wire_decode(ctx, f->model, shared_msg, shared_len, group_msgs, group_lens, G, w);
    if (rc) return rc;
    const size_t g = static_cast<size_t>(G);
    const uint32_t *st = w.stats.data();
    switch (f->model) {
        case DIST_B200_NICH:
            return dist_b200_nich_update_all(f, w.shared.data(), G, reinterpret_cast<const int32_t *>(st),
                                             reinterpret_cast<const float *>(st + g), reinterpret_cast<const float *>(st + 2 * g), stream);
        case DIST_B200_GP:
            if ((rc = dist_b200_gp_update_all(f, w.shared.data(), G, st, st + g, stream))) return rc;
            return G ? dist_b200_gp_set_log_prod(f, reinterpret_cast<const float *>(st + 2 * g), stream) : DIST_B200_OK;
        case DIST_B200_BNB:
            return dist_b200_bnb_update_all(f, w.shared.data(), w.keys[0], G, st, st + g, stream);
        case DIST_B200_BB:
            return dist_b200_bb_update_all(f, w.shared.data(), G, reinterpret_cast<const int32_t *>(st),
                                           reinterpret_cast<const int32_t *>(st + g), stream);
        case DIST_B200_DD:
            return dist_b200_dd_update_all(f, w.dim, w.shared.data(), G, reinterpret_cast<const int32_t *>(st), stream);
        case DIST_B200_DPD:
            return dist_b200_dpd_update_all(f, w.shared[1], w.shared[2], w.dim, w.keys.data(), w.shared.data() + 3, G,
                                            reinterpret_cast<const int32_t *>(st), stream);
        case DIST_B200_NIW: {
            const size_t d = static_cast<size_t>(w.dim);
            return dist_b200_niw_update_all(f, w.dim, w.shared.data() + 2, w.shared[0], w.shared.data() + 2 + d, w.shared[1], G,
                                            reinterpret_cast<const int32_t *>(st), reinterpret_cast<const float *>(st + g),
                                            reinterpret_cast<const float *>(st + g + g * d), stream);
        }
        default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "update_all_wire: unsupported model");
    }
}

// the reference's record stream (distributions/io/stream.py:141-153): [uint32 little-endian length][message] ...
static int split_stream(dist_b200_ctx *ctx, const void *bytes, size_t len, std::vector<const void *> &msgs,
                        std::vector<size_t> &lens) {
    const uint8_t *p = static_cast<const uint8_t *>(bytes), *end = p + len;
    while (p < end) {
        if (end - p < 4) return fail(ctx, DIST_B200_ERR_INVALID, "wire stream: truncated record length");
        const size_t n = static_cast<size_t>(p[0]) | (static_cast<size_t>(p[1]) << 8) | (static_cast<size_t>(p[2]) << 16) |
                         (static_cast<size_t>(p[3]) << 24);
        p += 4;
        if (n > static_cast<size_t>(end - p)) return fail(ctx, DIST_B200_ERR_INVALID, "wire stream: record runs past the end");
        msgs.push_back(p);
        lens.push_back(n);
        p += n;
    }
    return DIST_B200_OK;
}

int dist_b200_wire_split_stream(dist_b200_ctx *ctx, const void *stream_bytes, size_t stream_len, size_t *offsets_out,
                                size_t *lens_out, size_t capacity, size_t *n_records) {
    if ((!stream_bytes && stream_len) || !n_records) return DIST_B200_ERR_INVALID;  // ctx may be null
    std::vector<const void *> msgs;
    std::vector<size_t> lens;
    int rc = split_stream(ctx, stream_bytes, stream_len, msgs, lens);
    if (rc) return rc;
    *n_records = msgs.size();
    if (msgs.size() > capacity) return fail(ctx, DIST_B200_ERR_INVALID, "wire_split_stream: output arrays too small (count returned)");
    for (size_t i = 0; i < msgs.size(); ++i) {
        if (offsets_out) offsets_out[i] = static_cast<size_t>(static_cast<const uint8_t *>(msgs[i]) - static_cast<const uint8_t *>(stream_bytes));
        if (lens_out) lens_out[i] = lens[i];
    }
    return DIST_B200_OK;
}

int dist_b200_update_all_stream(dist_b200_feature *f, const void *shared_msg, size_t shared_len, const void *stream_bytes,
                                size_t stream_len, void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    if (!stream_bytes && stream_len) return fail(f->ctx, DIST_B200_ERR_INVALID, "update_all_stream: null stream");
    std::vector<const void *> msgs;
    std::vector<size_t> lens;
    int rc = split_stream(f->ctx, stream_bytes, stream_len, msgs, lens);
    if (rc) return rc;
    if (msgs.size() > 0x7FFFFFFFull) return fail(f->ctx, DIST_B200_ERR_UNSUPPORTED, "update_all_stream: too many groups");
    return dist_b200_update_all_wire(f, shared_msg, shared_len, msgs.data(), lens.data(), static_cast<int>(msgs.size()), stream);
}

int dist_b200_prior_wire_host(dist_b200_ctx *ctx, const void *clustering_msg, size_t len, int G,
                              const int32_t *group_sizes, float *prior_host) {
    if (!ctx || !clustering_msg || !group_sizes || !prior_host || G < 1) return DIST_B200_ERR_INVALID;
    int which = 0;
    float alpha = 0, d = 0;
    uint64_t dataset_size = 0;
    int rc = wire_decode_clustering(ctx, clustering_msg, len, &which, &alpha, &d, &dataset_size);
    if (rc) return rc;
    if (which == 1) return dist_b200_prior_pitman_yor_host(ctx, alpha, d, G, group_sizes, prior_host);
    if (dataset_size < 1 || dataset_size > 0x7FFFFFFFull) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "wire: LowEntropy dataset_size out of range");
    return dist_b200_prior_low_entropy_host(ctx, static_cast<int>(dataset_size), G, group_sizes, prior_host);
}

static int emit_messages(dist_b200_ctx *ctx, const std::vector<uint8_t> &bytes, const std::vector<size_t> &lens, void *out,
                         size_t capacity, size_t *lens_out, size_t *n_bytes) {
    if (n_bytes) *n_bytes = bytes.size();
    if (bytes.size() > capacity) return fail(ctx, DIST_B200_ERR_INVALID, "wire: output buffer too small (size returned in n_bytes)");
    if (!bytes.empty()) std::memcpy(out, bytes.data(), bytes.size());
    if (lens_out) for (size_t i = 0; i < lens.size(); ++i) lens_out[i] = lens[i];
    return DIST_B200_OK;
}

int dist_b200_wire_encode_groups(dist_b200_ctx *ctx, int model, int G, int dim, const uint32_t *keys, const uint32_t *stats,
                                 size_t stats_words, void *out, size_t capacity, size_t *lens_out, size_t *n_bytes) {
    std::vector<uint8_t> bytes;
    std::vector<size_t> lens;
    int rc = wire_encode_groups(ctx, model, G, dim, keys, stats, stats_words, bytes, lens);
    if (rc) return rc;
    return emit_messages(ctx, bytes, lens, out, capacity, lens_out, n_bytes);
}

int dist_b200_wire_encode_shared(dist_b200_ctx *ctx, int model, const float *shared, size_t n_shared, const uint32_t *keys,
                                 size_t n_keys, void *out, size_t capacity, size_t *n_bytes) {
    std::vector<uint8_t> bytes;
    int rc = wire_encode_shared(ctx, model, shared, n_shared, keys, n_keys, bytes);
    if (rc) return rc;
    return emit_messages(ctx, bytes, std::vector<size_t>(), out, capacity, nullptr, n_bytes);
}

int dist_b200_feature_dump_groups_wire(dist_b200_feature *f, void *out, size_t capacity, size_t *lens_out, size_t *n_bytes,
                                       void *stream) {
    if (!f || !f->ctx) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (!stats_resident(f) || f->G < 1) return fail(ctx, DIST_B200_ERR_STATE, "dump_groups_wire: no device statistics (update_all first)");
    const size_t g = static_cast<size_t>(f->G);
    const size_t words = g * (group_words(f) + (f->model == DIST_B200_GP ? 1 : 0));  // gp: + Group::log_prod
    std::vector<uint32_t> st(words, 0);
    size_t got = 0;
    int rc = dist_b200_feature_download_stats(f, st.data(), 4 * words, &got, stream);  // synchronises
    if (rc) return rc;
    if (f->model == DIST_B200_GP) {  // Group::log_prod is a required field of the message
        if (!f->log_prod_valid) return fail(ctx, DIST_B200_ERR_STATE, "dump_groups_wire: gp log_prod is stale (dist_b200_gp_set_log_prod)");
        DISTB200_CUDA(ctx, cudaMemcpy(st.data() + 2 * g, f->log_prod_dev, 4 * g, cudaMemcpyDeviceToHost));
    }
    // dpd: f->keys is update_all's key array, in the caller's order like the mirrored counts
    std::vector<uint32_t> keys;
    if (f->model == DIST_B200_DPD) {
        if (f->keys.size() != static_cast<size_t>(f->dim)) return fail(ctx, DIST_B200_ERR_STATE, "dump_groups_wire: dpd keys missing");
        keys = f->keys;
    }
    std::vector<uint8_t> bytes;
    std::vector<size_t> lens;
    if ((rc = wire_encode_groups(ctx, f->model, f->G, f->dim, keys.data(), st.data(), words, bytes, lens))) return rc;
    return emit_messages(ctx, bytes, lens, out, capacity, lens_out, n_bytes);
}

int dist_b200_feature_download_stats(const dist_b200_feature *f, void *out_host, size_t capacity_bytes, size_t *n_bytes,
                                     void *stream) {
    if (!f || !f->ctx || !out_host) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    if (!stats_resident(f)) return fail(ctx, DIST_B200_ERR_STATE, "download_stats: no device statistics (update_all first)");
    const size_t total = 4 * group_words(f) * f->G;
    if (n_bytes) *n_bytes = total;
    if (total > capacity_bytes) return fail(ctx, DIST_B200_ERR_INVALID, "download_stats: buffer too small");
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));
    char *out = static_cast<char *>(out_host);
    for (int a = 0; a < stat_arrays(f); ++a) {
        const size_t b = 4 * stat_elems(f, a) * f->G;
        DISTB200_CUDA(ctx, cudaMemcpyAsync(out, f->stats[a], b, cudaMemcpyDeviceToHost, s));
        out += b;
    }
    DISTB200_CUDA(ctx, cudaStreamSynchronize(s));
    return DIST_B200_OK;
}

int dist_b200_count_assignments(dist_b200_ctx *ctx, const int32_t *assign_dev, size_t n_rows, int G, int32_t *counts_dev,
                                int accumulate, void *stream) {
    if (!ctx || !assign_dev || !counts_dev || G < 1) return DIST_B200_ERR_INVALID;
    return launch_count_assignments(ctx, assign_dev, n_rows, G, counts_dev, accumulate, as_stream(stream));
}

int dist_b200_prior_pitman_yor_dev(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *group_sizes_dev,
                                   float *prior_dev, void *stream) {
    if (!ctx || G < 1 || !group_sizes_dev || !prior_dev) return DIST_B200_ERR_INVALID;
    return launch_prior_prep(ctx, alpha, d, G, group_sizes_dev, prior_dev, as_stream(stream));
}

int dist_b200_feature_download_caches(const dist_b200_feature *f, float *out_host, size_t capacity_floats,
                                      size_t *n_floats, void *stream) {
    if (!f || !f->ctx || !out_host) return DIST_B200_ERR_INVALID;
    dist_b200_ctx *ctx = f->ctx;
    size_t rows;
    switch (f->model) {
        case DIST_B200_NICH: rows = 4; break;
        case DIST_B200_GP: rows = 3; break;
        case DIST_B200_BNB: rows = 3; break;
        case DIST_B200_BB: rows = 2; break;
        case DIST_B200_DD: rows = f->dim; break;
        case DIST_B200_DPD: rows = f->dim + 1; break;
        default: return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "download_caches: unsupported model");
    }
    const size_t n = rows * f->G;
    if (n_floats) *n_floats = n;
    if (n > capacity_floats) return fail(ctx, DIST_B200_ERR_INVALID, "download_caches: buffer too small");
    if (n == 0) return DIST_B200_OK;
    int rc = ensure_scratch(ctx, n * sizeof(float));
    if (rc) return rc;
    cudaStream_t s = as_stream(stream);
    DISTB200_CUDA(ctx, cudaStreamWaitEvent(s, f->ready, 0));  // a batched add / remove may still be rebuilding the caches
    if ((rc = launch_unpack_caches(ctx, f, static_cast<float *>(ctx->scratch_dev), s))) return rc;
    DISTB200_CUDA(ctx, cudaMemcpyAsync(out_host, ctx->scratch_dev, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    DISTB200_CUDA(ctx, cudaStreamSynchronize(s));
    return DIST_B200_OK;
}

int dist_b200_prior_pitman_yor(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *group_sizes,
                               float *prior_dev, void *stream) {
    if (!ctx || G < 1 || !group_sizes || !prior_dev) return DIST_B200_ERR_INVALID;
    return prior_from_host_sizes(ctx, G, group_sizes, prior_dev, nullptr, as_stream(stream),
                                 [&](const int32_t *sz, float *out, cudaStream_t s) { return launch_prior_prep(ctx, alpha, d, G, sz, out, s); });
}

// LowEntropy clustering prior (clustering.hpp:245-331 through MixtureDriver::score_value): overwrite semantics
int dist_b200_prior_low_entropy_dev(dist_b200_ctx *ctx, int dataset_size, int G, const int32_t *sizes_dev,
                                    float *prior_dev, void *stream) {
    if (!ctx || G < 1 || !sizes_dev || !prior_dev || dataset_size < 1) return DIST_B200_ERR_INVALID;
    return launch_low_entropy_prep(ctx, dataset_size, G, sizes_dev, prior_dev, as_stream(stream));
}

int dist_b200_prior_low_entropy_host(dist_b200_ctx *ctx, int dataset_size, int G, const int32_t *group_sizes,
                                     float *prior_host) {
    if (!ctx || G < 1 || !group_sizes || !prior_host || dataset_size < 1) return DIST_B200_ERR_INVALID;
    return prior_from_host_sizes(ctx, G, group_sizes, nullptr, prior_host, ctx->own_stream, [&](const int32_t *sz, float *out, cudaStream_t s) {
        return launch_low_entropy_prep(ctx, dataset_size, G, sz, out, s);
    });
}

int dist_b200_prior_pitman_yor_host(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *group_sizes,
                                    float *prior_host) {
    if (!ctx || G < 1 || !group_sizes || !prior_host) return DIST_B200_ERR_INVALID;
    return prior_from_host_sizes(ctx, G, group_sizes, nullptr, prior_host, ctx->own_stream,
                                 [&](const int32_t *sz, float *out, cudaStream_t s) { return launch_prior_prep(ctx, alpha, d, G, sz, out, s); });
}

// ---- the hot path ---------------------------------------------------------------------------
// Make f's GammaPoisson value table current: grown with the feature's capacity, its rebuild queued in `tb` when stale
// (rebuilt lazily, stream-ordered, after any cache update).  The caller launches what remains queued.
static int queue_gp_table(dist_b200_ctx *ctx, dist_b200_feature *f, GpTableBatch &tb, cudaStream_t s) {
    const size_t bytes = sizeof(float) * 2 * kGpTableX * f->capacity;  // [capacity][x] | [x][capacity]
    if (bytes > f->gp_table_bytes) {
        if (int rc = grow(ctx, f->gp_table, f->gp_table_bytes, bytes)) return rc;
        f->gp_table_dirty = true;
    }
    if (!f->gp_table_dirty) return DIST_B200_OK;
    if (tb.n == kGpTableBatch) {
        int rc = launch_gp_table_batch(ctx, tb, s);
        if (rc) return rc;
        tb.n = 0;
    }
    tb.n_groups[tb.n] = f->capacity;
    tb.params[tb.n] = static_cast<const float4 *>(f->params);
    tb.table[tb.n] = f->gp_table;
    ++tb.n;
    f->gp_table_dirty = false;
    return DIST_B200_OK;
}

// Describe one row-mapped feature for the score kernel.  multi: GammaPoisson goes through its per-(group, value) table.
static int fill_desc(dist_b200_ctx *ctx, const dist_b200_feature *cf, const void *column, bool multi, FeatDesc &d,
                     GpTableBatch &tb, cudaStream_t s) {
    dist_b200_feature *f = const_cast<dist_b200_feature *>(cf);
    d.params = f->params;
    d.column = column;
    d.kind = f->model;
    d.vdim = f->dim;
    d.aux = nullptr;
    d.cap = f->capacity;
    d.pad_ = 0;
    if (multi && f->model == DIST_B200_GP) {
        if (int rc = queue_gp_table(ctx, f, tb, s)) return rc;
        d.params = f->gp_table;
        d.kind = kKindGpTable;
        d.vdim = kGpTableX;
        d.aux = f->params;
    }
    return DIST_B200_OK;
}

// rebuild every stale GammaPoisson value table of a multi-feature list on `s` (one launch per 128) and
// re-record the features' ready events, so that other streams order themselves behind the rebuild
static int refresh_gp_tables(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F, cudaStream_t s) {
    if (F < 2) return DIST_B200_OK;
    GpTableBatch tb;
    tb.n = 0;
    bool any = false;
    for (int f = 0; f < F; ++f) {
        if (!features[f] || features[f]->model != DIST_B200_GP) continue;
        const int queued = tb.n;
        int rc = queue_gp_table(ctx, const_cast<dist_b200_feature *>(features[f]), tb, s);
        if (rc) return rc;
        any = any || tb.n != queued;
    }
    if (!any) return DIST_B200_OK;
    int rc = launch_gp_table_batch(ctx, tb, s);
    if (rc) return rc;
    for (int f = 0; f < F; ++f)
        if (features[f] && features[f]->model == DIST_B200_GP) DISTB200_CUDA(ctx, cudaEventRecord(features[f]->ready, s));
    return DIST_B200_OK;
}

// argument checks of every score entry; G = the list's number of groups
static int check_score_args(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F, const void *const *columns,
                            const float *prior, const float *u, const int32_t *assign, const float *scores, int accumulate,
                            const float *logp, int &G) {
    if (!ctx || !features || !columns || F < 1) return DIST_B200_ERR_INVALID;
    if (!assign && !scores && !logp) return fail(ctx, DIST_B200_ERR_INVALID, "score: no output requested");
    if (assign && !u) return fail(ctx, DIST_B200_ERR_INVALID, "score_sample: u is required");
    if (accumulate && prior) return fail(ctx, DIST_B200_ERR_INVALID, "score: prior is an overwrite, not valid with accumulate");
    G = features[0] ? features[0]->G : 0;
    if (G < 1) return fail(ctx, DIST_B200_ERR_STATE, "score: feature 0 has no groups (call update_all)");
    for (int f = 0; f < F; ++f) {
        if (!features[f] || !columns[f]) return fail(ctx, DIST_B200_ERR_INVALID, "score: null feature / column");
        if (features[f]->ctx != ctx) return fail(ctx, DIST_B200_ERR_INVALID, "score: feature belongs to another context");
        if (features[f]->G != G) return fail(ctx, DIST_B200_ERR_STATE, "score: features disagree on the number of groups");
    }
    return DIST_B200_OK;
}

// Row-mapped models (nich/gp/bb/dd) fuse into one launch.  dpd (value-major table, warp per row) and
// niw (dense contraction) have their own kernels: alone they run directly, in mixed lists the scores
// are materialised, every feature accumulates, and the stand-alone sampler finishes.
static bool solo(const dist_b200_feature *f) { return f->model == DIST_B200_DPD || f->model == DIST_B200_NIW; }

// The row-mapped part of a feature list (solo features skipped), with each feature's observed mask in `ml` when `ml` is
// given; stale GammaPoisson value tables are rebuilt on `s`.  multi: see fill_desc.  At most kMaxFeatures row-mapped.
static int build_list(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F, const void *const *columns,
                      const uint32_t *const *observed, bool multi, FeatList &fl, MaskList *ml, cudaStream_t s) {
    GpTableBatch tb;
    tb.n = 0;
    fl.n = 0;
    for (int f = 0; f < F; ++f) {
        if (solo(features[f])) continue;
        if (ml) ml->m[fl.n] = observed[f];
        if (int rc = fill_desc(ctx, features[f], columns[f], multi, fl.f[fl.n++], tb, s)) return rc;
    }
    return launch_gp_table_batch(ctx, tb, s);
}

// Missing cells (dist_b200.h: "Missing cells"): observed[f] is NULL (feature f fully observed) or its mask; observed may
// be NULL.  A call is masked when any mask is non-NULL.  Then the row-mapped features run the masked feature-list kernel
// (a list of one too), and each masked dpd / niw feature is scored alone into a second [N][G] buffer and added where
// observed (masked_accumulate).  The single-feature routes are taken on unmasked calls only.
// logp != nullptr (assign = scores = nullptr): logp[n] = log sum_g exp(prior[g] + sum_f score_f) per row
static int score_dispatch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F, const void *const *columns,
                          const uint32_t *const *observed, size_t N, const float *prior, const float *u, int32_t *assign,
                          float *scores, int accumulate, cudaStream_t s, float *logp = nullptr) {
    int G = 0;
    if (int rc = check_score_args(ctx, features, F, columns, prior, u, assign, scores, accumulate, logp, G)) return rc;
    if (N == 0) return DIST_B200_OK;
    if (int rc = wait_ready(ctx, features, F, s)) return rc;
    bool masked = false, masked_solo = false;
    int n_solo = 0;
    for (int f = 0; f < F; ++f) {
        const bool m = observed && observed[f];
        masked = masked || m;
        masked_solo = masked_solo || (m && solo(features[f]));
        n_solo += solo(features[f]) ? 1 : 0;
    }
    if (!masked && F == 1) {
        dist_b200_feature *f0 = const_cast<dist_b200_feature *>(features[0]);
        // ONE table feature (dpd / dd / bb): every row with the same value has the same likelihood vector, so it is evaluated
        // once per distinct value (table_rows.cu).  SURVEY 8(d) "algorithmic shortcut".  DIST_B200_OPT_VALUE_CDF = 1 keeps
        // the per-cell kernels (what bench.py reports beside it), 2 = the round-2 tree search instead of the guide-table walk
        if (ctx->opt[DIST_B200_OPT_VALUE_CDF] != 1 &&
            (f0->model == DIST_B200_DPD || f0->model == DIST_B200_DD || f0->model == DIST_B200_BB)) {
            const int R = f0->model == DIST_B200_DPD ? f0->dim + 1 : (f0->model == DIST_B200_DD ? f0->dim : 2);  // table rows
            // sampling only: per-value CDF trees
            if (assign && !scores && !accumulate) {
                int rc = grow(ctx, f0->cdf_buf, f0->cdf_bytes, sizeof(float) * value_cdf_floats(R, G));
                if (!rc) rc = launch_value_cdf(ctx, f0, f0->cdf_buf, columns[0], N, prior, u, assign, s);
                if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
            }
            // logp: the log-normaliser is a function of the value alone, one log-sum-exp per table row and a gather per row
            if (logp) {
                int rc = grow(ctx, f0->cdf_buf, f0->cdf_bytes, sizeof(float) * R);
                if (!rc) rc = launch_value_logp(ctx, f0, f0->cdf_buf, columns[0], N, prior, logp, s);
                if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
            }
        }
        // one NIW<32> feature, sampling only: quadratic forms, scores and sample_from_scores in one tcgen05 kernel
        if (f0->model == DIST_B200_NIW && f0->dim == 32 && f0->niw_tc && assign && !scores && !accumulate &&
            ctx->opt[DIST_B200_OPT_NIW_PATH] == 0)
            return launch_niw_tc(ctx, G, f0->niw_tc, columns[0], N, prior, nullptr, 0, u, assign, s);
        // one NIW feature with d <= 8, sampling only: the fused FP32 kernel (DIST_B200_OPT_NIW_PATH = 1 keeps the materialising route)
        if (f0->model == DIST_B200_NIW && f0->dim <= 8 && assign && !scores && !accumulate && ctx->opt[DIST_B200_OPT_NIW_PATH] == 0) {
            const int rc = launch_niw_rows_small(ctx, f0, columns[0], N, prior, u, assign, s);
            if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
        }
        // logp over dpd / niw (alone or in a mixed list): the scores are materialised and reduced by logp_scores_kernel
        if (f0->model == DIST_B200_DPD && !logp) {
            if (assign && !scores && !accumulate && ctx->opt[DIST_B200_OPT_TABLE_KERNEL] != 1) {
                const int rc = launch_table_rows(ctx, f0, columns[0], N, prior, u, assign, s);
                if (rc != DIST_B200_ERR_UNSUPPORTED) return rc;
            }
            return launch_gather_rows(ctx, f0, columns[0], N, prior, u, assign, scores, accumulate, s);
        }
    }
    if (F - n_solo > kMaxFeatures) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "score: more than 512 features in one call");
    FeatList fl;
    MaskList ml;
    MaskList *masks = masked ? &ml : nullptr;
    int rc = build_list(ctx, features, F, columns, observed, F > 1, fl, masks, s);
    if (rc) return rc;
    if (n_solo == 0) return launch_score_rows(ctx, fl, G, N, prior, u, assign, scores, accumulate, s, nullptr, logp, masks);
    const size_t cells = N * static_cast<size_t>(G);
    float *buf = scores;
    if (!buf) {
        if ((rc = grow(ctx, ctx->scores_scratch, ctx->scores_scratch_bytes, sizeof(float) * cells))) return rc;
        buf = static_cast<float *>(ctx->scores_scratch);
    }
    float *tmp = nullptr;  // a masked dpd / niw feature's scores, before they are added where observed
    if (masked_solo) {
        if ((rc = grow(ctx, ctx->missing_scratch, ctx->missing_scratch_bytes, sizeof(float) * cells))) return rc;
        tmp = static_cast<float *>(ctx->missing_scratch);
    }
    bool started = accumulate != 0;
    if (fl.n) {
        if ((rc = launch_score_rows(ctx, fl, G, N, prior, nullptr, nullptr, buf, accumulate, s, nullptr, nullptr, masks))) return rc;
        started = true;
    }
    for (int f = 0; f < F; ++f) {
        const dist_b200_feature *feat = features[f];
        if (!solo(feat)) continue;
        const uint32_t *m = observed ? observed[f] : nullptr;
        float *dst = m ? tmp : buf;
        const float *p = m || started ? nullptr : prior;
        const int acc = !m && started ? 1 : 0;
        if (feat->model == DIST_B200_DPD) rc = launch_gather_rows(ctx, feat, columns[f], N, p, nullptr, nullptr, dst, acc, s);
        else rc = launch_niw_scores(ctx, feat, columns[f], N, p, dst, acc, s);
        if (!rc && m) rc = launch_masked_accumulate(ctx, buf, tmp, m, N, G, started ? nullptr : prior, started ? 1 : 0, s);
        if (rc) return rc;
        started = true;
    }
    if (assign) return launch_sample_scores(ctx, buf, N, G, u, assign, s);
    if (logp) return launch_logp_scores(ctx, buf, N, G, logp, s);
    return DIST_B200_OK;
}

int dist_b200_score_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                 const void *const *columns_dev, size_t n_rows, const float *prior_dev, float *scores_dev,
                                 int accumulate, const uint32_t *const *observed_dev, void *stream) {
    if (!scores_dev) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "score_batch: scores_dev is null") : DIST_B200_ERR_INVALID;
    return score_dispatch(ctx, features, n_features, columns_dev, observed_dev, n_rows, prior_dev, nullptr, nullptr, scores_dev,
                          accumulate, as_stream(stream));
}

int dist_b200_score_sample_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                        const void *const *columns_dev, size_t n_rows, const float *prior_dev,
                                        const float *u_dev, int32_t *assign_dev, float *scores_dev,
                                        const uint32_t *const *observed_dev, void *stream) {
    if (!assign_dev) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "score_sample_batch: assign_dev is null") : DIST_B200_ERR_INVALID;
    return score_dispatch(ctx, features, n_features, columns_dev, observed_dev, n_rows, prior_dev, u_dev, assign_dev, scores_dev, 0,
                          as_stream(stream));
}

int dist_b200_score_logp_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                      const void *const *columns_dev, size_t n_rows, const float *prior_dev, float *logp_dev,
                                      const uint32_t *const *observed_dev, void *stream) {
    if (!logp_dev) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "score_logp_batch: logp_dev is null") : DIST_B200_ERR_INVALID;
    return score_dispatch(ctx, features, n_features, columns_dev, observed_dev, n_rows, prior_dev, nullptr, nullptr, nullptr, 0,
                          as_stream(stream), logp_dev);
}

int dist_b200_score_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                          const void *const *columns_dev, size_t n_rows, const float *prior_dev, float *scores_dev,
                          int accumulate, void *stream) {
    if (!scores_dev) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "score_batch: scores_dev is null") : DIST_B200_ERR_INVALID;
    return score_dispatch(ctx, features, n_features, columns_dev, nullptr, n_rows, prior_dev, nullptr, nullptr, scores_dev,
                          accumulate, as_stream(stream));
}

int dist_b200_score_sample_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                 const void *const *columns_dev, size_t n_rows, const float *prior_dev,
                                 const float *u_dev, int32_t *assign_dev, float *scores_dev, void *stream) {
    if (!assign_dev) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "score_sample_batch: assign_dev is null") : DIST_B200_ERR_INVALID;
    return score_dispatch(ctx, features, n_features, columns_dev, nullptr, n_rows, prior_dev, u_dev, assign_dev, scores_dev, 0,
                          as_stream(stream));
}

int dist_b200_score_logp_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                               const void *const *columns_dev, size_t n_rows, const float *prior_dev, float *logp_dev,
                               void *stream) {
    if (!logp_dev) return ctx ? fail(ctx, DIST_B200_ERR_INVALID, "score_logp_batch: logp_dev is null") : DIST_B200_ERR_INVALID;
    return score_dispatch(ctx, features, n_features, columns_dev, nullptr, n_rows, prior_dev, nullptr, nullptr, nullptr, 0,
                          as_stream(stream), logp_dev);
}

int dist_b200_logp_from_scores(dist_b200_ctx *ctx, const float *scores_dev, size_t n_rows, int G, float *logp_dev,
                               void *stream) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    if (!scores_dev || !logp_dev || G < 1) return fail(ctx, DIST_B200_ERR_INVALID, "logp_from_scores: null buffer or G < 1");
    return launch_logp_scores(ctx, scores_dev, n_rows, G, logp_dev, as_stream(stream));
}

int dist_b200_sample_from_scores(dist_b200_ctx *ctx, const float *scores_dev, size_t n_rows, int G,
                                 const float *u_dev, int32_t *assign_dev, void *stream) {
    if (!ctx || !scores_dev || !u_dev || !assign_dev || G < 1) return DIST_B200_ERR_INVALID;
    return launch_sample_scores(ctx, scores_dev, n_rows, G, u_dev, assign_dev, as_stream(stream));
}

int dist_b200_peer_alloc(dist_b200_ctx *ctx, size_t bytes, void **dev_ptr, unsigned char handle_out[64]) {
    if (!ctx || !dev_ptr || !handle_out || bytes == 0) return DIST_B200_ERR_INVALID;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    DISTB200_CUDA(ctx, cudaMalloc(dev_ptr, bytes));
    DISTB200_CUDA(ctx, cudaMemset(*dev_ptr, 0, bytes));  // epoch flags start at 0
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, *dev_ptr);
    if (e != cudaSuccess) {
        cudaFree(*dev_ptr);
        *dev_ptr = nullptr;
        return fail(ctx, DIST_B200_ERR_CUDA, std::string("cudaIpcGetMemHandle: ") + cudaGetErrorString(e));
    }
    std::memcpy(handle_out, &h, 64);
    return DIST_B200_OK;
}

int dist_b200_peer_open(dist_b200_ctx *ctx, const unsigned char handle[64], void **dev_ptr) {
    if (!ctx || !handle || !dev_ptr) return DIST_B200_ERR_INVALID;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, handle, 64);
    DISTB200_CUDA(ctx, cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return DIST_B200_OK;
}

int dist_b200_peer_close(dist_b200_ctx *ctx, void *dev_ptr) {
    if (!ctx || !dev_ptr) return DIST_B200_ERR_INVALID;
    DISTB200_CUDA(ctx, cudaIpcCloseMemHandle(dev_ptr));
    return DIST_B200_OK;
}

int dist_b200_peer_free(dist_b200_ctx *ctx, void *dev_ptr) {
    if (!ctx || !dev_ptr) return DIST_B200_ERR_INVALID;
    DISTB200_CUDA(ctx, cudaDeviceSynchronize());
    DISTB200_CUDA(ctx, cudaFree(dev_ptr));
    return DIST_B200_OK;
}

int dist_b200_score_push_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F,
                               const void *const *columns_dev, size_t n_rows, size_t row0, const float *prior_dev,
                               void *const *slot_ptrs, int n_owners, size_t block_rows, void *stream) {
    if (!ctx || !features || !columns_dev || F < 1 || !slot_ptrs || n_owners < 1 || block_rows == 0) return DIST_B200_ERR_INVALID;
    if (n_owners > kMaxPushOwners) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "score_push: more than 16 owners");
    if (F > kMaxFeatures) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "score_push: more than 512 features in one call");
    const int G = features[0] ? features[0]->G : 0;
    if (G < 1) return fail(ctx, DIST_B200_ERR_STATE, "score_push: feature 0 has no groups");
    if ((row0 + n_rows + block_rows - 1) / block_rows > static_cast<size_t>(n_owners))
        return fail(ctx, DIST_B200_ERR_INVALID, "score_push: rows extend past the last owner's block");
    cudaStream_t s = as_stream(stream);
    int rc = wait_ready(ctx, features, F, s);
    if (rc) return rc;
    for (int f = 0; f < F; ++f) {
        if (!features[f] || !columns_dev[f] || features[f]->ctx != ctx || features[f]->G != G)
            return fail(ctx, DIST_B200_ERR_INVALID, "score_push: bad feature list");
        if (solo(features[f])) return fail(ctx, DIST_B200_ERR_UNSUPPORTED, "score_push: row-mapped models only");
    }
    // multi for a list of one too: a lone GammaPoisson shard is scored through its value table
    FeatList fl;
    if ((rc = build_list(ctx, features, F, columns_dev, nullptr, true, fl, nullptr, s))) return rc;
    PushTargets pt{};
    pt.n = n_owners;
    pt.row0 = row0;
    pt.block_rows = block_rows;
    for (int i = 0; i < n_owners; ++i) pt.ptr[i] = static_cast<float *>(slot_ptrs[i]);
    return launch_score_rows(ctx, fl, G, n_rows, prior_dev, nullptr, nullptr, nullptr, 0, s, &pt);
}

int dist_b200_sample_from_slots(dist_b200_ctx *ctx, const float *slots_dev, int n_slots, size_t slot_stride,
                                size_t n_rows, int G, const float *u_dev, int32_t *assign_dev, void *stream) {
    if (!ctx || !slots_dev || n_slots < 1 || !u_dev || !assign_dev || G < 1) return DIST_B200_ERR_INVALID;
    return launch_sample_scores(ctx, slots_dev, n_rows, G, u_dev, assign_dev, as_stream(stream), n_slots, slot_stride);
}

// The host-buffer form of score_dispatch.  Its per-row output is 4 bytes: the sampled group (u_host and assign_host given)
// or the row's log-normaliser (logp_host given, no u).
static int score_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F, const void *const *columns_host, size_t N,
                      const float *prior_host, const float *u_host, int32_t *assign_host, float *logp_host, float *scores_host) {
    void *out_host = logp_host ? static_cast<void *>(logp_host) : static_cast<void *>(assign_host);
    for (int f = 0; f < F; ++f)
        if (!features[f] || !columns_host[f]) return fail(ctx, DIST_B200_ERR_INVALID, "score_sample_host: null feature / column");
    const int G = features[0]->G;
    if (G < 1) return fail(ctx, DIST_B200_ERR_STATE, "score_sample_host: no groups");
    if (N == 0) return DIST_B200_OK;
    // Row chunks are pipelined over two streams: the H2D copy of chunk k+1 and the D2H copy of chunk
    // k-1 overlap the kernels of chunk k (rows are independent given frozen statistics).
    cudaStream_t st[2] = {ctx->own_stream, ctx->own_stream2};
    Staging stage(ctx, st[0], st[1]);
    // layout of the staging area (identical in the page-locked mirror and on the device):
    //   columns | prior | u (sampling only) | per-row output | scores (optional, device only + host out)
    std::vector<size_t> col_off(F);
    for (int f = 0; f < F; ++f) col_off[f] = stage.region(value_bytes(features[f]) * N);
    const size_t prior_off = stage.region(sizeof(float) * G);
    const size_t u_off = stage.region(u_host ? sizeof(float) * N : 0);
    const size_t out_off = stage.region(sizeof(int32_t) * N);
    const size_t scores_off = stage.region(scores_host ? sizeof(float) * N * G : 0);
    int rc;
    if ((rc = stage.reserve(scores_off))) return rc;
    // A caller buffer that is already page-locked (cudaHostAlloc / cudaHostRegister / torch pin_memory)
    // is copied from / to directly; pageable buffers go through the context's pinned staging area.
    auto is_pinned = [](const void *p) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
            cudaGetLastError();
            return false;
        }
        return at.type == cudaMemoryTypeHost;
    };
    std::vector<char> col_pinned(F);
    for (int f = 0; f < F; ++f) col_pinned[f] = is_pinned(columns_host[f]) ? 1 : 0;
    const bool u_pinned = !u_host || is_pinned(u_host), out_pinned = is_pinned(out_host);

    // per-row output of rows [lo, lo + n) at `out` (device / mapped), u of those rows at `uu`
    auto dispatch = [&](const void *const *cols, size_t n, const float *pr, const float *uu, char *out, float *sc, cudaStream_t str) {
        return score_dispatch(ctx, features, F, cols, nullptr, n, pr, uu, logp_host ? nullptr : reinterpret_cast<int32_t *>(out), sc, 0, str,
                              logp_host ? reinterpret_cast<float *>(out) : nullptr);
    };

    if ((rc = wait_ready(ctx, features, F, st[0]))) return rc;
    if ((rc = refresh_gp_tables(ctx, features, F, st[0]))) return rc;  // before the second stream starts reading them
    // the prior vector is re-read per table row by the dpd / dd kernels: it goes to the device on every route
    const float *prior_dev = prior_host ? stage.dev<const float>(prior_off) : nullptr;
    if (prior_host && (rc = stage.put(prior_off, prior_host, sizeof(float) * G, st[0], true))) return rc;
    // Zero-copy: when every caller buffer is page-locked, the kernels read the rows straight from host memory and write
    // the assignments straight back (device-accessible under unified addressing): ONE launch, the PCIe transfers overlap
    // the math row tile by row tile with no chunking, no staging copies and no second stream.
    // DIST_B200_OPT_HOST_ZEROCOPY: 0 = when all buffers are page-locked, 1 = never, 2 = same as 0 (A/B runs).
    {
        bool all_pinned = u_pinned && out_pinned && !scores_host;
        for (int f = 0; f < F; ++f) all_pinned = all_pinned && col_pinned[f];
        // niw keeps the staged path: its row images are built by a separate pack kernel, which would read the rows over
        // PCIe without any math to hide behind (measured: c5 e2e 6.1e10 staged vs 4.1e10 zero-copy)
        bool staged_only = ctx->opt[DIST_B200_OPT_HOST_ZEROCOPY] == 1;
        for (int f = 0; f < F; ++f) staged_only = staged_only || features[f]->model == DIST_B200_NIW;
        if (all_pinned && !staged_only) {
            std::vector<const void *> zc_cols(F);
            void *dp = nullptr;
            bool ok = true;
            for (int f = 0; f < F && ok; ++f) {
                ok = cudaHostGetDevicePointer(&dp, const_cast<void *>(columns_host[f]), 0) == cudaSuccess;
                zc_cols[f] = dp;
            }
            const float *u_zc = nullptr;
            if (ok && u_host) {
                ok = cudaHostGetDevicePointer(&dp, const_cast<float *>(u_host), 0) == cudaSuccess;
                u_zc = static_cast<const float *>(dp);
            }
            if (ok) ok = cudaHostGetDevicePointer(&dp, out_host, 0) == cudaSuccess;
            char *out_zc = static_cast<char *>(dp);
            if (ok) {
                if ((rc = dispatch(zc_cols.data(), N, prior_dev, u_zc, out_zc, nullptr, st[0]))) return rc;
                return stage.drain();
            }
            cudaGetLastError();  // not mappable: fall through to the staged path
        }
    }
    if ((rc = wait_ready(ctx, features, F, st[1]))) return rc;
    if (prior_host) {
        DISTB200_CUDA(ctx, cudaEventRecord(ctx->ev, st[0]));
        DISTB200_CUDA(ctx, cudaStreamWaitEvent(st[1], ctx->ev, 0));
    }
    const size_t min_chunk = 32768;
    // five chunks measured best at 1M rows (DIST_B200_OPT_HOST_CHUNKS overrides it for A/B runs)
    const size_t max_chunks = ctx->opt[DIST_B200_OPT_HOST_CHUNKS] > 0 ? static_cast<size_t>(ctx->opt[DIST_B200_OPT_HOST_CHUNKS]) : 5;
    size_t nchunks = std::min<size_t>(max_chunks, std::max<size_t>(1, N / min_chunk));
    // niw launches share the context's packed-row buffer and mixed dpd lists (and a dpd logp, which may materialise) its
    // single scores buffer: their kernels stay on ONE stream in chunk order; only the H2D copies of the later chunks run
    // ahead on the second stream
    bool one_compute_stream = false;
    for (int f = 0; f < F; ++f)
        if (features[f]->model == DIST_B200_NIW || (features[f]->model == DIST_B200_DPD && (F > 1 || logp_host))) one_compute_stream = true;
    if (one_compute_stream && scores_host) nchunks = 1;
    // chunk boundaries: equal interior chunks, half-size first and last ones -- the first H2D copy and the
    // last D2H copy are the only transfers no kernel hides
    std::vector<size_t> bounds(1, 0);
    if (nchunks >= 4) {
        const size_t unit = round_up((N + 2 * (nchunks - 1) - 1) / (2 * (nchunks - 1)), 256);  // half an interior chunk
        size_t at = unit;
        while (at < N && bounds.size() < nchunks - 1) {
            bounds.push_back(at);
            at += 2 * unit;
        }
        const size_t last = N > unit ? (N - unit) / 256 * 256 : 0;  // 256-row aligned like every other boundary
        if (last > bounds.back()) bounds.push_back(last);
    } else {
        const size_t chunk = round_up((N + nchunks - 1) / nchunks, 256);
        for (size_t at = chunk; at < N; at += chunk) bounds.push_back(at);
    }
    bounds.push_back(N);
    // with more than one chunk, one compute stream takes the copies on the second stream and the kernels on the first
    one_compute_stream = one_compute_stream && bounds.size() > 2;
    std::vector<const void *> cols(F);
    for (size_t k = 0; k + 1 < bounds.size(); ++k) {
        const size_t lo = bounds[k], n = bounds[k + 1] - lo;
        const cudaStream_t cs = one_compute_stream ? st[1] : st[k & 1], ks = one_compute_stream ? st[0] : st[k & 1];
        for (int f = 0; f < F; ++f) {
            const size_t vb = value_bytes(features[f]), at = col_off[f] + vb * lo;
            if ((rc = stage.put(at, static_cast<const char *>(columns_host[f]) + vb * lo, vb * n, cs, !col_pinned[f]))) return rc;
            cols[f] = stage.dev(at);
        }
        if (u_host && (rc = stage.put(u_off + 4 * lo, u_host + lo, 4 * n, cs, !u_pinned))) return rc;
        if (cs != ks) {
            DISTB200_CUDA(ctx, cudaEventRecord(ctx->ev, cs));
            DISTB200_CUDA(ctx, cudaStreamWaitEvent(ks, ctx->ev, 0));
        }
        if ((rc = dispatch(cols.data(), n, prior_dev, u_host ? stage.dev<const float>(u_off) + lo : nullptr, stage.dev(out_off + 4 * lo),
                           scores_host ? stage.dev<float>(scores_off) + lo * G : nullptr, ks)) ||
            (rc = stage.get(static_cast<char *>(out_host) + 4 * lo, out_off + 4 * lo, 4 * n, ks, !out_pinned)) ||
            (scores_host && (rc = stage.get(scores_host + lo * G, scores_off + sizeof(float) * lo * G, sizeof(float) * n * G, ks))))
            return rc;
    }
    if ((rc = stage.drain())) return rc;
    if (!out_pinned) std::memcpy(out_host, stage.pin(out_off), 4 * N);
    return DIST_B200_OK;
}

int dist_b200_score_sample_batch_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F,
                                      const void *const *columns_host, size_t N, const float *prior_host,
                                      const float *u_host, int32_t *assign_host, float *scores_host) {
    if (!ctx || !features || !columns_host || F < 1 || F > kMaxFeatures || !u_host || !assign_host) return DIST_B200_ERR_INVALID;
    return score_host(ctx, features, F, columns_host, N, prior_host, u_host, assign_host, nullptr, scores_host);
}

int dist_b200_score_logp_batch_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int F,
                                    const void *const *columns_host, size_t N, const float *prior_host, float *logp_host) {
    if (!ctx) return DIST_B200_ERR_INVALID;
    if (!features || !columns_host || F < 1 || F > kMaxFeatures || !logp_host)
        return fail(ctx, DIST_B200_ERR_INVALID, "score_logp_batch_host: null argument");
    return score_host(ctx, features, F, columns_host, N, prior_host, nullptr, nullptr, logp_host, nullptr);
}

int dist_b200_host_register(dist_b200_ctx *ctx, void *ptr, size_t bytes) {
    if (!ctx || !ptr || bytes == 0) return DIST_B200_ERR_INVALID;
    DISTB200_CUDA(ctx, cudaSetDevice(ctx->device));
    const cudaError_t e = cudaHostRegister(ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
    if (e == cudaErrorHostMemoryAlreadyRegistered) {
        cudaGetLastError();
        return DIST_B200_OK;
    }
    if (e != cudaSuccess) return fail(ctx, DIST_B200_ERR_CUDA, std::string("cudaHostRegister: ") + cudaGetErrorString(e));
    return DIST_B200_OK;
}

int dist_b200_host_unregister(dist_b200_ctx *ctx, void *ptr) {
    if (!ctx || !ptr) return DIST_B200_ERR_INVALID;
    DISTB200_CUDA(ctx, cudaSetDevice(ctx->device));
    DISTB200_CUDA(ctx, cudaDeviceSynchronize());  // no kernel may still be reading the range
    const cudaError_t e = cudaHostUnregister(ptr);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(ctx, DIST_B200_ERR_INVALID, std::string("cudaHostUnregister: ") + cudaGetErrorString(e));
    }
    return DIST_B200_OK;
}

int dist_b200_score_value_host(dist_b200_ctx *ctx, const dist_b200_feature *feature, const void *value_host,
                               float *scores_accum_host) {
    if (!ctx || !feature || !value_host || !scores_accum_host) return DIST_B200_ERR_INVALID;
    const int G = feature->G;
    if (G < 1) return fail(ctx, DIST_B200_ERR_STATE, "score_value: no groups");
    const size_t vb = value_bytes(feature);
    // zero-copy through the context's page-locked area (device-accessible under unified addressing): the kernel reads
    // the value from host memory and writes the G scores back to it, so a call is ONE launch + one synchronise instead
    // of two H2D copies, a launch and a D2H copy; the accumulation into the caller's (pageable) buffer is done here
    int rc = ensure_pinned(ctx, round_up(vb, 256) + sizeof(float) * G + 256);
    if (rc) return rc;
    char *pin = static_cast<char *>(ctx->pinned);
    float *sc = reinterpret_cast<float *>(pin + round_up(vb, 256));
    cudaStream_t s = ctx->own_stream;
    if ((rc = wait_ready(ctx, &feature, 1, s))) return rc;
    std::memcpy(pin, value_host, vb);
    const void *col = pin;
    rc = score_dispatch(ctx, &feature, 1, &col, nullptr, 1, nullptr, nullptr, nullptr, sc, 0, s);
    if (rc) return rc;
    DISTB200_CUDA(ctx, cudaStreamSynchronize(s));
    for (int g = 0; g < G; ++g) scores_accum_host[g] += sc[g];  // MixtureSlave::score_value accumulates (mixture.hpp:416-425)
    return DIST_B200_OK;
}

int dist_b200_numerics_probe(dist_b200_ctx *ctx, int fn, size_t n, const float *in_dev, float *out_dev, void *stream) {
    if (!ctx || !in_dev || !out_dev) return DIST_B200_ERR_INVALID;
    return launch_numerics_probe(ctx, fn, n, in_dev, out_dev, as_stream(stream));
}

}  // extern "C"
