// common.cuh -- shared host/device declarations of the B200 mixture-scoring library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/dist_b200.h"
#include "numerics.cuh"

namespace distb200 {

constexpr int kMaxPushOwners = 16;  // ranks of one NVLink domain a feature-sharded launch can push to
constexpr int kMaxFeatures = 512;  // feature descriptors travel in kernel-parameter space (20 KB)

// device view of one feature, consumed by the row-mapped score kernel
struct FeatDesc {
    const void *params;  // nich/gp/bb: float4[G]; dd: float[G][vdim]; dpd: float[(V+1)][G]
    const void *column;  // value column, N entries
    int kind;            // dist_b200_model, or kKindGpTable
    int vdim;            // dd: dim; gp table: kGpTableX
    const void *aux;     // gp table: the float4 caches, for values >= kGpTableX
    int cap;             // gp table: groups allocated = row stride of the transposed copy [kGpTableX][cap] that follows the table
    int pad_;
};

// internal kind: GammaPoisson scored through a per-(group, value) table for small counts
constexpr int kKindGpTable = 16;  // (6 is DIST_B200_BNB)
constexpr int kGpTableX = 32;

// destinations of a peer-push launch (see RowsArgs)
struct PushTargets {
    int n;
    size_t row0, block_rows;
    float *ptr[kMaxPushOwners];
};

struct FeatList {
    int n;
    FeatDesc f[kMaxFeatures];
};

// observed masks of a feature list: m[f] is NULL (feature f fully observed) or ceil(N / 32) words, bit n % 32 of word
// n / 32 set when row n's cell of feature f is observed (a separate kernel parameter: FeatList's layout is unchanged)
struct MaskList {
    const uint32_t *m[kMaxFeatures];
};

// GammaPoisson value tables of many features rebuilt in one launch (grid.y = feature)
constexpr int kGpTableBatch = 128;
struct GpTableBatch {
    int n;
    int n_groups[kGpTableBatch];
    const float4 *params[kGpTableBatch];
    float *table[kGpTableBatch];
};

// batched Group::add_value over the pooled-statistics models (nich / gp / bb) of one kind: up to
// kAddBatch features per launch, descriptors in kernel-parameter space
constexpr int kAddBatch = 128;
struct AddDesc {
    const void *column;          // value column, N entries
    uint32_t *st0, *st1, *st2;   // stored statistics (nich: count|mean|ctv, gp: count|sum, bb: heads|tails)
    float4 *params;              // hot caches, rebuilt after the merge
    float *aux;                  // nich: unscaled log_coeff_
    float shared[4];             // hyper-parameters
    int model, pad;
};
struct AddBatch {
    int n, G;
    int sign;                    // +1: add_value, -1: remove_value
    size_t N;
    const int32_t *assign;
    char *acc;                   // per feature: cnt_a[G] | cnt_b[G] (int) | sum_x[G] | sum_xx[G] (double)
    size_t acc_stride;           // bytes per feature
    const double *xchg;          // merge from an exchanged [feature][4][G] double buffer instead of acc (multi-GPU)
    int xchg_first;              // index of d[0] in that buffer
    AddDesc d[kAddBatch];
};
// observed masks of an AddBatch's features (dist_b200.h, missing cells): m[f] for d[f], NULL = fully observed.  A
// separate kernel parameter of the masked kernels, so AddBatch keeps its layout.
struct AddMasks {
    const uint32_t *m[kAddBatch];
};

}  // namespace distb200

struct dist_b200_ctx {
    int device = 0;
    int sm_count = 0;
    std::string last_error;
    distb200::NumericTables tables{};
    float *tables_storage = nullptr;  // one allocation backing `tables`
    // scratch for the host-buffer entry points
    void *pinned = nullptr;
    size_t pinned_bytes = 0;
    void *scratch_dev = nullptr;
    size_t scratch_bytes = 0;
    void *xpack = nullptr;            // niw tensor path: rows packed into A-operand images
    size_t xpack_bytes = 0;
    float *bbt = nullptr;             // kSub cross-cat kernel: compact [heads | tails] rows of the list's BetaBernoulli features
    size_t bbt_bytes = 0;
    void *scores_scratch = nullptr;   // [N][G] buffer of the materialising dispatch paths
    size_t scores_scratch_bytes = 0;
    void *missing_scratch = nullptr;  // masked entries: per-feature [N] assignments, or one feature's [N][G] scores
    size_t missing_scratch_bytes = 0;
    cudaStream_t own_stream = nullptr, own_stream2 = nullptr;
    cudaEvent_t ev = nullptr;
    void *add_acc = nullptr;          // batched add_value: per-feature accumulators (stats.cu)
    size_t add_acc_bytes = 0;
    cudaEvent_t add_done = nullptr;   // recorded after the last merge that read add_acc
    int opt[DIST_B200_OPT_COUNT_] = {0};  // dist_b200_ctx_set_option: A/B knobs of bench.py / the profiling scripts
};

struct dist_b200_feature {
    dist_b200_ctx *ctx = nullptr;
    int model = 0;
    int G = 0;          // packed group count
    int capacity = 0;   // groups allocated in the hot caches (params, aux, gp_table, log_prod_dev)
    int dim = 0;        // dd: dim, dpd: V, niw: d
    // scalar hyper-parameters of the last update_all (needed by update_group / add_group): nich mu kappa sigmasq nu;
    // gp alpha inv_beta; bnb alpha beta r; bb alpha beta; dpd alpha beta0; niw kappa nu
    float shared[4] = {0, 0, 0, 0};
    std::vector<float> alphas;        // host copy of alphas_dev
    std::vector<uint32_t> keys;       // dpd keys as given to update_all (the order of the counts columns)
    bool keys_dense = false;          // dpd: keys == 0..V-1
    float alpha_sum = 0;              // dd
    // device buffers
    void *params = nullptr;           // hot layout (see FeatDesc::params)
    size_t params_bytes = 0;
    float *aux = nullptr;             // nich: unscaled log_coeff_ per group (capacity floats)
    size_t aux_bytes = 0;
    float *gp_table = nullptr;        // gp: [capacity][kGpTableX] tabulated terms for values < kGpTableX
    size_t gp_table_bytes = 0;
    bool gp_table_dirty = true;
    cudaEvent_t ready = nullptr;      // recorded after every cache mutation; scoring streams wait on it
    // device-resident raw group statistics (mirror of the host Groups; the state that batched add_value updates in
    // place): stat_arrays arrays in update_all's argument order, each holding stats_cap groups of stat_elems 4-byte
    // elements
    //   nich: count | mean | count_times_variance     gp, bnb: count | sum     bb: heads | tails
    //   dd: counts[dim]     dpd: counts[V]     niw: count | sum_x[d] | sum_xxT[d][d]
    uint32_t *stats[3] = {nullptr, nullptr, nullptr};
    size_t stats_bytes[3] = {0, 0, 0};
    int stats_cap = 0;
    float *alphas_dev = nullptr;      // the Shared vector: dd alphas, dpd betas, niw mu[d] | psi[d][d]
    size_t alphas_bytes = 0;
    float *log_prod_dev = nullptr;    // gp: Group::log_prod per group (read by score_data only)
    size_t log_prod_bytes = 0;
    bool log_prod_valid = false;      // cleared by every statistics mutation that does not maintain it
    float *dpd_hot = nullptr;         // dpd: per-call scratch of table_rows.cu (the table with prior / row max folded in)
    size_t dpd_hot_bytes = 0;
    float *cdf_buf = nullptr;         // dpd / dd / bb: per-value CDF trees (rebuilt per scoring call: they carry the prior)
    size_t cdf_bytes = 0;
    uint32_t *keys_dev = nullptr;     // dpd sorted keys
    size_t keys_bytes = 0;
    int *key_rows_dev = nullptr;      // dpd: table row of sorted key i
    size_t key_rows_bytes = 0;
    // niw
    float *niw_buf = nullptr;         // per-group records (posterior, whitening matrix, constants)
    size_t niw_bytes = 0;
    float *niw_tc = nullptr;          // d = 32 and 32 < d <= 128: tensor-core operand images, b vectors, constants
    size_t niw_tc_bytes = 0;
    void *sample_buf = nullptr;       // sample_values: per-group records of the prep pass (sample_values.cu)
    size_t sample_bytes = 0;
};

namespace distb200 {

inline int fail(dist_b200_ctx *ctx, int code, const std::string &msg) {
    if (ctx) ctx->last_error = msg;
    return code;
}

#define DISTB200_CUDA(ctx, call)                                                                   \
    do {                                                                                           \
        cudaError_t e__ = (call);                                                                  \
        if (e__ != cudaSuccess)                                                                    \
            return ::distb200::fail((ctx), DIST_B200_ERR_CUDA,                                     \
                                    std::string(#call) + ": " + cudaGetErrorString(e__));          \
    } while (0)

// Grow-only device buffer: when `bytes` exceeds the allocation `have`, `buf` is replaced by an allocation of `bytes`.
// The first `keep` bytes of the old contents move over, and with `zero` the rest is zero-filled.  The device is
// synchronised before the old buffer is freed: kernels on any stream may still read it.
template <class T>
int grow(dist_b200_ctx *ctx, T *&buf, size_t &have, size_t bytes, size_t keep = 0, bool zero = false) {
    if (bytes <= have) return DIST_B200_OK;
    if (buf) DISTB200_CUDA(ctx, cudaDeviceSynchronize());
    if (buf && !keep) {  // freed first: the peak use stays one buffer
        DISTB200_CUDA(ctx, cudaFree(buf));
        buf = nullptr;
        have = 0;
    }
    void *fresh = nullptr;
    DISTB200_CUDA(ctx, cudaMalloc(&fresh, bytes));
    if (zero) DISTB200_CUDA(ctx, cudaMemset(static_cast<char *>(fresh) + keep, 0, bytes - keep));
    if (buf) DISTB200_CUDA(ctx, cudaMemcpy(fresh, buf, keep, cudaMemcpyDeviceToDevice));
    // the fill and the copy run on the legacy stream: they complete before any stream uses the buffer
    if (buf || zero) DISTB200_CUDA(ctx, cudaDeviceSynchronize());
    if (buf) DISTB200_CUDA(ctx, cudaFree(buf));
    buf = static_cast<T *>(fresh);
    have = bytes;
    return DIST_B200_OK;
}

// ---- kernel launchers implemented in the .cu files --------------------------------------------
// prep.cu
int launch_nich_prep(dist_b200_ctx *ctx, const float shared[4], int G, int g0, int n, const int32_t *count_dev,
                     const float *mean_dev, const float *ctv_dev, float4 *params, float *aux, cudaStream_t s);
int launch_gp_prep(dist_b200_ctx *ctx, const float shared[2], int g0, int n, const uint32_t *count_dev,
                   const uint32_t *sum_dev, float4 *params, cudaStream_t s);
int launch_bnb_prep(dist_b200_ctx *ctx, const float shared[3], int g0, int n, const uint32_t *count_dev,
                    const uint32_t *sum_dev, float4 *params, cudaStream_t s);
int launch_bb_prep(dist_b200_ctx *ctx, const float shared[2], int g0, int n, const int32_t *heads_dev,
                   const int32_t *tails_dev, float4 *params, cudaStream_t s);
int launch_dd_prep(dist_b200_ctx *ctx, int dim, const float *alphas_dev, float alpha_sum, int g0, int n,
                   const int32_t *counts_dev, float *table, cudaStream_t s);
int launch_dpd_prep(dist_b200_ctx *ctx, float alpha, float beta0, int V, const float *betas_dev, int G,
                    const int32_t *counts_dev, float *table, cudaStream_t s);
int launch_dpd_update_group(dist_b200_ctx *ctx, float alpha, float beta0, int V, const float *betas, int G, int g,
                            const int32_t *counts_row, float *table, cudaStream_t s);
int launch_prior_prep(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *sizes_dev, float *prior,
                      cudaStream_t s);
int launch_low_entropy_prep(dist_b200_ctx *ctx, int dataset_size, int G, const int32_t *sizes_dev, float *prior,
                            cudaStream_t s);
int launch_numerics_probe(dist_b200_ctx *ctx, int fn, size_t n, const float *in, float *out, cudaStream_t s);
// score_data_grid: log marginal likelihood of all groups under n_grid packed Shareds (acc: n_grid doubles of scratch)
int launch_score_data(dist_b200_ctx *ctx, const dist_b200_feature *f, const uint32_t *st0, const uint32_t *st1,
                      const uint32_t *st2, const float *betas, const float *log_prod, const float *shareds_dev,
                      size_t n_grid, size_t stride, double *acc, float *out_dev, cudaStream_t s);
int launch_unpack_caches(dist_b200_ctx *ctx, const dist_b200_feature *f, float *out_dev, cudaStream_t s);

// score_rows.cu: rows mapped to lanes, groups looped (nich / gp / bb / small-dim dd, any F).  logp != nullptr (with
// assign = scores = nullptr): logp[n] = log sum_g exp(prior[g] + scores of row n)
int launch_score_rows(dist_b200_ctx *ctx, const FeatList &feats, int G, size_t N, const float *prior,
                      const float *u, int32_t *assign, float *scores, int accumulate, cudaStream_t s,
                      const PushTargets *push = nullptr, float *logp = nullptr);
int launch_gp_table_batch(dist_b200_ctx *ctx, const GpTableBatch &b, cudaStream_t s);
// score_rows_masked*.cu: the feature-list kernel with missing cells (every feature row-mapped; assign, scores or logp)
int launch_score_rows_masked(dist_b200_ctx *ctx, const FeatList &feats, const MaskList &masks, int G, size_t N,
                             const float *prior, const float *u, int32_t *assign, float *scores, int accumulate,
                             float *logp, cudaStream_t s);
// missing.cu: out[n] = assign[n] where row n's bit equals `keep` (1: observed cells, 0: missing cells), else -1
int launch_mask_assign(dist_b200_ctx *ctx, const int32_t *assign, const uint32_t *observed, size_t N, int keep, int32_t *out,
                       cudaStream_t s);
// scores[n][g] = base + (bit of row n ? tmp[n][g] : 0), base = scores[n][g] (accumulate) or prior[g] (or 0 without a prior)
int launch_masked_accumulate(dist_b200_ctx *ctx, float *scores, const float *tmp, const uint32_t *observed, size_t N, int G,
                             const float *prior, int accumulate, cudaStream_t s);
// stats.cu: batched Group::add_value (segmented reduction of assigned rows into the device-side statistics)
// pooled models: accumulate `b.n` features in one launch (b.acc zeroed by the launcher), then merge + rebuild caches
int launch_add_rows_pooled(dist_b200_ctx *ctx, const AddBatch &b, cudaStream_t s, const AddMasks *masks = nullptr);
int launch_merge_prep_batch(dist_b200_ctx *ctx, const AddBatch &b, cudaStream_t s);  // prep.cu
int launch_pack_accumulators(dist_b200_ctx *ctx, const AddBatch &b, double *xchg, cudaStream_t s);  // prep.cu
// dd / dpd: counts updated in place
int launch_add_rows_counts(dist_b200_ctx *ctx, dist_b200_feature *f, const void *column, const int32_t *assign, size_t N,
                           int sign, cudaStream_t s, int32_t *dst = nullptr, const uint32_t *observed = nullptr);
int launch_counts_to_doubles(dist_b200_ctx *ctx, const int32_t *src, double *dst, size_t n, cudaStream_t s);
int launch_merge_counts(dist_b200_ctx *ctx, int32_t *counts, const double *delta, size_t n, int sign, cudaStream_t s);
size_t add_rows_acc_bytes(int G);
int launch_count_assignments(dist_b200_ctx *ctx, const int32_t *assign, size_t N, int G, int32_t *counts, int accumulate,
                             cudaStream_t s, const uint32_t *observed = nullptr);
// gather_rows.cu: one warp per row, groups mapped to lanes (value-major tables: dpd, wide dd) and the
// stand-alone sampler over materialised scores
int launch_gather_rows(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *column, size_t N,
                       const float *prior, const float *u, int32_t *assign, float *scores, int accumulate,
                       cudaStream_t s);
int launch_sample_scores(dist_b200_ctx *ctx, const float *scores, size_t N, int G, const float *u,
                         int32_t *assign, cudaStream_t s, int n_slots = 1, size_t slot_stride = 0);
// logp[n] = log sum_g exp(scores[n][g]) over materialised [N][G] scores
int launch_logp_scores(dist_b200_ctx *ctx, const float *scores, size_t N, int G, float *logp, cudaStream_t s);
// table_rows.cu: single table feature (dpd / dd / bb)
size_t table_hot_floats(int R, int G);
int launch_table_rows(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *column, size_t N, const float *prior,
                      const float *u, int32_t *assign, cudaStream_t s);
size_t value_cdf_floats(int R, int G);
int launch_value_cdf(dist_b200_ctx *ctx, const dist_b200_feature *f, float *buf, const void *column, size_t N,
                     const float *prior, const float *u, int32_t *assign, cudaStream_t s);
// the logp form of the per-value shortcut: one log-normaliser per table row (`buf`: table rows floats), then a gather
int launch_value_logp(dist_b200_ctx *ctx, const dist_b200_feature *f, float *buf, const void *column, size_t N,
                      const float *prior, float *logp, cudaStream_t s);
// niw.cu
int niw_padded_dim(int d);
int launch_niw_prep(dist_b200_ctx *ctx, int d, const float *mu, float kappa, const float *psi, float nu, int G,
                    const int32_t *count, const float *sum_x, const float *sum_xxT, float *recs, cudaStream_t s);
int launch_niw_rows_small(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *values, size_t N, const float *prior,
                          const float *u, int32_t *assign, cudaStream_t s);
int launch_niw_scores(dist_b200_ctx *ctx, const dist_b200_feature *f, const void *values, size_t N,
                      const float *prior, float *scores, int accumulate, cudaStream_t s);
int launch_score_data_finish(dist_b200_ctx *ctx, size_t n_grid, const double *acc, float *out_dev, cudaStream_t s);  // prep.cu
// niw_stats.cu (batched add_value / remove_value and score_data on the resident statistics)
inline size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }
size_t niw_add_rows_bytes(int G, int d, size_t N);
int launch_niw_accumulate(dist_b200_ctx *ctx, int G, int d, const void *values, const int32_t *assign, size_t N, double *acc,
                          void *work, cudaStream_t s, const uint32_t *observed = nullptr);
int launch_niw_apply(dist_b200_ctx *ctx, int G, int d, int sign, const double *acc, int32_t *count, float *sum_x, float *sum_xxT,
                     cudaStream_t s);
int launch_niw_score_data(dist_b200_ctx *ctx, int G, int d, const int32_t *count, const float *sum_x, const float *sum_xxT,
                          const float *shareds_dev, size_t n_grid, size_t stride, double *acc, cudaStream_t s);
// niw_tc.cu (tcgen05 / TMEM path, d = 32)
size_t niw_tc_floats(int G);
int launch_niw_tc_prep(dist_b200_ctx *ctx, int G, const float *recs, float *tc_buf, cudaStream_t s);
// scores != nullptr: [N][G] scores (optionally accumulated onto the buffer); scores == nullptr: the fused sampler writes assign[N]
int launch_niw_tc(dist_b200_ctx *ctx, int G, const float *tc_buf, const void *values, size_t N, const float *prior,
                  float *scores, int accumulate, const float *u, int32_t *assign, cudaStream_t s);
// niw_tc_wide.cu (tcgen05 / TMEM path, 32 < d <= 128, materialising): per-stage operand images built from the records
size_t niw_tc_wide_floats(int G, int d);
int launch_niw_tc_wide_prep(dist_b200_ctx *ctx, int G, int d, const float *recs, float *tc_buf, cudaStream_t s);
// [N][G] scores of x - mu0 (mu0 = Shared.mu, the centre the records' b vectors were built around), optionally accumulated
int launch_niw_tc_wide(dist_b200_ctx *ctx, int G, int d, const float *tc_buf, const float *mu0, const void *values, size_t N,
                       const float *prior, float *scores, int accumulate, cudaStream_t s);

// sample_values.cu: batched Group::sample_value of one feature.  The device-resident statistics it reads:
struct SampleSrc {
    int model, G, dim;                // dim: dd dim / dpd V / niw d
    float shared[4];                  // nich mu kappa sigmasq nu; gp alpha inv_beta; bnb alpha beta r; bb alpha beta;
                                      // dpd alpha beta0; niw kappa nu
    const uint32_t *st0, *st1, *st2;  // statistics arrays (see dist_b200_feature::stats)
    const float *alphas;              // dist_b200_feature::alphas_dev
    const uint32_t *keys_sorted;      // dpd: dist_b200_feature::keys_dev / key_rows_dev
    const int *key_rows;
};
int launch_sample_values(dist_b200_ctx *ctx, dist_b200_feature *f, const SampleSrc &src, uint32_t position, const int32_t *assign,
                         size_t N, uint64_t seed, uint64_t row0, void *out, cudaStream_t s);

// wire.cu: protobuf wire format of the reference (schema.proto) -> SoA.  Decoded feature: Shared floats
// (+ dpd keys) and the statistics arrays in update_all's argument order.
struct WireFeature {
    std::vector<float> shared;     // nich 4; gp 2; bb 2; bnb 3 (alpha, beta, r); dd alphas[dim]; dpd gamma, alpha, beta0, betas[V]
    std::vector<uint32_t> keys;    // dpd: Shared.values; bnb: r (exact)
    std::vector<uint32_t> stats;   // arrays of G (x dim) 4-byte elements, floats as their bit patterns
    int dim = 0;                   // dd dim / dpd V
};
int wire_decode(dist_b200_ctx *ctx, int model, const void *shared_msg, size_t shared_len, const void *const *group_msgs,
                const size_t *group_lens, int G, WireFeature &out);
int wire_decode_clustering(dist_b200_ctx *ctx, const void *msg, size_t len, int *which, float *alpha, float *d,
                           uint64_t *dataset_size);
int wire_encode_shared(dist_b200_ctx *ctx, int model, const float *shared, size_t n_shared, const uint32_t *keys,
                       size_t n_keys, std::vector<uint8_t> &out);
int wire_encode_groups(dist_b200_ctx *ctx, int model, int G, int dim, const uint32_t *keys, const uint32_t *stats,
                       size_t stats_words, std::vector<uint8_t> &out, std::vector<size_t> &lens);

}  // namespace distb200
