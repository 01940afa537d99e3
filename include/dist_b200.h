/* dist_b200.h -- C-ABI of the B200-native mixture-scoring hot path.
 *
 * Drop-in boundary for ONE path of forcedotcom/distributions (reference paths are relative to
 * /root/reference): batched `Mixture::score_value` for every row against every group of the
 * conjugate component models, plus the clustering prior's group-size term, followed by
 * `sample_from_scores`.  The reference has no FFI of its own for this path (SURVEY.md §8b): the
 * seam is the C++ template contract `MixtureSlave<Model, DataScorer, ValueScorer>`
 * (include/distributions/mixture.hpp:340-450) and its Cython mirror
 * (distributions/lp/models/_nich.pyx:85-138).  Each entry point below names the reference
 * interface it replaces; INTEGRATION.md shows the binding a maintainer of the reference would add.
 *
 * Conventions
 *   - plain C types only; every call returns a dist_b200_status (0 = ok) and never aborts or
 *     throws across the boundary (the reference aborts / throws: common.hpp:49-67).
 *   - `*_dev` pointers are CUDA device pointers on the context's device, `*_host` / unmarked
 *     statistics pointers are host pointers.  `stream` is a cudaStream_t passed as void*
 *     (NULL = the legacy default stream).  Calls taking a stream are asynchronous on it unless
 *     they return data to the host.
 *   - a "feature" is the device-side MixtureValueScorer of one Model::Mixture: the per-group
 *     caches of one feature column for G groups.  Features that share a partition (one cross-cat
 *     "kind") are scored together: scores[n][g] = prior[g] + sum_f score_f(x[n][f]; group g).
 *   - there is NO CPU fallback: every scoring / sampling entry launches sm_100a kernels.
 */
#ifndef DIST_B200_H_
#define DIST_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIST_B200_ABI_VERSION 1

typedef enum {
    DIST_B200_OK = 0,
    DIST_B200_ERR_INVALID = 1,     /* bad argument (null, size, range) */
    DIST_B200_ERR_CUDA = 2,        /* a CUDA runtime call failed; see dist_b200_last_error */
    DIST_B200_ERR_UNSUPPORTED = 3, /* valid request outside what this build implements */
    DIST_B200_ERR_STATE = 4        /* feature not initialised / G mismatch between features */
} dist_b200_status;

/* component models, include/distributions/models/{dd,dpd,bb,gp,nich,niw}.hpp */
typedef enum {
    DIST_B200_DD = 0,   /* DirichletDiscrete<max_dim>   value: int32   */
    DIST_B200_DPD = 1,  /* DirichletProcessDiscrete     value: uint32 (0xFFFFFFFF = OTHER, dpd.hpp:55) */
    DIST_B200_BB = 2,   /* BetaBernoulli                value: uint8 (0 / non-0) */
    DIST_B200_GP = 3,   /* GammaPoisson                 value: uint32  */
    DIST_B200_NICH = 4, /* NormalInverseChiSq           value: float   */
    DIST_B200_NIW = 5,  /* NormalInverseWishart<d>      value: float[d], rows contiguous */
    DIST_B200_BNB = 6   /* BetaNegativeBinomial         value: uint32  */
} dist_b200_model;

typedef struct dist_b200_ctx dist_b200_ctx;
typedef struct dist_b200_feature dist_b200_feature;

/* ---- context --------------------------------------------------------------------------------
 * Owns the device-side numerics tables that replace src/special.cc's statics (FastLog table
 * special.cc:35-44, lgamma_approx_coeff5 :144-211, log_factorial_table :213-230,
 * lgamma_nu_func_approx_coeff3 :232-269) and scratch buffers.  One context per device/thread. */
int dist_b200_abi_version(void);
int dist_b200_ctx_create(int device, dist_b200_ctx **out);
void dist_b200_ctx_destroy(dist_b200_ctx *ctx);
const char *dist_b200_last_error(const dist_b200_ctx *ctx);
int dist_b200_sm_count(const dist_b200_ctx *ctx);
/* Measurement knobs (bench.py and the profiling scripts A/B kernels with them; a production caller never sets
 * any: 0 = the library's default everywhere).  The library reads no environment variables. */
typedef enum {
    DIST_B200_OPT_VALUE_CDF = 0,   /* single dpd / dd / bb feature, sampling only: 0 = score once per distinct VALUE and
                                      search per-value CDFs (guide tables; 8-ary trees for G > 1024) per row (SURVEY.md 8d "algorithmic shortcut");
                                      1 = evaluate every (row, group) cell (the no-shortcut kernels),
                                      2 = the shortcut with 8-ary tree search instead of the guide-table walk (G <= 1024) */
    DIST_B200_OPT_ROW_TILE = 1,    /* score_rows register tile for G > 128: 0 = default (32; 64 when the [N][G] scores are written), else 32 / 64 */
    DIST_B200_OPT_HOST_CHUNKS = 2, /* row chunks of the host-buffer entry: 0 = default (5) */
    DIST_B200_OPT_NIW_PATH = 3,    /* d = 32: 0 = tcgen05 kernel, split fp16 operands (default), 1 = FP32 CUDA-core kernel;
                                      no effect at other d (32 < d <= 128 has one route, the centred tcgen05 kernel) */
    DIST_B200_OPT_TABLE_KERNEL = 4,/* dpd no-shortcut kernel: 0 = register kernel on the lane-segment layout (owner lane's walk staged through
                                      shared memory), 1 = round-1 gather kernel, 2 = register kernel with the walk inside the row loop (G in (384, 512]) */
    DIST_B200_OPT_SMALL_TILE = 5,  /* score_rows, single feature, 64 < G <= 128: 0 = default, 1 = one 128-group tile x 256 threads
                                      (round 1), 2 = 128 threads x 3 blocks / SM with a 128-group tile, 3 = four 32-group tiles;
                                      default: 128 threads x 3, tile = G rounded up to 16 when only sampling */
    DIST_B200_OPT_NICH_PACKED = 6, /* nich single feature: 0 = default (packed fp32x2; sampling-only G > 128: static softmax reference,
                                      four rows per thread), 1 = scalar loop (round 1), 2 = packed fp32x2 loop with one row per thread,
                                      3 = sampling-only G > 128 with per-tile maxima, two rows per thread (the kernel the default replaced) */
    DIST_B200_OPT_NIW_DEBUG = 7,   /* profiling only, results are WRONG when set: 1 = skip the fused sampling walk, 2 = also the epilogue math */
    DIST_B200_OPT_HOST_ZEROCOPY = 8, /* host-buffer entry with page-locked caller buffers: 0 = kernels read / write the host buffers
                                      directly (one launch, no staging), 1 = staged row chunks over two streams (round 1) */
    DIST_B200_OPT_EXP_OFFLOAD = 9, /* nich sampling kernel (G > 128): share of the softmax exp2 evaluated on the FMA pipe (Cody-Waite +
                                      degree-5 polynomial) instead of MUFU.EX2: 0 = default (5 of every 16 pairs), 1 = none, 1 + k = k of every 16 pairs (k = 4, 6, 8) */
    DIST_B200_OPT_COUNT_ = 16
} dist_b200_option;
int dist_b200_ctx_set_option(dist_b200_ctx *ctx, int option, int value);

/* ---- features: MixtureValueScorer::{resize, update_all, update_group, add_group, remove_group}
 * All statistics arrays are host pointers holding the reference's Group fields as
 * struct-of-arrays over the G packed group ids. */
int dist_b200_feature_create(dist_b200_ctx *ctx, int model, dist_b200_feature **out);
void dist_b200_feature_destroy(dist_b200_feature *f);
int dist_b200_feature_model(const dist_b200_feature *f);
int dist_b200_feature_groups(const dist_b200_feature *f); /* G, 0 before the first update_all */

/* NormalInverseChiSq::MixtureValueScorer::update_all (nich.hpp:344-352 -> Scorer::init :239-250,
 * Shared::plus_group :58-69).  shared = {mu, kappa, sigmasq, nu}; Group = {count, mean,
 * count_times_variance} (nich.hpp:98-101). */
int dist_b200_nich_update_all(dist_b200_feature *f, const float shared[4], int G, const int32_t *count,
                              const float *mean, const float *count_times_variance, void *stream);
/* GammaPoisson (gp.hpp:293-301 -> :198-207, :56-61).  shared = {alpha, inv_beta};
 * Group = {count, sum, log_prod} (gp.hpp:84-87; log_prod does not enter score_value). */
int dist_b200_gp_update_all(dist_b200_feature *f, const float shared[2], int G, const uint32_t *count,
                            const uint32_t *sum, void *stream);
/* BetaNegativeBinomial (bnb.hpp:285-293 -> Scorer::init :200-211, plus_group :57-63).  shared = {alpha, beta},
 * r failures; Group = {count, sum} (bnb.hpp:89-91).  Caches {score, post_beta, alpha + r * count + r}; a cell
 * is score + fast_lgamma(post_beta + v) - fast_lgamma(post_beta + v + alpha) (bnb.hpp:308-319). */
int dist_b200_bnb_update_all(dist_b200_feature *f, const float shared[2], uint32_t r, int G, const uint32_t *count,
                             const uint32_t *sum, void *stream);
/* BetaBernoulli (bb.hpp:276-292).  shared = {alpha, beta}; Group = {heads, tails} (bb.hpp:79-81). */
int dist_b200_bb_update_all(dist_b200_feature *f, const float shared[2], int G, const int32_t *heads,
                            const int32_t *tails, void *stream);
/* DirichletDiscrete<max_dim> (dd.hpp:399-421).  counts is [G][dim] row-major (Group::counts,
 * dd.hpp:89-92; count_sum is recomputed). */
int dist_b200_dd_update_all(dist_b200_feature *f, int dim, const float *alphas, int G,
                            const int32_t *counts, void *stream);
/* DirichletProcessDiscrete (dpd.hpp:471-497).  keys[V] are the values present in Shared::betas with
 * weights betas[V]; counts is [G][V] dense (column v <-> keys[v]); beta0 scores OTHER / unseen
 * values (dpd.hpp:533-537). */
int dist_b200_dpd_update_all(dist_b200_feature *f, float alpha, float beta0, int V, const uint32_t *keys,
                             const float *betas, int G, const int32_t *counts, void *stream);
/* NormalInverseWishart<d> has no Mixture in the reference; this is the batched form of looping
 * Group::score_value over groups (mixture.hpp:321-337 semantics; niw.hpp:82-103, :343-361,
 * random.hpp:160-185).  psi and sum_xxT[g] are [d][d] row-major; Group = {count, sum_x, sum_xxT}
 * (niw.hpp:187-190).  1 <= d <= 128; d > 128 returns DIST_B200_ERR_UNSUPPORTED (the group prep holds a d x d double
 * Cholesky factor in shared memory).  Scoring routes by d: d <= 8 sampling only, the fused FP32 kernel; d <= 32 the FP32
 * CUDA-core kernel, except d = 32: tcgen05 with split fp16 operands (DIST_B200_OPT_NIW_PATH); 32 < d <= 128: tcgen05 on
 * x - mu (Shared.mu) padded to 64 / 128, scores materialised and sampled / reduced by the stand-alone kernels. */
int dist_b200_niw_update_all(dist_b200_feature *f, int d, const float *mu, float kappa, const float *psi,
                             float nu, int G, const int32_t *count, const float *sum_x,
                             const float *sum_xxT, void *stream);

/* MixtureValueScorer::update_group after Group::add_value / remove_value touched one group
 * (nich.hpp:312-342, gp.hpp:262-291, bb.hpp:258-274, dd.hpp:381-397,458-467, dpd.hpp:430-469; niw: the batched
 * form of rebuilding one Group's Scorer, niw.hpp:247-276,343-361).  `stats` points at that single group's
 * statistics in the same order as the update_all arguments:
 *   nich {int32 count; float mean; float ctv}   gp / bnb {uint32 count; uint32 sum}
 *   bb {int32 heads; int32 tails}               dd int32 counts[dim]
 *   dpd int32 counts[V] (dense, column v <-> keys[v] of the last update_all)
 *   niw {int32 count; float sum_x[d]; float sum_xxT[d][d]} packed without padding
 * The hyper-parameters are the ones given to the last update_all.  A dpd update rewrites the group's column of the
 * value-major table (O(V)); new VALUES (Shared::add_value growing betas, dpd.hpp:66-84) need an update_all. */
int dist_b200_feature_update_group(dist_b200_feature *f, int groupid, const void *stats, void *stream);
/* packed_add of a fresh empty group / packed_remove = swap-with-last (vector.hpp:39-61,
 * mixture.hpp:361-375) on every per-group device array.  dpd keeps its table dense with stride G, so both rebuild
 * it from the device-resident counts (O(V G), a few microseconds at V = 4096, G = 512). */
int dist_b200_feature_add_group(dist_b200_feature *f, void *stream);
int dist_b200_feature_remove_group(dist_b200_feature *f, int groupid, void *stream);

/* ---- group births and deaths in one batch: the step that makes a blocked Gibbs pass a DP / Pitman-Yor mixture ------
 * The batched form of the per-value bookkeeping of MixtureDriver::add_value / remove_value (mixture.hpp:77-122: a value
 * landing in an empty group appends a fresh one, a group emptied by remove_value is packed_remove'd) and of
 * packed_add / packed_remove (vector.hpp:39-61), for one clustering and every feature of its kind at once.
 *   - counts_dev[G]: the group sizes (the clustering's counts, e.g. from dist_b200_count_assignments).  A group is ALIVE
 *     iff counts_dev[g] > 0.  Feature statistics never decide liveness (with missing cells, a live group may hold no
 *     observed cell of some feature).
 *   - Order (canonical and stable): the live groups keep their relative order and become 0 .. K+ - 1; exactly n_empty
 *     fresh empty groups follow, K+ .. K+ + n_empty - 1; *G_out = K+ + n_empty.  A group of size 0 is dropped even when
 *     it already was an empty group, and a fresh one replaces it.  This is NOT the order a sequence of swap-with-last
 *     dist_b200_feature_remove_group calls gives: callers with per-group data of their own follow remap_out_dev.
 *   - remap_out_dev[G] (nullable): the new id of every old group, -1 for a dropped one.
 *   - counts_out_dev (nullable, capacity >= G + n_empty): the compacted counts, zeros for the fresh groups: the group
 *     sizes dist_b200_prior_pitman_yor_dev / dist_b200_prior_low_entropy_dev take at the new G.
 *   - assign_dev[n_rows] (nullable when n_rows == 0) is relabelled in place: negative ids stay, an id >= 0 becomes its
 *     group's new id.  An id >= G, or one whose group was dropped, becomes -1; that happens only when counts_dev
 *     disagrees with the assignments.
 *   - Every feature of the list (n_features == 0 does the clustering part only): its statistics are compacted the same
 *     way, each fresh group is Group::init (every statistics word zero) and its G becomes the new G.  Afterwards
 *     download_stats / download_caches / score / sample / logp / sample_values are bit-identical to those of a feature
 *     loaded by update_all from the compacted statistics.  gp: a Group::log_prod that was valid moves with its group
 *     (0 for a fresh group) and stays valid; an invalid one stays invalid.  Hot-cache slots past the new G hold zeros,
 *     as after dist_b200_feature_remove_group.
 *   - Checked, with no state changed: every feature has resident statistics (ERR_STATE before its first update_all) and
 *     G == the feature's G (ERR_STATE); n_empty >= 1, the reference's invariant (mixture.hpp:150-153), and no null
 *     argument where one is required (ERR_INVALID).
 *   - Synchronisation: the new G must reach the host (grid sizes and the features' G live there), so the call reads
 *     K+ back once through page-locked memory, which drains `stream` once.  That is its only synchronisation (plus the
 *     device-wide one of a buffer that has to grow past its capacity).  Everything else is enqueued on `stream`, and the
 *     features' ready events are recorded as the other update entries do.
 * Launches: one remap block, one relabel pass, and per 128 per-group arrays one gather and one copy-back launch
 * (statistics and gathered caches, out of place through a context buffer), then the caches of the fresh groups: the
 * model's prep on the n_empty fresh groups only, per feature (dpd: its table rebuilt once at the new stride; niw: the
 * fresh records and the tensor-core images once; gp: the value table is marked stale).  The count does not depend on
 * how many groups die or are born.
 * Row shards (replicated statistics): all-reduce the counts over the ranks, then every rank calls this with the GLOBAL
 * counts on its replica and its own rows; every replica computes the same remap and stays bit-identical. */
int dist_b200_regroup_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                            const int32_t *counts_dev, int G, int n_empty,
                            int32_t *assign_dev, size_t n_rows,
                            int32_t *counts_out_dev, int32_t *remap_out_dev, int *G_out, void *stream);

/* ---- batched Group::add_value on the device (next row of the path: score -> sample -> UPDATE) -----
 * Folds n_rows values into the groups given by assign_dev[n] (packed ids; negative = skip) with one
 * segmented reduction, merges into the device-resident statistics (the arrays last given to update_all /
 * update_group) and rebuilds the caches, without a host round trip.  Reference, per value:
 * Group::add_value + MixtureValueScorer::add_value (nich.hpp:125-133,326-333; gp.hpp:109-116,275-282;
 * bb.hpp:102-107,258-265; dd.hpp:123-130,381-388; dpd.hpp:188-196,430-447).  Counts are exact; nich's
 * mean / count_times_variance use the pairwise merge of Group::merge (nich.hpp:167-179) instead of N
 * sequential Welford steps (agreement ~1e-6 relative).  niw (niw.hpp:247-276; column = rows of d floats): the rows
 * are bucketed by group and every group's count / sum_x / sum_xxT deltas are accumulated in double (a per-group
 * SYRK), then folded into the resident float statistics -- the correctly rounded sums, where the reference's
 * value-by-value float updates carry their accumulation error; the group records are rebuilt afterwards.  A group
 * the batch empties is reset to exact zeros (Group::init). */
int dist_b200_feature_add_rows(dist_b200_feature *f, const void *column_dev, const int32_t *assign_dev, size_t n_rows,
                               void *stream);
/* The same for all features of one cross-cat kind at once (the reference loops the features of a kind per
 * row, loom-style kinds over ProductModel): one accumulate launch and one merge + cache-rebuild launch per 128
 * nich / gp / bb features, everything enqueued on `stream` without draining it.  features[i] reads
 * columns_dev[i]; all share assign_dev. */
int dist_b200_add_rows_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                             const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, void *stream);
/* Batched Group::remove_value (nich.hpp:146-165, gp.hpp:128-135, bb.hpp:117-122, dd.hpp:142-149,
 * dpd.hpp:207-215): the rows leave the groups assign_dev[n] names -- the first half of a Gibbs sweep over a
 * block of rows.  Integer statistics exact; nich inverts the pairwise merge in double (a group emptied by the
 * batch is reset to count = mean = ctv = 0 as the reference does).  Emptied groups stay in place: removing
 * them (dist_b200_feature_remove_group) is the mixture driver's decision, as in mixture.hpp:95-122. */
int dist_b200_remove_rows_batch(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, void *stream);
int dist_b200_remove_rows_batch_host(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                     const void *const *columns_host, const int32_t *assign_host, size_t n_rows);
/* Row shards (one process per GPU, rows partitioned, statistics replicated): the update has a real exchange
 * step.  Every rank accumulates its own rows into xchg_dev, the caller sums the buffers over the ranks (one NCCL
 * all-reduce of float64), and every rank merges the global sums into its replica (sign +1 add_value, -1
 * remove_value), leaving all replicas bit-identical.  Layout of xchg_dev (doubles; dist_b200_rows_xchg_doubles
 * returns the total): first one [4][G] block per pooled-statistics feature (nich / gp / bb / bnb: count-like a,
 * count-like b, sum x, sum x^2; integers exact) in list order, then one [G][dim] block of delta counts per
 * count-table feature (dd: dd.hpp:123-149; dpd: dpd.hpp:188-214, dim = number of known values) and one
 * [G][1 + d + d * d] block {count, sum_x, sum_xxT} per niw feature, in list order.  All features with the same G. */
int dist_b200_rows_xchg_doubles(dist_b200_feature *const *features, int n_features, size_t *n_doubles);
int dist_b200_rows_accumulate(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                              const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, double *xchg_dev,
                              void *stream);
int dist_b200_rows_merge(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features, const double *xchg_dev,
                         int sign, void *stream);
/* Host-buffer form (the call a reference-side binding makes): columns_host[i] holds n_rows values of
 * features[i] (float / uint32 / int32, bool as uint8), assign_host the packed group ids.  Synchronous. */
int dist_b200_add_rows_batch_host(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                  const void *const *columns_host, const int32_t *assign_host, size_t n_rows);
/* ---- batched Group::sample_value: posterior-predictive draws from the same device-resident statistics -------------
 * For every row n with 0 <= assign_dev[n] < G, columns_out_dev[i][n] receives one draw from the posterior predictive of
 * group assign_dev[n] of features[i]: fresh parameters per value, as Sampler::init + Sampler::eval do (nich.hpp, gp.hpp,
 * bnb.hpp, bb.hpp, dd.hpp, dpd.hpp, niw.hpp), so rows are independent given the statistics.  Rows with a negative or
 * out-of-range id are left untouched (as add_rows_batch skips them).  Output types are the column types of
 * dist_b200_model (dpd: the key, 0xFFFFFFFF = OTHER; niw: rows of d floats), so the columns feed score_sample_batch and
 * add_rows_batch unchanged.  All features share G (ERR_STATE otherwise, and for a feature before its first update_all).
 * The launch waits on every feature's pending updates, so a preceding add_rows_batch is seen without a host synchronise.
 * Random numbers: Philox4x32-10 keyed by `seed`, counter (global row row0 + n, position i of the feature in the list,
 * draw index within the value).  A draw is a pure function of (seed, row0 + n, i, that group's statistics), independent
 * of launch geometry, n_rows and chunking: row shards passing their own row0 reproduce a single call bit for bit.  Two
 * features drawn in separate calls at the same list position get the same random stream: give such calls distinct seeds.
 * niw: coordinate c of a row draws its normal from block c of the row's stream and the chi-square from block max(32, d)
 * on, so no block serves two quantities at any d <= 128 (the draws at d <= 32 use block 32, as before).
 * The host form stages through the context (the output columns travel both ways, so skipped rows keep their values);
 * its results are bit-identical to the device form.  Synchronous. */
int dist_b200_sample_values_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                  const int32_t *assign_dev, size_t n_rows, uint64_t seed, uint64_t row0,
                                  void *const *columns_out_dev, void *stream);
int dist_b200_sample_values_batch_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                       const int32_t *assign_host, size_t n_rows, uint64_t seed, uint64_t row0,
                                       void *const *columns_out_host);
/* ---- score_data_grid: hyper-parameter inference over the same statistics ---------------------------
 * out[i] = log marginal likelihood of all groups of `f` under hyper-parameter setting i: the reference's
 * MixtureSlave::score_data_grid / score_data (mixture.hpp:427-438; nich.hpp:262-288, gp.hpp:220-241,
 * bb.hpp:207-229, dd.hpp:250-324, dpd.hpp:344-374) on the device-resident group statistics.  shareds:
 * n_grid packed Shareds, `stride` floats apart -- nich (mu, kappa, sigmasq, nu); gp (alpha, inv_beta);
 * bb (alpha, beta); dd alphas[dim]; dpd (alpha), with beta0 / betas of the last update_all; niw (niw.hpp:296-308)
 * kappa, nu, mu[d], psi[d][d].  Every term is
 * the reference's fp32 expression; the sum over groups is accumulated in double (the reference: fp32, group
 * order), so results agree to ~1e-6 of sum |term|.  gp reads Group::log_prod, which the hot path does not
 * carry: set it with dist_b200_gp_set_log_prod after update_all / any statistics change (ERR_STATE otherwise).
 * niw: the determinants come from Cholesky factorisations in double; fast_log(det) is the reference's while det is a
 * normal float -- beyond that (the reference's float determinant() overflows, always at d = 32, and its result is
 * meaningless) the exact log determinant is used, as in the reference's Python flavour (dbg/models/niw.py:213,216). */
int dist_b200_gp_set_log_prod(dist_b200_feature *f, const float *log_prod_host, void *stream);
int dist_b200_score_data_grid(dist_b200_feature *f, const float *shareds_dev, size_t n_grid, size_t stride,
                              float *out_dev, void *stream);
int dist_b200_score_data_grid_host(dist_b200_feature *f, const float *shareds_host, size_t n_grid, size_t stride,
                                   float *out_host);
/* ---- the reference's protobuf wire format (distributions/io/schema.proto:36-158) ----------------------
 * Load a feature from its serialized Shared message and G serialized Group messages (the records of the
 * reference's dumps / loom-style streams) without building host objects: the messages are decoded straight
 * into the SoA arrays of the model's update_all (dpd: dense counts in Shared.values order, beta0 =
 * max(0, 1 - sum betas) as Shared::protobuf_load, dpd.hpp:104-125; gp: log_prod is kept for score_data_grid).
 * Packed and unpacked repeated scalars are accepted, unknown fields skipped; a malformed message is
 * DIST_B200_ERR_INVALID, a uint64 count that does not fit the reference's 32-bit Group fields
 * DIST_B200_ERR_UNSUPPORTED.  niw (schema.proto:147-161): Shared.psi must be symmetric positive definite and every
 * Group.sum_xxT symmetric, as Shared / Group::protobuf_load assert (niw.hpp:105-134, :192-216). */
int dist_b200_update_all_wire(dist_b200_feature *f, const void *shared_msg, size_t shared_len,
                              const void *const *group_msgs, const size_t *group_lens, int G, void *stream);
/* The same with the Groups as one record stream of the reference's dumps (distributions/io/stream.py:141-153,
 * after decompression): [uint32 little-endian length][Group message] repeated; G = the number of records. */
int dist_b200_update_all_stream(dist_b200_feature *f, const void *shared_msg, size_t shared_len, const void *stream_bytes,
                                size_t stream_len, void *stream);
/* record boundaries of such a stream (no device; ctx may be NULL): offsets_out / lens_out[capacity] (nullable),
 * *n_records the count (also when capacity is too small) */
int dist_b200_wire_split_stream(dist_b200_ctx *ctx, const void *stream_bytes, size_t stream_len, size_t *offsets_out,
                                size_t *lens_out, size_t capacity, size_t *n_records);
/* The decode step alone (no device): shared_out = Shared floats (nich 4; gp 2; bb 2; bnb alpha, beta, r;
 * dd alphas; dpd gamma, alpha, beta0, betas[V]; niw kappa, nu, mu[d], psi[d][d]), keys_out = dpd Shared.values
 * (bnb: r), stats_out = the update_all arrays back to back, floats as bit patterns (gp: count | sum | log_prod;
 * niw: count[G] | sum_x[G][d] | sum_xxT[G][d][d]).  counts_out receives the
 * three lengths (also when a buffer is too small).  ctx may be NULL (no error text is recorded then). */
int dist_b200_wire_decode(dist_b200_ctx *ctx, int model, const void *shared_msg, size_t shared_len,
                          const void *const *group_msgs, const size_t *group_lens, int G, float *shared_out,
                          size_t shared_cap, uint32_t *keys_out, size_t keys_cap, uint32_t *stats_out, size_t stats_cap,
                          size_t counts_out[3]);
/* The way back: the feature's current device-resident statistics as G serialized Group messages,
 * concatenated into out[capacity]; lens_out[G] (nullable) the length of each, *n_bytes the total (also when
 * out is too small).  Canonical proto2 output (fields in number order, repeated scalars unpacked): byte-
 * identical to the reference's writer for the same Groups; dpd groups list their non-zero counts in
 * Shared.values order.  gp needs a valid log_prod (ERR_STATE otherwise).  Synchronises the stream. */
int dist_b200_feature_dump_groups_wire(dist_b200_feature *f, void *out, size_t capacity, size_t *lens_out, size_t *n_bytes,
                                       void *stream);
/* the encode step alone (no device; ctx may be NULL): stats = the arrays dist_b200_wire_decode returns */
int dist_b200_wire_encode_groups(dist_b200_ctx *ctx, int model, int G, int dim, const uint32_t *keys, const uint32_t *stats,
                                 size_t stats_words, void *out, size_t capacity, size_t *lens_out, size_t *n_bytes);
/* Shared message from the packed values dist_b200_wire_decode returns (nich, gp, bb, bnb with keys[0] = r, dd, niw;
 * dpd: keys = Shared.values[V] followed by the per-value totals Shared.counts[V] (dpd.hpp:64, :126-138), i.e. the
 * column sums of the groups' counts when every add_value went through Shared and a Group, as the drivers do) */
int dist_b200_wire_encode_shared(dist_b200_ctx *ctx, int model, const float *shared, size_t n_shared, const uint32_t *keys,
                                 size_t n_keys, void *out, size_t capacity, size_t *n_bytes);
/* Clustering message (pitman_yor = 1 | low_entropy = 2, schema.proto:36-53) -> the prior vector */
int dist_b200_prior_wire_host(dist_b200_ctx *ctx, const void *clustering_msg, size_t len, int G,
                              const int32_t *group_sizes, float *prior_host);
/* Device-resident statistics back to the host, arrays in update_all's argument order, G entries each
 * (nich: count,int32 | mean,f32 | ctv,f32; gp: count | sum; bb: heads | tails; dd: counts[G][dim];
 * dpd: counts[G][V]).  Synchronises the stream. */
int dist_b200_feature_download_stats(const dist_b200_feature *f, void *out_host, size_t capacity_bytes, size_t *n_bytes,
                                     void *stream);
/* MixtureDriver::counts() for a batch: counts_dev[g] (+)= #{n : assign_dev[n] == g}  (mixture.hpp:77-93). */
int dist_b200_count_assignments(dist_b200_ctx *ctx, const int32_t *assign_dev, size_t n_rows, int G, int32_t *counts_dev,
                                int accumulate, void *stream);
/* dist_b200_prior_pitman_yor with the group sizes already on the device. */
int dist_b200_prior_pitman_yor_dev(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *group_sizes_dev,
                                   float *prior_dev, void *stream);

/* Read the caches back in the reference's own struct-of-arrays layout (for parity tests):
 *   nich [4][G] score_, log_coeff_, precision_, mean_   (nich.hpp:379-384)
 *   gp   [3][G] score_, post_alpha_, score_coeff_       (gp.hpp:329-333)
 *   bb   [2][G] heads_scores_, tails_scores_            (bb.hpp:321-324)
 *   dd   [dim][G]  score_value_group(g, v) = scores_[v][g] - scores_shift_[g]  (dd.hpp:423-431)
 *   dpd  [V+1][G]  the same for keys[v], last row = the OTHER / unseen row      (dpd.hpp:499-515)
 * Synchronises the stream.  *n_floats receives the number of floats written. */
int dist_b200_feature_download_caches(const dist_b200_feature *f, float *out_host, size_t capacity_floats,
                                      size_t *n_floats, void *stream);

/* ---- clustering prior: Clustering<int>::PitmanYor::Mixture::{init, score_value}
 * (clustering.hpp:151-161, :195-230; CRP is d = 0).  Writes prior_dev[g] = shifted_scores_[g] -
 * fast_log(sample_size + alpha) for g < G from the group sizes (host). */
int dist_b200_prior_pitman_yor(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *group_sizes,
                               float *prior_dev, void *stream);

/* LowEntropy clustering prior (Clustering<int>::LowEntropy, clustering.hpp:245-331): prior[g] =
 * score_add_value(group_sizes[g], nonempty, sample_size, empty) as the uncached MixtureDriver::score_value
 * evaluates it (mixture.hpp:123-141).  OVERWRITES prior[G], like the Pitman-Yor vector; feed it to the same
 * `prior` argument of the score entries. */
int dist_b200_prior_low_entropy_host(dist_b200_ctx *ctx, int dataset_size, int G, const int32_t *group_sizes,
                                     float *prior_host);
int dist_b200_prior_low_entropy_dev(dist_b200_ctx *ctx, int dataset_size, int G, const int32_t *sizes_dev,
                                    float *prior_dev, void *stream);
/* Same with a HOST result buffer: the per-value CachedMixture::score_value(model, scores) drop-in
 * (clustering.hpp:195-208; overwrites prior_host[0..G)). */
int dist_b200_prior_pitman_yor_host(dist_b200_ctx *ctx, float alpha, float d, int G, const int32_t *group_sizes,
                                    float *prior_host);

/* ---- the hot path -----------------------------------------------------------------------------
 * columns_dev[f] is feature f's value column for the N rows, typed per model (see
 * dist_b200_model); feature-major storage, i.e. one contiguous array per feature.
 *
 * dist_b200_score_batch: batched MixtureSlave::score_value (mixture.hpp:416-425).
 *   accumulate != 0 : scores_dev[n][g] += sum_f ...        (the slave's ACCUMULATE semantic)
 *   accumulate == 0 : scores_dev[n][g]  = prior_dev[g] + sum_f ... (prior_dev may be NULL = 0;
 *                     this is clustering's OVERWRITE, clustering.hpp:195-208, followed by the slaves)
 * scores_dev is [N][G] row-major float32.
 * Precondition of the continuous models: the log argument of a cell, nich's 1 + precision (x - mean)^2 and niw's
 * 1 + q / dof, must be finite in float32.  A cell whose argument overflows scores -inf (the reference's table gives
 * 128 ln 2); a row that overflows in every group gets -inf from score_logp_batch and an unspecified draw.  On the niw
 * d = 32 tensor-core route such a row also makes the other rows of its 128-row tile score NaN (tile-wide scale).
 * niw d = 32 (tensor cores): the quadratic form's error follows |W x| + |W mu'|, not |W (x - mu')|.  It matches the FP32
 * kernel's accuracy on data and prior mean within a few standard deviations of the origin (measured); at 1e2 - 1e3
 * standard deviations, or beside a row ~1e4 x larger in its 128-row tile, it loses precision (DESIGN §6).
 * DIST_B200_OPT_NIW_PATH = 1 is translation-invariant.
 * niw 32 < d <= 128 (tensor cores, centred): the rows are split after subtracting Shared.mu and the groups' offsets
 * W (mu' - mu) are formed in double, so the error follows |W (x - mu)| + |W (mu' - mu)| -- the data's spread around the
 * prior mean, not its offset from the origin -- within the derived bound of DESIGN §6 ("d > 32").  As at d = 32 the scale
 * is per 128-row tile: a row far larger than its tile-mates (|x - mu| ~ 1e4 x) costs them precision, and a row whose
 * scaled square overflows makes them NaN. */
int dist_b200_score_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                          const void *const *columns_dev, size_t n_rows, const float *prior_dev,
                          float *scores_dev, int accumulate, void *stream);

/* dist_b200_score_sample_batch: the whole per-row assignment step of
 * examples/mixture/main.py:236-244 for N rows against frozen statistics, fused:
 * prior + features -> sample_from_scores_overwrite (random.hpp:360-366) with the caller's
 * uniforms u_dev[n] in [0,1) in place of sample_unif01(rng).  assign_dev[n] receives the packed
 * group id.  scores_dev (optional, may be NULL) also receives the [N][G] log scores. */
int dist_b200_score_sample_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features,
                                 int n_features, const void *const *columns_dev, size_t n_rows,
                                 const float *prior_dev, const float *u_dev, int32_t *assign_dev,
                                 float *scores_dev, void *stream);

/* dist_b200_sample_from_scores: sample_from_scores (random.hpp:386-392; scores are not
 * overwritten) for N rows of G materialised scores, e.g. after the feature-shard reduction. */
int dist_b200_sample_from_scores(dist_b200_ctx *ctx, const float *scores_dev, size_t n_rows, int G,
                                 const float *u_dev, int32_t *assign_dev, void *stream);

/* ---- row log-likelihood: how probable is each row under the mixture ---------------------------------------------
 * dist_b200_score_logp_batch: for every row n,
 *   logp_dev[n] = log sum_{g < G} exp(prior_dev[g] + sum_f score_f(columns_dev[f][n]; g))      (natural log, float32)
 * prior_dev may be NULL (= 0).  With the Pitman-Yor vector of dist_b200_prior_pitman_yor (group sizes including the empty
 * group; the prior weights then sum to 1) this is the log posterior-predictive density of the row under the mixture: the
 * quantity the reference's frozen-mixture example forms per pixel as exp(scores).sum() (examples/mixture/main.py:143-160)
 * with log_sum_exp as its primitive (src/random.cc:77-92).
 *   - logp_dev is OVERWRITTEN; there is no accumulate form.  The [N][G] scores are not materialised for row-mapped
 *     features (nich / gp / bnb / bb / dd, any list of them) and single table features; dpd in per-cell mode, niw and mixed
 *     lists containing them go through the context's scores buffer.
 *   - A row whose every term is -inf (e.g. a prior of -inf everywhere) gets -inf, never NaN.
 *   - Same feature-list rules, column types and error codes as dist_b200_score_sample_batch (ERR_STATE for a feature
 *     before its first update_all or features that disagree on G).  Waits on every feature's pending updates (ready
 *     events), like the other score entries, so a preceding add_rows_batch on another stream is seen.
 *   - Conditional densities: logp(A | B) = logp(features A and B) - logp(features B), two calls over nested feature lists
 *     with the same prior.
 * dist_b200_score_logp_batch_host: the same with host buffers (staged / zero-copy as dist_b200_score_sample_batch_host;
 * results bit-identical to the device form).  Synchronous.
 * dist_b200_logp_from_scores: the reduction alone over materialised [N][G] scores, e.g. a score_batch result or the sum
 * of feature-shard slots the caller formed (the counterpart of dist_b200_sample_from_scores). */
int dist_b200_score_logp_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                               const void *const *columns_dev, size_t n_rows, const float *prior_dev,
                               float *logp_dev, void *stream);
int dist_b200_score_logp_batch_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                    const void *const *columns_host, size_t n_rows, const float *prior_host,
                                    float *logp_host);
int dist_b200_logp_from_scores(dist_b200_ctx *ctx, const float *scores_dev, size_t n_rows, int G,
                               float *logp_dev, void *stream);

/* ---- missing cells: per-feature observed masks ------------------------------------------------------------------
 * A cross-cat table has holes.  As in loom's ProductModel, whose Value carries an `observed` flag per feature, an
 * unobserved feature simply does not enter the row's score or its group's statistics.  The *_masked entries take the
 * arguments of their unmasked form plus observed_dev: n_features device pointers, one per feature, each NULL (that
 * feature is fully observed) or ceil(n_rows / 32) uint32 words; bit n % 32 of word n / 32 is 1 when row n's cell is
 * observed (bits past n_rows are ignored).  np.packbits(column, bitorder="little") read as little-endian uint32 is this
 * layout.  observed_dev itself may be NULL (every feature fully observed).
 *   - Scoring: a missing cell contributes exactly 0: scores[n][g] = prior[g] + sum_f observed_f[n] * score_f(x_f[n]; g).
 *     Its stored value is never used in arithmetic (it may be NaN, a dd value >= dim, a huge count).  A row with every
 *     feature missing scores the prior alone: its draw comes from the prior and its logp is logsumexp(prior).
 *   - add / remove rows, rows_accumulate: a missing cell leaves that feature's statistics alone, exactly as if
 *     assign_dev[n] were -1 for that feature only.  The row's other features are unaffected.  The exchange layout of
 *     rows_accumulate is the unmasked one (merge with dist_b200_rows_merge).
 *   - Imputation (sample_values_batch_masked): a draw is written into every MISSING cell of a row with a valid
 *     assignment, and nothing else: observed cells and rows with an invalid id keep their values.  The draw is the one
 *     dist_b200_sample_values_batch writes for the same (seed, row0, row, list position), so the result is
 *     where(observed, column, unmasked draws) bit for bit.  Here a NULL mask means nothing is imputed for that feature.
 *   - With every mask NULL the score, sample, logp and rows entries ARE the unmasked entries (bit-identical results).
 *     Argument checks and error codes are those of the unmasked entries.
 * Routes and costs.  Lists of row-mapped features (nich / gp / bnb / bb / dd, including a list of one) run the
 * feature-list kernel with the masks as a separate kernel parameter: one broadcast word per warp and feature, and a
 * lane whose cell is missing sits that feature out.  dpd and niw features are scored alone (their own kernels) into a
 * second context [N][G] buffer and added where observed: one extra [N][G] write and read per masked dpd / niw feature
 * (fully observed ones accumulate directly).  The single-feature, nich_rows2, table, per-value and niw tensor-core
 * sampling kernels have no masked form; their features take the two routes above.  add / remove rows and
 * rows_accumulate run masked instantiations of the pooled, count-table and niw histogram / scatter kernels (one mask
 * word per 32 rows, pooled batches of up to 128 features as unmasked).  Imputation runs the unmasked sampling kernels
 * over an assignment vector with -1 in the observed rows: one extra N-int pass per masked feature.
 * Streams: the masked score route (with dpd / niw) and imputation use a context scratch buffer of their own, ordered
 * only by the stream of the call, as the context's scores buffer is: masked calls of one context on two streams at
 * once must not overlap.
 * There are no masked forms of dist_b200_score_push_batch or of the host-buffer entries. */
int dist_b200_score_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                 const void *const *columns_dev, size_t n_rows, const float *prior_dev, float *scores_dev,
                                 int accumulate, const uint32_t *const *observed_dev, void *stream);
int dist_b200_score_sample_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                        const void *const *columns_dev, size_t n_rows, const float *prior_dev,
                                        const float *u_dev, int32_t *assign_dev, float *scores_dev,
                                        const uint32_t *const *observed_dev, void *stream);
int dist_b200_score_logp_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                      const void *const *columns_dev, size_t n_rows, const float *prior_dev, float *logp_dev,
                                      const uint32_t *const *observed_dev, void *stream);
int dist_b200_add_rows_batch_masked(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                    const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows,
                                    const uint32_t *const *observed_dev, void *stream);
int dist_b200_remove_rows_batch_masked(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                       const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows,
                                       const uint32_t *const *observed_dev, void *stream);
int dist_b200_rows_accumulate_masked(dist_b200_ctx *ctx, dist_b200_feature *const *features, int n_features,
                                     const void *const *columns_dev, const int32_t *assign_dev, size_t n_rows, double *xchg_dev,
                                     const uint32_t *const *observed_dev, void *stream);
int dist_b200_sample_values_batch_masked(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                                         const int32_t *assign_dev, size_t n_rows, uint64_t seed, uint64_t row0,
                                         void *const *columns_out_dev, const uint32_t *const *observed_dev, void *stream);

/* ---- feature shards over NVLink peer memory (one process per GPU) ----------------------------------
 * scores[n][g] = prior[g] + sum_f s_f[n][g] is a sum over features (SURVEY.md §8e).  With the features of
 * a kind sharded over K ranks, each rank scores its features for every row and stores the partial row
 * DIRECTLY into the owning rank's memory -- owner = row / block_rows -- from inside the score kernel, so
 * the NVLink transfer overlaps the math tile by tile and the partial [N][G] tile never touches local HBM.
 * Every owner holds K slots [block_rows][G] (slot r written by rank r) and samples the fixed-order sum of
 * its slots (deterministic, unlike atomics).  Buffers are exchanged as CUDA IPC handles. */
int dist_b200_peer_alloc(dist_b200_ctx *ctx, size_t bytes, void **dev_ptr, unsigned char handle_out[64]);
int dist_b200_peer_open(dist_b200_ctx *ctx, const unsigned char handle[64], void **dev_ptr);
int dist_b200_peer_close(dist_b200_ctx *ctx, void *dev_ptr);
int dist_b200_peer_free(dist_b200_ctx *ctx, void *dev_ptr);
/* Partial scores of rows [row0, row0 + n_rows) for this rank's features, pushed to the owners' slots:
 * slot_ptrs[o] is the (peer-mapped) base of THIS rank's slot in owner o's buffer.  prior_dev is passed
 * by exactly one rank.  Row-mapped models only (nich / gp / bnb / bb / dd; dpd and niw return
 * DIST_B200_ERR_UNSUPPORTED).  Any block_rows >= 1 and any row0 are accepted.  When G % 4 == 0 every slot pointer
 * must be 16-byte aligned (rows are stored 16 bytes at a time). */
int dist_b200_score_push_batch(dist_b200_ctx *ctx, const dist_b200_feature *const *features, int n_features,
                               const void *const *columns_dev, size_t n_rows, size_t row0, const float *prior_dev,
                               void *const *slot_ptrs, int n_owners, size_t block_rows, void *stream);
/* Device-side signalling that replaces host barriers around the push.  Every owner holds one uint32 flag per
 * pusher (zero-initialised: dist_b200_peer_alloc clears its buffer); epochs only grow.
 *   dist_b200_peer_signal: after this rank's push kernel (same stream), raise flag[my_index] = epoch in every
 *     owner's flag array (flag_ptrs[o] = peer-mapped base of owner o's flags) with a system-scope release.
 *   dist_b200_peer_wait: stream-ordered wait until all n_peers local flags have reached `epoch` (system-scope
 *     acquire; traps after ~13 s instead of hanging the device).  The sampler enqueued behind it then sees every push.
 * Neither returns to the host: a step is push kernel, signal, wait, sampler on one stream. */
int dist_b200_peer_signal(dist_b200_ctx *ctx, void *const *flag_ptrs, int n_peers, int my_index, uint32_t epoch, void *stream);
int dist_b200_peer_wait(dist_b200_ctx *ctx, const void *flags_dev, int n_peers, uint32_t epoch, void *stream);
/* sample_from_scores over the sum of n_slots partial score blocks, slot_stride floats apart. */
int dist_b200_sample_from_slots(dist_b200_ctx *ctx, const float *slots_dev, int n_slots, size_t slot_stride,
                                size_t n_rows, int G, const float *u_dev, int32_t *assign_dev, void *stream);

/* ---- host-buffer forms: the call a reference-side binding makes (INTEGRATION.md).  Same
 * semantics with HOST pointers, results on the host before returning.  Pageable buffers are staged through the
 * context's page-locked area in row chunks over two streams (H2D of chunk k+1 and D2H of chunk k-1 under the kernel of
 * chunk k).  Buffers that are ALL page-locked already (cudaHostAlloc / cudaHostRegister / torch pin_memory) are not
 * copied at all: the kernels read the rows from and write the assignments to host memory directly (one launch; the
 * PCIe transfers overlap the math row tile by row tile) -- except with a niw feature, whose pack kernel has no math to
 * hide the reads behind.  dist_b200_score_value_host (per value) always goes through page-locked memory this way. */
int dist_b200_score_sample_batch_host(dist_b200_ctx *ctx, const dist_b200_feature *const *features,
                                      int n_features, const void *const *columns_host, size_t n_rows,
                                      const float *prior_host, const float *u_host, int32_t *assign_host,
                                      float *scores_host);
/* Page-lock a caller-owned host buffer once (cudaHostRegister, portable + mapped), so that every later host-entry call
 * on it takes the zero-copy route -- the data columns of a Gibbs sampler are the same arrays sweep after sweep (the
 * reference keeps them in std::vector / numpy storage, which is pageable).  Registering an already registered range is
 * OK.  The caller unregisters before freeing the buffer. */
int dist_b200_host_register(dist_b200_ctx *ctx, void *ptr, size_t bytes);
int dist_b200_host_unregister(dist_b200_ctx *ctx, void *ptr);
/* per-value MixtureSlave::score_value (mixture.hpp:416-425): scores_accum_host[G] += model term. */
int dist_b200_score_value_host(dist_b200_ctx *ctx, const dist_b200_feature *feature, const void *value_host,
                               float *scores_accum_host);

/* ---- numerics probes (parity tests of the device functions against special.hpp / fmath.hpp).
 * fn: 0 fast_log (table form, as used by the cache rebuilds)   1 fast_exp (sampler form)
 *     2 fast_lgamma   3 fast_lgamma_nu   4 fast_log_factorial (input bits as uint32)
 *     5 fast_log (per-cell form: truncated mantissa + MUFU.LG2; the argument must be finite: inf gives inf, where the
 *       table gives 128 ln 2 -- see the nich / niw score entries)
 *     6 fast_lgamma (exact restatement of the cache rebuilds)
 *     7 exp2 on the FMA pipe (poly_ex2_pair of the sampling kernels; arguments below -125 give 2^-125) */
int dist_b200_numerics_probe(dist_b200_ctx *ctx, int fn, size_t n, const float *in_dev, float *out_dev,
                             void *stream);

/* Register-only pipe probes for roofline denominators that MEASURED_PEAKS.json does not carry:
 * which = 0: MUFU (ex2/lg2) lane-ops per second, 1: FP32 FMA lane-ops per second, whole device;
 * which = 2: L2 gather BYTES per second with the dpd table kernel's access pattern (random 2 KB rows of an
 * L2-resident 8 MB table, LDG.128) -- the denominator of c4's gather bound (SURVEY.md 8d). */
int dist_b200_pipe_peak(dist_b200_ctx *ctx, int which, double *ops_per_s);

#ifdef __cplusplus
}
#endif
#endif /* DIST_B200_H_ */
