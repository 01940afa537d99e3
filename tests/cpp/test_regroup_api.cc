// The regroup follow-ups of the C++ host mirror (include/distributions_b200/mixture.hpp): MixtureIdTracker::regroup and
// the clustering drivers' regroup run here without a device; Mixture<Model>::regroup of every model is instantiated so
// that it compiles and links.  With the argument "gpu", a Mixture<NormalInverseChiSq> is also regrouped on the device
// by dist_b200_regroup_batch and its host Groups, re-read by Mixture::regroup, are checked against the compaction of the
// Groups it held before.  Prints "ok" when every check holds.
#include <distributions_b200/mixture.hpp>

#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>

using namespace distributions_b200;

#define CHECK(c)                                                        \
    do {                                                                \
        if (!(c)) {                                                     \
            std::fprintf(stderr, "check failed at line %d: %s\n", __LINE__, #c); \
            return 1;                                                   \
        }                                                               \
    } while (0)

template <class Model>
static bool instantiate() {
    void (Mixture<Model>::*fn)(const typename Model::Shared &, const std::vector<int32_t> &, size_t, rng_t &) = &Mixture<Model>::regroup;
    return fn != nullptr;
}

// six groups, three of them empty by the clustering's sizes; two fresh groups after the regroup
static int gpu_check() {
    auto ctx = std::make_shared<Context>(0);
    rng_t rng;
    const NormalInverseChiSq::Shared shared = NormalInverseChiSq::Shared::EXAMPLE();
    Mixture<NormalInverseChiSq> mixture(ctx);
    for (int g = 0; g < 6; ++g) {
        NormalInverseChiSq::Group grp;
        grp.init(shared, rng);
        for (int i = 0; i <= g; ++i) grp.add_value(shared, 0.5f * g + 0.25f * i, rng);
        mixture.groups().push_back(grp);
    }
    mixture.init(shared, rng);
    const std::vector<NormalInverseChiSq::Group> before = mixture.groups();
    const std::vector<int32_t> sizes = {3, 0, 1, 0, 0, 6};
    int32_t *sizes_dev = nullptr, *remap_dev = nullptr;
    CHECK(cudaMalloc(&sizes_dev, sizeof(int32_t) * 6) == cudaSuccess && cudaMalloc(&remap_dev, sizeof(int32_t) * 6) == cudaSuccess);
    CHECK(cudaMemcpy(sizes_dev, sizes.data(), sizeof(int32_t) * 6, cudaMemcpyHostToDevice) == cudaSuccess);
    dist_b200_feature *feats[1] = {mixture.feature()};
    int G_new = 0;
    ctx->check(dist_b200_regroup_batch(ctx->get(), feats, 1, sizes_dev, 6, 2, nullptr, 0, nullptr, remap_dev, &G_new, nullptr),
               "regroup_batch");
    std::vector<int32_t> remap(6);
    CHECK(cudaMemcpy(remap.data(), remap_dev, sizeof(int32_t) * 6, cudaMemcpyDeviceToHost) == cudaSuccess);
    cudaFree(sizes_dev);
    cudaFree(remap_dev);
    CHECK(G_new == 5);
    CHECK((remap == std::vector<int32_t>{0, -1, 1, -1, -1, 2}));
    mixture.regroup(shared, remap, 2, rng);
    CHECK(mixture.groups().size() == 5);
    const int kept[3] = {0, 2, 5};
    for (int i = 0; i < 5; ++i) {
        const NormalInverseChiSq::Group &got = mixture.groups(i);
        NormalInverseChiSq::Group want;
        want.init(shared, rng);
        if (i < 3) want = before[kept[i]];
        CHECK(got.count == want.count && std::memcmp(&got.mean, &want.mean, 4) == 0 &&
              std::memcmp(&got.count_times_variance, &want.count_times_variance, 4) == 0);
    }
    return 0;
}

int main(int argc, char **argv) {
    if (argc > 1 && std::strcmp(argv[1], "gpu") == 0 && gpu_check() != 0) return 1;
    // a mixture drops groups 1 and 3 (size 0) and keeps two empty groups
    std::vector<int32_t> sizes = {4, 0, 7, 0, 1};
    PitmanYor py{1.0f, 0.1f};
    PitmanYor::Mixture driver(nullptr);
    driver.counts() = sizes;
    driver.init(py);
    const std::vector<int32_t> remap = driver.regroup(py, 2);
    CHECK((remap == std::vector<int32_t>{0, -1, 1, -1, 2}));
    CHECK((driver.counts() == std::vector<int32_t>{4, 7, 1, 0, 0}));
    CHECK(driver.sample_size() == 12);
    CHECK(driver.empty_groupids().size() == 2 && driver.empty_groupids().count(3) && driver.empty_groupids().count(4));

    LowEntropy le{100};
    LowEntropy::Mixture le_driver(nullptr);
    le_driver.counts() = sizes;
    CHECK(le_driver.regroup(le, 1) == (std::vector<int32_t>{0, -1, 1, -1, 2}));
    CHECK((le_driver.counts() == std::vector<int32_t>{4, 7, 1, 0}));

    MixtureIdTracker ids;
    ids.init(5);
    ids.remove_group(0);  // global 4 moves to packed 0: packed -> global = 4 1 2 3
    ids.add_group();      // global 5
    std::vector<int32_t> rm = {0, -1, 1, -1, 2};  // drops globals 1 and 3
    ids.regroup(rm, 2);
    CHECK(ids.packed_size() == 5 && ids.global_size() == 8);
    CHECK(ids.packed_to_global(0) == 4 && ids.packed_to_global(1) == 2 && ids.packed_to_global(2) == 5);
    CHECK(ids.packed_to_global(3) == 6 && ids.packed_to_global(4) == 7);
    CHECK(ids.global_to_packed(2) == 1 && ids.global_to_packed(7) == 4);
    bool stale = false;
    try {
        ids.global_to_packed(3);
    } catch (const std::runtime_error &) {
        stale = true;
    }
    CHECK(stale);

    CHECK(instantiate<NormalInverseChiSq>() && instantiate<GammaPoisson>() && instantiate<BetaNegativeBinomial>() &&
          instantiate<BetaBernoulli>() && instantiate<DirichletDiscrete<16>>() && instantiate<DirichletProcessDiscrete>() &&
          instantiate<NormalInverseWishart<3>>());
    std::printf("ok\n");
    return 0;
}
