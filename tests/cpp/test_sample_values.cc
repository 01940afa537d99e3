// Drives Mixture<Model>::sample_values and CrossCat::sample_values of the C++ host mirror
// (include/distributions_b200/mixture.hpp): groups are filled with Group::add_value before init, then the draws are
// printed; tests/test_gpu_sample_values.py compares them with the C-ABI's draws for the same statistics and seed.
#include <distributions_b200/mixture.hpp>

#include <cstdio>

using namespace distributions_b200;

template <class T>
static void print_vec(const char * tag, const T * v, size_t n) {
    std::printf("%s", tag);
    for (size_t i = 0; i < n; ++i) std::printf(" %u", static_cast<unsigned>(v[i]));
    std::printf("\n");
}

int main() {
    auto ctx = std::make_shared<Context>(0);
    rng_t rng;
    const uint64_t seed = 7, row0 = 100;
    const size_t n = 8;
    const int32_t ids[n] = {0, 1, 2, 1, -1, 0, 3, 2};  // -1 and 3 (= G) keep their values

    GammaPoisson::Shared gs{2.f, 0.5f};
    Mixture<GammaPoisson> gp(ctx);
    gp.groups().resize(3);
    for (auto & g : gp.groups()) g.init(gs, rng);
    for (uint32_t v = 0; v < 20; ++v) gp.groups(1).add_value(gs, v, rng);
    for (uint32_t v = 0; v < 5; ++v) gp.groups(2).add_value(gs, 100 + v, rng);
    gp.init(gs, rng);
    std::vector<uint32_t> gv(n, 12345u);
    gp.sample_values(gs, ids, n, seed, row0, gv.data());
    print_vec("gp", gv.data(), n);

    BetaBernoulli::Shared bs{0.5f, 2.f};
    Mixture<BetaBernoulli> bb(ctx);
    bb.groups().resize(3);
    for (auto & g : bb.groups()) g.init(bs, rng);
    for (int i = 0; i < 10; ++i) bb.groups(1).add_value(bs, true, rng);
    for (int i = 0; i < 10; ++i) bb.groups(2).add_value(bs, false, rng);
    bb.init(bs, rng);
    bool bv[n] = {true, true, true, true, true, true, true, true};
    bb.sample_values(bs, ids, n, seed, row0, bv);
    print_vec("bb", bv, n);

    CrossCat kind(ctx);
    kind.add_feature(gp.feature(), nullptr);
    kind.add_feature(bb.feature(), nullptr);
    std::vector<uint32_t> c0(n, 12345u);
    std::vector<uint8_t> c1(n, 7);
    void * cols[2] = {c0.data(), c1.data()};
    kind.sample_values(n, ids, seed, row0, cols);
    print_vec("kind0", c0.data(), n);
    print_vec("kind1", c1.data(), n);
    return 0;
}
