// Drives Mixture<Model>::score_logp_values and CrossCat::score_logp_values of the C++ host mirror
// (include/distributions_b200/mixture.hpp): groups are filled with Group::add_value before init, then the row
// log-likelihoods are printed as float bit patterns; tests/test_gpu_score_logp.py compares them with the C-ABI's.
#include <distributions_b200/mixture.hpp>

#include <cstdio>
#include <cstring>

using namespace distributions_b200;

static void print_bits(const char * tag, const float * v, size_t n) {
    std::printf("%s", tag);
    for (size_t i = 0; i < n; ++i) {
        uint32_t b;
        std::memcpy(&b, v + i, 4);
        std::printf(" %u", static_cast<unsigned>(b));
    }
    std::printf("\n");
}

int main() {
    auto ctx = std::make_shared<Context>(0);
    rng_t rng;
    const size_t n = 8;
    const float prior[3] = {-0.5f, -1.25f, -2.f};

    GammaPoisson::Shared gs{2.f, 0.5f};
    Mixture<GammaPoisson> gp(ctx);
    gp.groups().resize(3);
    for (auto & g : gp.groups()) g.init(gs, rng);
    for (uint32_t v = 0; v < 20; ++v) gp.groups(1).add_value(gs, v, rng);
    for (uint32_t v = 0; v < 5; ++v) gp.groups(2).add_value(gs, 100 + v, rng);
    gp.init(gs, rng);
    const uint32_t gv[n] = {0, 3, 9, 17, 40, 101, 250, 1};
    float lp[n];
    gp.score_logp_values(gs, gv, n, prior, lp);
    print_bits("gp", lp, n);

    BetaBernoulli::Shared bs{0.5f, 2.f};
    Mixture<BetaBernoulli> bb(ctx);
    bb.groups().resize(3);
    for (auto & g : bb.groups()) g.init(bs, rng);
    for (int i = 0; i < 10; ++i) bb.groups(1).add_value(bs, true, rng);
    for (int i = 0; i < 10; ++i) bb.groups(2).add_value(bs, false, rng);
    bb.init(bs, rng);
    const bool bv[n] = {true, false, true, true, false, false, true, false};
    bb.score_logp_values(bs, bv, n, nullptr, lp);
    print_bits("bb", lp, n);

    CrossCat kind(ctx);
    const uint8_t bw[n] = {1, 0, 1, 1, 0, 0, 1, 0};
    kind.add_feature(gp.feature(), gv);
    kind.add_feature(bb.feature(), bw);
    kind.score_logp_values(n, prior, lp);
    print_bits("kind", lp, n);
    return 0;
}
