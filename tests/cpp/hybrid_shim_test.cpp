// GPU test of the hybrid method through the header-only shim (genomic_b200/host/cbs_gpu.hpp): the calls the reference leaves
// undefined become std::runtime_error (CBS_GPU_ERR_UNSUPPORTED), and cbs_gpu::fndcpt(hybrid) on kmax <= n <= 2 kmax markers
// equals the oracle restatement (liboracle.so), the engine used before and after.
#include <cmath>
#include <cstdio>
#include <random>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../genomic_b200/host/cbs_gpu.hpp"
#include "../../oracle/cbs_oracle.h"

static int fails = 0;
#define CHECK(c) do { if (!(c)) { std::printf("FAIL line %d: %s\n", __LINE__, #c); ++fails; } } while (0)

template <class F>
static bool refused(F f, const char* text) {
    try { f(); } catch (const std::runtime_error& e) { return std::string(e.what()).find(text) != std::string::npos; }
    return false;
}

int main() {
    std::mt19937_64 g(23);
    std::normal_distribution<double> nd(0.0, 0.2);
    std::vector<double> y(400);
    for (size_t i = 0; i < y.size(); ++i) y[i] = nd(g) + ((i >= 150 && i < 156) ? 1.0 : 0.0);
    const int nperm = 200;
    std::vector<int> sbdry(2000, nperm + 1);
    {   // cbs::segment with hybrid and nmin <= kmax
        std::mt19937_64 rng(1);
        CHECK(refused([&] { cbs_gpu::segment(y, false, 0.05, nperm, true, 2, 25, 25, 0.05, sbdry, 1e-6, rng); },
                      "hybrid CBS needs nmin >= kmax + 1"));
        CHECK(refused([&] { cbs_gpu::segment(y, false, 0.05, nperm, true, 2, 128, 0, 0.05, sbdry, 1e-6, rng); },
                      "hybrid CBS needs nmin >= kmax + 1"));
    }
    for (int n : {24, 26, 40, 50}) {  // cbs::fndcpt(hybrid, hk = 25): refused below hk + 2 with delta = 0, compared above
        std::vector<double> x(y.begin() + 140, y.begin() + 140 + n);
        double s = 0.0;
        for (double v : x) s += v;
        const double avg = s / (double)n;
        double tss = 0.0;
        for (auto& v : x) v -= avg;
        for (double v : x) tss += v * v;
        std::mt19937_64 rng(5);
        rng.discard(300);
        if (n < 27) {
            CHECK(refused([&] { cbs_gpu::fndcpt(x, tss, nperm, 0.05, false, true, 2, 25, 0.0, 100, sbdry, 1e-6, rng); },
                          "hybrid fndcpt needs n >= hk and delta < 1"));
            continue;
        }
        orc_rng orng;
        orc_rng_seed_mt(&orng, 5);
        orc_rng_discard(&orng, 300);
        const auto cp = cbs_gpu::fndcpt(x, tss, nperm, 0.05, false, true, 2, 25, 0.0, 100, sbdry, 1e-6, rng);
        const orc_cpt oc = orc_fndcpt(x.data(), n, tss, nperm, 0.05, 0, 1, 2, 25, 26.0 / n, 100, 1e-6, &orng);
        CHECK(cp.ncpt == oc.ncpt); CHECK(cp.iseg[0] == oc.iseg[0] && cp.iseg[1] == oc.iseg[1]); CHECK(cp.ostat == oc.ostat);
        if (oc.ncpt >= 1) CHECK(cp.icpt[0] == oc.icpt[0]);
        if (oc.ncpt == 2) CHECK(cp.icpt[1] == oc.icpt[1]);
        for (int i = 0; i < 5; ++i) CHECK(rng() == orc_rng_u64(&orng));  // both engines at the same position
    }
    std::printf("%s (%d failures)\n", fails ? "FAILED" : "ok", fails);
    return fails ? 1 : 0;
}
