// GPU test of binary segmentation through the header-only shim (genomic_b200/host/cbs_gpu.hpp): cbs_gpu::segment(x, true, ...)
// and cbs_gpu::fndcpt(..., ibin = true, ...) against the oracle restatement (liboracle.so), the engine used before and after.
#include <cmath>
#include <cstdio>
#include <random>
#include <vector>

#include "../../genomic_b200/host/cbs_gpu.hpp"
#include "../../oracle/cbs_oracle.h"

static int fails = 0;
#define CHECK(c) do { if (!(c)) { std::printf("FAIL line %d: %s\n", __LINE__, #c); ++fails; } } while (0)

int main() {
    std::mt19937_64 g(17);
    std::uniform_real_distribution<double> u(0.0, 1.0);
    std::vector<double> y(2400);
    for (size_t i = 0; i < y.size(); ++i) y[i] = u(g) < ((i >= 800 && i < 1300) ? 0.6 : 0.3) ? 1.0 : 0.0;
    for (int al0 : {2, 3}) {  // cbs::segment with ibin = true
        std::mt19937_64 rng(7);
        rng.discard(500);
        orc_rng orng;
        orc_rng_seed_mt(&orng, 7);
        orc_rng_discard(&orng, 500);
        const int nperm = 400;
        std::vector<int> sbdry(2000, nperm + 1);
        const auto seg = cbs_gpu::segment(y, true, 0.01, nperm, false, al0, 25, 200, 0.05, sbdry, 1e-6, rng);
        orc_seg_opts o = {1, 0.01, nperm, 0, al0, 25, 200, 0.05, 1e-6, 0, 0.05};
        std::vector<int> len(y.size());
        std::vector<double> mean(y.size());
        const int k = orc_segment(y.data(), (int)y.size(), &o, &orng, 7, 0, (int)y.size(), len.data(), mean.data(), nullptr, 0, nullptr);
        CHECK(k == (int)seg.lengths.size());
        CHECK(k >= 3);
        for (int i = 0; i < k && i < (int)seg.lengths.size(); ++i) { CHECK(len[i] == seg.lengths[i]); CHECK(mean[i] == seg.means[i]); }
        for (int i = 0; i < 5; ++i) CHECK(rng() == orc_rng_u64(&orng));  // both engines at the same position
    }
    {   // cbs::fndcpt with ibin = true on a centred segment
        double s = 0.0;
        for (double v : y) s += v;
        const double avg = s / (double)y.size();
        std::vector<double> yc(y);
        double tss = 0.0;
        for (auto& v : yc) v -= avg;
        for (double v : yc) tss += v * v;
        std::mt19937_64 rng(5);
        rng.discard(100);
        orc_rng orng;
        orc_rng_seed_mt(&orng, 5);
        orc_rng_discard(&orng, 100);
        const int nperm = 600;
        std::vector<int> sbdry(2000, nperm + 1);
        const auto cp = cbs_gpu::fndcpt(yc, tss, nperm, 0.05, true, false, 2, 25, 0.0, 100, sbdry, 1e-6, rng);
        const orc_cpt oc = orc_fndcpt(yc.data(), (int)yc.size(), tss, nperm, 0.05, 1, 0, 2, 25, 0.0, 100, 1e-6, &orng);
        CHECK(cp.ncpt == oc.ncpt); CHECK(cp.iseg[0] == oc.iseg[0] && cp.iseg[1] == oc.iseg[1]); CHECK(cp.ostat == oc.ostat);
        if (oc.ncpt >= 1) CHECK(cp.icpt[0] == oc.icpt[0]);
        if (oc.ncpt == 2) CHECK(cp.icpt[1] == oc.icpt[1]);
        for (int i = 0; i < 5; ++i) CHECK(rng() == orc_rng_u64(&orng));
    }
    {   // hybrid together with ibin is refused (CBS_GPU_ERR_UNSUPPORTED becomes std::runtime_error)
        std::mt19937_64 rng(1);
        std::vector<int> sbdry(400, 201);
        bool threw = false;
        try { cbs_gpu::segment(y, true, 0.01, 200, true, 2, 25, 200, 0.05, sbdry, 1e-6, rng); } catch (const std::runtime_error&) { threw = true; }
        CHECK(threw);
    }
    std::printf("%s (%d failures)\n", fails ? "FAILED" : "ok", fails);
    return fails ? 1 : 0;
}
