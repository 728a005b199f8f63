// cbs_gpu.cu -- host driver and C ABI (include/cbs_gpu.h) of libcbs_cuda.so.
//
// The host only stages buffers and enqueues rounds; every decision of the recursive split
// (cbs::segment / cbs::fndcpt) is taken on the device by k_sched over a device-resident
// worklist.  Rounds are enqueued in groups without reading anything back; a mapped
// host flag written by k_sched tells the host when to stop enqueueing.
#include <cub/cub.cuh>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstddef>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "../../include/cbs_gpu.h"
#include "host_math.h"
#include "kernels.cuh"
#include "binary.cuh"
#include "weighted.cuh"
#include "mt_jump.h"
#include "prune.h"
#include "smooth.cuh"

using namespace cbsg;

static_assert(GEN_SEG == cbsg::mtjump::SEG && GEN_NSEG == cbsg::mtjump::NSEG && GEN_LEAD == cbsg::mtjump::LEAD,
              "generator geometry must match the jump table");

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    template <class T> T* as() const { return (T*)p; }
};

enum KernelId { K_SCHED = 0, K_GEN, K_PREP, K_PERM, K_SCAN, K_EDGEPREP, K_EDGEPERM, K_MEANS, K_SMOOTH, K_SHUF0, K_SHUF1, K_SHUF2, K_SHUF3, K_PREFIX, K_COUNT };

}  // namespace

struct cbs_gpu_ctx {
    int device = 0;
    int sm_count = 148;
    size_t smem_optin = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::string err;
    int* h_done = nullptr;  // mapped pinned
    cudaGraphExec_t call_exec = nullptr;  // graph of a whole call: WHILE node around one scheduler round (run_cbs)
    std::vector<unsigned char> call_key;  // the launch configuration it was captured with
    unsigned long long round_launches = 0;
    int* d_done = nullptr;  // device alias of h_done
    DevBuf x, cur, gtab, factab, bbtab, unit_off, unit_ids, tasks, ring, act0, act1, chains, segs, splits, udraws, arena,
        rej, draws0, draws1, prep_task, items, item_prefix, edgeprep_task, edges, edge_prefix, gen_chain, means, seed312,
        dev, staging, fv, fidx, flab, lab, diffs, diffs_sorted, sm_keys, sm_gid, cn_scratch, gout, cubtmp, flag, goff, stream_buf, shuf, jump, tailp,
        wts, rw, cw, ycur;  // weighted CBS
    bool jump_ready = false;
    // lanes: a call with independent units is split into contiguous unit ranges that run as separate
    // worklists on their own streams (child contexts), so the latency-bound phases of one lane overlap
    // the other's; results are merged in unit order
    std::vector<cbs_gpu_ctx*> lanes;
    double mem_fraction = 0.80;  // share of free device memory the arenas of this context may take
    bool is_lane = false;
    bool profiling = false;   // per-launch CUDA events
    bool serial = false;      // all kernels of a round on one stream (non-overlapping per-kernel times)
    bool counting = false;    // scan work counters (atomics in the kernel: slows it, never combine with timing)
    double kms[K_COUNT] = {0};
    std::vector<cudaEvent_t> ev_pool;
    std::vector<std::pair<int, int>> ev_used;  // (kernel id, index of start event); stop = start+1
    size_t ev_next = 0;
    uint64_t launches = 0;
    uint64_t last_arcs = 0, last_slots = 0;
    cudaEvent_t e0 = nullptr, e1 = nullptr, e2 = nullptr, e3 = nullptr, e4 = nullptr;
    cudaEvent_t grp[2] = {nullptr, nullptr};
    // side streams: kernels of one round that do not depend on each other run concurrently
    cudaStream_t side[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t ev_sched = nullptr, ev_gen = nullptr, ev_side[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    cudaStream_t gen_stream = nullptr;  // the MT stream is generated one round ahead on this stream
    cudaEvent_t ev_ahead = nullptr;
};

namespace {

int fail(cbs_gpu_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg;
    return code;
}

#define CUDA_TRY(c, expr)                                                                                   \
    do {                                                                                                    \
        cudaError_t e__ = (expr);                                                                           \
        if (e__ != cudaSuccess)                                                                             \
            return fail(c, e__ == cudaErrorMemoryAllocation ? CBS_GPU_ERR_OOM : CBS_GPU_ERR_CUDA,           \
                        std::string(#expr) + ": " + cudaGetErrorString(e__));                               \
    } while (0)

int ensure(cbs_gpu_ctx* c, DevBuf& b, size_t bytes) {
    if (bytes <= b.cap && b.p) return CBS_GPU_OK;
    if (b.p) { cudaFree(b.p); b.p = nullptr; b.cap = 0; }
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&b.p, want);
    if (e != cudaSuccess) {
        cudaGetLastError();
        want = bytes + 256;
        e = cudaMalloc(&b.p, want);
    }
    if (e != cudaSuccess) { cudaGetLastError(); b.p = nullptr; return fail(c, CBS_GPU_ERR_OOM, "cudaMalloc failed for " + std::to_string(bytes) + " bytes"); }
    b.cap = want;
    return CBS_GPU_OK;
}
#define ENSURE(c, buf, bytes)                                   \
    do {                                                        \
        const int rc__ = ensure(c, buf, bytes);                 \
        if (rc__ != CBS_GPU_OK) return rc__;                    \
    } while (0)

// event-bracketed launch bookkeeping (profiling mode)
struct LaunchTimer {
    cbs_gpu_ctx* c;
    int kid;
    int idx = -1;
    cudaStream_t s;
    LaunchTimer(cbs_gpu_ctx* ctx, int k, cudaStream_t stream = nullptr) : c(ctx), kid(k), s(stream ? stream : ctx->stream) {
        c->launches++;
        if (!c->profiling) return;
        if (c->ev_next + 2 > c->ev_pool.size()) {
            const size_t old = c->ev_pool.size();
            c->ev_pool.resize(old + 1024);
            for (size_t i = old; i < c->ev_pool.size(); ++i) cudaEventCreate(&c->ev_pool[i]);
        }
        idx = (int)c->ev_next;
        c->ev_next += 2;
        cudaEventRecord(c->ev_pool[idx], s);
    }
    ~LaunchTimer() {
        if (idx < 0) return;
        cudaEventRecord(c->ev_pool[idx + 1], s);
        c->ev_used.emplace_back(kid, idx);
    }
};

void collect_timers(cbs_gpu_ctx* c) {
    // CBS_GPU_DEBUG_ROUNDS=1: timeline of the call on stderr, one line per round: kernel=start+duration in ms relative to the
    // first launch (launches shorter than 0.05 ms are left out)
    const bool dump = getenv("CBS_GPU_DEBUG_ROUNDS") != nullptr;
    static const char* names[] = {"sched", "gen", "prep", "perm", "scan", "edgeprep", "edgeperm", "means", "smooth", "shuf0", "shuf1", "shuf2", "shuf3", "prefix"};
    int round = 0;
    for (auto& u : c->ev_used) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, c->ev_pool[u.second], c->ev_pool[u.second + 1]) == cudaSuccess) c->kms[u.first] += ms;
        if (dump) {
            float at = 0.f;
            cudaEventElapsedTime(&at, c->ev_pool[c->ev_used[0].second], c->ev_pool[u.second]);
            if (u.first == K_SCHED) fprintf(stderr, "\n[round %d @%.2f]", round++, at);
            if (ms > 0.05f) fprintf(stderr, " %s=%.2f+%.2f", names[u.first], at, ms);
        }
    }
    if (dump) fprintf(stderr, "\n");
    c->ev_used.clear();
    c->ev_next = 0;
}

int validate_params(cbs_gpu_ctx* c, const cbs_gpu_params* p) {
    if (!p) return fail(c, CBS_GPU_ERR_INVALID, "params is NULL");
    if (p->ibin && p->hybrid) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "ibin=true with hybrid=true is not implemented: htmaxp has no binary variant");
    if (p->hybrid && (p->kmax < 1 || p->kmax > 128)) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "hybrid: kmax must be in 1..128");
    if (p->min_width < 1) return fail(c, CBS_GPU_ERR_INVALID, "min_width must be >= 1");
    if (p->nperm < 0) return fail(c, CBS_GPU_ERR_INVALID, "nperm must be >= 0");
    if (!(p->alpha >= 0.0)) return fail(c, CBS_GPU_ERR_INVALID, "alpha must be >= 0");
    if (p->rng_mode != CBS_GPU_RNG_MT19937_64 && p->rng_mode != CBS_GPU_RNG_PHILOX)
        return fail(c, CBS_GPU_ERR_INVALID, "unknown rng_mode");
    if (p->do_smooth) {
        if (p->smooth_region < 0) return fail(c, CBS_GPU_ERR_INVALID, "smooth_region must be non-negative");
        if (p->smooth_region > SM_MAX_REGION) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "smooth_region > 64 is not supported");
    }
    return CBS_GPU_OK;
}

// ---- smoothing on device buffers -------------------------------------------------------------
// xin: values (double, device, N), goff: device group offsets [n_groups+1], dlab: labels or nullptr
// (constant label per group), out: device N. host_off is the host copy of the offsets.
long long env_ll(const char* name, long long dflt) {
    const char* s = getenv(name);
    if (!s || !*s) return dflt;
    return atoll(s);
}

int smooth_device(cbs_gpu_ctx* c, const double* xin, const long long* goff, const int* dlab, int n_groups, long long N,
                  int region, double oscale, double sscale, double trim, double* out, const std::vector<long long>& host_off) {
    if (region < 0) return fail(c, CBS_GPU_ERR_INVALID, "smooth_region must be non-negative");
    if (region > SM_MAX_REGION) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "smooth_region > 64 is not supported");
    cudaStream_t st = c->stream;
    CUDA_TRY(c, cudaMemcpyAsync(out, xin, sizeof(double) * (size_t)N, cudaMemcpyDeviceToDevice, st));
    if (N == 0 || n_groups == 0) return CBS_GPU_OK;
    ENSURE(c, c->fv, sizeof(double) * (size_t)N);
    ENSURE(c, c->fidx, sizeof(int) * (size_t)N);
    if (dlab) ENSURE(c, c->flab, sizeof(int) * (size_t)N);
    ENSURE(c, c->diffs, sizeof(double) * (size_t)N);
    ENSURE(c, c->diffs_sorted, sizeof(double) * (size_t)N);
    ENSURE(c, c->gout, sizeof(SmoothGroupOut) * (size_t)n_groups);
    int* flab = dlab ? c->flab.as<int>() : nullptr;
    SmoothGroupOut* gout = c->gout.as<SmoothGroupOut>();
    {
        LaunchTimer t(c, K_SMOOTH);
        k_sm_compact<<<std::min(n_groups, c->sm_count * 8), 256, 0, st>>>(xin, goff, dlab, n_groups, c->fv.as<double>(),
                                                                         c->fidx.as<int>(), flab, gout);
    }
    // the reference validates trim only when it reaches inflfact (>= 2 finite values and n_keep > 0)
    std::vector<SmoothGroupOut> hg((size_t)n_groups);
    CUDA_TRY(c, cudaMemcpyAsync(hg.data(), gout, sizeof(SmoothGroupOut) * (size_t)n_groups, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    bool reaches = false;
    for (int g = 0; g < n_groups; ++g)
        if (hg[g].m >= 2 && llround((1.0 - 2.0 * trim) * (double)(hg[g].m - 1)) > 0) reaches = true;
    double infl = 1.0;
    if (reaches) {
        if (!(trim >= 0.0 && trim < 0.5)) return fail(c, CBS_GPU_ERR_INVALID, "trim must satisfy 0 <= trim < 0.5");
        if (trim == 0.0) return fail(c, CBS_GPU_ERR_OVERFLOW, "trim == 0: normal quantile at 1 overflows (boost::math::quantile raises overflow_error)");
        infl = inflfact(trim);
    }
    const int maxn = (int)std::min<long long>(N, 1 << 20);
    // Ascending order of the differences inside every group.  A segmented sort spends most of its time on the few very long
    // segments (1.7 ms for one SNP6 sample); two device-wide radix sorts do the same in a third of that: all (difference,
    // group) pairs by difference, then -- radix sorts are stable -- by the few bits of the group number.  24 B per marker of
    // scratch, so calls beyond CBS_GPU_SMOOTH_RADIX_MAX markers (default 256 M) keep the segmented sort.
    const bool radix = N <= env_ll("CBS_GPU_SMOOTH_RADIX_MAX", 256LL << 20) && n_groups > 1;
    if (radix) {
        ENSURE(c, c->sm_keys, sizeof(double) * (size_t)N);
        ENSURE(c, c->sm_gid, sizeof(int) * (size_t)N * 3);
    }
    int* gid0 = radix ? c->sm_gid.as<int>() : nullptr;
    {
        LaunchTimer t(c, K_SMOOTH);
        dim3 grid((unsigned)std::max(1, std::min((maxn + 255) / 256, 64)), (unsigned)std::min(n_groups, 65535));
        k_sm_diffs<<<grid, 256, 0, st>>>(c->fv.as<double>(), goff, n_groups, gout, c->diffs.as<double>(), gid0);
    }
    if (radix) {
        LaunchTimer t(c, K_SMOOTH);
        int* gid1 = gid0 + N;
        int* gid2 = gid1 + N;
        int gbits = 1;
        while ((1LL << gbits) < n_groups) ++gbits;
        size_t tmp1 = 0, tmp2 = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tmp1, c->diffs.as<double>(), c->sm_keys.as<double>(), gid0, gid1, (int)N, 0, 64, st);
        cub::DeviceRadixSort::SortPairs(nullptr, tmp2, gid1, gid2, c->sm_keys.as<double>(), c->diffs_sorted.as<double>(), (int)N, 0, gbits, st);
        ENSURE(c, c->cubtmp, std::max(tmp1, tmp2) + 16);
        CUDA_TRY(c, cub::DeviceRadixSort::SortPairs(c->cubtmp.p, tmp1, c->diffs.as<double>(), c->sm_keys.as<double>(), gid0, gid1, (int)N, 0, 64, st));
        CUDA_TRY(c, cub::DeviceRadixSort::SortPairs(c->cubtmp.p, tmp2, gid1, gid2, c->sm_keys.as<double>(), c->diffs_sorted.as<double>(), (int)N, 0, gbits, st));
    } else if (n_groups == 1) {
        LaunchTimer t(c, K_SMOOTH);
        size_t tmp = 0;
        cub::DeviceRadixSort::SortKeys(nullptr, tmp, c->diffs.as<double>(), c->diffs_sorted.as<double>(), (int)N, 0, 64, st);
        ENSURE(c, c->cubtmp, tmp + 16);
        CUDA_TRY(c, cub::DeviceRadixSort::SortKeys(c->cubtmp.p, tmp, c->diffs.as<double>(), c->diffs_sorted.as<double>(), (int)N, 0, 64, st));
    } else {
        LaunchTimer t(c, K_SMOOTH);
        size_t tmp = 0;
        cub::DeviceSegmentedSort::SortKeys(nullptr, tmp, c->diffs.as<double>(), c->diffs_sorted.as<double>(), (int)N, n_groups,
                                           goff, goff + 1, st);
        ENSURE(c, c->cubtmp, tmp + 16);
        CUDA_TRY(c, cub::DeviceSegmentedSort::SortKeys(c->cubtmp.p, tmp, c->diffs.as<double>(), c->diffs_sorted.as<double>(),
                                                       (int)N, n_groups, goff, goff + 1, st));
    }
    {
        LaunchTimer t(c, K_SMOOTH);
        k_sm_sd<<<std::min(n_groups, c->sm_count * 8), 32, 0, st>>>(c->diffs_sorted.as<double>(), goff, n_groups,
                                                                              trim, infl, oscale, sscale, gout);
    }
    {
        LaunchTimer t(c, K_SMOOTH);
        dim3 grid((unsigned)std::max(1, std::min((maxn + 255) / 256, 256)), (unsigned)std::min(n_groups, 65535));
        k_sm_window<<<grid, 256, 0, st>>>(c->fv.as<double>(), c->fidx.as<int>(), flab, goff, n_groups, region, gout, out);
    }
    CUDA_TRY(c, cudaGetLastError());
    (void)host_off;
    return CBS_GPU_OK;
}

// warps per scan CTA of kernel `kern` (k_scan_perm / k_scan_obs): the block and extrema tables are per CTA; take the CTA
// shape that keeps the most warps resident on an SM
bool pick_scan_warps(cbs_gpu_ctx* c, ScanLayout& lay, int* occ_out, const void* kern) {
    int best_w = 0, best_res = 0, best_occ = 1;
    const int forced = (int)env_ll("CBS_GPU_SCAN_WARPS", 0);  // experiments only
    for (int w : {8, 4, 2, 1}) {
        if (forced && w != forced) continue;
        lay.warps = w;
        if (lay.bytes() > c->smem_optin) continue;
        int occ = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, w * 32, lay.bytes()) != cudaSuccess) { cudaGetLastError(); continue; }
        if (occ * w > best_res || (occ * w == best_res && w == 8)) { best_res = occ * w; best_w = w; best_occ = occ; }
    }
    if (!best_w) return false;
    lay.warps = best_w;
    if (occ_out) *occ_out = std::max(1, best_occ);
    return true;
}
// the scan of the round's observed rows or of its permutation rows; the counting instantiations only when D->profile is set
void launch_scan(bool obs, bool prof, int grid, const ScanLayout& lay, cudaStream_t s, Dev* dD) {
    const unsigned threads = (unsigned)lay.warps * 32;
    if (obs) { if (prof) k_scan_obs<true><<<grid, threads, lay.bytes(), s>>>(dD, lay); else k_scan_obs<false><<<grid, threads, lay.bytes(), s>>>(dD, lay); }
    else { if (prof) k_scan_perm<true><<<grid, threads, lay.bytes(), s>>>(dD, lay); else k_scan_perm<false><<<grid, threads, lay.bytes(), s>>>(dD, lay); }
}
int obs_slice_cap() { return (int)std::min<long long>(64, std::max<long long>(1, env_ll("CBS_GPU_OBS_SLICES", OBS_SLICES_MAX))); }

// shared-memory shuffle classes (cbs_core.h): dynamic shared memory of a CTA = claim table + last[] of the longest segment
size_t shuffle_smem_bytes(int cls) { return ((size_t)4 << shuffle_class_hbits(cls)) + (((size_t)shuffle_class_max(cls) + 2) * 2 + 15) / 16 * 16; }
template <bool MT>
void launch_shuffle_t(Dev* dD, int cls, int grid, cudaStream_t ss) {
    const size_t smem = shuffle_smem_bytes(cls);
    const int hb = shuffle_class_hbits(cls);
    switch (shuffle_class_threads(cls)) {
    case 128: k_shuffle<128, 2, MT><<<grid, 128, smem, ss>>>(dD, cls, hb); break;
    case 256: k_shuffle<256, 2, MT><<<grid, 256, smem, ss>>>(dD, cls, hb); break;
    case 512: k_shuffle<512, 2, MT><<<grid, 512, smem, ss>>>(dD, cls, hb); break;
    default: k_shuffle<1024, 2, MT><<<grid, 1024, smem, ss>>>(dD, cls, hb); break;
    }
}
void launch_shuffle(Dev* dD, int cls, int grid, cudaStream_t ss, bool mt) {
    if (mt) launch_shuffle_t<true>(dD, cls, grid, ss); else launch_shuffle_t<false>(dD, cls, grid, ss);
}
template <bool MT>
void launch_shuffle_cluster_t(Dev* dD, int R, int cls, int hbits, int grid, size_t smem, cudaStream_t ss) {
    if (R == 2) k_shuffle_cluster<1024, 4, 2, MT><<<grid, 1024, smem, ss>>>(dD, cls, hbits);
    else if (R == 4) k_shuffle_cluster<1024, 4, 4, MT><<<grid, 1024, smem, ss>>>(dD, cls, hbits);
    else k_shuffle_cluster<1024, 4, 8, MT><<<grid, 1024, smem, ss>>>(dD, cls, hbits);
}
void launch_shuffle_cluster(Dev* dD, int R, int cls, int hbits, int grid, size_t smem, cudaStream_t ss, bool mt) {
    if (mt) launch_shuffle_cluster_t<true>(dD, R, cls, hbits, grid, smem, ss); else launch_shuffle_cluster_t<false>(dD, R, cls, hbits, grid, smem, ss);
}
int shuffle_occupancy(int cls) {
    int occ = 0;
    const size_t smem = shuffle_smem_bytes(cls);
    cudaError_t e;
    switch (shuffle_class_threads(cls)) {
    case 128: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_shuffle<128, 2, true>, 128, smem); break;
    case 256: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_shuffle<256, 2, true>, 256, smem); break;
    case 512: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_shuffle<512, 2, true>, 512, smem); break;
    default: e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_shuffle<1024, 2, true>, 1024, smem); break;
    }
    if (e != cudaSuccess) { cudaGetLastError(); occ = 1; }
    return std::max(1, occ);
}
template <class F>
bool set_max_smem(F* f, int bytes) { return cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes) == cudaSuccess; }

// resident clusters x R of k_shuffle_cluster for segments of up to nmax markers (0: does not fit / not schedulable)
int cluster_fit(cbs_gpu_ctx* c, int R, long long nmax, int hbits, size_t* smem_out) {
    const size_t smem = ((size_t)4 << hbits) + 4 * ((size_t)nmax / R + 4);
    if (smem > c->smem_optin) return 0;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(c->sm_count / R * R); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension; at[0].val.clusterDim.x = R; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int ncl = 0;
    cudaError_t e = R == 2 ? cudaOccupancyMaxActiveClusters(&ncl, k_shuffle_cluster<1024, 4, 2, true>, &cfg)
                  : R == 4 ? cudaOccupancyMaxActiveClusters(&ncl, k_shuffle_cluster<1024, 4, 4, true>, &cfg)
                           : cudaOccupancyMaxActiveClusters(&ncl, k_shuffle_cluster<1024, 4, 8, true>, &cfg);
    if (e != cudaSuccess || ncl < 1) { cudaGetLastError(); return 0; }
    *smem_out = smem;
    return ncl * R;
}

struct RunCaps {
    int task_cap, list_cap, seg_cap, split_cap, max_live;
    long long arena_cap, draws_cap, rej_cap;
};

// The core: x already resident (double, device, smoothed if requested) in c->x.
struct ApiMode {   // low-level entry points: ONE decision on the vector as given (cbs_core.h Dev::api_mode)
    int mode = 0;
    double tss = 0.0, delta = 0.0;
    int n1 = 0, n2 = 0;
};

int run_cbs(cbs_gpu_ctx* c, const std::vector<long long>& off, const uint64_t* unit_ids, int n_units,
            const cbs_gpu_params* p, const uint64_t* mt_next312, bool weighted /* weights resident in c->wts */, Dev& hD,
            const ApiMode& api = ApiMode()) {
    cudaStream_t st = c->stream;
    // CBS_GPU_DEBUG_SETUP=1: host wall clock of the set-up phases on stderr
    const bool setup_debug = getenv("CBS_GPU_DEBUG_SETUP") != nullptr;
    auto setup_t0 = std::chrono::steady_clock::now();
    auto setup_mark = [&](const char* what) {
        if (!setup_debug) return;
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[setup] %s %.3f ms\n", what, std::chrono::duration<double, std::milli>(now - setup_t0).count());
        setup_t0 = now;
    };
    // profiling bit 2: every kernel on the one stream, so that per-launch event times do not overlap (roofline time base)
    cudaStream_t side[5], gen_stream = c->serial ? st : c->gen_stream;
    for (int k = 0; k < 5; ++k) side[k] = c->serial ? st : c->side[k];
    const long long N = off[n_units];
    long long Nmax = 0;
    for (int u = 0; u < n_units; ++u) Nmax = std::max(Nmax, off[u + 1] - off[u]);
    if (Nmax > 1000000) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "units longer than 1,000,000 markers are not supported");
    if (N > 2000000000LL) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "more than 2e9 markers per call are not supported");
    const bool mt = p->rng_mode == CBS_GPU_RNG_MT19937_64;
    if (weighted && p->ibin) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "weighted CBS has no binary mode (cbs::segment_weighted takes no ibin)");
    if (weighted && p->hybrid && p->nmin < p->kmax + 2)
        return fail(c, CBS_GPU_ERR_UNSUPPORTED, "weighted hybrid CBS needs nmin >= kmax + 2");

    RunCaps cap;
    cap.task_cap = (int)std::min<long long>(std::max<long long>(4096, 64LL * n_units + 1024), 1 << 22);
    cap.task_cap = (int)std::max<long long>(64, std::min<long long>(env_ll("CBS_GPU_TASK_CAP", cap.task_cap), 1 << 24));  // env overrides: sane range only
    cap.list_cap = 4 * cap.task_cap + n_units + 16;
    cap.seg_cap = (int)std::min<long long>(N / 2 + n_units + 16, std::max<long long>(1 << 20, 256LL * n_units));
    cap.seg_cap = (int)std::max<long long>(n_units + 16, std::min<long long>(env_ll("CBS_GPU_SEG_CAP", cap.seg_cap), 1LL << 30));
    cap.split_cap = (p->record_splits || api.mode) ? 3 * cap.seg_cap + 16 : 1;
    cap.max_live = mt ? std::max(1, cap.task_cap / 16) : std::max(1, cap.task_cap / 4);
    // MT with one engine per unit: every chain reads the one shared stream from position 0 and the stream window only moves
    // forward once all chains have started, so admit them all in the first round
    if (mt && !p->chain) cap.max_live = std::max(cap.max_live, n_units);
    cap.rej_cap = 1 << 22;

    ENSURE(c, c->cur, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->gtab, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->factab, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->bbtab, sizeof(int) * (size_t)(N + 1));
    if (weighted) {
        ENSURE(c, c->rw, sizeof(double) * (size_t)(N + 1));
        ENSURE(c, c->cw, sizeof(double) * (size_t)(N + 1));
        ENSURE(c, c->ycur, sizeof(double) * (size_t)(N + 1));
        ENSURE(c, c->flag, sizeof(int));
    }
    ENSURE(c, c->unit_off, sizeof(long long) * (size_t)(n_units + 1));
    ENSURE(c, c->unit_ids, sizeof(uint64_t) * (size_t)(n_units + 1));
    ENSURE(c, c->tasks, sizeof(Task) * (size_t)cap.task_cap);
    ENSURE(c, c->ring, sizeof(int) * (size_t)cap.task_cap);
    ENSURE(c, c->act0, sizeof(int) * (size_t)cap.list_cap);
    ENSURE(c, c->act1, sizeof(int) * (size_t)cap.list_cap);
    const int n_chains = mt ? (p->chain ? 1 : n_units) : 0;
    ENSURE(c, c->chains, sizeof(Chain) * (size_t)std::max(1, n_chains));
    ENSURE(c, c->segs, sizeof(SegRec) * (size_t)cap.seg_cap);
    ENSURE(c, c->splits, sizeof(SplitRec) * (size_t)cap.split_cap);
    ENSURE(c, c->udraws, sizeof(uint64_t) * (size_t)(n_units + 1));
    ENSURE(c, c->rej, sizeof(int) * (size_t)cap.rej_cap);
    ENSURE(c, c->prep_task, sizeof(int) * (size_t)cap.list_cap);
    ENSURE(c, c->items, sizeof(PermItem) * (size_t)cap.list_cap);
    ENSURE(c, c->item_prefix, sizeof(int) * (size_t)(cap.list_cap + 1));
    ENSURE(c, c->edgeprep_task, sizeof(int) * (size_t)cap.list_cap);
    ENSURE(c, c->edges, sizeof(EdgeItem) * (size_t)cap.list_cap);
    ENSURE(c, c->edge_prefix, sizeof(int) * (size_t)(cap.list_cap + 1));
    ENSURE(c, c->gen_chain, sizeof(int) * (size_t)(n_chains + 1));
    ENSURE(c, c->shuf, sizeof(int) * (3 * SHUF_NCLS + 1) * (size_t)(cap.list_cap + 1));
    ENSURE(c, c->means, sizeof(double) * (size_t)cap.seg_cap);
    ENSURE(c, c->seed312, sizeof(uint64_t) * 312);
    ENSURE(c, c->dev, sizeof(Dev));
    if (p->hybrid) ENSURE(c, c->tailp, sizeof(double) * 100 * (size_t)cap.list_cap);  // tailp quadrature terms per new segment

    setup_mark("buffers");
    // arenas: sized from the workload, bounded by what the device has left
    const long long per_perm_max = 3 * Nmax + 64;
    long long want_arena = std::min<long long>(24LL * 4096 * std::max<long long>(N, 1), 32LL << 30) / 8;
    want_arena = std::max<long long>(want_arena, 16 * per_perm_max);
    want_arena = std::max<long long>(want_arena, (64LL << 20) / 8);
    const bool shared_stream = mt && !p->chain;
    long long want_draws = (mt && !shared_stream) ? std::max<long long>(want_arena / 3, 8 * (Nmax + 312)) : 1;
    // shared raw MT stream (chain == 0): as long as the largest consumption of any one unit
    // shared raw MT stream (chain == 0): a ring of 2^k words (default 16 GB, CBS_GPU_STREAM_MB) + a mirror of its first words
    // (any permutation and the generator's lead-in must be readable linearly).  The ring is a WINDOW on the stream: when the
    // fastest chain is a whole window ahead of the slowest it waits (cbs_core.h plan_perm), so a small ring costs time, never an error.
    const long long stream_mirror = shared_stream ? std::max<long long>(Nmax, GEN_LEAD) + 1024 : 0;
    long long stream_ring = 0;
    if (shared_stream) {
        const long long asked = std::max<long long>(env_ll("CBS_GPU_STREAM_MB", 16384), 1) * (1LL << 20) / 8;
        const long long least = 8 * (Nmax + 312) + 4 * GEN_LEAD;  // a quarter of the ring must hold one permutation
        stream_ring = 1;
        while (stream_ring < least) stream_ring <<= 1;
        while (stream_ring * 2 <= asked) stream_ring <<= 1;
    }
    long long want_stream = shared_stream ? stream_ring + stream_mirror : 0;
    const long long env_arena = env_ll("CBS_GPU_ARENA_MB", 0);
    if (env_arena > 0) { want_arena = env_arena * (1LL << 20) / 8; if (mt && !shared_stream) want_draws = std::max<long long>(want_arena / 3, 8 * (Nmax + 312)); }
    // (cudaMemGetInfo goes to the kernel driver and was measured to take tens of milliseconds now and then: it is asked only
    // when a buffer has to grow, i.e. normally on the first call of a context)
    const bool must_grow = (long long)(c->arena.cap / 8) < want_arena || (shared_stream && (long long)(c->stream_buf.cap / 8) < want_stream) ||
                           (mt && !shared_stream && (long long)(std::min(c->draws0.cap, c->draws1.cap) / 8) < want_draws);
    if (must_grow) {
        size_t free_b = 0, total_b = 0;
        CUDA_TRY(c, cudaMemGetInfo(&free_b, &total_b));
        const size_t have = c->arena.cap + c->draws0.cap + c->draws1.cap + c->stream_buf.cap;
        const double budget = c->mem_fraction * (double)(free_b + have);
        const double need = 8.0 * ((double)want_arena + 2.0 * (double)want_draws + (double)want_stream);
        if (need > budget) {
            const double f = budget / need;
            want_arena = (long long)((double)want_arena * f);
            want_draws = (long long)((double)want_draws * f);
            if (shared_stream) {  // the ring stays a power of two and never shrinks below what one permutation needs
                const long long least = 8 * (Nmax + 312) + 4 * GEN_LEAD;
                while (stream_ring / 2 >= least && (double)(stream_ring + stream_mirror) > (double)want_stream * f) stream_ring >>= 1;
                want_stream = stream_ring + stream_mirror;
            }
        }
    }
    if (want_arena < 4 * per_perm_max) return fail(c, CBS_GPU_ERR_OOM, "not enough device memory for the permutation arena");
    if ((long long)(c->arena.cap / 8) < want_arena) ENSURE(c, c->arena, (size_t)want_arena * 8);
    if (shared_stream && (long long)(c->stream_buf.cap / 8) < want_stream) ENSURE(c, c->stream_buf, (size_t)want_stream * 8);
    if (mt && !shared_stream) {
        if ((long long)(c->draws0.cap / 8) < want_draws) ENSURE(c, c->draws0, (size_t)want_draws * 8);
        if ((long long)(c->draws1.cap / 8) < want_draws) ENSURE(c, c->draws1, (size_t)want_draws * 8);
    }
    cap.arena_cap = (long long)(c->arena.cap / 8);
    cap.draws_cap = (mt && !shared_stream) ? (long long)(std::min(c->draws0.cap, c->draws1.cap) / 8) : 0;

    setup_mark("arenas");
    // ---- device state ---------------------------------------------------------------------
    memset(&hD, 0, sizeof(hD));
    hD.x = c->x.as<double>();
    hD.unit_off = c->unit_off.as<long long>();
    hD.unit_ids = unit_ids ? c->unit_ids.as<uint64_t>() : nullptr;
    hD.n_units = n_units;
    hD.prm.alpha = p->alpha; hD.prm.nperm = p->nperm; hD.prm.hybrid = p->hybrid; hD.prm.min_width = p->min_width;
    hD.prm.kmax = p->kmax; hD.prm.nmin = p->nmin; hD.prm.eta = p->eta; hD.prm.tol = p->tol; hD.prm.ibin = p->ibin;
    hD.prm.rng_mode = mt ? RNG_MT : RNG_PHILOX; hD.prm.chain = p->chain ? 1 : 0; hD.prm.seed = p->seed;
    hD.prm.first_batch = p->first_batch > 0 ? p->first_batch : 256;
    hD.prm.max_batch = p->max_batch > 0 ? p->max_batch : 4096;
    // a batch needs one rejection flag per permutation: never ask for more than the flag table holds (it would be deferred forever)
    hD.prm.first_batch = (int)std::min<long long>(hD.prm.first_batch, cap.rej_cap / 4);
    hD.prm.max_batch = (int)std::min<long long>(hD.prm.max_batch, cap.rej_cap / 4);
    if (hD.prm.max_batch < hD.prm.first_batch) hD.prm.max_batch = hD.prm.first_batch;
    hD.prm.record_splits = (p->record_splits || api.mode) ? 1 : 0;
    hD.api_mode = api.mode; hD.api_tss = api.tss; hD.api_delta = api.delta; hD.api_n1 = api.n1; hD.api_n2 = api.n2;
    if (api.mode) hD.prm.nmin = 0;  // cbs::fndcpt takes `hybrid` as given (cbs::segment derives it from nmin, CBS.cpp:983)
    hD.cur = c->cur.as<double>(); hD.gtab = c->gtab.as<double>(); hD.factab = c->factab.as<double>(); hD.bbtab = c->bbtab.as<int>();
    hD.tasks = c->tasks.as<Task>(); hD.task_cap = cap.task_cap; hD.free_ring = c->ring.as<int>();
    hD.free_head = 0; hD.free_tail = (unsigned)cap.task_cap;
    hD.active[0] = c->act0.as<int>(); hD.active[1] = c->act1.as<int>(); hD.list_cap = cap.list_cap;
    hD.chains = c->chains.as<Chain>(); hD.n_chains = n_chains;
    hD.units_started = 0; hD.max_live = cap.max_live;
    hD.segs = c->segs.as<SegRec>(); hD.seg_cap = cap.seg_cap;
    hD.splits = c->splits.as<SplitRec>(); hD.split_cap = cap.split_cap;
    hD.unit_draws = c->udraws.as<uint64_t>();
    hD.arena = c->arena.as<double>(); hD.arena_cap = cap.arena_cap;
    hD.rej = c->rej.as<int>(); hD.rej_cap = cap.rej_cap;
    hD.draws[0] = c->draws0.as<uint64_t>(); hD.draws[1] = c->draws1.as<uint64_t>(); hD.draws_cap = cap.draws_cap;
    hD.prep_task = c->prep_task.as<int>(); hD.items = c->items.as<PermItem>(); hD.item_prefix = c->item_prefix.as<int>();
    hD.edgeprep_task = c->edgeprep_task.as<int>(); hD.edges = c->edges.as<EdgeItem>(); hD.edge_prefix = c->edge_prefix.as<int>();
    hD.gen_chain = c->gen_chain.as<int>();
    for (int k = 0; k < SHUF_NCLS; ++k) {
        hD.shuf_item[k] = c->shuf.as<int>() + (size_t)(2 * k) * (cap.list_cap + 1);
        hD.shuf_prefix[k] = c->shuf.as<int>() + (size_t)(2 * k + 1) * (cap.list_cap + 1);
    }
    hD.item_uprefix = c->shuf.as<int>() + (size_t)(2 * SHUF_NCLS) * (cap.list_cap + 1);
    for (int k = 0; k < SHUF_NCLS; ++k) hD.shuf_p0[k] = c->shuf.as<int>() + (size_t)(2 * SHUF_NCLS + 1 + k) * (cap.list_cap + 1);
    hD.shared_stream = shared_stream ? 1 : 0;
    hD.stream = c->stream_buf.as<uint64_t>();
    hD.stream_cap = stream_ring; hD.stream_mask = stream_ring - 1; hD.stream_mirror = stream_mirror; hD.stream_lo = 0;
    hD.stream_len = 312; hD.stream_target = 312; hD.stream_target_prev = 312;
    hD.jump_polys = nullptr;
    hD.span_max = 1LL << 40;
    if (shared_stream && (long long)Nmax * hD.prm.first_batch > mtjump::SEG && !env_ll("CBS_GPU_NO_JUMP", 0)) {
        // parallel generation of the one stream: table of x^(c*S) mod phi, built once per process
        if (!c->jump_ready) {
            const mtjump::Table& T = mtjump::table();
            if (T.ok) {
                ENSURE(c, c->jump, sizeof(uint64_t) * T.polys.size());
                CUDA_TRY(c, cudaMemcpyAsync(c->jump.p, T.polys.data(), sizeof(uint64_t) * T.polys.size(), cudaMemcpyHostToDevice, st));
                CUDA_TRY(c, cudaStreamSynchronize(st));
                c->jump_ready = true;
            }
        }
        if (c->jump_ready) { hD.jump_polys = c->jump.as<uint64_t>(); hD.span_max = (long long)mtjump::NSEG * mtjump::SEG; }
    }
    hD.profile = c->counting ? 1 : 0;
    hD.shuf_arena = 1;  // decided below (cluster shuffle available?) and patched on the device before the first round
    hD.no_early = env_ll("CBS_GPU_NO_EARLY", 0) ? 1 : 0;
    hD.obs_slices = obs_slice_cap();
    if (weighted) {
        hD.w = c->wts.as<double>(); hD.rw = c->rw.as<double>(); hD.cw = c->cw.as<double>(); hD.ycur = c->ycur.as<double>();
        CUDA_TRY(c, cudaMemsetAsync(c->flag.p, 0, sizeof(int), st));
        if (N) { k_wsetup<<<std::min<long long>((N + 255) / 256, c->sm_count * 8), 256, 0, st>>>(hD.w, hD.rw, N, c->flag.as<int>()); c->launches++; }
        int bad = 0;
        CUDA_TRY(c, cudaMemcpyAsync(&bad, c->flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        if (bad) return fail(c, CBS_GPU_ERR_INVALID, "weights must be finite and positive");
    }
    CUDA_TRY(c, cudaMemcpyAsync(c->unit_off.p, off.data(), sizeof(long long) * (size_t)(n_units + 1), cudaMemcpyHostToDevice, st));
    if (unit_ids) CUDA_TRY(c, cudaMemcpyAsync(c->unit_ids.p, unit_ids, sizeof(uint64_t) * (size_t)n_units, cudaMemcpyHostToDevice, st));
    {
        std::vector<int> ring((size_t)cap.task_cap);
        for (int i = 0; i < cap.task_cap; ++i) ring[i] = i;
        CUDA_TRY(c, cudaMemcpyAsync(c->ring.p, ring.data(), sizeof(int) * ring.size(), cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaMemsetAsync(c->udraws.p, 0, sizeof(uint64_t) * (size_t)(n_units + 1), st));
        CUDA_TRY(c, cudaMemcpyAsync(c->dev.p, &hD, sizeof(Dev), cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));  // `ring` is a stack temporary
    }
    Dev* dD = c->dev.as<Dev>();
    if (api.mode == 2 && N) CUDA_TRY(c, cudaMemcpyAsync(c->cur.p, c->x.p, sizeof(double) * (size_t)N, cudaMemcpyDeviceToDevice, st));  // no k_prep in this mode
    if (mt) {
        uint64_t next[312];
        if (mt_next312) memcpy(next, mt_next312, sizeof(next)); else mt_seed_next312(p->seed, next);
        CUDA_TRY(c, cudaMemcpyAsync(c->seed312.p, next, sizeof(next), cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        k_init_chains<<<std::min(std::max(1, n_chains), 1024), 128, 0, st>>>(dD, c->seed312.as<uint64_t>());
        if (shared_stream) {  // positions 0..311 (and their mirror)
            CUDA_TRY(c, cudaMemcpyAsync(c->stream_buf.p, next, sizeof(next), cudaMemcpyHostToDevice, st));
            CUDA_TRY(c, cudaMemcpyAsync(c->stream_buf.as<uint64_t>() + stream_ring, next, sizeof(next), cudaMemcpyHostToDevice, st));
        }
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }

    setup_mark("device state");
    // ---- scan kernel configuration ------------------------------------------------------------
    ScanLayout lay;
    lay.nb_max = block_count((int)std::max<long long>(Nmax, 1)) + 2;
    lay.set_table(std::max<long long>(Nmax, 1));
    int scan_occ = 1, obs_occ = 1;
    ScanLayout lay_obs = lay;
    if (!pick_scan_warps(c, lay, &scan_occ, (const void*)k_scan_perm<false>) ||
        !pick_scan_warps(c, lay_obs, &obs_occ, (const void*)k_scan_obs<false>))
        return fail(c, CBS_GPU_ERR_UNSUPPORTED, "segment too long for the scan kernel's shared memory");
    const bool scan_prof = hD.profile != 0;
    const int obs_grid = c->sm_count * obs_occ;
    const size_t wscan_smem = ((sizeof(WScanSmem) + 15) & ~(size_t)15) + (size_t)lay.nb_max * (2 * sizeof(double) + 3 * sizeof(int)) + 16;
    const int scan_grid = c->sm_count * scan_occ;
    const size_t bscan_smem = ((sizeof(BinSmem) + 15) & ~(size_t)15) + (size_t)lay.nb_max * (2 * sizeof(double) + 3 * sizeof(int)) + 16;

    // shared-memory shuffle kernel, one launch per segment-length class present in this call
    int shuf_occ[SHUF_CL2]; bool shuf_on[SHUF_CL2];
    for (int cls = 0; cls < SHUF_CL2; ++cls) {
        shuf_on[cls] = (cls == 0) || Nmax > shuffle_class_max(cls - 1);  // no unit is long enough otherwise
        shuf_occ[cls] = shuf_on[cls] ? shuffle_occupancy(cls) : 1;
    }
    const bool l2_shuffle_on = Nmax > shuffle_class_max(SHUF_CL2 - 1);
    // segments > 65535 markers: a cluster of 2, 4 or 8 CTAs per permutation shares last[] through distributed shared
    // memory; units too long even for that (or CBS_GPU_SHUF_CLUSTER=0) fall back to k_perm (index arrays in the arena)
    int cl_R = 0, cl_grid = 0, cl2_grid = 0;
    const int cl_hbits = 12;
    size_t cl_smem = 0, cl2_smem = 0;
    auto cluster_fit_l = [&](int R, long long nmax, size_t* smem_out) -> int { return cluster_fit(c, R, nmax, cl_hbits, smem_out); };
    if (l2_shuffle_on && env_ll("CBS_GPU_SHUF_CLUSTER", 1)) {
        if (Nmax > SHUF_CL2_MAX) {
            for (int R : {4, 8}) { cl_grid = cluster_fit_l(R, Nmax, &cl_smem); if (cl_grid) { cl_R = R; break; } }
        } else cl_R = -1;  // nothing longer than the cluster-of-2 class
        if (cl_R) cl2_grid = cluster_fit_l(2, std::min<long long>(Nmax, SHUF_CL2_MAX), &cl2_smem);
        if (cl_R < 0) { cl_R = cl2_grid ? 2 : 0; }
    }
    static const int kShufTimer[SHUF_CL2] = {K_SHUF0, K_SHUF1, K_SHUF2, K_SHUF2, K_SHUF3, K_SHUF3};

    if (cl_R) {
        hD.shuf_arena = 0;
        hD.shuf_cl2 = cl2_grid ? 1 : 0;
        CUDA_TRY(c, cudaMemcpyAsync((char*)dD + offsetof(Dev, shuf_arena), &hD.shuf_arena, sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaMemcpyAsync((char*)dD + offsetof(Dev, shuf_cl2), &hD.shuf_cl2, sizeof(int), cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
    }

    int chain_occ = 4;
    if ((weighted ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&chain_occ, k_chain<true>, 32 * (1 + CP_STAT_WARPS), 0)
                  : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&chain_occ, k_chain<false>, 32 * (1 + CP_STAT_WARPS), 0)) != cudaSuccess) { cudaGetLastError(); chain_occ = 4; }
    chain_occ = std::max(1, chain_occ);

    setup_mark("launch configuration");
    // ---- rounds -------------------------------------------------------------------------------
    *c->h_done = 0;
    const int G = (int)std::min<long long>(64, std::max<long long>(1, env_ll("CBS_GPU_ROUND_GROUP", 16)));
    // rounds per group; two groups are kept in flight, so the host is 16-32 rounds ahead of the device and its scheduling
    // jitter cannot starve the GPU; the rounds enqueued beyond the last one find D->done set and every kernel returns at once
    const bool debug = env_ll("CBS_GPU_DEBUG", 0) != 0;
    int groups_in_flight = 0, rounds = 0;
    int gi = 0;
    // One round = one fork-join of launches over the main stream, the side streams and the generator stream, and every launch
    // configuration is fixed for the call.  The round is therefore captured ONCE as the body of a WHILE node of a CUDA graph
    // whose condition the scheduler kernel keeps at 1 until the work list is empty: the whole call is one graph launch, the
    // device runs exactly the rounds it needs and the host plays no part between them.  The instantiated graph is kept in
    // the context and reused by later calls with the same configuration.  Event-timed profiling, CBS_GPU_DEBUG and
    // CBS_GPU_GRAPH=0 enqueue the rounds from the host instead, in groups with a done flag polled in between.
    cudaGraphConditionalHandle loop_handle = 0;
    int looped = 0;
    auto enqueue_round = [&]() {
        bool ahead_pending = false;
        // One round.  Dependencies: everything after k_sched; shuffles after the generator;
        // k_prefix after the shuffles; k_scan_perm after k_prefix; k_scan_obs after k_prep; next k_sched after all.
        // A task's permutations are planned in a later round than its observed scan (Sched::step), so neither scan
        // of a round reads what the other writes, and the observed scans run beside the shuffles.
        //   main : sched, gen, [shuffle classes], prefix, scan_perm
        //   side0: prep, scan_obs  side1: edgeprep, edgeperm
        //   side2, side3: other shuffle classes      side4: shuffle of segments > 65535 markers
        { LaunchTimer t(c, K_SCHED); k_sched<<<1, 256, 0, st>>>(dD, c->d_done, loop_handle, looped); }
        cudaEventRecord(c->ev_sched, st);
        cudaStreamWaitEvent(side[0], c->ev_sched, 0);
        { LaunchTimer t(c, K_PREP, side[0]); k_tables<<<dim3(16, 64), 256, 0, side[0]>>>(dD); if (weighted) { k_wprep<<<c->sm_count * 8, 32, 0, side[0]>>>(dD); k_wtables<<<c->sm_count * 2, 256, 0, side[0]>>>(dD); c->launches++; if (p->hybrid) { k_wdelta<<<c->sm_count * 2, 32, 0, side[0]>>>(dD); c->launches++; } } else k_prep<<<c->sm_count * 8, 32, 0, side[0]>>>(dD); c->launches++; }
        const bool scan_split = !weighted && !p->ibin;
        if (scan_split) { LaunchTimer t(c, K_SCAN, side[0]); launch_scan(true, scan_prof, obs_grid, lay_obs, side[0], dD); }
        cudaEventRecord(c->ev_side[0], side[0]);
        cudaStreamWaitEvent(side[1], c->ev_sched, 0);
        { LaunchTimer t(c, K_EDGEPREP, side[1]); if (weighted) k_wedgeprep<<<c->sm_count * 4, 32, 0, side[1]>>>(dD); else k_edgeprep<<<c->sm_count * 4, 32, 0, side[1]>>>(dD); }
        if (mt) {
            LaunchTimer t(c, K_GEN);
            if (shared_stream) {
                k_gen_lead<<<1, 192, 0, st>>>(dD, 0);
                if (hD.jump_polys) { k_gen_par<<<GEN_NSEG, 320, 0, st>>>(dD); c->launches++; }
            } else k_gen<<<std::min(std::max(1, n_chains), c->sm_count * 4), 192, 0, st>>>(dD);
        }
        cudaEventRecord(c->ev_gen, st);
        // the edge permutations read this round's draws (plan_edge asked the generator for them): after the generator
        if (mt) cudaStreamWaitEvent(side[1], c->ev_gen, 0);
        { LaunchTimer t(c, K_EDGEPERM, side[1]); if (weighted) k_wedgeperm<<<c->sm_count * 4, 128, 0, side[1]>>>(dD); else k_edgeperm<<<c->sm_count * 4, 128, 0, side[1]>>>(dD); }
        cudaEventRecord(c->ev_side[1], side[1]);
        if (mt && shared_stream && hD.jump_polys) {
            // generate ahead for the next round, next to this round's shuffles and scan
            cudaStreamWaitEvent(gen_stream, c->ev_gen, 0);
            k_gen_lead<<<1, 192, 0, gen_stream>>>(dD, 1);
            k_gen_par<<<GEN_NSEG, 320, 0, gen_stream>>>(dD);
            c->launches += 2;
            cudaEventRecord(c->ev_ahead, gen_stream);
            ahead_pending = true;
        }
        // shuffles: classes alternate between the main stream and three side streams so that they run
        // concurrently (each class is latency bound on its own); the longest present class goes first
        bool used_side[5] = {false, false, false, false, false};
        {
            int slot = 0;
            if (l2_shuffle_on) {
                cudaStream_t ss = side[4];
                cudaStreamWaitEvent(ss, c->ev_gen, 0);
                used_side[4] = true;
                LaunchTimer t(c, K_PERM, ss);
                if (cl_R == 4 || cl_R == 8) launch_shuffle_cluster(dD, cl_R, SHUF_GLOBAL, cl_hbits, cl_grid, cl_smem, ss, mt);
                else if (cl_R == 0) k_perm<<<c->sm_count * 8, 128, 0, ss>>>(dD);
                if (cl2_grid) { launch_shuffle_cluster(dD, 2, SHUF_CL2, cl_hbits, cl2_grid, cl2_smem, ss, mt); c->launches++; }
            }
            for (int cls = SHUF_CL2 - 1; cls >= 0; --cls) {
                if (!shuf_on[cls]) continue;
                const int where = slot++ % 3;  // 0 = main stream, 1,2 = side[2], side[3]
                cudaStream_t ss = where == 0 ? st : side[1 + where];
                if (where != 0 && !used_side[1 + where]) { cudaStreamWaitEvent(ss, c->ev_gen, 0); used_side[1 + where] = true; }
                LaunchTimer t(c, kShufTimer[cls], ss);
                launch_shuffle(dD, cls, c->sm_count * shuf_occ[cls], ss, mt);
            }
        }
        for (int k = 2; k < 5; ++k) if (used_side[k]) { cudaEventRecord(c->ev_side[k], side[k]); cudaStreamWaitEvent(st, c->ev_side[k], 0); }
        { LaunchTimer t(c, K_PREFIX); if (weighted && p->hybrid) { k_wssq<<<c->sm_count * 8, 128, 0, st>>>(dD); c->launches++; } if (weighted) k_chain<true><<<c->sm_count * chain_occ, 32 * (1 + CP_STAT_WARPS), 0, st>>>(dD); else k_chain<false><<<c->sm_count * chain_occ, 32 * (1 + CP_STAT_WARPS), 0, st>>>(dD); }
        if (!scan_split) cudaStreamWaitEvent(st, c->ev_side[0], 0);
        { LaunchTimer t(c, K_SCAN);
          if (weighted) {
              k_wscan<1><<<c->sm_count * 4, 256, wscan_smem, st>>>(dD, lay.nb_max);   // observed rows, sliced over CTAs
              k_wobs_fin<<<8, 128, 0, st>>>(dD);
              k_wscan<0><<<c->sm_count * 4, 256, wscan_smem, st>>>(dD, lay.nb_max);   // permutation rows
              c->launches += 2;
          }
          else if (p->ibin) k_scan_binary<<<c->sm_count * 4, 256, bscan_smem, st>>>(dD, lay.nb_max);
          else launch_scan(false, scan_prof, scan_grid, lay, st, dD); }
        if (scan_split) cudaStreamWaitEvent(st, c->ev_side[0], 0);  // the tail probabilities read the observed statistics
        if (p->hybrid) {
            if (weighted) k_whscan<<<c->sm_count * 4, 256, 0, st>>>(dD); else k_hscan<<<c->sm_count * 4, 256, 0, st>>>(dD);
            k_tailp_terms<<<c->sm_count * 8, 128, 0, st>>>(dD, c->tailp.as<double>());
            k_tailp_sum<<<c->sm_count, 64, 0, st>>>(dD, c->tailp.as<double>());
            c->launches += 3;
        }
        cudaStreamWaitEvent(st, c->ev_side[1], 0);
        if (ahead_pending) cudaStreamWaitEvent(st, c->ev_ahead, 0);  // the next k_sched plans on the extended stream
    };
    const bool use_graph = !c->profiling && !debug && env_ll("CBS_GPU_GRAPH", 1) != 0;
    unsigned long long launches_per_round = 0;
    cudaGraphExec_t call_exec = nullptr;
    if (use_graph) {
        std::vector<unsigned char> key;
        auto put = [&](const void* v, size_t nbytes) { const unsigned char* b = (const unsigned char*)v; key.insert(key.end(), b, b + nbytes); };
#define KEY_POD(v) put(&(v), sizeof(v))
        const int flags[7] = {weighted ? 1 : 0, mt ? 1 : 0, shared_stream ? 1 : 0, hD.jump_polys ? 1 : 0, p->hybrid ? 1 : 0, l2_shuffle_on ? 1 : 0,
                              p->ibin ? 1 : 0};
        KEY_POD(dD); KEY_POD(st); KEY_POD(flags); KEY_POD(n_chains); KEY_POD(shuf_occ); KEY_POD(shuf_on); KEY_POD(cl_R); KEY_POD(cl_grid);
        KEY_POD(cl2_grid); KEY_POD(cl_smem); KEY_POD(cl2_smem); KEY_POD(chain_occ); KEY_POD(scan_grid); KEY_POD(obs_grid); KEY_POD(scan_prof);
        KEY_POD(wscan_smem); KEY_POD(bscan_smem); KEY_POD(lay); KEY_POD(lay_obs);
        const void* tailp_ptr = c->tailp.p; KEY_POD(tailp_ptr);
#undef KEY_POD
        if (c->call_exec && key == c->call_key) {
            call_exec = c->call_exec;
            launches_per_round = c->round_launches;
        } else {
            if (c->call_exec) { cudaGraphExecDestroy(c->call_exec); c->call_exec = nullptr; }
            const unsigned long long before = c->launches;
            cudaGraph_t graph = nullptr;
            cudaError_t ce = cudaGraphCreate(&graph, 0);
            if (ce == cudaSuccess) ce = cudaGraphConditionalHandleCreate(&loop_handle, graph, 1, cudaGraphCondAssignDefault);
            cudaGraphNodeParams wp = {cudaGraphNodeTypeConditional};
            wp.conditional.handle = loop_handle;
            wp.conditional.type = cudaGraphCondTypeWhile;
            wp.conditional.size = 1;
            cudaGraphNode_t wnode = nullptr;
            if (ce == cudaSuccess) ce = cudaGraphAddNode(&wnode, graph, nullptr, 0, &wp);
            if (ce == cudaSuccess) {
                looped = 1;
                ce = cudaStreamBeginCaptureToGraph(st, wp.conditional.phGraph_out[0], nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed);
                if (ce == cudaSuccess) {
                    enqueue_round();
                    ce = cudaStreamEndCapture(st, nullptr);
                }
                looped = 0;
            }
            launches_per_round = c->launches - before;
            c->launches = before;
            if (ce == cudaSuccess) ce = cudaGraphInstantiate(&call_exec, graph, 0);
            if (graph) cudaGraphDestroy(graph);
            if (ce != cudaSuccess) {
                // (a driver without conditional nodes, or a capture that could not be closed: rounds are enqueued by the host)
                cudaGetLastError();
                call_exec = nullptr;
                if (env_ll("CBS_GPU_GRAPH", 1) == 2) return fail(c, CBS_GPU_ERR_CUDA, std::string("call graph: ") + cudaGetErrorString(ce));
            } else {
                c->call_exec = call_exec;
                c->call_key = key;
                c->round_launches = launches_per_round;
            }
        }
    }
    setup_mark("graph");
    if (call_exec) {
        CUDA_TRY(c, cudaGraphLaunch(call_exec, st));
        CUDA_TRY(c, cudaStreamSynchronize(st));
        if (*(volatile int*)c->h_done == 0) return fail(c, CBS_GPU_ERR_CUDA, "the call graph ended before the scheduler was done");
    }
    for (; !call_exec;) {
        for (int r = 0; r < G; ++r) {
            enqueue_round();
            ++rounds;
        }
        CUDA_TRY(c, cudaEventRecord(c->grp[gi], st));
        gi ^= 1;
        ++groups_in_flight;
        if (groups_in_flight == 2) {
            CUDA_TRY(c, cudaEventSynchronize(c->grp[gi]));  // the older group
            --groups_in_flight;
            if (*(volatile int*)c->h_done != 0) break;
            if (debug) {
                Dev snap;
                cudaMemcpy(&snap, dD, sizeof(Dev), cudaMemcpyDeviceToHost);  // synchronises: debugging only
                fprintf(stderr, "[cbs_gpu] enq=%d round=%d live=%d items=%d perms=%d prep=%d edgeprep=%d edge=%d gen=%d segs=%d perms_done=%llu err=%d\n",
                        rounds, snap.round, snap.n_active[snap.cur_list], snap.n_items, snap.item_prefix ? -1 : 0, snap.n_prep,
                        snap.n_edgeprep, snap.n_edge, snap.n_gen, snap.n_segs, snap.stat_perms, snap.error);
            }
        }
        if (rounds > 50000000) { cudaDeviceSynchronize(); return fail(c, CBS_GPU_ERR_CUDA, "scheduler did not terminate"); }
    }
    // everything that was enqueued (up to two groups of rounds, on the main, generator and side streams) has to be over before
    // anything is read back or an error is reported
    for (int k = 0; k < 5; ++k) cudaStreamSynchronize(side[k]);
    CUDA_TRY(c, cudaStreamSynchronize(gen_stream));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpy(&hD, dD, sizeof(Dev), cudaMemcpyDeviceToHost));
    if (call_exec) c->launches += launches_per_round * (unsigned long long)std::max(1, hD.round);  // one body per scheduler round
    if (hD.error) {
        switch (hD.error) {
        case ERR_TASK_CAP: return fail(c, CBS_GPU_ERR_CAPACITY, "pending-segment pool exhausted (raise CBS_GPU_TASK_CAP)");
        case ERR_SEG_CAP: return fail(c, CBS_GPU_ERR_CAPACITY, "segment table exhausted (raise CBS_GPU_SEG_CAP)");
        case ERR_SPLIT_CAP: return fail(c, CBS_GPU_ERR_CAPACITY, "split log exhausted");
        case ERR_STALL: return fail(c, CBS_GPU_ERR_CUDA, "scheduler stalled: live segments but no work could be planned");
        case ERR_STREAM_CAP: return fail(c, CBS_GPU_ERR_CAPACITY, "MT stream window smaller than one permutation (raise CBS_GPU_STREAM_MB)");
        case ERR_ARENA: return fail(c, CBS_GPU_ERR_OOM, "permutation arena too small for one segment (raise CBS_GPU_ARENA_MB)");
        default: return fail(c, CBS_GPU_ERR_CUDA, "internal scheduler error " + std::to_string(hD.error));
        }
    }
    if (getenv("CBS_GPU_DEBUG_ROUNDS")) {
        fprintf(stderr, "[rounds] planned perms / markers per round:");
        for (int r = 0; r < std::min(hD.round, 64); ++r) fprintf(stderr, " %d:%llu/%.1fM", r, hD.round_perms[r], hD.round_elems[r] * 1e-6);
        fprintf(stderr, "\n");
        if (hD.shared_stream) fprintf(stderr, "[stream] words generated %.1fM, furthest word asked for %.1fM\n", hD.stream_len * 1e-6, hD.stream_target * 1e-6);
    }
    if (hD.n_segs > 0) {
        LaunchTimer t(c, K_MEANS);
        if (weighted) k_wmeans<<<std::min(hD.n_segs, c->sm_count * 8), 32, 0, st>>>(dD, c->means.as<double>());
        else k_means<<<std::min(hD.n_segs, c->sm_count * 8), 32, 0, st>>>(dD, c->means.as<double>());
    }
    CUDA_TRY(c, cudaGetLastError());
    return CBS_GPU_OK;
}

struct ResultOwner {
    cbs_gpu_result pub;
    std::vector<int64_t> seg_offsets;
    std::vector<int32_t> lengths;
    std::vector<double> means;
    std::vector<uint64_t> draws;
    std::vector<cbs_gpu_split> splits;
};

int fetch_results(cbs_gpu_ctx* c, const Dev& hD, int n_units, bool want_splits, ResultOwner* R, const cbs_gpu_params* prm = nullptr,
                  const std::vector<long long>* unit_off = nullptr, bool weighted = false) {
    cudaStream_t st = c->stream;
    const int ns = hD.n_segs;
    std::vector<SegRec> segs((size_t)ns);
    std::vector<double> means((size_t)ns);
    R->draws.assign((size_t)n_units, 0);
    if (ns) {
        CUDA_TRY(c, cudaMemcpyAsync(segs.data(), c->segs.p, sizeof(SegRec) * (size_t)ns, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(c, cudaMemcpyAsync(means.data(), c->means.p, sizeof(double) * (size_t)ns, cudaMemcpyDeviceToHost, st));
    }
    if (n_units) CUDA_TRY(c, cudaMemcpyAsync(R->draws.data(), c->udraws.p, sizeof(uint64_t) * (size_t)n_units, cudaMemcpyDeviceToHost, st));
    std::vector<SplitRec> sp;
    if (want_splits && hD.n_splits) {
        sp.resize((size_t)hD.n_splits);
        CUDA_TRY(c, cudaMemcpyAsync(sp.data(), c->splits.p, sizeof(SplitRec) * sp.size(), cudaMemcpyDeviceToHost, st));
    }
    CUDA_TRY(c, cudaStreamSynchronize(st));
    // order segments by (unit, lo)
    std::vector<int> order((size_t)ns);
    for (int i = 0; i < ns; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) {
        if (segs[a].unit != segs[b].unit) return segs[a].unit < segs[b].unit;
        return segs[a].lo < segs[b].lo;
    });
    R->seg_offsets.assign((size_t)n_units + 1, 0);
    R->lengths.resize((size_t)ns);
    R->means.resize((size_t)ns);
    for (int k = 0; k < ns; ++k) {
        const SegRec& s = segs[order[k]];
        R->lengths[k] = s.hi - s.lo;
        R->means[k] = means[order[k]];
        R->seg_offsets[(size_t)s.unit + 1]++;
    }
    for (int u = 0; u < n_units; ++u) R->seg_offsets[u + 1] += R->seg_offsets[u];
    if (prm && prm->undo_prune && unit_off) {
        // CBS.cpp:1013-1022: prune on the host, then means of the merged segments (sequential sums)
        const long long N = (*unit_off)[n_units];
        std::vector<double> hx((size_t)N);
        if (N) CUDA_TRY(c, cudaMemcpy(hx.data(), c->x.p, sizeof(double) * (size_t)N, cudaMemcpyDeviceToHost));
        std::vector<double> hw;
        if (weighted && N) { hw.resize((size_t)N); CUDA_TRY(c, cudaMemcpy(hw.data(), c->wts.p, sizeof(double) * (size_t)N, cudaMemcpyDeviceToHost)); }
        std::vector<int64_t> noff((size_t)n_units + 1, 0);
        std::vector<int32_t> nlen;
        std::vector<double> nmean;
        for (int u = 0; u < n_units; ++u) {
            std::vector<int> lseg(R->lengths.begin() + R->seg_offsets[u], R->lengths.begin() + R->seg_offsets[u + 1]);
            const double* xu = hx.data() + (*unit_off)[u];
            const int n = (int)((*unit_off)[u + 1] - (*unit_off)[u]);
            if (lseg.size() > 1) lseg = prune_lengths(xu, n, lseg, prm->undo_prune_cutoff);
            int pos = 0;
            for (int len : lseg) {
                nlen.push_back(len);
                if (weighted) {  // CBS.cpp:1091-1097 (prune_segments itself is unweighted in the reference, :1089)
                    const double* wu = hw.data() + (*unit_off)[u];
                    double sw = 0.0, swx = 0.0;
                    for (int i = pos; i < pos + len; ++i) { sw += wu[i]; swx += wu[i] * xu[i]; }
                    nmean.push_back(swx / sw);
                } else {
                    double acc = 0.0;
                    for (int i = pos; i < pos + len; ++i) acc += xu[i];
                    nmean.push_back(acc / (double)len);
                }
                pos += len;
            }
            noff[u + 1] = (int64_t)nlen.size();
        }
        R->seg_offsets.swap(noff); R->lengths.swap(nlen); R->means.swap(nmean);
    }
    R->splits.resize(sp.size());
    for (size_t k = 0; k < sp.size(); ++k) {
        cbs_gpu_split& o = R->splits[k];
        const SplitRec& s = sp[k];
        o.unit = s.unit; o.lo = s.lo; o.hi = s.hi; o.ostat = s.ostat; o.iseg0 = s.iseg0; o.iseg1 = s.iseg1;
        o.ncpt = s.ncpt; o.icpt0 = s.icpt0; o.icpt1 = s.icpt1; o.perms_run = s.perms_run; o.nrej = s.nrej;
        o.exit_code = s.exit_code; o.called = s.called; o.e_nrej0 = s.e_nrej0; o.e_nrej1 = s.e_nrej1;
        o.e_status0 = s.e_status0; o.e_status1 = s.e_status1;
    }
    R->pub.n_units = n_units;
    R->pub.n_segments = (int64_t)R->lengths.size();
    R->pub.seg_offsets = R->seg_offsets.data();
    R->pub.lengths = R->lengths.data();
    R->pub.means = R->means.data();
    R->pub.draws_consumed = R->draws.data();
    R->pub.n_splits = (int64_t)R->splits.size();
    R->pub.splits = R->splits.empty() ? nullptr : R->splits.data();
    R->pub.rounds = hD.round;
    R->pub.perms_run = hD.stat_perms;
    R->pub.perm_elements = hD.stat_perm_elems;
    return CBS_GPU_OK;
}

// stage `values` into c->x as double on the device
int stage_values(cbs_gpu_ctx* c, const void* values, int dtype, int memspace, long long N, double* dst) {
    cudaStream_t st = c->stream;
    if (N == 0) return CBS_GPU_OK;
    if (dtype == CBS_GPU_F64) {
        const cudaMemcpyKind kind = memspace == CBS_GPU_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        CUDA_TRY(c, cudaMemcpyAsync(dst, values, sizeof(double) * (size_t)N, kind, st));
    } else {
        const float* src = (const float*)values;
        if (memspace != CBS_GPU_DEVICE) {
            ENSURE(c, c->staging, sizeof(float) * (size_t)N);
            CUDA_TRY(c, cudaMemcpyAsync(c->staging.p, values, sizeof(float) * (size_t)N, cudaMemcpyHostToDevice, st));
            src = c->staging.as<float>();
        }
        k_widen_f32<<<std::min<long long>((N + 255) / 256, c->sm_count * 16), 256, 0, st>>>(src, dst, N);
        c->launches++;
    }
    return CBS_GPU_OK;
}

}  // namespace

// =========================================================================================
// C ABI
// =========================================================================================
extern "C" {

void cbs_gpu_default_params(cbs_gpu_params* p) {
    memset(p, 0, sizeof(*p));
    p->alpha = 0.01; p->nperm = 200; p->hybrid = 0; p->min_width = 2; p->kmax = 25; p->nmin = 200; p->eta = 0.05;
    p->tol = 1e-6; p->ibin = 0; p->undo_prune = 0; p->undo_prune_cutoff = 0.05;
    p->do_smooth = 1; p->smooth_region = 10; p->outlier_sd_scale = 4.0; p->smooth_sd_scale = 2.0; p->trim = 0.025;
    p->rng_mode = CBS_GPU_RNG_MT19937_64; p->chain = 1; p->seed = 1;
}

int cbs_gpu_create(const int* device_ids, int ndev, cbs_gpu_ctx** out) {
    if (!out) return CBS_GPU_ERR_INVALID;
    *out = nullptr;
    if (ndev != 1 || !device_ids) return CBS_GPU_ERR_INVALID;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return CBS_GPU_ERR_CUDA;  // no CPU fallback
    if (device_ids[0] < 0 || device_ids[0] >= count) return CBS_GPU_ERR_INVALID;
    cbs_gpu_ctx* c = new cbs_gpu_ctx();
    c->device = device_ids[0];
    if (cudaSetDevice(c->device) != cudaSuccess) { delete c; return CBS_GPU_ERR_CUDA; }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, c->device) != cudaSuccess) { delete c; return CBS_GPU_ERR_CUDA; }
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = prop.sharedMemPerBlockOptin - 1024;  // head room for the kernels' static shared memory
    // function attributes are process-wide per device: set them once to the device maximum, never per call
    // (concurrent lanes with different needs would otherwise shrink each other's limit)
    const int mx = (int)c->smem_optin;
    if (!set_max_smem(k_scan_perm<false>, mx) || !set_max_smem(k_scan_perm<true>, mx) || !set_max_smem(k_scan_obs<false>, mx) ||
        !set_max_smem(k_scan_obs<true>, mx) ||
        !set_max_smem(k_shuffle<128, 2, true>, mx) || !set_max_smem(k_shuffle<256, 2, true>, mx) || !set_max_smem(k_shuffle<512, 2, true>, mx) ||
        !set_max_smem(k_shuffle<1024, 2, true>, mx) || !set_max_smem(k_shuffle<128, 2, false>, mx) || !set_max_smem(k_shuffle<256, 2, false>, mx) ||
        !set_max_smem(k_shuffle<512, 2, false>, mx) || !set_max_smem(k_shuffle<1024, 2, false>, mx) ||
        !set_max_smem(k_shuffle_cluster<1024, 4, 2, true>, mx) || !set_max_smem(k_shuffle_cluster<1024, 4, 4, true>, mx) ||
        !set_max_smem(k_shuffle_cluster<1024, 4, 8, true>, mx) || !set_max_smem(k_shuffle_cluster<1024, 4, 2, false>, mx) ||
        !set_max_smem(k_shuffle_cluster<1024, 4, 4, false>, mx) || !set_max_smem(k_shuffle_cluster<1024, 4, 8, false>, mx)) {
        delete c;
        return CBS_GPU_ERR_CUDA;
    }
    if (cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking) != cudaSuccess) { delete c; return CBS_GPU_ERR_CUDA; }
    c->stream = c->own_stream;
    if (cudaHostAlloc((void**)&c->h_done, sizeof(int), cudaHostAllocMapped) != cudaSuccess) { delete c; return CBS_GPU_ERR_CUDA; }
    *c->h_done = 0;
    if (cudaHostGetDevicePointer((void**)&c->d_done, c->h_done, 0) != cudaSuccess) { delete c; return CBS_GPU_ERR_CUDA; }
    cudaEventCreate(&c->e0); cudaEventCreate(&c->e1); cudaEventCreate(&c->e2); cudaEventCreate(&c->e3); cudaEventCreate(&c->e4);
    cudaEventCreateWithFlags(&c->grp[0], cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->grp[1], cudaEventDisableTiming);
    for (int k = 0; k < 5; ++k) {
        cudaStreamCreateWithFlags(&c->side[k], cudaStreamNonBlocking);
        cudaEventCreateWithFlags(&c->ev_side[k], cudaEventDisableTiming);
    }
    cudaEventCreateWithFlags(&c->ev_sched, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_gen, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&c->ev_ahead, cudaEventDisableTiming);
    cudaStreamCreateWithFlags(&c->gen_stream, cudaStreamNonBlocking);
    *out = c;
    return CBS_GPU_OK;
}

void cbs_gpu_destroy(cbs_gpu_ctx* c) {
    if (!c) return;
    for (auto* l : c->lanes) cbs_gpu_destroy(l);
    c->lanes.clear();
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    DevBuf* bufs[] = {&c->x, &c->cur, &c->gtab, &c->factab, &c->bbtab, &c->unit_off, &c->unit_ids, &c->tasks, &c->ring, &c->act0,
                      &c->act1, &c->chains, &c->segs, &c->splits, &c->udraws, &c->arena, &c->rej, &c->draws0, &c->draws1,
                      &c->prep_task, &c->items, &c->item_prefix, &c->edgeprep_task, &c->edges, &c->edge_prefix, &c->gen_chain,
                      &c->means, &c->seed312, &c->dev, &c->staging, &c->fv, &c->fidx, &c->flab, &c->lab, &c->diffs,
                      &c->diffs_sorted, &c->sm_keys, &c->sm_gid, &c->cn_scratch, &c->gout, &c->cubtmp, &c->flag, &c->goff, &c->stream_buf, &c->shuf, &c->jump, &c->tailp,
                      &c->wts, &c->rw, &c->cw, &c->ycur};
    for (DevBuf* b : bufs) if (b->p) cudaFree(b->p);
    if (c->call_exec) cudaGraphExecDestroy(c->call_exec);
    if (c->h_done) cudaFreeHost(c->h_done);
    for (auto e : c->ev_pool) cudaEventDestroy(e);
    cudaEvent_t evs[] = {c->e0, c->e1, c->e2, c->e3, c->e4, c->grp[0], c->grp[1]};
    for (auto e : evs) if (e) cudaEventDestroy(e);
    for (int k = 0; k < 5; ++k) { if (c->side[k]) cudaStreamDestroy(c->side[k]); if (c->ev_side[k]) cudaEventDestroy(c->ev_side[k]); }
    if (c->ev_sched) cudaEventDestroy(c->ev_sched);
    if (c->ev_gen) cudaEventDestroy(c->ev_gen);
    if (c->ev_ahead) cudaEventDestroy(c->ev_ahead);
    if (c->gen_stream) cudaStreamDestroy(c->gen_stream);
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
}

const char* cbs_gpu_last_error(const cbs_gpu_ctx* c) { return c ? c->err.c_str() : "no context"; }

int cbs_gpu_set_stream(cbs_gpu_ctx* c, void* s) {
    if (!c) return CBS_GPU_ERR_INVALID;
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return CBS_GPU_OK;
}

int cbs_gpu_set_profiling(cbs_gpu_ctx* c, int on) {
    if (!c) return CBS_GPU_ERR_INVALID;
    c->profiling = (on & 1) != 0;
    c->counting = (on & 2) != 0;
    c->serial = (on & 4) != 0;
    return CBS_GPU_OK;
}

int cbs_gpu_last_kernel_ms(cbs_gpu_ctx* c, double* ms14) {
    if (!c || !ms14) return CBS_GPU_ERR_INVALID;
    for (int k = 0; k < 14; ++k) ms14[k] = c->kms[k];
    return CBS_GPU_OK;
}

int cbs_gpu_last_arc_evals(cbs_gpu_ctx* c, uint64_t* arcs, uint64_t* slots) {
    if (!c || !arcs || !slots) return CBS_GPU_ERR_INVALID;
    *arcs = c->last_arcs;
    *slots = c->last_slots;
    return CBS_GPU_OK;
}

int cbs_gpu_selftest(void) {
    // host-only checks (no device needed): the MT19937-64 jump-ahead table against sequential generation
    return mtjump::table().ok ? 0 : 1;
}

int cbs_gpu_measure_fp64(cbs_gpu_ctx* c, double* tera_inst_per_s) {
    if (!c || !tera_inst_per_s) return CBS_GPU_ERR_INVALID;
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    const int grid = c->sm_count * 8, block = 256, iters = 4096;
    ENSURE(c, c->staging, sizeof(double) * (size_t)grid * block);
    cudaStream_t st = c->stream;
    double best = 0.0;
    for (int rep = 0; rep < 5; ++rep) {
        CUDA_TRY(c, cudaEventRecord(c->e0, st));
        k_fp64_peak<<<grid, block, 0, st>>>(c->staging.as<double>(), iters, 1e-9);
        CUDA_TRY(c, cudaEventRecord(c->e1, st));
        CUDA_TRY(c, cudaEventSynchronize(c->e1));
        float ms = 0.f;
        cudaEventElapsedTime(&ms, c->e0, c->e1);
        // per thread: iters * 4 * 8 DADD
        const double inst = (double)grid * block * (double)iters * 32.0;
        if (rep > 0 && ms > 0.f) best = std::max(best, inst / (ms * 1e-3) / 1e12);
    }
    *tera_inst_per_s = best;
    return CBS_GPU_OK;
}

// ---- low level: cbs::tmaxo / cbs::tmaxp on vectors as given ------------------------------------
static int run_raw_scan(cbs_gpu_ctx* c, const double* xh, int n, int count, double tss, int al0, int ibin, int obs,
                        std::vector<Task>& tasks_out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (ibin) return fail(c, CBS_GPU_ERR_CUDA, "internal: binary data takes run_bin_scan");
    if (n < 2 || count < 1 || !xh) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (al0 < 1 || n < 2 * al0) return fail(c, CBS_GPU_ERR_INVALID, "need n >= 2*al0, al0 >= 1");
    if (n > 1000000) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "vectors longer than 1,000,000 are not supported");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    const long long N = (long long)n * count;
    const int nb = block_count(n);
    const long long per = Sched::sx_stride(n) + Sched::bs_stride(nb);
    ENSURE(c, c->x, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->cur, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->gtab, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->factab, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->bbtab, sizeof(int) * (size_t)(N + 1));
    ENSURE(c, c->unit_off, sizeof(long long) * (size_t)(count + 1));
    ENSURE(c, c->tasks, sizeof(Task) * (size_t)count);
    ENSURE(c, c->arena, sizeof(double) * (size_t)(per * count));
    ENSURE(c, c->rej, sizeof(int) * (size_t)count);
    ENSURE(c, c->prep_task, sizeof(int) * (size_t)count);
    ENSURE(c, c->items, sizeof(PermItem) * (size_t)count);
    ENSURE(c, c->item_prefix, sizeof(int) * (size_t)(count + 1));
    ENSURE(c, c->dev, sizeof(Dev));
    std::vector<long long> off((size_t)count + 1);
    std::vector<Task> tasks((size_t)count);
    std::vector<int> prep((size_t)count), prefix((size_t)count + 1);
    std::vector<PermItem> items((size_t)count);
    memset(tasks.data(), 0, sizeof(Task) * tasks.size());
    for (int u = 0; u <= count; ++u) off[u] = (long long)u * n;
    for (int u = 0; u < count; ++u) {
        Task& t = tasks[u];
        t.unit = u; t.lo = 0; t.hi = n; t.n = n; t.nb = nb; t.raw = 1; t.tss = tss; t.state = TS_OBS;
        t.off_sx = per * u; t.off_bs = per * u + Sched::sx_stride(n); t.off_rej = u; t.next = -1;
        prep[u] = u; prefix[u] = u;
        items[u].task = u; items[u].P = 1; items[u].obs = obs;
    }
    prefix[count] = count;
    Dev hD;
    memset(&hD, 0, sizeof(hD));
    hD.x = c->x.as<double>(); hD.unit_off = c->unit_off.as<long long>(); hD.n_units = count;
    hD.prm.min_width = al0; hD.prm.nperm = 0; hD.prm.rng_mode = RNG_PHILOX;
    hD.cur = c->cur.as<double>(); hD.gtab = c->gtab.as<double>(); hD.factab = c->factab.as<double>(); hD.bbtab = c->bbtab.as<int>();
    hD.tasks = c->tasks.as<Task>(); hD.task_cap = count;
    hD.arena = c->arena.as<double>(); hD.arena_cap = per * count; hD.rej = c->rej.as<int>(); hD.rej_cap = count;
    hD.n_prep = count; hD.prep_task = c->prep_task.as<int>();
    hD.n_items = count; hD.items = c->items.as<PermItem>(); hD.item_prefix = c->item_prefix.as<int>();
    hD.obs_slices = obs_slice_cap(); hD.obs_noloc = obs == 2 ? 1 : 0;
    hD.ctr[CTR_OBS_SLICES] = (unsigned)obs_slices(n, hD.obs_slices);
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, xh, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->unit_off.p, off.data(), sizeof(long long) * off.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->tasks.p, tasks.data(), sizeof(Task) * tasks.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->prep_task.p, prep.data(), sizeof(int) * prep.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->items.p, items.data(), sizeof(PermItem) * items.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->item_prefix.p, prefix.data(), sizeof(int) * prefix.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->dev.p, &hD, sizeof(Dev), cudaMemcpyHostToDevice, st));
    ScanLayout lay;
    lay.nb_max = nb + 2;
    lay.set_table(n);
    int occ = 1;
    if (!pick_scan_warps(c, lay, &occ, (const void*)k_scan_obs<false>)) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "vector too long for the scan kernel's shared memory");
    Dev* dD = c->dev.as<Dev>();
    k_tables<<<dim3(16, 64), 256, 0, st>>>(dD);
    k_prep<<<std::min(count, c->sm_count * 8), 32, 0, st>>>(dD);
    launch_scan(true, false, (int)std::min<long long>((long long)count * hD.ctr[CTR_OBS_SLICES], (long long)c->sm_count * occ), lay, st, dD);
    CUDA_TRY(c, cudaGetLastError());
    tasks_out.resize((size_t)count);
    CUDA_TRY(c, cudaMemcpyAsync(tasks_out.data(), c->tasks.p, sizeof(Task) * tasks_out.size(), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return CBS_GPU_OK;
}

// binary data (ibin = true): cbs::tmaxo_impl walked in the reference's own order, one warp per vector (binary.cuh)
static int run_bin_scan(cbs_gpu_ctx* c, const double* xh, int n, int count, double tss, int al0, std::vector<double>& stat,
                        std::vector<int>& left, std::vector<int>& right) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n < 2 || count < 1 || !xh) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (al0 < 1 || n < 2 * al0) return fail(c, CBS_GPU_ERR_INVALID, "need n >= 2*al0, al0 >= 1");
    if (n > 1000000) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "vectors longer than 1,000,000 are not supported");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    const long long N = (long long)n * count, per = bin_scratch_doubles(n);
    ENSURE(c, c->x, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->arena, sizeof(double) * (size_t)(per * count));
    ENSURE(c, c->means, sizeof(double) * (size_t)count);
    ENSURE(c, c->staging, sizeof(int) * 2 * (size_t)count);
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, xh, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, st));
    k_scan_bin<<<std::min(count, c->sm_count * 16), 32, 0, st>>>(c->x.as<double>(), n, count, tss, al0, 1, c->arena.as<double>(),
                                                               c->means.as<double>(), c->staging.as<int>(), c->staging.as<int>() + count);
    CUDA_TRY(c, cudaGetLastError());
    stat.resize((size_t)count); left.resize((size_t)count); right.resize((size_t)count);
    CUDA_TRY(c, cudaMemcpyAsync(stat.data(), c->means.p, sizeof(double) * (size_t)count, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(left.data(), c->staging.p, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(right.data(), c->staging.as<int>() + count, sizeof(int) * (size_t)count, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return CBS_GPU_OK;
}

int cbs_gpu_tmaxo(cbs_gpu_ctx* c, const double* x, int32_t n, double tss, int32_t al0, int32_t ibin, double* statistic,
                  int32_t* start, int32_t* end) {
    if (ibin) {
        std::vector<double> st; std::vector<int> l, r;
        const int rc = run_bin_scan(c, x, n, 1, tss, al0, st, l, r);
        if (rc) return rc;
        if (statistic) *statistic = st[0];
        if (start) *start = l[0] - 1;  // CBS.cpp:380
        if (end) *end = r[0] - 1;
        return CBS_GPU_OK;
    }
    std::vector<Task> t;
    const int rc = run_raw_scan(c, x, n, 1, tss, al0, ibin, 1, t);
    if (rc) return rc;
    if (statistic) *statistic = t[0].ostat;
    if (start) *start = t[0].tmaxi - 1;  // CBS.cpp:380
    if (end) *end = t[0].tmaxj - 1;
    return CBS_GPU_OK;
}

int cbs_gpu_tmaxp(cbs_gpu_ctx* c, const double* px, int32_t n, int32_t count, double tss, int32_t al0, int32_t ibin,
                  double* statistics) {
    if (ibin) {
        std::vector<double> st; std::vector<int> l, r;
        const int rc = run_bin_scan(c, px, n, count, tss, al0, st, l, r);
        if (rc) return rc;
        for (int k = 0; k < count; ++k) statistics[k] = st[k];
        return CBS_GPU_OK;
    }
    std::vector<Task> t;
    const int rc = run_raw_scan(c, px, n, count, tss, al0, ibin, 2, t);
    if (rc) return rc;
    for (int k = 0; k < count; ++k) statistics[k] = t[k].ostat;
    return CBS_GPU_OK;
}

static int segment_batch_impl(cbs_gpu_ctx* c, const void* values, int dtype, int memspace, const int64_t* unit_offsets,
                              const uint64_t* unit_ids, int32_t n_units, const cbs_gpu_params* params, cbs_gpu_result** out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!out) return fail(c, CBS_GPU_ERR_INVALID, "out is NULL");
    *out = nullptr;
    const auto wall0 = std::chrono::steady_clock::now();
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    int rc = validate_params(c, params);
    if (rc) return rc;
    if (n_units < 0 || !unit_offsets) return fail(c, CBS_GPU_ERR_INVALID, "bad unit table");
    if (dtype != CBS_GPU_F32 && dtype != CBS_GPU_F64) return fail(c, CBS_GPU_ERR_INVALID, "bad dtype");
    std::vector<long long> off((size_t)n_units + 1);
    for (int u = 0; u <= n_units; ++u) {
        off[u] = unit_offsets[u];
        if (u && off[u] < off[u - 1]) return fail(c, CBS_GPU_ERR_INVALID, "unit_offsets must be non-decreasing");
    }
    if (off[0] != 0) return fail(c, CBS_GPU_ERR_INVALID, "unit_offsets[0] must be 0");
    const long long N = off[n_units];
    if (N > 0 && !values) return fail(c, CBS_GPU_ERR_INVALID, "values is NULL");
    for (int k = 0; k < K_COUNT; ++k) c->kms[k] = 0.0;
    c->launches = 0;
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->flag, sizeof(int));
    CUDA_TRY(c, cudaEventRecord(c->e0, st));
    double* xdst = c->x.as<double>();
    if (params->do_smooth) {
        ENSURE(c, c->diffs_sorted, sizeof(double) * (size_t)(N + 1));  // reused below as the raw copy
        ENSURE(c, c->lab, sizeof(double) * (size_t)(N + 1));
        xdst = c->lab.as<double>();  // raw widened values; smoothing writes c->x
    }
    rc = stage_values(c, values, dtype, memspace, N, xdst);
    if (rc) return rc;
    CUDA_TRY(c, cudaEventRecord(c->e1, st));
    if (params->do_smooth) {
        ENSURE(c, c->goff, sizeof(long long) * (size_t)(n_units + 1));
        CUDA_TRY(c, cudaMemcpyAsync(c->goff.p, off.data(), sizeof(long long) * (size_t)(n_units + 1), cudaMemcpyHostToDevice, st));
        rc = smooth_device(c, xdst, c->goff.as<long long>(), nullptr, n_units, N, params->smooth_region, params->outlier_sd_scale,
                           params->smooth_sd_scale, params->trim, c->x.as<double>(), off);
        if (rc) return rc;
    }
    CUDA_TRY(c, cudaEventRecord(c->e2, st));
    // CBS needs finite input (the reference has no defined behaviour otherwise)
    CUDA_TRY(c, cudaMemsetAsync(c->flag.p, 0, sizeof(int), st));
    if (N) { k_count_nonfinite<<<std::min<long long>((N + 255) / 256, c->sm_count * 8), 256, 0, st>>>(c->x.as<double>(), N, c->flag.as<int>()); c->launches++; }
    int bad = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&bad, c->flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    if (bad) return fail(c, CBS_GPU_ERR_NONFINITE, "non-finite values reach CBS; remove them first (DNAcopy drops missing values before segmenting)");
    Dev hD;
    rc = run_cbs(c, off, unit_ids, n_units, params, nullptr, false, hD);
    if (rc) return rc;
    CUDA_TRY(c, cudaEventRecord(c->e3, st));
    ResultOwner* R = new ResultOwner();
    memset(&R->pub, 0, sizeof(R->pub));
    rc = fetch_results(c, hD, n_units, params->record_splits != 0, R, params, &off);
    if (rc) { delete R; return rc; }
    CUDA_TRY(c, cudaEventRecord(c->e4, st));
    CUDA_TRY(c, cudaEventSynchronize(c->e4));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->e0, c->e1); R->pub.ms_h2d = ms;
    cudaEventElapsedTime(&ms, c->e1, c->e2); R->pub.ms_smooth = ms;
    cudaEventElapsedTime(&ms, c->e2, c->e3); R->pub.ms_segment = ms;
    cudaEventElapsedTime(&ms, c->e3, c->e4); R->pub.ms_d2h = ms;
    R->pub.ms_call = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - wall0).count();
    if (c->profiling) collect_timers(c);
    R->pub.kernel_launches = c->launches;
    c->last_arcs = hD.stat_arcs;
    c->last_slots = hD.stat_slots;
    *out = &R->pub;
    return CBS_GPU_OK;
}

int cbs_gpu_segment_batch(cbs_gpu_ctx* c, const void* values, int dtype, int memspace, const int64_t* unit_offsets,
                          const uint64_t* unit_ids, int32_t n_units, const cbs_gpu_params* params, cbs_gpu_result** out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!out) return fail(c, CBS_GPU_ERR_INVALID, "out is NULL");
    *out = nullptr;
    int want_lanes = (int)env_ll("CBS_GPU_LANES", 1);  // opt-in: measured no gain on B200 (persistent grids fill the SMs)
    const bool serial_stream = params && params->rng_mode == CBS_GPU_RNG_MT19937_64 && params->chain;
    bool splittable = !c->is_lane && params && unit_offsets && n_units >= 2 && !serial_stream && (dtype == CBS_GPU_F32 || dtype == CBS_GPU_F64);
    if (splittable) {  // (malformed unit tables go to segment_batch_impl as they are: it reports them)
        if (unit_offsets[0] != 0) splittable = false;
        for (int u = 0; splittable && u < n_units; ++u) if (unit_offsets[u + 1] < unit_offsets[u]) splittable = false;
    }
    // Large cohorts are segmented in consecutive sub-batches of about CBS_GPU_CHUNK_MARKERS markers (default 96 M, some 50
    // SNP6 samples) so that a call of any size runs in bounded device memory (~100 B per marker of per-call buffers besides
    // the arenas).  Units are independent (Philox keys and chain == 0 streams do not depend on the neighbours), and the cost
    // per sample does not depend on the batch size beyond a few samples per call (125 samples: 6.77 s in one batch, 6.81 s in
    // five), so the split costs nothing.
    const long long chunk_max = std::max<long long>(1024, env_ll("CBS_GPU_CHUNK_MARKERS", 96LL << 20));
    const long long N_all = splittable ? (long long)unit_offsets[n_units] : 0;
    const bool parallel = splittable && want_lanes >= 2 && n_units >= 2 * want_lanes;
    if (!parallel && (!splittable || N_all <= chunk_max))
        return segment_batch_impl(c, values, dtype, memspace, unit_offsets, unit_ids, n_units, params, out);
    if (want_lanes > 4) want_lanes = 4;
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    int L = want_lanes;
    std::vector<int> cut;
    if (parallel) {
        while ((int)c->lanes.size() < L) {
            cbs_gpu_ctx* child = nullptr;
            const int ids[1] = {c->device};
            if (cbs_gpu_create(ids, 1, &child) != CBS_GPU_OK) return fail(c, CBS_GPU_ERR_CUDA, "cannot create lane context");
            child->is_lane = true;
            c->lanes.push_back(child);
        }
        // contiguous ranges balanced by sum n^1.5 (the cost of the permutation scans)
        std::vector<double> cost((size_t)n_units + 1, 0.0);
        for (int u = 0; u < n_units; ++u) {
            const double n = (double)(unit_offsets[u + 1] - unit_offsets[u]);
            cost[u + 1] = cost[u] + (n > 0 ? n * std::sqrt(n) : 0.0);
        }
        cut.assign((size_t)L + 1, 0);
        cut[L] = n_units;
        for (int l = 1; l < L; ++l) {
            const double target = cost[n_units] * l / L;
            int u = cut[l - 1];
            while (u < n_units && cost[u + 1] <= target) ++u;
            cut[l] = std::max(u, cut[l - 1]);
        }
    } else {
        // sub-batches of equal marker counts, cut at unit boundaries
        const int want = (int)std::min<long long>((N_all + chunk_max - 1) / chunk_max, n_units);
        cut.push_back(0);
        for (int k = 1; k < want; ++k) {
            const long long target = N_all * k / want;
            int u = cut.back();
            while (u < n_units && (long long)unit_offsets[u + 1] <= target) ++u;
            if (u > cut.back() && u < n_units) cut.push_back(u);
        }
        cut.push_back(n_units);
        L = (int)cut.size() - 1;
    }
    // the input must be complete before other streams read it
    if (memspace == CBS_GPU_DEVICE) cudaStreamSynchronize(c->stream);
    std::vector<uint64_t> ids_all((size_t)n_units);
    for (int u = 0; u < n_units; ++u) ids_all[u] = unit_ids ? unit_ids[u] : (uint64_t)u;  // keys must not depend on the split
    std::vector<int> rcs((size_t)L, CBS_GPU_OK);
    std::vector<cbs_gpu_result*> parts((size_t)L, nullptr);
    std::vector<std::vector<int64_t>> offs((size_t)L);
    std::vector<std::thread> th;
    const size_t esz = dtype == CBS_GPU_F32 ? 4 : 8;
    std::vector<std::vector<double>> part_kms((size_t)L, std::vector<double>((size_t)K_COUNT, 0.0));
    std::vector<unsigned long long> part_arcs((size_t)L, 0), part_slots((size_t)L, 0);
    for (int l = 0; l < L; ++l) {
        const int u0 = cut[l], u1 = cut[l + 1];
        offs[l].resize((size_t)(u1 - u0) + 1);
        for (int u = u0; u <= u1; ++u) offs[l][u - u0] = unit_offsets[u] - unit_offsets[u0];
        const char* base = (const char*)values + (size_t)unit_offsets[u0] * esz;
        if (parallel) {
            cbs_gpu_ctx* child = c->lanes[l];
            child->profiling = c->profiling; child->counting = c->counting; child->serial = c->serial;
            child->mem_fraction = 0.80 / L;
            th.emplace_back([=, &rcs, &parts, &offs, &ids_all]() {
                rcs[l] = segment_batch_impl(child, base, dtype, memspace, offs[l].data(), ids_all.data() + u0, u1 - u0, params, &parts[l]);
            });
        } else {
            rcs[l] = segment_batch_impl(c, base, dtype, memspace, offs[l].data(), ids_all.data() + u0, u1 - u0, params, &parts[l]);
            if (rcs[l] != CBS_GPU_OK) {
                for (auto* p : parts) if (p) cbs_gpu_result_free(p);
                return rcs[l];  // the message is already in c
            }
            for (int k = 0; k < K_COUNT; ++k) part_kms[l][k] = c->kms[k];
            part_arcs[l] = c->last_arcs; part_slots[l] = c->last_slots;
        }
    }
    for (auto& t : th) t.join();
    if (parallel)
        for (int l = 0; l < L; ++l) {
            if (rcs[l] != CBS_GPU_OK) {
                const std::string msg = cbs_gpu_last_error(c->lanes[l]);
                for (auto* p : parts) if (p) cbs_gpu_result_free(p);
                return fail(c, rcs[l], msg);
            }
            for (int k = 0; k < K_COUNT; ++k) part_kms[l][k] = c->lanes[l]->kms[k];
            part_arcs[l] = c->lanes[l]->last_arcs; part_slots[l] = c->lanes[l]->last_slots;
        }
    ResultOwner* R = new ResultOwner();
    memset(&R->pub, 0, sizeof(R->pub));
    R->seg_offsets.assign((size_t)n_units + 1, 0);
    R->draws.assign((size_t)n_units, 0);
    for (int k = 0; k < K_COUNT; ++k) c->kms[k] = 0.0;
    c->last_arcs = 0; c->last_slots = 0;
    for (int l = 0; l < L; ++l) {
        const cbs_gpu_result* p = parts[l];
        const int u0 = cut[l];
        const int64_t shift = (int64_t)R->lengths.size();
        for (int u = 0; u < p->n_units; ++u) {
            R->seg_offsets[(size_t)u0 + u + 1] = shift + p->seg_offsets[u + 1];
            R->draws[(size_t)u0 + u] = p->draws_consumed[u];
        }
        R->lengths.insert(R->lengths.end(), p->lengths, p->lengths + p->n_segments);
        R->means.insert(R->means.end(), p->means, p->means + p->n_segments);
        for (int64_t k = 0; k < p->n_splits; ++k) { cbs_gpu_split sp = p->splits[k]; sp.unit += u0; R->splits.push_back(sp); }
        R->pub.perms_run += p->perms_run; R->pub.perm_elements += p->perm_elements; R->pub.kernel_launches += p->kernel_launches;
        if (parallel) {  // lanes run side by side, sub-batches one after the other
            R->pub.rounds = std::max(R->pub.rounds, p->rounds);
            R->pub.ms_h2d = std::max(R->pub.ms_h2d, p->ms_h2d); R->pub.ms_smooth = std::max(R->pub.ms_smooth, p->ms_smooth);
            R->pub.ms_segment = std::max(R->pub.ms_segment, p->ms_segment); R->pub.ms_d2h = std::max(R->pub.ms_d2h, p->ms_d2h);
            R->pub.ms_call = std::max(R->pub.ms_call, p->ms_call);
        } else {
            R->pub.rounds += p->rounds;
            R->pub.ms_h2d += p->ms_h2d; R->pub.ms_smooth += p->ms_smooth; R->pub.ms_segment += p->ms_segment; R->pub.ms_d2h += p->ms_d2h;
            R->pub.ms_call += p->ms_call;
        }
        for (int k = 0; k < K_COUNT; ++k) c->kms[k] += part_kms[l][k];
        c->last_arcs += part_arcs[l]; c->last_slots += part_slots[l];
    }
    // empty leading/trailing units keep monotone offsets
    for (int u = 0; u < n_units; ++u) if (R->seg_offsets[u + 1] < R->seg_offsets[u]) R->seg_offsets[u + 1] = R->seg_offsets[u];
    for (auto* p : parts) cbs_gpu_result_free(p);
    R->pub.n_units = n_units;
    R->pub.n_segments = (int64_t)R->lengths.size();
    R->pub.seg_offsets = R->seg_offsets.data();
    R->pub.lengths = R->lengths.data();
    R->pub.means = R->means.data();
    R->pub.draws_consumed = R->draws.data();
    R->pub.n_splits = (int64_t)R->splits.size();
    R->pub.splits = R->splits.empty() ? nullptr : R->splits.data();
    *out = &R->pub;
    return CBS_GPU_OK;
}

// cbs::segment_weighted (CBS.cpp:1026-1099) for every unit; values and weights: float64, laid out alike
int cbs_gpu_segment_weighted_batch(cbs_gpu_ctx* c, const double* values, const double* weights, int memspace,
                                   const int64_t* unit_offsets, const uint64_t* unit_ids, int32_t n_units,
                                   const cbs_gpu_params* params, cbs_gpu_result** out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!out) return fail(c, CBS_GPU_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!params || !unit_offsets || n_units < 0) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cbs_gpu_params p = *params;
    p.do_smooth = 0;  // cbs::segment_weighted does not smooth
    int rc = validate_params(c, &p);
    if (rc) return rc;
    std::vector<long long> off((size_t)n_units + 1);
    for (int u = 0; u <= n_units; ++u) off[u] = unit_offsets[u];
    if (off[0] != 0) return fail(c, CBS_GPU_ERR_INVALID, "unit_offsets[0] must be 0");
    for (int u = 0; u < n_units; ++u) if (off[u + 1] < off[u]) return fail(c, CBS_GPU_ERR_INVALID, "unit_offsets must be non-decreasing");
    const long long N = off[n_units];
    if (N > 0 && (!values || !weights)) return fail(c, CBS_GPU_ERR_INVALID, "values / weights is NULL");
    for (int k = 0; k < K_COUNT; ++k) c->kms[k] = 0.0;
    c->launches = 0;
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->wts, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->flag, sizeof(int));
    CUDA_TRY(c, cudaEventRecord(c->e0, st));
    const cudaMemcpyKind kind = memspace == CBS_GPU_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    if (N) {
        CUDA_TRY(c, cudaMemcpyAsync(c->x.p, values, sizeof(double) * (size_t)N, kind, st));
        CUDA_TRY(c, cudaMemcpyAsync(c->wts.p, weights, sizeof(double) * (size_t)N, kind, st));
    }
    CUDA_TRY(c, cudaEventRecord(c->e1, st));
    CUDA_TRY(c, cudaMemsetAsync(c->flag.p, 0, sizeof(int), st));
    if (N) { k_count_nonfinite<<<std::min<long long>((N + 255) / 256, c->sm_count * 8), 256, 0, st>>>(c->x.as<double>(), N, c->flag.as<int>()); c->launches++; }
    int bad = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&bad, c->flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    if (bad) return fail(c, CBS_GPU_ERR_NONFINITE, "non-finite values reach CBS");
    CUDA_TRY(c, cudaEventRecord(c->e2, st));
    Dev hD;
    rc = run_cbs(c, off, unit_ids, n_units, &p, nullptr, true, hD);
    if (rc) return rc;
    CUDA_TRY(c, cudaEventRecord(c->e3, st));
    ResultOwner* R = new ResultOwner();
    memset(&R->pub, 0, sizeof(R->pub));
    rc = fetch_results(c, hD, n_units, p.record_splits != 0, R, &p, &off, true);
    if (rc) { delete R; return rc; }
    CUDA_TRY(c, cudaEventRecord(c->e4, st));
    CUDA_TRY(c, cudaEventSynchronize(c->e4));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, c->e0, c->e1); R->pub.ms_h2d = ms;
    cudaEventElapsedTime(&ms, c->e2, c->e3); R->pub.ms_segment = ms;
    cudaEventElapsedTime(&ms, c->e3, c->e4); R->pub.ms_d2h = ms;
    if (c->profiling) collect_timers(c);
    R->pub.kernel_launches = c->launches;
    *out = &R->pub;
    return CBS_GPU_OK;
}

// cbs::segment_weighted on one vector (CBS.hpp:115-128)
int cbs_gpu_segment_weighted(cbs_gpu_ctx* c, const double* x, const double* weights, int32_t n, const cbs_gpu_params* params,
                             const uint64_t* mt_next312, int32_t cap, int32_t* lengths, double* means, int32_t* n_segments,
                             uint64_t* draws_consumed) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n < 0 || (n > 0 && (!x || !weights)) || !n_segments || !params) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cbs_gpu_params p = *params;
    p.do_smooth = 0;
    int rc = validate_params(c, &p);
    if (rc) return rc;
    *n_segments = 0;
    if (draws_consumed) *draws_consumed = 0;
    if (n == 0) return CBS_GPU_OK;
    for (int i = 0; i < n; ++i) if (!std::isfinite(x[i])) return fail(c, CBS_GPU_ERR_NONFINITE, "non-finite values reach CBS");
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->wts, sizeof(double) * (size_t)(n + 1));
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->wts.p, weights, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    std::vector<long long> off = {0, (long long)n};
    Dev hD;
    for (int k = 0; k < K_COUNT; ++k) c->kms[k] = 0.0;
    rc = run_cbs(c, off, nullptr, 1, &p, mt_next312, true, hD);
    if (rc) return rc;
    ResultOwner R;
    memset(&R.pub, 0, sizeof(R.pub));
    rc = fetch_results(c, hD, 1, false, &R, &p, &off, true);
    if (rc) return rc;
    if (c->profiling) collect_timers(c);
    *n_segments = (int32_t)R.pub.n_segments;
    if (draws_consumed) *draws_consumed = R.draws[0];
    if (R.pub.n_segments > cap) return fail(c, CBS_GPU_ERR_CAPACITY, "output capacity too small");
    for (int64_t k = 0; k < R.pub.n_segments; ++k) { lengths[k] = R.lengths[k]; means[k] = R.means[k]; }
    return CBS_GPU_OK;
}

// ---- low level: one decision on a vector as given -------------------------------------------------------------
static int decision_impl(cbs_gpu_ctx* c, const double* x, const double* weights, int32_t n, const cbs_gpu_params* params,
                         const ApiMode& api, const uint64_t* mt_next312, cbs_gpu_split* out, uint64_t* draws_consumed) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n < 2 || !x || !params || !out) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cbs_gpu_params p = *params;
    p.do_smooth = 0; p.undo_prune = 0; p.chain = 0; p.record_splits = 1;
    int rc = validate_params(c, &p);
    if (rc) return rc;
    for (int i = 0; i < n; ++i) if (!std::isfinite(x[i])) return fail(c, CBS_GPU_ERR_NONFINITE, "non-finite values reach CBS");
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(n + 1));
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    if (weights) {
        ENSURE(c, c->wts, sizeof(double) * (size_t)(n + 1));
        CUDA_TRY(c, cudaMemcpyAsync(c->wts.p, weights, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    }
    std::vector<long long> off = {0, (long long)n};
    Dev hD;
    for (int k = 0; k < K_COUNT; ++k) c->kms[k] = 0.0;
    rc = run_cbs(c, off, nullptr, 1, &p, mt_next312, weights != nullptr, hD, api);
    if (rc) return rc;
    if (hD.n_splits < 1) return fail(c, CBS_GPU_ERR_CUDA, "internal: the decision was not recorded");
    SplitRec s;
    uint64_t draws = 0;
    CUDA_TRY(c, cudaMemcpyAsync(&s, c->splits.p, sizeof(SplitRec), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaMemcpyAsync(&draws, c->udraws.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    if (c->profiling) collect_timers(c);
    memset(out, 0, sizeof(*out));
    out->unit = 0; out->lo = s.lo; out->hi = s.hi; out->ostat = s.ostat; out->iseg0 = s.iseg0; out->iseg1 = s.iseg1;
    out->ncpt = s.ncpt; out->icpt0 = s.icpt0; out->icpt1 = s.icpt1; out->perms_run = s.perms_run; out->nrej = s.nrej;
    out->exit_code = s.exit_code; out->called = s.called; out->e_nrej0 = s.e_nrej0; out->e_nrej1 = s.e_nrej1;
    out->e_status0 = s.e_status0; out->e_status1 = s.e_status1;
    if (draws_consumed) *draws_consumed = draws;
    return CBS_GPU_OK;
}

int cbs_gpu_fndcpt(cbs_gpu_ctx* c, const double* x, int32_t n, double tss, const cbs_gpu_params* params, double delta,
                   int32_t ngrid, const uint64_t* mt_next312, cbs_gpu_split* out, uint64_t* draws_consumed) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (params && params->hybrid && ngrid != 100) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "hybrid: ngrid must be 100");
    if (params && n < 2 * params->min_width) return fail(c, CBS_GPU_ERR_INVALID, "need n >= 2*al0");
    ApiMode api;
    api.mode = 1; api.tss = tss; api.delta = delta;
    return decision_impl(c, x, nullptr, n, params, api, mt_next312, out, draws_consumed);
}

int cbs_gpu_wfindcpt(cbs_gpu_ctx* c, const double* x, const double* weights, int32_t n, double tss, const cbs_gpu_params* params,
                     int32_t ngrid, const uint64_t* mt_next312, cbs_gpu_split* out, uint64_t* draws_consumed) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!weights) return fail(c, CBS_GPU_ERR_INVALID, "weights is NULL");
    if (params && params->hybrid && ngrid != 100) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "hybrid: ngrid must be 100");
    if (params && n < 2 * params->min_width) return fail(c, CBS_GPU_ERR_INVALID, "need n >= 2*al0");
    ApiMode api;
    api.mode = 1; api.tss = tss;
    return decision_impl(c, x, weights, n, params, api, mt_next312, out, draws_consumed);
}

int cbs_gpu_tpermp(cbs_gpu_ctx* c, const double* x, int32_t n1, int32_t n2, const cbs_gpu_params* params,
                   const uint64_t* mt_next312, double* pvalue, uint64_t* draws_consumed) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n1 < 1 || n2 < 1 || !pvalue || !params) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (params->nperm < 1) return fail(c, CBS_GPU_ERR_INVALID, "nperm must be >= 1");
    ApiMode api;
    api.mode = 2; api.n1 = n1; api.n2 = n2;
    cbs_gpu_split s;
    cbs_gpu_params p = *params;
    p.hybrid = 0; p.min_width = 1;
    const int rc = decision_impl(c, x, nullptr, n1 + n2, &p, api, mt_next312, &s, draws_consumed);
    if (rc) return rc;
    *pvalue = s.e_status0 == 1 ? 1.0 : s.e_status0 == 2 ? 0.0 : (double)s.e_nrej0 / (double)p.nperm;  // CBS.cpp:499,522,535
    return CBS_GPU_OK;
}

int cbs_gpu_wtmaxo(cbs_gpu_ctx* c, const double* x, const double* weights, int32_t n, double tss, int32_t al0,
                   double* statistic, int32_t* start, int32_t* end) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!weights) return fail(c, CBS_GPU_ERR_INVALID, "weights is NULL");
    if (al0 < 1 || n < 2 * al0) return fail(c, CBS_GPU_ERR_INVALID, "need n >= 2*al0, al0 >= 1");
    cbs_gpu_params p;
    cbs_gpu_default_params(&p);
    p.min_width = al0; p.nperm = 0; p.hybrid = 0;
    ApiMode api;
    api.mode = 3; api.tss = tss;
    cbs_gpu_split s;
    const int rc = decision_impl(c, x, weights, n, &p, api, nullptr, &s, nullptr);
    if (rc) return rc;
    if (statistic) *statistic = s.ostat;
    if (start) *start = s.iseg0;
    if (end) *end = s.iseg1;
    return CBS_GPU_OK;
}

// cbs::xperm / cbs::wxperm: ONE permutation with the engine state given as its next 312 raw words.  The raw words the
// permutation consumes are produced on the host with the engine's recurrence (n words, trivial next to the transfer) and the
// shuffle runs in the same kernels the worklist uses (shuffle.cuh), from a hand-built single-item plan.
int cbs_gpu_xperm(cbs_gpu_ctx* c, const double* x, const double* rwts, int32_t n, const uint64_t* mt_next312, uint64_t seed,
                  double* px) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n < 1 || !x || !px) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (n > 1000000) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "vectors longer than 1,000,000 are not supported");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    std::vector<uint64_t> words((size_t)n + 312);
    if (mt_next312) memcpy(words.data(), mt_next312, sizeof(uint64_t) * 312); else mt_seed_next312(seed, words.data());
    for (long long k = 312; k < (long long)n + 312; ++k) words[(size_t)k] = mt_twist(words[(size_t)k - 312], words[(size_t)k - 311], words[(size_t)k - 156]);
    std::vector<double> y(x, x + n);
    if (rwts) for (int i = 0; i < n; ++i) y[(size_t)i] = x[i] * rwts[i];  // CBS.cpp:540
    const long long stride = Sched::sx_stride(n);
    ENSURE(c, c->x, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->cur, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->ycur, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->rw, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->wts, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->unit_off, sizeof(long long) * 2);
    ENSURE(c, c->tasks, sizeof(Task));
    ENSURE(c, c->arena, sizeof(double) * (size_t)(stride + Sched::idx_stride(n) + 16));
    ENSURE(c, c->draws0, sizeof(uint64_t) * (size_t)(n + 312));
    ENSURE(c, c->items, sizeof(PermItem));
    ENSURE(c, c->shuf, sizeof(int) * 8);
    ENSURE(c, c->dev, sizeof(Dev));
    // which kernel takes a segment of n markers (cbs_core.h shuffle classes)
    int cls = shuffle_class(n, false), cl_R = 0, cl_grid = 0;
    size_t cl_smem = 0;
    if (cls == SHUF_GLOBAL)
        for (int R : {2, 4, 8}) { cl_grid = cluster_fit(c, R, n, 12, &cl_smem); if (cl_grid) { cl_R = R; break; } }
    Task t;
    memset(&t, 0, sizeof(t));
    t.unit = 0; t.lo = 0; t.hi = n; t.n = n; t.nb = block_count(n); t.raw = 1; t.off_sx = 0; t.off_A = stride; t.off_draw = 0;
    const PermItem item = {0, 1, 0};
    const int plan[8] = {0 /*shuf_item*/, 0, 1 /*shuf_prefix*/, 0 /*shuf_p0*/, 0, 0, 0, 0};
    const long long off[2] = {0, n};
    Dev hD;
    memset(&hD, 0, sizeof(hD));
    hD.x = c->x.as<double>(); hD.cur = c->cur.as<double>(); hD.unit_off = c->unit_off.as<long long>(); hD.n_units = 1;
    hD.prm.rng_mode = RNG_MT;
    hD.tasks = c->tasks.as<Task>(); hD.task_cap = 1;
    hD.arena = c->arena.as<double>(); hD.arena_cap = (long long)(c->arena.cap / 8);
    hD.draws[0] = c->draws0.as<uint64_t>(); hD.draws[1] = c->draws0.as<uint64_t>();
    hD.items = c->items.as<PermItem>(); hD.n_items = 1;
    for (int k = 0; k < SHUF_NCLS; ++k) { hD.shuf_item[k] = c->shuf.as<int>(); hD.shuf_prefix[k] = c->shuf.as<int>() + 1; hD.shuf_p0[k] = c->shuf.as<int>() + 3; }
    hD.n_shuf[cls] = 1;
    hD.shuf_arena = (cls == SHUF_GLOBAL && !cl_R) ? 1 : 0;
    if (rwts) { hD.w = c->wts.as<double>(); hD.rw = c->rw.as<double>(); hD.ycur = c->ycur.as<double>(); }
    CUDA_TRY(c, cudaMemcpyAsync(c->cur.p, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    if (rwts) {
        CUDA_TRY(c, cudaMemcpyAsync(c->ycur.p, y.data(), sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaMemcpyAsync(c->rw.p, rwts, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(c, cudaMemcpyAsync(c->draws0.p, words.data(), sizeof(uint64_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->unit_off.p, off, sizeof(off), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->tasks.p, &t, sizeof(t), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->items.p, &item, sizeof(item), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->shuf.p, plan, sizeof(plan), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->dev.p, &hD, sizeof(Dev), cudaMemcpyHostToDevice, st));
    Dev* dD = c->dev.as<Dev>();
    if (cls < SHUF_CL2) launch_shuffle(dD, cls, 1, st, true);
    else if (cl_R) launch_shuffle_cluster(dD, cl_R, SHUF_GLOBAL, 12, cl_R, cl_smem, st, true);
    else k_perm<<<1, 128, 0, st>>>(dD);
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(px, c->arena.as<double>() + 1, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return CBS_GPU_OK;
}

// cbs::htmaxp (CBS.hpp:34, CBS.cpp:387-485) for `count` vectors of n values laid end to end
int cbs_gpu_htmaxp(cbs_gpu_ctx* c, const double* px, int32_t n, int32_t count, double tss, int32_t k, int32_t al0, int32_t ibin,
                   double* statistics) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (ibin) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "htmaxp with ibin=true is not implemented");
    if (n < 2 || count < 1 || !px || !statistics) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (al0 < 1 || k < al0 || k > 128 || n <= 2 * k) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "need al0 <= k <= 128 and n > 2k");
    if (n > 1000000) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "vectors longer than 1,000,000 are not supported");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    const long long N = (long long)n * count;
    const int nb = block_count(n);
    const long long per = Sched::sx_stride(n) + Sched::bs_stride(nb);
    ENSURE(c, c->x, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->cur, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->gtab, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->factab, sizeof(double) * (size_t)(N + 1));
    ENSURE(c, c->bbtab, sizeof(int) * (size_t)(N + 1));
    ENSURE(c, c->unit_off, sizeof(long long) * (size_t)(count + 1));
    ENSURE(c, c->tasks, sizeof(Task) * (size_t)count);
    ENSURE(c, c->arena, sizeof(double) * (size_t)(per * count));
    ENSURE(c, c->rej, sizeof(int) * (size_t)count);
    ENSURE(c, c->prep_task, sizeof(int) * (size_t)count);
    ENSURE(c, c->items, sizeof(PermItem) * (size_t)count);
    ENSURE(c, c->item_prefix, sizeof(int) * (size_t)(count + 1));
    ENSURE(c, c->dev, sizeof(Dev));
    std::vector<long long> off((size_t)count + 1);
    std::vector<Task> tasks((size_t)count);
    std::vector<int> prep((size_t)count), prefix((size_t)count + 1);
    std::vector<PermItem> items((size_t)count);
    memset(tasks.data(), 0, sizeof(Task) * tasks.size());
    for (int u = 0; u <= count; ++u) off[(size_t)u] = (long long)u * n;
    for (int u = 0; u < count; ++u) {
        Task& t = tasks[(size_t)u];
        t.unit = u; t.lo = 0; t.hi = n; t.n = n; t.nb = nb; t.raw = 1; t.tss = tss; t.state = TS_PERM; t.use_hybrid = 1;
        t.off_sx = per * u; t.off_bs = per * u + Sched::sx_stride(n); t.off_rej = u; t.next = -1;
        prep[(size_t)u] = u; prefix[(size_t)u] = u;
        items[(size_t)u].task = u; items[(size_t)u].P = 1; items[(size_t)u].obs = 0;  // a "permutation" row: k_hscan takes it
    }
    prefix[(size_t)count] = count;
    Dev hD;
    memset(&hD, 0, sizeof(hD));
    hD.x = c->x.as<double>(); hD.unit_off = c->unit_off.as<long long>(); hD.n_units = count;
    hD.prm.min_width = al0; hD.prm.kmax = k; hD.prm.hybrid = 1; hD.prm.nperm = 0; hD.prm.rng_mode = RNG_PHILOX;
    hD.cur = c->cur.as<double>(); hD.gtab = c->gtab.as<double>(); hD.factab = c->factab.as<double>(); hD.bbtab = c->bbtab.as<int>();
    hD.tasks = c->tasks.as<Task>(); hD.task_cap = count;
    hD.arena = c->arena.as<double>(); hD.arena_cap = per * count; hD.rej = c->rej.as<int>(); hD.rej_cap = count;
    hD.n_prep = count; hD.prep_task = c->prep_task.as<int>();
    hD.n_items = count; hD.items = c->items.as<PermItem>(); hD.item_prefix = c->item_prefix.as<int>();
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, px, sizeof(double) * (size_t)N, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->unit_off.p, off.data(), sizeof(long long) * off.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->tasks.p, tasks.data(), sizeof(Task) * tasks.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->prep_task.p, prep.data(), sizeof(int) * prep.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->items.p, items.data(), sizeof(PermItem) * items.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->item_prefix.p, prefix.data(), sizeof(int) * prefix.size(), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->dev.p, &hD, sizeof(Dev), cudaMemcpyHostToDevice, st));
    Dev* dD = c->dev.as<Dev>();
    k_tables<<<dim3(16, 64), 256, 0, st>>>(dD);
    k_prep<<<std::min(count, c->sm_count * 8), 32, 0, st>>>(dD);  // prefix sums of the vectors as given (CBS.cpp:396-398)
    k_hscan<<<std::min(count, c->sm_count * 4), 256, 0, st>>>(dD);
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(tasks.data(), c->tasks.p, sizeof(Task) * tasks.size(), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    for (int u = 0; u < count; ++u) statistics[u] = tasks[(size_t)u].pval1;
    return CBS_GPU_OK;
}

// cbs::tailp (CBS.hpp:29, CBS.cpp:324-339); ngrid must be 100 (the device kernels' quadrature size)
int cbs_gpu_tailp(cbs_gpu_ctx* c, double b, double delta, int32_t m, int32_t ngrid, double tol, double* out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!out || m < 1) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (ngrid != TAILP_NGRID) return fail(c, CBS_GPU_ERR_UNSUPPORTED, "ngrid must be 100");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    ENSURE(c, c->tasks, sizeof(Task));
    ENSURE(c, c->prep_task, sizeof(int));
    ENSURE(c, c->tailp, sizeof(double) * TAILP_NGRID);
    ENSURE(c, c->dev, sizeof(Dev));
    Task t;
    memset(&t, 0, sizeof(t));
    t.n = m; t.hi = m; t.use_hybrid = 1; t.ostat = b * b;
    Dev hD;
    memset(&hD, 0, sizeof(hD));
    hD.prm.hybrid = 1; hD.prm.tol = tol; hD.api_mode = 4; hD.api_delta = delta;
    hD.tasks = c->tasks.as<Task>(); hD.n_prep = 1; hD.prep_task = c->prep_task.as<int>();
    const int zero = 0;
    CUDA_TRY(c, cudaMemcpyAsync(c->tasks.p, &t, sizeof(t), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->prep_task.p, &zero, sizeof(int), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->dev.p, &hD, sizeof(Dev), cudaMemcpyHostToDevice, st));
    k_tailp_terms<<<32, 128, 0, st>>>(c->dev.as<Dev>(), c->tailp.as<double>());
    k_tailp_sum<<<1, 64, 0, st>>>(c->dev.as<Dev>(), c->tailp.as<double>());
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(&t, c->tasks.p, sizeof(t), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    *out = t.pval1;
    return CBS_GPU_OK;
}

// cbs::btmax (CBS.hpp:31) / cbs::btailp (CBS.hpp:30): binary-data helpers (binary.cuh, kernels.cuh)
int cbs_gpu_btmax(cbs_gpu_ctx* c, const double* x, int32_t n, double* out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!x || !out || n < 1) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->means, sizeof(double) * 2);
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    k_btmax<<<1, 32, 0, st>>>(c->x.as<double>(), n, c->means.as<double>());
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(out, c->means.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return CBS_GPU_OK;
}

int cbs_gpu_btailp(cbs_gpu_ctx* c, double b, int32_t m, int32_t ng, double tol, double* out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (!out || m < 5 || ng < 1 || ng > 100000) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    ENSURE(c, c->tailp, sizeof(double) * (size_t)(ng + 2));
    ENSURE(c, c->means, sizeof(double) * 2);
    k_btailp_terms<<<std::min(c->sm_count, (ng + 4) / 4), 128, 0, st>>>(b, m, ng, tol, c->tailp.as<double>());
    k_btailp_sum<<<1, 32, 0, st>>>(b, m, ng, c->tailp.as<double>(), c->means.as<double>());
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(out, c->means.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    return CBS_GPU_OK;
}

void cbs_gpu_result_free(cbs_gpu_result* r) {
    if (!r) return;
    delete reinterpret_cast<ResultOwner*>(r);  // pub is the first member
}

int cbs_gpu_summarize_cn(cbs_gpu_ctx* c, const int64_t* seg_offsets, int32_t n_units, const uint64_t* seg_start,
                         const uint64_t* seg_end, const float* seg_value, int32_t direction, double cutoff,
                         const int64_t* pos_offsets, const uint64_t* positions, int64_t* out_offsets, uint64_t* out_pos,
                         double* out_value) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (direction != 1 && direction != -1) return fail(c, CBS_GPU_ERR_INVALID, "direction must be 1 or -1.");  // summarize.cpp:49-51
    if (n_units < 0 || !seg_offsets || !out_offsets) return fail(c, CBS_GPU_ERR_INVALID, "bad segment table");
    if (seg_offsets[0] != 0) return fail(c, CBS_GPU_ERR_INVALID, "seg_offsets[0] must be 0");
    for (int u = 0; u < n_units; ++u) if (seg_offsets[u + 1] < seg_offsets[u]) return fail(c, CBS_GPU_ERR_INVALID, "seg_offsets must be non-decreasing");
    const long long S = seg_offsets[n_units];
    if (S > 0 && (!seg_start || !seg_end || !seg_value)) return fail(c, CBS_GPU_ERR_INVALID, "segment columns are NULL");
    if (positions && !pos_offsets) return fail(c, CBS_GPU_ERR_INVALID, "positions without pos_offsets");
    // output positions per unit: given, or the sorted distinct starts and ends (summarize.cpp:24-36; a few per unit: host)
    std::vector<long long> poff((size_t)n_units + 1, 0);
    std::vector<unsigned long long> pos;
    for (int u = 0; u < n_units; ++u) {
        if (positions) {
            if (pos_offsets[u + 1] < pos_offsets[u] || pos_offsets[0] != 0) return fail(c, CBS_GPU_ERR_INVALID, "pos_offsets must start at 0 and be non-decreasing");
            pos.insert(pos.end(), positions + pos_offsets[u], positions + pos_offsets[u + 1]);
        } else {
            const size_t at = pos.size();
            for (long long k = seg_offsets[u]; k < seg_offsets[u + 1]; ++k) { pos.push_back(seg_start[k]); pos.push_back(seg_end[k]); }
            std::sort(pos.begin() + (long)at, pos.end());
            pos.erase(std::unique(pos.begin() + (long)at, pos.end()), pos.end());
        }
        poff[(size_t)u + 1] = (long long)pos.size();
        // the reference meets a segment with start > end while it scans for the first position of the unit (summarize.cpp:59-61)
        if (poff[(size_t)u + 1] > poff[(size_t)u])
            for (long long k = seg_offsets[u]; k < seg_offsets[u + 1]; ++k)
                if (seg_start[k] > seg_end[k]) return fail(c, CBS_GPU_ERR_INVALID, "Segment start is greater than end.");
    }
    for (int u = 0; u <= n_units; ++u) out_offsets[u] = poff[(size_t)u];
    const long long P = poff[(size_t)n_units];
    if (P == 0) return CBS_GPU_OK;
    if (!out_pos || !out_value) return fail(c, CBS_GPU_ERR_INVALID, "output arrays are NULL");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = c->stream;
    std::vector<long long> soff((size_t)n_units + 1);
    for (int u = 0; u <= n_units; ++u) soff[(size_t)u] = seg_offsets[u];
    // one scratch buffer: start | end | positions (8 B each), offsets, values (4 B), output
    const size_t b_start = 0, b_end = b_start + 8 * (size_t)S, b_pos = b_end + 8 * (size_t)S, b_soff = b_pos + 8 * (size_t)P,
                 b_poff = b_soff + 8 * ((size_t)n_units + 1), b_out = b_poff + 8 * ((size_t)n_units + 1), b_val = b_out + 8 * (size_t)P;
    ENSURE(c, c->cn_scratch, b_val + 4 * (size_t)S + 16);
    char* base = (char*)c->cn_scratch.p;
    if (S) {
        CUDA_TRY(c, cudaMemcpyAsync(base + b_start, seg_start, 8 * (size_t)S, cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaMemcpyAsync(base + b_end, seg_end, 8 * (size_t)S, cudaMemcpyHostToDevice, st));
        CUDA_TRY(c, cudaMemcpyAsync(base + b_val, seg_value, 4 * (size_t)S, cudaMemcpyHostToDevice, st));
    }
    CUDA_TRY(c, cudaMemcpyAsync(base + b_pos, pos.data(), 8 * (size_t)P, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(base + b_soff, soff.data(), 8 * ((size_t)n_units + 1), cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(base + b_poff, poff.data(), 8 * ((size_t)n_units + 1), cudaMemcpyHostToDevice, st));
    k_summarize_cn<<<(unsigned)std::min<long long>((P + 127) / 128, c->sm_count * 16), 128, 0, st>>>(
        (const unsigned long long*)(base + b_start), (const unsigned long long*)(base + b_end), (const float*)(base + b_val),
        (const long long*)(base + b_soff), (const long long*)(base + b_poff), n_units, (const unsigned long long*)(base + b_pos),
        direction, cutoff, (double*)(base + b_out));
    c->launches++;
    CUDA_TRY(c, cudaGetLastError());
    CUDA_TRY(c, cudaMemcpyAsync(out_value, base + b_out, 8 * (size_t)P, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    for (long long i = 0; i < P; ++i) out_pos[i] = pos[(size_t)i];
    return CBS_GPU_OK;
}

int cbs_gpu_smooth(cbs_gpu_ctx* c, const double* values, const int32_t* chrom, int64_t n, int32_t smooth_region,
                   double outlier_sd_scale, double smooth_sd_scale, double trim, double* out) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n < 0 || (n > 0 && (!values || !chrom || !out))) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (smooth_region < 0) return fail(c, CBS_GPU_ERR_INVALID, "smooth_region must be non-negative");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    if (n == 0) return CBS_GPU_OK;
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->lab, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->staging, sizeof(int) * (size_t)n);
    ENSURE(c, c->goff, sizeof(long long) * 2);
    const long long goff[2] = {0, (long long)n};
    std::vector<long long> off(goff, goff + 2);
    CUDA_TRY(c, cudaMemcpyAsync(c->lab.p, values, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->staging.p, chrom, sizeof(int) * (size_t)n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(c, cudaMemcpyAsync(c->goff.p, goff, sizeof(goff), cudaMemcpyHostToDevice, st));
    const int rc = smooth_device(c, c->lab.as<double>(), c->goff.as<long long>(), c->staging.as<int>(), 1, n, smooth_region,
                                 outlier_sd_scale, smooth_sd_scale, trim, c->x.as<double>(), off);
    if (rc) return rc;
    CUDA_TRY(c, cudaMemcpyAsync(out, c->x.p, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(c, cudaStreamSynchronize(st));
    if (c->profiling) collect_timers(c);
    return CBS_GPU_OK;
}

int cbs_gpu_segment(cbs_gpu_ctx* c, const double* x, int32_t n, const cbs_gpu_params* params, const uint64_t* mt_next312,
                    int32_t cap, int32_t* lengths, double* means, int32_t* n_segments, uint64_t* draws_consumed) {
    if (!c) return CBS_GPU_ERR_INVALID;
    if (n < 0 || (n > 0 && !x) || !n_segments) return fail(c, CBS_GPU_ERR_INVALID, "bad arguments");
    if (cudaSetDevice(c->device) != cudaSuccess) return fail(c, CBS_GPU_ERR_CUDA, "cudaSetDevice failed");
    cbs_gpu_params p = *params;
    p.do_smooth = 0;  // cbs::segment does not smooth
    int rc = validate_params(c, &p);
    if (rc) return rc;
    *n_segments = 0;
    if (draws_consumed) *draws_consumed = 0;
    if (n == 0) return CBS_GPU_OK;  // cbs::segment on an empty vector returns no segments
    cudaStream_t st = c->stream;
    ENSURE(c, c->x, sizeof(double) * (size_t)(n + 1));
    ENSURE(c, c->flag, sizeof(int));
    CUDA_TRY(c, cudaMemcpyAsync(c->x.p, x, sizeof(double) * (size_t)n, cudaMemcpyHostToDevice, st));
    for (int i = 0; i < n; ++i) if (!std::isfinite(x[i])) return fail(c, CBS_GPU_ERR_NONFINITE, "non-finite values reach CBS");
    std::vector<long long> off = {0, (long long)n};
    Dev hD;
    for (int k = 0; k < K_COUNT; ++k) c->kms[k] = 0.0;
    rc = run_cbs(c, off, nullptr, 1, &p, mt_next312, false, hD);
    if (rc) return rc;
    ResultOwner R;
    memset(&R.pub, 0, sizeof(R.pub));
    rc = fetch_results(c, hD, 1, false, &R, &p, &off);
    if (rc) return rc;
    if (c->profiling) collect_timers(c);
    *n_segments = (int32_t)R.pub.n_segments;
    if (draws_consumed) *draws_consumed = R.draws[0];
    if (R.pub.n_segments > cap) return fail(c, CBS_GPU_ERR_CAPACITY, "output capacity too small");
    for (int64_t k = 0; k < R.pub.n_segments; ++k) { lengths[k] = R.lengths[k]; means[k] = R.means[k]; }
    return CBS_GPU_OK;
}

}  // extern "C"
