// weighted.cuh -- sm_100a kernels of weighted CBS (cbs::segment_weighted, /root/reference lib/cbs/CBS.cpp:1026-1099).
//
// The control flow of wfindcpt (CBS.cpp:894-957) is the one of fndcpt, so the device worklist and its scheduler
// (cbs_core.h) are shared with the unweighted path; what changes is the arithmetic of every kernel:
//   k_wsetup   rw = sqrt(w) for the whole call (CBS.cpp:1056), weights validated
//   k_wprep    per pending segment: all-equal test, weighted mean, centring, weighted tss, cw = cumsum(w)/sqrt(sum w),
//              prefix sums of cur*w (CBS.cpp:1051-1067, wtmaxo :621-637) -- every sum is ONE sequential chain on lane 0
//   (shuffle)  perm_warp gathers ycur[idx]/rw[pos] (wxperm, CBS.cpp:538-547, including its j == i quirk)
//   (k_chain)  multiplies the gathered values by w before the sequential prefix chain (wtmaxo :623,627)
//   k_wscan    wtmaxo / wtmaxp (CBS.cpp:610-743): CTA per (segment, permutation)
//   k_wedgeprep, k_wedgeperm   wtpermp (CBS.cpp:549-591)
//   k_wmeans   weighted segment means (CBS.cpp:1091-1097)
//   k_wdelta, k_wssq, k_whscan   the weighted hybrid method (getmncwt :593-608, hwtmaxp :745-828)
#pragma once

namespace cbsg {

__global__ void k_wsetup(const double* __restrict__ w, double* __restrict__ rw, long long N, int* bad) {
    int b = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < N; i += (long long)gridDim.x * blockDim.x) {
        const double v = w[i];
        if (!(v > 0.0) || isinf(v)) b = 1;
        rw[i] = sqrt(v);
    }
    if (b) atomicOr(bad, 1);
}

// ------------------------------------------------------------------------------------
// k_wprep: one warp per new pending segment (CBS.cpp:1046-1067 and the prefix sums of wtmaxo :621-637 on observed data)
// ------------------------------------------------------------------------------------
#define WPREP_CHUNK 512
#define WPREP_Q (WPREP_CHUNK / 32)
__device__ void wprep_warp(Dev* D, Task& t, int lane, double* __restrict__ bx, double* __restrict__ bw) {
    const long long base = D->unit_off[t.unit] + t.lo;
    const double* __restrict__ x = D->x + base;
    const double* __restrict__ w = D->w + base;
    const double* __restrict__ rw = D->rw + base;
    double* __restrict__ cur = D->cur + base;
    double* __restrict__ cw = D->cw + base;
    double* __restrict__ ycur = D->ycur + base;
    const int n = t.n;
    // CBS.cpp:1051 all-equal test (loads batched in registers: a warp has nothing else to hide their latency with)
    const double x0 = x[0];
    bool flat = true;
    for (int i0 = 0; i0 < n; i0 += 32 * WPREP_Q) {
        double v[WPREP_Q];
#pragma unroll
        for (int q = 0; q < WPREP_Q; ++q) { const int i = i0 + lane + 32 * q; v[q] = (i < n) ? x[i] : x0; }
#pragma unroll
        for (int q = 0; q < WPREP_Q; ++q) if (!(fabs(v[q] - x0) < 1e-12)) flat = false;
    }
    flat = __all_sync(FULL, flat) && !t.raw;  // cbs::wfindcpt (low-level entry) takes the vector as it is
    if (lane == 0) { t.alleq = flat ? 1 : 0; t.w_level = 0ull; t.w_found = 0ull; t.w_set = 0; t.w_lock = 0; t.w_tie = 0; t.w_init = -1.0; }
    if (flat) return;
    // CBS.cpp:1053-1058: wsum, wxsum.  Every sum is sequential, but the sums are independent of each other: lane 0 runs
    // them as interleaved DADD chains over values the whole warp staged in shared memory (products included: they are
    // rounded before the addition, as in the reference).  The partial sums of w are kept: they are cw before scaling.
    double wsum = 0.0, wxsum = 0.0;
    double vx[WPREP_Q], vw[WPREP_Q];  // the next chunk, in flight while lane 0 walks the current one
#pragma unroll
    for (int q = 0; q < WPREP_Q; ++q) { const int k = lane + 32 * q; vx[q] = (k < n) ? x[k] : 0.0; vw[q] = (k < n) ? w[k] : 0.0; }
    for (int c0 = 0; c0 < n; c0 += WPREP_CHUNK) {
        const int cnt = min(WPREP_CHUNK, n - c0);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < WPREP_Q; ++q) { const int k = lane + 32 * q; bw[k] = vw[q]; bx[k] = vw[q] * vx[q]; }
        __syncwarp();
        if (c0 + WPREP_CHUNK < n) {
#pragma unroll
            for (int q = 0; q < WPREP_Q; ++q) { const int i = c0 + WPREP_CHUNK + lane + 32 * q; vx[q] = (i < n) ? x[i] : 0.0; vw[q] = (i < n) ? w[i] : 0.0; }
        }
        if (lane == 0) {  // two independent chains interleaved in one thread: both advance at the DADD latency
            int k = 0;
            for (; k + 8 <= cnt; k += 8) {  // operands of 8 steps in registers first: the loads do not wait for the stores
                double a[8], b[8];
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const double2 va = *reinterpret_cast<const double2*>(bw + k + u), vb = *reinterpret_cast<const double2*>(bx + k + u);
                    a[u] = va.x; a[u + 1] = va.y; b[u] = vb.x; b[u + 1] = vb.y;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) { wsum = wsum + a[u]; a[u] = wsum; wxsum = wxsum + b[u]; }
#pragma unroll
                for (int u = 0; u < 8; u += 2) *reinterpret_cast<double2*>(bw + k + u) = make_double2(a[u], a[u + 1]);
            }
            for (; k < cnt; ++k) { wsum = wsum + bw[k]; wxsum = wxsum + bx[k]; bw[k] = wsum; }
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < WPREP_Q; ++q) { const int k = lane + 32 * q; if (k < cnt) cw[c0 + k] = bw[k]; }  // unscaled csum (CBS.cpp:1065)
    }
    wsum = shfl_d(wsum, 0); wxsum = shfl_d(wxsum, 0);
    const double avg = t.raw ? 0.0 : wxsum / wsum;  // raw: x is already centred and its tss is the caller's (wfindcpt arguments)
    const double cwscale = sqrt(wsum);
    // CBS.cpp:1061-1066 centring, weighted tss, cw; wtmaxo :623,627 prefix sums of cur*w
    double* __restrict__ sx = D->arena + t.off_sx;
    double wxx = 0.0, run = 0.0;
    if (lane == 0) sx[0] = 0.0;
#pragma unroll
    for (int q = 0; q < WPREP_Q; ++q) { const int k = lane + 32 * q; vx[q] = (k < n) ? x[k] : 0.0; vw[q] = (k < n) ? w[k] : 0.0; }
    for (int c0 = 0; c0 < n; c0 += WPREP_CHUNK) {
        const int cnt = min(WPREP_CHUNK, n - c0);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < WPREP_Q; ++q) {
            const int k = lane + 32 * q;
            const double v = vx[q] - avg, ww = vw[q];
            bx[k] = v * ww;       // :623,627
            bw[k] = ww * v * v;   // :1063
            if (k < cnt) cur[c0 + k] = v;
        }
        __syncwarp();
        if (c0 + WPREP_CHUNK < n) {
#pragma unroll
            for (int q = 0; q < WPREP_Q; ++q) { const int i = c0 + WPREP_CHUNK + lane + 32 * q; vx[q] = (i < n) ? x[i] : 0.0; vw[q] = (i < n) ? w[i] : 0.0; }
        }
        if (lane == 0) {
            int k = 0;
            for (; k + 8 <= cnt; k += 8) {
                double a[8], b[8];
#pragma unroll
                for (int u = 0; u < 8; u += 2) {
                    const double2 va = *reinterpret_cast<const double2*>(bx + k + u), vb = *reinterpret_cast<const double2*>(bw + k + u);
                    a[u] = va.x; a[u + 1] = va.y; b[u] = vb.x; b[u + 1] = vb.y;
                }
#pragma unroll
                for (int u = 0; u < 8; ++u) { run = run + a[u]; a[u] = run; wxx = wxx + b[u]; }
#pragma unroll
                for (int u = 0; u < 8; u += 2) *reinterpret_cast<double2*>(bx + k + u) = make_double2(a[u], a[u + 1]);
            }
            for (; k < cnt; ++k) { run = run + bx[k]; wxx = wxx + bw[k]; bx[k] = run; }
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < WPREP_Q; ++q) { const int k = lane + 32 * q; if (k < cnt) sx[c0 + 1 + k] = bx[k]; }
    }
    // elementwise tail with all lanes: ycur = cur*rw (what wxperm shuffles, :540), cw scaled (:1066)
    for (int i0 = 0; i0 < n; i0 += 32 * 8) {
        double a[8], b[8], c2[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) { const int i = i0 + lane + 32 * q; const bool in = i < n; a[q] = in ? cur[i] : 0.0; b[q] = in ? rw[i] : 0.0; c2[q] = in ? cw[i] : 0.0; }
#pragma unroll
        for (int q = 0; q < 8; ++q) { const int i = i0 + lane + 32 * q; if (i < n) { ycur[i] = a[q] * b[q]; cw[i] = c2[q] / cwscale; } }
    }
    wxx = shfl_d(wxx, 0);
    run = shfl_d(run, 0);
    for (int k = lane; k < SX_PAD; k += 32) sx[n + 1 + k] = run;
    if (lane == 0 && !t.raw) t.tss = wxx;
}

__global__ void __launch_bounds__(32) k_wprep(Dev* D) {
    __shared__ __align__(16) double bx[WPREP_CHUNK];
    __shared__ __align__(16) double bw[WPREP_CHUNK];
    if (D->done) return;
    for (int k = blockIdx.x; k < D->n_prep; k += gridDim.x) wprep_warp(D, D->tasks[D->prep_task[k]], threadIdx.x, bx, bw);
}

// k_wtables: per new segment and block b the smallest weight of an arc of al0 markers inside the block (bound of the
// diagonal pair (b,b), CBS.cpp:662-664) and across the boundary to block b+1 (pair (b,b+1), :665-667).  They depend on cw
// only, not on the row, so every permutation of the segment reuses them (the reference recomputes them per call).
// Stored in the per-marker tables the unweighted scan uses for g[L] / fac[L] (unused by weighted CBS), at the segment's
// offset.  Runs after k_wprep on the same stream.
__global__ void __launch_bounds__(256) k_wtables(Dev* D) {
    if (D->done) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int al0 = D->prm.min_width;
    for (int k = blockIdx.x; k < D->n_prep; k += gridDim.x) {
        const Task& t = D->tasks[D->prep_task[k]];
        if (t.alleq) continue;
        const long long base = D->unit_off[t.unit] + t.lo;
        const double* __restrict__ cw = D->cw + base;
        const int* __restrict__ bb = D->bbtab + base;
        double* dmin = D->gtab + base;
        double* adjmin = D->factab + base;
        const int n = t.n, nb = t.nb;
        const double inf = __longlong_as_double(0x7ff0000000000000LL);
        for (int b = 1 + warp; b <= nb; b += nwarps) {
            const int ilo = bb[b - 1] + 1, ihi = bb[b];
            double m1 = inf, m2 = inf;
            if (lane == 0) m1 = cw[min(ilo + al0, n) - 1] - cw[ilo - 1];
            for (int kk = ilo + 1 + lane; kk <= ihi - al0; kk += 32) m1 = fmin(m1, cw[kk + al0 - 1] - cw[kk - 1]);
            if (b < nb) {
                const int jlo = ihi + 1;
                if (lane == 0) m2 = cw[jlo - 1] - cw[max(jlo - al0, 1) - 1];
                for (int kk = max(jlo - al0 + 1, 1) + lane; kk <= ihi; kk += 32) m2 = fmin(m2, cw[min(kk + al0, n) - 1] - cw[kk - 1]);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { m1 = fmin(m1, shfl_d(m1, lane ^ o)); m2 = fmin(m2, shfl_d(m2, lane ^ o)); }
            if (lane == 0) { dmin[b - 1] = m1; adjmin[b - 1] = m2; }
        }
    }
}

// ------------------------------------------------------------------------------------
// k_wscan: wtmaxo (observed data: statistic and location) / wtmaxp (permutation: reject decision), CBS.cpp:610-743.
//
// The reference lists the block pairs whose bound reaches the statistic of the global-extrema arc (:650-693), visits
// them by descending corner statistic and scans, per pair, the arcs (i, j) whose weight awt1 = cw[j-1]-cw[i-1] lies in
// the pair's bands awt1 <= awtmax (:708-719) and awt1 >= psrn-awtmax (:721-733); a pair is skipped when the running
// maximum exceeds its bound.  The bound is an upper bound of every arc of the pair, so the maximum is the maximum over
// the arcs of all listed pairs: here the warps of a CTA take the pairs 32 at a time, each lane evaluates the bound of
// one pair, and the warp scans the pairs that reach the current level (rows of the pair one after the other, the lanes
// along j; cw is monotone, so a row ends at the first 32 arcs outside the band).  An arc costs two subtractions and
// three multiplications (s*s > level*den); only a hit divides.  Permutations only need their reject decision: the level
// starts at the statistic M* a permutation must reach to reject (decision mode, as in k_scan).
// Location (observed data): ties follow the reference's visiting order -- the global-extrema arc first, then pairs by
// descending corner statistic, low band (i descending, j ascending) before high band (i ascending, j descending); it is
// resolved in a second pass over the arcs that attain the maximum.  Pairs with EQUAL corner statistics are ordered by
// their position in the list (the reference's std::sort order is unspecified there).
// ------------------------------------------------------------------------------------
struct WScanSmem {
    unsigned long long level;  // bit pattern of the prune level (positive doubles order like integers)
    unsigned long long found;  // bit pattern of the best statistic found
    double g_min, g_max;
    int g_imin, g_imax;
    int next_pair, lock;
    unsigned long long* glevel; unsigned long long* gfound;  // copies of WRow's
    int decided;  // decision mode: an arc that makes the permutation reject has been found, stop scanning
    double rej_at;  // smallest statistic that certainly rejects (decision mode), +inf otherwise
    // location record: best arc among those that attain the maximum
    double r_corner, r_v;
    int r_q, r_phase, r_o1, r_o2, r_i, r_j, r_set;
    int tie;  // wcand_tied was seen: the location needs the ordered walk
};

struct WRow {
    int n, nb, al0, nal0;
    const double* sx;   // prefix sums sx[0..n]
    const double* cw;   // cw[0..n-1]
    const int* bb;      // smem bb[0..nb]
    const double* bmin; const double* bmax; const int* amin; const int* amax;  // smem, per block (0-based)
    const double* dmin; const double* adjmin;  // k_wtables
    int q_first, q_stride;                     // pairs of this CTA: batches of 32 starting at q_first, q_stride apart
    unsigned long long* glevel; unsigned long long* gfound;  // observed scan shared by several CTAs (else nullptr)
    double psrn, psrnov2, init;
};

struct WPair {
    int bi, bj, ilo1, ihi, jlo, jhi;
    double bsslim;   // bound (:676)
    double awt;      // weight of the corner arc (:683,686)
    double corner;   // its statistic bssbij (:684,687)
    bool listed;     // bssmax0 <= bsslim (:677)
};

__device__ __forceinline__ void wpair_from_index(int q, int nb, int& bi, int& bj) { pair_from_index(q, nb, bi, bj); }

// bound and corner of block pair (bi, bj), 1-based (CBS.cpp:652-689)
__device__ void wpair_eval(const WRow& r, int bi, int bj, WPair& p) {
    const double* cw = r.cw;
    p.bi = bi; p.bj = bj;
    p.ilo1 = r.bb[bi - 1] + 1; p.ihi = r.bb[bi]; p.jlo = r.bb[bj - 1] + 1; p.jhi = r.bb[bj];
    const int al0 = r.al0;
    double awthi = cw[p.jhi - 1] - cw[p.ilo1 - 1];
    if (p.jhi - p.ilo1 > r.nal0) {
        awthi = 0.0;
        for (int kk = 1; kk <= al0; ++kk) awthi = fmax(awthi, cw[r.nal0 + kk - 1] - cw[kk - 1]);
    }
    double awtlo;
    if (bi == bj) {
        awtlo = r.dmin[bi - 1];    // :662-664 (k_wtables)
    } else if (bi + 1 == bj) {
        awtlo = r.adjmin[bi - 1];  // :665-667
    } else {
        awtlo = cw[p.jlo - 1] - cw[p.ihi - 1];
    }
    const double sij1 = fabs(r.bmax[bj - 1] - r.bmin[bi - 1]);
    const double sij2 = fabs(r.bmax[bi - 1] - r.bmin[bj - 1]);
    const double sijmx0 = fmax(sij1, sij2);
    p.bsslim = (sijmx0 * sijmx0) / fmin(awtlo * (r.psrn - awtlo), awthi * (r.psrn - awthi));
    p.listed = r.init <= p.bsslim;
    if (sij1 > sij2) {
        p.awt = fabs(cw[r.amax[bj - 1] - 1] - cw[r.amin[bi - 1] - 1]);
        p.corner = (sij1 * sij1) / (p.awt * (r.psrn - p.awt));
    } else {
        p.awt = fabs(cw[r.amin[bj - 1] - 1] - cw[r.amax[bi - 1] - 1]);
        p.corner = (sij2 * sij2) / (p.awt * (r.psrn - p.awt));
    }
}

struct WCand {
    double corner;
    int q, phase, o1, o2, i, j;
    bool set;
    double v;  // statistic of the arc
};
// true if a is visited before b by the reference
__device__ __forceinline__ bool wcand_before(const WCand& a, const WCand& b) {
    if (!b.set) return a.set;
    if (!a.set) return false;
    if (a.corner != b.corner) return a.corner > b.corner;
    // equal corner statistics: the reference's std::sort leaves short runs of equal keys in enumeration order (its final
    // insertion sort is stable) and visits the sorted list from the back, so the LATER pair of the enumeration comes first
    if (a.q != b.q) return a.q > b.q;
    if (a.phase != b.phase) return a.phase < b.phase;
    if (a.o1 != b.o1) return a.o1 < b.o1;
    return a.o2 < b.o2;
}

// the same maximum in two different pairs whose corner statistics are EQUAL: which one the reference visits first depends on
// where std::sort leaves equal keys (it is not stable beyond 16 elements), which the keys above cannot express
__device__ __forceinline__ bool wcand_tied(const WCand& a, const WCand& b) {
    return a.set && b.set && a.v == b.v && a.corner == b.corner && a.q != b.q;
}

// larger statistic first, then the reference's visiting order
__device__ __forceinline__ bool wcand_better(const WCand& a, const WCand& b) {
    if (!b.set) return a.set;
    if (!a.set) return false;
    if (a.v != b.v) return a.v > b.v;
    return wcand_before(a, b);
}

// one warp scans the two bands of a pair (CBS.cpp:700-734), raising level/found.  LOC == true (observed rows): every
// lane also keeps the best arc it has seen -- largest statistic, earliest in the reference's visiting order among equals.
// An arc that attains the final maximum M always passes the filter (the level never exceeds M) and its pair is never
// skipped (bound >= M >= level), so the reduction of these records over lanes, warps and CTAs is the reference's location.
// Mapping: every lane owns a row i (its S_i and cw_i stay in registers) and the warp walks j together, so the two loads
// of a step (S_j, cw_j) are broadcasts that hit L1, independent from step to step (pipelined), and a step evaluates 32
// arcs.  cw is monotone, hence a row's band is one interval of j: the walk ends when every lane has left its interval.
template <bool LOC>
__device__ __forceinline__ void warc_eval(const WPair& p, int q, WScanSmem* sm, WCand& best, double lvl,
                                          double d, double a1, double psrn, int phase, int o1, int o2, int i, int j) {
    const double d2 = d * d, den = a1 * (psrn - a1);
    if (d2 > lvl * den) {
        const double v = d2 / den;
        if (LOC) {
            WCand c{p.corner, q, phase, o1, o2, i, j, true, v};
            if (wcand_tied(c, best)) sm->tie = 1;
            if (wcand_better(c, best)) best = c;
        }
        if (v > __longlong_as_double((long long)*((volatile unsigned long long*)&sm->level))) {
            atomicMax(&sm->found, (unsigned long long)__double_as_longlong(v));
            atomicMax(&sm->level, (unsigned long long)__double_as_longlong(v));
            if (sm->gfound) { atomicMax(sm->gfound, (unsigned long long)__double_as_longlong(v)); atomicMax(sm->glevel, (unsigned long long)__double_as_longlong(v)); }
            // rej_at is +inf when the early decision is off; an infinite arc (weight 0, only where cw is not strictly
            // increasing) must not match it: the reference's statistic is then NaN, which never rejects (CBS.cpp:933)
            if (v >= sm->rej_at && sm->rej_at < __longlong_as_double(0x7ff0000000000000LL)) sm->decided = 1;
        }
    }
}

template <bool LOC>
__device__ void wscan_pair(const WRow& r, const WPair& p, int q, WScanSmem* sm, WCand& best, int lane) {
    const double* __restrict__ sx = r.sx;
    const double* __restrict__ cw = r.cw;
    const double psrn = r.psrn;
    double awtmax = p.awt;
    const double awthi = cw[p.jhi - 1] - cw[p.ilo1 - 1];
    const double awtlo = (p.bi == p.bj) ? 0.0 : (cw[p.jlo - 1] - cw[p.ihi - 1]);
    if (awtmax > psrn - awtmax) awtmax = psrn - awtmax;
    const volatile unsigned long long* vlevel = &sm->level;
    if (awtlo <= r.psrnov2) {
        // low band: i = ihi1 .. ilo1 (descending in the reference), j = max(i+al0, jlo) .. jhi while awt1 <= awtmax
        const int ihi1 = (p.bi == p.bj) ? p.ihi - r.al0 : p.ihi;
        for (int g0 = ihi1; g0 >= p.ilo1; g0 -= 32) {
            if (__any_sync(FULL, *((volatile int*)&sm->decided))) break;  // warp-uniform exit
            const int i = g0 - lane;
            const bool active = i >= p.ilo1;
            const double sxi = active ? sx[i] : 0.0, cwi = active ? cw[i - 1] : 0.0;
            const int jlo1 = active ? max(i + r.al0, p.jlo) : 0x7fffffff;
            double lvl = __longlong_as_double((long long)*vlevel) * (1.0 - 1e-12);
            // the lanes' first j differ only on the diagonal pair: start at the smallest
            int jstart = jlo1;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) jstart = min(jstart, __shfl_xor_sync(FULL, jstart, o));
            bool done = !active;
            for (int j0 = jstart; j0 <= p.jhi; j0 += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 + u;
                    if (j <= p.jhi) {
                        const double sj = sx[j], cj = cw[j - 1];
                        if (!done && j >= jlo1) {
                            const double a1 = cj - cwi;
                            if (a1 <= awtmax) warc_eval<LOC>(p, q, sm, best, lvl, sj - sxi, a1, psrn, 0, ihi1 - i, j, i, j);
                            else done = true;
                        }
                    }
                }
                if (__all_sync(FULL, done)) break;
                if (((j0 - jstart) & 63) == 60) lvl = __longlong_as_double((long long)*vlevel) * (1.0 - 1e-12);
            }
        }
    }
    awtmax = psrn - awtmax;
    if (awthi >= r.psrnov2) {
        // high band: i = ilo1 .. ihi (ascending), j = jhi1 .. jlo (descending) while awt1 >= psrn - awtmax
        const bool wrap = (p.bi == 1) && (p.bj == r.nb);
        for (int g0 = p.ilo1; g0 <= p.ihi; g0 += 32) {
            if (__any_sync(FULL, *((volatile int*)&sm->decided))) break;
            const int i = g0 + lane;
            const bool active = i <= p.ihi;
            const double sxi = active ? sx[i] : 0.0, cwi = active ? cw[i - 1] : 0.0;
            const int jhi1 = active ? (wrap ? min(p.jhi, p.jhi - r.al0 + i) : p.jhi) : -1;
            double lvl = __longlong_as_double((long long)*vlevel) * (1.0 - 1e-12);
            int jstart = jhi1;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) jstart = max(jstart, __shfl_xor_sync(FULL, jstart, o));
            bool done = !active;
            for (int j0 = jstart; j0 >= p.jlo; j0 -= 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const int j = j0 - u;
                    if (j >= p.jlo) {
                        const double sj = sx[j], cj = cw[j - 1];
                        if (!done && j <= jhi1) {
                            const double a1 = cj - cwi;
                            if (a1 >= awtmax) warc_eval<LOC>(p, q, sm, best, lvl, sj - sxi, a1, psrn, 1, i - p.ilo1, -j, i, j);
                            else done = true;
                        }
                    }
                }
                if (__all_sync(FULL, done)) break;
                if (((jstart - j0) & 63) == 60) lvl = __longlong_as_double((long long)*vlevel) * (1.0 - 1e-12);
            }
        }
    }
}

// all warps of the CTA walk the pair list once
template <bool LOC>
__device__ void wscan_pass(const WRow& r, WScanSmem* sm, int lane) {
    const int npairs = r.nb * (r.nb + 1) / 2;
    WCand best;
    best.set = false; best.corner = 0.0; best.q = 0; best.phase = 0; best.o1 = 0; best.o2 = 0; best.i = 0; best.j = 0; best.v = 0.0;
    for (;;) {
        int q0 = 0;
        if (lane == 0) {
            q0 = atomicAdd(&sm->next_pair, r.q_stride);
            // level found by the other CTAs that scan this row
            if (r.glevel) atomicMax(&sm->level, *((volatile unsigned long long*)r.glevel));
        }
        q0 = __shfl_sync(FULL, q0, 0);
        if (q0 >= npairs) break;
        if (__any_sync(FULL, *((volatile int*)&sm->decided))) break;
        const int q = q0 + lane;
        WPair p;
        bool alive = false;
        if (q < npairs) {
            int bi, bj;
            wpair_from_index(q, r.nb, bi, bj);
            wpair_eval(r, bi, bj, p);
            const double lvl = __longlong_as_double((long long)*((volatile unsigned long long*)&sm->level));
            alive = p.listed && !(p.bsslim * (1.0 + 1e-12) < lvl);
        }
        unsigned mask = __ballot_sync(FULL, alive);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            WPair s;
            s.bi = __shfl_sync(FULL, p.bi, src); s.bj = __shfl_sync(FULL, p.bj, src);
            s.ilo1 = __shfl_sync(FULL, p.ilo1, src); s.ihi = __shfl_sync(FULL, p.ihi, src);
            s.jlo = __shfl_sync(FULL, p.jlo, src); s.jhi = __shfl_sync(FULL, p.jhi, src);
            s.bsslim = shfl_d(p.bsslim, src); s.awt = shfl_d(p.awt, src); s.corner = shfl_d(p.corner, src);
            s.listed = true;
            {  // the level may have risen since the bound was evaluated (read once per warp: uniform branch)
                double lvl = 0.0;
                if (lane == 0) lvl = __longlong_as_double((long long)*((volatile unsigned long long*)&sm->level));
                lvl = shfl_d(lvl, 0);
                if (s.bsslim * (1.0 + 1e-12) < lvl) continue;
            }
            wscan_pair<LOC>(r, s, q0 + src, sm, best, lane);
        }
    }
    if (LOC) {
        // warp reduction of the first-visited arc, then merge into the CTA's record under a lock
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            WCand c;
            c.corner = shfl_d(best.corner, lane ^ o);
            c.q = __shfl_xor_sync(FULL, best.q, o); c.phase = __shfl_xor_sync(FULL, best.phase, o);
            c.o1 = __shfl_xor_sync(FULL, best.o1, o); c.o2 = __shfl_xor_sync(FULL, best.o2, o);
            c.i = __shfl_xor_sync(FULL, best.i, o); c.j = __shfl_xor_sync(FULL, best.j, o);
            c.set = __shfl_xor_sync(FULL, best.set ? 1 : 0, o) != 0;
            c.v = shfl_d(best.v, lane ^ o);
            if (wcand_tied(c, best)) sm->tie = 1;
            if (wcand_better(c, best)) best = c;
        }
        if (lane == 0 && best.set) {
            while (atomicCAS(&sm->lock, 0, 1) != 0) {}
            __threadfence_block();
            WCand cur{sm->r_corner, sm->r_q, sm->r_phase, sm->r_o1, sm->r_o2, sm->r_i, sm->r_j, sm->r_set != 0, sm->r_v};
            if (wcand_tied(best, cur)) sm->tie = 1;
            if (wcand_better(best, cur)) {
                sm->r_v = best.v;
                sm->r_corner = best.corner; sm->r_q = best.q; sm->r_phase = best.phase; sm->r_o1 = best.o1; sm->r_o2 = best.o2;
                sm->r_i = best.i; sm->r_j = best.j; sm->r_set = 1;
            }
            __threadfence_block();
            atomicExch(&sm->lock, 0);
        }
    }
}

// MODE 0: the permutation rows of the round, one CTA per row (reject decision).
// MODE 1: the observed rows (PermItem::obs == 1), each spread over WOBS_SLICES CTAs that take interleaved batches of
//         block pairs and share the running maximum through Task::w_level / w_found: an observed scan is ~n^1.5 arcs
//         (1e8 for a 150 000 marker chromosome) and a round has only a few of them, so one CTA per row leaves the GPU idle.
//         Every CTA merges its best arc into the row's record (Task::w_v, w_i, w_j, ...); k_wobs_fin then writes
//         ostat / tmaxi / tmaxj (the kernel boundary is the grid-wide barrier).
#define WOBS_SLICES 24
template <int MODE>
__global__ void __launch_bounds__(256) k_wscan(Dev* D, int nb_max) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (D->done) return;
    WScanSmem* sm = (WScanSmem*)smem_raw;
    double* s_bmin = (double*)(smem_raw + ((sizeof(WScanSmem) + 15) & ~(size_t)15));
    double* s_bmax = s_bmin + nb_max;
    int* s_amin = (int*)(s_bmax + nb_max);
    int* s_amax = s_amin + nb_max;
    int* s_bb = s_amax + nb_max;
    __shared__ int s_g;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = blockDim.x >> 5;
    const int total = MODE == 0 ? D->item_prefix[D->n_items] : D->n_items * WOBS_SLICES;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_g = (int)atomicAdd(&D->ctr[MODE == 0 ? 1 : 5], 1u);
        __syncthreads();
        const int gidx = s_g;
        if (gidx >= total) break;
        int k, p = 0, slice = 0;
        if (MODE == 0) { k = find_item(D->item_prefix, D->n_items, gidx); p = gidx - D->item_prefix[k]; }
        else { k = gidx / WOBS_SLICES; slice = gidx - k * WOBS_SLICES; }
        const PermItem it = D->items[k];
        if ((MODE == 0) != (it.obs != 1)) continue;  // observed rows: MODE 1/2 only
        Task& t = D->tasks[it.task];
        if (it.obs && t.alleq) continue;
        if (!it.obs && t.use_hybrid) continue;  // k_whscan
        const int n = t.n, nb = t.nb;
        const long long base = D->unit_off[t.unit] + t.lo;
        WRow r;
        r.n = n; r.nb = nb; r.al0 = D->prm.min_width; r.nal0 = n - r.al0;
        r.sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        r.cw = D->cw + base;
        r.dmin = D->gtab + base; r.adjmin = D->factab + base;
        r.bb = s_bb; r.bmin = s_bmin; r.bmax = s_bmax; r.amin = s_amin; r.amax = s_amax;
        r.q_first = MODE == 0 ? 0 : 32 * slice;
        r.q_stride = MODE == 0 ? 32 : 32 * WOBS_SLICES;
        r.glevel = MODE == 1 ? &t.w_level : nullptr;
        r.gfound = MODE == 1 ? &t.w_found : nullptr;
        const int* bbg = D->bbtab + base;
        for (int b = tid; b <= nb; b += blockDim.x) s_bb[b] = bbg[b];
        __syncthreads();
        // per-block extrema of the prefix sums with their FIRST occurrence (CBS.cpp:624-633): a warp per block
        for (int b = warp; b < nb; b += nwarps) {
            const int first = s_bb[b] + 1, last = s_bb[b + 1];
            double lo = __longlong_as_double(0x7ff0000000000000LL), hi = -lo;
            int ilo = 0x7fffffff, ihi = 0x7fffffff;
            for (int i = first + lane; i <= last; i += 32) {
                const double v = r.sx[i];
                if (v < lo) { lo = v; ilo = i; }
                if (v > hi) { hi = v; ihi = i; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double olo = shfl_d(lo, lane ^ o), ohi = shfl_d(hi, lane ^ o);
                const int oilo = __shfl_xor_sync(FULL, ilo, o), oihi = __shfl_xor_sync(FULL, ihi, o);
                if (olo < lo || (olo == lo && oilo < ilo)) { lo = olo; ilo = oilo; }
                if (ohi > hi || (ohi == hi && oihi < ihi)) { hi = ohi; ihi = oihi; }
            }
            if (lane == 0) { s_bmin[b] = lo; s_bmax[b] = hi; s_amin[b] = ilo; s_amax[b] = ihi; }
        }
        __syncthreads();
        // global extrema: first block that attains them, only if below / above 0.0 (CBS.cpp:619-620, 634-635)
        if (warp == 0) {
            double lo = __longlong_as_double(0x7ff0000000000000LL), hi = -lo;
            int blo = 0x7fffffff, bhi = 0x7fffffff;
            for (int b = lane; b < nb; b += 32) {
                if (s_bmin[b] < lo) { lo = s_bmin[b]; blo = b; }
                if (s_bmax[b] > hi) { hi = s_bmax[b]; bhi = b; }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double olo = shfl_d(lo, lane ^ o), ohi = shfl_d(hi, lane ^ o);
                const int oblo = __shfl_xor_sync(FULL, blo, o), obhi = __shfl_xor_sync(FULL, bhi, o);
                if (olo < lo || (olo == lo && oblo < blo)) { lo = olo; blo = oblo; }
                if (ohi > hi || (ohi == hi && obhi < bhi)) { hi = ohi; bhi = obhi; }
            }
            if (lane == 0) {
                const bool below = lo < 0.0, above = hi > 0.0;
                sm->g_min = below ? lo : 0.0; sm->g_imin = below ? s_amin[blo] : n;
                sm->g_max = above ? hi : 0.0; sm->g_imax = above ? s_amax[bhi] : n;
            }
        }
        __syncthreads();
        const double psdiff = sm->g_max - sm->g_min;
        const int gimin = sm->g_imin, gimax = sm->g_imax;
        const int fi = min(gimax, gimin), fj = max(gimax, gimin);
        const double rn = (double)n;
        double best = 0.0;
        bool decided = false;
        if (MODE == 1 && slice == 0) {
            // strictly increasing, finite cw <=> every arc weight a and psrn - a is positive, so no arc statistic of this
            // segment can be inf or NaN: the precondition of the early reject decision of its permutations (an inf
            // statistic makes the reference's pstat NaN, which never rejects)
            int bad = 0;
            for (int i = tid; i < n; i += blockDim.x) {
                const double ci = r.cw[i], cp = i ? r.cw[i - 1] : 0.0;
                if (!(ci > cp) || isinf(ci)) bad = 1;
            }
            bad = __syncthreads_or(bad);
            // location: the seed arc unless MODE 2 finds better; without spread the reference reports it unshifted (:642-645)
            if (tid == 0) { t.w_ok = bad ? 0 : 1; t.tmaxi = psdiff > 0.0 ? fi : fi + 1; t.tmaxj = psdiff > 0.0 ? fj : fj + 1; }
        }
        if (psdiff > 0.0) {  // else CBS.cpp:642-645
            r.psrn = r.cw[n - 1];
            r.psrnov2 = r.psrn / 2.0;
            const double psrj = fabs(r.cw[gimax - 1] - r.cw[gimin - 1]);
            r.init = (psdiff * psdiff) / (psrj * (r.psrn - psrj));  // :649
            const unsigned long long init_bits = (unsigned long long)__double_as_longlong(r.init);
            __syncthreads();
            if (tid == 0) {
                double level = r.init;
                if (MODE == 0) {
                    // decision mode: reject <=> thresh <= f(M), f(M) = M/(((M+1)-M)/(n-2)) ~ M(n-2) (tss = 0 makes the
                    // reference replace tss by M+1); M* sits 1e-9 below the solution, f(M*) < thresh is verified
                    const double thresh = t.ostat * 0.99999;
                    const double mstar = thresh / (rn - 2.0) * (1.0 - 1e-9);
                    if (mstar > level) {
                        const double f = mstar / (((mstar + 1.0) - mstar) / (rn - 2.0));
                        if (f < thresh) level = mstar;
                    }
                }
                sm->decided = 0;
                sm->rej_at = __longlong_as_double(0x7ff0000000000000LL);
                if (MODE == 0 && !D->no_early && t.w_ok && r.init < 1e300) {  // (init is inf when the seed arc is empty)
                    // early decision: f(M) = M(n-2)(1 +- (M+1) 2^-52) is increasing up to that wobble, so any arc with
                    // M >= rej_at = thresh/(n-2) (1+1e-9) settles "reject" whatever the maximum turns out to be
                    const double thresh = t.ostat * 0.99999;
                    const double ra = thresh / (rn - 2.0) * (1.0 + 1e-9);
                    const double f = ra / (((ra + 1.0) - ra) / (rn - 2.0));
                    if (ra < 1e5 && f >= thresh * (1.0 + 5e-10)) {
                        sm->rej_at = ra;
                        if (r.init >= ra) sm->decided = 1;
                    }
                }
                sm->glevel = r.glevel; sm->gfound = r.gfound;
                if (MODE == 1) {  // the seed arc counts for every slice; then join the level the other slices reached
                    atomicMax(&t.w_found, init_bits);
                    atomicMax(&t.w_level, init_bits);
                    if (slice == 0) t.w_init = r.init;
                    const double gl = __longlong_as_double((long long)*((volatile unsigned long long*)&t.w_level));
                    if (gl > level) level = gl;
                }
                sm->level = (unsigned long long)__double_as_longlong(level);
                sm->found = init_bits;
                sm->next_pair = r.q_first; sm->lock = 0; sm->r_set = 0; sm->tie = 0;
                sm->r_corner = 0.0; sm->r_q = 0; sm->r_phase = 0; sm->r_o1 = 0; sm->r_o2 = 0; sm->r_i = 0; sm->r_j = 0;
            }
            __syncthreads();
            if (MODE == 1) {
                wscan_pass<true>(r, sm, lane);
                __syncthreads();
                if (tid == 0 && sm->r_set) {  // this CTA's best arc into the row's record
                    WCand mine{sm->r_corner, sm->r_q, sm->r_phase, sm->r_o1, sm->r_o2, sm->r_i, sm->r_j, true, sm->r_v};
                    while (atomicCAS(&t.w_lock, 0, 1) != 0) {}
                    __threadfence();
                    const volatile Task& vt = t;
                    WCand cur{vt.w_corner, vt.w_q, vt.w_phase, vt.w_o1, vt.w_o2, vt.w_i, vt.w_j, vt.w_set != 0, vt.w_v};
                    if (sm->tie || wcand_tied(mine, cur)) t.w_tie = 1;
                    if (wcand_better(mine, cur)) {
                        t.w_v = mine.v; t.w_corner = mine.corner; t.w_q = mine.q; t.w_phase = mine.phase; t.w_o1 = mine.o1;
                        t.w_o2 = mine.o2; t.w_i = mine.i; t.w_j = mine.j; t.w_set = 1;
                    }
                    __threadfence();
                    atomicExch(&t.w_lock, 0);
                }
            } else {
                if (!sm->decided) wscan_pass<false>(r, sm, lane);
                __syncthreads();
                best = __longlong_as_double((long long)sm->found);
                decided = sm->decided != 0;
            }
        }
        if (MODE == 0 && tid == 0) {
            double tss = 0.0;  // wtmaxp passes tss = 0.0 (CBS.cpp:741-743): mirrored, not "fixed"
            if (tss <= best + 0.0001) tss = best + 1.0;  // CBS.cpp:643,737
            const double stat = best / ((tss - best) / (rn - 2.0));
            if (it.obs == 2) t.ostat = stat;
            else D->rej[t.off_rej + p] = (decided || t.ostat * 0.99999 <= stat) ? 1 : 0;  // CBS.cpp:900,933
        }
    }
}

// cbs::wtmaxo (CBS.cpp:610-739) walked in the reference's own order by one warp: lane 0 runs the control flow (block extrema,
// pair list, std::sort order of the corner statistics, descending visit with the running maximum), the lanes share the inner
// loop over j.  Only used for an observed row whose maximum is attained in pairs with equal corner statistics (structured
// data: constant stretches, periodic signals), where the location depends on std::sort's treatment of equal keys.
__device__ void wtmaxo_ordered(const double* __restrict__ sx, const double* __restrict__ cw, const int* __restrict__ bb, int n, int nb,
                               int al0, double* scratch, int lane, double& bss_out, int& ti_out, int& tj_out) {
    const int nb2 = nb * (nb + 1) / 2;
    double* bpsmax = scratch;
    double* bpsmin = bpsmax + nb + 1;
    double* bssbij = bpsmin + nb + 1;
    double* bssijmax = bssbij + nb2 + 1;
    double* awt = bssijmax + nb2 + 1;
    int* ibmin = (int*)(awt + nb2 + 1);
    int* ibmax = ibmin + nb + 1;
    int* bloc = ibmax + nb + 1;   // (i << 16) | j
    int* loc = bloc + nb2 + 1;
    double psmin0 = 0.0, psmax0 = 0.0;
    int ipsmin0 = n, ipsmax0 = n;
    if (lane == 0) {  // :621-637 from the prefix sums that k_wprep wrote
        for (int j = 1; j <= nb; ++j) {
            const int ilo = bb[j - 1] + 1;
            double psmin = sx[ilo], psmax = sx[ilo];
            int ipsmin = ilo, ipsmax = ilo;
            for (int i = ilo + 1; i <= bb[j]; ++i) {
                if (sx[i] < psmin) { psmin = sx[i]; ipsmin = i; }
                if (sx[i] > psmax) { psmax = sx[i]; ipsmax = i; }
            }
            ibmin[j] = ipsmin; ibmax[j] = ipsmax; bpsmin[j] = psmin; bpsmax[j] = psmax;
            if (psmin < psmin0) { psmin0 = psmin; ipsmin0 = ipsmin; }
            if (psmax > psmax0) { psmax0 = psmax; ipsmax0 = ipsmax; }
        }
    }
    __syncwarp();
    psmin0 = shfl_d(psmin0, 0); psmax0 = shfl_d(psmax0, 0);
    ipsmin0 = __shfl_sync(FULL, ipsmin0, 0); ipsmax0 = __shfl_sync(FULL, ipsmax0, 0);
    double bssmax = 0.0;
    int tmaxi = min(ipsmax0, ipsmin0), tmaxj = max(ipsmax0, ipsmin0);
    const double psdiff = psmax0 - psmin0;
    if (psdiff <= 0.0) { bss_out = 0.0; ti_out = tmaxi; tj_out = tmaxj; return; }
    const double psrn = cw[n - 1];
    {
        const double psrj = fabs(cw[ipsmax0 - 1] - cw[ipsmin0 - 1]);
        bssmax = (psdiff * psdiff) / (psrj * (psrn - psrj));
    }
    const double psrnov2 = psrn / 2.0;
    const int nal0 = n - al0;
    int l = 0;
    for (int i = 1; i <= nb; ++i) {  // :650-693, the list keeps the (i, j) order (ballot compaction)
        for (int j0 = i; j0 <= nb; j0 += 32) {
            const int j = j0 + lane;
            bool take = false;
            double e_lim = 0.0, e_bij = 0.0, e_awt = 0.0;
            if (j <= nb) {
                const int ilo1 = (i == 1) ? 1 : bb[i - 1] + 1, ihi = bb[i];
                const int jlo = (j == 1) ? 1 : bb[j - 1] + 1, jhi = bb[j];
                double awthi = cw[jhi - 1] - cw[ilo1 - 1];
                if (jhi - ilo1 > nal0) {
                    awthi = 0.0;
                    for (int kk = 1; kk <= al0; ++kk) awthi = fmax(awthi, cw[nal0 + kk - 1] - cw[kk - 1]);
                }
                double awtlo;
                if (i == j) {
                    awtlo = cw[ilo1 + al0 - 1] - cw[ilo1 - 1];
                    for (int kk = ilo1 + 1; kk <= ihi - al0; ++kk) awtlo = fmin(awtlo, cw[kk + al0 - 1] - cw[kk - 1]);
                } else if (i + 1 == j) {
                    awtlo = cw[jlo - 1] - cw[jlo - al0 - 1];
                    for (int kk = jlo - al0 + 1; kk <= ihi; ++kk) awtlo = fmin(awtlo, cw[kk + al0 - 1] - cw[kk - 1]);
                } else awtlo = cw[jlo - 1] - cw[ihi - 1];
                const double sij1 = fabs(bpsmax[j] - bpsmin[i]), sij2 = fabs(bpsmax[i] - bpsmin[j]);
                const double sijmx0 = fmax(sij1, sij2);
                const double bsslim = (sijmx0 * sijmx0) / fmin(awtlo * (psrn - awtlo), awthi * (psrn - awthi));
                if (bssmax <= bsslim) {
                    take = true; e_lim = bsslim;
                    if (sij1 > sij2) { e_awt = fabs(cw[ibmax[j] - 1] - cw[ibmin[i] - 1]); e_bij = (sij1 * sij1) / (e_awt * (psrn - e_awt)); }
                    else { e_awt = fabs(cw[ibmin[j] - 1] - cw[ibmax[i] - 1]); e_bij = (sij2 * sij2) / (e_awt * (psrn - e_awt)); }
                }
            }
            const unsigned mask = __ballot_sync(FULL, take);
            if (take) {
                const int pos = l + 1 + __popc(mask & ((1u << lane) - 1u));
                loc[pos] = pos; bloc[pos] = (i << 16) | j; bssijmax[pos] = e_lim; awt[pos] = e_awt; bssbij[pos] = e_bij;
            }
            l += __popc(mask);
        }
    }
    const int nb1 = l;
    __syncwarp();
    if (lane == 0) { IdxSort srt{loc + 1, bssbij}; srt.run(nb1); }
    __syncwarp();
    for (int ll = nb1; ll >= 1; --ll) {  // :698-735
        const int k = loc[ll];
        if (bssmax > bssijmax[k]) continue;
        const int bi = bloc[k] >> 16, bj = bloc[k] & 0xffff;
        double awtmax = awt[k];
        const int ilo1 = (bi == 1) ? 1 : bb[bi - 1] + 1, ihi = bb[bi];
        const int jlo = (bj == 1) ? 1 : bb[bj - 1] + 1, jhi = bb[bj];
        const double awthi = cw[jhi - 1] - cw[ilo1 - 1];
        const double awtlo = (bi == bj) ? 0.0 : (cw[jlo - 1] - cw[ihi - 1]);
        if (awtmax > psrn - awtmax) awtmax = psrn - awtmax;
        if (awtlo <= psrnov2) {
            const int ihi1 = (bi == bj) ? ihi - al0 : ihi;
            for (int i = ihi1; i >= ilo1; --i) {
                const int jlo1 = max(i + al0, jlo);
                double rv = -1.0;
                int rj = 0x7fffffff;
                for (int j = jlo1 + lane; j <= jhi; j += 32) {  // ascending j: the first j that attains the row's maximum counts
                    const double awt1 = cw[j - 1] - cw[i - 1];
                    if (awt1 <= awtmax) {
                        const double d = sx[j] - sx[i];
                        const double v = (d * d) / (awt1 * (psrn - awt1));
                        if (v > rv) { rv = v; rj = j; }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = shfl_d(rv, lane ^ o);
                    const int oj = __shfl_xor_sync(FULL, rj, o);
                    if (ov > rv || (ov == rv && oj < rj)) { rv = ov; rj = oj; }
                }
                if (rv > bssmax) { bssmax = rv; tmaxi = i; tmaxj = rj; }
            }
        }
        awtmax = psrn - awtmax;
        if (awthi >= psrnov2) {
            for (int i = ilo1; i <= ihi; ++i) {
                const int jhi1 = ((bi == 1) && (bj == nb)) ? min(jhi, jhi - al0 + i) : jhi;
                double rv = -1.0;
                int rj = -1;
                for (int j = jhi1 - lane; j >= jlo; j -= 32) {  // descending j: the LARGEST j among equal maxima is met first
                    const double awt1 = cw[j - 1] - cw[i - 1];
                    if (awt1 >= awtmax) {
                        const double d = sx[j] - sx[i];
                        const double v = (d * d) / (awt1 * (psrn - awt1));
                        if (v > rv) { rv = v; rj = j; }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ov = shfl_d(rv, lane ^ o);
                    const int oj = __shfl_xor_sync(FULL, rj, o);
                    if (ov > rv || (ov == rv && oj > rj)) { rv = ov; rj = oj; }
                }
                if (rv > bssmax) { bssmax = rv; tmaxi = i; tmaxj = rj; }
            }
        }
    }
    bss_out = bssmax; ti_out = tmaxi; tj_out = tmaxj;
}

// observed rows: statistic and location from the shared records (after k_wscan<1> and k_wscan<2>); a warp per row
__global__ void k_wobs_fin(Dev* D) {
    if (D->done) return;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int k = warp; k < D->n_items; k += nwarps) {
        const PermItem it = D->items[k];
        if (it.obs != 1) continue;
        Task& t = D->tasks[it.task];
        if (t.alleq) continue;
        const double best = __longlong_as_double((long long)t.w_found);  // 0.0 when the prefix sums have no spread
        int ti = t.tmaxi, tj = t.tmaxj;
        // the seed arc is visited first and wins ties; otherwise the first-visited arc that attains the maximum
        if (t.w_set && t.w_v == best && best > t.w_init) { ti = t.w_i; tj = t.w_j; }
        if (t.w_tie && t.off_A >= 0) {  // equal corner statistics and equal maxima: take the location from the reference's own walk
            const long long base = D->unit_off[t.unit] + t.lo;
            double b2;
            int i2, j2;
            wtmaxo_ordered(D->arena + t.off_sx, D->cw + base, D->bbtab + base, t.n, t.nb, D->prm.min_width, D->arena + t.off_A, lane, b2, i2, j2);
            if (b2 == best) { ti = i2; tj = j2; }
        }
        if (lane == 0) {
            double tss = t.tss;
            if (tss <= best + 0.0001) tss = best + 1.0;  // CBS.cpp:643,737
            t.ostat = best / ((tss - best) / ((double)t.n - 2.0));
            t.tmaxi = ti; t.tmaxj = tj;
        }
    }
}

// ------------------------------------------------------------------------------------
// weighted hybrid method (wfindcpt :908-921): delta from the weights (getmncwt :593-608), hwtmaxp (:745-828)
//   k_wdelta  per new segment: smallest weight of an arc of kmax+1 markers (wrap-around arcs included) / total weight;
//             k_tailp_* then evaluate the tail probability with it
//   k_wssq    per permutation row, BEFORE the chain turns the row into prefix sums: ssq = sum w*px*px, sequential (:757,762)
//   k_whscan  hwtmaxp for one permutation per CTA.  Its pruning (lengths are abandoned once the bound from mncwt drops
//             below the running maximum) only skips arcs that cannot exceed the maximum, so the value is the maximum of
//             d^2/(a(W-a)) over ALL arcs of al0..k markers, wrap-around arcs included; evaluated by brute force like
//             k_hscan, with the division only for arcs that can raise the thread's maximum.  mncwt itself is not needed.
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_wdelta(Dev* D) {
    if (D->done || !D->prm.hybrid) return;
    const int lane = threadIdx.x;
    for (int k = blockIdx.x; k < D->n_prep; k += gridDim.x) {
        Task& t = D->tasks[D->prep_task[k]];
        if (!t.use_hybrid || t.alleq) continue;
        const double* __restrict__ cw = D->cw + D->unit_off[t.unit] + t.lo;
        const int n = t.n, len = D->prm.kmax + 1, rest = n - len;
        if (rest < 1) { if (lane == 0) t.w_delta = 0.5; continue; }
        const double total = cw[n - 1];
        double m = cw[len - 1];
        for (int i = 1 + lane; i <= rest; i += 32) m = fmin(m, cw[i + len - 1] - cw[i - 1]);
        for (int i = 1 + lane; i <= len; i += 32) m = fmin(m, total - (cw[i + rest - 1] - cw[i - 1]));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m = fmin(m, shfl_d(m, lane ^ o));
        if (lane == 0) t.w_delta = m / total;
    }
}

__global__ void __launch_bounds__(128) k_wssq(Dev* D) {
    __shared__ __align__(16) double buf_all[4][WPREP_CHUNK];
    if (D->done || !D->prm.hybrid) return;
    const int lane = threadIdx.x & 31;
    double* __restrict__ buf = buf_all[threadIdx.x >> 5];
    const int total = D->item_prefix[D->n_items];
    for (;;) {
        int g = 0;
        if (lane == 0) g = (int)atomicAdd(&D->ctr[7], 1u);
        g = __shfl_sync(FULL, g, 0);
        if (g >= total) break;
        const int k = find_item(D->item_prefix, D->n_items, g);
        const PermItem it = D->items[k];
        const Task& t = D->tasks[it.task];
        if (it.obs || !t.use_hybrid) continue;
        const int p = g - D->item_prefix[k], n = t.n;
        const double* __restrict__ px = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n) + 1;
        const double* __restrict__ w = D->w + D->unit_off[t.unit] + t.lo;
        double ssq = 0.0;
        for (int c0 = 0; c0 < n; c0 += WPREP_CHUNK) {
            const int cnt = min(WPREP_CHUNK, n - c0);
            double v[WPREP_Q];
#pragma unroll
            for (int q = 0; q < WPREP_Q; ++q) {
                const int kk = lane + 32 * q;
                const double a = (kk < cnt) ? px[c0 + kk] : 0.0, ww = (kk < cnt) ? w[c0 + kk] : 0.0;
                v[q] = ww * a * a;
            }
            __syncwarp();
#pragma unroll
            for (int q = 0; q < WPREP_Q; ++q) buf[lane + 32 * q] = v[q];
            __syncwarp();
            if (lane == 0) {
                int kk = 0;
                for (; kk + 8 <= cnt; kk += 8) {
                    double a[8];
#pragma unroll
                    for (int u = 0; u < 8; u += 2) { const double2 va = *reinterpret_cast<const double2*>(buf + kk + u); a[u] = va.x; a[u + 1] = va.y; }
#pragma unroll
                    for (int u = 0; u < 8; ++u) ssq = ssq + a[u];
                }
                for (; kk < cnt; ++kk) ssq = ssq + buf[kk];
            }
        }
        if (lane == 0) BlockStats(D->arena + t.off_bs + (long long)p * Sched::bs_stride(t.nb), t.nb).result() = ssq;
        __syncwarp();
    }
}

__global__ void __launch_bounds__(256) k_whscan(Dev* D) {
    __shared__ double s_red[8];
    __shared__ int s_g;
    if (D->done || !D->prm.hybrid) return;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int total = D->item_prefix[D->n_items];
    const int kk = D->prm.kmax, al0 = D->prm.min_width;
    for (;;) {
        __syncthreads();
        if (tid == 0) s_g = (int)atomicAdd(&D->ctr[4], 1u);
        __syncthreads();
        const int gidx = s_g;
        if (gidx >= total) break;
        const int it_k = find_item(D->item_prefix, D->n_items, gidx);
        const PermItem it = D->items[it_k];
        Task& t = D->tasks[it.task];
        if (it.obs || !t.use_hybrid) continue;
        const int p = gidx - D->item_prefix[it_k];
        const int n = t.n;
        const double* __restrict__ sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        const double* __restrict__ cw = D->cw + D->unit_off[t.unit] + t.lo;
        const double W = cw[n - 1];
        double best = 0.0;
        for (int i = 1 + tid; i <= n; i += blockDim.x) {
            const double si = sx[i], ci = cw[i - 1];
            for (int j = al0; j <= kk; ++j) {  // arcs (i, i+j) (:763-775, :795-805)
                const int e = i + j;
                if (e > n) break;
                const double d = sx[e] - si, a = cw[e - 1] - ci;
                const double d2 = d * d, den = a * (W - a);
                if (d2 > best * den * (1.0 - 1e-12)) { const double v = d2 / den; if (v > best) best = v; }
            }
            for (int j = (i > al0 ? i : al0); j <= kk; ++j) {  // wrap-around arcs: i <= j, against i+n-j (:780-790)
                const int e = i + n - j;
                const double d = sx[e] - si, a = cw[e - 1] - ci;
                const double d2 = d * d, den = a * (W - a);
                if (d2 > best * den * (1.0 - 1e-12)) { const double v = d2 / den; if (v > best) best = v; }
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const double o2 = shfl_d(best, lane ^ o); if (o2 > best) best = o2; }
        if (lane == 0) s_red[warp] = best;
        __syncthreads();
        if (tid == 0) {
            double m = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) if (s_red[w] > m) m = s_red[w];
            const double ssq = BlockStats(D->arena + t.off_bs + (long long)p * Sched::bs_stride(t.nb), t.nb).result();
            const double mean = sx[n] / W;
            double tss = ssq - mean * mean;  // :776
            if (tss <= m + 0.0001) tss = m + 1.0;
            const double stat = m / ((tss - m) / ((double)n - 2.0));
            D->rej[t.off_rej + p] = (t.ostat * 0.99999 <= stat) ? 1 : 0;
        }
    }
}

// ------------------------------------------------------------------------------------
// wtpermp (CBS.cpp:549-591)
// ------------------------------------------------------------------------------------
__device__ void wedgeprep_warp(Dev* D, Task& t, int s, int lane, double* bx, double* bw) {
    const int n1 = t.e_n1[s], n2 = t.e_n2[s], n = n1 + n2;
    const long long base = D->unit_off[t.unit] + t.lo + t.e_off[s];
    const double* __restrict__ x = D->cur + base;
    const double* __restrict__ w = D->w + base;
    if (n1 == 1 || n2 == 1) { if (lane == 0) { t.e_status[s] = 1; t.e_m1[s] = 0; t.e_nrej[s] = 0; } return; }
    double xsum1 = 0.0, xsum2 = 0.0, tss = 0.0, rn1 = 0.0, rn2 = 0.0;  // :553-565, one chain across both sides for tss
    for (int c0 = 0; c0 < n; c0 += WPREP_CHUNK) {
        const int cnt = min(WPREP_CHUNK, n - c0);
        __syncwarp();
        for (int k = lane; k < cnt; k += 32) { bx[k] = x[c0 + k]; bw[k] = w[c0 + k]; }
        __syncwarp();
        if (lane == 0)
            for (int k = 0; k < cnt; ++k) {
                const double v = bx[k], ww = bw[k];
                if (c0 + k < n1) { xsum1 = xsum1 + ww * v; tss = tss + ww * v * v; rn1 = rn1 + ww; }
                else { xsum2 = xsum2 + ww * v; tss = tss + ww * v * v; rn2 = rn2 + ww; }
            }
    }
    if (lane == 0) {
        t.e_nrej[s] = 0;
        const double rn = rn1 + rn2;
        const double xbar = (xsum1 + xsum2) / rn;
        tss -= rn * (xbar * xbar);
        int m1; double rm1, ostat, tstat;
        if (n1 <= n2) { m1 = n1; rm1 = rn1; ostat = 0.99999 * fabs(xsum1 / rn1 - xbar); tstat = (ostat * ostat) * rn1 * rn / rn2; }
        else          { m1 = n2; rm1 = rn2; ostat = 0.99999 * fabs(xsum2 / rn2 - xbar); tstat = (ostat * ostat) * rn2 * rn / rn1; }
        tstat /= ((tss - tstat) / ((double)n - 2.0));
        t.e_m1[s] = m1; t.e_rm1[s] = rm1; t.e_ostat[s] = ostat; t.e_xbar[s] = xbar;
        t.e_status[s] = (tstat > 25.0 && m1 >= 10) ? 2 : 0;
    }
}

__global__ void __launch_bounds__(32) k_wedgeprep(Dev* D) {
    __shared__ __align__(16) double bx[WPREP_CHUNK];
    __shared__ __align__(16) double bw[WPREP_CHUNK];
    if (D->done) return;
    for (int k = blockIdx.x; k < 2 * D->n_edgeprep; k += gridDim.x)
        wedgeprep_warp(D, D->tasks[D->edgeprep_task[k >> 1]], k & 1, threadIdx.x, bx, bw);
}

// value at position k before any swap (CBS.cpp:574-575): x*rw on the left side, x on the right
__device__ __forceinline__ double wedge_src(const double* x, const double* rw, int n1, int k) {
    return (k < n1) ? x[k] * rw[k] : x[k];
}

// m1 <= 64: override list in local memory (see edge_sparse_thread)
__device__ int wedge_sparse_thread(const Dev& D, const Task& t, const EdgeItem& e, int r) {
    const int s = e.side, m1 = t.e_m1[s], n1 = t.e_n1[s], n = n1 + t.e_n2[s];
    const long long base = D.unit_off[t.unit] + t.lo + t.e_off[s];
    const double* x = D.cur + base;
    const double* rw = D.rw + base;
    DrawSrc src;
    edge_draw_src(D, t, e, r, src);
    int okey[64];
    double oval[64];
    int cnt = 0;
    double acc = 0.0;
    uint32_t kd = 0;
    for (int i = n; i >= n - m1 + 1; --i) {
        const int j = draw_index(src.u64(kd++), i);
        double vi = wedge_src(x, rw, n1, i - 1);
        for (int q = 0; q < cnt; ++q) if (okey[q] == i - 1) vi = oval[q];
        double vj;
        int slot = -1;
        if (j == i) vj = vi;
        else {
            vj = wedge_src(x, rw, n1, j - 1);
            for (int q = 0; q < cnt; ++q) if (okey[q] == j - 1) { vj = oval[q]; slot = q; }
            if (slot < 0) { slot = cnt++; okey[slot] = j - 1; }
            oval[slot] = vi;
        }
        acc += vj * rw[i - 1];  // :580
    }
    const double pstat = fabs(acc / t.e_rm1[s] - t.e_xbar[s]);
    return t.e_ostat[s] <= pstat ? 1 : 0;
}

// general case: scratch column with undo (see edge_general_thread)
__device__ int wedge_general_thread(const Dev& D, const Task& t, const EdgeItem& e, int c) {
    const int s = e.side, m1 = t.e_m1[s], n1 = t.e_n1[s], n = n1 + t.e_n2[s];
    const long long base = D.unit_off[t.unit] + t.lo + t.e_off[s];
    const double* x = D.cur + base;
    const double* rw = D.rw + base;
    double* A = D.arena + e.off_scratch;
    const long long C = e.cols;
    for (int k = 0; k < n; ++k) A[(long long)k * C + c] = wedge_src(x, rw, n1, k);
    int rejections = 0;
    for (int q = 0; q < e.Q; ++q) {
        const int r = c + q * e.cols;
        if (r >= e.P) break;
        DrawSrc src;
        edge_draw_src(D, t, e, r, src);
        double acc = 0.0;
        uint32_t kd = 0;
        for (int i = n; i >= n - m1 + 1; --i) {
            const int j = draw_index(src.u64(kd++), i);
            const double a = A[(long long)(i - 1) * C + c], b = A[(long long)(j - 1) * C + c];
            A[(long long)(i - 1) * C + c] = b;
            A[(long long)(j - 1) * C + c] = a;
            acc += b * rw[i - 1];
        }
        const double pstat = fabs(acc / t.e_rm1[s] - t.e_xbar[s]);
        if (t.e_ostat[s] <= pstat) ++rejections;
        if (q + 1 < e.Q && r + e.cols < e.P) {
            for (int i = n - m1 + 1; i <= n; ++i) {  // undo, last swap first
                const int j = draw_index(src.u64((uint32_t)(n - i)), i);
                const double a = A[(long long)(i - 1) * C + c], b = A[(long long)(j - 1) * C + c];
                A[(long long)(i - 1) * C + c] = b;
                A[(long long)(j - 1) * C + c] = a;
            }
        }
    }
    return rejections;
}

__global__ void __launch_bounds__(128) k_wedgeperm(Dev* D) {
    if (D->done) return;
    __shared__ int s_base;
    const int total = D->edge_prefix[D->n_edge];
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_base = (int)atomicAdd(&D->ctr[2], (unsigned)blockDim.x);
        __syncthreads();
        const int g = s_base + threadIdx.x;
        if (s_base >= total) break;
        if (g >= total) continue;
        const int k = find_item(D->edge_prefix, D->n_edge, g);
        const EdgeItem e = D->edges[k];
        Task& t = D->tasks[e.task];
        const int th = g - D->edge_prefix[k];
        const int r = e.sparse ? wedge_sparse_thread(*D, t, e, th) : wedge_general_thread(*D, t, e, th);
        if (r) atomicAdd(&t.e_nrej[e.side], r);
    }
}

// weighted mean of every final segment (CBS.cpp:1091-1097), sequential sums
__global__ void __launch_bounds__(32) k_wmeans(const Dev* D, double* means) {
    __shared__ __align__(16) double bx[WPREP_CHUNK];
    __shared__ __align__(16) double bw[WPREP_CHUNK];
    const int lane = threadIdx.x;
    for (int k = blockIdx.x; k < D->n_segs; k += gridDim.x) {
        const SegRec sg = D->segs[k];
        const long long base = D->unit_off[sg.unit] + sg.lo;
        const double* __restrict__ x = D->x + base;
        const double* __restrict__ w = D->w + base;
        const int n = sg.hi - sg.lo;
        double sw = 0.0, swx = 0.0;
        for (int c0 = 0; c0 < n; c0 += WPREP_CHUNK) {
            const int cnt = min(WPREP_CHUNK, n - c0);
            __syncwarp();
            for (int q = lane; q < cnt; q += 32) { bx[q] = x[c0 + q]; bw[q] = w[c0 + q]; }
            __syncwarp();
            if (lane == 0)
                for (int q = 0; q < cnt; ++q) { sw = sw + bw[q]; swx = swx + bw[q] * bx[q]; }
        }
        if (lane == 0) means[k] = swx / sw;
        __syncwarp();
    }
}

}  // namespace cbsg
