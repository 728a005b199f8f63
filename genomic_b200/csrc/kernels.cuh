// kernels.cuh -- sm_100a kernels of the CBS hot path.
//
//   k_sched          count phase + the single-thread worklist scheduler (cbs_core.h); holds the loop condition of the
//                    call graph (cbs_gpu.cu run_cbs: one scheduler round = the body of a WHILE node)
//   k_gen_lead/par   MT19937-64 raw stream, one shared ring for all units, extended in parallel with jump-ahead
//                    polynomials (mt_jump.h); k_gen: one CTA per chain when ONE engine is shared serially (chain mode)
//   k_tables, k_prep per new pending segment: block ends, g[L] and fac[L]; all-equal test, mean, centring, tss and the
//                    observed prefix sums as lane-0 chains                              (CBS.cpp:985-989, :71-97)
//   k_shuffle, k_shuffle_cluster   xperm as an exact parallel Fisher-Yates, CTA or thread-block cluster per permutation
//                    (shuffle.cuh; CBS.cpp:487-493); k_perm: fallback with index arrays in L2 for units no cluster holds
//   k_chain          prefix sums of the permuted rows (one dependent DADD chain per row) + the row statistics the scan
//                    prunes with                                                          (CBS.cpp:83-94)
//   k_scan_perm      CTA per permutation: branch-and-bound max-t arc scan, reject decision (CBS.cpp:99-224)
//   k_scan_obs       the same scan of the observed rows, up to 24 CTAs per row: maximum and location
//   k_hscan, k_tailp_*   hybrid p-values: htmaxp (CBS.cpp:387-485) and tailp (:324-339)
//   k_edgeprep       tpermp set-up sums (CBS.cpp:496-522)
//   k_edgeperm       tpermp permutation loop (CBS.cpp:524-534)
//   k_means          segment means (CBS.cpp:1014-1022)
//   (binary.cuh: the ibin = true scan, btmax; weighted.cuh: the weighted variants; smooth.cuh: smoothing, summarize_cn)
//
// All floating point that feeds a comparison is plain IEEE double with the reference's
// operation order; the library is compiled with -fmad=false.
#pragma once
#include <cuda_runtime.h>

#include "cbs_threads.h"
#include "shuffle.cuh"

namespace cbsg {

#define FULL 0xffffffffu

// ------------------------------------------------------------------------------------
// small device helpers
// ------------------------------------------------------------------------------------
__device__ __forceinline__ double shfl_d(double v, int src) { return __shfl_sync(FULL, v, src); }

__device__ __forceinline__ void atomic_max_pos_double(double* addr, double v) {
    // non-negative doubles order like their bit patterns
    atomicMax((unsigned long long*)addr, (unsigned long long)__double_as_longlong(v));
}

// order-preserving map between doubles and signed 64-bit integers (its own inverse on the bit pattern)
__device__ __forceinline__ long long dkey(double v) {
    const long long b = __double_as_longlong(v);
    return b ^ ((b >> 63) & 0x7fffffffffffffffLL);
}
__device__ __forceinline__ double dunkey(long long k) { return __longlong_as_double(k ^ ((k >> 63) & 0x7fffffffffffffffLL)); }

// map a global work index to (item, offset) through an exclusive prefix array
__device__ __forceinline__ int find_item(const int* prefix, int n_items, int g) {
    int lo = 0, hi = n_items;  // prefix[lo] <= g < prefix[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (prefix[mid] <= g) lo = mid; else hi = mid;
    }
    return lo;
}

// ------------------------------------------------------------------------------------
// k_sched
// ------------------------------------------------------------------------------------
__device__ void count_item_warp(Dev* D, const PermItem& it, int lane) {
    if (it.obs) return;
    Task& t = D->tasks[it.task];
    const int* rej = D->rej + t.off_rej;
    const int P = it.P, base = t.nrej, nrejc = t.nrejc;
    int running = 0, hit = -1;
    for (int p0 = 0; p0 < P; p0 += 32) {
        const int f = (p0 + lane < P) ? rej[p0 + lane] : 0;
        const unsigned mask = __ballot_sync(FULL, f != 0);
        const int incl = __popc(mask & (0xffffffffu >> (31 - lane)));
        const unsigned over = __ballot_sync(FULL, f != 0 && base + running + incl > nrejc);
        if (over) {
            const int l = __ffs(over) - 1;
            hit = p0 + l;
            running += __popc(mask & (0xffffffffu >> (31 - l)));
            break;
        }
        running += __popc(mask);
    }
    if (lane == 0) { t.cnt_exit = hit; t.cnt_nrej = running; }
}

// `looped`: the round is the body of a WHILE node of a CUDA graph (cbs_gpu.cu run_cbs) and `loop` its condition: the
// scheduler keeps it at 1 until the work list is empty (or an error is raised), so the whole call is one graph launch.
__global__ void __launch_bounds__(256) k_sched(Dev* D, volatile int* host_done, cudaGraphConditionalHandle loop, int looped) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (D->done) {
        if (looped && threadIdx.x == 0) cudaGraphSetConditional(loop, 0);
        return;
    }
    for (int k = warp; k < D->n_items; k += 8) count_item_warp(D, D->items[k], lane);
    __syncthreads();
    if (threadIdx.x == 0) {
        Sched S(*D);
        S.run_round();
        if (D->done) { __threadfence_system(); *host_done = D->error ? -D->error : 1; }
        if (looped) cudaGraphSetConditional(loop, D->done ? 0u : 1u);
    }
}

// ------------------------------------------------------------------------------------
// k_gen: one CTA per chain. hist = the next 312 raw words of the chain's engine.  Commit the
// words consumed from last round's window, then write this round's window: the 312 known
// words followed by need_len further words of the recurrence (4 barriers per 312 words).
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(192) k_gen(Dev* D) {
    __shared__ uint64_t st[312];
    if (D->done) return;
    const int par = D->round & 1;
    for (int g = blockIdx.x; g < D->n_gen; g += gridDim.x) {
        Chain& ch = D->chains[D->gen_chain[g]];
        const uint64_t d = ch.commit_d;
        const uint64_t* prev = D->draws[par ^ 1];
        const uint64_t need = ch.need_len;
        __syncthreads();
        for (int u = threadIdx.x; u < 312; u += blockDim.x) {
            const uint64_t v = d ? prev[ch.prev_off + (long long)d + u] : ch.hist[u];
            st[u] = v;
            if (d) ch.hist[u] = v;
        }
        __syncthreads();
        if (need == 0) continue;
        uint64_t* out = D->draws[par] + ch.need_off;
        for (int u = threadIdx.x; u < 312; u += blockDim.x) out[u] = st[u];
        const int k = threadIdx.x;
        for (uint64_t w0 = 312; w0 < need + 312; w0 += 312) {
            uint64_t v = 0;
            if (k < 156) v = mt_twist(st[k], st[k + 1], st[k + 156]);
            __syncthreads();
            if (k < 156) { st[k] = v; if (w0 + k < need + 312) out[w0 + k] = v; }
            __syncthreads();
            if (k < 156) { const int kk = k + 156; v = mt_twist(st[kk], st[(kk + 1) % 312], st[kk - 156]); }
            __syncthreads();
            if (k < 156) { st[k + 156] = v; if (w0 + 156 + k < need + 312) out[w0 + 156 + k] = v; }
            __syncthreads();
        }
    }
}

// ------------------------------------------------------------------------------------
// k_prep: one warp per pending segment.  The sums of the reference are strictly sequential
// (CBS.cpp:986-989 mean and tss, :83-87 prefix sums), so lane 0 runs them as ONE dependent DADD chain
// (8 cycles per marker on B200) over chunks staged in shared memory, while the other lanes already have
// the next chunk of the segment in flight in registers; the results equal the reference's bit for bit.
// The per-block extrema are computed by k_scan.
// ------------------------------------------------------------------------------------
#define PREP_CHUNK 1024
__device__ void prep_warp(Dev* D, Task& t, int lane, double* buf) {
    const long long base = D->unit_off[t.unit] + t.lo;
    const double* __restrict__ x = D->x + base;
    double* cur = D->cur + base;
    const int n = t.n;
    const bool raw = t.raw != 0;
    double avg = 0.0;
    double r[PREP_CHUNK / 32];
    if (!raw) {
        // CBS.cpp:985
        // (the all-equal test rides on the loads of the mean pass: one pass over x less for the one warp)
        const double x0 = x[0];
        bool flat = true;
        // CBS.cpp:986 mean, sequential
        double s = 0.0;
#pragma unroll
        for (int q = 0; q < PREP_CHUNK / 32; ++q) { const int i = lane + 32 * q; r[q] = (i < n) ? x[i] : x0; }
        for (int c0 = 0; c0 < n; c0 += PREP_CHUNK) {
            const int cnt = min(PREP_CHUNK, n - c0);
            __syncwarp();
#pragma unroll
            for (int q = 0; q < PREP_CHUNK / 32; ++q) { buf[lane + 32 * q] = r[q]; if (!(fabs(r[q] - x0) < 1e-12)) flat = false; }
            __syncwarp();
            if (c0 + PREP_CHUNK < n) {
#pragma unroll
                for (int q = 0; q < PREP_CHUNK / 32; ++q) { const int i = c0 + PREP_CHUNK + lane + 32 * q; r[q] = (i < n) ? x[i] : x0; }
            }
            if (lane == 0) {
                int k = 0;
#pragma unroll 8
                for (; k + 1 < cnt; k += 2) {
                    const double2 v = *reinterpret_cast<const double2*>(buf + k);
                    s = s + v.x;
                    s = s + v.y;
                }
                if (k < cnt) s = s + buf[k];
            }
        }
        flat = __all_sync(FULL, flat);
        if (lane == 0) t.alleq = flat ? 1 : 0;
        if (flat) return;
        s = shfl_d(s, 0);
        avg = s / (double)n;
    }
    // (block ends, fac[L] and g[L] of the segment: k_tables, which runs before this kernel on the same stream)
    // CBS.cpp:987-989 centring and tss, :83-87 prefix sums
    double* sx = D->arena + t.off_sx;
    double run = 0.0, tss = 0.0;
    if (lane == 0) sx[0] = 0.0;
#pragma unroll
    for (int q = 0; q < PREP_CHUNK / 32; ++q) { const int i = lane + 32 * q; r[q] = (i < n) ? x[i] : 0.0; }
    for (int c0 = 0; c0 < n; c0 += PREP_CHUNK) {
        const int cnt = min(PREP_CHUNK, n - c0);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < PREP_CHUNK / 32; ++q) {
            const int i = c0 + lane + 32 * q;
            const double v = raw ? r[q] : r[q] - avg;
            buf[lane + 32 * q] = v;
            if (i < n) cur[i] = v;
        }
        __syncwarp();
        if (c0 + PREP_CHUNK < n) {
#pragma unroll
            for (int q = 0; q < PREP_CHUNK / 32; ++q) { const int i = c0 + PREP_CHUNK + lane + 32 * q; r[q] = (i < n) ? x[i] : 0.0; }
        }
        if (lane == 0) {
            int k = 0;
#pragma unroll 8
            for (; k + 1 < cnt; k += 2) {
                double2 v = *reinterpret_cast<const double2*>(buf + k);
                run = run + v.x; tss = tss + v.x * v.x; v.x = run;
                run = run + v.y; tss = tss + v.y * v.y; v.y = run;
                *reinterpret_cast<double2*>(buf + k) = v;
            }
            if (k < cnt) { const double v = buf[k]; run = run + v; tss = tss + v * v; buf[k] = run; }
        }
        __syncwarp();
        for (int k = lane; k < cnt; k += 32) sx[c0 + 1 + k] = buf[k];
    }
    run = shfl_d(run, 0);
    for (int k = lane; k < SX_PAD; k += 32) sx[n + 1 + k] = run;  // finite padding behind S_n (read by k_scan)
    if (lane == 0 && !raw) t.tss = tss;
}

// k_tables: per new segment the block ends bb[0..nb] (CBS.cpp:71,77), fac[L] = n/(L(n-L)) (the reference's expression,
// :191-193) and g[L] = sqrt(L(n-L)/n); divisions and square roots in double, spread over the whole grid
__global__ void __launch_bounds__(256) k_tables(Dev* D) {
    if (D->done) return;
    for (int k = blockIdx.y; k < D->n_prep; k += gridDim.y) {
        const Task& t = D->tasks[D->prep_task[k]];
        const long long base = D->unit_off[t.unit] + t.lo;
        const int n = t.n, nb = t.nb;
        const double rn = (double)n;
        for (int L = blockIdx.x * blockDim.x + threadIdx.x; L < n; L += gridDim.x * blockDim.x) {
            if (L <= nb) D->bbtab[base + L] = block_end(n, nb, L);
            if (L >= 1) {
                const double rr = (double)L;
                const double prod = rr * (rn - rr);
                D->factab[base + L] = rn / prod;
                D->gtab[base + L] = sqrt(prod / rn);
            }
        }
        if (n <= nb && blockIdx.x == 0 && threadIdx.x == 0) for (int b = n; b <= nb; ++b) D->bbtab[base + b] = block_end(n, nb, b);
    }
}

__global__ void __launch_bounds__(32) k_prep(Dev* D) {
    __shared__ __align__(16) double buf[PREP_CHUNK];
    if (D->done) return;
    for (int k = blockIdx.x; k < D->n_prep; k += gridDim.x) prep_warp(D, D->tasks[D->prep_task[k]], threadIdx.x, buf);
}

// ------------------------------------------------------------------------------------
// Shared MT stream (chain == 0: every unit starts from the same engine state, so all chains read
// ONE raw stream W[0..)).  It is extended on demand, in parallel (mt_jump.h):
//   k_gen_lead  one CTA: sequential lead-in of GEN_LEAD words after the current end (or the whole
//               extension if it is short / no jump table)
//   k_gen_par   CTA c: first 312 words of segment c as the GF(2) combination
//               W[base+c*S+u] = XOR_{i: g_cS[i]=1} W[base+u+i], then the ordinary recurrence to the
//               end of the segment.  All segments advance concurrently.
// ------------------------------------------------------------------------------------
#define GEN_SEG (1LL << 18)
#define GEN_NSEG 512
#define GEN_LEAD 20480

// extend the raw stream (ring + mirror, cbs_core.h) sequentially from position `from` to `to` (state = the 312 words
// before `from`); called by all threads of a CTA with >= 156 threads
__device__ void gen_sequential(const Dev& D, long long from, long long to, uint64_t* st) {
    const int k = threadIdx.x;
    __syncthreads();
    for (int u = k; u < 312; u += blockDim.x) st[u] = stream_get(D, from - 312 + u);
    __syncthreads();
    for (long long pos = from; pos < to; pos += 312) {
        uint64_t v = 0;
        if (k < 156) v = mt_twist(st[k], st[k + 1], st[k + 156]);
        __syncthreads();
        if (k < 156) { st[k] = v; if (pos + k < to) stream_put(D, pos + k, v); }
        __syncthreads();
        if (k < 156) { const int kk = k + 156; v = mt_twist(st[kk], st[(kk + 1) % 312], st[kk - 156]); }
        __syncthreads();
        if (k < 156) { st[k + 156] = v; if (pos + 156 + k < to) stream_put(D, pos + 156 + k, v); }
        __syncthreads();
    }
}

// ahead = 0: extend the stream to what this round's shuffles need (normally nothing: see ahead = 1).
// ahead = 1: runs on its own stream next to the shuffles and the scan of the round and extends the stream
//            GEN_AHEAD words beyond the need, so that the next round usually finds its words already generated.
// The stream never grows beyond stream_lo + stream_cap - 312: positions from stream_lo on are still needed by a chain.
#define GEN_AHEAD (64LL << 20)
__global__ void __launch_bounds__(192) k_gen_lead(Dev* D, int ahead) {
    __shared__ uint64_t st[312];
    if (D->done || !D->shared_stream) return;
    if (ahead) {  // fold the extension of the ahead = 0 pass of this round (k_sched folds the last one of a round)
        __syncthreads();
        if (threadIdx.x == 0 && D->gen_E > 0) { D->stream_len = D->gen_base + D->gen_E; D->gen_E = 0; }
        __syncthreads();
    }
    const long long len = D->stream_len;
    long long target = D->stream_target;
    if (ahead) {
        // How far ahead: a launch costs about the same for one segment or for all of them (the GF(2) combination of the
        // segment heads dominates), and a round whose need outruns the stream pays a whole generator launch on its critical
        // path -- but words nobody reads are HBM writes and SM time taken from the shuffles running next to this kernel.
        // So: twice the growth of the need over the last round, at least GEN_AHEAD, at most the span of one launch.
        long long extra = GEN_AHEAD;
        if (D->jump_polys) {
            const long long growth = target - D->stream_target_prev;
            if (2 * growth > extra) extra = 2 * growth;
            if (extra > D->span_max) extra = D->span_max;
        }
        __syncthreads();
        if (threadIdx.x == 0) D->stream_target_prev = target;
        target += extra;
        if (target > len + D->span_max) target = len + D->span_max;
    }
    if (target > D->stream_lo + D->stream_cap - 312) target = D->stream_lo + D->stream_cap - 312;  // the scheduler never asks for more
    if (len >= target) { if (threadIdx.x == 0) { D->gen_base = len; D->gen_E = 0; } return; }
    const long long E = target - len;
    long long lead_end = target;
    if (D->jump_polys && E > GEN_SEG) lead_end = len + GEN_LEAD;
    gen_sequential(*D, len, lead_end, st);
    if (threadIdx.x == 0) { D->gen_base = len; D->gen_E = E; D->gen_lead_end = lead_end; }
}

__global__ void __launch_bounds__(320) k_gen_par(Dev* D) {
    __shared__ uint64_t st[312];
    __shared__ uint64_t sp[312];
    if (D->done || !D->shared_stream || !D->jump_polys) return;
    const long long base = D->gen_base, E = D->gen_E;
    if (E <= GEN_SEG) return;  // k_gen_lead did everything
    const int c = blockIdx.x;
    if ((long long)c * GEN_SEG >= E) return;
    const long long seg_lo = base + (long long)c * GEN_SEG;
    const long long seg_hi = base + ((E < (long long)(c + 1) * GEN_SEG) ? E : (long long)(c + 1) * GEN_SEG);
    long long from = D->gen_lead_end;
    if (c > 0) {
        const uint64_t* g = D->jump_polys + (size_t)c * 312;
        for (int u = threadIdx.x; u < 312; u += blockDim.x) sp[u] = g[u];
        __syncthreads();
        if (threadIdx.x < 312) {
            // the lead-in W[base .. base+GEN_LEAD) is read linearly from the ring slot of `base` (the mirror covers it)
            const uint64_t* src = D->stream + (base & D->stream_mask) + threadIdx.x;
            uint64_t acc0 = 0, acc1 = 0;
            for (int wd = 0; wd < 312; ++wd) {
                const uint64_t bits = sp[wd];
                const uint64_t* s0 = src + wd * 64;
#pragma unroll 8
                for (int bpos = 0; bpos < 64; bpos += 2) {
                    if ((bits >> bpos) & 1ULL) acc0 ^= s0[bpos];
                    if ((bits >> (bpos + 1)) & 1ULL) acc1 ^= s0[bpos + 1];
                }
            }
            stream_put(*D, seg_lo + threadIdx.x, acc0 ^ acc1);
        }
        __syncthreads();
        from = seg_lo + 312;
    }
    if (from < seg_hi) gen_sequential(*D, from, seg_hi, st);
}

// ------------------------------------------------------------------------------------
// k_perm_smem: one warp per permutation, segments of up to 65535 markers.
//   * the permutation is built on a 16-bit INDEX array in shared memory (2 B per marker), so
//     the Fisher-Yates random accesses never leave the SM;
//   * 32 consecutive steps of CBS.cpp:489-492 are taken per warp iteration: a step commutes
//     with the others of its group unless it shares a position with one of them; those few
//     (detected with match.any / redux.or) are replayed in order afterwards -- the result is
//     the sequential shuffle, bit for bit;
//   * the prefix sums are then accumulated in index order: every lane runs the same
//     dependent DADD chain on shuffled-in values x[idx[k]], lane k keeps S_k and stores it
//     coalesced (CBS.cpp:83-90 order, hence identical rounding).
// ------------------------------------------------------------------------------------
// index-array accessors: shared memory (16-bit) or global memory (32-bit, L2 only: ld/st.cg)
struct IdxSmem {
    static constexpr bool kClaimTable = true;   // conflicts through the claim table (a false positive costs ~80 cycles)
    unsigned short* a;
    __device__ __forceinline__ int ld(int k) const { return a[k]; }
    __device__ __forceinline__ void st(int k, int v) const { a[k] = (unsigned short)v; }
};
struct IdxGlobal {
    static constexpr bool kClaimTable = false;  // a replayed step costs an L2 round trip: exact detection (match.any)
    unsigned int* a;
    __device__ __forceinline__ int ld(int k) const { return (int)__ldcg(a + k); }
    __device__ __forceinline__ void st(int k, int v) const { __stcg(a + k, (unsigned int)v); }
};

// 32 consecutive Fisher-Yates steps (CBS.cpp:489-492) taken by the 32 lanes at once: lane l swaps row i-1
// (i = i0-l) with row j-1.  A step commutes with the others of its group unless it shares a row with one of
// them; those few are replayed in order afterwards, so the result is the sequential shuffle.  Sharing is
// detected through a small table in shared memory (match.any costs ~400 cycles on B200): every lane writes its
// id into slot j mod 8192 and reads it back -- whoever does not find itself shares the slot with the winner
// (same target, or a harmless hash collision); a target inside the group's own rows flags the owner of that row.
#define FY_TAB 8192
#define FY_SCRATCH (FY_TAB + 256)  // bytes of per-warp scratch: claim table + one flag per step of a round
template <class Idx>
__device__ __forceinline__ void fy_group(Idx s_idx, unsigned char* tab, int i0, int i, int j, int lane) {
    if (!Idx::kClaimTable) {
        const int vi = s_idx.ld(i - 1), vj = s_idx.ld(j - 1);  // in flight while match.any resolves
        const unsigned same = __match_any_sync(FULL, j);
        const int m = i0 - j;  // lane whose row is my target
        const bool tgt = (m >= 0) && (m < 32) && (m != lane);
        const unsigned tmask = __reduce_or_sync(FULL, tgt ? (1u << m) : 0u);
        const bool conflict = (__popc(same) > 1) || tgt || ((tmask >> lane) & 1u);
        __syncwarp();
        if (!conflict) { s_idx.st(i - 1, vj); s_idx.st(j - 1, vi); }
        __syncwarp();
        unsigned cm = __ballot_sync(FULL, conflict);
        while (cm) {
            const int l = __ffs(cm) - 1;
            cm &= cm - 1;
            if (lane == l) {
                const int a = s_idx.ld(i - 1), b = s_idx.ld(j - 1);
                s_idx.st(i - 1, b); s_idx.st(j - 1, a);
            }
            __syncwarp();
        }
        return;
    }
    unsigned char* cflag = tab + FY_TAB;
    const int slot = j & (FY_TAB - 1);
    const int m = i0 - j;  // lane whose row is my target
    const bool tgt = (m >= 0) && (m < 32) && (m != lane);
    tab[slot] = (unsigned char)lane;
    if (tgt) cflag[m] = 1;
    __syncwarp();
    const int w = tab[slot];
    const bool loser = (w != lane);
    if (loser) cflag[w] = 1;
    const int vi = s_idx.ld(i - 1), vj = s_idx.ld(j - 1);
    __syncwarp();
    const bool conflict = loser || tgt || (cflag[lane] != 0);
    cflag[lane] = 0;
    if (!conflict) { s_idx.st(i - 1, vj); s_idx.st(j - 1, vi); }
    __syncwarp();
    unsigned cm = __ballot_sync(FULL, conflict);
    while (cm) {
        const int l = __ffs(cm) - 1;
        cm &= cm - 1;
        if (lane == l) {
            const int a = s_idx.ld(i - 1), b = s_idx.ld(j - 1);
            s_idx.st(i - 1, b); s_idx.st(j - 1, a);
        }
        __syncwarp();
    }
}

// K*32 consecutive steps at once: lane l takes steps i = i0 - 32k - l, k = 0..K-1 (step id 32k+l).  Same scheme as
// fy_group with one round of claims for all K*32 steps, so the three shared-memory round trips of a round are
// paid once per K*32 steps.  Used while i0 is large (few steps of a round share a row).
template <int K, class Idx>
__device__ __forceinline__ void fy_multi(Idx s_idx, unsigned char* tab, int i0, const int (&j)[K], int lane) {
    unsigned char* cflag = tab + FY_TAB;
    bool tgt[K], dup[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        const int m = i0 - j[k];  // id of the step whose row is my target
        tgt[k] = (m >= 0) && (m < 32 * K) && (m != 32 * k + lane);
        tab[j[k] & (FY_TAB - 1)] = (unsigned char)(32 * k + lane);
        if (tgt[k]) cflag[m] = 1;
        dup[k] = false;
    }
    __syncwarp();
    int vi[K], vj[K];
    bool loser[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        vi[k] = s_idx.ld(i0 - 32 * k - lane - 1);
        vj[k] = s_idx.ld(j[k] - 1);
        loser[k] = (tab[j[k] & (FY_TAB - 1)] != 32 * k + lane);
    }
    // a step that lost its slot shares it with a step of the same target (a real conflict) or merely of the same
    // hash: settle it exactly, the targets of all K*32 steps are in registers
#pragma unroll
    for (int k = 0; k < K; ++k) {
        unsigned lm = __ballot_sync(FULL, loser[k]);
        while (lm) {
            const int l = __ffs(lm) - 1;
            lm &= lm - 1;
            const int jj = __shfl_sync(FULL, j[k], l);
            bool hit = false;
#pragma unroll
            for (int k2 = 0; k2 < K; ++k2) {
                const bool same = (j[k2] == jj) && !(k2 == k && lane == l);
                dup[k2] |= same;
                hit |= same;
            }
            if (__any_sync(FULL, hit) && lane == l) dup[k] = true;
        }
    }
    __syncwarp();
    bool conflict[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
        conflict[k] = dup[k] || tgt[k] || (cflag[32 * k + lane] != 0);
        cflag[32 * k + lane] = 0;
        if (!conflict[k]) { s_idx.st(i0 - 32 * k - lane - 1, vj[k]); s_idx.st(j[k] - 1, vi[k]); }
    }
    __syncwarp();
#pragma unroll
    for (int k = 0; k < K; ++k) {
        unsigned cm = __ballot_sync(FULL, conflict[k]);
        while (cm) {
            const int l = __ffs(cm) - 1;
            cm &= cm - 1;
            if (lane == l) {
                const int r = i0 - 32 * k - lane - 1;
                const int a = s_idx.ld(r), b = s_idx.ld(j[k] - 1);
                s_idx.st(r, b); s_idx.st(j[k] - 1, a);
            }
            __syncwarp();
        }
    }
}
#define FY_MULTI_MIN 8192    // rounds of 128 steps while i0 is at least this
#define FY_MULTI8_MIN 20480  // rounds of 256 steps while i0 is at least this

#define PERM_CHUNK 1024
template <class Idx>
__device__ void perm_warp(Dev* D, const Task& t, int p, Idx s_idx, unsigned char* tab, int lane) {
    const int n = t.n;
    const long long base = D->unit_off[t.unit] + t.lo;
    const double* __restrict__ cur = D->cur + base;
    const bool mt = D->prm.rng_mode == RNG_MT;
    const uint64_t* win = nullptr;
    if (mt) win = draw_window(*D, t.off_draw + (long long)p * n);
    const uint32_t k0 = (uint32_t)t.key, k1 = (uint32_t)(t.key >> 32), permno = (uint32_t)(t.perms_done + p);
    for (int k = lane; k < n; k += 32) s_idx.st(k, k);
    __syncwarp();
    // groups of 32 steps while i0 >= 64; group g covers steps i = n-32g .. n-32g-31, lane l takes i = n-32g-l
    // and draw number 32g+l of this permutation
    const int G = (n >= 64) ? ((n - 64) / 32 + 1) : 0;
    int i0 = n;
    if (mt) {
        // the raw words of the next 8 groups are in flight (registers) while 8 groups are shuffled: the
        // stream lives in HBM / L2, one load per group would expose its latency in every group
        uint64_t raw[8], nxt[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) raw[q] = (q < G) ? win[32 * q + lane] : 0ull;
        for (int g0 = 0; g0 < G; g0 += 8) {
            // the stream lives in HBM: pull the words of four blocks ahead into L2 (2 KB = 16 lines per block), the
            // register prefetch one block ahead then only pays an L2 hit
            if (lane < 16 && g0 + 40 < G) asm volatile("prefetch.global.L2 [%0];" ::"l"(win + 32 * (g0 + 32) + 16 * lane));
#pragma unroll
            for (int q = 0; q < 8; ++q) { const int g = g0 + 8 + q; nxt[q] = (g < G) ? win[32 * g + lane] : 0ull; }
            if (Idx::kClaimTable && g0 + 7 < G && i0 >= FY_MULTI8_MIN) {
                int j8[8];
#pragma unroll
                for (int k = 0; k < 8; ++k) j8[k] = draw_index(mt_temper(raw[k]), i0 - 32 * k - lane);
                fy_multi<8>(s_idx, tab, i0, j8, lane);
                i0 -= 256;
            } else
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                if (Idx::kClaimTable && g0 + 4 * h + 3 < G && i0 >= FY_MULTI_MIN) {
                    int j4[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) j4[k] = draw_index(mt_temper(raw[4 * h + k]), i0 - 32 * k - lane);
                    fy_multi<4>(s_idx, tab, i0, j4, lane);
                    i0 -= 128;
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if (g0 + 4 * h + k < G) {
                            const int i = i0 - lane;
                            fy_group(s_idx, tab, i0, i, draw_index(mt_temper(raw[4 * h + k]), i), lane);
                            i0 -= 32;
                        }
                    }
                }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) raw[q] = nxt[q];
        }
        // tail (i0 < 64 steps): the remaining raw words are loaded once, lane 0 replays the steps
        const uint64_t w0 = (lane < i0) ? win[32 * G + lane] : 0ull;
        const uint64_t w1 = (32 + lane < i0) ? win[32 * G + 32 + lane] : 0ull;
        for (int tt = 0; tt < i0; ++tt) {
            const uint64_t rw = __shfl_sync(FULL, (tt < 32) ? w0 : w1, tt & 31);
            if (lane == 0) {
                const int i = i0 - tt;
                const int j = draw_index(mt_temper(rw), i);
                const int a = s_idx.ld(i - 1), b = s_idx.ld(j - 1);
                s_idx.st(i - 1, b); s_idx.st(j - 1, a);
            }
        }
    } else {
        auto philox_j = [&](int i) {
            const uint32_t kd = (uint32_t)(n - i);
            uint32_t o[4];
            philox4x32_10(kd >> 1, permno, 0u, 0u, k0, k1, o);
            const uint64_t u = (kd & 1u) ? (((uint64_t)o[3] << 32) | o[2]) : (((uint64_t)o[1] << 32) | o[0]);
            return draw_index(u, i);
        };
        int g = 0;
        for (; Idx::kClaimTable && g + 7 < G && i0 >= FY_MULTI8_MIN; g += 8, i0 -= 256) {
            int j8[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) j8[k] = philox_j(i0 - 32 * k - lane);
            fy_multi<8>(s_idx, tab, i0, j8, lane);
        }
        for (; Idx::kClaimTable && g + 3 < G && i0 >= FY_MULTI_MIN; g += 4, i0 -= 128) {
            int j4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) j4[k] = philox_j(i0 - 32 * k - lane);
            fy_multi<4>(s_idx, tab, i0, j4, lane);
        }
        for (; g < G; ++g, i0 -= 32) {
            const int i = i0 - lane;
            fy_group(s_idx, tab, i0, i, philox_j(i), lane);
        }
        if (lane == 0) {
            DrawSrc src;
            src.init_philox(t.key, 0u, permno);
            for (int i = i0; i >= 1; --i) {
                const int j = draw_index(src.u64((uint32_t)(n - i)), i);
                const int a = s_idx.ld(i - 1), b = s_idx.ld(j - 1);
                s_idx.st(i - 1, b); s_idx.st(j - 1, a);
            }
        }
    }
    __syncwarp();
    // gather the permuted values into the prefix-sum slots: S[k+1] <- x[idx[k]] (coalesced stores); k_chain turns
    // them into prefix sums in place.  (The chain is a separate kernel because it needs no index array: an SM holds
    // only a few index arrays, but dozens of chains.)
    double* sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
    if (D->w) {
        // weighted CBS, wxperm (CBS.cpp:538-547): the Fisher-Yates runs on y = cur*rw and position i-1 receives
        // y[.]/rw[i-1] at step i -- unless the step drew j == i, in which case the reference's swap restores the
        // undivided value.  Draw number n-i of the permutation belongs to step i.
        const double* __restrict__ ycur = D->ycur + base;
        const double* __restrict__ rw = D->rw + base;
        for (int k = lane; k < n; k += 32) {
            const int i = k + 1;
            uint64_t u;
            if (mt) u = mt_temper(win[n - i]);
            else {
                const uint32_t kd = (uint32_t)(n - i);
                uint32_t o[4];
                philox4x32_10(kd >> 1, permno, 0u, 0u, k0, k1, o);
                u = (kd & 1u) ? (((uint64_t)o[3] << 32) | o[2]) : (((uint64_t)o[1] << 32) | o[0]);
            }
            const double y = ycur[s_idx.ld(k)];
            sx[k + 1] = (draw_index(u, i) == i) ? y : y / rw[k];
        }
        __syncwarp();
        return;
    }
    int k = lane;
    for (; k + 480 < n; k += 512) {
        int id[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) id[q] = s_idx.ld(k + 32 * q);
        double v[16];
#pragma unroll
        for (int q = 0; q < 16; ++q) v[q] = __ldg(cur + id[q]);
#pragma unroll
        for (int q = 0; q < 16; ++q) sx[k + 1 + 32 * q] = v[q];
    }
    for (; k < n; k += 32) sx[k + 1] = cur[s_idx.ld(k)];
    __syncwarp();
}

// k_shuffle: xperm (CBS.cpp:487-493) for segments of up to 65535 markers, one CTA per permutation (shuffle.cuh):
// exact parallel replay of the Fisher-Yates, last[] (16 bit per marker) and the claim table in shared memory; the
// permuted values go straight into the S row of the permutation (k_chain turns them into prefix sums in place).
template <int T, int K, bool MT>
__global__ void __launch_bounds__(T) k_shuffle(Dev* D, int cls, int hbits) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_g;
    unsigned* claim = (unsigned*)smem_raw;
    unsigned short* last = (unsigned short*)(smem_raw + ((size_t)4 << hbits));
    if (D->done) return;
    const int hmask = (1 << hbits) - 1;
    for (int k = threadIdx.x; k <= hmask; k += T) claim[k] = 0u;
    unsigned epoch = 0;
    const int nl = D->n_shuf[cls];
    const int total = D->shuf_prefix[cls][nl];
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) s_g = (int)atomicAdd(&D->ctr[8 + cls], 1u);
        __syncthreads();
        const int g = s_g;
        if (g >= total) break;
        const int k = find_item(D->shuf_prefix[cls], nl, g);
        const PermItem it = D->items[D->shuf_item[cls][k]];
        const Task& t = D->tasks[it.task];
        const int p = D->shuf_p0[cls][k] + (g - D->shuf_prefix[cls][k]);
        const int n = t.n;
        const long long base = D->unit_off[t.unit] + t.lo;
        ShufDraws<MT> src;
        src.win = MT ? draw_window(*D, t.off_draw + (long long)p * n) : nullptr;
        src.k0 = (uint32_t)t.key; src.k1 = (uint32_t)(t.key >> 32); src.permno = (uint32_t)(t.perms_done + p);
        double* sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        // weighted CBS (wxperm, CBS.cpp:538-547): the shuffle runs on y = cur*rw, position i-1 receives y[.]/rw[i-1]
        const double* vals = D->w ? D->ycur + base : D->cur + base;
        const double* rdiv = D->w ? D->rw + base : nullptr;
        shuffle_cta<T, K>(LastSmem16{last}, claim, hmask, epoch, n, src, vals, rdiv, sx);
    }
}

// k_shuffle_cluster: the same for segments of more than 65535 markers; a cluster of R CTAs per permutation shares
// last[] (32 bit per marker) through distributed shared memory (shuffle.cuh)
template <int T, int K, int R, bool MT>
__global__ void __cluster_dims__(R, 1, 1) __launch_bounds__(T) k_shuffle_cluster(Dev* D, int cls, int hbits) {
    namespace cg = cooperative_groups;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ int s_g;
    unsigned* claim = (unsigned*)smem_raw;
    unsigned* last = (unsigned*)(smem_raw + ((size_t)4 << hbits));
    if (D->done) return;
    cg::cluster_group cl = cg::this_cluster();
    const int hmask = (1 << hbits) - 1;
    for (int k = threadIdx.x; k <= hmask; k += T) claim[k] = 0u;
    unsigned epoch = 0;
    const int nl = D->n_shuf[cls];
    const int total = D->shuf_prefix[cls][nl];
    for (;;) {
        cl.sync();  // the previous permutation's root walks (remote reads of last[]) are over
        if (cl.block_rank() == 0 && threadIdx.x == 0) {
            const int g = (int)atomicAdd(&D->ctr[8 + cls], 1u);
            for (int r = 0; r < R; ++r) *cl.map_shared_rank(&s_g, r) = g;
        }
        cl.sync();
        const int g = s_g;
        if (g >= total) break;
        const int k = find_item(D->shuf_prefix[cls], nl, g);
        const PermItem it = D->items[D->shuf_item[cls][k]];
        const Task& t = D->tasks[it.task];
        const int p = D->shuf_p0[cls][k] + (g - D->shuf_prefix[cls][k]);
        const int n = t.n;
        const long long base = D->unit_off[t.unit] + t.lo;
        ShufDraws<MT> src;
        src.win = MT ? draw_window(*D, t.off_draw + (long long)p * n) : nullptr;
        src.k0 = (uint32_t)t.key; src.k1 = (uint32_t)(t.key >> 32); src.permno = (uint32_t)(t.perms_done + p);
        double* sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        const double* vals = D->w ? D->ycur + base : D->cur + base;
        const double* rdiv = D->w ? D->rw + base : nullptr;
        shuffle_cluster<T, K, R>(last, claim, hmask, epoch, n, src, vals, rdiv, sx);
    }
}

// ------------------------------------------------------------------------------------
// k_perm: the same warp-per-permutation shuffle for segments of 65536+ markers, whose index
// array (32-bit) does not fit in shared memory and lives in the arena (L2-resident accesses).
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_perm(Dev* D) {
    if (D->done) return;
    const int lane = threadIdx.x & 31;
    unsigned char* tab = nullptr;  // IdxGlobal does not use the claim table (measured: 128-step rounds lose on L2 arrays)
    const int nl = D->n_shuf[SHUF_GLOBAL];
    const int total = D->shuf_prefix[SHUF_GLOBAL][nl];
    for (;;) {
        int g = 0;
        if (lane == 0) g = (int)atomicAdd(&D->ctr[0], 1u);
        g = __shfl_sync(FULL, g, 0);
        if (g >= total) break;
        const int k = find_item(D->shuf_prefix[SHUF_GLOBAL], nl, g);
        const PermItem it = D->items[D->shuf_item[SHUF_GLOBAL][k]];
        const Task& t = D->tasks[it.task];
        const int slot = g - D->shuf_prefix[SHUF_GLOBAL][k];  // the entry's permutations have consecutive index arrays
        const int p = D->shuf_p0[SHUF_GLOBAL][k] + slot;
        const long long idxd = Sched::idx_stride(t.n);  // doubles per permutation (cbs_core.h plan_perm)
        unsigned int* idx = (unsigned int*)(D->arena + t.off_A + (long long)slot * idxd);
        perm_warp(D, t, p, IdxGlobal{idx}, tab, lane);
    }
}

// ------------------------------------------------------------------------------------
// k_chain: turns the gathered values S[1..n] of every permutation into prefix sums IN PLACE with ONE strictly
// sequential DADD chain per permutation (the reference's order, CBS.cpp:83-90, hence identical rounding), and writes
// the row's statistics for the scan next to it: per block of the reference's sqrt(n) blocks the extrema with their FIRST
// occurrence (CBS.cpp:88-94), and per aligned run of 32 prefix sums the extrema in single precision rounded outwards.
// A CTA is one summing warp and CP_STAT_WARPS = 4 statistics warps, and owns CHAIN_Q = 4 consecutive permutations of a batch:
//   warp A   stages chunks of the four rows in shared memory (the next chunk is already in flight in registers); lanes
//            0, 8, 16, 24 each walk one row at the DADD latency (8 cycles per marker on B200), so one warp instruction
//            advances four chains and nothing else is ever on their critical path;
//   warps B  take each finished chunk, one warp per row: store it coalesced and compute the statistics (block extrema
//            reduced with redux.sync on order-preserving keys), while A is already summing the next chunk.  One
//            statistics warp for all four rows (the first form of this layout) could not keep up with the summing warp.
// The chunks go through a ring of CP_SLOTS buffers; the hand-over is two monotone chunk counters in shared memory.
// Round 1 gave a permutation one warp that did both jobs in turn with one active lane: ~5.4 warp instructions per
// marker, issue bound at a fraction of the FP64 pipe; here the summing warp issues ~1.3 per marker and the
// statistics warps, on the other schedulers of the SM, the rest (4.2 in total, profiles/r02_ncu_round4_final.md).
// ------------------------------------------------------------------------------------
#define CP_CHUNK 256
#define CP_ROW (CP_CHUNK + 4)  // doubles: +4 puts the four rows on different banks for the 128-bit accesses of the summing lanes
#define CP_SLOTS 3

// order-preserving map between floats and signed 32-bit integers (its own inverse on the bit pattern)
__device__ __forceinline__ int fkey(float v) { const int b = __float_as_int(v); return b ^ ((b >> 31) & 0x7fffffff); }
__device__ __forceinline__ float funkey(int k) { return __int_as_float(k ^ ((k >> 31) & 0x7fffffff)); }

// first occurrence of the smallest (largest) value among the lanes of `gmask`: three redux.sync on the order-preserving key
__device__ __forceinline__ void group_argmin(double& v, int& idx, unsigned gmask) {
    const long long key = dkey(v + 0.0);  // -0.0 and +0.0 compare equal in the reference: one key
    const int hi = (int)(key >> 32);
    const unsigned lo = (unsigned)key;
    const int mhi = __reduce_min_sync(gmask, hi);
    const unsigned mlo = __reduce_min_sync(gmask, hi == mhi ? lo : 0xffffffffu);
    const bool win = hi == mhi && lo == mlo;
    idx = __reduce_min_sync(gmask, win ? idx : 0x7fffffff);
    v = dunkey(((long long)mhi << 32) | (long long)mlo);
}
__device__ __forceinline__ void group_argmax(double& v, int& idx, unsigned gmask) {
    const long long key = dkey(v + 0.0);
    const int hi = (int)(key >> 32);
    const unsigned lo = (unsigned)key;
    const int mhi = __reduce_max_sync(gmask, hi);
    const unsigned mlo = __reduce_max_sync(gmask, hi == mhi ? lo : 0u);
    const bool win = hi == mhi && lo == mlo;
    idx = __reduce_min_sync(gmask, win ? idx : 0x7fffffff);
    v = dunkey(((long long)mhi << 32) | (long long)mlo);
}

#define CP_STAT_WARPS 4                       // warps B: each takes CHAIN_Q / CP_STAT_WARPS rows of the chunk
#define CP_LPR (32 * CP_STAT_WARPS / CHAIN_Q)  // lanes of a warp B per row (32: a warp per row)
template <bool WEIGHTED>  // weighted CBS: the chain adds px*w (wtmaxo, CBS.cpp:623,627); the product is rounded before the addition
__global__ void __launch_bounds__(32 * (1 + CP_STAT_WARPS)) k_chain(Dev* D) {
    __shared__ __align__(16) double bufs[CP_SLOTS][CHAIN_Q][CP_ROW];
    __shared__ volatile int s_full, s_done[CP_STAT_WARPS];
    __shared__ int s_g;
    if (D->done) return;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool summing = warp == 0;  // warp A
    if (threadIdx.x == 0) { s_full = 0; for (int w = 0; w < CP_STAT_WARPS; ++w) s_done[w] = 0; }
    __syncthreads();
    const int total = D->item_uprefix[D->n_items];
    const double dinf = __longlong_as_double(0x7ff0000000000000LL);
    int seq = 0;  // chunks handled so far (the same number in all warps)
    for (;;) {
        if (threadIdx.x == 0) s_g = (int)atomicAdd(&D->ctr[3], 1u);
        __syncthreads();
        const int g = s_g;
        __syncthreads();
        if (g >= total) break;
        const int k = find_item(D->item_uprefix, D->n_items, g);
        const PermItem it = D->items[k];
        if (it.obs) continue;  // k_prep wrote the prefix sums of observed data
        const Task& t = D->tasks[it.task];
        const int n = t.n, nb = t.nb;
        const int p0 = (g - D->item_uprefix[k]) * CHAIN_Q;
        const int nq = min(CHAIN_Q, it.P - p0);
        const long long stride = Sched::sx_stride(n);
        double* sx0 = D->arena + t.off_sx + (long long)p0 * stride;
        const int nchunks = (n + CP_CHUNK - 1) / CP_CHUNK;
        if (summing) {
            const int q = lane >> 3;  // lanes 0, 8, 16, 24 sum rows 0..3
            const double* __restrict__ wt = WEIGHTED ? D->w + D->unit_off[t.unit] + t.lo : nullptr;
            double run = 0.0;
            double r[CHAIN_Q][CP_CHUNK / 32];
#pragma unroll
            for (int q2 = 0; q2 < CHAIN_Q; ++q2)
#pragma unroll
                for (int j = 0; j < CP_CHUNK / 32; ++j) {
                    const int i = lane + 32 * j;
                    const bool ok = q2 < nq && i < n;
                    double v = ok ? sx0[(long long)q2 * stride + 1 + i] : 0.0;
                    if (WEIGHTED && ok) v = v * wt[i];
                    r[q2][j] = v;
                }
            for (int c = 0; c < nchunks; ++c) {
                const int c0 = c * CP_CHUNK, cnt = min(CP_CHUNK, n - c0);
                double (*buf)[CP_ROW] = bufs[(seq + c) % CP_SLOTS];
                // the slot's previous chunk has been consumed by every warp B (plain spin: a sleep overshoots by more than a chunk takes)
#pragma unroll
                for (int w = 0; w < CP_STAT_WARPS; ++w) while (s_done[w] < seq + c - (CP_SLOTS - 1)) {}
                __syncwarp();
#pragma unroll
                for (int q2 = 0; q2 < CHAIN_Q; ++q2)
#pragma unroll
                    for (int j = 0; j < CP_CHUNK / 32; ++j) buf[q2][lane + 32 * j] = r[q2][j];
                __syncwarp();
                if (c + 1 < nchunks) {
#pragma unroll
                    for (int q2 = 0; q2 < CHAIN_Q; ++q2)
#pragma unroll
                        for (int j = 0; j < CP_CHUNK / 32; ++j) {
                            const int i = c0 + CP_CHUNK + lane + 32 * j;
                            const bool ok = q2 < nq && i < n;
                            double v = ok ? sx0[(long long)q2 * stride + 1 + i] : 0.0;
                            if (WEIGHTED && ok) v = v * wt[i];
                            r[q2][j] = v;
                        }
                }
                if ((lane & 7) == 0 && q < nq) {
                    double* row = buf[q];
                    int kk = 0;
#pragma unroll 8
                    for (; kk + 1 < cnt; kk += 2) {
                        double2 v = *reinterpret_cast<const double2*>(row + kk);
                        run = run + v.x; v.x = run;
                        run = run + v.y; v.y = run;
                        *reinterpret_cast<double2*>(row + kk) = v;
                    }
                    if (kk < cnt) { run = run + row[kk]; row[kk] = run; }
                }
                __syncwarp();
                if (lane == 0) { __threadfence_block(); s_full = seq + c + 1; }
            }
        } else {
            const int bw = warp - 1;                       // which warp B
            const int sub = lane % CP_LPR;                 // lane within the row's group
            const int q = bw * (32 / CP_LPR) + lane / CP_LPR;  // row of this lane
            const bool valid = q < nq;
            const int qr = valid ? q : nq - 1;  // lanes of unused rows shadow the last row (uniform control flow), without writing
            const unsigned gmask = (CP_LPR == 32 ? 0xffffffffu : ((1u << CP_LPR) - 1u)) << (CP_LPR * (lane / CP_LPR));
            double* sxg = sx0 + (long long)qr * stride;
            BlockStats bs(D->arena + t.off_bs + (long long)(p0 + qr) * Sched::bs_stride(nb), nb);
            const int* __restrict__ bb = D->bbtab + D->unit_off[t.unit] + t.lo;
            float* tmin = (float*)(sxg + Sched::tbl_offset(n));
            float* tmax = tmin + Sched::tbl_entries(n);
            int b = 1;
            double blo = dinf, bhi = -dinf;
            int ilo = 0x7fffffff, ihi = 0x7fffffff;
            double prev_last = 0.0;  // S[0]
            if (valid && sub == 0) sxg[0] = 0.0;
            const int q_first = bw * (32 / CP_LPR), q_end = min(nq, q_first + 32 / CP_LPR);  // rows this warp stores
            for (int c = 0; c < nchunks; ++c) {
                const int c0 = c * CP_CHUNK, cnt = min(CP_CHUNK, n - c0), hi_idx = c0 + cnt;
                const double (*buf)[CP_ROW] = bufs[(seq + c) % CP_SLOTS];
                while (s_full < seq + c + 1) __nanosleep(256);  // B is the faster side and has two slots of slack: do not burn issue slots
                __threadfence_block();
                __syncwarp();
                for (int q2 = q_first; q2 < q_end; ++q2) {
                    double* dst = sx0 + (long long)q2 * stride + c0 + 1;
                    for (int kk = lane; kk < cnt; kk += 32) dst[kk] = buf[q2][kk];
                }
                const double* row = buf[qr];
                // per-block extrema with their first occurrence; the blocks are those of the segment, the same for all rows
                while (b <= nb) {
                    const int first = bb[b - 1] + 1, last = bb[b];
                    const int a = max(first, c0 + 1), z = min(last, hi_idx);
                    if (a > z) break;
                    double lo = dinf, hi = -dinf;
                    int jlo = 0x7fffffff, jhi = 0x7fffffff;
                    for (int i = a + sub; i <= z; i += CP_LPR) {
                        const double v = row[i - c0 - 1];
                        if (v < lo) { lo = v; jlo = i; }
                        if (v > hi) { hi = v; jhi = i; }
                    }
                    group_argmin(lo, jlo, gmask);
                    group_argmax(hi, jhi, gmask);
                    if (lo < blo) { blo = lo; ilo = jlo; }  // the part seen earlier holds the earlier indices: it wins ties
                    if (hi > bhi) { bhi = hi; ihi = jhi; }
                    if (last > hi_idx) break;  // the block continues in the next chunk
                    if (valid && sub == 0) { bs.bmin()[b - 1] = blo; bs.bmax()[b - 1] = bhi; bs.amin()[b - 1] = ilo; bs.amax()[b - 1] = ihi; }
                    ++b; blo = dinf; bhi = -dinf; ilo = 0x7fffffff; ihi = 0x7fffffff;
                }
                // table entries e = c0/32 + l cover S[32e .. 32e+31] = row[32l-1 .. 32l+30] (row[-1] = prev_last).  One pass per
                // entry: the row's group of lanes reads the run coalesced, converts (rounded outwards) and reduces with
                // redux.sync on order-preserving keys; the passes are independent, so their latencies overlap.  The entry that
                // starts with the chunk's last value is only complete in the last chunk.
                const bool last_chunk = hi_idx >= n;
                float mylo = 0.f, myhi = 0.f;
#pragma unroll
                for (int l = 0; l <= CP_CHUNK / 32; ++l) {
                    if (32 * l - 1 > cnt - 1 || (l == CP_CHUNK / 32 && !last_chunk)) continue;  // uniform
                    int klo = 0x7fffffff, khi = (int)0x80000000;
                    for (int u = sub; u < 32; u += CP_LPR) {
                        const int kx = 32 * l - 1 + u;
                        if (kx <= cnt - 1) {
                            // order-preserving key of the HIGH word of the double: integer work only (two f64 -> f32 conversions per
                            // prefix sum saturate the XU pipe, about one lane per clock and SM on B200)
                            const int hk = fkey(__int_as_float(__double2hiint((kx < 0) ? prev_last : row[kx])));
                            klo = min(klo, hk); khi = max(khi, hk);
                        }
                    }
                    klo = __reduce_min_sync(gmask, klo); khi = __reduce_max_sync(gmask, khi);
                    if (sub == (l % CP_LPR)) {
                        // all doubles with the extreme high words lie between these two; rounded outwards to single precision
                        const int hlo = __float_as_int(funkey(klo)), hhi = __float_as_int(funkey(khi));
                        mylo = __double2float_rd(__hiloint2double(hlo, hlo < 0 ? -1 : 0));
                        myhi = __double2float_ru(__hiloint2double(hhi, hhi < 0 ? 0 : -1));
                        if (valid) { tmin[(c0 >> 5) + l] = mylo; tmax[(c0 >> 5) + l] = myhi; }
                    }
                }
                prev_last = row[cnt - 1];
                __syncwarp();
                if (lane == 0) s_done[bw] = seq + c + 1;
            }
            // the scan reads up to SX_PAD values behind S_n without bounds checks: keep them finite
            for (int q2 = q_first; q2 < q_end; ++q2) {
                const double lastv = shfl_d(prev_last, CP_LPR * (q2 - q_first));
                double* dst = sx0 + (long long)q2 * stride + n + 1;
                for (int kk = lane; kk < SX_PAD; kk += 32) dst[kk] = lastv;
            }
        }
        seq += nchunks;
    }
}

// ------------------------------------------------------------------------------------
// k_scan -- the max-t arc scan.
//
// One CTA per (segment, permutation).  The reference finds max over arcs (i,j) of
// fac(L) * (S_j - S_i)^2, L = j - i, by visiting sqrt(n) x sqrt(n) block pairs in order of
// their corner statistic and pruning with the running maximum (CBS.cpp:119-216).  Here:
//   phase 0 the per-block extrema of the prefix sums with their first occurrence (CBS.cpp:88-94) and a
//           table of the extrema of every aligned run of 32 (64, 128) prefix sums, in shared memory;
//   pass 1  every thread evaluates corner arcs of block pairs; the best VALID corner gives a
//           lower bound LB on the answer (it is an arc the reference also evaluates);
//   pass 2  warps claim block pairs whose upper bound reaches the current level.  A pair is cut
//           into units of 32 positions x 8 arc lengths on the global index grid.  A unit can only hold
//           an arc above level M if max|S_j - S_i| over the values it touches exceeds
//           sqrt(M) * min g[L], g[L] = sqrt(L(n-L)/n): this is decided from the table (first for 32
//           lengths at once, then per unit) without reading a prefix sum.  Surviving units go through
//           a per-warp queue so that all 32 lanes examine arcs: one DADD (S_j - S_i) and one integer
//           max of the high word per arc against per-length thresholds in registers; a hit (rare)
//           re-evaluates the unit exactly as fac*s*s and raises the level.
// The set of arcs considered per block pair is exactly the reference's (its restricted
// length ranges [lenlo,lenmax] and [n-lenmax,lenhi], CBS.cpp:179-215), so the maximum is the
// same double; ties for the observed scan follow the reference's visiting order.
// ------------------------------------------------------------------------------------
struct ScanSmem {
    double level;     // prune level (monotone, atomicMax)
    double sms;       // sqrt(level)*(1-1e-12) (monotone)
    double found;     // best statistic found (perm mode)
    // LOC record (observed scan): best arc under the reference's visiting order
    double r_stat, r_corner;
    int r_q, r_key, r_i, r_j;
    int lock;
    int next_pair;
    double red[8];
    double g_min, g_max;  // global extrema of the prefix sums (0.0 unless below / above it)
    int g_imin, g_imax;
    int n_list, pop;      // list of block pairs that reach the level: entries / next entry to scan
    // decision mode, early exit: the reject decision is f(max) >= thresh with f(M) = M/((tss-M)/(n-2)); every floating
    // point operation in f is monotone in M, so the COMPUTED f is non-decreasing while M + 0.0001 < tss (beyond, the
    // reference replaces tss).  Once an arc with f(stat) >= thresh is found the permutation rejects whatever the
    // maximum is -- provided no arc of the row can get within 0.0001 of tss, which pass 1 establishes from the pair bounds.
    double rej_at;        // smallest statistic known to reject (+inf when the early exit is off)
    int decided;
};

struct Cand {
    double stat, corner;
    int q, key, i, j;
};
// true if a precedes b: larger statistic, else earlier in the reference's visiting order
__device__ __forceinline__ bool cand_better(const Cand& a, const Cand& b) {
    if (a.stat != b.stat) return a.stat > b.stat;
    if (a.corner != b.corner) return a.corner > b.corner;
    if (a.q != b.q) return a.q > b.q;
    if (a.key != b.key) return a.key < b.key;
    return a.i < b.i;
}

#define SCAN_QUEUE 256  // per-warp ring of surviving units (entries)
#define SCAN_GRING 64   // per-warp ring of surviving groups of 128 arc lengths (entries)
#define SCAN_LIST 2048  // per-CTA list of block pairs that reach the level (entries)
#define SCAN_LSMALL 128 // arcs shorter than this are swept row by row over the whole segment, not pair by pair
#define PCODE_FLAT 0xffffffffu  // unit of the short-arc sweep: the block pair is looked up per arc

struct PairGeo {
    int ilo, ihi, jlo, jhi;
    int lenlo, lenhi;
    int bandLo[2], bandHi[2];  // arc-length bands actually scanned (empty if lo > hi)
    double corner;
    int q;
};

__device__ __forceinline__ void pair_from_index(int q, int nb, int& bi, int& bj) {
    // rows bi = 1..nb, row r (0-based) starts at r*nb - r*(r-1)/2
    // single precision estimate (all quantities are integers below 2^24), corrected exactly below
    const float t = 2.0f * (float)nb + 1.0f;
    int r = (int)((t - __fsqrt_rn(t * t - 8.0f * (float)q)) * 0.5f);
    if (r < 0) r = 0;
    if (r > nb - 1) r = nb - 1;
    while (r + 1 <= nb - 1 && (long long)(r + 1) * nb - (long long)(r + 1) * r / 2 <= q) ++r;
    while (r > 0 && (long long)r * nb - (long long)r * (r - 1) / 2 > q) --r;
    const int off = (int)((long long)r * nb - (long long)r * (r - 1) / 2);
    bi = r + 1;
    bj = bi + (q - off);
}

struct ScanCtx {
    int n, nb, al0;
    double rn, half;
    float inv_n_rd;         // 1/n rounded down
    const int* bb;          // smem
    const double* bmin; const double* bmax; const int* amin; const int* amax;  // smem
    const float* tmin; const float* tmax;  // smem: extrema of prefix sums [e << tsh, (e+1) << tsh), rounded outwards
    int tsh;
    const double* sx;       // global, this permutation's prefix sums sx[0..n] (+ SX_PAD finite values)
    const double* gtab; const double* factab;  // global, index by L
    bool loc;
    unsigned long long* slots;  // profiling counters (PROF instantiations only)
    unsigned long long* arcs;
    int slice, nslices;         // observed rows: this CTA's share of the row (1 slice: the whole row)
    unsigned long long* glevel; // observed rows over several slices: the row's level (Task::o_level), else nullptr
};

// corner of a block pair (CBS.cpp:132-155): length of the corner arc and its raw spread
__device__ __forceinline__ void pair_corner(const ScanCtx& c, int bi, int bj, double& s1, double& s2, int& clen) {
    s1 = fabs(c.bmax[bj - 1] - c.bmin[bi - 1]);
    s2 = fabs(c.bmax[bi - 1] - c.bmin[bj - 1]);
    clen = (s1 > s2) ? abs(c.amax[bj - 1] - c.amin[bi - 1]) : abs(c.amin[bj - 1] - c.amax[bi - 1]);
}

__device__ __forceinline__ void pair_lengths(const ScanCtx& c, int bi, int bj, int& ilo, int& ihi, int& jlo, int& jhi,
                                             int& lenlo, int& lenhi) {
    ilo = c.bb[bi - 1] + 1; ihi = c.bb[bi]; jlo = c.bb[bj - 1] + 1; jhi = c.bb[bj];
    lenhi = min(jhi - ilo, c.n - c.al0);
    lenlo = (bi == bj) ? 1 : (jlo - ihi);
    if (lenlo < c.al0) lenlo = c.al0;
}

// can the pair hold an arc of SCAN_LSMALL markers or more at or above the level?  (shorter arcs: sweep_short)
// bound = rn/min(L(n-L)) * (corner spread)^2, division free
__device__ __forceinline__ bool pair_alive(const ScanCtx& c, int bi, int bj, double level) {
    int ilo, ihi, jlo, jhi, lenlo, lenhi;
    pair_lengths(c, bi, bj, ilo, ihi, jlo, jhi, lenlo, lenhi);
    if (lenlo < SCAN_LSMALL) lenlo = SCAN_LSMALL;
    if (lenlo > lenhi) return false;
    double s1, s2; int clen;
    pair_corner(c, bi, bj, s1, s2, clen);
    const double smx = (s1 > s2) ? s1 : s2;
    const double rlo = (double)lenlo, rhi = (double)lenhi;
    const double a = rlo * (c.rn - rlo), b2 = rhi * (c.rn - rhi);
    const double mn = (b2 < a) ? b2 : a;
    return c.rn * smx * smx >= level * mn * (1.0 - 1e-12);
}

// block (1-based) that holds prefix index i, 1 <= i <= n
__device__ __forceinline__ int block_of(const ScanCtx& c, int i) {
    int lo = 0, hi = c.nb;  // bb[lo] < i <= bb[hi]
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (c.bb[mid] < i) lo = mid; else hi = mid;
    }
    return hi;
}

// geometry of a block pair: blocks, tie-break data and the two arc-length bands (CBS.cpp:179-180, 198-199)
__device__ __forceinline__ void pair_geometry(const ScanCtx& c, int bi, int bj, PairGeo& g, bool loc) {
    pair_lengths(c, bi, bj, g.ilo, g.ihi, g.jlo, g.jhi, g.lenlo, g.lenhi);
    // position of the pair in the reference's enumeration (row bi, then bj): the tie-break key of LOC mode
    g.q = (bi - 1) * c.nb - ((bi - 1) * (bi - 2)) / 2 + (bj - bi);
    double s1, s2; int clen;
    pair_corner(c, bi, bj, s1, s2, clen);
    g.corner = 0.0;
    if (loc) g.corner = c.factab[min(max(clen, 1), c.n - 1)] * ((s1 > s2) ? s1 : s2) * ((s1 > s2) ? s1 : s2);
    int lenmax = clen;
    if (lenmax > c.n - lenmax) lenmax = c.n - lenmax;
    g.bandLo[0] = 1; g.bandHi[0] = 0; g.bandLo[1] = 1; g.bandHi[1] = 0;
    if (((double)g.lenlo <= c.half) && (g.lenlo <= lenmax)) { g.bandLo[0] = g.lenlo; g.bandHi[0] = lenmax; }
    const int lenmax2 = c.n - lenmax;
    if (((double)g.lenhi >= c.half) && (g.lenhi >= lenmax2)) { g.bandLo[1] = lenmax2; g.bandHi[1] = g.lenhi; }
}

// exact re-evaluation of one unit (slow path): rows i0..i0+31, arc lengths L0..L0+7.  A unit of a block pair is
// restricted to the pair's blocks and to the band of its side; a unit of the short-arc sweep (PCODE_FLAT) looks
// the pair of every arc up and keeps the arc only if its length lies in one of that pair's bands.
template <bool OBS>
__device__ void scan_unit_exact(const ScanCtx& c, unsigned pcode, int i0, int L0, double sms, ScanSmem* sm) {
    const bool flat = pcode == PCODE_FLAT;
    const bool loc = OBS && c.loc;
    PairGeo g;
    int side = 0, La, Lb, ia, ib, cbi = -1, cbj = -1;
    if (!flat) {
        side = (int)(pcode & 1u);
        pair_geometry(c, (int)(pcode >> 16), (int)((pcode >> 1) & 0x7fffu), g, loc);
        La = max(g.bandLo[side], SCAN_LSMALL); Lb = g.bandHi[side];
        ia = max(i0, g.ilo); ib = min(i0 + 31, g.ihi);
    } else {
        La = c.al0; Lb = min(c.n - c.al0, SCAN_LSMALL - 1);
        ia = max(i0, 1); ib = min(i0 + 31, c.n);
        g.jlo = 1; g.jhi = c.n;
    }
    double best = 0.0;
    double th[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int L = L0 + r;
        th[r] = (L >= La && L <= Lb) ? sms * c.gtab[L] : __longlong_as_double(0x7ff0000000000000LL);
    }
    Cand cb; cb.stat = -1.0; cb.corner = 0.0; cb.q = 0; cb.key = 0; cb.i = 0; cb.j = 0;
    for (int i = ia; i <= ib; ++i) {
        const double a = c.sx[i];
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int L = L0 + r, j = i + L;
            if (L < La || L > Lb) continue;
            if (flat ? (j > c.n) : (j < g.jlo || j > g.jhi)) continue;
            const double s = fabs(c.sx[j] - a);
            if (!(s > th[r])) continue;
            if (flat) {
                const int bi = block_of(c, i), bj = block_of(c, j);
                if (bi != cbi || bj != cbj) { pair_geometry(c, bi, bj, g, loc); cbi = bi; cbj = bj; }
                if (L >= g.bandLo[0] && L <= g.bandHi[0]) side = 0;
                else if (L >= g.bandLo[1] && L <= g.bandHi[1]) side = 1;
                else continue;  // not an arc the reference evaluates
            }
            const double stat = c.factab[L] * s * s;  // CBS.cpp:191-193
            if (!loc) { if (stat > best) best = stat; }
            else {
                Cand x;
                x.stat = stat; x.corner = g.corner; x.q = g.q;
                x.key = side ? (0x40000000 + (c.n - L)) : L;  // low side: L ascending; high side: L descending
                x.i = i; x.j = j;
                if (cb.stat < 0.0 || cand_better(x, cb)) cb = x;
            }
        }
    }
    if (!loc) {
        if (best > 0.0) {
            if (best >= sm->rej_at) sm->decided = 1;
            atomic_max_pos_double(&sm->found, best);
            atomic_max_pos_double(&sm->level, best);
            atomic_max_pos_double(&sm->sms, sqrt(best) * (1.0 - 1e-12));
            if (OBS && c.glevel) atomicMax(c.glevel, (unsigned long long)__double_as_longlong(best));
        }
    } else if (cb.stat >= 0.0) {
        bool done = false;
        while (!done) {
            if (atomicCAS(&sm->lock, 0, 1) == 0) {
                Cand r;
                r.stat = sm->r_stat; r.corner = sm->r_corner; r.q = sm->r_q; r.key = sm->r_key; r.i = sm->r_i; r.j = sm->r_j;
                if (cand_better(cb, r)) {
                    sm->r_stat = cb.stat; sm->r_corner = cb.corner; sm->r_q = cb.q; sm->r_key = cb.key; sm->r_i = cb.i; sm->r_j = cb.j;
                }
                __threadfence_block();
                atomicExch(&sm->lock, 0);
                done = true;
            }
        }
        atomic_max_pos_double(&sm->level, cb.stat);
        atomic_max_pos_double(&sm->sms, sqrt(cb.stat) * (1.0 - 1e-12));
        if (OBS && c.glevel) atomicMax(c.glevel, (unsigned long long)__double_as_longlong(cb.stat));
    }
}

// observed row over several slices: take over the level another slice of the row has reached (a value some arc attains,
// so the arcs that attain the maximum are still examined by the slice that owns them)
template <bool OBS>
__device__ __forceinline__ void join_level(const ScanCtx& c, ScanSmem* sm) {
    if (!OBS || !c.glevel) return;
    const double g = __longlong_as_double((long long)*((volatile unsigned long long*)c.glevel));
    if (g > *((volatile double*)&sm->level)) {
        atomic_max_pos_double(&sm->level, g);
        atomic_max_pos_double(&sm->sms, sqrt(g) * (1.0 - 1e-12));
    }
}

// lower bound (single precision, every operation rounded down) of g[L] = sqrt(L(n-L)/n); L, n-L < 2^24 are exact
__device__ __forceinline__ float g_lower(const ScanCtx& c, int L) {
    return __fsqrt_rd(__fmul_rd(__fmul_rd((float)L, (float)(c.n - L)), c.inv_n_rd));
}
// lower bound of min g[L] over L in [l0, l1]: g increases up to n/2 and decreases behind it
__device__ __forceinline__ float g_lower_min(const ScanCtx& c, int l0, int l1) {
    if (2 * l1 <= c.n) return g_lower(c, l0);
    if (2 * l0 >= c.n) return g_lower(c, l1);
    return fminf(g_lower(c, l0), g_lower(c, l1));
}
// upper bound of max |S_j - S_i| over i in the aligned row starting at i0 and j in [js, je], from the table
__device__ __forceinline__ float window_bound(const ScanCtx& c, int i0, int js, int je) {
    const int re = i0 >> c.tsh;
    const float rmin = c.tmin[re], rmax = c.tmax[re];
    const int e1 = min(je, c.n) >> c.tsh;
    int e = js >> c.tsh;
    float wmin = c.tmin[e], wmax = c.tmax[e];
    for (++e; e <= e1; ++e) { wmin = fminf(wmin, c.tmin[e]); wmax = fmaxf(wmax, c.tmax[e]); }
    return fmaxf(__fsub_ru(wmax, rmin), __fsub_ru(rmax, wmin));
}

// per-warp ring of units that survived the pruning tests; it lives across the pairs of a permutation so that the
// arcs are (almost) always examined by 32 busy lanes
struct UnitQueue {
    int* q;             // SCAN_QUEUE x (unit code, pair code)
    unsigned head, n;   // entries [head, head+n)
};

// examine the arcs of one queued unit (fast path): rows i0..i0+31 x lengths L0..L0+7, 4 steps of 8 rows x 8 lengths
// from registers.  Nothing is clipped here: arcs outside the pair's blocks or band, and the values behind S_n
// (finite padding), can only produce a spurious hit, which the exact re-evaluation discards.
template <bool OBS>
__device__ __forceinline__ void scan_unit(const ScanCtx& c, unsigned code, unsigned pcode, ScanSmem* sm) {
    const int i0 = (int)(code >> 17) << 5, L0 = (int)(code & 0x1ffffu) << 3;
    // Thresholds for the 8 lengths.  The fast path never compares doubles (DSETP issues at a quarter of the DADD
    // rate on B200): an arc can only beat the level if |S_j - S_i| > th, and then the high word of |S_j - S_i|
    // is >= the high word of th.  Per length the maximum of (hi << 1) (the shift drops the sign) is kept with one
    // integer instruction per arc (VIADDMNMX.U32) next to the DADD.
    const double sms = *((volatile double*)&sm->sms);
    unsigned thk[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const int L = L0 + k;
        const bool in = (L >= c.al0 && L <= c.n - c.al0);
        thk[k] = in ? (((unsigned)__double2hiint(sms * c.gtab[in ? L : 1])) << 1) : 0xffffffffu;
    }
    const double2* pa = reinterpret_cast<const double2*>(c.sx + i0);        // i0 is a multiple of 32,
    const double2* pb = reinterpret_cast<const double2*>(c.sx + i0 + L0);   // L0 of 8: 16-byte aligned
    double w[8], nw[8];
    unsigned m[8];
#pragma unroll
    for (int k = 0; k < 4; ++k) { const double2 v = __ldg(pb + k); w[2 * k] = v.x; w[2 * k + 1] = v.y; }
#pragma unroll
    for (int k = 0; k < 8; ++k) m[k] = 0u;
#pragma unroll
    for (int it = 0; it < 4; ++it) {
        double av[8];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const double2 v = __ldg(pb + 4 * (it + 1) + k); nw[2 * k] = v.x; nw[2 * k + 1] = v.y;
            const double2 u = __ldg(pa + 4 * it + k); av[2 * k] = u.x; av[2 * k + 1] = u.y;
        }
#pragma unroll
        for (int s = 0; s < 8; ++s) {
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const double xv = (s + k < 8) ? w[s + k] : nw[s + k - 8];
                m[k] = max(m[k], ((unsigned)__double2hiint(xv - av[s])) << 1);
            }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) w[k] = nw[k];
    }
    bool flag = false;
#pragma unroll
    for (int k = 0; k < 8; ++k) flag |= (m[k] >= thk[k]);
    if (flag) scan_unit_exact<OBS>(c, pcode, i0, L0, sms, sm);
}

// examine queued units 32 at a time (all of them if `all`)
template <bool OBS>
__device__ __forceinline__ void drain_units(const ScanCtx& c, UnitQueue& uq, ScanSmem* sm, int lane, bool all) {
    while (uq.n >= 32 || (all && uq.n > 0)) {
        const unsigned take = min(uq.n, 32u);
        if (lane < take) {
            const int2 e = *reinterpret_cast<const int2*>(uq.q + 2 * ((uq.head + lane) & (SCAN_QUEUE - 1)));
            scan_unit<OBS>(c, (unsigned)e.x, (unsigned)e.y, sm);
        }
        __syncwarp();
        uq.head += take; uq.n -= take;
    }
}

// Can the arcs with rows [32a, 32a+31] and lengths [L0, L0+width) that belong to the pair and to the band [La, Lb]
// reach the level?  False if there are none, or if the extrema of the values they touch stay below the smallest
// threshold of their lengths.
__device__ __forceinline__ bool group_may_reach(const ScanCtx& c, const PairGeo& g, const ScanSmem* sm, int a, int L0,
                                                int width, int La, int Lb) {
    const int i0 = a << 5;
    const int imin = max(i0, g.ilo), imax = min(i0 + 31, g.ihi);
    const int l0 = max(L0, La), l1 = min(L0 + width - 1, Lb);
    if (l0 > l1 || imax + l1 < g.jlo || imin + l0 > g.jhi) return false;
    const float smsf = __double2float_rd(*((volatile const double*)&sm->sms));
    const float th = __fmul_rd(smsf, g_lower_min(c, l0, l1));
    return !(window_bound(c, i0, i0 + L0, i0 + 31 + L0 + width - 1) < th);
}

// append the surviving units of this lane's 32-length group (bit t of keep4: unit t) to the warp's unit queue
__device__ __forceinline__ void push_units(UnitQueue& uq, unsigned keep4, unsigned code0, unsigned pcode, int lane) {
    const int cnt = __popc(keep4);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
    const int added = __shfl_sync(FULL, incl, 31);
    if (added) {
        const unsigned at = uq.head + uq.n + (unsigned)(incl - cnt);
#pragma unroll
        for (int t = 0; t < 4; ++t)
            if ((keep4 >> t) & 1u)
                *reinterpret_cast<int2*>(uq.q + 2 * ((at + __popc(keep4 & ((1u << t) - 1u))) & (SCAN_QUEUE - 1))) =
                    make_int2((int)(code0 + (unsigned)t), (int)pcode);
        uq.n += (unsigned)added;
        __syncwarp();
    }
}

// Short arcs (length below SCAN_LSMALL) have low thresholds whatever block pair they belong to, so the pair bounds
// cannot discard them; they are swept here over the whole segment, row by row (32 rows x 32 lengths, then units of
// 32 x 8), with the same table tests.  The warps of the CTA (and the slices of an observed row) share the rows.
template <bool OBS, bool PROF>
__device__ void sweep_short(const ScanCtx& c, UnitQueue& uq, ScanSmem* sm, int warp, int nwarps, int lane) {
    PairGeo gs;
    gs.ilo = 1; gs.ihi = c.n; gs.jlo = 1; gs.jhi = c.n;
    const int La = c.al0, Lb = min(c.n - c.al0, SCAN_LSMALL - 1);
    if (La > Lb) return;
    const int ngs = (Lb >> 5) + 1, total = ((c.n >> 5) + 1) * ngs;
    unsigned long long my_arcs = 0, my_slots = 0;
    for (int base = (c.slice * nwarps + warp) * 32; base < total; base += c.nslices * nwarps * 32) {
        if (__any_sync(FULL, *((volatile int*)&sm->decided))) break;  // decision mode: settled
        join_level<OBS>(c, sm);
        const int idx = base + lane;
        unsigned keep4 = 0, code0 = 0;
        if (idx < total) {
            const int a = idx / ngs, Ls = (idx - a * ngs) << 5;
            code0 = ((unsigned)a << 17) | (unsigned)(Ls >> 3);
            if (group_may_reach(c, gs, sm, a, Ls, 32, La, Lb)) {
#pragma unroll
                for (int t = 0; t < 4; ++t)
                    if (group_may_reach(c, gs, sm, a, Ls + 8 * t, 8, La, Lb)) keep4 |= 1u << t;
            }
            if (PROF && keep4) {  // profiling: arcs inside the queued units
                const int i0 = a << 5;
                for (int k = 0; k < 32; ++k) {
                    const int L = Ls + k;
                    if (!((keep4 >> (k >> 3)) & 1u) || L < La || L > Lb) continue;
                    const int ia = max(i0, 1), ib = min(i0 + 31, c.n - L);
                    if (ib >= ia) my_arcs += (unsigned long long)(ib - ia + 1);
                }
                my_slots += 256ull * __popc(keep4);
            }
        }
        push_units(uq, keep4, code0, PCODE_FLAT, lane);
        drain_units<OBS>(c, uq, sm, lane, false);
    }
    if (PROF && my_slots) atomicAdd(c.slots, my_slots);
    if (PROF && my_arcs) atomicAdd(c.arcs, my_arcs);
    __syncwarp();
}

// scan one arc-length band [La, Lb] of a block pair with the whole warp.  The (row, length) plane of the pair is
// refined top down: groups of 32 rows x 128 lengths, then x 32 lengths, then units of 32 x 8; the survivors of
// each level are compacted through small rings in shared memory so that all 32 lanes stay busy at the next level.
template <bool OBS, bool PROF>
__device__ void scan_band(const ScanCtx& c, const PairGeo& g, unsigned pcode, UnitQueue& uq, int* gring, int La, int Lb,
                          ScanSmem* sm, int lane) {
    const int a0 = g.ilo >> 5, nra = (g.ihi >> 5) - a0 + 1;    // aligned rows of 32 positions meeting block i
    const int c0 = La >> 7, ncg = (Lb >> 7) - c0 + 1;          // aligned groups of 128 arc lengths meeting the band
    const int total = nra * ncg;
    unsigned long long my_arcs = 0, my_slots = 0;
    unsigned ghead = 0, gn = 0;   // ring of surviving 128-length groups
    for (int base = 0;; base += 32) {
        const bool more = base < total;
        if (more) {
            const int idx = base + lane;
            bool keep = false;
            unsigned code = 0;
            if (idx < total) {
                const int ar = idx / ncg;
                const int a = a0 + ar, Lc = (c0 + (idx - ar * ncg)) << 7;
                keep = group_may_reach(c, g, sm, a, Lc, 128, La, Lb);
                code = ((unsigned)a << 17) | (unsigned)(Lc >> 3);
            }
            const unsigned mask = __ballot_sync(FULL, keep);
            if (mask) {
                if (keep) gring[(ghead + gn + __popc(mask & ((1u << lane) - 1u))) & (SCAN_GRING - 1)] = (int)code;
                gn += __popc(mask);
                __syncwarp();
            }
        }
        // 8 surviving groups -> 32 groups of 32 lengths, one per lane
        while (gn >= 8 || (!more && gn > 0)) {
            const unsigned gtake = min(gn, 8u);
            unsigned keep4 = 0, code0 = 0;  // surviving 8-length units of this lane's 32-length group
            if ((unsigned)(lane >> 2) < gtake) {
                const unsigned gc = (unsigned)gring[(ghead + (lane >> 2)) & (SCAN_GRING - 1)];
                const int a = (int)(gc >> 17), Ls = ((int)(gc & 0x1ffffu) << 3) + 32 * (lane & 3);
                code0 = ((unsigned)a << 17) | (unsigned)(Ls >> 3);
                if (group_may_reach(c, g, sm, a, Ls, 32, La, Lb)) {
#pragma unroll
                    for (int t = 0; t < 4; ++t)
                        if (group_may_reach(c, g, sm, a, Ls + 8 * t, 8, La, Lb)) keep4 |= 1u << t;
                }
                if (PROF && keep4) {  // profiling: arcs of the pair and band inside the queued units
                    const int i0 = a << 5;
                    for (int k = 0; k < 32; ++k) {
                        const int L = Ls + k;
                        if (!((keep4 >> (k >> 3)) & 1u) || L < La || L > Lb) continue;
                        const int ia = max(max(i0, g.ilo), g.jlo - L), ib = min(min(i0 + 31, g.ihi), g.jhi - L);
                        if (ib >= ia) my_arcs += (unsigned long long)(ib - ia + 1);
                    }
                    my_slots += 256ull * __popc(keep4);
                }
            }
            __syncwarp();
            ghead += gtake; gn -= gtake;
            push_units(uq, keep4, code0, pcode, lane);
            drain_units<OBS>(c, uq, sm, lane, false);
        }
        if (!more) break;
    }
    if (PROF && my_slots) atomicAdd(c.slots, my_slots);
    if (PROF && my_arcs) atomicAdd(c.arcs, my_arcs);
    __syncwarp();
}

// the two bands of one block pair
template <bool OBS, bool PROF>
__device__ void scan_pair(const ScanCtx& c, int bi, int bj, UnitQueue& uq, int* gring, ScanSmem* sm, int lane) {
    PairGeo g;
    pair_geometry(c, bi, bj, g, OBS && c.loc);
    const unsigned pcode = (((unsigned)bi << 15) | (unsigned)bj) << 1;
    // arcs shorter than SCAN_LSMALL are covered by sweep_short
    const int lo0 = max(g.bandLo[0], SCAN_LSMALL), lo1 = max(g.bandLo[1], SCAN_LSMALL);
    if (lo0 <= g.bandHi[0]) scan_band<OBS, PROF>(c, g, pcode, uq, gring, lo0, g.bandHi[0], sm, lane);
    if (lo1 <= g.bandHi[1]) scan_band<OBS, PROF>(c, g, pcode | 1u, uq, gring, lo1, g.bandHi[1], sm, lane);
}

// Slice of an observed row that owns block pair (bi, bj).  Pass 2 enumerates the pairs diagonal by diagonal,
// q = d*nb - d*(d-1)/2 + (bi-1) with d = bj - bi, and deals chunks of 32 consecutive q round-robin over the slices; pass 1
// uses the very same ownership, so every pair belongs to exactly one slice whether or not that slice's list overflows.
__device__ __forceinline__ int pair_slice(int bi, int bj, int nb, int nsl) {
    const int d = bj - bi;
    return ((d * nb - d * (d - 1) / 2 + bi - 1) >> 5) % nsl;
}

// dynamic shared memory layout helper (host + device)
struct ScanLayout {
    int nb_max;   // blocks of the longest segment + 1
    int nt;       // entries of the extrema table
    int tsh;      // log2 of the run of prefix sums one table entry covers
    int warps;
    CBS_HD size_t bytes() const {
        return ((sizeof(ScanSmem) + 15) & ~(size_t)15) + 2 * (size_t)nb_max * 8 + 3 * (size_t)nb_max * 4 + 2 * (size_t)nt * 4 +
               (size_t)warps * (2 * SCAN_QUEUE + SCAN_GRING) * 4 + (size_t)SCAN_LIST * 4 + 64;
    }
    // table geometry for units of up to nmax markers: at most 16384 entries (128 KB)
    CBS_HD void set_table(long long nmax) {
        tsh = 5;
        while (((nmax >> tsh) + 2) > 16384) ++tsh;
        nt = (int)(nmax >> tsh) + 2;
    }
};

// The scan of one kind of row.  OBS = false (k_scan_perm): the permutation rows of the round, one CTA per row, reject
// decision only.  OBS = true (k_scan_obs): the observed rows (one per pending segment planned this round, prefix sums
// written by k_prep), exact maximum and, unless D->obs_noloc, its location; a row is spread over obs_slices(n) CTAs
// (slice-major work list, so that every row starts early) that share the pair list and the short-arc rows, the running
// level (Task::o_level) and, at the end, the best arc (Task::o_*, merged with cand_better, a total order: the result does
// not depend on the order in which slices finish); the last slice to finish writes the result.  PROF: scan work
// counters (D->profile), compiled out of the timed kernels.
template <bool OBS, bool PROF>
__device__ __forceinline__ void scan_rows(Dev* D, const ScanLayout& lay) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (D->done) return;
    ScanSmem* sm = (ScanSmem*)smem_raw;
    double* s_bmin = (double*)(smem_raw + ((sizeof(ScanSmem) + 15) & ~(size_t)15));
    double* s_bmax = s_bmin + lay.nb_max;
    int* s_amin = (int*)(s_bmax + lay.nb_max);
    int* s_amax = s_amin + lay.nb_max;
    int* s_bb = s_amax + lay.nb_max;
    float* s_tmin = (float*)(s_bb + lay.nb_max);
    float* s_tmax = s_tmin + lay.nt;
    int* s_queue = (int*)(((size_t)(s_tmax + lay.nt) + 7) & ~(size_t)7);  // entries are int2
    int* s_list = s_queue + lay.warps * (2 * SCAN_QUEUE + SCAN_GRING);
    __shared__ int s_g, s_last;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int nwarps = blockDim.x >> 5;
    const int n_prep = D->n_prep;
    // observed rows: entry g is slice g / n_prep of row g % n_prep, up to the most slices any row of the round takes; an
    // entry beyond its row's own count is skipped (one counter increment and two barriers).  A per-row prefix would avoid
    // those, but it would be a second array the scheduler fills for every observed row, in every caller of Sched.
    const int total = OBS ? n_prep * (int)D->ctr[CTR_OBS_SLICES] : D->item_prefix[D->n_items];
    const float finf = __int_as_float(0x7f800000);
    for (;;) {
        __syncthreads();
        if (tid == 0) s_g = (int)atomicAdd(&D->ctr[OBS ? CTR_SCAN_OBS : CTR_SCAN_PERM], 1u);
        __syncthreads();
        const int gidx = s_g;
        if (gidx >= total) break;
        int p = 0, slice = 0, nsl = 1, task;
        if (OBS) {
            slice = gidx / n_prep;
            task = D->prep_task[gidx - slice * n_prep];
        } else {
            const int k = find_item(D->item_prefix, D->n_items, gidx);
            const PermItem it = D->items[k];
            if (it.obs) continue;  // k_scan_obs
            task = it.task;
            p = gidx - D->item_prefix[k];
        }
        Task& t = D->tasks[task];
        if (OBS) {
            if (t.alleq) continue;
            nsl = obs_slices(t.n, D->obs_slices);
            if (slice >= nsl) continue;
        } else if (t.use_hybrid) continue;  // k_hscan
        const int n = t.n, nb = t.nb;
        const long long base = D->unit_off[t.unit] + t.lo;
        ScanCtx c;
        c.n = n; c.nb = nb; c.al0 = D->prm.min_width; c.rn = (double)n; c.half = c.rn / 2.0;
        c.inv_n_rd = __frcp_rd((float)n);
        c.bb = s_bb; c.bmin = s_bmin; c.bmax = s_bmax; c.amin = s_amin; c.amax = s_amax;
        c.tmin = s_tmin; c.tmax = s_tmax; c.tsh = lay.tsh;
        c.sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        c.gtab = D->gtab + base; c.factab = D->factab + base;
        c.loc = OBS && !D->obs_noloc;
        const bool decide = !OBS;
        c.slots = PROF ? &D->stat_slots : nullptr;
        c.arcs = PROF ? &D->stat_arcs : nullptr;
        c.slice = slice; c.nslices = nsl;
        c.glevel = nsl > 1 ? &t.o_level : nullptr;
        BlockStats bs(D->arena + t.off_bs + (long long)p * Sched::bs_stride(nb), nb);
        const int* bbg = D->bbtab + base;
        for (int b = tid; b <= nb; b += blockDim.x) s_bb[b] = bbg[b];
        if (OBS) {
            // observed data (one row per pending segment, written by k_prep): the statistics are computed here (by
            // every slice of the row: n * 8 bytes from L2)
            __syncthreads();
        // ---- phase 0a: extrema table.  A warp takes 1024 consecutive prefix sums (coalesced loads); a
            // reduce-scatter over the lanes leaves lane l with the extrema of run l of 32, in single precision
            // rounded outwards; runs are merged 2 or 4 to an entry when the table is coarser (tsh 6, 7).
            for (int c0 = warp * 1024; c0 <= n; c0 += nwarps * 1024) {
                float lo[32], hi[32];
    #pragma unroll
                for (int r = 0; r < 32; ++r) {
                    const int e = c0 + 32 * r + lane;
                    if (e <= n) { const double v = c.sx[e]; lo[r] = __double2float_rd(v); hi[r] = __double2float_ru(v); }
                    else { lo[r] = finf; hi[r] = -finf; }
                }
    #pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const bool up = (lane & o) != 0;
    #pragma unroll
                    for (int r = 0; r < o; ++r) {
                        const float keep_lo = up ? lo[r + o] : lo[r], send_lo = up ? lo[r] : lo[r + o];
                        const float keep_hi = up ? hi[r + o] : hi[r], send_hi = up ? hi[r] : hi[r + o];
                        lo[r] = fminf(keep_lo, __shfl_xor_sync(FULL, send_lo, o));
                        hi[r] = fmaxf(keep_hi, __shfl_xor_sync(FULL, send_hi, o));
                    }
                }
                float l0 = lo[0], h0 = hi[0];
                for (int sft = 5; sft < lay.tsh; ++sft) {
                    const int o = 1 << (sft - 5);
                    l0 = fminf(l0, __shfl_xor_sync(FULL, l0, o));
                    h0 = fmaxf(h0, __shfl_xor_sync(FULL, h0, o));
                }
                const int per = 1 << (lay.tsh - 5);  // runs per entry
                if ((lane & (per - 1)) == 0 && c0 + 32 * lane <= n) {
                    const int e = (c0 + 32 * lane) >> lay.tsh;
                    s_tmin[e] = l0; s_tmax[e] = h0;
                }
            }
            __syncthreads();
            // ---- phase 0b: per-block extrema with their FIRST occurrence (CBS.cpp:88-94): a warp per block
            for (int b = warp; b < nb; b += nwarps) {
                const int first = s_bb[b] + 1, last = s_bb[b + 1];
                double lo = __longlong_as_double(0x7ff0000000000000LL), hi = -lo;
                int ilo = 0x7fffffff, ihi = 0x7fffffff;
                for (int i = first + lane; i <= last; i += 32) {
                    const double v = c.sx[i];
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
        } else {
            // ---- phase 0: the statistics of the row were written next to it by k_chain: the extrema of every
            // aligned run of 32 prefix sums (merged 2 or 4 to an entry when the table is coarser) and the per-block
            // extrema with their first occurrence (CBS.cpp:88-94)
            {
                const float* gmin = (const float*)(c.sx + Sched::tbl_offset(n));
                const float* gmax = gmin + Sched::tbl_entries(n);
                const int fine = (n >> 5) + 1, per = 1 << (lay.tsh - 5);
                for (int e = tid; e <= (n >> lay.tsh); e += blockDim.x) {
                    float lo = finf, hi = -finf;
                    for (int r = 0; r < per; ++r) {
                        const int f = e * per + r;
                        if (f < fine) { lo = fminf(lo, gmin[f]); hi = fmaxf(hi, gmax[f]); }
                    }
                    s_tmin[e] = lo; s_tmax[e] = hi;
                }
                for (int b2 = tid; b2 < nb; b2 += blockDim.x) {
                    s_bmin[b2] = bs.bmin()[b2]; s_bmax[b2] = bs.bmax()[b2]; s_amin[b2] = bs.amin()[b2]; s_amax[b2] = bs.amax()[b2];
                }
            }
            __syncthreads();
        }
        // global extrema: the first block that attains the overall minimum / maximum, and only if it is
        // below / above 0.0 (CBS.cpp:80-81, 93-94)
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
                sm->n_list = 0;
                sm->decided = 0; sm->rej_at = __longlong_as_double(0x7ff0000000000000LL);
            }
        }
        __syncthreads();
        const double gmin = sm->g_min, gmax = sm->g_max;
        const int gimin = sm->g_imin, gimax = sm->g_imax;
        const double spread = gmax - gmin;
        const double tss0 = t.tss;
        double final_best;
        int fi = min(gimax, gimin), fj = max(gimax, gimin);
        if (spread <= 0.0) {  // CBS.cpp:102-111
            final_best = -1.0;
            if (OBS && slice != 0) continue;  // every slice of the row gets here: slice 0 writes the result
        } else {
            // CBS.cpp:113-117 initial candidate: global extrema of the prefix sums
            const double rj = (double)abs(gimax - gimin);
            const double init = c.rn / (rj * (c.rn - rj)) * spread * spread;
            // ---- pass 1: best valid corner -> lower bound; the pairs whose bound reaches a provisional level (the
            // level before the corners are known) are appended to the pair list on the way, so that the pairs are
            // normally enumerated once.  Thread t takes pairs t, t+256, ... and steps (bi, bj) incrementally.
            const int npairs = nb * (nb + 1) / 2;
            double prov = init;
            if (decide) {
                const double thresh = t.ostat * 0.99999;
                const double mstar = thresh * tss0 / (c.rn - 2.0 + thresh) * (1.0 - 1e-9);
                if (mstar > prov && mstar + 0.001 < tss0 && mstar / ((tss0 - mstar) / (c.rn - 2.0)) < thresh) prov = mstar;
            }
            double lb = 0.0;
            // early exit of decision mode needs max + 0.0001 < tss for every arc of the row: rn*smx^2/min(L(n-L)) bounds
            // the arcs of a pair, so  rn*smx^2 < ublim*min(L(n-L))  for all pairs (division free) establishes it
            const double ublim = (tss0 - 0.001) * (1.0 - 1e-9);
            bool ub_ok = decide && !D->no_early && init + 0.001 < tss0;
            {
                int bi = 1, bj = 1;
                if (tid < npairs) pair_from_index(tid, nb, bi, bj);
                for (int q0 = 0; q0 < npairs; q0 += blockDim.x) {
                    const int q = q0 + tid;
                    bool alive = false;
                    if (q < npairs) {
                        double s1, s2; int clen;
                        pair_corner(c, bi, bj, s1, s2, clen);
                        const double smx = (s1 > s2) ? s1 : s2;
                        if (clen >= c.al0 && clen <= n - c.al0) {
                            // fac[clen] recomputed (same expression as the table: one division instead of an L2 round trip)
                            const double rr = (double)clen;
                            const double v = c.rn / (rr * (c.rn - rr)) * smx * smx;
                            if (v > lb) lb = v;
                        }
                        int ilo, ihi, jlo, jhi, lenlo, lenhi;
                        pair_lengths(c, bi, bj, ilo, ihi, jlo, jhi, lenlo, lenhi);
                        if (ub_ok && lenlo <= lenhi) {
                            const double rlo = (double)lenlo, rhi = (double)lenhi;
                            const double a = rlo * (c.rn - rlo), b2 = rhi * (c.rn - rhi);
                            if (!(c.rn * smx * smx < ublim * ((b2 < a) ? b2 : a))) ub_ok = false;
                        }
                        if (lenlo < SCAN_LSMALL) lenlo = SCAN_LSMALL;
                        if (lenlo <= lenhi) {
                            const double rlo = (double)lenlo, rhi = (double)lenhi;
                            const double a = rlo * (c.rn - rlo), b2 = rhi * (c.rn - rhi);
                            alive = c.rn * smx * smx >= prov * ((b2 < a) ? b2 : a) * (1.0 - 1e-12);
                        }
                        if (OBS && nsl > 1 && pair_slice(bi, bj, nb, nsl) != slice) alive = false;  // another slice's pair
                    }
                    const unsigned mask = __ballot_sync(FULL, alive);
                    if (mask) {
                        int at = 0;
                        if (lane == 0) at = atomicAdd(&sm->n_list, __popc(mask));
                        at = __shfl_sync(FULL, at, 0) + __popc(mask & ((1u << lane) - 1u));
                        if (alive && at < SCAN_LIST) s_list[at] = (bi << 16) | bj;
                    }
                    // advance by blockDim.x pairs: row bi holds bj = bi..nb
                    bj += blockDim.x;
                    while (bj > nb && bi <= nb) { const int excess = bj - nb; ++bi; bj = bi - 1 + excess; }
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) { const double o2 = shfl_d(lb, lane ^ o); if (o2 > lb) lb = o2; }
            if (lane == 0) sm->red[warp] = lb;
            const int ub_all = __syncthreads_and(ub_ok ? 1 : 0);
            if (tid == 0) {
                double m = init;
                for (int w = 0; w < nwarps; ++w) if (sm->red[w] > m) m = sm->red[w];
                sm->rej_at = __longlong_as_double(0x7ff0000000000000LL);
                sm->decided = 0;
                if (decide && ub_all) {
                    const double thresh = t.ostat * 0.99999;
                    const double ra = thresh * tss0 / (c.rn - 2.0 + thresh) * (1.0 + 1e-9);
                    if (ra > 0.0 && ra + 0.001 < tss0 && ra / ((tss0 - ra) / (c.rn - 2.0)) >= thresh) {
                        sm->rej_at = ra;
                        if (m >= ra) sm->decided = 1;  // the seed arc or the best valid corner already rejects
                    }
                }
                if (OBS && c.glevel) {  // publish the row's lower bound, then join the level the other slices reached
                    atomicMax(c.glevel, (unsigned long long)__double_as_longlong(m));
                    const double gl = __longlong_as_double((long long)*((volatile unsigned long long*)c.glevel));
                    if (gl > m) m = gl;
                }
                double level = m;
                if (decide) {
                    // decision mode: only arcs that could make this permutation reject matter.
                    // reject <=> thresh <= f(M), f(M) = M/((tss-M)/(n-2)) increasing for M < tss-1e-4
                    const double thresh = t.ostat * 0.99999;
                    const double mstar = thresh * tss0 / (c.rn - 2.0 + thresh) * (1.0 - 1e-9);
                    if (mstar > level && mstar + 0.001 < tss0) {
                        const double f = mstar / ((tss0 - mstar) / (c.rn - 2.0));
                        if (f < thresh) level = mstar;
                    }
                }
                sm->level = level;
                sm->sms = sqrt(level) * (1.0 - 1e-12);
                sm->found = init;
                sm->r_stat = init; sm->r_corner = __longlong_as_double(0x7ff0000000000000LL);
                sm->r_q = 0x7fffffff; sm->r_key = -1; sm->r_i = fi; sm->r_j = fj;
                sm->lock = 0; sm->pop = 0;
                // the list is complete unless it overflowed: then pass 2 enumerates the pairs again, list by list
                // (next_pair counts this slice's pairs: chunk q0 of the slice is q0 * nsl + 32 * slice of the row)
                if (sm->n_list > SCAN_LIST) { sm->n_list = 0; sm->next_pair = 0; } else sm->next_pair = npairs;
            }
            __syncthreads();
            // ---- pass 2: scan surviving block pairs ----------------------------------------
            // (a) the warps evaluate the pair bounds 32 pairs at a time and append the pairs that reach the level to
            // a list in shared memory; (b) the warps pop ONE pair at a time and scan it, so that the load is balanced
            // at the grain of a pair.  Repeated while pairs remain (the list is bounded).
            UnitQueue uq;
            uq.q = s_queue + warp * (2 * SCAN_QUEUE + SCAN_GRING);
            uq.head = 0; uq.n = 0;
            int* gring = uq.q + 2 * SCAN_QUEUE;
            const bool settled = sm->decided != 0;  // uniform: written before the barrier above
            if (!settled) sweep_short<OBS, PROF>(c, uq, sm, warp, nwarps, lane);
            for (; !settled;) {
                for (;;) {
                    if (*((volatile int*)&sm->n_list) > SCAN_LIST - 32 * nwarps) break;  // every warp may still add 32
                    int q0 = 0;
                    if (lane == 0) q0 = atomicAdd(&sm->next_pair, 32);
                    q0 = __shfl_sync(FULL, q0, 0) * nsl + 32 * slice;
                    if (q0 >= npairs) break;
                    // pairs are enumerated diagonal by diagonal (bj - bi = 0, 1, 2, ...): the pairs with the longest
                    // arc-length bands come first
                    const int q = q0 + lane;
                    bool alive = false;
                    int bi = 1, bj = 1;
                    if (q < npairs) {
                        int da, db; pair_from_index(q, nb, da, db);
                        bi = db - da + 1; bj = bi + (da - 1);
                        alive = pair_alive(c, bi, bj, *((volatile double*)&sm->level));
                    }
                    const unsigned mask = __ballot_sync(FULL, alive);
                    if (mask) {
                        int at = 0;
                        if (lane == 0) at = atomicAdd(&sm->n_list, __popc(mask));
                        at = __shfl_sync(FULL, at, 0);
                        if (alive) s_list[at + __popc(mask & ((1u << lane) - 1u))] = (bi << 16) | bj;
                    }
                }
                __syncthreads();
                const int n_list = sm->n_list;
                for (;;) {
                    int w = 0;
                    if (lane == 0) w = atomicAdd(&sm->pop, 1);
                    w = __shfl_sync(FULL, w, 0);
                    if (w >= n_list) break;
                    if (__any_sync(FULL, *((volatile int*)&sm->decided))) break;  // decision mode: settled
                    const int code = s_list[w];
                    const int bi = code >> 16, bj = code & 0xffff;
                    join_level<OBS>(c, sm);
                    if (!pair_alive(c, bi, bj, *((volatile double*)&sm->level))) continue;  // the level may have risen
                    scan_pair<OBS, PROF>(c, bi, bj, uq, gring, sm, lane);
                }
                drain_units<OBS>(c, uq, sm, lane, true);  // the level may still rise: flush before the next list
                __syncthreads();
                const bool finished = (long long)sm->next_pair * nsl + 32 * slice >= npairs || sm->decided;
                __syncthreads();
                if (finished) break;
                if (tid == 0) { sm->n_list = 0; sm->pop = 0; }
                __syncthreads();
            }
            __syncthreads();
            final_best = c.loc ? sm->r_stat : sm->found;
            if (c.loc) { fi = sm->r_i; fj = sm->r_j; }
            if (OBS && nsl > 1) {
                // merge this slice's result into the row's record; the last slice to finish writes the result
                if (tid == 0) {
                    if (c.loc) {
                        Cand mine;
                        mine.stat = sm->r_stat; mine.corner = sm->r_corner; mine.q = sm->r_q; mine.key = sm->r_key;
                        mine.i = sm->r_i; mine.j = sm->r_j;
                        while (atomicCAS(&t.o_lock, 0, 1) != 0) {}
                        __threadfence();
                        const volatile Task& vt = t;
                        Cand cur;
                        cur.stat = vt.o_stat; cur.corner = vt.o_corner; cur.q = vt.o_q; cur.key = vt.o_key; cur.i = vt.o_i; cur.j = vt.o_j;
                        if (!vt.o_set || cand_better(mine, cur)) {
                            t.o_stat = mine.stat; t.o_corner = mine.corner; t.o_q = mine.q; t.o_key = mine.key;
                            t.o_i = mine.i; t.o_j = mine.j; t.o_set = 1;
                        }
                        __threadfence();
                        atomicExch(&t.o_lock, 0);
                    } else {
                        atomicMax(&t.o_found, (unsigned long long)__double_as_longlong(sm->found));
                    }
                    __threadfence();
                    const int last = atomicAdd(&t.o_done, 1) == nsl - 1;
                    if (last) {
                        __threadfence();
                        const volatile Task& vt = t;
                        if (c.loc) { final_best = vt.o_stat; fi = vt.o_i; fj = vt.o_j; }
                        else final_best = __longlong_as_double((long long)vt.o_found);
                    }
                    s_last = last;
                }
                __syncthreads();
                if (!s_last) continue;
            }
        }
        if (tid == 0) {
            double tss = tss0, stat;
            if (final_best < 0.0) {
                if (tss <= 0.0001) tss = 1.0;
                stat = 0.0 / ((tss - 0.0) / (c.rn - 2.0));
            } else {  // CBS.cpp:221-223
                if (tss <= final_best + 0.0001) tss = final_best + 1.0;
                stat = final_best / ((tss - final_best) / (c.rn - 2.0));
            }
            if (!OBS) D->rej[t.off_rej + p] = (sm->decided || t.ostat * 0.99999 <= stat) ? 1 : 0;  // CBS.cpp:838,863
            else if (c.loc) { t.ostat = stat; t.tmaxi = fi; t.tmaxj = fj; }
            else t.ostat = stat;
            bs.result() = stat;
        }
    }
}

template <bool PROF>
__global__ void __launch_bounds__(256, 3) k_scan_perm(Dev* D, ScanLayout lay) { scan_rows<false, PROF>(D, lay); }
template <bool PROF>
__global__ void __launch_bounds__(256, 2) k_scan_obs(Dev* D, ScanLayout lay) { scan_rows<true, PROF>(D, lay); }

// ------------------------------------------------------------------------------------
// hybrid p-values (DNAcopy's default method; `cna segment --hybrid true`)
//   k_tailp : analytic tail probability of the observed statistic for arcs longer than kmax
//             (tailp/nu/it1tsq/fpnorm, CBS.cpp:14-51, :324-339), one thread per new segment.  Uses the
//             CUDA double-precision erfc/log/exp/pow (<= 4 ulp), so pval1 agrees with the reference's
//             libm value to ~1e-15 relative, not bit for bit.
//   k_hscan : htmaxp (CBS.cpp:387-485) for one permutation per CTA.  htmaxp's pruning only skips arcs
//             that cannot exceed the running maximum, so its value is the exact maximum of
//             fac(j)*d*d over ALL arcs of length al0..k (inside its ~k-wide blocks, straddling
//             adjacent blocks, and wrapping around the end), plus the per-block (argmin,argmax)
//             candidates, which use the other rounding fac*(d*d) (:415-416).  It is evaluated
//             here by brute force, 25 arcs per marker.
// ------------------------------------------------------------------------------------
__device__ double dev_fpnorm(double x) { return 0.5 * erfc(-x / sqrt(2.0)); }
__device__ double dev_nu(double x, double tol) {
    if (x > 0.01) {
        double lnu1 = log(2.0) - 2.0 * log(x);
        double lnu0 = lnu1;
        int k = 2;
        double dk = 0.0;
        for (int i = 1; i <= k; ++i) { dk += 1.0; lnu1 -= 2.0 * dev_fpnorm(-x * sqrt(dk) / 2.0) / dk; }
        while (fabs((lnu1 - lnu0) / lnu1) > tol) {
            lnu0 = lnu1;
            for (int i = 1; i <= k; ++i) { dk += 1.0; lnu1 -= 2.0 * dev_fpnorm(-x * sqrt(dk) / 2.0) / dk; }
            k *= 2;
            if (k > (1 << 24)) break;
        }
        return exp(lnu1);
    }
    return exp(-0.583 * x);
}
__device__ double dev_it1tsq(double x, double a) {
    double y = x + a - 0.5;
    double out = (8.0 * y) / (1.0 - 4.0 * y * y) + 2.0 * log((1.0 + 2.0 * y) / (1.0 - 2.0 * y));
    y = x - 0.5;
    out -= (8.0 * y) / (1.0 - 4.0 * y * y) + 2.0 * log((1.0 + 2.0 * y) / (1.0 - 2.0 * y));
    return out;
}
// nu() (CBS.cpp:18-41) by a whole warp: the terms 2*Phi(-x*sqrt(dk)/2)/dk of the series are evaluated 32 at a time
// (dk is an exact integer, so lane l evaluates the very expression the sequential loop would), and subtracted from
// lnu1 in the sequential order by every lane (the value stays uniform over the warp).
__device__ double warp_nu(double x, double tol, int lane) {
    if (!(x > 0.01)) return exp(-0.583 * x);
    double lnu1 = log(2.0) - 2.0 * log(x);
    double lnu0 = lnu1;
    long long done = 0;  // terms subtracted so far (= dk)
    auto take = [&](int k) {  // the next k terms
        for (int c0 = 0; c0 < k; c0 += 32) {
            const int cnt = min(32, k - c0);
            const double dk = (double)(done + lane + 1);
            const double term = (lane < cnt) ? 2.0 * dev_fpnorm(-x * sqrt(dk) / 2.0) / dk : 0.0;
            for (int q = 0; q < cnt; ++q) lnu1 -= shfl_d(term, q);
            done += cnt;
        }
    };
    int k = 2;
    take(k);
    while (fabs((lnu1 - lnu0) / lnu1) > tol) {
        lnu0 = lnu1;
        take(k);
        k *= 2;
        if (k > (1 << 24)) break;
    }
    return exp(lnu1);
}

// tailp (CBS.cpp:324-339).  k_tailp_terms: a warp per quadrature point (ngrid = 100 per segment; a point's nu() series
// has up to ~1e6 terms for the small x of SNP6-scale segments); k_tailp_sum: the terms are added in the reference's order.
#define TAILP_NGRID 100
__global__ void __launch_bounds__(128) k_tailp_terms(Dev* D, double* terms) {
    if (D->done || !D->prm.hybrid) return;
    const int lane = threadIdx.x & 31;
    const int total = D->n_prep * TAILP_NGRID;
    for (int w = blockIdx.x * 4 + (threadIdx.x >> 5); w < total; w += gridDim.x * 4) {
        const int k = w / TAILP_NGRID, i = w - k * TAILP_NGRID + 1;  // quadrature point i = 1..ngrid of prep task k
        const Task& t = D->tasks[D->prep_task[k]];
        if (!t.use_hybrid || t.alleq) continue;
        const double b = sqrt(t.ostat);
        if (!(b > 0.1) && D->api_mode != 4) continue;  // (cbs::tailp itself has no such shortcut: api_mode 4)
        const double delta = D->w ? t.w_delta : (D->api_mode && D->api_delta > 0.0) ? D->api_delta
                                                : (double)(D->prm.kmax + 1) / (double)t.n;  // CBS.cpp:984; weighted: getmncwt (:908)
        const double dincr = (0.5 - delta) / (double)TAILP_NGRID;
        const double bsqrtm = b / sqrt((double)t.n);
        // tl and t after i increments of dincr, accumulated as the reference does (repeated addition)
        double tl = 0.5 - dincr, tt = 0.5 - 0.5 * dincr;
        for (int q = 0; q < i; ++q) { tl += dincr; tt += dincr; }
        const double x = bsqrtm / sqrt(tt * (1.0 - tt));
        const double nux = warp_nu(x, D->prm.tol, lane);
        if (lane == 0) terms[(long long)k * TAILP_NGRID + (i - 1)] = (nux * nux) * dev_it1tsq(tl, dincr);
    }
}
__global__ void __launch_bounds__(64) k_tailp_sum(Dev* D, const double* terms) {
    if (D->done || !D->prm.hybrid) return;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < D->n_prep; k += gridDim.x * blockDim.x) {
        Task& t = D->tasks[D->prep_task[k]];
        if (!t.use_hybrid || t.alleq) continue;
        const double b = sqrt(t.ostat);
        if (!(b > 0.1) && D->api_mode != 4) { t.pval1 = 1.0; continue; }
        double out = 0.0;
        for (int q = 0; q < TAILP_NGRID; ++q) out += terms[(long long)k * TAILP_NGRID + q];
        out = 9.973557e-2 * pow(b, 3.0) * exp(-b * b / 2.0) * out;
        t.pval1 = 2.0 * out;
    }
}

// cbs::btailp (CBS.cpp:341-361): nu(x1)/x at the ng+1 quadrature points, a warp per point (x advances by repeated addition
// as in the reference), then the trapezoid sum in order.  Off the `cna segment` path (binary data).
__global__ void __launch_bounds__(128) k_btailp_terms(double b, int m, int ng, double tol, double* vals) {
    const int lane = threadIdx.x & 31;
    const double dm = (double)m;
    const double ll = b * sqrt(1.0 / (double)(m - 2) - 1.0 / dm);
    const double ul = b * sqrt(1.0 / 2.0 - 1.0 / dm);
    const double dincr = (ul - ll) / (double)ng;
    for (int i = blockIdx.x * 4 + (threadIdx.x >> 5); i <= ng; i += gridDim.x * 4) {
        double x = ll;
        for (int q = 0; q < i; ++q) x += dincr;
        const double x1 = x + (b * b) / (dm * x);
        const double v = warp_nu(x1, tol, lane) / x;
        if (lane == 0) vals[i] = v;
    }
}
__global__ void k_btailp_sum(double b, int m, int ng, const double* vals, double* out) {
    if (threadIdx.x || blockIdx.x) return;
    const double dm = (double)m;
    const double ll = b * sqrt(1.0 / (double)(m - 2) - 1.0 / dm);
    const double ul = b * sqrt(1.0 / 2.0 - 1.0 / dm);
    const double dincr = (ul - ll) / (double)ng;
    double acc = 0.0, nulo = vals[0];
    for (int i = 1; i <= ng; ++i) { const double nuhi = vals[i]; acc += (nuhi + nulo) * dincr; nulo = nuhi; }
    acc = b * exp(-b * b / 2.0) * acc * 0.39894228040143267794;  // 1/sqrt(2 pi)
    acc += 2.0 * (1.0 - dev_fpnorm(b));
    *out = acc;
}

__global__ void __launch_bounds__(256) k_hscan(Dev* D) {
    __shared__ double s_fac[132];
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
        const double rn = (double)n;
        const double* __restrict__ sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        for (int j = tid; j <= kk && j < 132; j += blockDim.x) {
            const double rj = (double)j;
            s_fac[j] = (j >= 1) ? rn / (rj * (rn - rj)) : 0.0;
        }
        __syncthreads();
        double best = 0.0;
        // all arcs (i, i+j), 1 <= i <= n-j, and the wrap-around arcs i = 1..j against i+n-j
        for (int i = 1 + tid; i <= n; i += blockDim.x) {
            const double si = sx[i];
            for (int j = al0; j <= kk; ++j) {
                double d;
                if (i + j <= n) d = fabs(sx[i + j] - si);
                else continue;
                const double v = s_fac[j] * d * d;
                if (v > best) best = v;
            }
            for (int j = (i > al0 ? i : al0); j <= kk; ++j) {  // wrap: i <= j
                const double d = fabs(sx[i + n - j] - si);
                const double v = s_fac[j] * d * d;
                if (v > best) best = v;
            }
        }
        // per-block (argmin, argmax) candidates of htmaxp's own blocks, nb = int(n/k) (CBS.cpp:390-419)
        const int nbh = (int)(rn / (double)kk);
        for (int b = 1 + tid; b <= nbh; b += blockDim.x) {
            const int first = block_end(n, nbh, b - 1) + 1, last = block_end(n, nbh, b);
            double lo = sx[first], hi = lo;
            int ilo = first, ihi = first;
            for (int i = first + 1; i <= last; ++i) {
                const double v = sx[i];
                if (v < lo) { lo = v; ilo = i; }
                if (v > hi) { hi = v; ihi = i; }
            }
            const int d = abs(ilo - ihi);
            if (d <= kk && d >= al0) {
                const double rj = (double)d;
                const double fac = rn / (rj * (rn - rj));
                const double df = hi - lo;
                const double v = fac * (df * df);
                if (v > best) best = v;
            }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) { const double o2 = shfl_d(best, lane ^ o); if (o2 > best) best = o2; }
        if (lane == 0) s_red[warp] = best;
        __syncthreads();
        if (tid == 0) {
            double m = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) if (s_red[w] > m) m = s_red[w];
            double tss = t.tss;
            if (tss <= m + 0.0001) tss = m + 1.0;  // CBS.cpp:483-484
            const double stat = m / ((tss - m) / (rn - 2.0));
            D->rej[t.off_rej + p] = (t.ostat * 0.99999 <= stat) ? 1 : 0;
            if (t.raw) t.pval1 = stat;  // cbs::htmaxp through the low-level entry point: the statistic itself
        }
    }
}

// ------------------------------------------------------------------------------------
// edge tests
// ------------------------------------------------------------------------------------
// lane 0: sum = sum + x[k], tss = tss + x[k]*x[k] for k = 0..n-1, strictly in order (one dependent DADD
// chain each); the other lanes stage chunks through shared memory and keep the next one in flight
__device__ void chain_sum_sq(const double* __restrict__ x, int n, double* buf, int lane, double& sum, double& tss) {
    double r[PREP_CHUNK / 32];
#pragma unroll
    for (int q = 0; q < PREP_CHUNK / 32; ++q) { const int i = lane + 32 * q; r[q] = (i < n) ? x[i] : 0.0; }
    for (int c0 = 0; c0 < n; c0 += PREP_CHUNK) {
        const int cnt = min(PREP_CHUNK, n - c0);
        __syncwarp();
#pragma unroll
        for (int q = 0; q < PREP_CHUNK / 32; ++q) buf[lane + 32 * q] = r[q];
        __syncwarp();
        if (c0 + PREP_CHUNK < n) {
#pragma unroll
            for (int q = 0; q < PREP_CHUNK / 32; ++q) { const int i = c0 + PREP_CHUNK + lane + 32 * q; r[q] = (i < n) ? x[i] : 0.0; }
        }
        if (lane == 0) {
            int k = 0;
#pragma unroll 8
            for (; k + 1 < cnt; k += 2) {
                const double2 v = *reinterpret_cast<const double2*>(buf + k);
                sum = sum + v.x; tss = tss + v.x * v.x;
                sum = sum + v.y; tss = tss + v.y * v.y;
            }
            if (k < cnt) { const double v = buf[k]; sum = sum + v; tss = tss + v * v; }
        }
    }
    __syncwarp();
}

__device__ void edgeprep_warp(Dev* D, Task& t, int s, int lane, double* buf) {
    const int n1 = t.e_n1[s], n2 = t.e_n2[s];
    const double* x = D->cur + D->unit_off[t.unit] + t.lo + t.e_off[s];
    if (n1 == 1 || n2 == 1) { if (lane == 0) { t.e_status[s] = 1; t.e_m1[s] = 0; t.e_nrej[s] = 0; } return; }
    double sum1 = 0.0, sum2 = 0.0, tss = 0.0;  // CBS.cpp:503-512
    chain_sum_sq(x, n1, buf, lane, sum1, tss);
    chain_sum_sq(x + n1, n2, buf, lane, sum2, tss);
    if (lane == 0) { t.e_nrej[s] = 0; edgeprep_finish(t, s, sum1, sum2, tss); }
}

__global__ void __launch_bounds__(32) k_edgeprep(Dev* D) {
    __shared__ __align__(16) double buf[PREP_CHUNK];
    if (D->done) return;
    for (int k = blockIdx.x; k < 2 * D->n_edgeprep; k += gridDim.x)
        edgeprep_warp(D, D->tasks[D->edgeprep_task[k >> 1]], k & 1, threadIdx.x, buf);
}

__global__ void __launch_bounds__(128) k_edgeperm(Dev* D) {
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
        const int r = e.sparse ? edge_sparse_thread(*D, t, e, th) : edge_general_thread(*D, t, e, th);
        if (r) atomicAdd(&t.e_nrej[e.side], r);
    }
}

// ------------------------------------------------------------------------------------
// k_means: sequential sum of the (uncentred) values of each final segment
// ------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) k_means(const Dev* D, double* means) {
    __shared__ __align__(16) double buf[PREP_CHUNK];
    const int lane = threadIdx.x;
    for (int k = blockIdx.x; k < D->n_segs; k += gridDim.x) {
        const SegRec sg = D->segs[k];
        const double* x = D->x + D->unit_off[sg.unit] + sg.lo;
        const int n = sg.hi - sg.lo;
        double s = 0.0, sq = 0.0;
        chain_sum_sq(x, n, buf, lane, s, sq);
        if (lane == 0) means[k] = s / (double)n;
    }
}

// FP64 issue-rate microbenchmark: independent DADDs, 8 accumulators per thread.  The scan kernel's
// algorithmic work is one DADD per arc examined (the compare runs on the integer pipe), so this is
// the pipe peak its roofline is quoted against (MEASURED_PEAKS.json has no FP64 figure).
__global__ void __launch_bounds__(256) k_fp64_peak(double* out, int iters, double step) {
    double a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = (double)(threadIdx.x + k) * 1e-3;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int r = 0; r < 4; ++r) {
#pragma unroll
            for (int k = 0; k < 8; ++k) a[k] = a[k] + step;
        }
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += a[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

__global__ void k_widen_f32(const float* in, double* out, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        out[i] = (double)in[i];
}

__global__ void k_init_chains(Dev* D, const uint64_t* seed_state /* next 312 raw words */) {
    const int chain = D->prm.chain;
    for (int c = blockIdx.x; c < D->n_chains; c += gridDim.x) {
        Chain& ch = D->chains[c];
        for (int u = threadIdx.x; u < 312; u += blockDim.x) ch.hist[u] = seed_state[u];
        if (threadIdx.x == 0) {
            ch.top = -1; ch.unit_cur = -1;
            ch.unit_next = chain ? 0 : c; ch.unit_last = chain ? D->n_units : c + 1;
            ch.cursor = 0; ch.unit_cursor0 = 0; ch.commit_d = 0;
            ch.prev_off = -1; ch.prev_len = 0; ch.need_off = -1; ch.need_len = 0;
        }
    }
}

}  // namespace cbsg
