// cbs_core.h -- types, RNG helpers and the worklist scheduler shared by the CUDA
// kernels (kernels.cu) and, for logic tests only, a host build (tests/emul).
//
// Path implemented: the reference's CBS hot path, lib/cbs/CBS.cpp (segment :959-1024,
// fndcpt :830-892, tmaxo_impl :68-227, xperm :487-493, tpermp :495-536) as driven by
// src/cna_segment.hpp:127-159.  See DESIGN.md for the data layout.
#pragma once
#include <math.h>
#include <stdint.h>
#include <string.h>

#ifdef __CUDACC__
#define CBS_HD __host__ __device__ __forceinline__
#else
#define CBS_HD inline
#endif

namespace cbsg {

enum { RNG_MT = 0, RNG_PHILOX = 1 };
enum { SHUF_NCLS_MAX = 12 };  // room for the shuffle class tables (cbs_core.h: SHUF_NCLS)
enum { SX_PAD = 48 };
enum { CHAIN_Q = 4 };  // permutations of a batch that one pair of warps of k_chain turns into prefix sums together  // finite values kept behind the prefix sums of every permutation

// mirrors the reference call arguments 1:1 (CBS.hpp:100-113) + rng selection
struct Params {
    double alpha;
    int nperm;
    int hybrid;
    int min_width;
    int kmax;
    int nmin;
    double eta;
    double tol;
    int ibin;
    int rng_mode;
    int chain;  // MT only: one serial stream across all units (what `cna segment` does)
    uint64_t seed;
    int first_batch;   // permutations in the first batch of a max-t test
    int max_batch;     // cap on permutations per batch
    int record_splits;
};

// ------------------------------------------------------------------------------------
// RNG helpers
// ------------------------------------------------------------------------------------
CBS_HD uint64_t mt_temper(uint64_t y) {
    y ^= (y >> 29) & 0x5555555555555555ULL;
    y ^= (y << 17) & 0x71D67FFFEDA60000ULL;
    y ^= (y << 37) & 0xFFF7EEE000000000ULL;
    y ^= (y >> 43);
    return y;
}
CBS_HD uint64_t mt_twist(uint64_t a, uint64_t b, uint64_t m) {
    const uint64_t y = (a & 0xFFFFFFFF80000000ULL) | (b & 0x7FFFFFFFULL);
    return m ^ (y >> 1) ^ ((y & 1ULL) ? 0xB5026F5AA96619E9ULL : 0ULL);
}
// libstdc++ generate_canonical<double,53> on a 64-bit engine (SURVEY A.2): double(v)*2^-64,
// clamped just below 1.  The scaling by a power of two is exact.
CBS_HD double canonical_from_u64(uint64_t v) {
    double u = (double)v * 5.421010862427522170037264004349708557128906250e-20;
    if (u >= 1.0) u = 0.99999999999999988897769753748434595763683319091796875;
    return u;
}
// j = int(u*i) + 1 (CBS.cpp:490,528); returns 1-based index.
// The reference's expression needs a u64 -> f64 conversion and an f64 -> int truncation per draw; on B200 these run on
// the XU pipe at about half a lane per clock and SM, which made the shuffle kernels XU bound.  The same integer comes
// out of integer arithmetic: with r = v*i/2^64 exactly, the double computation yields p = RNE(RNE(v)*2^-64 * i) with
// |p - r| <= i*2^-54 + ulp(p)/2 <= 2^-33 for i <= 2^20 (the clamp below 1 moves u by at most 2^-53), so
// floor(p) == floor(r) whenever frac(r) lies in [2^-32, 1 - 2^-32); only then is the fast path taken (all but one draw
// in 2^31), otherwise the reference's own floating-point expression is evaluated.
CBS_HD int draw_index(uint64_t v, int i) {
    if (i <= (1 << 20)) {
        const uint64_t a = (uint64_t)(uint32_t)v * (uint64_t)(uint32_t)i;
        const uint64_t b = (v >> 32) * (uint64_t)(uint32_t)i;
        const uint64_t s = b + (a >> 32);  // floor(v*i / 2^32): integer part of r in the high word, top 32 fraction bits below
        const uint32_t f = (uint32_t)s;
        if (f - 1u < 0xFFFFFFFEu) return (int)(s >> 32) + 1;
    }
    return (int)(canonical_from_u64(v) * (double)i) + 1;
}

CBS_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                          uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        const uint32_t n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        const uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
CBS_HD uint64_t mix64(uint64_t z) {
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
// philox key of one split decision: a pure function of (seed, global unit id, lo, hi)
CBS_HD uint64_t task_key(uint64_t seed, uint64_t unit_id, uint32_t lo, uint32_t hi) {
    uint64_t h = mix64(seed + 0x9E3779B97F4A7C15ULL);
    h = mix64(h ^ (unit_id + 0x9E3779B97F4A7C15ULL));
    h = mix64(h ^ (((uint64_t)lo << 32) | (uint64_t)hi));
    return h;
}

// Uniform source for one permutation: draw k (0-based) of (stage, perm).
//   MT    : tempered word of the chain's window, win[k]
//   Philox: counter (k>>1, perm, stage, 0), key = task key, lanes 0/1 -> even k, 2/3 -> odd k
struct DrawSrc {
    const uint64_t* win;  // MT: points at this permutation's first raw word; nullptr => philox
    uint32_t k0, k1, stage, perm;
    uint32_t cached_pair;
    uint64_t c_even, c_odd;
    CBS_HD void init_mt(const uint64_t* w) { win = w; cached_pair = 0xFFFFFFFFu; }
    CBS_HD void init_philox(uint64_t key, uint32_t st, uint32_t pm) {
        win = nullptr; k0 = (uint32_t)key; k1 = (uint32_t)(key >> 32); stage = st; perm = pm;
        cached_pair = 0xFFFFFFFFu;
    }
    CBS_HD uint64_t u64(uint32_t k) {
        if (win) return mt_temper(win[k]);
        const uint32_t pair = k >> 1;
        if (pair != cached_pair) {
            uint32_t o[4];
            philox4x32_10(pair, perm, stage, 0u, k0, k1, o);
            c_even = ((uint64_t)o[1] << 32) | o[0];
            c_odd = ((uint64_t)o[3] << 32) | o[2];
            cached_pair = pair;
        }
        return (k & 1u) ? c_odd : c_even;
    }
};

// ------------------------------------------------------------------------------------
// Block geometry (CBS.cpp:71,77)
// ------------------------------------------------------------------------------------
CBS_HD int block_count(int n) { return n >= 50 ? (int)lround(sqrt((double)n)) : 1; }

// The observed scan of a pending segment (k_scan_obs) is spread over one CTA per OBS_SLICE_MARKERS markers, at most
// `cap` CTAs: a round holds only a few observed rows, and one CTA per row leaves most SMs idle (round 0: 23 rows).
enum { OBS_SLICE_MARKERS = 8192, OBS_SLICES_MAX = 24 };
CBS_HD int obs_slices(int n, int cap) {
    const int s = (n + OBS_SLICE_MARKERS - 1) / OBS_SLICE_MARKERS;
    return s < 1 ? 1 : (s > cap ? (cap < 1 ? 1 : cap) : s);
}
// work-stealing counters of the plain scan kernels, and the most slices any observed row of the round takes
enum { CTR_SCAN_PERM = 16, CTR_SCAN_OBS = 17, CTR_OBS_SLICES = 18 };
CBS_HD int block_end(int n, int nb, int b) {  // 1-based b; block_end(.,.,0) == 0
    return (int)lround((double)n * ((double)b / (double)nb));
}

// ------------------------------------------------------------------------------------
// Binary data (ibin = true): the reject decision of a permutation (CBS.cpp:218-224, 862-864) is thresh <= M / (tss'/n)
// with tss' = tss, or 1 when tss <= 1e-4.  A division by a positive constant is monotone in M, so the decision is
// M >= Lstar for the smallest double Lstar that passes the reference's own expression: found by stepping from the estimate.
// ------------------------------------------------------------------------------------
CBS_HD double bin_reject_level(double ostat, double tss, int n) {
    const double c = (tss <= 0.0001 ? 1.0 : tss) / (double)n;
    const double thresh = ostat * 0.99999;
    const double inf = HUGE_VAL;
    double m = thresh * c;
    if (!(m > 0.0)) m = 0.0;
    for (int k = 0; k < 64 && m / c < thresh; ++k) m = nextafter(m, inf);
    for (int k = 0; k < 64 && m > 0.0 && nextafter(m, 0.0) / c >= thresh; ++k) m = nextafter(m, 0.0);
    return m;
}
// fac * (s - 0.5)^2 <= fac_max / 4 for every |S_j - S_i| = s < 0.5 of an arc inside the bands (al0 <= L <= n - al0), so above
// that level only arcs with s >= 0.5 can reject, where the statistic is monotone in s.  Below it (a "weak" threshold) the
// reference's order-dependent pair skipping decides, and the permutations take the ordered walk (binary.cuh, DESIGN 4c).
CBS_HD bool bin_weak(double lstar, int n, int al0) {
    const double rn = (double)n, ra = (double)al0;
    return !(lstar > 0.25 * (rn / (ra * (rn - ra))));
}

// ------------------------------------------------------------------------------------
// Worklist records
// ------------------------------------------------------------------------------------
enum TaskState {
    TS_FREE = 0,
    TS_NEW,        // pending segment, nothing computed yet
    TS_OBS,        // prep + observed scan submitted
    TS_PERM,       // a permutation batch of the max-t test submitted
    TS_EDGEPREP,   // edge-test sums submitted
    TS_EDGEPERM,   // an edge permutation batch submitted
};

enum ExitCode { EX_NONE = 0, EX_SMALL_T = 1, EX_BIG_T = 2, EX_EARLY = 3, EX_TAILP = 4 };

struct Task {
    int unit, lo, hi, n;
    int state;
    int next;  // chain stack link (MT) / unused
    int nb;
    int alleq;       // written by prep
    int use_hybrid;  // hybrid && nmin < n (CBS.cpp:983): htmaxp permutations + analytic tail probability
    double pval1;    // tailp(sqrt(ostat), (kmax+1)/n, n, 100, tol), written by k_tailp (CBS.cpp:846)
    int raw;         // low-level API (tmaxo/tmaxp): use x as given with the supplied tss, no centring
    int deferred;    // did not get arena space this round
    int obs_round;   // round in which prep + observed scan were planned (results exist from the next round on)
    double tss;      // written by prep
    // observed scan result (written by scan kernel, LOC mode)
    double ostat;
    int tmaxi, tmaxj;  // 1-based prefix indices (reference tmaxi/tmaxj)
    // max-t permutation test
    int nrejc, perms_done, nrej, exit_code;
    int batch_P;
    int cnt_exit, cnt_nrej;  // written by the count phase: index in batch of the exiting perm (-1) / rejections in batch
    // edge tests (tpermp), side 0 = left boundary, 1 = right boundary
    int e_n1[2], e_n2[2], e_off[2], e_m1[2];
    int e_status[2];  // 0 needs permutations, 1 => p = 1.0, 2 => p = 0.0   (written by edgeprep)
    double e_ostat[2], e_xbar[2], e_rm1[2];
    int e_nrej[2];    // accumulated by edgeperm (atomics)
    int e_side, e_done;  // side in flight, permutations of that side already done
    int e_batch_P;
    // per-round arena slots
    long long off_sx, off_bs, off_A, off_rej;
    long long off_draw;  // MT: offset of this batch's window inside the draws arena
    uint64_t key;        // philox task key
    int w_ok;            // weighted CBS: cw of the segment is finite and strictly increasing (written by the observed scan)
    // weighted CBS, observed scan spread over several CTAs (weighted.cuh, k_wscan<1>/<2>, k_wobs_fin): running maximum
    // shared through global memory (bit patterns of positive doubles) and the first-visited arc that attains it
    unsigned long long w_level, w_found;
    double w_init, w_corner, w_v;
    int w_q, w_phase, w_o1, w_o2, w_i, w_j, w_set, w_lock;
    // observed scan spread over several CTAs (k_scan_obs): running level (bit pattern of a positive double), the best
    // arc of the finished slices (o_stat ... o_j; o_found: exact maximum without location) and the slices finished
    unsigned long long o_level, o_found;
    double o_stat, o_corner;
    int o_q, o_key, o_i, o_j, o_set, o_lock, o_done;
    int w_tie;           // the maximum was attained in two pairs with EQUAL corner statistics: k_wobs_fin walks the pairs in the reference's
                         // own (std::sort) order to get the location (weighted.cuh wtmaxo_ordered)
    double w_delta;      // weighted hybrid: min weight of a (kmax+1)-marker arc / total weight (getmncwt, CBS.cpp:602-607)
    long long off_bin;   // binary data: scratch of the ordered walk (binary.cuh) for the observed row / every row of a weak batch, or -1
};

struct Chain {        // MT replay: one serial stream
    int top;          // top of the pending-segment stack (task index) or -1
    int unit_next;    // chain==1: next unit to start; chain==0: unused
    int unit_last;    // one past the last unit of this chain
    int unit_cur;     // unit currently being segmented
    uint64_t cursor;  // uniforms consumed so far
    uint64_t unit_cursor0;
    // generator plan for the coming round
    uint64_t commit_d;      // draws consumed from last round's window (to be committed into hist)
    long long prev_off;     // last round's window offset (arena of the previous round)
    uint64_t prev_len;
    long long need_off;     // this round's window
    uint64_t need_len;
    uint64_t hist[312];     // the NEXT 312 raw (untempered) MT words: output k of the stream, k = cursor+u,
                            // is mt_temper(hist[u]).  A window of `need_len` words is stored as
                            // need_len+312 raw words so that any prefix can later be committed.
};

struct SegRec { int unit, lo, hi; };

struct SplitRec {  // one per fndcpt decision (parity diagnostics)
    int unit, lo, hi;
    double ostat;
    int iseg0, iseg1, ncpt, icpt0, icpt1, perms_run, nrej, exit_code, called;
    int e_nrej0, e_nrej1, e_status0, e_status1;
};

struct PermItem {  // one scan/shuffle work item of a round
    int task;
    int P;       // permutations (1 for the observed scan)
    int obs;     // 0 = permutation of the max-t test: only its reject decision is needed
                 // 1 = observed data (prep wrote sx / block stats): exact maximum AND location
                 // 2 = exact maximum, no location (cbs::tmaxp through the low-level API)
};
struct EdgeItem {
    int task, side;
    int perm0, P;    // permutations [perm0, perm0+P) of this side
    int cols, Q;     // general kernel: columns and permutations per column
    int sparse;      // 1 = register/local-memory kernel (m1 small)
    long long off_scratch;
    long long off_draw;
};

struct Dev {
    // ---- inputs -------------------------------------------------------------
    const double* x;            // values to segment (after smoothing), units end to end
    const long long* unit_off;  // [n_units+1]
    const uint64_t* unit_ids;   // global unit ids (philox keys)
    int n_units;
    Params prm;
    // ---- per-marker work arrays (same offsets as x) -------------------------------
    double* cur;     // centred values of the pending segment covering the marker
    double* gtab;    // g[L] = sqrt(L(n-L)/n) at offset seg_start+L
    double* factab;  // fac[L] = n/(L(n-L))
    int* bbtab;      // block ends bb[0..nb] at offset seg_start
    // ---- task pool ------------------------------------------------------------------
    Task* tasks;
    int task_cap;
    int* free_ring;
    unsigned free_head, free_tail;
    int* active[2];
    int n_active[2];
    int list_cap;
    int cur_list;
    Chain* chains;
    int n_chains;
    int units_started;  // next unit (philox) / chain (MT) to admit
    int max_live;       // admission limit on concurrently live root entries
    // ---- outputs ----------------------------------------------------------------------
    SegRec* segs;
    int seg_cap, n_segs;
    SplitRec* splits;
    int split_cap, n_splits;
    uint64_t* unit_draws;  // MT: draws consumed per unit
    // ---- arenas -----------------------------------------------------------------------
    double* arena;          // sx / block stats / shuffle scratch, in doubles
    long long arena_cap;
    int* rej;               // rejection flags of this round's permutations
    long long rej_cap;
    uint64_t* draws[2];     // MT per-chain windows (chain==1), ping-pong by round parity
    long long draws_cap;
    // MT, chain==0: every unit starts from the same engine state, so all chains read ONE raw stream
    // W[0..) that is generated once and extended on demand (positions are absolute cursors)
    // The stream is kept as a WINDOW: a ring of stream_cap words (a power of two; position p lives at p & stream_mask)
    // followed by a mirror of the ring's first stream_mirror words, so that any stream_mirror consecutive positions
    // can be read linearly from the ring slot of the first.  Positions below stream_lo (the smallest cursor of any
    // live chain) are dead and may be overwritten; a request that would reach beyond stream_lo + stream_cap is
    // deferred until the slower chains have moved on, so no input can exhaust the buffer.
    int shared_stream;
    uint64_t* stream;
    long long stream_cap, stream_mask, stream_mirror, stream_lo, stream_len, stream_target;
    long long stream_target_prev;             // the need one round ago (k_gen_lead sizes its look-ahead on the growth)
    const uint64_t* jump_polys;             // table g_{c*S} (mt_jump.h) or nullptr: sequential generation only
    long long gen_base, gen_E, gen_lead_end;  // extension in flight (written by k_gen_lead)
    long long span_max;                       // words the generator may add per round
    // ---- round plan -------------------------------------------------------------------
    int round;
    int n_prep;   int* prep_task;
    int n_items;  PermItem* items; int* item_prefix;  // exclusive prefix of P, [n_items+1]
    int* item_uprefix;                                 // exclusive prefix of ceil(P/CHAIN_Q): work units of k_chain
    int n_edgeprep; int* edgeprep_task;
    int n_edge;   EdgeItem* edges; int* edge_prefix;  // exclusive prefix of threads, [n_edge+1]
    int n_gen;    int* gen_chain;
    // shuffle work lists by segment-length class (shuffle_class below)
    int n_shuf[SHUF_NCLS_MAX]; int* shuf_item[SHUF_NCLS_MAX]; int* shuf_prefix[SHUF_NCLS_MAX];
    int* shuf_p0[SHUF_NCLS_MAX];   // first permutation of the item that the entry covers
    // work-stealing counters (reset every round): 0 global shuffle, 1 binary / weighted scan, 2 edge, 3 prefix, 4 hscan,
    // 8+cls shared-memory shuffle of class cls, CTR_SCAN_* (k_scan_perm / k_scan_obs); ctr[CTR_OBS_SLICES] is written by the scheduler
    unsigned ctr[24];
    // ---- status -----------------------------------------------------------------------
    int done;
    int stall;  // consecutive rounds with live tasks but no planned work
    int error;  // 0 ok; see cbs_gpu.h status codes
    unsigned long long stat_perms, stat_rounds_active;
    unsigned long long stat_perm_elems;     // sum over max-t permutations of the segment length
    unsigned long long round_elems[64], round_perms[64];  // per round (first 64): planned permutations and their markers (timeline)
    int profile;                            // count scan work (bench / roofline)
    unsigned long long stat_slots, stat_arcs;  // arc slots issued by the scan fast path / of them real arcs
    // ---- weighted CBS (cbs::segment_weighted, CBS.cpp:1026-1099); w == nullptr otherwise ----------
    const double* w;  // weights, laid out like x
    double* rw;       // sqrt(w) (CBS.cpp:1056)
    double* cw;       // per pending segment, at the segment's offset: cumsum(w)/sqrt(sum w) (CBS.cpp:1062-1066)
    double* ycur;     // cur * rw: what wxperm shuffles (CBS.cpp:540)
    // ---- low-level entry points (cbs::fndcpt / cbs::tpermp on a vector as given) run ONE decision through the same worklist ----
    int api_mode;     // 0: cbs::segment; 1: one fndcpt decision on unit 0 (x and tss as given, no children); 2: one tpermp test;
                      // 3: observed scan only (wtmaxo); 4: tailp of a given b (hand-built task, no worklist)
    double api_tss, api_delta;  // fndcpt: tss argument; hybrid: delta argument (0: (kmax+1)/n)
    int api_n1, api_n2;         // tpermp: sizes of the two sides
    int shuf_cl2;     // segments of 65536..SHUF_CL2_MAX markers have their own class (cluster of 2 CTAs)
    int shuf_arena;   // segments > 65535 markers are shuffled by k_perm on 32-bit index arrays in the arena (fallback of k_shuffle_cluster)
    int obs_slices;   // most CTAs per observed row (CBS_GPU_OBS_SLICES; 1: one CTA per row)
    int obs_noloc;    // observed rows need the exact maximum only (cbs::tmaxp through the low-level API)
    int no_early;     // CBS_GPU_NO_EARLY=1: decision-mode scans never stop at the first rejecting arc (A/B switch)
};

// shared MT stream (ring + mirror): store one word / linear read pointer for a run of <= stream_mirror positions
CBS_HD void stream_put(const Dev& D, long long pos, uint64_t v) {
    const long long idx = pos & D.stream_mask;
    D.stream[idx] = v;
    if (idx < D.stream_mirror) D.stream[idx + D.stream_cap] = v;
}
CBS_HD uint64_t stream_get(const Dev& D, long long pos) { return D.stream[pos & D.stream_mask]; }
// raw words of `off .. ` for one permutation (max-t or edge test): this round's per-chain window or the shared ring
CBS_HD const uint64_t* draw_window(const Dev& D, long long off) {
    return D.shared_stream ? D.stream + (off & D.stream_mask) : D.draws[D.round & 1] + off;
}

enum { ERR_TASK_CAP = 101, ERR_SEG_CAP = 102, ERR_ARENA = 103, ERR_SPLIT_CAP = 104, ERR_INTERNAL = 105, ERR_STALL = 106, ERR_STREAM_CAP = 107 };

// Shuffle classes (shuffle.cuh).  0..5: one CTA per permutation, last[] (16 bit per marker) and the claim table in
// shared memory; the class fixes the CTA size and the array size, hence how many permutations an SM holds at once
// (16 / 8 / 4 / 3 / 2 / 1 CTAs).  6, 7: segments of more than 65535 markers, last[] (32 bit per marker) spread over
// the shared memory of a cluster of 2 (up to SHUF_CL2_MAX markers) or more CTAs.
enum { SHUF_NCLS = 8, SHUF_CL2 = 6, SHUF_GLOBAL = 7, SHUF_CL2_MAX = 105000 };
CBS_HD int shuffle_class_max(int cls) {
    return cls == 0 ? 2048 : cls == 1 ? 8192 : cls == 2 ? 20000 : cls == 3 ? 29500 : cls == 4 ? 48500 : cls == 5 ? 65535 : SHUF_CL2_MAX;
}
CBS_HD int shuffle_class_threads(int cls) { return cls == 0 ? 128 : cls == 1 ? 256 : cls <= 4 ? 512 : 1024; }
CBS_HD int shuffle_class_hbits(int cls) { return cls <= 1 ? 11 : cls <= 4 ? 12 : 13; }  // log2 of the claim-table slots
CBS_HD int shuffle_class(int n, bool cl2) {
    for (int cls = 0; cls < SHUF_CL2; ++cls) if (n <= shuffle_class_max(cls)) return cls;
    return (cl2 && n <= SHUF_CL2_MAX) ? SHUF_CL2 : SHUF_GLOBAL;
}

// ------------------------------------------------------------------------------------
// Scheduler (runs in ONE thread per round; plain sequential C++ so that the very same
// code is exercised on the host by tests/emul).  Restates the control flow of
// cbs::segment (CBS.cpp:973-1005) and cbs::fndcpt (CBS.cpp:834-891) as a state machine
// over a device-resident pool of pending segments.
// ------------------------------------------------------------------------------------
struct Sched {
    Dev& D;
    int* out_list;
    int n_out;
    long long arena_used, rej_used, draws_used;
    CBS_HD explicit Sched(Dev& d) : D(d), out_list(nullptr), n_out(0), arena_used(0), rej_used(0), draws_used(0) {}

    CBS_HD int alloc_task() {
        if (D.free_head == D.free_tail) { D.error = ERR_TASK_CAP; return -1; }
        const int idx = D.free_ring[D.free_head % (unsigned)D.task_cap];
        D.free_head++;
        return idx;
    }
    CBS_HD void free_task(int idx) {
        D.tasks[idx].state = TS_FREE;
        D.free_ring[D.free_tail % (unsigned)D.task_cap] = idx;
        D.free_tail++;
    }
    CBS_HD int new_task(int unit, int lo, int hi) {
        const int idx = alloc_task();
        if (idx < 0) return -1;
        Task& t = D.tasks[idx];
        t.unit = unit; t.lo = lo; t.hi = hi; t.n = hi - lo;
        t.state = TS_NEW; t.next = -1; t.nb = 0; t.alleq = 0; t.raw = 0; t.deferred = 0;
        t.use_hybrid = (D.prm.hybrid && D.prm.nmin < t.n) ? 1 : 0; t.pval1 = 0.0; t.obs_round = -1;
        t.tss = 0.0; t.ostat = 0.0; t.tmaxi = 0; t.tmaxj = 0;
        t.nrejc = 0; t.perms_done = 0; t.nrej = 0; t.exit_code = EX_NONE; t.batch_P = 0;
        t.cnt_exit = -1; t.cnt_nrej = 0;
        t.e_side = 0; t.e_done = 0; t.e_batch_P = 0;
        for (int s = 0; s < 2; ++s) { t.e_status[s] = 0; t.e_nrej[s] = 0; t.e_m1[s] = 0; t.e_n1[s] = 0; t.e_n2[s] = 0; t.e_off[s] = 0; }
        t.off_bin = -1;
        t.key = task_key(D.prm.seed, D.unit_ids ? D.unit_ids[unit] : (uint64_t)unit, (uint32_t)lo, (uint32_t)hi);
        return idx;
    }
    // root task of a unit; the low-level entry points hand the vector over as is (cbs::fndcpt gets centred data and its tss)
    CBS_HD int new_root(int unit, int n) {
        const int idx = new_task(unit, 0, n);
        if (idx < 0 || !D.api_mode) return idx;
        Task& t = D.tasks[idx];
        t.raw = 1; t.tss = D.api_tss;
        if (D.api_mode == 2) {  // cbs::tpermp(n1, n2, n, x, ...): only the test of "side 0"; side 1 gets a one-point side: p = 1, no draws
            t.e_n1[0] = D.api_n1; t.e_n2[0] = D.api_n2; t.e_off[0] = 0;
            t.e_n1[1] = 1; t.e_n2[1] = 1; t.e_off[1] = 0;
            t.state = TS_EDGEPREP;
            D.edgeprep_task[D.n_edgeprep++] = idx;
            t.obs_round = D.round;  // the sums are computed by this round's k_edgeprep
        }
        return idx;
    }
    CBS_HD void emit_segment(const Task& t) {
        if (D.n_segs >= D.seg_cap) { D.error = ERR_SEG_CAP; return; }
        SegRec& s = D.segs[D.n_segs++];
        s.unit = t.unit; s.lo = t.lo; s.hi = t.hi;
    }
    CBS_HD void log_split(const Task& t, int called, int ncpt, int icpt0, int icpt1) {
        if (!D.prm.record_splits) return;
        if (D.n_splits >= D.split_cap) { D.error = ERR_SPLIT_CAP; return; }
        SplitRec& r = D.splits[D.n_splits++];
        r.unit = t.unit; r.lo = t.lo; r.hi = t.hi;
        r.ostat = called ? t.ostat : 0.0;
        r.iseg0 = called ? t.tmaxi - 1 : 0; r.iseg1 = called ? t.tmaxj - 1 : 0;
        r.ncpt = ncpt; r.icpt0 = icpt0; r.icpt1 = icpt1;
        r.perms_run = t.perms_done; r.nrej = t.nrej; r.exit_code = t.exit_code; r.called = called;
        r.e_nrej0 = t.e_nrej[0]; r.e_nrej1 = t.e_nrej[1]; r.e_status0 = t.e_status[0]; r.e_status1 = t.e_status[1];
    }
    CBS_HD Chain* chain_of(const Task& t) {
        if (D.prm.rng_mode != RNG_MT) return nullptr;
        return &D.chains[D.prm.chain ? 0 : t.unit];
    }

    // arena helpers ---------------------------------------------------------------------
    // One row per permutation: S[0..n], SX_PAD finite values (the scan's fast path reads whole 32 x 8 units), then
    // the extrema table of the row: tbl_entries(n) floats of minima and as many of maxima, entry e = extrema of
    // S[32e .. 32e+31], rounded outwards (written next to the prefix sums by k_chain / k_prep, read by k_scan)
    CBS_HD static long long tbl_offset(int n) { return ((long long)n + 1 + SX_PAD + 3) & ~3LL; }  // in doubles
    CBS_HD static long long tbl_entries(int n) { return ((long long)n >> 5) + 2; }
    CBS_HD static long long sx_stride(int n) { return tbl_offset(n) + ((tbl_entries(n) + 3) & ~3LL); }
    CBS_HD static long long bs_stride(int nb) { return (3LL * nb + 4 + 3) & ~3LL; }
    // scratch of wtmaxo_ordered (weighted.cuh), in doubles: per block 2 doubles + 2 ints, per block pair 3 doubles + 3 ints
    CBS_HD static long long wexact_stride(int nb) { const long long nb2 = (long long)nb * (nb + 1) / 2; return (3 * (nb + 1) + 5 * (nb2 + 1) + 8 + 3) & ~3LL; }
    // scratch of the binary ordered walk (binary.cuh), in doubles: per block pair a (corner statistic, index) record of 2
    // doubles, the pair bound and 2 ints (pair, corner length)
    CBS_HD static long long bin_stride(int nb) { const long long e = (long long)nb * (nb + 1) / 2 + 1; return (4 * e + 3) & ~3LL; }
    // 32-bit index array of the global-memory shuffle, in doubles; all strides are multiples of 4 doubles so
    // that every row of prefix sums starts on a 32-byte boundary (k_prefix moves rows with 128-bit accesses)
    CBS_HD static long long idx_stride(int n) { return (((long long)n + 1) / 2 + 1 + 3) & ~3LL; }

    // Task finished with `ncpt` change points at 0-based icpt (relative to lo):
    // emits the final segment or creates the children (CBS.cpp:996-1004).
    //   MT    : children go on the chain's stack, right-most on top (the reference always
    //           continues with the right-most pending segment, :976-978)
    //   philox: children are independent and are queued for this very round
    CBS_HD void finish(int idx, int called, int ncpt, int icpt0, int icpt1) {
        Task& t = D.tasks[idx];
        log_split(t, called, ncpt, icpt0, icpt1);
        Chain* ch = chain_of(t);
        const int unit = t.unit, lo = t.lo, hi = t.hi, below = t.next;
        if (D.api_mode) {  // a single decision was asked for: it is in the split log, nothing follows
            free_task(idx);
            if (ch) ch->top = below;
            return;
        }
        if (ncpt == 0) {
            emit_segment(t);
            free_task(idx);
            if (ch) ch->top = below;
            return;
        }
        const int c1 = lo + icpt0 + 1;
        const int c2 = (ncpt == 2) ? lo + icpt1 + 1 : hi;
        free_task(idx);
        int kids[3]; int nk = 0;
        kids[nk++] = new_task(unit, lo, c1);
        if (ncpt == 2) kids[nk++] = new_task(unit, c1, c2);
        kids[nk++] = new_task(unit, (ncpt == 2) ? c2 : c1, hi);
        for (int k = 0; k < nk; ++k) if (kids[k] < 0) return;
        if (ch) {
            int link = below;
            for (int k = 0; k < nk; ++k) { D.tasks[kids[k]].next = link; link = kids[k]; }
            ch->top = link;
            // The serial RNG stream only orders the PERMUTATION tests.  The observed scan of a pending
            // segment draws nothing, so the siblings that wait below the top are prepared and scanned
            // now; when their turn comes they continue from TS_OBS without spending a round on it.
            for (int k = 0; k + 1 < nk; ++k) {
                Task& kid = D.tasks[kids[k]];
                if (kid.n >= 2 * D.prm.min_width && plan_obs(kids[k])) kid.state = TS_OBS;
                else kid.deferred = 0;
            }
        } else {
            for (int k = 0; k < nk; ++k) push_out(kids[k]);
        }
    }
    CBS_HD void push_out(int idx) {
        if (n_out >= D.list_cap) { D.error = ERR_TASK_CAP; return; }
        out_list[n_out++] = idx;
    }
    // MT: make sure the chain has a pending segment: start its next unit if the stack is empty.
    // Returns false when the chain has nothing left.
    CBS_HD bool chain_refill(Chain* ch) {
        if (ch->top >= 0) return true;
        if (ch->unit_cur >= 0 && D.unit_draws) D.unit_draws[ch->unit_cur] = ch->cursor + ch->commit_d - ch->unit_cursor0;
        ch->unit_cur = -1;
        while (ch->unit_next < ch->unit_last) {
            const int u = ch->unit_next++;
            const long long n = D.unit_off[u + 1] - D.unit_off[u];
            if (n <= 0) continue;  // cna_segment.hpp:138
            const int idx = new_root(u, (int)n);
            if (idx < 0) return false;
            ch->top = idx;
            ch->unit_cur = u;
            ch->unit_cursor0 = ch->cursor + ch->commit_d;
            return true;
        }
        return false;
    }

    // request slots for the observed scan of task idx (prep + scan this round)
    CBS_HD bool plan_obs(int idx) {
        Task& t = D.tasks[idx];
        t.nb = block_count(t.n);
        const long long wx = D.w ? wexact_stride(t.nb) : 0;  // weighted: scratch of the ordered walk (only used when maxima tie)
        const long long bx = D.prm.ibin ? bin_stride(t.nb) : 0;  // binary data: scratch of the ordered walk
        const long long need = sx_stride(t.n) + bs_stride(t.nb) + wx + bx;
        if (need > D.arena_cap) { D.error = ERR_ARENA; return false; }
        if (arena_used + need > D.arena_cap || rej_used + 1 > D.rej_cap) { t.deferred = 1; return false; }
        t.off_sx = arena_used; t.off_bs = arena_used + sx_stride(t.n); t.off_A = wx ? t.off_bs + bs_stride(t.nb) : -1;
        t.off_bin = bx ? t.off_bs + bs_stride(t.nb) : -1;
        arena_used += need;
        t.off_rej = rej_used; rej_used += 1;
        t.o_level = 0; t.o_found = 0; t.o_set = 0; t.o_lock = 0; t.o_done = 0;
        const unsigned ns = (unsigned)obs_slices(t.n, D.obs_slices);
        if (ns > D.ctr[CTR_OBS_SLICES]) D.ctr[CTR_OBS_SLICES] = ns;
        D.prep_task[D.n_prep++] = idx;
        PermItem& it = D.items[D.n_items];
        it.task = idx; it.P = 1; it.obs = 1;
        t.obs_round = D.round;
        D.item_prefix[D.n_items + 1] = D.item_prefix[D.n_items] + 1;
        D.item_uprefix[D.n_items + 1] = D.item_uprefix[D.n_items] + 1;
        D.n_items++;
        t.deferred = 0;
        return true;
    }
    // request a permutation batch for the max-t test
    CBS_HD bool plan_perm(int idx) {
        Task& t = D.tasks[idx];
        const Params& p = D.prm;
        int want;
        if (t.perms_done == 0) want = p.first_batch;
        else {
            // expected permutations still needed to collect the missing rejections, +25%
            const double rate = (double)(t.nrej > 0 ? t.nrej : 1) / (double)t.perms_done;
            const double need = (double)(t.nrejc + 1 - t.nrej) / rate * 1.25 + 16.0;
            want = need > (double)p.max_batch ? p.max_batch : (int)need;
            if (want < p.first_batch) want = p.first_batch;
        }
        if (want > p.max_batch) want = p.max_batch;
        if (want > p.nperm - t.perms_done) want = p.nperm - t.perms_done;
        const int cls = shuffle_class(t.n, D.shuf_cl2 != 0);
        // fallback shuffle of segments > 65535 markers (k_perm): a 32-bit index array per permutation in the arena
        const long long idxd = (cls == SHUF_GLOBAL && D.shuf_arena) ? idx_stride(t.n) : 0;  // doubles per permutation
        // binary data with a weak reject level: every permutation takes the ordered walk and needs its scratch
        const long long bx = (p.ibin && bin_weak(bin_reject_level(t.ostat, t.tss, t.n), t.n, p.min_width)) ? bin_stride(t.nb) : 0;
        const long long per = idxd + sx_stride(t.n) + bs_stride(t.nb) + bx;
        const bool mtwin = p.rng_mode == RNG_MT && !D.shared_stream;
        // never let one task take more than half of the arena
        long long fit = (D.arena_cap / 2) / per;
        if (mtwin) { const long long f2 = (D.draws_cap / 2 - 312) / t.n; if (f2 < fit) fit = f2; }
        if (fit < 1) { D.error = ERR_ARENA; return false; }
        if (want > fit) want = (int)fit;
        if (D.shared_stream && p.rng_mode == RNG_MT) {
            // a batch must fit in one generator span and in a quarter of the stream window (the chain with the
            // smallest cursor then always gets its batch: no deadlock)
            long long by_span = D.span_max / t.n;
            const long long by_win = (D.stream_cap / 4) / t.n;
            if (by_win < by_span) by_span = by_win;
            if (by_span < 1) { D.error = ERR_STREAM_CAP; return false; }
            if (want > by_span) want = (int)by_span;
        }
        const int gpart = (cls == SHUF_GLOBAL) ? want : 0;
        const long long need = idxd * gpart + (sx_stride(t.n) + bs_stride(t.nb) + bx) * want;
        const long long dneed = (p.rng_mode == RNG_MT) ? (long long)want * t.n : 0;
        if (arena_used + need > D.arena_cap || rej_used + want > D.rej_cap || (mtwin && draws_used + dneed + 312 > D.draws_cap)) {
            t.deferred = 1;
            return false;
        }
        if (p.rng_mode == RNG_MT) {
            Chain* ch = chain_of(t);
            if (D.shared_stream) {
                const long long pos = (long long)(ch->cursor + ch->commit_d);
                // outside the window (slower chains still need its low end) or beyond the generator's span per round: wait
                if (pos + dneed + 312 > D.stream_lo + D.stream_cap || pos + dneed > D.stream_len + D.span_max) { t.deferred = 1; return false; }
                t.off_draw = pos;
                if (pos + dneed > D.stream_target) D.stream_target = pos + dneed;
            } else {
                t.off_draw = draws_used;
                ch->need_off = draws_used; ch->need_len = (uint64_t)dneed;
                draws_used += dneed + 312;  // the generator appends the 312 words that follow the window
            }
        }
        t.off_A = gpart ? arena_used : -1;
        t.off_sx = arena_used + idxd * gpart;
        t.off_bs = t.off_sx + sx_stride(t.n) * want;
        t.off_bin = bx ? t.off_bs + bs_stride(t.nb) * want : -1;
        arena_used += need;
        t.off_rej = rej_used; rej_used += want;
        t.batch_P = want;
        t.cnt_exit = -1; t.cnt_nrej = 0;
        PermItem& it = D.items[D.n_items];
        it.task = idx; it.P = want; it.obs = 0;
        D.item_prefix[D.n_items + 1] = D.item_prefix[D.n_items] + want;
        D.item_uprefix[D.n_items + 1] = D.item_uprefix[D.n_items] + (want + CHAIN_Q - 1) / CHAIN_Q;
        if (want - gpart > 0) {  // permutations [0, want-gpart): the class's own shuffle
            const int q = D.n_shuf[cls];
            D.shuf_item[cls][q] = D.n_items; D.shuf_p0[cls][q] = 0;
            D.shuf_prefix[cls][q + 1] = D.shuf_prefix[cls][q] + (want - gpart);
            D.n_shuf[cls] = q + 1;
        }
        if (gpart > 0) {  // permutations [want-gpart, want): L2 shuffle (all of them for segments > 65535 markers)
            const int q = D.n_shuf[SHUF_GLOBAL];
            D.shuf_item[SHUF_GLOBAL][q] = D.n_items; D.shuf_p0[SHUF_GLOBAL][q] = want - gpart;
            D.shuf_prefix[SHUF_GLOBAL][q + 1] = D.shuf_prefix[SHUF_GLOBAL][q] + gpart;
            D.n_shuf[SHUF_GLOBAL] = q + 1;
        }
        D.n_items++;
        t.deferred = 0;
        t.state = TS_PERM;
        return true;
    }
    // request an edge permutation batch (side t.e_side)
    CBS_HD bool plan_edge(int idx) {
        Task& t = D.tasks[idx];
        const Params& p = D.prm;
        const int s = t.e_side;
        const int m1 = t.e_m1[s];
        const int n12 = t.e_n1[s] + t.e_n2[s];
        const int remaining = p.nperm - t.e_done;
        EdgeItem e;
        e.task = idx; e.side = s; e.perm0 = t.e_done; e.off_scratch = -1; e.off_draw = -1;
        const bool mtwin = p.rng_mode == RNG_MT && !D.shared_stream;
        long long aneed = 0;
        if (m1 <= 64) {
            e.sparse = 1; e.cols = 0; e.Q = 1;
            e.P = remaining;
            if (mtwin) {
                long long fit = (D.draws_cap / 2 - 312) / m1;
                if (fit < 1) { D.error = ERR_ARENA; return false; }
                if (e.P > fit) e.P = (int)fit;
            }
        } else {
            e.sparse = 0;
            long long cols = (D.arena_cap / 4) / n12;
            if (cols < 1) { D.error = ERR_ARENA; return false; }
            if (cols > 4096) cols = 4096;
            if (cols > remaining) cols = remaining;
            int Q = (remaining + (int)cols - 1) / (int)cols;
            if (Q > 8) Q = 8;
            long long P = cols * Q;
            if (P > remaining) P = remaining;
            if (mtwin) {
                long long fit = (D.draws_cap / 2 - 312) / m1;
                if (fit < 1) { D.error = ERR_ARENA; return false; }
                if (P > fit) { P = fit; if (cols > P) cols = P; Q = (int)((P + cols - 1) / cols); }
            }
            e.cols = (int)cols; e.Q = Q; e.P = (int)P;
            aneed = cols * n12;
        }
        if (D.shared_stream && p.rng_mode == RNG_MT) {  // as plan_perm: a quarter of the window / one generator span at most
            long long fit = (D.stream_cap / 4) / m1;
            if (D.span_max / m1 < fit) fit = D.span_max / m1;
            if (fit < 1) { D.error = ERR_STREAM_CAP; return false; }
            if (e.P > fit) {
                e.P = (int)fit;
                if (!e.sparse) { if (e.cols > e.P) e.cols = e.P; e.Q = (e.P + e.cols - 1) / e.cols; aneed = (long long)e.cols * n12; }
            }
        }
        const long long dneed = (p.rng_mode == RNG_MT) ? (long long)e.P * m1 : 0;
        if (arena_used + aneed > D.arena_cap || (mtwin && draws_used + dneed + 312 > D.draws_cap)) { t.deferred = 1; return false; }
        if (p.rng_mode == RNG_MT) {
            Chain* ch = chain_of(t);
            if (D.shared_stream) {
                const long long pos = (long long)(ch->cursor + ch->commit_d);
                if (pos + dneed + 312 > D.stream_lo + D.stream_cap || pos + dneed > D.stream_len + D.span_max) { t.deferred = 1; return false; }
                e.off_draw = pos;
                if (pos + dneed > D.stream_target) D.stream_target = pos + dneed;
            } else {
                e.off_draw = draws_used;
                ch->need_off = draws_used; ch->need_len = (uint64_t)dneed;
                draws_used += dneed + 312;
            }
        }
        if (aneed) { e.off_scratch = arena_used; arena_used += aneed; }
        t.e_batch_P = e.P;
        const int threads = e.sparse ? e.P : e.cols;
        D.edges[D.n_edge] = e;
        D.edge_prefix[D.n_edge + 1] = D.edge_prefix[D.n_edge] + threads;
        D.n_edge++;
        t.deferred = 0;
        t.state = TS_EDGEPERM;
        return true;
    }

    // consume draws of the task's chain (MT): they become a commit for the generator
    CBS_HD void consume(Task& t, uint64_t d) {
        Chain* ch = chain_of(t);
        if (!ch) return;
        ch->commit_d += d;
    }

    // after the max-t test said "significant" (or was skipped): CBS.cpp:869-890
    CBS_HD bool begin_edges(int idx) {  // returns true if the task is finished
        Task& t = D.tasks[idx];
        const int iseg1 = t.tmaxi, iseg2 = t.tmaxj, n = t.n;  // 1-based, as in the reference
        if (iseg2 == n) { finish(idx, 1, 1, iseg1 - 1, 0); return true; }
        if (iseg1 == 0) { finish(idx, 1, 1, iseg2 - 1, 0); return true; }  // unreachable (SURVEY A.1)
        t.e_n1[0] = iseg1; t.e_n2[0] = iseg2 - iseg1; t.e_off[0] = 0;
        t.e_n2[1] = n - iseg2; t.e_n1[1] = (n - iseg1) - (n - iseg2); t.e_off[1] = iseg1;
        t.e_nrej[0] = t.e_nrej[1] = 0;
        t.state = TS_EDGEPREP;
        D.edgeprep_task[D.n_edgeprep++] = idx;
        return false;
    }
    CBS_HD void finish_edges(int idx) {
        Task& t = D.tasks[idx];
        const Params& p = D.prm;
        int ncpt = 0, ic[2] = {0, 0};
        for (int s = 0; s < 2; ++s) {
            double pv;
            if (t.e_status[s] == 1) pv = 1.0;
            else if (t.e_status[s] == 2) pv = 0.0;
            else pv = (double)t.e_nrej[s] / (double)p.nperm;
            if (pv <= p.alpha) {
                if (s == 0) { ncpt = 1; ic[0] = t.tmaxi - 1; }
                else if (ncpt < 2) { ic[ncpt] = t.tmaxj - 1; ++ncpt; }
            }
        }
        finish(idx, 1, ncpt, ic[0], ic[1]);
    }
    // choose the next edge side that still needs permutations; false if none
    CBS_HD bool next_edge_side(Task& t) {
        while (t.e_side < 2) {
            if (t.e_status[t.e_side] == 0 && t.e_done < D.prm.nperm) return true;
            t.e_side++; t.e_done = 0;
        }
        return false;
    }

    // One scheduling step of a task. Returns true if the task is still alive AND waits for
    // kernels of this round (or is deferred); false if it finished (children were queued).
    CBS_HD bool step(int idx) {
        Task& t = D.tasks[idx];
        const Params& p = D.prm;
        for (;;) {
            switch (t.state) {
            case TS_NEW: {
                if (t.n < 2 * p.min_width) { t.exit_code = EX_NONE; finish(idx, 0, 0, 0, 0); return false; }  // CBS.cpp:981
                if (!plan_obs(idx)) return true;
                t.state = TS_OBS;
                return true;
            }
            case TS_OBS: {
                if (t.obs_round == D.round) return true;  // planned ahead in this very round: kernels have not run yet
                if (t.alleq) { finish(idx, 0, 0, 0, 0); return false; }  // CBS.cpp:985
                if (D.api_mode == 3) { finish(idx, 1, 0, 0, 0); return false; }  // cbs::wtmaxo entry: the observed scan is all that was asked for
                const double t1 = sqrt(t.ostat);
                if (t1 <= 0.1) { t.exit_code = EX_SMALL_T; finish(idx, 1, 0, 0, 0); return false; }  // :839
                const int i1 = t.tmaxi, i2 = t.tmaxj;
                int arc = i2 - i1; if (t.n - i2 + i1 < arc) arc = t.n - i2 + i1;
                if (t1 >= 7.0 && arc >= 10) {  // :843
                    t.exit_code = EX_BIG_T;
                    if (begin_edges(idx)) return false;
                    return true;
                }
                if (t.use_hybrid) {  // :846-848
                    if (t.pval1 > p.alpha) { t.exit_code = EX_TAILP; finish(idx, 1, 0, 0, 0); return false; }
                    t.nrejc = (int)((p.alpha - t.pval1) * (double)p.nperm);
                } else t.nrejc = (int)(p.alpha * (double)p.nperm);  // :858
                t.perms_done = 0; t.nrej = 0;
                if (p.nperm <= 0) { if (begin_edges(idx)) return false; return true; }
                t.state = TS_PERM;
                if (!plan_perm(idx)) return true;
                return true;
            }
            case TS_PERM: {
                if (t.deferred) { plan_perm(idx); return true; }
                // results of the batch (count phase): ordered early exit, CBS.cpp:860-866
                if (t.cnt_exit >= 0) {
                    const int used = t.cnt_exit + 1;
                    t.perms_done += used; t.nrej = t.nrejc + 1; t.exit_code = EX_EARLY;
                    consume(t, (uint64_t)used * (uint64_t)t.n);
                    D.stat_perms += (unsigned long long)used;
                    D.stat_perm_elems += (unsigned long long)used * (unsigned long long)t.n;
                    finish(idx, 1, 0, 0, 0);
                    return false;
                }
                t.perms_done += t.batch_P; t.nrej += t.cnt_nrej;
                consume(t, (uint64_t)t.batch_P * (uint64_t)t.n);
                D.stat_perms += (unsigned long long)t.batch_P;
                D.stat_perm_elems += (unsigned long long)t.batch_P * (unsigned long long)t.n;
                if (t.perms_done >= p.nperm) {
                    if (begin_edges(idx)) return false;
                    return true;
                }
                plan_perm(idx);
                return true;
            }
            case TS_EDGEPREP: {
                if (D.api_mode == 2 && t.obs_round == D.round) return true;  // cbs::tpermp entry: k_edgeprep runs in this round
                t.e_side = 0; t.e_done = 0;
                if (!next_edge_side(t)) { finish_edges(idx); return false; }
                t.state = TS_EDGEPERM; t.deferred = 1;
                continue;
            }
            case TS_EDGEPERM: {
                if (!t.deferred) {
                    t.e_done += t.e_batch_P;
                    consume(t, (uint64_t)t.e_batch_P * (uint64_t)t.e_m1[t.e_side]);
                }
                if (!next_edge_side(t)) { finish_edges(idx); return false; }
                plan_edge(idx);
                return true;
            }
            default:
                D.error = ERR_INTERNAL;
                return false;
            }
        }
    }

    // One round: consume last round's results, advance every live task as far as possible
    // without kernels, and write the plan for this round's kernels.
    // Active entries are chain indices (MT) or task indices (philox).
    CBS_HD void run_round() {
        const int in = D.cur_list, outl = in ^ 1;
        const int* in_list = D.active[in];
        const int n_in = D.n_active[in];
        out_list = D.active[outl];
        n_out = 0;
        D.n_prep = 0; D.n_items = 0; D.n_edgeprep = 0; D.n_edge = 0; D.n_gen = 0;
        D.item_prefix[0] = 0; D.item_uprefix[0] = 0; D.edge_prefix[0] = 0;
        for (int k = 0; k < SHUF_NCLS; ++k) { D.n_shuf[k] = 0; D.shuf_prefix[k][0] = 0; }
        for (int k = 0; k < 24; ++k) D.ctr[k] = 0;
        arena_used = 0; rej_used = 0; draws_used = 0;
        const bool mt = D.prm.rng_mode == RNG_MT;
        if (D.shared_stream && D.gen_E > 0) { D.stream_len = D.gen_base + D.gen_E; D.gen_E = 0; }
        int wpos = 0;
        if (mt) {
            // carried-over chains first, then admit new ones up to max_live
            int k = 0;
            for (;;) {
                int c;
                if (k < n_in) c = in_list[k++];
                else if (D.units_started < D.n_chains && wpos < D.max_live) c = D.units_started++;
                else break;
                if (D.error) break;
                Chain& ch = D.chains[c];
                // last round's window becomes "previous"; its consumption is committed below
                ch.cursor += ch.commit_d;
                ch.commit_d = 0;
                ch.prev_off = ch.need_off; ch.prev_len = ch.need_len;
                ch.need_off = -1; ch.need_len = 0;
                bool alive = false;
                while (!D.error && chain_refill(&ch)) {
                    if (step(ch.top)) { alive = true; break; }
                }
                if (alive) {
                    out_list[wpos++] = c;
                    if (!D.shared_stream && (ch.commit_d || ch.need_len)) D.gen_chain[D.n_gen++] = c;
                }
            }
            n_out = wpos;
            if (D.shared_stream && D.units_started >= D.n_chains) {  // low end of the stream window: the smallest cursor of a live
                // chain (chains that have not started yet will read from position 0: the window waits for them)
                long long lo = D.stream_len;
                for (int k2 = 0; k2 < wpos; ++k2) {
                    const Chain& ch = D.chains[out_list[k2]];
                    const long long cpos = (long long)(ch.cursor + ch.commit_d);
                    if (cpos < lo) lo = cpos;
                }
                if (lo > D.stream_lo) D.stream_lo = lo;
            }
        } else {
            for (int k = 0; k < n_in; ++k) out_list[n_out++] = in_list[k];
            int qhead = 0;
            for (;;) {
                if (D.error) break;
                if (qhead == n_out) {
                    // admit new units while there is room
                    bool added = false;
                    while (D.units_started < D.n_units && wpos + (n_out - qhead) < D.max_live) {
                        const int u = D.units_started++;
                        const long long n = D.unit_off[u + 1] - D.unit_off[u];
                        if (n <= 0) continue;
                        const int idx = new_root(u, (int)n);
                        if (idx < 0) break;
                        push_out(idx);
                        added = true;
                        break;
                    }
                    if (!added) break;
                }
                const int idx = out_list[qhead++];
                if (step(idx)) out_list[wpos++] = idx;
            }
            n_out = wpos;
        }
        if (D.round < 64) {
            unsigned long long pe = 0, pp = 0;
            for (int k = 0; k < D.n_items; ++k) if (!D.items[k].obs) { pp += (unsigned long long)D.items[k].P; pe += (unsigned long long)D.items[k].P * (unsigned long long)D.tasks[D.items[k].task].n; }
            D.round_elems[D.round] = pe; D.round_perms[D.round] = pp;
        }
        D.n_active[outl] = n_out;
        D.cur_list = outl;
        D.round++;
        if (n_out == 0 && !D.error) {
            const bool more = mt ? (D.units_started < D.n_chains) : (D.units_started < D.n_units);
            if (!more) D.done = 1;
        }
        if (D.n_items || D.n_edge || D.n_edgeprep || D.n_prep) { D.stat_rounds_active++; D.stall = 0; }
        else if (n_out > 0 && ++D.stall > 16) D.error = ERR_STALL;  // a livelock must not spin forever
        if (D.error) D.done = 1;
    }
};

}  // namespace cbsg
