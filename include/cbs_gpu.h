/* cbs_gpu.h -- C ABI of libcbs_cuda.so: the B200 (sm_100a) implementation of the CBS +
 * outlier-smoothing hot path of djhshih/genomic (`cna segment`).
 *
 * The reference has no FFI layer; its boundary for this path is the C++ free-function
 * surface of lib/cbs that src/cna_segment.hpp:140-141 and tests/cbs_test.cpp call.  Each entry
 * point below names the reference interface it replaces (paths relative to the reference
 * root).  Plain pointers and sizes only; no C++ types, no exceptions cross this boundary:
 * every call returns a status code and cbs_gpu_last_error() gives the text.
 * The header-only C++ shim genomic_b200/host/cbs_gpu.hpp wraps these with the reference's
 * exact signatures (namespace cbs_gpu) and rethrows std::invalid_argument / runtime_error.
 */
#ifndef CBS_GPU_H
#define CBS_GPU_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CBS_GPU_OK 0
#define CBS_GPU_ERR_INVALID 1      /* what the reference reports as std::invalid_argument */
#define CBS_GPU_ERR_CUDA 2
#define CBS_GPU_ERR_OOM 3
#define CBS_GPU_ERR_CAPACITY 4     /* an internal table overflowed (message says which knob) */
#define CBS_GPU_ERR_UNSUPPORTED 5  /* argument combination not implemented on the GPU path */
#define CBS_GPU_ERR_NONFINITE 6    /* non-finite value reached CBS */
#define CBS_GPU_ERR_OVERFLOW 7     /* reference: std::overflow_error from boost quantile (trim == 0) */

#define CBS_GPU_RNG_MT19937_64 0   /* bit-exact replay of std::mt19937_64 + generate_canonical */
#define CBS_GPU_RNG_PHILOX 1       /* Philox4x32-10 counter mode, keyed per (seed, unit, segment) */

#define CBS_GPU_F32 0
#define CBS_GPU_F64 1
#define CBS_GPU_HOST 0
#define CBS_GPU_DEVICE 1

typedef struct cbs_gpu_ctx cbs_gpu_ctx;

/* One POD mirroring 1:1 the arguments of cbs::segment (lib/cbs/CBS.hpp:100-113) and cbs::smooth
 * (lib/cbs/smooth.hpp:8-13), i.e. the options of `cna segment` (src/cna_segment.hpp:67-79). */
typedef struct cbs_gpu_params {
    double alpha;
    int32_t nperm;
    int32_t hybrid;
    int32_t min_width;
    int32_t kmax;
    int32_t nmin;
    double eta; /* accepted, unused -- as in the reference */
    double tol;
    int32_t ibin;          /* binary data (CBS.cpp:99-224, ibin branches); not with hybrid, not on the weighted entries */
    int32_t undo_prune;
    double undo_prune_cutoff;
    int32_t do_smooth;
    int32_t smooth_region;
    double outlier_sd_scale;
    double smooth_sd_scale;
    double trim;
    int32_t rng_mode; /* CBS_GPU_RNG_* */
    int32_t chain;    /* MT only. 1: ONE stream shared serially by all units, exactly what
                         `cna segment` does (cna_segment.hpp:129); 0: a fresh engine seeded with
                         `seed` per unit (what tests/cbs_test.cpp does per call) -- units independent */
    uint64_t seed;
    int32_t first_batch;   /* scheduling knobs, 0 = default; never change results */
    int32_t max_batch;
    int32_t record_splits; /* keep one record per split decision (parity diagnostics) */
    int32_t reserved;
} cbs_gpu_params;

/* CLI defaults of `cna segment` (src/cna_segment.hpp:67-79): alpha .01, nperm 200, min_width 2,
 * kmax 25, nmin 200, eta .05, tol 1e-6, hybrid 0, smoothing on (10, 4.0, 2.0, .025), MT seed 1, chain 1 */
void cbs_gpu_default_params(cbs_gpu_params* p);

/* One record per call of the reference's fndcpt (CBS.cpp:830-892) */
typedef struct cbs_gpu_split {
    int32_t unit, lo, hi;       /* segment tested, [lo,hi) in markers of the unit */
    double ostat;               /* observed max-t statistic (ChangePointResult::ostat) */
    int32_t iseg0, iseg1;       /* ChangePointResult::iseg (0-based) */
    int32_t ncpt, icpt0, icpt1; /* ChangePointResult::ncpt / icpt */
    int32_t perms_run, nrej, exit_code, called;
    int32_t e_nrej0, e_nrej1, e_status0, e_status1;
} cbs_gpu_split;

/* Library-allocated result of a batched call; release with cbs_gpu_result_free. */
typedef struct cbs_gpu_result {
    int32_t n_units;
    int64_t n_segments;
    const int64_t* seg_offsets;     /* [n_units+1] into lengths/means */
    const int32_t* lengths;         /* SegmentationResult::lengths, concatenated */
    const double* means;            /* SegmentationResult::means, concatenated */
    const uint64_t* draws_consumed; /* [n_units], uniforms taken from the engine (MT mode) */
    int64_t n_splits;
    const cbs_gpu_split* splits;    /* only with record_splits */
    int32_t rounds;                 /* scheduler rounds executed */
    uint64_t perms_run;             /* max-t permutations actually evaluated */
    uint64_t perm_elements;         /* sum over those permutations of the segment length (markers shuffled) */
    uint64_t kernel_launches;       /* kernels launched by this call */
    double ms_h2d, ms_smooth, ms_segment, ms_d2h; /* CUDA-event timings on the call's stream */
    double ms_call;                 /* host wall clock of the whole call (buffer growth, staging and read-back included) */
} cbs_gpu_result;

/* ---- context -----------------------------------------------------------------------
 * One context drives ONE device (the process-per-GPU model); device_ids[0] is used, ndev must
 * be 1.  A context is not thread-safe. */
int cbs_gpu_create(const int* device_ids, int ndev, cbs_gpu_ctx** out);
void cbs_gpu_destroy(cbs_gpu_ctx* ctx);
const char* cbs_gpu_last_error(const cbs_gpu_ctx* ctx);
/* launch the round kernels on this CUDA stream (cudaStream_t) instead of the context's own */
int cbs_gpu_set_stream(cbs_gpu_ctx* ctx, void* cuda_stream);

/* ---- batched entry: replaces the loop body of Segment::segment_raw ------------------
 * (src/cna_segment.hpp:132-157): for every unit (one chromosome of one sample):
 *   x = widen(values[unit]);  if do_smooth: x = cbs::smooth(x, const label);  cbs::segment(x, ...)
 * values: all units end to end, float32 or float64, in host or device memory;
 * unit_offsets: host, [n_units+1]; unit_ids: host, global ids used for Philox keys (NULL = index).
 * Empty units yield zero segments (cna_segment.hpp:138). */
int cbs_gpu_segment_batch(cbs_gpu_ctx* ctx, const void* values, int dtype, int memspace, const int64_t* unit_offsets,
                          const uint64_t* unit_ids, int32_t n_units, const cbs_gpu_params* params,
                          cbs_gpu_result** out);
void cbs_gpu_result_free(cbs_gpu_result* r);

/* ---- single-call surface -------------------------------------------------------------
 * cbs::smooth (lib/cbs/smooth.hpp:8-13, smooth.cpp:119-153): values/chrom/out host arrays of n. */
int cbs_gpu_smooth(cbs_gpu_ctx* ctx, const double* values, const int32_t* chrom, int64_t n, int32_t smooth_region,
                   double outlier_sd_scale, double smooth_sd_scale, double trim, double* out);

/* cbs::segment (lib/cbs/CBS.hpp:100-113, CBS.cpp:959-1024) on one vector.
 * mt_next312 (MT mode, may be NULL): the NEXT 312 raw (untempered) words of the caller's
 * std::mt19937_64, i.e. the engine state in the form the device generator continues from;
 * NULL = engine freshly seeded with params->seed.  *draws_consumed tells the caller how far to
 * discard() its engine afterwards.  Returns CBS_GPU_ERR_CAPACITY if cap is too small
 * (*n_segments then holds the needed size). */
int cbs_gpu_segment(cbs_gpu_ctx* ctx, const double* x, int32_t n, const cbs_gpu_params* params,
                    const uint64_t* mt_next312, int32_t cap, int32_t* lengths, double* means, int32_t* n_segments,
                    uint64_t* draws_consumed);

/* cbs::segment_weighted (lib/cbs/CBS.hpp:115-128, CBS.cpp:1026-1099) on one vector: wfindcpt / wtmaxo / wtmaxp (with the
 * reference's tss = 0 placeholder, CBS.cpp:741-743, mirrored) / wxperm / wtpermp on the device.  weights must be finite
 * and positive.  hybrid = 1 selects the weighted hybrid method (getmncwt / hwtmaxp, CBS.cpp:593-608, 745-828) for
 * segments longer than nmin, as in the reference.  Other arguments as cbs_gpu_segment. */
int cbs_gpu_segment_weighted(cbs_gpu_ctx* ctx, const double* x, const double* weights, int32_t n,
                             const cbs_gpu_params* params, const uint64_t* mt_next312, int32_t cap, int32_t* lengths,
                             double* means, int32_t* n_segments, uint64_t* draws_consumed);
/* the same for many units at once (values and weights: float64, laid out alike, host or device memory); no smoothing */
int cbs_gpu_segment_weighted_batch(cbs_gpu_ctx* ctx, const double* values, const double* weights, int memspace,
                                   const int64_t* unit_offsets, const uint64_t* unit_ids, int32_t n_units,
                                   const cbs_gpu_params* params, cbs_gpu_result** out);

/* cbs::tmaxo (CBS.hpp:32, CBS.cpp:378-381): max-t statistic and 0-based arc of x as given
 * (no centring), with tss supplied by the caller. */
int cbs_gpu_tmaxo(cbs_gpu_ctx* ctx, const double* x, int32_t n, double tss, int32_t al0, int32_t ibin,
                  double* statistic, int32_t* start, int32_t* end);
/* cbs::tmaxp (CBS.hpp:33, CBS.cpp:383-385) for `count` vectors of length n laid end to end */
int cbs_gpu_tmaxp(cbs_gpu_ctx* ctx, const double* px, int32_t n, int32_t count, double tss, int32_t al0, int32_t ibin,
                  double* statistics);

/* ---- low-level call surface (lib/cbs/CBS.hpp:29-98), each ONE decision on the vector as given ---------------------
 * cbs::fndcpt (CBS.hpp:68-80, CBS.cpp:830-892): x is the centred segment, tss its sum of squares (both as the caller
 * computed them); params supplies cpval (alpha), nperm, hybrid, al0 (min_width), hk (kmax), tol and the RNG; delta is the
 * hybrid method's argument (0: (kmax+1)/n), ngrid must be 100.  sbdry is not an argument: `cna segment` disables the
 * sequential boundary (src/cna_segment.hpp:130) and so does this library.  The result comes back as a split record:
 * ncpt, icpt0/icpt1, iseg0/iseg1 (0-based, as cbs::ChangePointResult), ostat, plus perms_run, nrej and the edge tests'
 * counts for diagnostics.  mt_next312 / draws_consumed as in cbs_gpu_segment. */
int cbs_gpu_fndcpt(cbs_gpu_ctx* ctx, const double* x, int32_t n, double tss, const cbs_gpu_params* params, double delta,
                   int32_t ngrid, const uint64_t* mt_next312, cbs_gpu_split* out, uint64_t* draws_consumed);
/* cbs::wfindcpt (CBS.hpp:81-97, CBS.cpp:894-957).  The reference also takes rwts = sqrt(wts) and cwts =
 * cumsum(wts)/sqrt(sum wts); they are derived from `weights` on the device with the reference's own expressions
 * (CBS.cpp:1056-1066), and delta comes from getmncwt as in wfindcpt (:908). */
int cbs_gpu_wfindcpt(cbs_gpu_ctx* ctx, const double* x, const double* weights, int32_t n, double tss,
                     const cbs_gpu_params* params, int32_t ngrid, const uint64_t* mt_next312, cbs_gpu_split* out,
                     uint64_t* draws_consumed);
/* cbs::tpermp (CBS.hpp:35-36, CBS.cpp:495-536): permutation p-value of the boundary between x[0..n1) and x[n1..n1+n2);
 * params supplies nperm and the RNG */
int cbs_gpu_tpermp(cbs_gpu_ctx* ctx, const double* x, int32_t n1, int32_t n2, const cbs_gpu_params* params,
                   const uint64_t* mt_next312, double* pvalue, uint64_t* draws_consumed);

/* cbs::wtmaxo (CBS.hpp:54-58, CBS.cpp:610-739): weighted max-t statistic and 0-based arc of x as given, tss supplied by
 * the caller; cwts is derived from `weights` as in cbs::segment_weighted (CBS.cpp:1062-1066). */
int cbs_gpu_wtmaxo(cbs_gpu_ctx* ctx, const double* x, const double* weights, int32_t n, double tss, int32_t al0,
                   double* statistic, int32_t* start, int32_t* end);
/* cbs::xperm (CBS.hpp:37, CBS.cpp:487-493) and, with rwts != NULL, cbs::wxperm (CBS.hpp:39-42, CBS.cpp:538-547): ONE
 * permutation px of x drawn from the engine whose next 312 raw words are mt_next312 (NULL: std::mt19937_64(seed)); the
 * engine advances by exactly n draws. */
int cbs_gpu_xperm(cbs_gpu_ctx* ctx, const double* x, const double* rwts, int32_t n, const uint64_t* mt_next312, uint64_t seed,
                  double* px);
/* cbs::htmaxp (CBS.hpp:34, CBS.cpp:387-485) for `count` vectors of length n laid end to end; ibin must be 0 */
int cbs_gpu_htmaxp(cbs_gpu_ctx* ctx, const double* px, int32_t n, int32_t count, double tss, int32_t k, int32_t al0,
                   int32_t ibin, double* statistics);
/* cbs::tailp (CBS.hpp:29, CBS.cpp:324-339); ngrid must be 100.  Evaluated with the CUDA erfc/log/exp/pow (<= 4 ulp each), so
 * the value agrees with the reference's libm result to ~1e-14 relative, not bit for bit. */
int cbs_gpu_tailp(cbs_gpu_ctx* ctx, double b, double delta, int32_t m, int32_t ngrid, double tol, double* out);
/* binary-data helpers, off the `cna segment` path: cbs::btmax (CBS.hpp:31, CBS.cpp:363-376), cbs::btailp (CBS.hpp:30,
 * CBS.cpp:341-361); cbs_gpu_tmaxo / cbs_gpu_tmaxp accept ibin = 1 (CBS.cpp:68-227, ibin branches) */
int cbs_gpu_btmax(cbs_gpu_ctx* ctx, const double* x, int32_t n, double* out);
int cbs_gpu_btailp(cbs_gpu_ctx* ctx, double b, int32_t m, int32_t ng, double tol, double* out);

/* ---- downstream of the segment table (SURVEY 8 row f4) ---------------------------------
 * cngpld::summarize_cn (lib/cngpld/summarize.hpp:28-34, summarize.cpp:77-100) for every unit (one chromosome of one
 * sample) of a segment table: at every position -- by default the sorted distinct segment starts and ends of the unit
 * (summarize.cpp:24-36) -- the sum of exp(direction * value) over the overlapping segments with direction * value > cutoff,
 * divided by the number of overlapping segments (0 if none is altered; summarize.cpp:41-75).
 * seg_offsets: [n_units+1] into seg_start / seg_end / seg_value (float = the reference's rvalue).
 * positions == NULL: default positions; out_offsets [n_units+1], out_pos / out_value need room for 2 * n_segments.
 * positions != NULL: pos_offsets [n_units+1] into positions; out_pos / out_value need room for pos_offsets[n_units]
 * (out_pos receives a copy).  direction must be 1 or -1 and every segment needs start <= end (INVALID otherwise, the
 * reference's std::invalid_argument). */
int cbs_gpu_summarize_cn(cbs_gpu_ctx* ctx, const int64_t* seg_offsets, int32_t n_units, const uint64_t* seg_start,
                         const uint64_t* seg_end, const float* seg_value, int32_t direction, double cutoff,
                         const int64_t* pos_offsets, const uint64_t* positions, int64_t* out_offsets, uint64_t* out_pos,
                         double* out_value);

/* host-only self test (needs no device): 0 if the MT19937-64 jump-ahead polynomials reproduce
 * sequential generation */
int cbs_gpu_selftest(void);

/* ---- device info / peak measurement helpers (used by bench.py) -------------------------
 * Measured FP64 add+compare issue rate of this device with the library's own microbenchmark:
 * returns 1e12 double-precision pipe instructions per second. */
int cbs_gpu_measure_fp64(cbs_gpu_ctx* ctx, double* tera_inst_per_s);
/* timing (CUDA events) of the kernels of the last batched call, ms summed per kernel:
 * order: sched, gen, prep, perm (global-memory shuffle), scan, edgeprep, edgeperm, means, smooth,
 * shuf0..shuf3 (shared-memory shuffle by length class), prefix */
int cbs_gpu_last_kernel_ms(cbs_gpu_ctx* ctx, double* ms14);
/* bit 0: bracket every kernel launch with CUDA events (cbs_gpu_last_kernel_ms);
 * bit 1: count scan-kernel work with device atomics (cbs_gpu_last_arc_evals) -- this slows the scan
 * kernel several times, so time and count in separate calls;
 * bit 2: launch every kernel of a round on the one stream instead of the side streams, so that the per-launch event
 * times do not overlap (time base of the per-kernel roofline; slower than the normal, overlapped schedule) */
int cbs_gpu_set_profiling(cbs_gpu_ctx* ctx, int on);
/* scan-kernel work of the last batched call (needs profiling on): arcs = real (i,j) pairs examined
 * by the inner loop, slots = compare slots issued (arcs + padding of partially filled units) */
int cbs_gpu_last_arc_evals(cbs_gpu_ctx* ctx, uint64_t* arcs, uint64_t* slots);

#ifdef __cplusplus
}
#endif
#endif
