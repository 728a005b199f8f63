/* TEST INFRASTRUCTURE -- NOT PRODUCT CODE.
 *
 * CPU restatement (plain C) of the reference's CBS + smoothing hot path
 * (djhshih/genomic: lib/cbs/CBS.cpp, lib/cbs/smooth.cpp, src/cna_segment.hpp:127-159).
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
 * legs may load liboracle.so, and only as the checker.
 *
 * Parity pin: every entry point here is checked bit-for-bit against the UNMODIFIED
 * reference sources compiled into oracle/_ref/libcbs_ref.so (tests/test_oracle_vs_ref.py)
 * and against the reference's own golden vectors (tests/golden/, SURVEY 8c).
 */
#ifndef CBS_ORACLE_H
#define CBS_ORACLE_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- random sources ---------------------------------------------------------
 * kind 0: std::mt19937_64 replay (one serial stream; CBS.cpp:53-55 + libstdc++ 13
 *         generate_canonical<double,53>, see SURVEY A.2)
 * kind 1: Philox4x32-10 counter mode used by the product's fast mode; the uniform for
 *         (stage, perm, k) is a pure function of (key, stage, perm, k).            */
typedef struct orc_rng {
    int kind;
    uint64_t mt[312];
    int mti;
    uint64_t draws; /* uniforms handed out so far (MT: stream position) */
    uint32_t key0, key1;
    uint32_t stage, perm, k;
} orc_rng;

void orc_rng_seed_mt(orc_rng* r, uint64_t seed);
void orc_rng_seed_philox(orc_rng* r, uint64_t seed);
/* philox: derive the per-task key from (seed, unit id, lo, hi) */
void orc_rng_set_task(orc_rng* r, uint64_t seed, uint64_t unit_id, uint32_t lo, uint32_t hi);
void orc_rng_begin(orc_rng* r, uint32_t stage, uint32_t perm);
uint64_t orc_rng_u64(orc_rng* r);
double orc_rng_unif(orc_rng* r);
void orc_rng_discard(orc_rng* r, uint64_t n);
void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
uint64_t orc_task_key(uint64_t seed, uint64_t unit_id, uint32_t lo, uint32_t hi);

/* ---- max-t arc scan (CBS.cpp:68-227, 378-385) ------------------------------- */
typedef struct orc_tmax {
    double stat;
    int start, end; /* 0-based as cbs::tmaxo returns them (tmaxi-1, tmaxj-1) */
} orc_tmax;
orc_tmax orc_tmaxo(const double* x, int n, double tss, int al0, int ibin);
double orc_tmaxp(const double* px, int n, double tss, int al0, int ibin);
double orc_htmaxp(const double* px, int n, double tss, int k, int al0, int ibin);
double orc_tailp(double b, double delta, int m, int ngrid, double tol);

/* instrumentation: arcs evaluated by the inner loops since last reset */
uint64_t orc_arc_evals(void);
void orc_arc_evals_reset(void);

/* ---- permutation pieces (CBS.cpp:487-536) ------------------------------------ */
void orc_xperm(const double* x, int n, double* px, orc_rng* rng);
double orc_tpermp(int n1, int n2, int n, const double* x, int nperm, orc_rng* rng, double* scratch);

/* ---- one split decision (CBS.cpp:830-892) ------------------------------------- */
typedef struct orc_cpt {
    int ncpt;
    int icpt[2];
    int iseg[2];
    double ostat;
    /* diagnostics (not in the reference struct) */
    int perms_run; /* permutations executed in the max-t loop */
    int nrej;
    int exit_code;   /* 0 none, 1 t<=0.1, 2 shortcut t>=7, 3 early exit nrej>nrejc, 4 hybrid tail p>alpha */
    double edge_p[2]; /* tpermp p-values, -1 when not run */
} orc_cpt;
orc_cpt orc_fndcpt(const double* x, int n, double tss, int nperm, double cpval, int ibin, int hybrid, int al0, int hk,
                   double delta, int ngrid, double tol, orc_rng* rng);

/* ---- recursive driver (CBS.cpp:959-1024) --------------------------------------- */
typedef struct orc_split_rec {
    int lo, hi;     /* segment tested, [lo,hi) within the unit */
    double ostat;   /* observed statistic (0 when fndcpt was not called) */
    int iseg0, iseg1;
    int ncpt, icpt0, icpt1;
    int perms_run, nrej, exit_code;
    int called; /* 1 if fndcpt ran, 0 if skipped (too short / all equal) */
    double edge_p0, edge_p1; /* tpermp p-values of the two boundaries (CBS.cpp:877,883), -1 when not run */
} orc_split_rec;

typedef struct orc_seg_opts {
    int ibin;
    double alpha;
    int nperm;
    int hybrid;
    int min_width;
    int kmax;
    int nmin;
    double eta; /* accepted, unused (as in the reference) */
    double tol;
    int undo_prune;
    double undo_prune_cutoff;
} orc_seg_opts;

/* returns number of segments (lengths/means filled up to cap) or -needed.
 * log/log_cap/log_n may be NULL/0: split log in processing order.
 * philox mode: unit_id + seed are needed to key each task. */
int orc_segment(const double* x, int n, const orc_seg_opts* o, orc_rng* rng, uint64_t seed, uint64_t unit_id, int cap,
                int* lengths, double* means, orc_split_rec* log, int log_cap, int* log_n);

/* ---- smoothing (smooth.cpp:13-153) -------------------------------------------- */
double orc_norm_quantile(double p);
double orc_inflfact(double trim); /* NaN if trim invalid */
/* 0 ok; 1 invalid argument (what the reference throws std::invalid_argument for);
 * 2 overflow (trim == 0 reaches boost quantile(nd, 1.0) -> std::overflow_error) */
int orc_smooth(const double* values, const int* chrom, int64_t n, int smooth_region, double outlier_sd_scale,
               double smooth_sd_scale, double trim, double* out);

/* ---- cohort loop (cna_segment.hpp:127-159) -------------------------------------- */
typedef struct orc_cohort_opts {
    orc_seg_opts seg;
    int do_smooth;
    int smooth_region;
    double outlier_sd_scale, smooth_sd_scale, trim;
    int rng_kind; /* 0 MT replay, 1 philox */
    uint64_t seed;
    int chain; /* MT only: 1 = one stream across all units, 0 = fresh stream per unit */
} orc_cohort_opts;

/* unit_ids may be NULL (then unit id = index).  draws_out[u] (may be NULL): MT draws
 * consumed by unit u.  Returns total segments, -1 if cap too small, -2 invalid argument. */
int64_t orc_segment_units(const double* values, const int64_t* unit_off, const int* chrom_label,
                          const uint64_t* unit_ids, int n_units, const orc_cohort_opts* o, int64_t cap, int* seg_count,
                          int* lengths, double* means, uint64_t* draws_out, orc_split_rec* log, int64_t log_cap,
                          int64_t* log_n, int* log_unit);

/* ---- weighted CBS (cbs_oracle_weighted.c; CBS.cpp:538-591, 610-743, 894-957, 1026-1099) ---------------
 * cw = cumsum(w)/sqrt(sum w) as segment_weighted builds it (:1062-1066); rw = sqrt(w). */
orc_tmax orc_wtmaxo(const double* x, const double* w, const double* cw, int n, double tss, int al0);
double orc_wtmaxp(const double* px, const double* w, const double* cw, int n, int al0);
void orc_wxperm(const double* x, const double* rw, int n, double* px, orc_rng* rng);
double orc_wtpermp(int n1, int n2, int n, const double* x, const double* w, const double* rw, int nperm, orc_rng* rng,
                   double* scratch);
void orc_getmncwt(const double* cw, int n, int k, double* mn, double* delta);
double orc_hwtmaxp(const double* px, const double* w, const double* cw, const double* mn, int n, int k, int al0);
/* one wfindcpt decision on x as given (centred, with the caller's tss); rw = sqrt(w) and cw are derived from w as
 * segment_weighted derives them */
orc_cpt orc_wfindcpt(const double* x, const double* w, int n, double tss, int nperm, double cpval, int hybrid, int al0,
                     int hk, int ngrid, double tol, orc_rng* rng);
/* segments, or -needed-16 if cap is too small, or -4 (ORC_W_SELF_SPLIT) when a decision would re-create its own segment.
 *
 * -4 is the one place where this restatement knowingly departs from the reference.  When one weight carries nearly all of
 * the total, cw is not strictly increasing, an arc of weight 0 has an infinite statistic and ostat becomes NaN; no
 * permutation rejects and the change point lands on the segment's last marker, so [lo,hi) splits into [lo,hi) and
 * [hi,hi).  The reference (CBS.cpp:996-1004) then tests [lo,hi) again, with the same outcome, forever.  Here the driver
 * stops at the first decision that would re-create its own segment and returns -4; the split log ends with that decision.
 * The _log forms also fill a split log in processing order, as orc_segment does. */
int orc_segment_weighted(const double* x, const double* w, int n, const orc_seg_opts* o, orc_rng* rng, uint64_t seed,
                         uint64_t unit_id, int cap, int* lengths, double* means);
int orc_segment_weighted_log(const double* x, const double* w, int n, const orc_seg_opts* o, orc_rng* rng, uint64_t seed,
                             uint64_t unit_id, int cap, int* lengths, double* means, orc_split_rec* log, int log_cap,
                             int* log_n);
/* total segments, -1 if cap is too small, -4 as above */
int64_t orc_segment_weighted_units(const double* values, const double* weights, const int64_t* unit_off,
                                   const uint64_t* unit_ids, int n_units, const orc_cohort_opts* o, int64_t cap,
                                   int* seg_count, int* lengths, double* means, uint64_t* draws_out);
int64_t orc_segment_weighted_units_log(const double* values, const double* weights, const int64_t* unit_off,
                                       const uint64_t* unit_ids, int n_units, const orc_cohort_opts* o, int64_t cap,
                                       int* seg_count, int* lengths, double* means, uint64_t* draws_out,
                                       orc_split_rec* log, int64_t log_cap, int64_t* log_n, int* log_unit);

#ifdef __cplusplus
}
#endif
#endif
