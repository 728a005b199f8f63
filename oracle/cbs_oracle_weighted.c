/* TEST INFRASTRUCTURE -- never imported by the product path.
 *
 * Weighted CBS: CPU restatement of cbs::segment_weighted and what it calls
 * (/root/reference lib/cbs/CBS.cpp: wxperm :538-547, wtpermp :549-591, wtmaxo :610-739,
 * wtmaxp :741-743, wfindcpt :894-957, segment_weighted :1026-1099).
 * Compiled as part of cbs_oracle.c (included at its end: it uses that file's RNG, its
 * libstdc++-style index sort and its prune restatement).
 *
 * Pinned: bit-identical to the compiled reference (oracle/_ref, ref_segment_weighted) on
 * randomized inputs, and reproduces the inline KAT of tests/cbs_test.cpp:309-330
 * (15/15/15/15, means 0/2/-1.5/0) -- tests/test_oracle.py.
 *
 * The weighted hybrid method (getmncwt :593-608, hwtmaxp :745-828, the hybrid branch of wfindcpt
 * :908-921) is restated too and pinned the same way.
 */

#define ORC_W_UNSUPPORTED (-3) /* kept for the ABI of the python wrapper; no longer returned */
#define ORC_W_SELF_SPLIT (-4)  /* see cbs_oracle.h: a decision that would re-create its own segment */

/* ---- wtmaxo / wtmaxp ------------------------------------------------------------ */
typedef struct {
    int n, nb, al0;
    const double* s;  /* weighted prefix sums s[0..n] */
    const double* cw; /* cumulative weights (scaled), cw[0..n-1] */
    const int* bb;    /* block ends bb[0..nb], bb[0] = 0 */
    double total;     /* cw[n-1] */
} wrow;

typedef struct { double best; int i, j; } wbest;

/* statistic of the arc (i, j), 1-based prefix indices, arc weight a (:714,728) */
static inline double warc(const wrow* r, int i, int j, double a) {
    const double d = r->s[j] - r->s[i];
    return (d * d) / (a * (r->total - a));
}

/* low band of a block pair (:708-719): arcs with weight <= cap, i descending, j ascending */
static void wscan_low(const wrow* r, int bi, int bj, double cap, wbest* m) {
    const int ilo = r->bb[bi - 1] + 1, ihi = r->bb[bi], jlo = r->bb[bj - 1] + 1, jhi = r->bb[bj];
    const int itop = (bi == bj) ? ihi - r->al0 : ihi;
    for (int i = itop; i >= ilo; --i) {
        const int jfirst = imax(i + r->al0, jlo);
        for (int j = jfirst; j <= jhi; ++j) {
            const double a = r->cw[j - 1] - r->cw[i - 1];
            if (a <= cap) {
                const double v = warc(r, i, j, a);
                if (v > m->best) { m->best = v; m->i = i; m->j = j; }
            }
        }
    }
}

/* high band (:721-733): arcs with weight >= floor_, i ascending, j descending; the pair (1, nb) keeps al0 markers out */
static void wscan_high(const wrow* r, int bi, int bj, double floor_, wbest* m) {
    const int ilo = r->bb[bi - 1] + 1, ihi = r->bb[bi], jlo = r->bb[bj - 1] + 1, jhi = r->bb[bj];
    const int wrap = (bi == 1) && (bj == r->nb);
    for (int i = ilo; i <= ihi; ++i) {
        const int jtop = wrap ? imin(jhi, jhi - r->al0 + i) : jhi;
        for (int j = jtop; j >= jlo; --j) {
            const double a = r->cw[j - 1] - r->cw[i - 1];
            if (a >= floor_) {
                const double v = warc(r, i, j, a);
                if (v > m->best) { m->best = v; m->i = i; m->j = j; }
            }
        }
    }
}

orc_tmax orc_wtmaxo(const double* x, const double* w, const double* cw, int n, double tss, int al0) {
    const double rn = (double)n;
    const int nb = block_count(n);
    const int npair = nb * (nb + 1) / 2;
    double* s = (double*)calloc((size_t)n + 1, sizeof(double));
    int* bb = (int*)malloc(sizeof(int) * (size_t)(nb + 1));
    double* bmin = (double*)malloc(sizeof(double) * (size_t)(nb + 1));
    double* bmax = (double*)malloc(sizeof(double) * (size_t)(nb + 1));
    int* amin = (int*)malloc(sizeof(int) * (size_t)(nb + 1));
    int* amax = (int*)malloc(sizeof(int) * (size_t)(nb + 1));
    double* corner = (double*)malloc(sizeof(double) * (size_t)(npair + 1));
    double* bound = (double*)malloc(sizeof(double) * (size_t)(npair + 1));
    double* cornw = (double*)malloc(sizeof(double) * (size_t)(npair + 1));
    int* pi = (int*)malloc(sizeof(int) * (size_t)(npair + 1));
    int* pj = (int*)malloc(sizeof(int) * (size_t)(npair + 1));
    int* order = (int*)malloc(sizeof(int) * (size_t)(npair + 1));
    bb[0] = 0;
    block_ends(n, nb, bb);

    /* :617-637 sequential weighted prefix sums, block extrema with their first occurrence, global extrema
       (start at 0.0 with index n) */
    double g_lo = 0.0, g_hi = 0.0;
    int gi_lo = n, gi_hi = n;
    for (int b = 1; b <= nb; ++b) {
        const int first = bb[b - 1] + 1, last = bb[b];
        for (int i = first; i <= last; ++i) s[i] = s[i - 1] + x[i - 1] * w[i - 1];
        double lo = s[first], hi = s[first];
        int ilo = first, ihi = first;
        for (int i = first + 1; i <= last; ++i) {
            if (s[i] < lo) { lo = s[i]; ilo = i; }
            if (s[i] > hi) { hi = s[i]; ihi = i; }
        }
        bmin[b] = lo; bmax[b] = hi; amin[b] = ilo; amax[b] = ihi;
        if (lo < g_lo) { g_lo = lo; gi_lo = ilo; }
        if (hi > g_hi) { g_hi = hi; gi_hi = ihi; }
    }

    orc_tmax out;
    wbest m;
    m.best = 0.0; m.i = imin(gi_hi, gi_lo); m.j = imax(gi_hi, gi_lo);
    const double spread = g_hi - g_lo;
    int degenerate = 0;
    if (spread <= 0.0) {
        degenerate = 1; /* :642-645: location returned WITHOUT the -1 shift */
    } else {
        wrow r;
        r.n = n; r.nb = nb; r.al0 = al0; r.s = s; r.cw = cw; r.bb = bb; r.total = cw[n - 1];
        const double half = r.total / 2.0;
        const double a0 = fabs(cw[gi_hi - 1] - cw[gi_lo - 1]);
        m.best = (spread * spread) / (a0 * (r.total - a0)); /* :649 */
        const int nal0 = n - al0;
        int nlist = 0;
        for (int bi = 1; bi <= nb; ++bi) {
            for (int bj = bi; bj <= nb; ++bj) {
                const int ilo = bb[bi - 1] + 1, ihi = bb[bi], jlo = bb[bj - 1] + 1, jhi = bb[bj];
                /* largest and smallest arc weight of the pair (:656-671) */
                double whi = cw[jhi - 1] - cw[ilo - 1];
                if (jhi - ilo > nal0) {
                    whi = 0.0;
                    for (int k = 1; k <= al0; ++k) whi = fmax(whi, cw[nal0 + k - 1] - cw[k - 1]);
                }
                double wlo;
                if (bi == bj) {
                    wlo = cw[ilo + al0 - 1] - cw[ilo - 1];
                    for (int k = ilo + 1; k <= ihi - al0; ++k) wlo = fmin(wlo, cw[k + al0 - 1] - cw[k - 1]);
                } else if (bi + 1 == bj) {
                    wlo = cw[jlo - 1] - cw[jlo - al0 - 1];
                    for (int k = jlo - al0 + 1; k <= ihi; ++k) wlo = fmin(wlo, cw[k + al0 - 1] - cw[k - 1]);
                } else {
                    wlo = cw[jlo - 1] - cw[ihi - 1];
                }
                const double d1 = fabs(bmax[bj] - bmin[bi]), d2 = fabs(bmax[bi] - bmin[bj]);
                const double dmax = fmax(d1, d2);
                const double lim = (dmax * dmax) / fmin(wlo * (r.total - wlo), whi * (r.total - whi));
                if (m.best <= lim) { /* :677-690 */
                    ++nlist;
                    order[nlist] = nlist; pi[nlist] = bi; pj[nlist] = bj; bound[nlist] = lim;
                    if (d1 > d2) {
                        cornw[nlist] = fabs(cw[amax[bj] - 1] - cw[amin[bi] - 1]);
                        corner[nlist] = (d1 * d1) / (cornw[nlist] * (r.total - cornw[nlist]));
                    } else {
                        cornw[nlist] = fabs(cw[amin[bj] - 1] - cw[amax[bi] - 1]);
                        corner[nlist] = (d2 * d2) / (cornw[nlist] * (r.total - cornw[nlist]));
                    }
                }
            }
        }
        sort_indices_like_libstdcxx(order + 1, order + nlist + 1, corner); /* :695 */
        for (int t = nlist; t >= 1; --t) {
            const int k = order[t];
            if (m.best > bound[k]) continue;
            const int bi = pi[k], bj = pj[k];
            const int ilo = bb[bi - 1] + 1, ihi = bb[bi], jlo = bb[bj - 1] + 1, jhi = bb[bj];
            const double whi = cw[jhi - 1] - cw[ilo - 1];
            const double wlo = (bi == bj) ? 0.0 : (cw[jlo - 1] - cw[ihi - 1]);
            double cap = cornw[k];
            if (cap > r.total - cap) cap = r.total - cap;
            if (wlo <= half) wscan_low(&r, bi, bj, cap, &m);
            if (whi >= half) wscan_high(&r, bi, bj, r.total - cap, &m);
        }
    }
    if (tss <= m.best + 0.0001) tss = m.best + 1.0;
    out.stat = m.best / ((tss - m.best) / (rn - 2.0));
    out.start = degenerate ? m.i : m.i - 1;
    out.end = degenerate ? m.j : m.j - 1;
    free(s); free(bb); free(bmin); free(bmax); free(amin); free(amax); free(corner); free(bound); free(cornw);
    free(pi); free(pj); free(order);
    return out;
}

/* :741-743 -- the reference passes tss = 0.0 (placeholder); mirrored */
double orc_wtmaxp(const double* px, const double* w, const double* cw, int n, int al0) {
    return orc_wtmaxo(px, w, cw, n, 0.0, al0).stat;
}

/* ---- permutations ---------------------------------------------------------------- */
/* :538-547: Fisher-Yates on x*rw; the element that lands on position i-1 is divided by rw[i-1] -- except when j == i,
   where the final store puts the undivided value back */
void orc_wxperm(const double* x, const double* rw, int n, double* px, orc_rng* rng) {
    for (int i = 0; i < n; ++i) px[i] = x[i] * rw[i];
    for (int i = n; i >= 1; --i) {
        const int j = (int)(orc_rng_unif(rng) * (double)i) + 1;
        const double keep = px[i - 1];
        px[i - 1] = px[j - 1] / rw[i - 1];
        px[j - 1] = keep;
    }
}

/* :549-591 */
double orc_wtpermp(int n1, int n2, int n, const double* x, const double* w, const double* rw, int nperm, orc_rng* rng,
                   double* px) {
    if (n1 == 1 || n2 == 1) return 1.0;
    double sum1 = 0.0, sum2 = 0.0, tss = 0.0, w1 = 0.0, w2 = 0.0;
    for (int i = 0; i < n1; ++i) { sum1 += w[i] * x[i]; tss += w[i] * x[i] * x[i]; w1 += w[i]; }
    for (int i = n1; i < n; ++i) { sum2 += w[i] * x[i]; tss += w[i] * x[i] * x[i]; w2 += w[i]; }
    const double wt = w1 + w2;
    const double xbar = (sum1 + sum2) / wt;
    tss -= wt * (xbar * xbar);
    int m1;
    double wm1, ostat, tstat;
    if (n1 <= n2) { m1 = n1; wm1 = w1; ostat = 0.99999 * fabs(sum1 / w1 - xbar); tstat = (ostat * ostat) * w1 * wt / w2; }
    else          { m1 = n2; wm1 = w2; ostat = 0.99999 * fabs(sum2 / w2 - xbar); tstat = (ostat * ostat) * w2 * wt / w1; }
    tstat /= ((tss - tstat) / ((double)n - 2.0));
    if (tstat > 25.0 && m1 >= 10) return 0.0;
    int nrej = 0;
    const uint32_t stage = rng->stage;
    for (int np = 1; np <= nperm; ++np) {
        orc_rng_begin(rng, stage, (uint32_t)(np - 1));
        for (int i = 0; i < n1; ++i) px[i] = x[i] * rw[i];
        for (int i = n1; i < n; ++i) px[i] = x[i];
        double acc = 0.0;
        for (int i = n; i >= n - m1 + 1; --i) {
            const int j = (int)(orc_rng_unif(rng) * (double)i) + 1;
            const double t = px[i - 1]; px[i - 1] = px[j - 1]; px[j - 1] = t;
            acc += px[i - 1] * rw[i - 1];
        }
        if (ostat <= fabs(acc / wm1 - xbar)) ++nrej;
    }
    return (double)nrej / (double)nperm;
}

/* ---- weighted hybrid pieces ------------------------------------------------------------ */
/* smallest weight of an arc of `len` markers, wrap-around arcs included (the loop body of getmncwt, :597-601 / :603-607) */
static double min_arc_weight(const double* cw, int n, int len) {
    const double total = cw[n - 1];
    const int rest = n - len;
    double m = cw[len - 1];
    for (int i = 1; i <= rest; ++i) m = fmin(m, cw[i + len - 1] - cw[i - 1]);
    for (int i = 1; i <= len; ++i) m = fmin(m, total - (cw[i + rest - 1] - cw[i - 1]));
    return m;
}

/* getmncwt :593-608: mn[1..k] and delta = min weight of a (k+1)-marker arc / total weight */
void orc_getmncwt(const double* cw, int n, int k, double* mn, double* delta) {
    mn[0] = 0.0;
    for (int j = 1; j <= k; ++j) mn[j] = min_arc_weight(cw, n, j);
    *delta = min_arc_weight(cw, n, k + 1) / cw[n - 1];
}

/* arcs of al0..k markers starting in [from, to-len] / wrapping around / ending just behind `seam`; a length is only
   looked at while its bound spread^2/(mn(total-mn)) reaches the running maximum (:763-775, :780-790, :795-805) */
static double hw_short_arcs(const double* s, const double* cw, const double* mn, double total, int al0, int k, int n,
                            int mode, int from, int to, int seam, double spread, double out) {
    const double spread_sq = spread * spread;
    for (int len = al0; len <= k; ++len) {
        const double lim = spread_sq / (mn[len] * (total - mn[len]));
        if (lim < out) break;
        int i0, i1, shift;
        if (mode == 0) { i0 = from; i1 = to - len; shift = len; }
        else if (mode == 1) { i0 = 1; i1 = len; shift = n - len; }
        else { i0 = seam + 1 - len; i1 = seam; shift = len; }
        for (int i = i0; i <= i1; ++i) {
            const int j = i + shift;
            const double a = cw[j - 1] - cw[i - 1];
            const double d = s[j] - s[i];
            const double v = (d * d) / (a * (total - a));
            if (v > out) out = v;
        }
    }
    return out;
}

/* hwtmaxp :745-828 */
double orc_hwtmaxp(const double* px, const double* w, const double* cw, const double* mn, int n, int k, int al0) {
    const double rn = (double)n;
    const int nb = (int)(rn / (double)k);
    double* s = (double*)calloc((size_t)n + 2, sizeof(double));
    int* bb = (int*)malloc(sizeof(int) * (size_t)(nb + 1));
    double* bmin = (double*)malloc(sizeof(double) * (size_t)(nb + 1));
    double* bmax = (double*)malloc(sizeof(double) * (size_t)(nb + 1));
    bb[0] = 0;
    block_ends(n, nb, bb);
    const double total = cw[n - 1];
    double run = 0.0, ssq = 0.0, out = 0.0;
    for (int b = 1; b <= nb; ++b) {
        const int first = bb[b - 1] + 1;
        double lo = 0.0, hi = 0.0;
        int ilo = first, ihi = first;
        for (int i = first; i <= bb[b]; ++i) {
            run = run + px[i - 1] * w[i - 1];
            ssq += w[i - 1] * px[i - 1] * px[i - 1];
            s[i] = run;
            if (i == first || run < lo) { lo = run; ilo = i; }
            if (i == first || run > hi) { hi = run; ihi = i; }
        }
        bmin[b] = lo; bmax[b] = hi;
        const int d = abs(ilo - ihi);
        if (d <= k && d >= al0) {
            const double a = fabs(cw[ihi - 1] - cw[ilo - 1]);
            const double df = hi - lo;
            const double v = (df * df) / (a * (total - a));
            if (out < v) out = v;
        }
    }
    const double mean = s[n] / total;
    double tss = ssq - mean * mean; /* :776 */
    out = hw_short_arcs(s, cw, mn, total, al0, k, n, 0, 1, bb[1], 0, bmax[1] - bmin[1], out);
    out = hw_short_arcs(s, cw, mn, total, al0, k, n, 1, 0, 0, 0,
                        fmax(fabs(bmax[1] - bmin[nb]), fabs(bmax[nb] - bmin[1])), out);
    for (int l = 2; l <= nb; ++l) {
        out = hw_short_arcs(s, cw, mn, total, al0, k, n, 0, bb[l - 1] + 1, bb[l], 0, bmax[l] - bmin[l], out);
        out = hw_short_arcs(s, cw, mn, total, al0, k, n, 2, 0, 0, bb[l - 1],
                            fmax(fabs(bmax[l] - bmin[l - 1]), fabs(bmax[l - 1] - bmin[l])), out);
    }
    free(s); free(bb); free(bmin); free(bmax);
    if (tss <= out + 0.0001) tss = out + 1.0;
    return out / ((tss - out) / (rn - 2.0));
}

/* ---- one split decision (wfindcpt :894-957) -------------------------------------------- */
static orc_cpt orc_wfndcpt(const double* x, int n, double tss, const double* w, const double* rw, const double* cw,
                           int nperm, double cpval, int hybrid, int al0, int hk, int ngrid, double tol, orc_rng* rng) {
    orc_cpt r;
    memset(&r, 0, sizeof(r));
    r.edge_p[0] = r.edge_p[1] = -1.0;
    double* px = (double*)malloc(sizeof(double) * (size_t)(n > 0 ? n : 1));
    const orc_tmax obs = orc_wtmaxo(x, w, cw, n, tss, al0);
    r.ostat = obs.stat;
    r.iseg[0] = obs.start;
    r.iseg[1] = obs.end;
    const double t1 = sqrt(obs.stat);
    const double thresh = obs.stat * 0.99999;
    if (t1 <= 0.1) { r.exit_code = 1; free(px); return r; }
    const int i1 = obs.start + 1, i2 = obs.end + 1;
    const int arc = imin(i2 - i1, n - i2 + i1);
    if (!(t1 >= 7.0 && arc >= 10)) {
        int nrejc = (int)(cpval * (double)nperm);
        double* mn = NULL;
        if (hybrid) { /* :908-913: delta is recomputed from the weights */
            double delta = 0.0;
            mn = (double*)malloc(sizeof(double) * (size_t)(hk + 2));
            orc_getmncwt(cw, n, hk, mn, &delta);
            const double p1 = orc_tailp(t1, delta, n, ngrid, tol);
            if (p1 > cpval) { r.exit_code = 4; free(mn); free(px); return r; }
            nrejc = (int)((cpval - p1) * (double)nperm);
        }
        for (int np = 1; np <= nperm; ++np) { /* sbdry never fires on this path (see orc_fndcpt) */
            orc_rng_begin(rng, 0u, (uint32_t)(np - 1));
            orc_wxperm(x, rw, n, px, rng);
            const double p = hybrid ? orc_hwtmaxp(px, w, cw, mn, n, hk, al0) : orc_wtmaxp(px, w, cw, n, al0);
            r.perms_run = np;
            if (thresh <= p) ++r.nrej;
            if (r.nrej > nrejc) { r.exit_code = 3; free(mn); free(px); return r; }
        }
        free(mn);
    } else {
        r.exit_code = 2;
    }
    if (i2 == n) {
        r.ncpt = 1; r.icpt[0] = obs.start;
    } else if (i1 == 0) {
        r.ncpt = 1; r.icpt[0] = obs.end;
    } else {
        int n1 = i1, n12 = i2, n2 = n12 - n1;
        rng->stage = 1u;
        double p = orc_wtpermp(n1, n2, n12, x, w, rw, nperm, rng, px);
        r.edge_p[0] = p;
        if (p <= cpval) { r.ncpt = 1; r.icpt[0] = obs.start; }
        n12 = n - i1; n2 = n - i2; n1 = n12 - n2;
        rng->stage = 2u;
        p = orc_wtpermp(n1, n2, n12, x + i1, w + i1, rw + i1, nperm, rng, px);
        r.edge_p[1] = p;
        if (p <= cpval && r.ncpt < 2) { r.icpt[r.ncpt] = obs.end; ++r.ncpt; }
    }
    free(px);
    return r;
}

/* wfindcpt on a segment as given (the low-level entry): rw and cw derived from w as segment_weighted does (:1056-1066) */
orc_cpt orc_wfindcpt(const double* x, const double* w, int n, double tss, int nperm, double cpval, int hybrid, int al0,
                     int hk, int ngrid, double tol, orc_rng* rng) {
    const size_t nn = (size_t)(n > 0 ? n : 1);
    double* rw = (double*)malloc(sizeof(double) * nn);
    double* cw = (double*)malloc(sizeof(double) * nn);
    double wsum = 0.0;
    for (int i = 0; i < n; ++i) { rw[i] = sqrt(w[i]); wsum += w[i]; }
    const double scale = sqrt(wsum);
    double run = 0.0;
    for (int i = 0; i < n; ++i) { run += w[i]; cw[i] = run / scale; }
    const orc_cpt r = orc_wfndcpt(x, n, tss, w, rw, cw, nperm, cpval, hybrid, al0, hk, ngrid, tol, rng);
    free(rw); free(cw);
    return r;
}

/* ---- recursive driver (segment_weighted :1026-1099) ---------------------------------- */
int orc_segment_weighted(const double* x, const double* w, int n, const orc_seg_opts* o, orc_rng* rng, uint64_t seed,
                         uint64_t unit_id, int cap, int* lengths, double* means) {
    return orc_segment_weighted_log(x, w, n, o, rng, seed, unit_id, cap, lengths, means, NULL, 0, NULL);
}

int orc_segment_weighted_log(const double* x, const double* w, int n, const orc_seg_opts* o, orc_rng* rng, uint64_t seed,
                             uint64_t unit_id, int cap, int* lengths, double* means, orc_split_rec* log, int log_cap,
                             int* log_n) {
    int ends_cap = 64, nends = 2;
    int* ends = (int*)malloc(sizeof(int) * (size_t)ends_cap);
    ends[0] = 0; ends[1] = n;
    int done_cap = 64, ndone = 0;
    int* done = (int*)malloc(sizeof(int) * (size_t)done_cap);
    const size_t nn = (size_t)(n > 0 ? n : 1);
    double* cur = (double*)malloc(sizeof(double) * nn);
    double* rw = (double*)malloc(sizeof(double) * nn);
    double* cw = (double*)malloc(sizeof(double) * nn);
    int unsupported = 0, self_split = 0, nlog = 0;
    while (nends > 1) {
        const int k = nends - 1;
        const int lo = ends[k - 1], hi = ends[k], len = hi - lo;
        orc_cpt z;
        memset(&z, 0, sizeof(z));
        int called = 0;
        if (len >= 2 * o->min_width) {
            const int use_hybrid = o->hybrid && (o->nmin < len);
            int flat = 1;
            for (int i = 0; i < len; ++i) if (!(fabs(x[lo + i] - x[lo]) < 1e-12)) { flat = 0; break; }
            if (!flat) {
                const double* ws = w + lo;
                double wsum = 0.0, wxsum = 0.0;
                for (int i = 0; i < len; ++i) { rw[i] = sqrt(ws[i]); wsum += ws[i]; wxsum += ws[i] * x[lo + i]; }
                const double avg = wxsum / wsum, scale = sqrt(wsum);
                double wxx = 0.0, run = 0.0;
                for (int i = 0; i < len; ++i) {
                    cur[i] = x[lo + i] - avg;
                    wxx += ws[i] * cur[i] * cur[i];
                    run += ws[i];
                    cw[i] = run / scale;
                }
                orc_rng_set_task(rng, seed, unit_id, (uint32_t)lo, (uint32_t)hi);
                z = orc_wfndcpt(cur, len, wxx, ws, rw, cw, o->nperm, o->alpha, use_hybrid, o->min_width, o->kmax, 100, o->tol, rng);
                called = 1;
            }
        }
        if (log && nlog < log_cap) {
            orc_split_rec* e = &log[nlog];
            e->lo = lo; e->hi = hi; e->ostat = z.ostat; e->iseg0 = z.iseg[0]; e->iseg1 = z.iseg[1];
            e->ncpt = z.ncpt; e->icpt0 = z.icpt[0]; e->icpt1 = z.icpt[1];
            e->perms_run = z.perms_run; e->nrej = z.nrej; e->exit_code = z.exit_code; e->called = called;
            e->edge_p0 = called ? z.edge_p[0] : -1.0; e->edge_p1 = called ? z.edge_p[1] : -1.0;
        }
        ++nlog;
        if (z.ncpt > 0) {  /* children [lo,c1) [c1,c2) [c2,hi): one equal to [lo,hi) would be tested again, forever */
            const int c1 = lo + z.icpt[0] + 1, c2 = (z.ncpt == 2) ? lo + z.icpt[1] + 1 : hi;
            if (c1 == hi || (c1 == lo && c2 == hi) || c2 == lo) { self_split = 1; break; }
        }
        if (nends + 2 > ends_cap) { ends_cap *= 2; ends = (int*)realloc(ends, sizeof(int) * (size_t)ends_cap); }
        if (z.ncpt == 0) {
            if (ndone == done_cap) { done_cap *= 2; done = (int*)realloc(done, sizeof(int) * (size_t)done_cap); }
            done[ndone++] = ends[k];
            --nends;
        } else if (z.ncpt == 1) {
            ends[k + 1] = ends[k];
            ends[k] = lo + z.icpt[0] + 1;
            nends += 1;
        } else {
            ends[k + 2] = ends[k];
            ends[k] = lo + z.icpt[0] + 1;
            ends[k + 1] = lo + z.icpt[1] + 1;
            nends += 2;
        }
    }
    if (log_n) *log_n = nlog;
    int ret;
    if (unsupported) ret = ORC_W_UNSUPPORTED;
    else if (self_split) ret = ORC_W_SELF_SPLIT;
    else {
        int nseg = ndone;
        int* lseg = (int*)malloc(sizeof(int) * (size_t)(nseg > 0 ? nseg + 2 : 2));
        int prev = 0;
        for (int s = 0; s < nseg; ++s) { const int e = done[ndone - 1 - s]; lseg[s] = e - prev; prev = e; }
        if (o->undo_prune && nseg > 1) nseg = prune_lengths(x, n, lseg, nseg, o->undo_prune_cutoff); /* :1089, unweighted */
        if (nseg > cap) ret = -nseg - 16;
        else {
            int ll = 0;
            for (int s = 0; s < nseg; ++s) {
                double sw = 0.0, swx = 0.0;
                for (int i = ll; i < ll + lseg[s]; ++i) { sw += w[i]; swx += w[i] * x[i]; }
                lengths[s] = lseg[s];
                means[s] = swx / sw;
                ll += lseg[s];
            }
            ret = nseg;
        }
        free(lseg);
    }
    free(ends); free(done); free(cur); free(rw); free(cw);
    return ret;
}

/* cohort form: every unit through orc_segment_weighted; rng handling as orc_segment_units.
 * Returns total segments, -1 if cap too small, -3 unsupported (weighted hybrid), -4 self split. */
int64_t orc_segment_weighted_units(const double* values, const double* weights, const int64_t* unit_off,
                                   const uint64_t* unit_ids, int n_units, const orc_cohort_opts* o, int64_t cap,
                                   int* seg_count, int* lengths, double* means, uint64_t* draws_out) {
    return orc_segment_weighted_units_log(values, weights, unit_off, unit_ids, n_units, o, cap, seg_count, lengths, means,
                                          draws_out, NULL, 0, NULL, NULL);
}

int64_t orc_segment_weighted_units_log(const double* values, const double* weights, const int64_t* unit_off,
                                       const uint64_t* unit_ids, int n_units, const orc_cohort_opts* o, int64_t cap,
                                       int* seg_count, int* lengths, double* means, uint64_t* draws_out,
                                       orc_split_rec* log, int64_t log_cap, int64_t* log_n, int* log_unit) {
    orc_rng rng;
    if (o->rng_kind == 0) orc_rng_seed_mt(&rng, o->seed); else orc_rng_seed_philox(&rng, o->seed);
    int64_t total = 0, nlog = 0;
    if (log_n) *log_n = 0;
    for (int u = 0; u < n_units; ++u) {
        const int64_t lo = unit_off[u], hi = unit_off[u + 1];
        seg_count[u] = 0;
        if (draws_out) draws_out[u] = 0;
        if (hi <= lo) continue;
        const int n = (int)(hi - lo);
        if (o->rng_kind == 0 && !o->chain) orc_rng_seed_mt(&rng, o->seed);
        const uint64_t d0 = rng.draws;
        const int64_t room = cap - total;
        int this_log = 0;
        const int k = orc_segment_weighted_log(values + lo, weights + lo, n, &o->seg, &rng, o->seed,
                                               unit_ids ? unit_ids[u] : (uint64_t)u,
                                               room > 2147483647 ? 2147483647 : (int)room, lengths + total, means + total,
                                               log ? log + nlog : NULL,
                                               (int)((log_cap - nlog) > 2147483647 ? 2147483647 : (log_cap - nlog)), &this_log);
        if (log_unit) for (int i = 0; i < this_log && nlog + i < log_cap; ++i) log_unit[nlog + i] = u;
        nlog += this_log;
        if (log_n) *log_n = nlog;
        if (k == ORC_W_UNSUPPORTED) return -3;
        if (k == ORC_W_SELF_SPLIT) return -4;
        if (k < 0) return -1;
        seg_count[u] = k;
        total += k;
        if (draws_out) draws_out[u] = rng.draws - d0;
    }
    return total;
}
