// binary.cuh -- binary data (ibin = true): cbs::tmaxo / cbs::tmaxp (CBS.cpp:68-227, the ibin branches), the scan of the
// segmentation worklist for cbs::segment / cbs::fndcpt with ibin = true, cbs::btmax (:363-376) and cbs::btailp (:341-361).
//
// `cna segment` always passes ibin = false (src/cna_segment.hpp:141); binary segmentation is reached through the library
// surface (cbs_gpu_segment[_batch], cbs_gpu_fndcpt with params.ibin = 1).  With the continuity correction the statistic of an
// arc length is fac * (max_i |S_{i+L} - S_i| - 0.5)^2: it is not monotone in |d|, the reference's block-pair bound is not an
// upper bound any more, and which pairs it skips depends on the ORDER in which it visits them.  An exact maximum therefore
// walks the pairs in that order.  k_scan_bin (low-level tmaxo / tmaxp) does it with one warp per vector: lane 0 runs the
// sequential control flow (prefix sums, pair list, libstdc++'s introsort order of the corner statistics, descending visit
// with the running maximum), all lanes share the innermost loop over the start positions of an arc length.  k_scan_binary
// (worklist) spreads each pair over a CTA and decides most permutations without the order (DESIGN 4c).
#pragma once
#include <cuda_runtime.h>

#include "cbs_core.h"
#include "kernels.cuh"

namespace cbsg {

// ---- std::sort of an array by key, ties ordered as libstdc++'s introsort orders them (median-of-3 quicksort to depth
// 2*log2 n, heap sort fallback, final insertion sort, threshold 16): the reference sorts candidate block pairs with it
// (CBS.cpp:63-66,160) and visits equal keys in whatever order it leaves them. ----------------------------------------------
template <class E, class Less>
struct Introsort {
    E* a;       // the elements being sorted, a[0..len)
    Less less;  // strict order of two elements
    __device__ void sift(long hole, long len, E value) {
        const long top = hole;
        long child = hole;
        while (child < (len - 1) / 2) {
            child = 2 * (child + 1);
            if (less(a[child], a[child - 1])) --child;
            a[hole] = a[child];
            hole = child;
        }
        if ((len & 1) == 0 && child == (len - 2) / 2) {
            child = 2 * (child + 1);
            a[hole] = a[child - 1];
            hole = child - 1;
        }
        long parent = (hole - 1) / 2;
        while (hole > top && less(a[parent], value)) {
            a[hole] = a[parent];
            hole = parent;
            parent = (hole - 1) / 2;
        }
        a[hole] = value;
    }
    __device__ void heap_range(long lo, long hi) {  // heap sort of a[lo..hi)
        E* base = a + lo;
        E* keep = a;
        a = base;
        const long len = hi - lo;
        for (long parent = (len - 2) / 2; len >= 2; --parent) {
            sift(parent, len, a[parent]);
            if (parent == 0) break;
        }
        for (long last = len - 1; last >= 1; --last) {
            const E value = a[last];
            a[last] = a[0];
            sift(0, last, value);
        }
        a = keep;
    }
    __device__ void slide_back(long pos) {  // a[pos] moves left past larger elements (a smaller one is known to stop it)
        const E val = a[pos];
        long nxt = pos - 1;
        while (less(val, a[nxt])) { a[pos] = a[nxt]; pos = nxt; --nxt; }
        a[pos] = val;
    }
    __device__ void insertion(long lo, long hi) {
        for (long i = lo + 1; i < hi; ++i) {
            if (less(a[i], a[lo])) {
                const E val = a[i];
                for (long k = i; k > lo; --k) a[k] = a[k - 1];
                a[lo] = val;
            } else slide_back(i);
        }
    }
    __device__ void run(long len) {
        if (len <= 0) return;
        long lg = 0;
        for (long m = len; m > 1; m >>= 1) ++lg;
        // the quicksort phase, with an explicit stack of (lo, hi, depth): the right part is sorted first, as the recursion does
        long st_lo[64], st_hi[64], st_d[64];
        int sp = 0;
        st_lo[0] = 0; st_hi[0] = len; st_d[0] = 2 * lg; sp = 1;
        while (sp > 0) {
            --sp;
            long lo = st_lo[sp], hi = st_hi[sp], depth = st_d[sp];
            while (hi - lo > 16) {
                if (depth == 0) { heap_range(lo, hi); break; }
                --depth;
                const long mid = lo + (hi - lo) / 2;
                {   // median of a[lo+1], a[mid], a[hi-1] goes to a[lo]
                    const long x = lo + 1, y = mid, z = hi - 1;
                    long pick;
                    if (less(a[x], a[y])) pick = less(a[y], a[z]) ? y : (less(a[x], a[z]) ? z : x);
                    else pick = less(a[x], a[z]) ? x : (less(a[y], a[z]) ? z : y);
                    const E t = a[lo]; a[lo] = a[pick]; a[pick] = t;
                }
                long f = lo + 1, l = hi;
                for (;;) {
                    while (less(a[f], a[lo])) ++f;
                    --l;
                    while (less(a[lo], a[l])) --l;
                    if (!(f < l)) break;
                    const E t = a[f]; a[f] = a[l]; a[l] = t;
                    ++f;
                }
                // recursion on [f, hi) happens BEFORE the loop continues with [lo, f): the order of the two does not change the
                // result (disjoint ranges), so the right part is simply stacked
                if (sp < 64) { st_lo[sp] = f; st_hi[sp] = hi; st_d[sp] = depth; ++sp; }
                hi = f;
            }
        }
        if (len > 16) {
            insertion(0, 16);
            for (long i = 16; i < len; ++i) slide_back(i);
        } else insertion(0, len);
    }
};

// indices ordered by key[index] (k_scan_bin)
struct KeyOfIdx {
    const double* key;
    __device__ bool operator()(int x, int y) const { return key[x] < key[y]; }
};
typedef Introsort<int, KeyOfIdx> IdxSort;
// (key, index) records ordered by key: the same comparisons and moves as IdxSort, but the key travels with the index, so the
// partitions read memory sequentially instead of one dependent random load per comparison (k_scan_binary)
struct KeyIdx { double key; int idx; int pad; };
struct KeyIdxLess {
    __device__ bool operator()(const KeyIdx& x, const KeyIdx& y) const { return x.key < y.key; }
};

// scratch of one vector, carved out of one allocation: doubles first, then ints
__host__ __device__ inline long long bin_scratch_doubles(int n) {
    const long long nb = block_count(n), nb2 = nb * (nb + 1) / 2;
    const long long d = ((long long)n + 1) + 2 * (nb + 1) + 2 * (nb2 + 1);
    const long long i = 3 * (nb + 1) + 4 * (nb2 + 1);
    return d + (i + 1) / 2 + 8;
}

// warp-wide version of `sxmx < absx` with the SMALLEST index winning among equal maxima (CBS.cpp:186-190)
__device__ __forceinline__ void warp_first_max(double& v, int& idx) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, v, o);
        const int oi = __shfl_xor_sync(0xffffffffu, idx, o);
        if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
    }
}

// cbs::tmaxo_impl (CBS.cpp:68-227) as written, for `count` vectors of n values laid end to end; one warp per vector
__global__ void __launch_bounds__(32) k_scan_bin(const double* __restrict__ xall, int n, int count, double tss_in, int al0, int ibin,
                                                 double* scratch_all, double* stat_out, int* left_out, int* right_out) {
    const int lane = threadIdx.x;
    for (int v = blockIdx.x; v < count; v += gridDim.x) {
        const double* x = xall + (long long)v * n;
        const double rn = (double)n;
        const int nb = block_count(n);
        const int nb2 = nb * (nb + 1) / 2;
        double* sx = scratch_all + (long long)v * bin_scratch_doubles(n);
        double* bpsmax = sx + n + 1;
        double* bpsmin = bpsmax + nb + 1;
        double* bssbij = bpsmin + nb + 1;
        double* bssijmax = bssbij + nb2 + 1;
        int* bb = (int*)(bssijmax + nb2 + 1);
        int* ibmin = bb + nb + 1;
        int* ibmax = ibmin + nb + 1;
        int* bloci = ibmax + nb + 1;
        int* blocj = bloci + nb2 + 1;
        int* loc = blocj + nb2 + 1;
        int* alen = loc + nb2 + 1;
        double tss = tss_in;
        // :77 block ends, :79-97 prefix sums and block extrema (sequential: lane 0)
        double psmin0 = 0.0, psmax0 = 0.0;
        int ipsmin0 = n, ipsmax0 = n;
        if (lane == 0) {
            bb[0] = 0;
            for (int i = 1; i <= nb; ++i) bb[i] = block_end(n, nb, i);
            sx[0] = 0.0;
            int ilo = 1;
            double psum = 0.0;
            for (int j = 1; j <= nb; ++j) {
                sx[ilo] = psum + x[ilo - 1];
                double psmin = sx[ilo], psmax = sx[ilo];
                int ipsmin = ilo, ipsmax = ilo;
                for (int i = ilo + 1; i <= bb[j]; ++i) {
                    sx[i] = sx[i - 1] + x[i - 1];
                    if (sx[i] < psmin) { psmin = sx[i]; ipsmin = i; }
                    if (sx[i] > psmax) { psmax = sx[i]; ipsmax = i; }
                }
                ibmin[j] = ipsmin; ibmax[j] = ipsmax;
                bpsmin[j] = psmin; bpsmax[j] = psmax;
                if (psmin < psmin0) { psmin0 = psmin; ipsmin0 = ipsmin; }
                if (psmax > psmax0) { psmax0 = psmax; ipsmax0 = ipsmax; }
                psum = sx[bb[j]];
                ilo = bb[j] + 1;
            }
        }
        __syncwarp();
        psmin0 = __shfl_sync(0xffffffffu, psmin0, 0); psmax0 = __shfl_sync(0xffffffffu, psmax0, 0);
        ipsmin0 = __shfl_sync(0xffffffffu, ipsmin0, 0); ipsmax0 = __shfl_sync(0xffffffffu, ipsmax0, 0);
        const double psdiff = psmax0 - psmin0;
        double bssmax = 0.0;
        int tmaxi = min(ipsmax0, ipsmin0), tmaxj = max(ipsmax0, ipsmin0);
        if (psdiff <= 0.0) {  // :101-110
            if (tss <= 0.0001) tss = 1.0;
            bssmax = ibin ? 0.0 / (tss / rn) : 0.0 / ((tss - 0.0) / (rn - 2.0));
            if (lane == 0) { stat_out[v] = bssmax; left_out[v] = tmaxi; right_out[v] = tmaxj; }
            continue;
        }
        {
            const double rj = (double)abs(ipsmax0 - ipsmin0);
            const double rnjov1 = rn / (rj * (rn - rj));
            bssmax = ibin ? rnjov1 * ((psdiff - 0.5) * (psdiff - 0.5)) : rnjov1 * psdiff * psdiff;  // pow(., 2.0) is the exact square
        }
        const double rnov2 = rn / 2.0;
        const int nal0 = n - al0;
        // :119-158 candidate pairs in (i, j) order; the list keeps that order (ballot compaction, 32 pairs at a time)
        int l = 0;
        for (int i = 1; i <= nb; ++i) {
            for (int j0 = i; j0 <= nb; j0 += 32) {
                const int j = j0 + lane;
                bool take = false;
                double e_lim = 0.0, e_bij = 0.0;
                int e_len = 0;
                if (j <= nb) {
                    const int ilo1 = (i == 1) ? 1 : bb[i - 1] + 1, ihi = bb[i];
                    const int jlo = (j == 1) ? 1 : bb[j - 1] + 1, jhi = bb[j];
                    int alenhi = jhi - ilo1;
                    if (alenhi > nal0) alenhi = nal0;
                    int alenlo = (i == j) ? 1 : (jlo - ihi);
                    if (alenlo < al0) alenlo = al0;
                    const double sij1 = fabs(bpsmax[j] - bpsmin[i]);
                    const double sij2 = fabs(bpsmax[i] - bpsmin[j]);
                    const double sijmx0 = fmax(sij1, sij2);
                    const double rjlo = (double)alenlo, rjhi = (double)alenhi;
                    const double rnjov1 = rn / fmin(rjlo * (rn - rjlo), rjhi * (rn - rjhi));
                    const double bsslim = ibin ? rnjov1 * ((sijmx0 - 0.5) * (sijmx0 - 0.5)) : rnjov1 * sijmx0 * sijmx0;
                    if (bssmax <= bsslim) {
                        take = true;
                        e_lim = bsslim;
                        const double sij = (sij1 > sij2) ? sij1 : sij2;
                        e_len = (sij1 > sij2) ? abs(ibmax[j] - ibmin[i]) : abs(ibmin[j] - ibmax[i]);
                        const double rr = (double)e_len;
                        const double fac = rn / (rr * (rn - rr));
                        e_bij = ibin ? fac * ((sij - 0.5) * (sij - 0.5)) : fac * sij * sij;
                    }
                }
                const unsigned mask = __ballot_sync(0xffffffffu, take);
                if (take) {
                    const int pos = l + 1 + __popc(mask & ((1u << lane) - 1u));
                    loc[pos] = pos; bloci[pos] = i; blocj[pos] = j; bssijmax[pos] = e_lim; alen[pos] = e_len; bssbij[pos] = e_bij;
                }
                l += __popc(mask);
            }
        }
        const int nb1 = l;
        __syncwarp();
        if (lane == 0) { IdxSort srt{loc + 1, KeyOfIdx{bssbij}}; srt.run(nb1); }  // :160, ascending by corner statistic
        __syncwarp();
        // :162-216 descending visit
        for (int ll = nb1; ll >= 1; --ll) {
            const int k = loc[ll];
            const double bsslim = bssijmax[k];
            if (bssmax > bsslim) continue;
            const int bi = bloci[k], bj = blocj[k];
            int alenmax = alen[k];
            const int ilo1 = (bi == 1) ? 1 : bb[bi - 1] + 1, ihi = bb[bi];
            const int jlo = (bj == 1) ? 1 : bb[bj - 1] + 1, jhi = bb[bj];
            int alenhi = jhi - ilo1;
            if (alenhi > nal0) alenhi = nal0;
            int alenlo = (bi == bj) ? 1 : (jlo - ihi);
            if (alenlo < al0) alenlo = al0;
            const double rjlo = (double)alenlo, rjhi = (double)alenhi;
            if (alenmax > n - alenmax) alenmax = n - alenmax;
            for (int band = 0; band < 2; ++band) {
                int from, to, step;
                if (band == 0) { if (!((rjlo <= rnov2) && (alenlo <= alenmax))) continue; from = alenlo; to = alenmax; step = 1; }
                else {
                    const int amax2 = n - alenmax;
                    if (!((rjhi >= rnov2) && (alenhi >= amax2))) continue;
                    from = alenhi; to = amax2; step = -1;
                }
                for (int i2j = from; step > 0 ? i2j <= to : i2j >= to; i2j += step) {
                    const int ixlo = max(0, jlo - ilo1 - i2j), ixhi = max(0, ihi + i2j - jhi);
                    double sxmx = 0.0;
                    int sxmxi = ilo1;
                    for (int i = ilo1 + ixlo + lane; i <= ihi - ixhi; i += 32) {
                        const double absx = fabs(sx[i + i2j] - sx[i]);
                        if (sxmx < absx) { sxmx = absx; sxmxi = i; }
                    }
                    warp_first_max(sxmx, sxmxi);
                    const double rr = (double)i2j;
                    const double fac = rn / (rr * (rn - rr));
                    const double bijbss = ibin ? fac * ((sxmx - 0.5) * (sxmx - 0.5)) : fac * sxmx * sxmx;
                    if (bijbss > bssmax) { bssmax = bijbss; tmaxi = sxmxi; tmaxj = sxmxi + i2j; }
                }
            }
        }
        if (ibin) {  // :218-224
            if (tss <= 0.0001) tss = 1.0;
            bssmax /= (tss / rn);
        } else {
            if (tss <= bssmax + 0.0001) tss = bssmax + 1.0;
            bssmax /= ((tss - bssmax) / (rn - 2.0));
        }
        if (lane == 0) { stat_out[v] = bssmax; left_out[v] = tmaxi; right_out[v] = tmaxj; }
    }
}

// ------------------------------------------------------------------------------------
// k_scan_binary -- the worklist's scan for binary data (ibin = true), one CTA per row (observed segment or permutation).
//
// Observed rows (exact maximum and location) and the permutations of tasks with a weak reject level (bin_weak) walk the
// block pairs in the reference's order (CBS.cpp:119-216): the candidate list in (i, j) order, libstdc++'s introsort of the
// corner statistics, a descending visit that skips pairs whose bound is below the running maximum.  Inside one pair the
// result only depends on the running maximum at its start, so the warps take its arc lengths in parallel and the pair is
// reduced in visiting order (largest statistic, first length among equals; strict > against the running maximum).
// Permutations whose reject level Lstar lies above fac_max/4 take the decision scan instead (DESIGN 4c): the reference
// rejects iff the seed arc or some arc of a pair whose bound reaches Lstar, inside that pair's bands, has a statistic
// >= Lstar, whatever the visiting order.  The warps take such pairs in any order, per length only the arcs with
// |S_j - S_i| >= 0.5 + sqrt(Lstar)*g[L] are re-evaluated exactly, and the first hit settles the row.
// ------------------------------------------------------------------------------------
struct BinSmem {
    double best;          // running maximum (ordered walk)
    int bi, bj;           // its arc, 1-based prefix indices
    int decided;          // permutation rows: the row rejects
    int next_pair;        // decision scan: next block pair to claim
    int n_list;           // ordered walk: entries of the candidate list
    double g_min, g_max;
    int g_imin, g_imax;
    double w_stat[32];    // per warp: best length of the pair being walked
    int w_v[32], w_i[32], w_cnt[32];
};

__device__ __forceinline__ void bin_pair_lengths(const int* bb, int n, int al0, int bi, int bj, int& ilo, int& ihi, int& jlo,
                                                 int& jhi, int& lenlo, int& lenhi) {
    ilo = bb[bi - 1] + 1; ihi = bb[bi]; jlo = bb[bj - 1] + 1; jhi = bb[bj];  // (bb[0] = 0: block 1 starts at 1)
    lenhi = min(jhi - ilo, n - al0);
    lenlo = (bi == bj) ? 1 : (jlo - ihi);
    if (lenlo < al0) lenlo = al0;
}

// bound and corner arc of a block pair (CBS.cpp:126-156, ibin branches); blocks are 1-based, the smem arrays 0-based
__device__ __forceinline__ void bin_pair_bound(const double* bmin, const double* bmax, const int* amin, const int* amax, double rn,
                                               int bi, int bj, int lenlo, int lenhi, double& bsslim, double& corner, int& clen,
                                               double& smax) {
    const double sij1 = fabs(bmax[bj - 1] - bmin[bi - 1]);
    const double sij2 = fabs(bmax[bi - 1] - bmin[bj - 1]);
    smax = fmax(sij1, sij2);
    const double rjlo = (double)lenlo, rjhi = (double)lenhi;
    const double rnjov1 = rn / fmin(rjlo * (rn - rjlo), rjhi * (rn - rjhi));
    bsslim = rnjov1 * ((smax - 0.5) * (smax - 0.5));
    const double sij = (sij1 > sij2) ? sij1 : sij2;
    clen = (sij1 > sij2) ? abs(amax[bj - 1] - amin[bi - 1]) : abs(amin[bj - 1] - amax[bi - 1]);
    const double rr = (double)clen;
    corner = rn / (rr * (rn - rr)) * ((sij - 0.5) * (sij - 0.5));
}

// the two arc-length bands of a listed pair (CBS.cpp:179-180, 198-199): [lo0, hi0] visited ascending, then [lo1, hi1]
// descending; a band is empty when its count is 0
__device__ __forceinline__ void bin_bands(int n, int clen, int lenlo, int lenhi, int& cnt0, int& cnt1, int& hi1) {
    int lenmax = clen;
    if (lenmax > n - lenmax) lenmax = n - lenmax;
    const double rnov2 = (double)n / 2.0;
    cnt0 = ((double)lenlo <= rnov2 && lenlo <= lenmax) ? lenmax - lenlo + 1 : 0;
    const int amax2 = n - lenmax;
    cnt1 = ((double)lenhi >= rnov2 && lenhi >= amax2) ? lenhi - amax2 + 1 : 0;
    hi1 = lenhi;
}

__global__ void __launch_bounds__(256) k_scan_binary(Dev* D, int nb_max) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    if (D->done) return;
    BinSmem* s = (BinSmem*)smem_raw;
    double* s_bmin = (double*)(smem_raw + ((sizeof(BinSmem) + 15) & ~(size_t)15));
    double* s_bmax = s_bmin + nb_max;
    int* s_amin = (int*)(s_bmax + nb_max);
    int* s_amax = s_amin + nb_max;
    int* s_bb = s_amax + nb_max;
    __shared__ int s_g;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int total = D->item_prefix[D->n_items];
    const double dinf = __longlong_as_double(0x7ff0000000000000LL);
    for (;;) {
        __syncthreads();
        if (tid == 0) s_g = (int)atomicAdd(&D->ctr[1], 1u);
        __syncthreads();
        const int gidx = s_g;
        if (gidx >= total) break;
        const int k = find_item(D->item_prefix, D->n_items, gidx);
        const PermItem it = D->items[k];
        Task& t = D->tasks[it.task];
        if (it.obs && t.alleq) continue;
        const int p = gidx - D->item_prefix[k];
        const int n = t.n, nb = t.nb, al0 = D->prm.min_width;
        const double rn = (double)n;
        const long long base = D->unit_off[t.unit] + t.lo;
        const double* sx = D->arena + t.off_sx + (long long)p * Sched::sx_stride(n);
        const int* bbg = D->bbtab + base;
        for (int b = tid; b <= nb; b += blockDim.x) s_bb[b] = bbg[b];
        __syncthreads();
        if (it.obs) {  // k_prep wrote the prefix sums; the per-block extrema with their first occurrence (CBS.cpp:88-94)
            for (int b = warp; b < nb; b += nwarps) {
                const int first = s_bb[b] + 1, last = s_bb[b + 1];
                double lo = dinf, hi = -dinf;
                int ilo = 0x7fffffff, ihi = 0x7fffffff;
                for (int i = first + lane; i <= last; i += 32) {
                    const double v = sx[i];
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
        } else {  // written next to the row by k_chain
            BlockStats bs(D->arena + t.off_bs + (long long)p * Sched::bs_stride(nb), nb);
            for (int b = tid; b < nb; b += blockDim.x) {
                s_bmin[b] = bs.bmin()[b]; s_bmax[b] = bs.bmax()[b]; s_amin[b] = bs.amin()[b]; s_amax[b] = bs.amax()[b];
            }
        }
        __syncthreads();
        // global extrema: the first block attaining them, and only below / above 0.0 (CBS.cpp:80-81, 93-94)
        if (warp == 0) {
            double lo = dinf, hi = -dinf;
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
                s->g_min = below ? lo : 0.0; s->g_imin = below ? s_amin[blo] : n;
                s->g_max = above ? hi : 0.0; s->g_imax = above ? s_amax[bhi] : n;
                s->decided = 0; s->n_list = 0; s->next_pair = 0;
            }
        }
        __syncthreads();
        const double psdiff = s->g_max - s->g_min;
        const int gimin = s->g_imin, gimax = s->g_imax;
        const bool exact = it.obs != 0;
        const double lstar = exact ? dinf : bin_reject_level(t.ostat, t.tss, n);
        double seed = 0.0;
        if (psdiff > 0.0) {  // CBS.cpp:113-117
            const double rj = (double)abs(gimax - gimin);
            seed = rn / (rj * (rn - rj)) * ((psdiff - 0.5) * (psdiff - 0.5));
        }
        if (tid == 0) {
            s->best = seed; s->bi = min(gimax, gimin); s->bj = max(gimax, gimin);
            if (!exact && seed >= lstar) s->decided = 1;
        }
        __syncthreads();
        const int npairs = nb * (nb + 1) / 2;
        if (psdiff > 0.0 && !s->decided) {
            if (exact || bin_weak(lstar, n, al0)) {
                // ---- the reference's order.  Scratch: (corner, index) records, then bounds, pairs and corner lengths (1-based)
                double* scr = D->arena + t.off_bin + (exact ? 0 : (long long)p * Sched::bin_stride(nb));
                const long long e = (long long)npairs + 1;
                KeyIdx* rec = (KeyIdx*)scr;
                double* lim = scr + 2 * e;
                int* pcode = (int*)(lim + e);
                int* plen = pcode + e;
                // :119-158 candidate pairs in (i, j) order: CTA-wide stable compaction, blockDim pairs at a time
                for (int q0 = 0; q0 < npairs; q0 += blockDim.x) {
                    const int q = q0 + tid;
                    bool take = false;
                    double e_lim = 0.0, e_key = 0.0;
                    int e_len = 0, bi = 1, bj = 1;
                    if (q < npairs) {
                        pair_from_index(q, nb, bi, bj);
                        int ilo, ihi, jlo, jhi, lenlo, lenhi;
                        bin_pair_lengths(s_bb, n, al0, bi, bj, ilo, ihi, jlo, jhi, lenlo, lenhi);
                        double smax;
                        bin_pair_bound(s_bmin, s_bmax, s_amin, s_amax, rn, bi, bj, lenlo, lenhi, e_lim, e_key, e_len, smax);
                        take = seed <= e_lim;
                    }
                    const unsigned mask = __ballot_sync(FULL, take);
                    if (lane == 0) s->w_cnt[warp] = __popc(mask);
                    __syncthreads();
                    int before = 0, all = 0;
                    for (int w = 0; w < nwarps; ++w) { const int c = s->w_cnt[w]; if (w < warp) before += c; all += c; }
                    if (take) {
                        const int pos = s->n_list + 1 + before + __popc(mask & ((1u << lane) - 1u));
                        rec[pos].key = e_key; rec[pos].idx = pos; lim[pos] = e_lim; pcode[pos] = (bi << 16) | bj; plen[pos] = e_len;
                    }
                    __syncthreads();
                    if (tid == 0) s->n_list += all;
                }
                __syncthreads();
                const int nb1 = s->n_list;
                if (tid == 0) { Introsort<KeyIdx, KeyIdxLess> srt{rec + 1, KeyIdxLess{}}; srt.run(nb1); }  // :160
                __syncthreads();
                // :162-216 descending visit
                for (int ll = nb1; ll >= 1; --ll) {
                    const int kk = rec[ll].idx;
                    if (s->best > lim[kk]) continue;  // uniform: s->best only changes between the barriers below
                    const int bi = pcode[kk] >> 16, bj = pcode[kk] & 0xffff;
                    int ilo, ihi, jlo, jhi, lenlo, lenhi, cnt0, cnt1, hi1;
                    bin_pair_lengths(s_bb, n, al0, bi, bj, ilo, ihi, jlo, jhi, lenlo, lenhi);
                    bin_bands(n, plen[kk], lenlo, lenhi, cnt0, cnt1, hi1);
                    double wbest = -1.0;
                    int wv = 0x7fffffff, wi = 0;
                    for (int v = warp; v < cnt0 + cnt1; v += nwarps) {  // visiting order v: band 0 ascending, then band 1 descending
                        const int L = v < cnt0 ? lenlo + v : hi1 - (v - cnt0);
                        const int ixlo = max(0, jlo - ilo - L), ixhi = max(0, ihi + L - jhi);
                        double sxmx = 0.0;
                        int sxmxi = ilo;
                        for (int i = ilo + ixlo + lane; i <= ihi - ixhi; i += 32) {
                            const double absx = fabs(sx[i + L] - sx[i]);
                            if (sxmx < absx) { sxmx = absx; sxmxi = i; }
                        }
                        warp_first_max(sxmx, sxmxi);
                        const double rr = (double)L;
                        const double stat = rn / (rr * (rn - rr)) * ((sxmx - 0.5) * (sxmx - 0.5));
                        if (stat > wbest) { wbest = stat; wv = v; wi = sxmxi; }
                    }
                    if (lane == 0) { s->w_stat[warp] = wbest; s->w_v[warp] = wv; s->w_i[warp] = wi; }
                    __syncthreads();
                    if (tid == 0) {
                        double b = -1.0;
                        int bv = 0x7fffffff, bi2 = 0;
                        for (int w = 0; w < nwarps; ++w)
                            if (s->w_stat[w] > b || (s->w_stat[w] == b && s->w_v[w] < bv)) { b = s->w_stat[w]; bv = s->w_v[w]; bi2 = s->w_i[w]; }
                        if (bv != 0x7fffffff && b > s->best) {
                            const int L = bv < cnt0 ? lenlo + bv : hi1 - (bv - cnt0);
                            s->best = b; s->bi = bi2; s->bj = bi2 + L;
                            if (b >= lstar) s->decided = 1;  // permutation: the running maximum only grows
                        }
                    }
                    __syncthreads();
                    if (s->decided) break;
                }
            } else {
                // ---- decision scan (Lstar > fac_max/4): pairs whose bound reaches Lstar, in any order
                const double sql = sqrt(lstar);
                for (;;) {
                    int q0 = 0;
                    if (lane == 0) q0 = atomicAdd(&s->next_pair, 32);
                    q0 = __shfl_sync(FULL, q0, 0);
                    if (q0 >= npairs || *((volatile int*)&s->decided)) break;
                    const int q = q0 + lane;
                    bool alive = false;
                    int bi = 1, bj = 1, clen = 0;
                    double smax = 0.0;
                    if (q < npairs) {
                        pair_from_index(q, nb, bi, bj);
                        int ilo, ihi, jlo, jhi, lenlo, lenhi;
                        bin_pair_lengths(s_bb, n, al0, bi, bj, ilo, ihi, jlo, jhi, lenlo, lenhi);
                        double bsslim, corner;
                        bin_pair_bound(s_bmin, s_bmax, s_amin, s_amax, rn, bi, bj, lenlo, lenhi, bsslim, corner, clen, smax);
                        alive = bsslim >= lstar;
                    }
                    unsigned mask = __ballot_sync(FULL, alive);
                    while (mask) {
                        const int src = __ffs(mask) - 1;
                        mask &= mask - 1;
                        const int pbi = __shfl_sync(FULL, bi, src), pbj = __shfl_sync(FULL, bj, src), pclen = __shfl_sync(FULL, clen, src);
                        const double psmax = shfl_d(smax, src);
                        int ilo, ihi, jlo, jhi, lenlo, lenhi, cnt0, cnt1, hi1;
                        bin_pair_lengths(s_bb, n, al0, pbi, pbj, ilo, ihi, jlo, jhi, lenlo, lenhi);
                        bin_bands(n, pclen, lenlo, lenhi, cnt0, cnt1, hi1);
                        bool hit = false;
                        for (int v = 0; v < cnt0 + cnt1 && !hit; ++v) {
                            if ((v & 15) == 0 && *((volatile int*)&s->decided)) break;
                            const int L = v < cnt0 ? lenlo + v : hi1 - (v - cnt0);
                            const double rr = (double)L;
                            // an arc reaches Lstar only if |S_j - S_i| >= 0.5 + sqrt(Lstar)*g[L]; the threshold is lowered by
                            // 1e-12 relative so that rounding cannot drop an arc, and every arc above it is evaluated exactly
                            const double thr = 0.5 + sql * sqrt(rr * (rn - rr) / rn) * (1.0 - 1e-12);
                            if (psmax < thr) continue;
                            const double fac = rn / (rr * (rn - rr));
                            const int ixlo = max(0, jlo - ilo - L), ixhi = max(0, ihi + L - jhi);
                            bool h = false;
                            for (int i = ilo + ixlo + lane; i <= ihi - ixhi; i += 32) {
                                const double d = fabs(sx[i + L] - sx[i]);
                                if (d >= thr && fac * ((d - 0.5) * (d - 0.5)) >= lstar) h = true;
                            }
                            hit = __any_sync(FULL, h);
                        }
                        if (hit) {
                            if (lane == 0) s->decided = 1;
                            break;
                        }
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            if (exact) {  // CBS.cpp:101-110, 218-224
                double tss = t.tss;
                if (tss <= 0.0001) tss = 1.0;
                const double stat = s->best / (tss / rn);
                t.ostat = stat;
                if (it.obs == 1) { t.tmaxi = s->bi; t.tmaxj = s->bj; }
            } else D->rej[t.off_rej + p] = s->decided;  // CBS.cpp:862-864
        }
    }
}

// cbs::btmax (CBS.cpp:363-376): one dependent chain
__global__ void k_btmax(const double* __restrict__ x, int n, double* out) {
    if (threadIdx.x || blockIdx.x) return;
    double sumxi = x[0], ostat = 0.0, di = 1.0;
    const double dn = (double)n;
    for (int i = 2; i <= n - 2; ++i) {
        di += 1.0;
        sumxi += x[i - 1];
        const double b = dn * (sumxi * sumxi) / (di * (dn - di));
        if (ostat < b) ostat = b;
    }
    *out = sqrt(ostat);
}

}  // namespace cbsg
