// smooth.cuh -- outlier smoothing (DNAcopy smooth.CNA as ported in lib/cbs/smooth.cpp).
//
// Per "group" (one call of cbs::smooth; on the cna segment path one chromosome of one
// sample, cna_segment.hpp:139-140):
//   k_sm_compact  drop non-finite values, keep their indices            (smooth.cpp:135-141)
//   k_sm_diffs    |v[i+1]-v[i]| of the finite subsequence               (smooth.cpp:37-39)
//   (ascending sort of the differences within each group: two radix sorts, by value and then -- stable -- by group;
//    cub::DeviceSegmentedSort for very large calls)
//   k_sm_sd       sum of the n_keep smallest squares in ascending order -> trimmed SD (:36-44,:144-148)
//   k_sm_window   per finite marker: +-k window outlier test, median shrink (smooth.cpp:76-115), k <= SM_MAX_REGION
//   (wider windows: k_sm_run_*, k_sm_wide, k_sm_median below)
// The window kernel is the HBM-streaming part (24 B per marker); the sort only feeds one
// scalar per group but has to be exact because the sum is taken in sorted order.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cbsg {

struct SmoothGroupOut {
    double oSD, sSD;
    int valid;   // thresholds usable (>= 2 finite values, finite non-negative variance)
    int m;       // number of finite values
};

// one CTA per group: stable compaction of finite values
__global__ void __launch_bounds__(256) k_sm_compact(const double* __restrict__ x, const long long* __restrict__ off,
                                                    const int* __restrict__ lab, int n_groups, double* __restrict__ fv,
                                                    int* __restrict__ fidx, int* __restrict__ flab,
                                                    SmoothGroupOut* __restrict__ gout) {
    __shared__ int s_warp[8];
    __shared__ int s_base;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const long long lo = off[g];
        const int n = (int)(off[g + 1] - lo);
        if (threadIdx.x == 0) s_base = 0;
        __syncthreads();
        for (int c0 = 0; c0 < n; c0 += 256) {
            const int i = c0 + threadIdx.x;
            double v = 0.0;
            bool fin = false;
            if (i < n) { v = x[lo + i]; fin = isfinite(v); }
            const unsigned m = __ballot_sync(0xffffffffu, fin);
            const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
            if (lane == 0) s_warp[w] = __popc(m);
            __syncthreads();
            int before = s_base;
            for (int k = 0; k < w; ++k) before += s_warp[k];
            const int pos = before + __popc(m & ((1u << lane) - 1u));
            if (fin) {
                fv[lo + pos] = v;
                fidx[lo + pos] = i;
                if (flab) flab[lo + pos] = lab[lo + i];
            }
            __syncthreads();
            if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < 8; ++k) t += s_warp[k]; s_base += t; }
            __syncthreads();
        }
        if (threadIdx.x == 0) { gout[g].m = s_base; gout[g].valid = 0; gout[g].oSD = 0.0; gout[g].sSD = 0.0; }
        __syncthreads();
    }
}

// |differences| of the finite subsequence; slots beyond m-1 of a group are filled with +inf so
// that a segmented sort over the fixed group extents leaves them at the end
// gid (optional): the group of every slot, the second key of the two-pass radix sort (smooth_device)
__global__ void k_sm_diffs(const double* __restrict__ fv, const long long* __restrict__ off, int n_groups,
                           const SmoothGroupOut* __restrict__ gout, double* __restrict__ d, int* __restrict__ gid) {
    for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
        const long long lo = off[g];
        const int n = (int)(off[g + 1] - lo);
        const int m = gout[g].m;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
            d[lo + i] = (i + 1 < m) ? fabs(fv[lo + i + 1] - fv[lo + i]) : __longlong_as_double(0x7ff0000000000000LL);
            if (gid) gid[lo + i] = g;
        }
    }
}

// one warp per group: ascending-order sum of squares, exactly as the reference accumulates it (lane 0 runs the
// dependent chain over chunks staged in shared memory, chain_sum_sq in kernels.cuh)
__global__ void __launch_bounds__(32) k_sm_sd(const double* __restrict__ dsorted, const long long* __restrict__ off,
                                              int n_groups, double trim, double inflfact, double outlier_scale,
                                              double smooth_scale, SmoothGroupOut* __restrict__ gout) {
    __shared__ __align__(16) double buf[PREP_CHUNK];
    const int lane = threadIdx.x;
    for (int g = blockIdx.x; g < n_groups; g += gridDim.x) {
        const int m = gout[g].m;
        if (m < 2) continue;  // smooth.cpp:142
        double tvar = 0.0;
        const long long keep = llround((1.0 - 2.0 * trim) * (double)(m - 1));  // smooth.cpp:36
        if (keep > 0) {
            double sum = 0.0, ss = 0.0;
            chain_sum_sq(dsorted + off[g], (int)keep, buf, lane, sum, ss);
            tvar = inflfact * (ss / (2.0 * (double)keep));
        }
        if (lane == 0) {
            if (isfinite(tvar) && !(tvar < 0.0)) {  // smooth.cpp:145
                const double sd = sqrt(tvar);
                gout[g].oSD = outlier_scale * sd;
                gout[g].sSD = smooth_scale * sd;
                gout[g].valid = 1;
            }
        }
    }
}

#define SM_MAX_REGION 64  // widest window of k_sm_window (per-thread sort buffer); wider ones take k_sm_wide

// thread per finite marker
__global__ void __launch_bounds__(256) k_sm_window(const double* __restrict__ fv, const int* __restrict__ fidx,
                                                   const int* __restrict__ flab, const long long* __restrict__ off,
                                                   int n_groups, int region, const SmoothGroupOut* __restrict__ gout,
                                                   double* __restrict__ out) {
    for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
        const SmoothGroupOut go = gout[g];
        if (!go.valid) continue;
        const long long lo = off[g];
        const double* v = fv + lo;
        const int m = go.m;
        const double oSD = go.oSD, sSD = go.sSD;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
            // window clipped to the run of equal labels (smooth.cpp:47-61, :84-85)
            int wlo = i, whi = i;
            if (flab) {
                const int* lb = flab + lo;
                const int mine = lb[i];
                for (int s = 1; s <= region && i - s >= 0 && lb[i - s] == mine; ++s) wlo = i - s;
                for (int s = 1; s <= region && i + s < m && lb[i + s] == mine; ++s) whi = i + s;
            } else {
                wlo = max(0, i - region);
                whi = min(m - 1, i + region);
            }
            const double xi = v[i];
            double above = 100.0 * oSD, below = 100.0 * oSD;
            bool keep = false;
            for (int j = wlo; j <= whi; ++j) {
                if (j == i) continue;
                const double dist = xi - v[j];
                if (fabs(dist) <= oSD) { keep = true; break; }
                if (dist < above) above = dist;
                if (-dist < below) below = -dist;
            }
            double y = xi;
            if (!keep && !((above <= 0.0) && (below <= 0.0))) {
                double buf[2 * SM_MAX_REGION + 1];
                const int cnt = whi - wlo + 1;
                for (int j = 0; j < cnt; ++j) {  // insertion sort, ascending
                    const double val = v[wlo + j];
                    int k = j;
                    while (k > 0 && buf[k - 1] > val) { buf[k] = buf[k - 1]; --k; }
                    buf[k] = val;
                }
                const int h = cnt / 2;
                const double med = (cnt == 2 * h) ? (buf[h - 1] + buf[h]) / 2.0 : buf[h];
                if (above > 0.0) y = med + sSD;
                if (below > 0.0) y = med - sSD;
            }
            out[lo + fidx[lo + i]] = y;
        }
    }
}

// ---- windows wider than SM_MAX_REGION markers (smooth_device takes this path for region > 64) ------------------------
//   k_sm_run_mark, k_sm_run_end  the first and last position of every finite marker's run of equal labels, so that the
//                  window is clipped without walking `region` labels (cbs_gpu_smooth; in segment_batch a group has one
//                  label and its run is the whole group)
//   k_sm_wide      the outlier test, nearest neighbours first; markers that need a median go to a list
//   k_sm_median    the window median of each listed marker by an exact radix select
// The window [max(run_lo, i-R), min(run_hi, i+R)] is computed in 64 bits: R may be anything up to INT_MAX.
// No scratch of its own per marker: the run bounds (2 ints) take the slot of the sorted differences' input, the median
// list (8 B per entry) that of the sorted differences, both free once k_sm_sd has run.

// an entry of the median list: group (31 bits), finite index in the group (31 bits), above > 0, below > 0
__device__ __forceinline__ unsigned long long sm_med_item(int g, int i, bool above_pos, bool below_pos) {
    return ((unsigned long long)g << 33) | ((unsigned long long)i << 2) | (above_pos ? 2ULL : 0ULL) | (below_pos ? 1ULL : 0ULL);
}

// window of finite index i of a group of m finite values (positions lo..): clipped to its label run, or to the group when
// run_start == nullptr
__device__ __forceinline__ void sm_wide_window(int i, long long lo, int m, const int* __restrict__ run_start,
                                               const int* __restrict__ run_end, int region, int& wlo, int& whi) {
    int rlo = 0, rhi = m - 1;
    if (run_start) {
        const int s = run_start[lo + i];
        rlo = (int)(s - lo);
        rhi = (int)(run_end[s] - lo);
    }
    wlo = (int)max((long long)rlo, (long long)i - region);
    whi = (int)min((long long)rhi, (long long)i + region);
}

// start[p] = p at the first position of a run (and at the non-finite tail slots of a group), else 0; an inclusive max-scan
// (smooth_device) then gives every position the start of its run.  Positions are global and fit an int (fidx is int).
__global__ void k_sm_run_mark(const int* __restrict__ flab, const long long* __restrict__ off, int n_groups,
                              const SmoothGroupOut* __restrict__ gout, int* __restrict__ start) {
    for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
        const long long lo = off[g];
        const int n = (int)(off[g + 1] - lo), m = gout[g].m;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
            start[lo + i] = (i == 0 || i >= m || flab[lo + i] != flab[lo + i - 1]) ? (int)(lo + i) : 0;
    }
}
struct SmMaxInt {
    __host__ __device__ int operator()(int a, int b) const { return a > b ? a : b; }
};
// end_at[s] = last position of the run that starts at s
__global__ void k_sm_run_end(const int* __restrict__ flab, const long long* __restrict__ off, int n_groups,
                             const SmoothGroupOut* __restrict__ gout, const int* __restrict__ start, int* __restrict__ end_at) {
    for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
        const long long lo = off[g];
        const int m = gout[g].m;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x)
            if (i == m - 1 || flab[lo + i + 1] != flab[lo + i]) end_at[start[lo + i]] = (int)(lo + i);
    }
}

// Thread per finite marker.  The reference scans the window left to right and stops at the first neighbour within oSD;
// whether such a neighbour exists does not depend on the order, so the scan here goes nearest-first (i-1, i+1, i-2, ...)
// and ends after O(1) neighbours on noisy data.  A marker that is not kept has seen its whole window, and `above` and
// `below` are minima, which do not depend on the order either.  run_start == nullptr: the run is the whole group.
__global__ void __launch_bounds__(256) k_sm_wide(const double* __restrict__ fv, const int* __restrict__ fidx,
                                                 const int* __restrict__ run_start, const int* __restrict__ run_end,
                                                 const long long* __restrict__ off, int n_groups, int region,
                                                 const SmoothGroupOut* __restrict__ gout, double* __restrict__ out,
                                                 unsigned long long* __restrict__ med, unsigned* __restrict__ n_med) {
    for (int g = blockIdx.y; g < n_groups; g += gridDim.y) {
        const SmoothGroupOut go = gout[g];
        if (!go.valid) continue;
        const long long lo = off[g];
        const double* v = fv + lo;
        const int m = go.m;
        const double oSD = go.oSD;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
            int wlo, whi;
            sm_wide_window(i, lo, m, run_start, run_end, region, wlo, whi);
            const double xi = v[i];
            double above = 100.0 * oSD, below = 100.0 * oSD;
            bool keep = false;
            const int reach = max(i - wlo, whi - i);
            for (int s = 1; s <= reach; ++s) {
                if (i - s >= wlo) {
                    const double dist = xi - v[i - s];
                    if (fabs(dist) <= oSD) { keep = true; break; }
                    if (dist < above) above = dist;
                    if (-dist < below) below = -dist;
                }
                if (i + s <= whi) {
                    const double dist = xi - v[i + s];
                    if (fabs(dist) <= oSD) { keep = true; break; }
                    if (dist < above) above = dist;
                    if (-dist < below) below = -dist;
                }
            }
            if (keep || ((above <= 0.0) && (below <= 0.0))) { out[lo + fidx[lo + i]] = xi; continue; }
            const unsigned k = atomicAdd(n_med, 1u);
            med[k] = sm_med_item(g, i, above > 0.0, below > 0.0);
        }
    }
}

// order-preserving 64-bit keys of doubles (finite values: the compacted subsequence)
__device__ __forceinline__ unsigned long long sm_key(double x) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(x);
    return (u >> 63) ? ~u : (u | 0x8000000000000000ULL);
}
__device__ __forceinline__ double sm_unkey(unsigned long long k) {
    return __longlong_as_double((long long)((k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k));
}

// The value of rank `rank` (0-based, ascending) among v[0..cnt), by the whole CTA: eight passes of an 8-bit radix select
// on sm_key.  Exact: it returns the same order statistic as a sort, except that -0.0 ranks below +0.0 here, while the
// reference's sort leaves equal zeros in the order its algorithm happens to produce (see k_sm_median).
__device__ double cta_select(const double* v, int cnt, int rank, unsigned* s_hist, unsigned long long* s_pref, int* s_rank) {
    const int tid = threadIdx.x, lane = tid & 31;
    unsigned long long prefix = 0, mask = 0;
    for (int shift = 56; shift >= 0; shift -= 8) {
        for (int b = tid; b < 256; b += blockDim.x) s_hist[b] = 0u;
        __syncthreads();
        for (int j = tid; j < cnt; j += blockDim.x) {
            const unsigned long long k = sm_key(v[j]);
            if ((k & mask) == prefix) atomicAdd(&s_hist[(k >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (tid < 32) {  // lane l owns bins 8l..8l+7: the bin that holds `rank`, by a warp prefix sum
            unsigned c[8], tot = 0;
#pragma unroll
            for (int q = 0; q < 8; ++q) { c[q] = s_hist[8 * lane + q]; tot += c[q]; }
            unsigned incl = tot;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned y = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += y; }
            unsigned below = incl - tot;
            if (below <= (unsigned)rank && (unsigned)rank < incl) {
                for (int q = 0; q < 8; ++q) {
                    if ((unsigned)rank < below + c[q]) {
                        *s_pref = prefix | ((unsigned long long)(8 * lane + q) << shift);
                        *s_rank = rank - (int)below;
                        break;
                    }
                    below += c[q];
                }
            }
        }
        __syncthreads();
        prefix = *s_pref;
        rank = *s_rank;
        mask |= 0xffULL << shift;
    }
    return sm_unkey(prefix);
}

#define SM_MED_SMEM_VALUES 12288  // windows of up to this many markers are staged in shared memory (96 KB)

// CTA per listed marker: the median of its window including x_i (smooth.cpp:108-113, the mean of the two middle values for
// an even count), then median +- sSD as the reference applies it.  Windows up to SM_MED_SMEM_VALUES markers are copied to
// shared memory first; longer ones are selected from global memory.  Any exact selection returns the reference's values;
// the one exception is the sign of a zero median when sSD = 0 (the key order puts -0.0 before +0.0, the reference's sort
// does not order them), and -0.0 == 0.0 as a value.
__global__ void __launch_bounds__(256) k_sm_median(const double* __restrict__ fv, const int* __restrict__ fidx,
                                                   const int* __restrict__ run_start, const int* __restrict__ run_end,
                                                   const long long* __restrict__ off, int region,
                                                   const SmoothGroupOut* __restrict__ gout,
                                                   const unsigned long long* __restrict__ med, const unsigned* __restrict__ n_med,
                                                   double* __restrict__ out) {
    extern __shared__ __align__(16) double s_win[];
    __shared__ unsigned s_hist[256];
    __shared__ unsigned long long s_pref;
    __shared__ int s_rank;
    const unsigned total = *n_med;
    for (unsigned k = blockIdx.x; k < total; k += gridDim.x) {
        const unsigned long long it = med[k];
        const int g = (int)(it >> 33), i = (int)((it >> 2) & 0x7fffffffULL);
        const long long lo = off[g];
        int wlo, whi;
        sm_wide_window(i, lo, gout[g].m, run_start, run_end, region, wlo, whi);
        const int cnt = whi - wlo + 1;
        const double* src = fv + lo + wlo;
        __syncthreads();  // the previous item's readers of s_win are done
        if (cnt <= SM_MED_SMEM_VALUES) {
            for (int j = threadIdx.x; j < cnt; j += blockDim.x) s_win[j] = src[j];
            __syncthreads();
            src = s_win;
        }
        const int h = cnt / 2;
        double mv;
        if (cnt == 2 * h) {
            const double a = cta_select(src, cnt, h - 1, s_hist, &s_pref, &s_rank);
            const double b = cta_select(src, cnt, h, s_hist, &s_pref, &s_rank);
            mv = (a + b) / 2.0;
        } else mv = cta_select(src, cnt, h, s_hist, &s_pref, &s_rank);
        if (threadIdx.x == 0) {
            const double sSD = gout[g].sSD;
            double y = fv[lo + i];
            if (it & 2ULL) y = mv + sSD;  // above > 0
            if (it & 1ULL) y = mv - sSD;  // below > 0
            out[lo + fidx[lo + i]] = y;
        }
    }
}

// cngpld::summarize_cn (lib/cngpld/summarize.cpp:41-75): thread per output position; `pos_off` delimits the positions of a
// unit, `seg_off` its segments.  Overlap and altered counts and the sum follow the reference's loop order.
__global__ void k_summarize_cn(const unsigned long long* __restrict__ start, const unsigned long long* __restrict__ end,
                               const float* __restrict__ value, const long long* __restrict__ seg_off,
                               const long long* __restrict__ pos_off, int n_units, const unsigned long long* __restrict__ pos,
                               int direction, double cutoff, double* __restrict__ out) {
    const long long total = pos_off[n_units];
    for (long long p = blockIdx.x * (long long)blockDim.x + threadIdx.x; p < total; p += (long long)gridDim.x * blockDim.x) {
        int lo = 0, hi = n_units;  // unit u with pos_off[u] <= p < pos_off[u+1]
        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (pos_off[mid] <= p) lo = mid; else hi = mid; }
        const unsigned long long q = pos[p];
        long long overlap = 0, altered = 0;
        double sum = 0.0;
        for (long long k = seg_off[lo]; k < seg_off[lo + 1]; ++k) {
            if (start[k] <= q && q <= end[k]) {
                ++overlap;
                const double adj = (double)direction * (double)value[k];
                if (adj > cutoff) { sum += exp(adj); ++altered; }
            }
        }
        out[p] = altered == 0 ? 0.0 : sum / (double)overlap;
    }
}

__global__ void k_count_nonfinite(const double* x, long long n, int* flag) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        if (!isfinite(x[i])) *flag = 1;
}

}  // namespace cbsg
