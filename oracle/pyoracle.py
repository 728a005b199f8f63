"""TEST INFRASTRUCTURE -- ctypes bindings for the two CPU checkers.

* ``Oracle``  -> oracle/liboracle.so   (our C restatement, oracle/cbs_oracle.c)
* ``Ref``     -> oracle/_ref/libcbs_ref.so (the UNMODIFIED reference lib/cbs sources,
  compiled by oracle/Makefile; absent if it was never built)

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from dataclasses import dataclass

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)
c_i64_p = C.POINTER(C.c_int64)
c_u64_p = C.POINTER(C.c_uint64)


def _dp(a):
    return a.ctypes.data_as(c_double_p)


def _ip(a):
    return a.ctypes.data_as(c_int_p)


def build(ref: bool = True) -> None:
    """Compile liboracle.so (always) and _ref/libcbs_ref.so (when /root/reference exists)."""
    targets = ["oracle"] + (["ref"] if ref else [])
    subprocess.run(["make", "-s", "-C", HERE] + targets, check=True)


class OrcRng(C.Structure):
    _fields_ = [
        ("kind", C.c_int),
        ("mt", C.c_uint64 * 312),
        ("mti", C.c_int),
        ("draws", C.c_uint64),
        ("key0", C.c_uint32),
        ("key1", C.c_uint32),
        ("stage", C.c_uint32),
        ("perm", C.c_uint32),
        ("k", C.c_uint32),
    ]


class OrcTmax(C.Structure):
    _fields_ = [("stat", C.c_double), ("start", C.c_int), ("end", C.c_int)]


class OrcCpt(C.Structure):
    _fields_ = [
        ("ncpt", C.c_int),
        ("icpt", C.c_int * 2),
        ("iseg", C.c_int * 2),
        ("ostat", C.c_double),
        ("perms_run", C.c_int),
        ("nrej", C.c_int),
        ("exit_code", C.c_int),
        ("edge_p", C.c_double * 2),
    ]


class OrcSplitRec(C.Structure):
    _fields_ = [
        ("lo", C.c_int),
        ("hi", C.c_int),
        ("ostat", C.c_double),
        ("iseg0", C.c_int),
        ("iseg1", C.c_int),
        ("ncpt", C.c_int),
        ("icpt0", C.c_int),
        ("icpt1", C.c_int),
        ("perms_run", C.c_int),
        ("nrej", C.c_int),
        ("exit_code", C.c_int),
        ("called", C.c_int),
        ("edge_p0", C.c_double),
        ("edge_p1", C.c_double),
    ]


class OrcSegOpts(C.Structure):
    _fields_ = [
        ("ibin", C.c_int),
        ("alpha", C.c_double),
        ("nperm", C.c_int),
        ("hybrid", C.c_int),
        ("min_width", C.c_int),
        ("kmax", C.c_int),
        ("nmin", C.c_int),
        ("eta", C.c_double),
        ("tol", C.c_double),
        ("undo_prune", C.c_int),
        ("undo_prune_cutoff", C.c_double),
    ]


class OrcCohortOpts(C.Structure):
    _fields_ = [
        ("seg", OrcSegOpts),
        ("do_smooth", C.c_int),
        ("smooth_region", C.c_int),
        ("outlier_sd_scale", C.c_double),
        ("smooth_sd_scale", C.c_double),
        ("trim", C.c_double),
        ("rng_kind", C.c_int),
        ("seed", C.c_uint64),
        ("chain", C.c_int),
    ]


class SplitIntoItself(RuntimeError):
    """The weighted driver reached a decision that would re-create its own segment (oracle/cbs_oracle.h, code -4): the
    reference would test that segment again forever."""


def weight_tables(w):
    """rw = sqrt(w) and cw = cumsum(w)/sqrt(sum w), summed in order as cbs::segment_weighted (and the device) does."""
    w = np.ascontiguousarray(w, dtype=np.float64)
    csum = np.cumsum(w)  # sequential
    return np.sqrt(w), csum / np.sqrt(csum[-1])


@dataclass
class SegParams:
    """Mirror of the `cna segment` options (src/cna_segment.hpp:67-79)."""

    alpha: float = 0.01
    nperm: int = 200
    hybrid: bool = False
    min_width: int = 2
    kmax: int = 25
    nmin: int = 200
    eta: float = 0.05
    tol: float = 1e-6
    ibin: bool = False
    undo_prune: bool = False
    undo_prune_cutoff: float = 0.05
    do_smooth: bool = True
    smooth_region: int = 10
    outlier_sd_scale: float = 4.0
    smooth_sd_scale: float = 2.0
    trim: float = 0.025
    rng_kind: int = 0  # 0 = mt19937_64 replay, 1 = philox
    seed: int = 1
    chain: bool = False

    def seg_opts(self) -> OrcSegOpts:
        return OrcSegOpts(int(self.ibin), self.alpha, self.nperm, int(self.hybrid), self.min_width, self.kmax,
                          self.nmin, self.eta, self.tol, int(self.undo_prune), self.undo_prune_cutoff)

    def cohort_opts(self) -> OrcCohortOpts:
        return OrcCohortOpts(self.seg_opts(), int(self.do_smooth), self.smooth_region, self.outlier_sd_scale,
                             self.smooth_sd_scale, self.trim, self.rng_kind, self.seed, int(self.chain))


class Oracle:
    """Our C restatement."""

    def __init__(self, path: str | None = None):
        path = path or os.path.join(HERE, "liboracle.so")
        if not os.path.exists(path):
            build(ref=False)
        L = self.lib = C.CDLL(path)
        L.orc_tmaxo.restype = OrcTmax
        L.orc_tmaxo.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_int]
        L.orc_tmaxp.restype = C.c_double
        L.orc_tmaxp.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_int]
        L.orc_htmaxp.restype = C.c_double
        L.orc_htmaxp.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int]
        L.orc_tailp.restype = C.c_double
        L.orc_tailp.argtypes = [C.c_double, C.c_double, C.c_int, C.c_int, C.c_double]
        L.orc_arc_evals.restype = C.c_uint64
        L.orc_rng_seed_mt.argtypes = [C.POINTER(OrcRng), C.c_uint64]
        L.orc_rng_seed_philox.argtypes = [C.POINTER(OrcRng), C.c_uint64]
        L.orc_rng_set_task.argtypes = [C.POINTER(OrcRng), C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        L.orc_rng_begin.argtypes = [C.POINTER(OrcRng), C.c_uint32, C.c_uint32]
        L.orc_rng_u64.restype = C.c_uint64
        L.orc_rng_u64.argtypes = [C.POINTER(OrcRng)]
        L.orc_rng_unif.restype = C.c_double
        L.orc_rng_unif.argtypes = [C.POINTER(OrcRng)]
        L.orc_rng_discard.argtypes = [C.POINTER(OrcRng), C.c_uint64]
        L.orc_task_key.restype = C.c_uint64
        L.orc_task_key.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32]
        L.orc_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.orc_xperm.argtypes = [c_double_p, C.c_int, c_double_p, C.POINTER(OrcRng)]
        L.orc_tpermp.restype = C.c_double
        L.orc_tpermp.argtypes = [C.c_int, C.c_int, C.c_int, c_double_p, C.c_int, C.POINTER(OrcRng), c_double_p]
        L.orc_fndcpt.restype = OrcCpt
        L.orc_fndcpt.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_double, C.c_int, C.c_double, C.POINTER(OrcRng)]
        L.orc_segment.restype = C.c_int
        L.orc_segment.argtypes = [c_double_p, C.c_int, C.POINTER(OrcSegOpts), C.POINTER(OrcRng), C.c_uint64,
                                  C.c_uint64, C.c_int, c_int_p, c_double_p, C.POINTER(OrcSplitRec), C.c_int, c_int_p]
        L.orc_norm_quantile.restype = C.c_double
        L.orc_norm_quantile.argtypes = [C.c_double]
        L.orc_inflfact.restype = C.c_double
        L.orc_inflfact.argtypes = [C.c_double]
        L.orc_smooth.restype = C.c_int
        L.orc_smooth.argtypes = [c_double_p, c_int_p, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_double,
                                 c_double_p]
        L.orc_segment_units.restype = C.c_int64
        L.orc_segment_units.argtypes = [c_double_p, c_i64_p, c_int_p, c_u64_p, C.c_int, C.POINTER(OrcCohortOpts),
                                        C.c_int64, c_int_p, c_int_p, c_double_p, c_u64_p, C.POINTER(OrcSplitRec),
                                        C.c_int64, c_i64_p, c_int_p]
        L.orc_segment_weighted.restype = C.c_int
        L.orc_segment_weighted.argtypes = [c_double_p, c_double_p, C.c_int, C.POINTER(OrcSegOpts), C.POINTER(OrcRng),
                                           C.c_uint64, C.c_uint64, C.c_int, c_int_p, c_double_p]
        L.orc_segment_weighted_units.restype = C.c_int64
        L.orc_segment_weighted_units.argtypes = [c_double_p, c_double_p, c_i64_p, c_u64_p, C.c_int,
                                                 C.POINTER(OrcCohortOpts), C.c_int64, c_int_p, c_int_p, c_double_p,
                                                 c_u64_p]
        L.orc_segment_weighted_units_log.restype = C.c_int64
        L.orc_segment_weighted_units_log.argtypes = [c_double_p, c_double_p, c_i64_p, c_u64_p, C.c_int,
                                                     C.POINTER(OrcCohortOpts), C.c_int64, c_int_p, c_int_p, c_double_p,
                                                     c_u64_p, C.POINTER(OrcSplitRec), C.c_int64, c_i64_p, c_int_p]
        L.orc_wtmaxo.restype = OrcTmax
        L.orc_wtmaxo.argtypes = [c_double_p, c_double_p, c_double_p, C.c_int, C.c_double, C.c_int]
        L.orc_wtmaxp.restype = C.c_double
        L.orc_wtmaxp.argtypes = [c_double_p, c_double_p, c_double_p, C.c_int, C.c_int]
        L.orc_wxperm.argtypes = [c_double_p, c_double_p, C.c_int, c_double_p, C.POINTER(OrcRng)]
        L.orc_wtpermp.restype = C.c_double
        L.orc_wtpermp.argtypes = [C.c_int, C.c_int, C.c_int, c_double_p, c_double_p, c_double_p, C.c_int,
                                  C.POINTER(OrcRng), c_double_p]
        L.orc_getmncwt.argtypes = [c_double_p, C.c_int, C.c_int, c_double_p, c_double_p]
        L.orc_hwtmaxp.restype = C.c_double
        L.orc_hwtmaxp.argtypes = [c_double_p, c_double_p, c_double_p, c_double_p, C.c_int, C.c_int, C.c_int]
        L.orc_wfindcpt.restype = OrcCpt
        L.orc_wfindcpt.argtypes = [c_double_p, c_double_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int, C.c_int,
                                   C.c_int, C.c_int, C.c_double, C.POINTER(OrcRng)]

    # -- rng ---------------------------------------------------------------
    def rng_mt(self, seed: int) -> OrcRng:
        r = OrcRng()
        self.lib.orc_rng_seed_mt(C.byref(r), seed)
        return r

    def rng_philox(self, seed: int) -> OrcRng:
        r = OrcRng()
        self.lib.orc_rng_seed_philox(C.byref(r), seed)
        return r

    # -- kernels ------------------------------------------------------------
    def summarize_cn(self, start, end, value, direction, cutoff, positions=None):
        """cngpld::summarize_cn for the segments of one sample and chromosome (oracle/cngpld_oracle.c).
        Returns (positions uint64, values float64); raises ValueError where the reference throws invalid_argument."""
        L = self.lib
        L.orc_summarize_cn.restype = C.c_longlong
        st = np.ascontiguousarray(start, np.uint64)
        en = np.ascontiguousarray(end, np.uint64)
        va = np.ascontiguousarray(value, np.float32)
        n = len(st)
        ps = None if positions is None else np.ascontiguousarray(positions, np.uint64)
        cap = max(2 * n, 0 if ps is None else len(ps), 1)
        out_pos = np.zeros(cap, np.uint64)
        out_val = np.zeros(cap, np.float64)
        got = L.orc_summarize_cn(st.ctypes.data_as(C.c_void_p), en.ctypes.data_as(C.c_void_p), va.ctypes.data_as(C.c_void_p),
                                 C.c_longlong(n), C.c_int(direction), C.c_double(cutoff),
                                 None if ps is None else ps.ctypes.data_as(C.c_void_p),
                                 C.c_longlong(0 if ps is None else len(ps)), out_pos.ctypes.data_as(C.c_void_p),
                                 out_val.ctypes.data_as(C.c_void_p))
        if got < 0:
            raise ValueError("invalid_argument")
        return out_pos[:got].copy(), out_val[:got].copy()

    def tmaxo(self, x, tss, al0=2, ibin=False):
        x = np.ascontiguousarray(x, dtype=np.float64)
        r = self.lib.orc_tmaxo(_dp(x), len(x), tss, al0, int(ibin))
        return r.stat, r.start, r.end

    def tmaxp(self, px, tss, al0=2, ibin=False):
        px = np.ascontiguousarray(px, dtype=np.float64)
        return self.lib.orc_tmaxp(_dp(px), len(px), tss, al0, int(ibin))

    def htmaxp(self, px, tss, k, al0=2, ibin=False):
        px = np.ascontiguousarray(px, dtype=np.float64)
        return self.lib.orc_htmaxp(_dp(px), len(px), tss, k, al0, int(ibin))

    def tailp(self, b, delta, m, ngrid=100, tol=1e-6):
        return self.lib.orc_tailp(b, delta, m, ngrid, tol)

    def xperm(self, x, rng: OrcRng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        px = np.empty_like(x)
        self.lib.orc_xperm(_dp(x), len(x), _dp(px), C.byref(rng))
        return px

    def tpermp(self, n1, n2, x, nperm, rng: OrcRng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        scratch = np.empty(max(1, n1 + n2), dtype=np.float64)
        return self.lib.orc_tpermp(n1, n2, n1 + n2, _dp(x), nperm, C.byref(rng), _dp(scratch))

    def fndcpt(self, x, tss, nperm, cpval, rng: OrcRng, ibin=False, hybrid=False, al0=2, hk=25, delta=0.0, ngrid=100,
               tol=1e-6) -> OrcCpt:
        x = np.ascontiguousarray(x, dtype=np.float64)
        return self.lib.orc_fndcpt(_dp(x), len(x), tss, nperm, cpval, int(ibin), int(hybrid), al0, hk, delta, ngrid,
                                   tol, C.byref(rng))

    def segment(self, x, p: SegParams, rng: OrcRng | None = None, unit_id: int = 0, want_log: bool = False):
        x = np.ascontiguousarray(x, dtype=np.float64)
        if rng is None:
            rng = self.rng_mt(p.seed) if p.rng_kind == 0 else self.rng_philox(p.seed)
        cap = max(16, len(x))
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        log_cap = 4 * cap + 16 if want_log else 0
        log = (OrcSplitRec * max(1, log_cap))()
        nlog = C.c_int(0)
        opts = p.seg_opts()
        k = self.lib.orc_segment(_dp(x), len(x), C.byref(opts), C.byref(rng), p.seed, unit_id, cap, _ip(lengths),
                                 _dp(means), log if want_log else None, log_cap, C.byref(nlog))
        assert k >= 0
        out = (lengths[:k].copy(), means[:k].copy())
        if want_log:
            return out + ([log[i] for i in range(nlog.value)],)
        return out

    def segment_weighted(self, x, w, p: SegParams, rng: OrcRng | None = None, unit_id: int = 0):
        """cbs::segment_weighted restated (cbs_oracle_weighted.c) -> (lengths, means)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        if rng is None:
            rng = self.rng_philox(p.seed) if p.rng_kind else self.rng_mt(p.seed)
        cap = max(16, len(x))
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        opts = p.seg_opts()
        k = self.lib.orc_segment_weighted(_dp(x), _dp(w), len(x), C.byref(opts), C.byref(rng), p.seed, unit_id, cap,
                                          _ip(lengths), _dp(means))
        if k == -3:
            raise NotImplementedError("weighted hybrid method is not restated")
        assert k >= 0, k
        return lengths[:k].copy(), means[:k].copy()

    def segment_weighted_units(self, values, weights, unit_off, p: SegParams, unit_ids=None, want_log=False):
        """Weighted segmentation of every unit; with want_log, also the split log as segment_units returns it.
        Raises SplitIntoItself where the reference would not terminate."""
        values = np.ascontiguousarray(values, dtype=np.float64)
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        unit_off = np.ascontiguousarray(unit_off, dtype=np.int64)
        n_units = len(unit_off) - 1
        cap = int(len(values)) + n_units + 16
        seg_count = np.zeros(n_units, dtype=np.int32)
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        draws = np.zeros(n_units, dtype=np.uint64)
        uid = None if unit_ids is None else np.ascontiguousarray(unit_ids, dtype=np.uint64)
        log_cap = (4 * cap) if want_log else 0
        log = (OrcSplitRec * max(1, log_cap))()
        log_unit = np.zeros(max(1, log_cap), dtype=np.int32)
        nlog = C.c_int64(0)
        opts = p.cohort_opts()
        tot = self.lib.orc_segment_weighted_units_log(
            _dp(values), _dp(weights), unit_off.ctypes.data_as(c_i64_p),
            uid.ctypes.data_as(c_u64_p) if uid is not None else None, n_units, C.byref(opts), cap, _ip(seg_count),
            _ip(lengths), _dp(means), draws.ctypes.data_as(c_u64_p), log if want_log else None, log_cap,
            C.byref(nlog), _ip(log_unit))
        if tot == -3:
            raise NotImplementedError("weighted hybrid method is not restated")
        if tot == -4:
            last = log[nlog.value - 1] if want_log and nlog.value else None
            raise SplitIntoItself("a weighted split decision would re-create its own segment"
                                  + (f" (unit {log_unit[nlog.value - 1]}, [{last.lo}, {last.hi}))" if last else ""))
        assert tot >= 0, tot
        res = dict(seg_count=seg_count, lengths=lengths[:tot].copy(), means=means[:tot].copy(), draws=draws)
        if want_log:
            res["log"] = [(int(log_unit[i]), log[i]) for i in range(nlog.value)]
        return res

    # -- weighted low-level functions (CBS.cpp:538-957); rw and cw derived from w by weight_tables() ----------------
    def wtmaxo(self, x, w, tss, al0=2):
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        _, cw = weight_tables(w)
        r = self.lib.orc_wtmaxo(_dp(x), _dp(w), _dp(cw), len(x), tss, al0)
        return r.stat, r.start, r.end

    def wtmaxp(self, px, w, al0=2):
        px = np.ascontiguousarray(px, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        _, cw = weight_tables(w)
        return self.lib.orc_wtmaxp(_dp(px), _dp(w), _dp(cw), len(px), al0)

    def wxperm(self, x, w, rng: OrcRng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        rw, _ = weight_tables(w)
        px = np.empty_like(x)
        self.lib.orc_wxperm(_dp(x), _dp(rw), len(x), _dp(px), C.byref(rng))
        return px

    def wtpermp(self, n1, n2, x, w, nperm, rng: OrcRng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        rw, _ = weight_tables(w)
        scratch = np.empty(max(1, n1 + n2), dtype=np.float64)
        return self.lib.orc_wtpermp(n1, n2, n1 + n2, _dp(x), _dp(w), _dp(rw), nperm, C.byref(rng), _dp(scratch))

    def getmncwt(self, w, k):
        """(mn[0..k], delta) of the weighted hybrid method"""
        _, cw = weight_tables(w)
        mn = np.zeros(k + 1, dtype=np.float64)
        delta = C.c_double()
        self.lib.orc_getmncwt(_dp(cw), len(cw), k, _dp(mn), C.byref(delta))
        return mn, delta.value

    def hwtmaxp(self, px, w, k, al0=2):
        px = np.ascontiguousarray(px, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        _, cw = weight_tables(w)
        mn, _ = self.getmncwt(w, k)
        return self.lib.orc_hwtmaxp(_dp(px), _dp(w), _dp(cw), _dp(mn), len(px), k, al0)

    def wfindcpt(self, x, w, tss, nperm, cpval, rng: OrcRng, hybrid=False, al0=2, hk=25, ngrid=100, tol=1e-6) -> OrcCpt:
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        return self.lib.orc_wfindcpt(_dp(x), _dp(w), len(x), tss, nperm, cpval, int(hybrid), al0, hk, ngrid, tol,
                                     C.byref(rng))

    def smooth(self, values, chrom, smooth_region=10, outlier_sd_scale=4.0, smooth_sd_scale=2.0, trim=0.025):
        values = np.ascontiguousarray(values, dtype=np.float64)
        chrom = np.ascontiguousarray(chrom, dtype=np.int32)
        if len(values) != len(chrom):
            raise ValueError("values and chrom must have same length")
        out = np.empty_like(values)
        rc = self.lib.orc_smooth(_dp(values), _ip(chrom), len(values), smooth_region, outlier_sd_scale,
                                 smooth_sd_scale, trim, _dp(out))
        if rc == 2:
            raise OverflowError("quantile overflow (trim == 0)")
        if rc:
            raise ValueError("invalid argument")
        return out

    def segment_units(self, values, unit_off, chrom_label, p: SegParams, unit_ids=None, want_log=False):
        values = np.ascontiguousarray(values, dtype=np.float64)
        unit_off = np.ascontiguousarray(unit_off, dtype=np.int64)
        n_units = len(unit_off) - 1
        chrom_label = np.ascontiguousarray(chrom_label, dtype=np.int32)
        cap = int(len(values)) + n_units + 16
        seg_count = np.zeros(n_units, dtype=np.int32)
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        draws = np.zeros(n_units, dtype=np.uint64)
        uid = None
        if unit_ids is not None:
            uid = np.ascontiguousarray(unit_ids, dtype=np.uint64)
        log_cap = (4 * cap) if want_log else 0
        log = (OrcSplitRec * max(1, log_cap))()
        log_unit = np.zeros(max(1, log_cap), dtype=np.int32)
        nlog = C.c_int64(0)
        opts = p.cohort_opts()
        tot = self.lib.orc_segment_units(
            _dp(values), unit_off.ctypes.data_as(c_i64_p), _ip(chrom_label),
            uid.ctypes.data_as(c_u64_p) if uid is not None else None, n_units, C.byref(opts), cap, _ip(seg_count),
            _ip(lengths), _dp(means), draws.ctypes.data_as(c_u64_p), log if want_log else None, log_cap,
            C.byref(nlog), _ip(log_unit))
        if tot == -2:
            raise ValueError("invalid argument")
        assert tot >= 0, tot
        res = dict(seg_count=seg_count, lengths=lengths[:tot].copy(), means=means[:tot].copy(), draws=draws)
        if want_log:
            res["log"] = [(int(log_unit[i]), log[i]) for i in range(nlog.value)]
        return res


class Ref:
    """The compiled, unmodified reference (oracle/_ref/libcbs_ref.so)."""

    @staticmethod
    def available() -> bool:
        return os.path.exists(os.path.join(HERE, "_ref", "libcbs_ref.so"))

    def __init__(self, path: str | None = None):
        path = path or os.path.join(HERE, "_ref", "libcbs_ref.so")
        L = self.lib = C.CDLL(path)
        L.ref_rng_new.restype = C.c_void_p
        L.ref_rng_new.argtypes = [C.c_uint64]
        L.ref_rng_free.argtypes = [C.c_void_p]
        L.ref_rng_discard.argtypes = [C.c_void_p, C.c_uint64]
        L.ref_rng_next_u64.restype = C.c_uint64
        L.ref_rng_next_u64.argtypes = [C.c_void_p]
        L.ref_rng_next_canonical.restype = C.c_double
        L.ref_rng_next_canonical.argtypes = [C.c_void_p]
        L.ref_rng_equals.restype = C.c_int
        L.ref_rng_equals.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64]
        L.ref_tmaxo.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_int, c_double_p, c_int_p, c_int_p]
        L.ref_tmaxp.restype = C.c_double
        L.ref_tmaxp.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_int]
        L.ref_htmaxp.restype = C.c_double
        L.ref_htmaxp.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int]
        L.ref_tailp.restype = C.c_double
        L.ref_tailp.argtypes = [C.c_double, C.c_double, C.c_int, C.c_int, C.c_double]
        L.ref_xperm.argtypes = [c_double_p, C.c_int, c_double_p, C.c_void_p]
        L.ref_tpermp.restype = C.c_double
        L.ref_tpermp.argtypes = [C.c_int, C.c_int, C.c_int, c_double_p, C.c_int, C.c_void_p]
        L.ref_fndcpt.argtypes = [c_double_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int,
                                 C.c_int, C.c_double, C.c_int, C.c_double, C.c_void_p, c_int_p, c_int_p, c_int_p,
                                 c_double_p]
        L.ref_segment.restype = C.c_int
        L.ref_segment.argtypes = [c_double_p, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_int, C.c_double, C.c_int, c_int_p,
                                  c_double_p]
        L.ref_segment_weighted.restype = C.c_int
        L.ref_segment_weighted.argtypes = [c_double_p, c_double_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.c_double, C.c_double, C.c_void_p, C.c_int, C.c_double,
                                           C.c_int, c_int_p, c_double_p]
        L.ref_smooth.restype = C.c_int
        L.ref_smooth.argtypes = [c_double_p, c_int_p, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_double,
                                 c_double_p]
        L.ref_segment_units.restype = C.c_int64
        L.ref_segment_units.argtypes = [c_double_p, c_i64_p, c_int_p, C.c_int, C.c_int, C.c_int, C.c_double,
                                        C.c_double, C.c_double, C.c_double, C.c_int, C.c_int, C.c_int, C.c_int,
                                        C.c_int, C.c_double, C.c_double, C.c_int, C.c_double, C.c_uint64, C.c_int,
                                        C.c_int, C.c_int64, c_int_p, c_int_p, c_double_p]

        L.ref_btmax.restype = C.c_double
        L.ref_btmax.argtypes = [c_double_p, C.c_int]
        L.ref_btailp.restype = C.c_double
        L.ref_btailp.argtypes = [C.c_double, C.c_int, C.c_int, C.c_double]
        L.ref_wtmaxo.argtypes = [c_double_p, c_double_p, C.c_int, C.c_double, C.c_int, c_double_p, c_int_p, c_int_p]
        L.ref_wxperm.argtypes = [c_double_p, c_double_p, C.c_int, c_double_p, C.c_void_p]
        L.ref_wfindcpt.argtypes = [c_double_p, c_double_p, C.c_int, C.c_double, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int,
                                   C.c_int, C.c_double, C.c_void_p, c_int_p, c_int_p, c_int_p, c_double_p]
        L.ref_perm_reject_flags.argtypes = [c_double_p, C.c_int, C.c_double, C.c_double, C.c_int, C.c_uint64, C.c_uint64,
                                            C.c_int64, C.c_int64, C.c_int, C.c_void_p]

    def perm_reject_flags(self, x, tss, thresh, seed, start_draw, perm0, nperms, nthreads, al0=2):
        """flags[k] = permutation perm0+k of fndcpt's max-t loop rejects (reference xperm + tmaxp, threads over the range)"""
        x = np.ascontiguousarray(x, dtype=np.float64)
        flags = np.zeros(int(nperms), dtype=np.uint8)
        self.lib.ref_perm_reject_flags(_dp(x), len(x), float(tss), float(thresh), al0, int(seed), int(start_draw), int(perm0),
                                       int(nperms), int(nthreads), flags.ctypes.data_as(C.c_void_p))
        return flags

    def btmax(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        return self.lib.ref_btmax(_dp(x), len(x))

    def btailp(self, b, m, ng, tol=1e-6):
        return self.lib.ref_btailp(b, m, ng, tol)

    def wtmaxo(self, x, w, tss, al0=2):
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        stat, s, e = C.c_double(), C.c_int(), C.c_int()
        self.lib.ref_wtmaxo(_dp(x), _dp(w), len(x), tss, al0, C.byref(stat), C.byref(s), C.byref(e))
        return stat.value, s.value, e.value

    def wxperm(self, x, rwts, rng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        rw = np.ascontiguousarray(rwts, dtype=np.float64)
        px = np.zeros_like(x)
        self.lib.ref_wxperm(_dp(x), _dp(rw), len(x), _dp(px), rng.h)
        return px

    def wfindcpt(self, x, w, tss, nperm, cpval, rng, hybrid=False, al0=2, hk=25, ngrid=100, tol=1e-6):
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        ncpt, icpt, iseg, ostat = C.c_int(), (C.c_int * 2)(), (C.c_int * 2)(), C.c_double()
        self.lib.ref_wfindcpt(_dp(x), _dp(w), len(x), tss, nperm, cpval, int(hybrid), al0, hk, ngrid, tol, rng.h, C.byref(ncpt), icpt,
                              iseg, C.byref(ostat))
        return dict(ncpt=ncpt.value, icpt=(icpt[0], icpt[1]), iseg=(iseg[0], iseg[1]), ostat=ostat.value)

    class Rng:
        def __init__(self, lib, seed):
            self.lib = lib
            self.h = lib.ref_rng_new(seed)

        def __del__(self):
            if getattr(self, "h", None):
                self.lib.ref_rng_free(self.h)
                self.h = None

    def rng(self, seed: int) -> "Ref.Rng":
        return Ref.Rng(self.lib, seed)

    def rng_equals(self, rng, seed, draws) -> bool:
        return bool(self.lib.ref_rng_equals(rng.h, seed, draws))

    def tmaxo(self, x, tss, al0=2, ibin=False):
        x = np.ascontiguousarray(x, dtype=np.float64)
        stat, s, e = C.c_double(), C.c_int(), C.c_int()
        self.lib.ref_tmaxo(_dp(x), len(x), tss, al0, int(ibin), C.byref(stat), C.byref(s), C.byref(e))
        return stat.value, s.value, e.value

    def tmaxp(self, px, tss, al0=2, ibin=False):
        px = np.ascontiguousarray(px, dtype=np.float64)
        return self.lib.ref_tmaxp(_dp(px), len(px), tss, al0, int(ibin))

    def htmaxp(self, px, tss, k, al0=2, ibin=False):
        px = np.ascontiguousarray(px, dtype=np.float64)
        return self.lib.ref_htmaxp(_dp(px), len(px), tss, k, al0, int(ibin))

    def tailp(self, b, delta, m, ngrid=100, tol=1e-6):
        return self.lib.ref_tailp(b, delta, m, ngrid, tol)

    def xperm(self, x, rng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        px = np.empty_like(x)
        self.lib.ref_xperm(_dp(x), len(x), _dp(px), rng.h)
        return px

    def tpermp(self, n1, n2, x, nperm, rng):
        x = np.ascontiguousarray(x, dtype=np.float64)
        return self.lib.ref_tpermp(n1, n2, n1 + n2, _dp(x), nperm, rng.h)

    def fndcpt(self, x, tss, nperm, cpval, rng, ibin=False, hybrid=False, al0=2, hk=25, delta=0.0, ngrid=100,
               tol=1e-6):
        x = np.ascontiguousarray(x, dtype=np.float64)
        ncpt = C.c_int()
        icpt = (C.c_int * 2)()
        iseg = (C.c_int * 2)()
        ostat = C.c_double()
        self.lib.ref_fndcpt(_dp(x), len(x), tss, nperm, cpval, int(ibin), int(hybrid), al0, hk, delta, ngrid, tol,
                            rng.h, C.byref(ncpt), icpt, iseg, C.byref(ostat))
        return dict(ncpt=ncpt.value, icpt=(icpt[0], icpt[1]), iseg=(iseg[0], iseg[1]), ostat=ostat.value)

    def segment(self, x, p: SegParams, rng=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        rng = rng or self.rng(p.seed)
        cap = max(16, len(x))
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        k = self.lib.ref_segment(_dp(x), len(x), int(p.ibin), p.alpha, p.nperm, int(p.hybrid), p.min_width, p.kmax,
                                 p.nmin, p.eta, p.tol, rng.h, int(p.undo_prune), p.undo_prune_cutoff, cap,
                                 _ip(lengths), _dp(means))
        assert k >= 0
        return lengths[:k].copy(), means[:k].copy()

    def segment_weighted(self, x, w, p: SegParams, rng=None):
        x = np.ascontiguousarray(x, dtype=np.float64)
        w = np.ascontiguousarray(w, dtype=np.float64)
        rng = rng or self.rng(p.seed)
        cap = max(16, len(x))
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        k = self.lib.ref_segment_weighted(_dp(x), _dp(w), len(x), p.alpha, p.nperm, int(p.hybrid), p.min_width, p.kmax,
                                          p.nmin, p.eta, p.tol, rng.h, int(p.undo_prune), p.undo_prune_cutoff, cap,
                                          _ip(lengths), _dp(means))
        assert k >= 0
        return lengths[:k].copy(), means[:k].copy()

    def smooth(self, values, chrom, smooth_region=10, outlier_sd_scale=4.0, smooth_sd_scale=2.0, trim=0.025):
        values = np.ascontiguousarray(values, dtype=np.float64)
        chrom = np.ascontiguousarray(chrom, dtype=np.int32)
        if len(values) != len(chrom):
            raise ValueError("values and chrom must have same length")
        out = np.empty_like(values)
        rc = self.lib.ref_smooth(_dp(values), _ip(chrom), len(values), smooth_region, outlier_sd_scale,
                                 smooth_sd_scale, trim, _dp(out))
        if rc == 2:
            raise OverflowError("quantile overflow (trim == 0)")
        if rc:
            raise ValueError("invalid argument")
        return out

    def segment_units(self, values, unit_off, chrom_label, p: SegParams, nthreads: int = 1):
        values = np.ascontiguousarray(values, dtype=np.float64)
        unit_off = np.ascontiguousarray(unit_off, dtype=np.int64)
        n_units = len(unit_off) - 1
        chrom_label = np.ascontiguousarray(chrom_label, dtype=np.int32)
        cap = int(len(values)) + n_units + 16
        seg_count = np.zeros(n_units, dtype=np.int32)
        lengths = np.zeros(cap, dtype=np.int32)
        means = np.zeros(cap, dtype=np.float64)
        tot = self.lib.ref_segment_units(
            _dp(values), unit_off.ctypes.data_as(c_i64_p), _ip(chrom_label), n_units, int(p.do_smooth),
            p.smooth_region, p.outlier_sd_scale, p.smooth_sd_scale, p.trim, p.alpha, p.nperm, int(p.hybrid),
            p.min_width, p.kmax, p.nmin, p.eta, p.tol, int(p.undo_prune), p.undo_prune_cutoff, p.seed, int(p.chain),
            nthreads, cap, _ip(seg_count), _ip(lengths), _dp(means))
        if tot == -2:
            raise ValueError("invalid argument")
        assert tot >= 0, tot
        return dict(seg_count=seg_count, lengths=lengths[:tot].copy(), means=means[:tot].copy())
