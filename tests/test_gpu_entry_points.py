"""-m gpu: the C ABI entry points (include/cbs_gpu.h) through ctypes: the status code of every entry point for malformed
arguments, and the batched entry points on one unit against the single-vector ones."""
import ctypes as C

import numpy as np
import pytest

import genomic_b200
from genomic_b200 import Params, RNG_MT19937_64, RNG_PHILOX
from genomic_b200.binding import (CResult, CSplit, ERR_INVALID, ERR_NONFINITE, ERR_UNSUPPORTED, F64, HOST, OK)

pytestmark = pytest.mark.gpu

MAX_UNIT = 8388608  # CBS_GPU_MAX_UNIT
DP, I32P, I64P = C.POINTER(C.c_double), C.POINTER(C.c_int32), C.POINTER(C.c_int64)


@pytest.fixture(scope="module")
def api():
    lib = genomic_b200.load_library()
    ctx = genomic_b200.Context(0, lib=lib)
    yield lib, ctx
    ctx.close()


def dp(a):
    return None if a is None else a.ctypes.data_as(DP)


def step_vector(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(0.0, 1.0, n)
    x[n // 3: n // 2] += 1.5
    x[3 * n // 4:] -= 1.0
    return x


def status_cases(lib, h):
    """(name, call, status): each call passes exactly one malformed argument; status is the code it returns."""
    good = step_vector(200, 1)
    w = np.full(200, 1.0)
    bad = good.copy(); bad[17] = np.nan
    badw = w.copy(); badw[5] = np.inf
    huge = np.zeros(MAX_UNIT + 1)
    hw = np.ones(MAX_UNIT + 1)
    prm = Params(nperm=100, do_smooth=False).c()
    tss = float(((good - good.mean()) ** 2).sum())
    out = C.POINTER(CResult)()
    res = []

    def batch(values, off, params=prm, out_=C.byref(out), weights=None, weighted=False):
        off = np.ascontiguousarray(off, dtype=np.int64)
        o = off.ctypes.data_as(I64P)
        if weighted:
            rc = lib.cbs_gpu_segment_weighted_batch(h, dp(values), dp(weights), HOST, o, None, len(off) - 1,
                                                    None if params is None else C.byref(params), out_)
        else:
            rc = lib.cbs_gpu_segment_batch(h, None if values is None else values.ctypes.data_as(C.c_void_p), F64, HOST, o, None,
                                           len(off) - 1, None if params is None else C.byref(params), out_)
        if rc == OK:
            lib.cbs_gpu_result_free(out)
        return rc

    n = len(good)
    for wtd in (False, True):
        name = "segment_weighted_batch" if wtd else "segment_batch"
        ww = w if wtd else None
        res += [
            (f"{name} out=NULL", lambda wtd=wtd, ww=ww: batch(good, [0, n], out_=None, weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} params=NULL", lambda wtd=wtd, ww=ww: batch(good, [0, n], params=None, weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} values=NULL", lambda wtd=wtd, ww=ww: batch(None, [0, n], weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} offsets[0]!=0", lambda wtd=wtd, ww=ww: batch(good, [1, 100, n], weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} decreasing offsets", lambda wtd=wtd, ww=ww: batch(good, [0, 150, 100, n], weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} unit too long", lambda wtd=wtd, ww=ww: batch(huge, [0, MAX_UNIT + 1], weights=hw if wtd else None, weighted=wtd),
             ERR_UNSUPPORTED),
            (f"{name} non-finite", lambda wtd=wtd, ww=ww: batch(bad, [0, n], weights=ww, weighted=wtd), ERR_NONFINITE),
        ]
    res += [
        ("segment_weighted_batch weights=NULL", lambda: batch(good, [0, n], weighted=True), ERR_INVALID),
        ("segment_weighted_batch non-finite weight", lambda: batch(good, [0, n], weights=badw, weighted=True), ERR_INVALID),
    ]

    lengths, means = np.zeros(n, np.int32), np.zeros(n)
    nseg, draws = C.c_int32(0), C.c_uint64(0)

    def one(x, weights=None, weighted=False, params=prm, nseg_=C.byref(nseg)):
        m = n if x is None else len(x)
        p = None if params is None else C.byref(params)
        if weighted:
            return lib.cbs_gpu_segment_weighted(h, dp(x), dp(weights), m, p, None, n, lengths.ctypes.data_as(I32P),
                                                dp(means), nseg_, C.byref(draws))
        return lib.cbs_gpu_segment(h, dp(x), m, p, None, n, lengths.ctypes.data_as(I32P), dp(means), nseg_, C.byref(draws))

    for wtd in (False, True):
        name = "segment_weighted" if wtd else "segment"
        ww = w if wtd else None
        res += [
            (f"{name} values=NULL", lambda wtd=wtd, ww=ww: one(None, ww, wtd), ERR_INVALID),
            (f"{name} n_segments=NULL", lambda wtd=wtd, ww=ww: one(good, ww, wtd, nseg_=None), ERR_INVALID),
            (f"{name} unit too long", lambda wtd=wtd: one(huge, hw if wtd else None, wtd), ERR_UNSUPPORTED),
            (f"{name} non-finite", lambda wtd=wtd, ww=ww: one(bad, ww, wtd), ERR_NONFINITE),
        ]
    res += [
        ("segment_weighted params=NULL", lambda: one(good, w, True, params=None), ERR_INVALID),
        ("segment_weighted weights=NULL", lambda: one(good, None, True), ERR_INVALID),
    ]

    stat, s0, s1 = C.c_double(), C.c_int32(), C.c_int32()
    stats = np.zeros(4)
    tmaxo = lambda x, m, al0, ibin: lib.cbs_gpu_tmaxo(h, dp(x), m, tss, al0, ibin, C.byref(stat), C.byref(s0), C.byref(s1))
    tmaxp = lambda x, m, al0, ibin: lib.cbs_gpu_tmaxp(h, dp(x), m, 1, tss, al0, ibin, dp(stats))
    for ibin in (0, 1):
        for name, f in (("tmaxo", tmaxo), ("tmaxp", tmaxp)):
            res += [
                (f"{name}(ibin={ibin}) values=NULL", lambda f=f, ibin=ibin: f(None, n, 2, ibin), ERR_INVALID),
                (f"{name}(ibin={ibin}) n < 2*al0", lambda f=f, ibin=ibin: f(good, 5, 3, ibin), ERR_INVALID),
                (f"{name}(ibin={ibin}) too long", lambda f=f, ibin=ibin: f(huge, MAX_UNIT + 1, 2, ibin), ERR_UNSUPPORTED),
            ]
    htmaxp = lambda x, m, k, al0, out_: lib.cbs_gpu_htmaxp(h, dp(x), m, 1, C.c_double(tss), k, al0, 0, out_)
    res += [
        ("htmaxp values=NULL", lambda: htmaxp(None, n, 25, 2, dp(stats)), ERR_INVALID),
        ("htmaxp statistics=NULL", lambda: htmaxp(good, n, 25, 2, None), ERR_INVALID),
        ("htmaxp n < k", lambda: htmaxp(good, 20, 25, 2, dp(stats)), ERR_UNSUPPORTED),
        ("htmaxp too long", lambda: htmaxp(huge, MAX_UNIT + 1, 25, 2, dp(stats)), ERR_UNSUPPORTED),
    ]

    split = CSplit()
    pval = C.c_double()

    def fnd(x, m, params=prm, out_=C.byref(split), weights=None, weighted=False):
        p = None if params is None else C.byref(params)
        if weighted:
            return lib.cbs_gpu_wfindcpt(h, dp(x), dp(weights), m, C.c_double(tss), p, 100, None, out_, C.byref(draws))
        return lib.cbs_gpu_fndcpt(h, dp(x), m, C.c_double(tss), p, C.c_double(0.0), 100, None, out_, C.byref(draws))

    for wtd in (False, True):
        name = "wfindcpt" if wtd else "fndcpt"
        ww = w if wtd else None
        res += [
            (f"{name} values=NULL", lambda wtd=wtd, ww=ww: fnd(None, n, weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} params=NULL", lambda wtd=wtd, ww=ww: fnd(good, n, params=None, weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} out=NULL", lambda wtd=wtd, ww=ww: fnd(good, n, out_=None, weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} n < 2*al0", lambda wtd=wtd, ww=ww: fnd(good, 3, weights=ww, weighted=wtd), ERR_INVALID),
            (f"{name} non-finite", lambda wtd=wtd, ww=ww: fnd(bad, n, weights=ww, weighted=wtd), ERR_NONFINITE),
        ]
    res += [
        ("fndcpt too long", lambda: fnd(huge, MAX_UNIT + 1), ERR_UNSUPPORTED),
        ("wfindcpt weights=NULL", lambda: fnd(good, n, weighted=True), ERR_INVALID),
        ("tpermp params=NULL", lambda: lib.cbs_gpu_tpermp(h, dp(good), 100, 100, None, None, C.byref(pval), C.byref(draws)),
         ERR_INVALID),
        ("tpermp pvalue=NULL", lambda: lib.cbs_gpu_tpermp(h, dp(good), 100, 100, C.byref(prm), None, None, C.byref(draws)),
         ERR_INVALID),
        ("tpermp non-finite", lambda: lib.cbs_gpu_tpermp(h, dp(bad), 100, 100, C.byref(prm), None, C.byref(pval),
                                                         C.byref(draws)), ERR_NONFINITE),
        ("wtmaxo weights=NULL", lambda: lib.cbs_gpu_wtmaxo(h, dp(good), None, n, C.c_double(tss), 2, C.byref(stat),
                                                           C.byref(s0), C.byref(s1)), ERR_INVALID),
        ("wtmaxo n < 2*al0", lambda: lib.cbs_gpu_wtmaxo(h, dp(good), dp(w), 3, C.c_double(tss), 2, C.byref(stat),
                                                        C.byref(s0), C.byref(s1)), ERR_INVALID),
        ("wtmaxo non-finite", lambda: lib.cbs_gpu_wtmaxo(h, dp(bad), dp(w), n, C.c_double(tss), 2, C.byref(stat),
                                                         C.byref(s0), C.byref(s1)), ERR_NONFINITE),
        ("xperm values=NULL", lambda: lib.cbs_gpu_xperm(h, None, None, n, None, C.c_uint64(1), dp(np.zeros(n))), ERR_INVALID),
        ("xperm too long", lambda: lib.cbs_gpu_xperm(h, dp(huge), None, MAX_UNIT + 1, None, C.c_uint64(1), dp(huge)),
         ERR_UNSUPPORTED),
    ]
    return res


def test_malformed_arguments_status(api):
    lib, ctx = api
    cases = status_cases(lib, ctx.h)
    got = {name: call() for name, call, _ in cases}
    want = {name: code for name, _, code in cases}
    assert got == want
    # the context stays usable after every refusal
    x = step_vector(3000, 2)
    assert len(ctx.segment(x, Params(nperm=200))[0]) >= 1


def test_segment_without_params_is_refused(api):
    lib, ctx = api
    x = step_vector(100, 3)
    lengths, means = np.zeros(100, np.int32), np.zeros(100)
    nseg, draws = C.c_int32(0), C.c_uint64(0)
    rc = lib.cbs_gpu_segment(ctx.h, dp(x), len(x), None, None, 100, lengths.ctypes.data_as(I32P), dp(means), C.byref(nseg),
                             C.byref(draws))
    assert rc == ERR_INVALID
    assert lib.cbs_gpu_last_error(ctx.h).decode() == "bad arguments"


@pytest.mark.parametrize("rng_mode,chain", [(RNG_MT19937_64, True), (RNG_MT19937_64, False), (RNG_PHILOX, False)])
def test_one_unit_batches_equal_single_vector_calls(api, rng_mode, chain):
    _, ctx = api
    x = step_vector(20000, 4)
    w = np.random.default_rng(5).uniform(0.5, 2.0, len(x))
    p = Params(nperm=1000, rng_mode=rng_mode, chain=chain, seed=7, do_smooth=False)
    off = np.array([0, len(x)], np.int64)

    lengths, means, draws = ctx.segment(x, p)
    b = ctx.segment_batch(x, off, p)
    assert len(lengths) > 1
    assert np.array_equal(b.lengths, lengths) and np.array_equal(b.means, means) and int(b.draws[0]) == draws

    lengths, means, draws = ctx.segment_weighted(x, w, p)
    b = ctx.segment_weighted_batch(x, w, off, p)
    assert len(lengths) > 1
    assert np.array_equal(b.lengths, lengths) and np.array_equal(b.means, means) and int(b.draws[0]) == draws
