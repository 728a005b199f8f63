"""-m gpu: the low-level call surface of lib/cbs (CBS.hpp:29-98) through the C ABI against the COMPILED reference (oracle/_ref):
fndcpt, wfindcpt, tpermp, xperm, wxperm, htmaxp, wtmaxo, tailp, and the binary-data variants tmaxo/tmaxp(ibin=true), btmax,
btailp.  Integer results and the engine position are identical; floating point results are bit-identical except where the
device evaluates erfc/log/exp/pow (tailp, btailp, hybrid p-values): there the tolerance is written in the test."""
import numpy as np
import pytest

from helpers import equal_arrays, f32, make_unit
from genomic_b200 import Params, RNG_MT19937_64

pytestmark = pytest.mark.gpu


def centred(x):
    cur = x - np.cumsum(x)[-1] / len(x)          # CBS.cpp:986-988, sequential sums
    return cur, float(np.cumsum(cur * cur)[-1])


def test_kat_binary_tmaxo(ctx, ref):
    # tests/cbs_test.cpp:163-175: case1 with ibin=true -> [0,58], statistic > 10 (the compiled reference gives 900.259...)
    x = np.array([0.0] * 20 + [1.5] * 20 + [0.0] * 20)
    tss = float((x * x).sum() - x.sum() ** 2 / len(x))
    got = ctx.tmaxo(x, tss, 2, True)
    assert got == ref.tmaxo(x, tss, 2, True)
    assert (got[1], got[2]) == (0, 58) and got[0] > 10.0 and abs(got[0] - 900.259) < 1e-3


def test_binary_tmaxo_tmaxp_match_reference(ctx, ref):
    rng = np.random.default_rng(71)
    for trial in range(60):
        n = int(rng.integers(4, 3000))
        kind = trial % 4
        if kind == 0:
            x = rng.integers(0, 2, n).astype(float)                       # binary data, what ibin is for
        elif kind == 1:
            x = (rng.random(n) < 0.2).astype(float); x[n // 3: n // 2] = (rng.random(n // 2 - n // 3) < 0.7)
        else:
            x = make_unit(rng, n, trial % 5)
        xc, tss = centred(x)
        for al0 in (2, 3):
            if n < 2 * al0:
                continue
            assert ctx.tmaxo(xc, tss, al0, True) == ref.tmaxo(xc, tss, al0, True), (trial, n, al0)
        m = np.stack([rng.permutation(xc) for _ in range(5)])
        assert np.array_equal(ctx.tmaxp(m, tss, 2, True), np.array([ref.tmaxp(r, tss, 2, True) for r in m])), (trial, n)
    n = 60000
    x = (rng.random(n) < 0.3).astype(float); x[20000:26000] = (rng.random(6000) < 0.36)
    xc, tss = centred(x)
    assert ctx.tmaxo(xc, tss, 2, True) == ref.tmaxo(xc, tss, 2, True)


def test_btmax_btailp(ctx, ref):
    rng = np.random.default_rng(72)
    for n in (5, 40, 1000, 20000):
        x = rng.normal(0, 1, n)
        assert ctx.btmax(x) == ref.btmax(x)
    for b, m, ng in ((3.0, 200, 50), (4.5, 5000, 100), (2.2, 37, 10)):
        got, want = ctx.btailp(b, m, ng), ref.btailp(b, m, ng)
        assert abs(got - want) <= 1e-12 * abs(want), (b, m, ng, got, want)  # CUDA erfc/log/exp vs libm


def test_tailp(ctx, ref):
    for b, delta, m in ((3.5, 26 / 5000, 5000), (5.0, 26 / 150000, 150000), (0.05, 0.1, 300), (7.5, 0.01, 2000)):
        got, want = ctx.tailp(b, delta, m), ref.tailp(b, delta, m)
        assert abs(got - want) <= 1e-12 * abs(want), (b, delta, m, got, want)  # CUDA erfc/log/exp/pow vs libm


def test_xperm_wxperm_match_reference(ctx, ref):
    rng = np.random.default_rng(73)
    for n in (1, 2, 37, 2049, 9000, 30000, 70000, 147726):   # every shuffle class, incl. the cluster kernels
        x = rng.normal(0, 1, n)
        for seed in (1, 99):
            r = ref.rng(seed)
            want = ref.xperm(x, r)
            assert equal_arrays(ctx.xperm(x, seed=seed), want), (n, seed)
            assert ref.rng_equals(r, seed, n)
        if n >= 2:
            rw = np.sqrt(rng.uniform(0.5, 2.0, n))
            assert equal_arrays(ctx.xperm(x, seed=5, rwts=rw), ref.wxperm(x, rw, ref.rng(5))), n


def test_htmaxp_matches_reference(ctx, ref):
    rng = np.random.default_rng(74)
    for n in (60, 201, 1000, 5000):
        for k in (5, 25):
            if n <= 2 * k:
                continue
            m = np.stack([f32(rng.normal(0, 0.2, n)) for _ in range(12)])
            m -= m.mean(axis=1, keepdims=True)
            tss = float((m[0] * m[0]).sum())
            assert np.array_equal(ctx.htmaxp(m, tss, k, 2), np.array([ref.htmaxp(r, tss, k, 2) for r in m])), (n, k)


def test_tpermp_matches_reference(ctx, ref):
    rng = np.random.default_rng(75)
    for trial in range(14):
        n1, n2 = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        if trial == 0:
            n1, n2 = 1, 50          # p = 1 shortcut (CBS.cpp:499)
        if trial == 1:
            n1, n2 = 3000, 120      # m1 > 64: the general edge kernel
        x = rng.normal(0, 0.2, n1 + n2)
        x[:n1] += float(rng.choice([0.0, 0.05, 0.3, 2.0]))   # 2.0: the tstat > 25 shortcut (CBS.cpp:522)
        nperm = int(rng.choice([50, 500]))
        r = ref.rng(7)
        want = ref.tpermp(n1, n2, x, nperm, r)
        got, draws = ctx.tpermp(n1, n2, x, Params(nperm=nperm, seed=7))
        assert got == want, (trial, n1, n2, got, want)
        assert ref.rng_equals(r, 7, draws)


@pytest.mark.parametrize("hybrid", [False, True])
def test_fndcpt_matches_reference(ctx, ref, hybrid):
    rng = np.random.default_rng(76 + int(hybrid))
    for trial in range(16):
        n = int(rng.integers(60 if hybrid else 8, 2500))
        xc, tss = centred(make_unit(rng, n, trial % 5))
        if float(np.ptp(xc)) == 0.0:
            continue
        nperm, alpha = int(rng.choice([100, 1000])), float(rng.choice([0.01, 0.05]))
        r = ref.rng(3)
        want = ref.fndcpt(xc, tss, nperm, alpha, r, hybrid=hybrid, al0=2, hk=25, delta=26.0 / n)
        got = ctx.fndcpt(xc, tss, Params(alpha=alpha, nperm=nperm, hybrid=hybrid, min_width=2, kmax=25, seed=3), delta=26.0 / n)
        assert (got["ncpt"], got["iseg"]) == (want["ncpt"], want["iseg"]), (trial, n, got, want)
        assert got["ostat"] == want["ostat"]
        if want["ncpt"] >= 1:
            assert got["icpt"][0] == want["icpt"][0]
        if want["ncpt"] == 2:
            assert got["icpt"][1] == want["icpt"][1]
        assert ref.rng_equals(r, 3, got["draws"]), (trial, n)   # the caller's engine ends where the reference's does


def test_wtmaxo_kat_and_reference(ctx, ref):
    # tests/cbs_test.cpp:179-203: case2 -> [0,58] (al0=2), [0,57] (al0=3)
    x = np.array([0.0] * 15 + [2.0] * 15 + [-1.5] * 15 + [0.0] * 15)
    w = np.array([1.0] * 15 + [0.5] * 15 + [2.0] * 15 + [1.0] * 15)
    tss = float((w * x * x).sum() - (w * x).sum() ** 2 / w.sum())
    for al0, loc in ((2, (0, 58)), (3, (0, 57))):
        got = ctx.wtmaxo(x, w, tss, al0)
        assert got == ref.wtmaxo(x, w, tss, al0)
        assert (got[1], got[2]) == loc
    rng = np.random.default_rng(77)
    for trial in range(25):
        n = int(rng.integers(8, 4000))
        x = make_unit(rng, n, trial % 5)
        w = rng.uniform(0.5, 2.0, n)
        xc = x - (w * x).sum() / w.sum()
        tss = float((w * xc * xc).sum())
        assert ctx.wtmaxo(xc, w, tss, 2) == ref.wtmaxo(xc, w, tss, 2), (trial, n)


def test_wfindcpt_matches_reference(ctx, ref):
    rng = np.random.default_rng(78)
    for trial in range(12):
        n = int(rng.integers(8, 2500))
        x = make_unit(rng, n, trial % 5)
        if float(np.ptp(x)) == 0.0:
            continue
        w = rng.uniform(0.5, 2.0, n)
        # centring and weighted tss exactly as cbs::segment_weighted (CBS.cpp:1053-1066): sequential sums
        wsum = float(np.cumsum(w)[-1]); wxsum = float(np.cumsum(w * x)[-1])
        xc = x - wxsum / wsum
        tss = float(np.cumsum(w * xc * xc)[-1])
        nperm, alpha = int(rng.choice([100, 1000])), float(rng.choice([0.01, 0.05]))
        r = ref.rng(4)
        want = ref.wfindcpt(xc, w, tss, nperm, alpha, r)
        got = ctx.wfindcpt(xc, w, tss, Params(alpha=alpha, nperm=nperm, min_width=2, seed=4))
        assert (got["ncpt"], got["iseg"], got["ostat"]) == (want["ncpt"], want["iseg"], want["ostat"]), (trial, n, got, want)
        if want["ncpt"] >= 1:
            assert got["icpt"][0] == want["icpt"][0]
        if want["ncpt"] == 2:
            assert got["icpt"][1] == want["icpt"][1]
        assert ref.rng_equals(r, 4, got["draws"]), (trial, n)


def structured_vectors():
    for n in (400, 900, 1600, 2500, 10000):
        b = int(round(np.sqrt(n)))
        yield n, "alt", np.tile([1.0, -1.0], n // 2)
        yield n, "saw4", np.tile([1.0, 1.0, -1.0, -1.0], n // 4)
        yield n, "saw10", np.tile([1.0] * 5 + [-1.0] * 5, n // 10)
        yield n, "blocks", np.tile([1.0] * (b // 2) + [-1.0] * (b - b // 2), n // b + 1)[:n]
        yield n, "steps3", np.tile([2.0, -1.0, -1.0], n // 3 + 1)[:n]


def test_tied_maxima_follow_the_references_visiting_order(ctx, ref):
    """Periodic / piecewise constant vectors: many block pairs have EQUAL corner statistics and the maximum is attained by
    many arcs, so the reported arc is decided by the reference's visiting order, including where std::sort (not stable
    beyond 16 elements) leaves equal keys.  Unweighted: the scan's canonical-order key; weighted: a tie between pairs with
    equal corner statistics is detected and the location is taken from a walk in the reference's own order (wtmaxo_ordered).
    Round 1 documented both as known gaps without a test."""
    checked = 0
    for n, name, x in structured_vectors():
        for raw in (True, False):
            xc, tss = (x, float((x * x).sum())) if raw else centred(x)
            for al0 in (2, 3):
                assert ctx.tmaxo(xc, tss, al0) == ref.tmaxo(xc, tss, al0), (n, name, raw, al0)
                w = np.ones(n) if al0 == 2 else np.tile([1.0, 2.0], n // 2 + 1)[:n]
                assert ctx.wtmaxo(xc, w, tss, al0) == ref.wtmaxo(xc, w, tss, al0), (n, name, raw, al0)
                checked += 2
    assert checked == 200


def test_segment_structured_inputs_match_reference(ctx, ref):
    """cbs::segment / cbs::segment_weighted on tie-heavy vectors (constant stretches with exact steps, periodic signals)."""
    from oracle.pyoracle import SegParams
    rng = np.random.default_rng(79)
    for trial in range(10):
        n = int(rng.choice([400, 900, 1600]))
        x = np.tile([1.0] * 5 + [-1.0] * 5, n // 10 + 1)[:n] * float(rng.choice([0.01, 1.0]))
        a = int(rng.integers(50, n // 2)); b = int(rng.integers(a + 40, n - 20))
        x[a:b] += float(rng.choice([0.0, 2.0, 4.0]))
        p = SegParams(nperm=200, alpha=0.01, do_smooth=False, seed=trial + 1)
        gp = Params(nperm=200, alpha=0.01, do_smooth=False, seed=trial + 1)
        wl, wm = ref.segment(x, p)
        gl, gm, _ = ctx.segment(x, gp)
        assert np.array_equal(gl, wl) and np.array_equal(gm, wm), (trial, n)
        w = np.tile([1.0, 2.0, 0.5], n // 3 + 1)[:n]
        wl, wm = ref.segment_weighted(x, w, p)
        gl, gm, _ = ctx.segment_weighted(x, w, gp)
        assert np.array_equal(gl, wl) and np.array_equal(gm, wm), (trial, n, "weighted")
