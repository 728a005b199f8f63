"""-m gpu: the option ranges `cna segment` accepts beyond the device's fixed-size paths, bit for bit against the C oracle.

Smoothing windows wider than 64 markers (smooth_region > SM_MAX_REGION: k_sm_run_mark / k_sm_run_end, k_sm_wide,
k_sm_median in smooth.cuh) and hybrid kmax above 128 (k_hscan<true> with its length tiles and htmaxp_one_block_cta in
kernels.cuh; the weighted k_whscan / k_wdelta, which have no fixed-size table).  The narrow paths (k_sm_window,
k_hscan<false>) are covered by test_gpu_parity.py, test_gpu_fullsize.py and test_gpu_hybrid.py."""
import os
import subprocess

import numpy as np
import pytest

from helpers import check_split_log, engine_after, f32, gparams, pack, weighted_centre
from oracle.pyoracle import SegParams
from test_gpu_hybrid import Tally, centred, decision_input, htmaxp_rows, long_unit, short_unit
from test_gpu_weighted_decisions import check_weighted_log, segment_mix
from genomic_b200 import CbsGpuError, Params
from genomic_b200.binding import ERR_UNSUPPORTED

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
DRIVER = os.path.join(os.path.dirname(HERE), "genomic_b200", "cna_segment_gpu")
REGIONS = (64, 65, 100, 257, 1000, 5000, 10 ** 6, 2 ** 31 - 1)


# ---- smoothing -----------------------------------------------------------------------------------------------------------
def noisy(rng, n, spikes=True, nonfinite=False):
    """noise, rare outliers of several sizes (isolated ones get a median, clustered ones are kept), optional NaN/inf"""
    x = rng.normal(0, 0.2, n)
    if spikes:
        i = rng.integers(0, n, max(1, n // 700))
        x[i] += rng.choice([-1.0, 1.0], len(i)) * (2.0 + np.abs(rng.normal(0, 3.0, len(i))))
    x = f32(x)
    if nonfinite:
        i = rng.integers(0, n, max(1, n // 100))
        x[i] = rng.choice([np.nan, np.inf, -np.inf], len(i))
    return x


def labels(rng, n, layout, region):
    if layout == "single":
        return np.full(n, 3, np.int32)
    if layout == "chroms":
        cuts = np.sort(rng.choice(np.arange(1, n), 2, replace=False))
        return np.repeat(np.array([1, 2, 7], np.int32), np.diff(np.concatenate([[0], cuts, [n]])))
    # many short runs: one-marker runs and runs shorter than the window; a label may come back after another
    lens = []
    while sum(lens) < n:
        lens.append(int(rng.choice([1, 1, 2, 3, int(rng.integers(1, max(2, min(region, 3000))))])))
    lab = np.repeat(rng.integers(1, 5, len(lens)).astype(np.int32), lens)[:n]
    return lab


def check_smooth(ctx, oracle, x, lab, region, **kw):
    got = ctx.smooth(x, lab, region, **kw)
    want = oracle.smooth(x, lab, region, **kw)
    assert np.array_equal(got, want, equal_nan=True), (region, np.flatnonzero(~((got == want) | np.isnan(want)))[:5])
    fin = np.isfinite(x)
    return int(np.count_nonzero(want[fin] != x[fin]))  # markers the median branch replaced


@pytest.mark.parametrize("region", REGIONS)
def test_smooth_wide_windows(ctx, oracle, region):
    """ctx.smooth against orc_smooth at n up to 200 000: one label, three chromosome runs, many short runs; with and
    without non-finite values.  The median branch must have fired."""
    rng = np.random.default_rng(2100 + region % 1000)
    changed = 0
    for n in (3000, 200000):
        for layout in ("single", "chroms", "runs"):
            for nonfinite in (False, True):
                x = noisy(rng, n, nonfinite=nonfinite)
                changed += check_smooth(ctx, oracle, x, labels(rng, n, layout, region), region)
    assert changed >= 20, changed


def test_smooth_wide_long_unit(ctx, oracle):
    """one unit of 2.5 M markers: windows in shared memory (R = 1000) and in global memory (R = 10^6)"""
    rng = np.random.default_rng(2201)
    n = 2_500_000
    x = noisy(rng, n, nonfinite=True)
    lab = np.repeat(np.array([1, 2], np.int32), [1_700_000, n - 1_700_000])
    changed = sum(check_smooth(ctx, oracle, x, lab, r) for r in (1000, 10 ** 6))
    assert changed >= 100, changed


def test_smooth_wide_constant_and_outliers(ctx, oracle):
    """Constant data with a few outliers (sd = 0: oSD = 0 makes above = below = 0 from the start, nothing changes).
    Integer data, mostly 0, with outliers and smooth_sd_scale = 0: outliers become a zero median exactly, whose sign may
    differ from the reference's (-0.0 == 0.0).  Input where every marker is an outlier: alternating +-5 on a slow ramp
    with outlier_sd_scale 1e-6, so that every neighbour is farther than oSD and every window is scanned to its ends."""
    rng = np.random.default_rng(2301)
    for region in (65, 100, 5000, 2 ** 31 - 1):
        for c in (0.0, 1.5):
            x = np.full(20000, c)
            x[rng.integers(0, 20000, 15)] = rng.choice([-3.0, 4.0], 15)
            for layout in ("single", "runs"):
                assert check_smooth(ctx, oracle, x, labels(rng, 20000, layout, region), region) == 0
        x = rng.choice([-1.0, 0.0, 0.0, 0.0, 1.0], 20000)
        x[rng.choice(20000, 3, replace=False)] = (9.0, -15.0, 25.0)  # farther than oSD from each other
        assert check_smooth(ctx, oracle, x, labels(rng, 20000, "single", region), region, smooth_sd_scale=0.0) > 0
    n = 20000
    alt = f32(np.where(np.arange(n) % 2 == 0, 5.0, -5.0) + 1e-3 * np.arange(n))
    for region in (65, 1000, 10 ** 6):
        for layout in ("single", "runs"):
            changed = check_smooth(ctx, oracle, alt, labels(rng, n, layout, region), region, outlier_sd_scale=1e-6)
            assert changed > 0, (region, layout)


def test_smooth_region_refusals(ctx):
    """smooth_region < 0 stays an error (std::invalid_argument in the reference: ValueError here)"""
    x = np.zeros(100)
    with pytest.raises(ValueError, match="smooth_region must be non-negative"):
        ctx.smooth(x, np.ones(100, np.int32), -1)
    with pytest.raises(ValueError, match="smooth_region must be non-negative"):
        ctx.segment_batch(x, np.array([0, 100]), Params(smooth_region=-1))


@pytest.mark.parametrize("mode", ["mt_chain", "mt_unit", "philox"])
def test_segment_batch_smooth_region_100(ctx, oracle, mode):
    """segment_batch with do_smooth and R = 100 (each unit one label) against orc_segment_units"""
    rng = np.random.default_rng(2401 + len(mode))
    units = [noisy(rng, int(n)) for n in rng.integers(50, 20000, 12)] + [noisy(rng, 150000)]
    for u in units[:6]:
        u[len(u) // 3: len(u) // 2] += 0.5
    vals, off = pack(units)
    p = SegParams(nperm=500, alpha=0.01, do_smooth=True, smooth_region=100, rng_kind=1 if mode == "philox" else 0,
                  chain=(mode == "mt_chain"), seed=5)
    want = oracle.segment_units(vals, off, np.ones(len(units), np.int32), p)
    got = ctx.segment_batch(vals, off, gparams(p))
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    assert np.array_equal(got.means, want["means"])
    if mode != "philox":
        assert np.array_equal(got.draws, want["draws"])


def test_cli_smooth_region_100(ctx, tmp_path):
    """cna_segment_gpu --smooth_region 100 on a generated .cn file equals the Python batched call"""
    from cnio import cohort_from_cn, seg_text
    rng = np.random.default_rng(2501)
    n = {1: 3000, 2: 1800, 23: 900}
    rows = ["marker\tchromosome\tposition\ts1\ts2"]
    for c, m in n.items():
        a, b = noisy(rng, m), noisy(rng, m)
        a[m // 3: m // 2] += 0.6
        b[m // 2:] -= 0.5
        name = "chrX" if c == 23 else f"chr{c}"
        for k in range(m):
            rows.append(f"m{c}_{k}\t{name}\t{1000 * (k + 1)}\t{a[k]:.4f}\t{b[k]:.4f}")
    cn = tmp_path / "in.cn"
    cn.write_text("\n".join(rows) + "\n")
    out = tmp_path / "out.seg"
    assert subprocess.run([DRIVER, str(cn), str(out), "--nperm", "500", "--smooth_region", "100"]).returncode == 0
    names, positions, _, values, off, lab, units = cohort_from_cn(str(cn))
    got = ctx.segment_batch(values, off, Params(nperm=500, smooth_region=100))
    assert out.read_text() == seg_text(names, positions, units, got.seg_count, got.lengths, got.means)


# ---- hybrid kmax > 128 ---------------------------------------------------------------------------------------------------
WIDE_KMAXES = (129, 130, 200, 256, 500, 1000, 4096)


@pytest.mark.parametrize("k", WIDE_KMAXES)
def test_htmaxp_wide_bit_exact(ctx, oracle, k):
    """k_hscan<true> against orc_htmaxp, al0 1/2/3/5: n in [k, 2k) (htmaxp_one_block_cta) and from 2k to 147 726"""
    rng = np.random.default_rng(2600 + k)
    ns = sorted({k, k + 1, 2 * k - 1, 2 * k, 2 * k + 1, 3 * k, 10 * k + 7, 50000, 147726})
    for al0 in (1, 2, 3, 5):
        for n in ns:
            m = htmaxp_rows(rng, n, k, 12 if n <= 3 * k else 6 if n < 50000 else 3)
            tss = float((m[0] * m[0]).sum())
            got = ctx.htmaxp(m, tss, k, al0)
            want = np.array([oracle.htmaxp(r, tss, k, al0) for r in m])
            bad = np.flatnonzero(got != want)
            assert not len(bad), (k, al0, n, bad[:5], got[bad[:3]], want[bad[:3]])


def test_htmaxp_wide_1m_row(ctx, oracle):
    rng = np.random.default_rng(2701)
    n, k = 1_000_003, 500
    m = htmaxp_rows(rng, n, k, 2)
    tss = float((m[0] * m[0]).sum())
    for al0 in (2, 5):
        assert np.array_equal(ctx.htmaxp(m, tss, k, al0), np.array([oracle.htmaxp(r, tss, k, al0) for r in m])), al0


def test_fndcpt_hybrid_wide(ctx, oracle):
    """cbs_gpu_fndcpt(hybrid) at kmax 129/200/500 with a caller-owned engine already in use, n from kmax to 20 000"""
    rng = np.random.default_rng(2801)
    tally, refused = Tally(), 0
    for kmax in (129, 200, 500):
        for n in sorted({kmax - 1, kmax, kmax + 1, kmax + 2, 2 * kmax - 1, 2 * kmax, 2 * kmax + 1, 3000, 20000}):
            for kind in ("spike", "weak", "step", "null"):
                al0 = int(rng.choice([1, 2, 3, 5]))
                xc, tss = centred(decision_input(rng, kind, n))
                nperm = int(rng.choice([100, 300]))
                alpha = float(rng.choice([0.01, 0.05]))
                p = Params(alpha=alpha, nperm=nperm, min_width=al0, hybrid=True, kmax=kmax, seed=9)
                eng, nxt = engine_after(oracle, 9, int(rng.integers(0, 3000)))
                msg = (kmax, n, kind, al0)
                delta = (kmax + 1) / n
                if n < kmax or delta >= 1.0:
                    with pytest.raises(CbsGpuError) as e:
                        ctx.fndcpt(xc, tss, p, mt_next312=nxt)
                    assert e.value.code == ERR_UNSUPPORTED and "hybrid fndcpt needs n >= hk and delta < 1" in str(e.value), msg
                    refused += 1
                    continue
                d0 = eng.draws
                want = oracle.fndcpt(xc, tss, nperm, alpha, eng, hybrid=True, al0=al0, hk=kmax, delta=delta)
                got = ctx.fndcpt(xc, tss, p, mt_next312=nxt)
                assert got["ostat"] == want.ostat and got["iseg"] == tuple(want.iseg), msg
                assert (got["ncpt"], got["perms_run"], got["nrej"], got["exit_code"]) == \
                    (want.ncpt, want.perms_run, want.nrej, want.exit_code), msg
                assert got["icpt"][:want.ncpt] == tuple(want.icpt)[:want.ncpt], msg
                assert got["draws"] == eng.draws - d0, msg
                tally.hybrid_decision(ctx, oracle, n, kmax, want.ostat, want.exit_code, want.nrej, want.perms_run, alpha,
                                      nperm, 1e-6, delta, msg)
    tally.report("fndcpt kmax > 128")
    assert tally.short >= 20 and refused >= 6, (tally.short, refused)


# (mode, kmax, nmin, min_width)
WIDE_SPLIT_CONFIGS = [("mt_chain", 129, 130, 2), ("philox", 129, 300, 3), ("mt_unit", 200, 201, 5),
                      ("mt_chain", 200, 450, 2), ("philox", 500, 501, 2), ("mt_unit", 500, 1100, 3)]


def test_split_logs_hybrid_wide(ctx, oracle):
    """split logs at kmax 129/200/500 with nmin = kmax + 1 and nmin > 2 kmax, in MT-chain, MT-unit and Philox modes"""
    rng = np.random.default_rng(2901)
    tally = Tally()
    for mode, kmax, nmin, mw in WIDE_SPLIT_CONFIGS:
        lens = [nmin, nmin + 1, nmin + 2] + [int(v) for v in rng.integers(nmin + 1, max(nmin + 2, 2 * kmax + 1), 6)]
        lens += [int(v) for v in rng.integers(nmin + 1, 6000, 6)]
        units = [short_unit(rng, n) for n in lens]
        units.insert(3, long_unit(rng, int(rng.choice([20000, 61003]))))
        p = SegParams(nperm=int(rng.choice([100, 200])), alpha=float(rng.choice([0.01, 0.05])), hybrid=True, kmax=kmax,
                      nmin=nmin, min_width=mw, do_smooth=False, rng_kind=1 if mode == "philox" else 0,
                      chain=(mode == "mt_chain"), seed=int(rng.integers(1, 100)))
        vals, off = pack(units)
        want = oracle.segment_units(vals, off, np.ones(len(units), np.int32), p, want_log=True)
        got = ctx.segment_batch(vals, off, gparams(p, record_splits=True))
        for u, w, _ in check_split_log(got, want, p, exact_draws=not p.rng_kind):
            n = w.hi - w.lo
            if p.nmin < n:
                tally.hybrid_decision(ctx, oracle, n, p.kmax, w.ostat, w.exit_code, w.nrej, w.perms_run, p.alpha, p.nperm,
                                      p.tol, (p.kmax + 1) / n, (u, w.lo, w.hi))
    tally.report("split logs kmax > 128")
    assert tally.tailp_exit >= 20 and tally.early >= 20 and tally.full_mid >= 5 and tally.short >= 20, vars(tally)


def test_weighted_hybrid_kmax_200(ctx, oracle):
    """k_wdelta / k_wssq / k_whscan at kmax = 200: single wfindcpt calls and a split log against the weighted oracle.
    k_whscan's brute force is hwtmaxp's value for n >= 2 kmax (DESIGN 4a), so hybrid segments start there."""
    rng = np.random.default_rng(3001)
    kmax = 200
    for n in (2 * kmax, 2 * kmax + 1, 450, 3000, 20000):
        for kind in ("spike", "weak", "step", "null"):
            x = decision_input(rng, kind, n)
            w = rng.uniform(0.5, 2.0, n)
            xc, tss = weighted_centre(x, w)
            al0 = int(rng.choice([2, 3]))
            eng, nxt = engine_after(oracle, 9, int(rng.integers(0, 3000)))
            d0 = eng.draws
            want = oracle.wfindcpt(xc, w, tss, 200, 0.05, eng, hybrid=True, al0=al0, hk=kmax)
            got = ctx.wfindcpt(xc, w, tss, Params(alpha=0.05, nperm=200, min_width=al0, hybrid=True, kmax=kmax,
                                                  nmin=kmax + 2, seed=9), mt_next312=nxt)
            msg = (n, kind, al0)
            assert got["ostat"] == want.ostat and got["iseg"] == tuple(want.iseg), msg
            assert (got["ncpt"], got["perms_run"], got["nrej"], got["exit_code"]) == \
                (want.ncpt, want.perms_run, want.nrej, want.exit_code), msg
            assert got["draws"] == eng.draws - d0, msg
    units = [segment_mix(rng, int(n)) for n in rng.integers(kmax + 3, 4000, 10)] + [segment_mix(rng, 30000)]
    vals, off = pack(units)
    w = rng.uniform(0.5, 2.0, len(vals))
    p = SegParams(nperm=200, alpha=0.05, do_smooth=False, rng_kind=0, chain=True, seed=6, hybrid=True, kmax=kmax,
                  nmin=2 * kmax)
    want = oracle.segment_weighted_units(vals, w, off, p, want_log=True)
    got = ctx.segment_weighted_batch(vals, w, off, gparams(p, record_splits=True))
    check_weighted_log(got, want, p, exact_draws=True)


def test_hybrid_wide_refusals(ctx):
    """the refusals where the reference is undefined stay, with their messages, at kmax > 128"""
    rng = np.random.default_rng(3101)
    x = short_unit(rng, 600)
    for kmax, nmin in ((200, 199), (200, 200), (4096, 4000)):
        q = Params(hybrid=True, kmax=kmax, nmin=nmin, do_smooth=False)
        for call in (lambda: ctx.segment(x, q), lambda: ctx.segment_batch(x, np.array([0, 600]), q)):
            with pytest.raises(CbsGpuError) as e:
                call()
            assert e.value.code == ERR_UNSUPPORTED and "hybrid CBS needs nmin >= kmax + 1" in str(e.value), (kmax, nmin)
    with pytest.raises(CbsGpuError) as e:
        ctx.segment_weighted_batch(x, np.ones(600), np.array([0, 600]), Params(hybrid=True, kmax=200, nmin=201, do_smooth=False))
    assert e.value.code == ERR_UNSUPPORTED and "weighted hybrid CBS needs nmin >= kmax + 2" in str(e.value)
    for k in (129, 1000):
        with pytest.raises(CbsGpuError) as e:
            ctx.htmaxp(np.zeros((1, k - 1)) + np.arange(k - 1), 1.0, k, 2)
        assert e.value.code == ERR_UNSUPPORTED, k
    with pytest.raises(CbsGpuError) as e:
        ctx.segment(x, Params(hybrid=True, kmax=0, nmin=200, do_smooth=False))
    assert e.value.code == ERR_UNSUPPORTED


def unsupported(call, msg):
    with pytest.raises(CbsGpuError) as e:
        call()
    assert e.value.code == ERR_UNSUPPORTED and msg in str(e.value), (msg, str(e.value))


def test_hybrid_kmax_int_max_refused(ctx):
    """kmax = 2^31 - 1 with the default nmin: the nmin rules are compared in 64 bits, so kmax + 1 and kmax + 2 cannot wrap
    around, on the unweighted and the weighted entries"""
    rng = np.random.default_rng(3201)
    x = short_unit(rng, 600)
    w = rng.uniform(0.5, 2.0, 600)
    big = 2 ** 31 - 1
    for kmax in (big, big - 1):
        q = Params(hybrid=True, kmax=kmax, do_smooth=False)
        unsupported(lambda: ctx.segment(x, q), "hybrid CBS needs nmin >= kmax + 1")
        unsupported(lambda: ctx.segment_batch(x, np.array([0, 600]), q), "hybrid CBS needs nmin >= kmax + 1")
        unsupported(lambda: ctx.segment_weighted(x, w, q), "weighted hybrid CBS needs nmin >= kmax + 2")
        unsupported(lambda: ctx.segment_weighted_batch(x, w, np.array([0, 600]), q), "weighted hybrid CBS needs nmin >= kmax + 2")
        xc, tss = centred(x)
        unsupported(lambda: ctx.fndcpt(xc, tss, q), "hybrid fndcpt needs n >= hk and delta < 1")
        xw, tssw = weighted_centre(x, w)
        for nmin in (200, big):
            unsupported(lambda: ctx.wfindcpt(xw, w, tssw, Params(hybrid=True, kmax=kmax, nmin=nmin)),
                        "weighted hybrid wfindcpt needs n >= 2*hk")
        unsupported(lambda: ctx.htmaxp(x.reshape(1, -1), 1.0, kmax, 2), "need 1 <= al0 <= k and n >= k")


def test_weighted_hybrid_short_segments_refused(ctx):
    """Weighted hybrid segments of fewer than 2*kmax markers, where k_whscan's all-arcs maximum is not hwtmaxp's value,
    are refused instead of answered differently from the reference: nmin < 2*kmax - 1, and wfindcpt with n < 2*hk.
    nmin = 2*kmax - 1 and n = 2*hk are accepted."""
    rng = np.random.default_rng(3301)
    x = short_unit(rng, 1200)
    w = rng.uniform(0.5, 2.0, 1200)
    for kmax, nmin in ((25, 27), (25, 48), (101, 200), (129, 200), (200, 398)):
        q = Params(hybrid=True, kmax=kmax, nmin=nmin, do_smooth=False)
        unsupported(lambda: ctx.segment_weighted(x, w, q), "weighted hybrid CBS needs nmin >= 2*kmax - 1")
        unsupported(lambda: ctx.segment_weighted_batch(x, w, np.array([0, 1200]), q), "weighted hybrid CBS needs nmin >= 2*kmax - 1")
    for kmax in (25, 200):
        ctx.segment_weighted_batch(x, w, np.array([0, 1200]), Params(hybrid=True, kmax=kmax, nmin=2 * kmax - 1, do_smooth=False))
        for n in (kmax - 1, kmax + 2, 2 * kmax - 1):
            xw, tss = weighted_centre(x[:n], w[:n])
            unsupported(lambda: ctx.wfindcpt(xw, w[:n], tss, Params(hybrid=True, kmax=kmax, nmin=kmax + 2)),
                        "weighted hybrid wfindcpt needs n >= 2*hk")
        xw, tss = weighted_centre(x[:2 * kmax], w[:2 * kmax])
        ctx.wfindcpt(xw, w[:2 * kmax], tss, Params(hybrid=True, kmax=kmax, nmin=kmax + 2))
