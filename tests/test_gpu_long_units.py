"""-m gpu: units longer than 1,000,000 markers, up to CBS_GPU_MAX_UNIT = 2^23 = 8,388,608 markers.

Segments that no thread-block cluster holds (more than ~432 000 markers) are shuffled by k_perm; the scan's extrema table
is coarsened up to 1024 prefix sums per entry, and its queued units keep rows and arc lengths of up to 2^23 (a unit code
of 15 row bits wrapped rows at 2^20 before).  Everything is compared with the oracle bit for bit: single permutations
(engine position included), observed scans with maxima past row 2^20 and arcs longer than 2^20, and batches whose
decisions are matched one by one through the split log."""
import os
import subprocess

import numpy as np
import pytest

from helpers import engine_after, f32, pack
from oracle.pyoracle import SegParams
from genomic_b200 import Params, RNG_MT19937_64, RNG_PHILOX
from genomic_b200.binding import CbsGpuError, ERR_UNSUPPORTED

pytestmark = pytest.mark.gpu

MAX_UNIT = 8388608  # CBS_GPU_MAX_UNIT (include/cbs_gpu.h)
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "genomic_b200", "cna_segment_gpu")


def gparams(p: SegParams, **kw) -> Params:
    return Params(alpha=p.alpha, nperm=p.nperm, hybrid=p.hybrid, min_width=p.min_width, kmax=p.kmax, nmin=p.nmin,
                  ibin=p.ibin, do_smooth=p.do_smooth, rng_mode=RNG_PHILOX if p.rng_kind else RNG_MT19937_64,
                  chain=p.chain, seed=p.seed, **kw)


def centred(x):
    xc = x - x.mean()
    return xc, float((xc * xc).sum())


def long_unit(rng, n):
    """noise with steps of several sizes and lengths, weak shifts at both ends and weak arcs inside short segments:
    decisions of every kind, edge tests with 0 < p < 1"""
    x = rng.normal(0, 0.2, n)
    x[n // 3: n // 2] += 0.3
    x[:4000] += 0.048
    x[n - 4000:] -= 0.048
    x[(3 * n) // 4: (3 * n) // 4 + 30000] += 0.012
    x[(5 * n) // 6: (5 * n) // 6 + 8000] -= 0.024
    a = (9 * n) // 10
    x[a: a + 1500] += 0.5
    x[a + 600: a + 900] += 0.12
    b = (2 * n) // 10
    x[b: b + 3000] -= 0.4
    x[b + 1000: b + 2000] -= 0.06
    return f32(x)


@pytest.mark.parametrize("n", [440000, 1048577, 4000000, MAX_UNIT])  # 440 000: past the 8-CTA cluster (~432 100)
def test_xperm_wxperm(ctx, oracle, n):
    rng = np.random.default_rng(n)
    x = f32(rng.normal(0, 1, n))
    eng, nxt = engine_after(oracle, 11, 777)
    want = oracle.xperm(x, eng)
    assert np.array_equal(ctx.xperm(x, mt_next312=nxt), want)
    w = rng.uniform(0.2, 5.0, n)
    eng, nxt = engine_after(oracle, 12, 31)
    want = oracle.wxperm(x, w, eng)
    assert np.array_equal(ctx.xperm(x, mt_next312=nxt, rwts=np.sqrt(w)), want)


@pytest.mark.parametrize("n", [1200000, 2500000])
def test_tmaxo_tmaxp(ctx, oracle, n):
    """null vectors, a weak short arc past row 2^20 (not a block corner), and a weak arc longer than 2^20"""
    rng = np.random.default_rng(n)
    null = f32(rng.normal(0, 0.2, n))
    late = null.copy()
    late[n - 90007: n - 89300] += 0.12
    wide = null.copy()
    wide[n // 10: n // 10 + 1100003] += 0.004
    for name, x in (("null", null), ("late", late), ("wide", wide)):
        xc, tss = centred(x)
        want = oracle.tmaxo(xc, tss, 2)
        assert ctx.tmaxo(xc, tss, 2) == want, (n, name)
        assert ctx.tmaxp(xc, tss, 2) == oracle.tmaxp(xc, tss, 2), (n, name)
        if name == "late":
            assert want[1] >= 1 << 20, want  # the maximum starts past row 2^20


def test_tmaxo_longest_unit(ctx, oracle):
    x = f32(np.random.default_rng(23).normal(0, 0.2, MAX_UNIT))
    xc, tss = centred(x)
    assert ctx.tmaxo(xc, tss, 2) == oracle.tmaxo(xc, tss, 2)


def check_log(got, want, p, long_unit_id):
    """every logged decision equals the oracle's, matched by (unit, lo, hi); returns, for the long unit, the number of
    edge tests that ended with 0 < p < 1 and of max-t tests that ran to the end with 0 < nrej"""
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    if p.hybrid:  # the hybrid means are compared as in the other hybrid tests
        assert np.allclose(got.means, want["means"], rtol=1e-9, atol=0)
    else:
        assert np.array_equal(got.means, want["means"])
    if not p.rng_kind:
        assert np.array_equal(got.draws, want["draws"])
    assert len(got.splits) == len(want["log"])
    by_key = {(g["unit"], g["lo"], g["hi"]): g for g in got.splits}
    edge_mid = nrej_mid = 0
    for u, w in want["log"]:
        key = (u, w.lo, w.hi)
        g = by_key[key]
        assert (g["called"], g["ncpt"]) == (w.called, w.ncpt), key
        if not w.called:
            continue
        assert g["ostat"] == w.ostat, key
        assert (g["iseg0"], g["iseg1"], g["perms_run"], g["nrej"], g["exit_code"]) == \
            (w.iseg0, w.iseg1, w.perms_run, w.nrej, w.exit_code), key
        assert (g["icpt0"], g["icpt1"])[:w.ncpt] == (w.icpt0, w.icpt1)[:w.ncpt], key
        for s, (st, nr, wp) in enumerate(((g["e_status0"], g["e_nrej0"], w.edge_p0), (g["e_status1"], g["e_nrej1"], w.edge_p1))):
            if wp >= 0:
                gp = 1.0 if st == 1 else 0.0 if st == 2 else nr / p.nperm
                assert gp == wp, (key, s)
        if u == long_unit_id:
            edge_mid += int(0.0 < w.edge_p0 < 1.0) + int(0.0 < w.edge_p1 < 1.0)
            nrej_mid += int(w.exit_code != 3 and 0 < w.nrej)
    return edge_mid, nrej_mid


def mixed_batch(seed, n):
    rng = np.random.default_rng(seed)
    head = f32(rng.normal(0, 0.2, 3000))
    head[1000:1400] += 0.4
    return pack([head, long_unit(rng, n), f32(rng.normal(0, 0.2, 700))])


@pytest.mark.parametrize("mode", ["mt_unit", "philox"])
def test_batch_with_a_2_5m_unit(ctx, oracle, mode):
    vals, off = mixed_batch(3, 2500000)
    p = SegParams(nperm=40, alpha=0.05, do_smooth=False, rng_kind=1 if mode == "philox" else 0, chain=False, seed=3)
    want = oracle.segment_units(vals, off, np.ones(3, np.int32), p, want_log=True)
    got = ctx.segment_batch(vals, off, gparams(p, record_splits=True))
    edge_mid, nrej_mid = check_log(got, want, p, 1)
    assert nrej_mid >= 1, (edge_mid, nrej_mid)  # a max-t test of the long unit ran all 40 permutations with 0 < nrej


def test_mt_chain_1_2m(ctx, oracle):
    vals, off = mixed_batch(5, 1200000)
    p = SegParams(nperm=100, alpha=0.05, do_smooth=True, rng_kind=0, chain=True, seed=5)
    want = oracle.segment_units(vals, off, np.ones(3, np.int32), p, want_log=True)
    got = ctx.segment_batch(vals, off, gparams(p, record_splits=True))
    check_log(got, want, p, 1)


def test_units_between_cluster_and_1m(ctx, oracle):
    """430 000 - 1 000 000 markers: the longest segments are beyond every cluster class"""
    rng = np.random.default_rng(8)
    vals, off = pack([long_unit(rng, 700000), long_unit(rng, 450000), f32(rng.normal(0, 0.2, 5000))])
    p = SegParams(nperm=200, alpha=0.01, do_smooth=False, rng_kind=0, chain=False, seed=8)
    want = oracle.segment_units(vals, off, np.ones(3, np.int32), p, want_log=True)
    check_log(ctx.segment_batch(vals, off, gparams(p, record_splits=True)), want, p, 0)


def test_hybrid_1_2m(ctx, oracle):
    vals, off = mixed_batch(6, 1200000)
    p = SegParams(nperm=100, alpha=0.05, do_smooth=False, rng_kind=0, chain=False, seed=6, hybrid=True)
    want = oracle.segment_units(vals, off, np.ones(3, np.int32), p, want_log=True)
    check_log(ctx.segment_batch(vals, off, gparams(p, record_splits=True)), want, p, 1)


def test_binary_1_1m(ctx, oracle):
    rng = np.random.default_rng(9)
    n = 1100000
    prob = np.full(n, 0.3)
    prob[n // 5: n // 2] = 0.6
    prob[(3 * n) // 4: (3 * n) // 4 + 2000] = 0.9
    x = (rng.random(n) < prob).astype(np.float64)
    vals, off = pack([x, (rng.random(4000) < 0.5).astype(np.float64)])
    p = SegParams(nperm=50, alpha=0.05, do_smooth=False, rng_kind=1, chain=False, seed=9, ibin=True)
    want = oracle.segment_units(vals, off, np.ones(2, np.int32), p, want_log=True)
    check_log(ctx.segment_batch(vals, off, gparams(p, record_splits=True)), want, p, 0)


def test_weighted_1_2m(ctx, oracle):
    vals, off = mixed_batch(10, 1200000)
    w = np.random.default_rng(10).uniform(0.5, 2.0, len(vals))
    p = SegParams(nperm=60, alpha=0.05, do_smooth=False, rng_kind=0, chain=False, seed=10)
    want = oracle.segment_weighted_units(vals, w, off, p, want_log=True)
    check_log(ctx.segment_weighted_batch(vals, w, off, gparams(p, record_splits=True)), want, p, 1)


def test_driver_on_a_1_5m_row_chromosome(ctx, tmp_path):
    """cna_segment_gpu on a .cn file: its .seg rows are what the Python batched call gives for the same values"""
    from cnio import cohort_from_cn, seg_text
    rng = np.random.default_rng(12)
    sizes = {1: 1500000, 2: 20000}
    rows = ["marker\tchromosome\tposition\ts1"]
    for c, m in sizes.items():
        a = rng.normal(0, 0.2, m)
        a[m // 3: m // 2] += 0.4
        a[(3 * m) // 4] += 4.0
        pos = 100 * (np.arange(m) + 1)
        rows.extend(f"m{c}_{k}\tchr{c}\t{pos[k]}\t{a[k]:.4f}" for k in range(m))
    cn = tmp_path / "in.cn"
    cn.write_text("\n".join(rows) + "\n")
    out = tmp_path / "out.seg"
    assert subprocess.run([DRIVER, str(cn), str(out), "--nperm", "200"]).returncode == 0
    names, positions, _, values, off, lab, units = cohort_from_cn(str(cn))
    got = ctx.segment_batch(values, off, Params(nperm=200, chain=True, do_smooth=True))
    assert out.read_text() == seg_text(names, positions, units, got.seg_count, got.lengths, got.means)


def test_longer_units_are_rejected(ctx):
    x = np.zeros(MAX_UNIT + 1)
    calls = [lambda: ctx.tmaxo(x, 1.0, 2), lambda: ctx.xperm(x, seed=1),
             lambda: ctx.segment_batch(x, np.array([0, MAX_UNIT + 1]), Params(do_smooth=False))]
    for call in calls:
        with pytest.raises(CbsGpuError) as e:
            call()
        assert e.value.code == ERR_UNSUPPORTED and "8,388,608" in str(e.value)
