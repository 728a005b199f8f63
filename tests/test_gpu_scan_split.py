"""-m gpu: the observed scan spread over several CTAs per row (k_scan_obs, one slice per 8192 markers).  The slices share
the running level and merge their best arcs with the scan's total order on candidates, so the location of a maximum that
several slices attain, the statistic and everything downstream (segments, split log, draws) must be what the oracle
computes, and what one CTA per row (CBS_GPU_OBS_SLICES=1) computes."""
import numpy as np
import pytest

from helpers import f32, pack
from oracle.pyoracle import SegParams
import genomic_b200
from genomic_b200 import Params, RNG_MT19937_64, RNG_PHILOX

pytestmark = pytest.mark.gpu


def gparams(p: SegParams, **kw) -> Params:
    return Params(alpha=p.alpha, nperm=p.nperm, min_width=p.min_width, do_smooth=p.do_smooth,
                  rng_mode=RNG_PHILOX if p.rng_kind else RNG_MT19937_64, chain=p.chain, seed=p.seed, **kw)


def tied_vectors():
    """Vectors long enough for several slices whose maximum is attained by many arcs in different slices."""
    for n in (20000, 61003):
        yield n, "runs", np.tile([1.0] * 700 + [-1.0] * 700, n // 1400 + 1)[:n]
        yield n, "motif", np.tile([0.5, 0.5, -1.0, 0.25, 0.25, -0.5], n // 6 + 1)[:n]
        x = np.zeros(n); x[n // 5: 3 * n // 5] = 1.0
        yield n, "two_level", x
        yield n, "saw10", np.tile([1.0] * 5 + [-1.0] * 5, n // 10 + 1)[:n]


def centred(x):
    xc = x - x.mean()
    return xc, float((xc * xc).sum())


def test_tied_maxima_across_slices(ctx, oracle):
    for n, name, x in tied_vectors():
        for raw in (True, False):
            xc, tss = (x, float((x * x).sum())) if raw else centred(x)
            for al0 in (2, 3):
                assert ctx.tmaxo(xc, tss, al0) == oracle.tmaxo(xc, tss, al0), (n, name, raw, al0)
            assert ctx.tmaxp(xc, tss, 2) == oracle.tmaxp(xc, tss, 2), (n, name, raw)


def test_tmaxo_tmaxp_long_vectors(ctx, oracle):
    rng = np.random.default_rng(401)
    for n in (100000, 147726):
        x = f32(rng.normal(0, 0.2, n))
        for step in (False, True):
            if step:
                x[n // 4: n // 3] += 0.3
            xc, tss = centred(x)
            assert ctx.tmaxo(xc, tss, 2) == oracle.tmaxo(xc, tss, 2), (n, step)
            assert ctx.tmaxp(xc, tss, 2) == oracle.tmaxp(xc, tss, 2), (n, step)
    xs = np.stack([f32(rng.normal(0, 0.2, 30000)) for _ in range(3)])
    xs = xs - xs.mean(axis=1, keepdims=True)
    tss = float((xs[0] * xs[0]).sum())
    got = ctx.tmaxp(xs, tss, 2)
    assert [float(v) for v in got] == [oracle.tmaxp(r, tss, 2) for r in xs]


SCAN_LIST = 2048  # per-CTA list of block pairs (kernels.cuh)


def pass1_list_sizes(x, al0=2):
    """Host restatement of the first pass of the observed scan: the block pairs of arcs of 128 markers or more whose bound
    reaches the seed arc's statistic, counted per slice (diagonal chunks of 32 pairs dealt round-robin over the slices).
    Only used to check that the test below reaches lists on both sides of SCAN_LIST (the device rounds the same way up to
    the order of the prefix sums, so a count may differ by a few pairs)."""
    n = len(x)
    nb = int(round(np.sqrt(n)))
    S = np.concatenate([[0.0], np.cumsum(x)])
    bb = np.array([int(round(n * (b / nb))) for b in range(nb + 1)])
    blocks = [S[bb[b] + 1: bb[b + 1] + 1] for b in range(nb)]
    bmin = np.array([v.min() for v in blocks]); bmax = np.array([v.max() for v in blocks])
    amin = np.array([bb[b] + 1 + v.argmin() for b, v in enumerate(blocks)])
    amax = np.array([bb[b] + 1 + v.argmax() for b, v in enumerate(blocks)])
    gimin = amin[bmin.argmin()] if bmin.min() < 0 else n
    gimax = amax[bmax.argmax()] if bmax.max() > 0 else n
    spread = max(bmax.max(), 0.0) - min(bmin.min(), 0.0)
    rj = abs(gimax - gimin)
    init = n / (rj * (n - rj)) * spread * spread
    bi, bj = np.triu_indices(nb)
    bi, bj = bi + 1, bj + 1
    smx = np.maximum(np.abs(bmax[bj - 1] - bmin[bi - 1]), np.abs(bmax[bi - 1] - bmin[bj - 1]))
    lenhi = np.minimum(bb[bj] - bb[bi - 1] - 1, n - al0)
    lenlo = np.maximum(np.where(bi == bj, 1, bb[bj - 1] + 1 - bb[bi]), max(al0, 128)).astype(float)
    lo_hi = np.minimum(lenlo * (n - lenlo), lenhi * (n - lenhi.astype(float)))
    alive = (lenlo <= lenhi) & (n * smx * smx >= init * lo_hi * (1 - 1e-12))
    nsl = min(24, -(-n // 8192))
    d = bj - bi
    owner = ((d * nb - d * (d - 1) // 2 + bi - 1) >> 5) % nsl
    return [int(np.sum(alive & (owner == s))) for s in range(nsl)]


def test_pair_lists_on_both_sides_of_the_list_capacity(ctx, oracle, monkeypatch):
    """Slices of one row whose pair lists overflow (pass 2 enumerates the pairs again) next to slices whose lists do not:
    every block pair must still be scanned by exactly one slice.  Noisy periodic vectors with maxima of ~150 markers,
    i.e. inside the block pairs, not in the short-arc sweep."""
    n = 40000
    z = np.random.default_rng(5).normal(0, 1, n)
    straddle = 0
    cases = []
    for amp in (0.072, 0.074, 0.076):
        x = np.sin(2 * np.pi * np.arange(n) / 412.5) + amp * z
        x = x - x.mean()
        sizes = pass1_list_sizes(x)
        straddle += int(min(sizes) <= SCAN_LIST < max(sizes))
        tss = float((x * x).sum())
        want = oracle.tmaxo(x, tss, 2)
        assert want[2] - want[1] >= 128, want
        assert ctx.tmaxo(x, tss, 2) == want, (amp, sizes)
        assert ctx.tmaxp(x, tss, 2) == oracle.tmaxp(x, tss, 2), (amp, sizes)
        cases.append((x, tss, want))
    assert straddle >= 2
    monkeypatch.setenv("CBS_GPU_OBS_SLICES", "1")
    for x, tss, want in cases:
        assert ctx.tmaxo(x, tss, 2) == want


def check_split_log(got, want):
    assert len(got.splits) == len(want["log"])
    by_key = {(g["unit"], g["lo"], g["hi"]): g for g in got.splits}  # decisions are logged in order of completion
    for u, w in want["log"]:
        g = by_key[(u, w.lo, w.hi)]
        assert (g["called"], g["ncpt"]) == (w.called, w.ncpt), (u, w.lo, w.hi)
        if w.called:
            assert g["ostat"] == w.ostat, (u, w.lo, w.hi)
            assert (g["iseg0"], g["iseg1"], g["perms_run"], g["nrej"], g["exit_code"]) == \
                (w.iseg0, w.iseg1, w.perms_run, w.nrej, w.exit_code), (u, w.lo, w.hi)


@pytest.mark.parametrize("mode", ["mt_unit", "philox"])
def test_long_units_match_oracle(ctx, oracle, mode):
    rng = np.random.default_rng(411)
    null = f32(rng.normal(0, 0.2, 100000))
    steps = f32(rng.normal(0, 0.2, 147726))
    steps[30000:52000] += 0.5
    steps[90000:90900] -= 0.8
    runs = np.tile([0.3] * 900 + [-0.3] * 1100, 60)[:118000] + f32(rng.normal(0, 0.05, 118000))
    vals, off = pack([null, steps, runs])
    p = SegParams(nperm=100, alpha=0.01, do_smooth=False, rng_kind=1 if mode == "philox" else 0, chain=False, seed=21)
    want = oracle.segment_units(vals, off, np.ones(3, np.int32), p, want_log=True)
    got = ctx.segment_batch(vals, off, gparams(p, record_splits=True))
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    assert np.array_equal(got.means, want["means"])
    if mode != "philox":
        assert np.array_equal(got.draws, want["draws"])
    check_split_log(got, want)


def test_one_slice_per_row_gives_the_same_results(monkeypatch):
    from genomic_b200 import synth
    vals, off, lab, ids = synth.cohort([0], scale=0.25)
    p = Params(nperm=1000, rng_mode=RNG_MT19937_64, chain=False, seed=3, record_splits=True)
    c = genomic_b200.Context(0)
    try:
        sliced = c.segment_batch(vals, off, p, unit_ids=ids)
        monkeypatch.setenv("CBS_GPU_OBS_SLICES", "1")
        single = c.segment_batch(vals, off, p, unit_ids=ids)
    finally:
        c.close()
    for f in ("seg_count", "lengths", "means", "draws"):
        assert np.array_equal(getattr(sliced, f), getattr(single, f)), f
    key = lambda g: (g["unit"], g["lo"], g["hi"])
    assert sorted(sliced.splits, key=key) == sorted(single.splits, key=key)
