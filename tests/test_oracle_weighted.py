"""CPU (-m "not gpu"): the weighted oracle's split log and low-level bindings (oracle/cbs_oracle_weighted.c) agree with
its driver, and the driver stops where the reference would re-split a segment into itself."""
import time

import numpy as np
import pytest

from helpers import f32, make_unit, pack, weighted_centre
from oracle.pyoracle import SegParams, SplitIntoItself


def cohort(seed):
    rng = np.random.default_rng(seed)
    units = [make_unit(rng, int(rng.integers(1, 1200)), k % 5) for k in range(6)]
    units.insert(2, np.zeros(0))
    vals, off = pack(units)
    w = rng.choice([rng.uniform(0.5, 2.0, len(vals)), 10.0 ** rng.uniform(-3, 3, len(vals))])
    return vals, w, off


@pytest.mark.parametrize("mode,hybrid,undo_prune", [("mt_unit", False, False), ("mt_chain", False, True),
                                                    ("philox", False, False), ("mt_unit", True, False)])
def test_split_log_changes_nothing_and_replays(oracle, mode, hybrid, undo_prune):
    vals, w, off = cohort({"mt_unit": 1, "mt_chain": 2, "philox": 3}[mode] + 10 * hybrid)
    p = SegParams(nperm=200, alpha=0.05, do_smooth=False, rng_kind=1 if mode == "philox" else 0,
                  chain=(mode == "mt_chain"), seed=7, hybrid=hybrid, nmin=200, undo_prune=undo_prune)
    plain = oracle.segment_weighted_units(vals, w, off, p)
    logged = oracle.segment_weighted_units(vals, w, off, p, want_log=True)
    for f in ("seg_count", "lengths", "means", "draws"):
        assert np.array_equal(plain[f], logged[f]), f
    assert any(r.ncpt > 0 for _, r in logged["log"])
    if undo_prune:
        return
    # replay: a depth-first walk over the logged decisions, right-most pending segment first (CBS.cpp:976-1004)
    log = iter(logged["log"])
    lengths = []
    for u in range(len(off) - 1):
        n = int(off[u + 1] - off[u])
        if n == 0:
            continue
        ends, done = [0, n], []
        while len(ends) > 1:
            lo, hi = ends[-2], ends[-1]
            lu, r = next(log)
            assert (lu, r.lo, r.hi) == (u, lo, hi)
            cuts = [lo + c + 1 for c in (r.icpt0, r.icpt1)[:r.ncpt]]
            if not cuts:
                done.append(ends.pop())
            else:
                ends[-1:] = cuts + [hi]
        lengths += list(np.diff([0] + done[::-1]))
    assert next(log, None) is None
    assert lengths == logged["lengths"].tolist()


@pytest.mark.parametrize("hybrid", [False, True])
def test_wfindcpt_and_wtmaxo_equal_the_root_decision(oracle, hybrid):
    rng = np.random.default_rng(21 + hybrid)
    for trial in range(8):
        n = int(rng.integers(250 if hybrid else 8, 4000))
        x = make_unit(rng, n, trial % 5)
        w = [rng.uniform(0.5, 2.0, n), rng.choice([0.5, 1.0, 2.0], n), 10.0 ** rng.uniform(-3, 3, n)][trial % 3]
        al0 = int(rng.choice([2, 3, 5]))
        p = SegParams(nperm=300, alpha=0.05, min_width=al0, do_smooth=False, seed=5, hybrid=hybrid, nmin=200,
                      kmax=int(rng.choice([10, 25])))
        vals, off = pack([x])
        root = oracle.segment_weighted_units(vals, w, off, p, want_log=True)["log"][0][1]
        assert (root.lo, root.hi) == (0, n)
        if not root.called:
            continue
        xc, tss = weighted_centre(x, w)
        eng = oracle.rng_mt(p.seed)
        d = oracle.wfindcpt(xc, w, tss, p.nperm, p.alpha, eng, hybrid=hybrid, al0=al0, hk=p.kmax)
        assert (d.ostat, tuple(d.iseg)) == (root.ostat, (root.iseg0, root.iseg1)), trial
        assert (d.ncpt, d.perms_run, d.nrej, d.exit_code) == (root.ncpt, root.perms_run, root.nrej, root.exit_code), trial
        assert tuple(d.icpt)[:d.ncpt] == (root.icpt0, root.icpt1)[:d.ncpt]
        assert tuple(d.edge_p) == (root.edge_p0, root.edge_p1)
        assert oracle.wtmaxo(xc, w, tss, al0) == (root.ostat, root.iseg0, root.iseg1), trial


def test_low_level_bindings_are_consistent(oracle):
    rng = np.random.default_rng(31)
    n = 600
    x = make_unit(rng, n, 1)
    w = rng.uniform(0.5, 2.0, n)
    xc, tss = weighted_centre(x, w)
    eng = oracle.rng_mt(3)
    px = oracle.wxperm(xc, w, eng)
    assert eng.draws == n and not np.array_equal(px, xc)
    stat = oracle.wtmaxp(px, w, 2)
    assert stat == oracle.wtmaxo(px, w, 0.0, 2)[0]  # wtmaxp is wtmaxo with the reference's tss = 0 placeholder
    mn, delta = oracle.getmncwt(w, 25)
    assert mn[0] == 0.0 and np.all(np.diff(mn) > 0) and 0 < delta < 1
    assert oracle.hwtmaxp(px, w, 25) > 0
    p = oracle.wtpermp(200, n - 200, xc, w, 100, oracle.rng_mt(3))
    assert 0.0 <= p <= 1.0


def test_split_into_itself_is_reported(oracle):
    """One weight carries essentially all of the total: cw stalls, an arc of weight 0 has an infinite statistic, ostat is
    NaN, nothing rejects and the split point is the segment's last marker.  The reference would test [0, 400) again
    forever; the oracle stops and says so."""
    x = f32(np.random.default_rng(1).normal(0, 0.2, 400))
    x[150:250] += 1.0
    w = np.ones(400)
    w[200] = 1e20
    p = SegParams(nperm=200, alpha=0.05, do_smooth=False, seed=3)
    t0 = time.time()
    with pytest.raises(SplitIntoItself, match=r"unit 0, \[0, 400\)"):
        oracle.segment_weighted_units(x, w, np.array([0, 400]), p, want_log=True)
    with pytest.raises(SplitIntoItself):
        oracle.segment_weighted_units(x, w, np.array([0, 400]), p)
    assert time.time() - t0 < 10
    xc, tss = weighted_centre(x, w)
    d = oracle.wfindcpt(xc, w, tss, 200, 0.05, oracle.rng_mt(3))
    assert np.isnan(d.ostat) and (d.ncpt, d.icpt[0]) == (1, 399)
    # the same weight at index 0 terminates
    w0 = np.r_[1e20, np.ones(399)]
    r = oracle.segment_weighted_units(x, w0, np.array([0, 400]), p, want_log=True)
    assert r["lengths"].sum() == 400
