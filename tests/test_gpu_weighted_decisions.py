"""-m gpu: weighted CBS (DESIGN 4a) decision by decision against the C oracle (oracle/cbs_oracle_weighted.c).

Final segment lengths say little about the weighted path: the reference's wtmaxp passes tss = 0, so nearly every
permutation rejects, and a max-t test usually ends after nrejc + 1 permutations or takes the t >= 7 shortcut.  So these
tests compare what each decision computed: the observed statistic and its arc (k_wscan<1> over up to 24 CTAs,
k_wobs_fin, the wtmaxo_ordered tie fallback), the permutation counts (k_wscan<0> and its early decision), the edge
tests (k_wedgeprep/k_wedgeperm), the weighted hybrid kernels, and inputs whose weights make the statistic infinite."""
import re

import numpy as np
import pytest

from helpers import engine_after, f32, make_unit, pack, weighted_centre
from oracle.pyoracle import SegParams, SplitIntoItself, weight_tables
from test_gpu_scan_split import tied_vectors
from genomic_b200 import CbsGpuError, Params, RNG_MT19937_64, RNG_PHILOX
from genomic_b200.binding import ERR_UNSUPPORTED

pytestmark = pytest.mark.gpu


def gparams(p: SegParams, **kw) -> Params:
    return Params(alpha=p.alpha, nperm=p.nperm, hybrid=p.hybrid, min_width=p.min_width, kmax=p.kmax, nmin=p.nmin,
                  do_smooth=False, rng_mode=RNG_PHILOX if p.rng_kind else RNG_MT19937_64, chain=p.chain, seed=p.seed,
                  undo_prune=p.undo_prune, undo_prune_cutoff=p.undo_prune_cutoff, **kw)


def weight_sets(rng, n):
    return {"uniform": rng.uniform(0.5, 2.0, n), "three": rng.choice([0.5, 1.0, 2.0], n),
            "logu3": 10.0 ** rng.uniform(-3, 3, n)}


def arc_statistic(x, w, tss, start, end):
    """statistic of the arc (start, end] from sequential prefix sums, with the reference's expressions (CBS.cpp:714,
    737-738): independent of the oracle's scan"""
    s = np.concatenate([[0.0], np.cumsum(x * w)])
    _, cw = weight_tables(w)
    d = s[end + 1] - s[start + 1]
    a = cw[end] - cw[start]
    m = (d * d) / (a * (cw[-1] - a))
    if tss <= m + 0.0001:
        tss = m + 1.0
    return m / ((tss - m) / (len(x) - 2.0))


@pytest.mark.parametrize("n", [20000, 70000, 147726, 600000])
def test_wtmaxo_long_vectors(ctx, oracle, n):
    rng = np.random.default_rng(n)
    x = f32(rng.normal(0, 0.2, n))
    for step in (False, True):
        if step:
            x[n // 4: n // 3] += 0.3
            x[n // 2: n // 2 + 40] -= 0.6
        for wname, w in weight_sets(rng, n).items():
            xc, tss = weighted_centre(x, w)
            for al0 in (2, 3, 5):
                got = ctx.wtmaxo(xc, w, tss, al0)
                assert got == oracle.wtmaxo(xc, w, tss, al0), (n, step, wname, al0)
                assert got[0] == arc_statistic(xc, w, tss, got[1], got[2]), (n, step, wname, al0)


@pytest.mark.parametrize("n", [20000, 61003, 147726])
def test_tied_maxima_across_slices(ctx, oracle, n):
    """Maxima attained by many arcs in different slices, with weights that keep the ties (wcand_tied -> w_tie ->
    wtmaxo_ordered in k_wobs_fin)."""
    for _, name, x in tied_vectors((n,)):
        for wname, w in (("ones", np.ones(n)), ("1,2", np.tile([1.0, 2.0], n)[:n]),
                         ("1,2,0.5", np.tile([1.0, 2.0, 0.5], n)[:n])):
            for raw in (True, False):
                xc, tss = (x, float(np.cumsum(w * x * x)[-1])) if raw else weighted_centre(x, w)
                for al0 in (2, 3):
                    got, want = ctx.wtmaxo(xc, w, tss, al0), oracle.wtmaxo(xc, w, tss, al0)
                    assert np.array_equal(got, want, equal_nan=True), (n, name, wname, raw, al0)  # NaN: raw, weight 0 arcs


def decision_input(rng, kind, n):
    x = rng.normal(0, 0.2, n)
    if kind == "spike":  # short high arcs: no t >= 7 shortcut, the permutations run
        for _ in range(int(rng.integers(1, 3))):
            a = int(rng.integers(0, max(1, n - 8)))
            x[a:a + int(rng.integers(1, 8))] += float(rng.choice([1.5, 3.0, 6.0]))
    elif kind == "weak":
        x[n // 4: n // 2] += float(rng.choice([0.02, 0.05, 0.1]))
    elif kind == "step":
        x[n // 3:] += 1.0
    elif kind == "zero":  # t <= 0.1
        x[:] = 0.0
    return f32(x)


def check_edge_p(status, nrej, want_p, nperm, msg):
    """tpermp p-values of both boundaries: the device reports the rejection counts and the shortcut status"""
    for side in (0, 1):
        if want_p[side] < 0:
            continue  # not run
        got_p = 1.0 if status[side] == 1 else 0.0 if status[side] == 2 else nrej[side] / nperm
        assert got_p == want_p[side], (msg, side, status, nrej, want_p)


def test_wfindcpt_single_calls(ctx, oracle):
    """cbs::wfindcpt with a caller-owned engine that has already been used: every field of the decision and the draws."""
    rng = np.random.default_rng(501)
    exits = set()
    cases = []
    for n in (8, 9, 60, 500, 3000, 20000, 147726):
        for kind in ("spike", "weak", "step", "zero", "null"):
            for hybrid in (False, True):
                if hybrid and n < 250:
                    continue
                cases.append((n, kind, hybrid))
    for k, (n, kind, hybrid) in enumerate(cases):
        x = decision_input(rng, kind, n)
        w = list(weight_sets(rng, n).values())[k % 3]
        xc, tss = weighted_centre(x, w)
        al0 = 2 if n < 20 else int(rng.choice([2, 3, 5]))
        kmax = int(rng.choice([10, 25]))
        nperm = 200 if n > 20000 else 500
        eng, nxt = engine_after(oracle, 9, int(rng.integers(0, 5000)))
        d0 = eng.draws
        want = oracle.wfindcpt(xc, w, tss, nperm, 0.05, eng, hybrid=hybrid, al0=al0, hk=kmax)
        got = ctx.wfindcpt(xc, w, tss, Params(alpha=0.05, nperm=nperm, min_width=al0, hybrid=hybrid, kmax=kmax,
                                              nmin=kmax + 2, seed=9), mt_next312=nxt)
        msg = (n, kind, hybrid, al0)
        assert got["ostat"] == want.ostat and got["iseg"] == tuple(want.iseg), msg
        assert (got["ncpt"], got["perms_run"], got["nrej"], got["exit_code"]) == \
            (want.ncpt, want.perms_run, want.nrej, want.exit_code), msg
        assert got["icpt"][:want.ncpt] == tuple(want.icpt)[:want.ncpt], msg
        check_edge_p(got["e_status"], got["e_nrej"], tuple(want.edge_p), nperm, msg)
        assert got["draws"] == eng.draws - d0, msg
        exits.add(want.exit_code)
    assert exits == {0, 1, 2, 3, 4}


def segment_mix(rng, n):
    """noise with a few short spikes and weak steps: decisions of every kind, edge tests with 0 < p < 1"""
    x = rng.normal(0, 0.2, n)
    for _ in range(int(rng.integers(1, 4))):
        a = int(rng.integers(0, max(1, n - 8)))
        x[a:a + int(rng.integers(2, 8))] += float(rng.choice([-1.0, 1.0])) * float(rng.choice([0.6, 1.0, 2.0]))
    for _ in range(int(rng.integers(1, 3))):
        a = int(rng.integers(0, n))
        x[a:int(rng.integers(a, n + 1))] += float(rng.choice([0.05, 0.1, 0.2]))
    return f32(x)


def step_unit(rng, n):
    """noise with three overlapping steps: long segments whose decisions end early or take the t >= 7 shortcut"""
    x = rng.normal(0, 0.2, n)
    for _ in range(3):
        a = int(rng.integers(0, n))
        x[a:int(rng.integers(a, n + 1))] += float(rng.choice([-0.5, 0.3, 0.6]))
    return f32(x)


def check_weighted_log(got, want, p, exact_draws):
    """every logged decision of the device equals the oracle's, matched by (unit, lo, hi); returns coverage counts"""
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    if p.hybrid:  # as in the other hybrid tests
        assert np.allclose(got.means, want["means"], rtol=1e-9, atol=0)
    else:
        assert np.array_equal(got.means, want["means"])
    if exact_draws:
        assert np.array_equal(got.draws, want["draws"])
    assert len(got.splits) == len(want["log"])
    by_key = {(g["unit"], g["lo"], g["hi"]): g for g in got.splits}
    assert len(by_key) == len(got.splits)
    edge_mid = nrej_mid = 0
    for u, w in want["log"]:
        key = (u, w.lo, w.hi)
        g = by_key[key]
        assert (g["called"], g["ncpt"]) == (w.called, w.ncpt), key
        if not w.called:
            continue
        assert np.array_equal(g["ostat"], w.ostat, equal_nan=True), key
        assert (g["iseg0"], g["iseg1"], g["perms_run"], g["nrej"], g["exit_code"]) == \
            (w.iseg0, w.iseg1, w.perms_run, w.nrej, w.exit_code), key
        assert (g["icpt0"], g["icpt1"])[:w.ncpt] == (w.icpt0, w.icpt1)[:w.ncpt], key
        check_edge_p((g["e_status0"], g["e_status1"]), (g["e_nrej0"], g["e_nrej1"]), (w.edge_p0, w.edge_p1), p.nperm, key)
        edge_mid += int(0.0 < w.edge_p0 < 1.0) + int(0.0 < w.edge_p1 < 1.0)
        nrej_mid += int(w.exit_code != 3 and 0 < w.nrej)
    return edge_mid, nrej_mid


def test_split_logs_all_modes(ctx, oracle):
    """MT chain, MT unit and Philox; short units next to 100 000- to 147 726-marker units; several batch sizes and
    undo_prune.  Decisions compared field by field."""
    rng = np.random.default_rng(511)
    long_units = {n: step_unit(rng, n) for n in (100000, 118000, 147726)}
    edge_mid = nrej_mid = 0
    for trial, (mode, nlong, hybrid, undo) in enumerate((("mt_chain", 100000, False, False), ("mt_unit", 118000, False, True),
                                                         ("philox", 147726, False, False), ("mt_chain", 147726, True, False),
                                                         ("mt_unit", 100000, True, False), ("philox", 118000, False, True))):
        units = [segment_mix(rng, int(n)) for n in rng.integers(8, 4000, 16)]
        units.insert(3, long_units[nlong])
        units.insert(5, np.zeros(0))
        vals, off = pack(units)
        w = list(weight_sets(rng, len(vals)).values())[trial % 3]
        p = SegParams(nperm=int(rng.choice([200, 500])), alpha=float(rng.choice([0.05, 0.1])), do_smooth=False, rng_kind=1 if mode == "philox" else 0,
                      chain=(mode == "mt_chain"), seed=int(rng.integers(1, 100)), hybrid=hybrid, undo_prune=undo,
                      min_width=int(rng.choice([2, 3])))
        want = oracle.segment_weighted_units(vals, w, off, p, want_log=True)
        got = ctx.segment_weighted_batch(vals, w, off, gparams(p, record_splits=True, first_batch=int(rng.choice([16, 64, 256])),
                                                                max_batch=int(rng.choice([64, 256, 2048]))))
        e, r = check_weighted_log(got, want, p, exact_draws=(mode != "philox"))
        edge_mid += e
        nrej_mid += r
    assert edge_mid >= 15  # permutation edge tests with 0 < p < 1 were compared
    assert nrej_mid >= 10  # max-t tests that ran to the end with 0 < nrej <= nrejc were compared


@pytest.mark.parametrize("kmax", [25, 10])
def test_hybrid_long_units(ctx, oracle, kmax):
    """k_wdelta (wrap-around arcs included), k_wssq and k_whscan on units of 20 000 to 147 726 markers."""
    rng = np.random.default_rng(521 + kmax)
    units = [step_unit(rng, n) for n in (20000, 61003, 147726)] + [segment_mix(rng, 3000)]
    vals, off = pack(units)
    w = rng.uniform(0.5, 2.0, len(vals))
    p = SegParams(nperm=200, alpha=0.05, do_smooth=False, rng_kind=0, chain=False, seed=6, hybrid=True, kmax=kmax)
    want = oracle.segment_weighted_units(vals, w, off, p)
    got = ctx.segment_weighted_batch(vals, w, off, gparams(p, first_batch=64))
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    assert np.array_equal(got.draws, want["draws"])
    assert np.allclose(got.means, want["means"], rtol=1e-9, atol=0)


def extreme_weight_cases():
    n = 400
    x = f32(np.random.default_rng(1).normal(0, 0.2, n))
    x[150:250] += 1.0
    y = make_unit(np.random.default_rng(5), n, 1)
    lu = 10.0 ** np.random.default_rng(6).uniform(-8, 8, n)
    alt = np.tile([1e9, 1e-9], n // 2)
    first = np.r_[1e20, np.ones(n - 1)]
    mid = np.r_[np.ones(200), 1e20, np.ones(199)]
    return [("alternating", x, alt), ("alternating", y, alt), ("logu8", x, lu), ("logu8", y, lu),
            ("first", x, first), ("first", y, first), ("middle", x, mid), ("middle", y, mid)]


def test_extreme_weights(ctx, oracle):
    """cw not strictly increasing (w_ok = 0: no early decision), infinite arc statistics, NaN ostat.  Where the oracle
    terminates, results and split log are equal; where a decision would re-create its own segment (the reference would
    loop), the device stops with CBS_GPU_ERR_UNSUPPORTED naming the segment."""
    outcomes = set()
    for name, x, w in extreme_weight_cases():
        for mode in ("mt_chain", "philox"):
            vals, off = pack([x, make_unit(np.random.default_rng(7), 300, 1)])
            ww = np.r_[w, np.random.default_rng(8).uniform(0.5, 2.0, 300)]
            p = SegParams(nperm=200, alpha=0.05, do_smooth=False, rng_kind=1 if mode == "philox" else 0,
                          chain=(mode == "mt_chain"), seed=3)
            try:
                want = oracle.segment_weighted_units(vals, ww, off, p, want_log=True)
            except SplitIntoItself as e:
                outcomes.add("self_split")
                with pytest.raises(CbsGpuError) as info:
                    ctx.segment_weighted_batch(vals, ww, off, gparams(p, record_splits=True))
                assert info.value.code == ERR_UNSUPPORTED, (name, mode)
                where = r"unit (\d+), (?:segment )?\[(\d+), (\d+)\)"
                assert re.search(where, str(info.value)).groups() == re.search(where, str(e)).groups(), (name, mode)
                continue
            outcomes.add("terminates")
            outcomes.update("nan" for _, r in want["log"] if r.called and np.isnan(r.ostat))
            got = ctx.segment_weighted_batch(vals, ww, off, gparams(p, record_splits=True))
            check_weighted_log(got, want, p, exact_draws=(mode != "philox"))
        xc, tss = weighted_centre(x, w)
        eng, nxt = engine_after(oracle, 3, 0)
        want = oracle.wfindcpt(xc, w, tss, 200, 0.05, eng)
        got = ctx.wfindcpt(xc, w, tss, Params(alpha=0.05, nperm=200, seed=3), mt_next312=nxt)
        assert np.array_equal(got["ostat"], want.ostat, equal_nan=True) and got["iseg"] == tuple(want.iseg), name
        assert (got["ncpt"], got["perms_run"], got["nrej"], got["exit_code"]) == \
            (want.ncpt, want.perms_run, want.nrej, want.exit_code), name
        assert got["icpt"][:want.ncpt] == tuple(want.icpt)[:want.ncpt], name
        assert got["draws"] == eng.draws, name
    assert outcomes == {"self_split", "terminates", "nan"}
