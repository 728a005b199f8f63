"""-m gpu: the unweighted hybrid method (DNAcopy's default, `cna segment --hybrid true`) decision by decision against the C
oracle (oracle/cbs_oracle.c) over the whole kmax range 1..128.

The hybrid method tests a segment's observed statistic with htmaxp permutations (k_hscan: bit-exact) after the analytic
tail probability tailp (k_tailp_terms / k_tailp_sum: CUDA erfc/log/exp/pow, within ~1e-15 of libm, not bit-exact; DESIGN
2).  That p-value drives two integer decisions of the scheduler (cbs_core.h, Sched::step): the EX_TAILP exit
(pval1 > alpha) and the rejection budget nrejc = (int)((alpha - pval1) * nperm).  So every decision compared here also
shows that the oracle's pval1 is clear of both boundaries by more than the tailp tolerance (boundary_clear): an input that
drifts onto one fails with that message instead of flaking."""
import math
import os
import subprocess

import numpy as np
import pytest

from helpers import check_split_log, engine_after, f32, gparams, pack
from oracle.pyoracle import SegParams
from genomic_b200 import CbsGpuError, Params
from genomic_b200.binding import ERR_UNSUPPORTED

pytestmark = pytest.mark.gpu

TAILP_RTOL = 1e-12  # CUDA erfc/log/exp/pow against libm (test_gpu_lowlevel.py::test_tailp)
TAILP_ATOL = 1e-300  # where the result underflows: subnormal on one side, 0 on the other
KMAXES = (1, 2, 3, 10, 25, 64, 127, 128)


def tailp_error(got, want):
    """error of the device's tailp in units of the tolerance (<= 1 passes)"""
    return abs(got - want) / (TAILP_RTOL * abs(want) + TAILP_ATOL)


def x_range(b, delta, m):
    """smallest and largest argument x = b/sqrt(m t(1-t)) of nu() over tailp's quadrature points"""
    dincr = (0.5 - delta) / 100
    ends = [(0.5 + 0.5 * dincr) * (0.5 - 0.5 * dincr), (0.5 - 99.5 * dincr) * (0.5 + 99.5 * dincr)]
    xs = [b / math.sqrt(m) / math.sqrt(v) for v in ends]
    return min(xs), max(xs)


def tailp_grid():
    """(b, delta, m, tol): m from just above nmin up to 2^23 with the segmenter's delta = (kmax+1)/m, explicit deltas, b
    from just above 0.1 to past the underflow of exp(-b^2/2), and b where x = b/sqrt(m t(1-t)) crosses 0.01 inside the
    quadrature (both branches of nu).  Where every x is in (0.01, 0.2), nu() sums 1e4 to 1e6 terms per point in the
    oracle; only a few such points are kept, to bound the oracle's time."""
    ms = (3, 12, 27, 66, 130, 201, 257, 1000, 4099, 20000, 147726, 1048577, 1 << 23)
    bs = (0.1000001, 0.25, 0.7, 1.5, 2.5, 3.5, 5.0, 7.0, 10.0, 15.0, 25.0, 37.0, 38.2, 38.7, 40.0)
    pts, slow = [], []
    for kmax in (1, 10, 25, 64, 128):
        for m in ms:
            if m < kmax + 2:  # nmin >= kmax + 1 (cbs_gpu.cu run_cbs)
                continue
            delta = (kmax + 1) / m
            for b in bs:
                lo, hi = x_range(b, delta, m)
                (pts if lo >= 0.2 or hi <= 0.01 else slow).append((b, delta, m))
    for delta in (1e-7, 1e-3, 0.05, 0.25, 0.49, 0.75):
        for m in (201, 20000, 1 << 23):
            pts += [(b, delta, m) for b in (0.3, 2.0, 6.0, 30.0) if x_range(b, delta, m)[0] >= 0.2 or x_range(b, delta, m)[1] <= 0.01]
    pts += slow[::max(1, len(slow) // 4)]
    for m, kmax in ((1000, 25), (147726, 128), (1 << 23, 25)):  # x = 0.01 at t = 0.1
        pts.append((0.01 * math.sqrt(m * 0.09), (kmax + 1) / m, m))
    return [(b, d, m, tol) for (b, d, m) in pts for tol in (1e-6, 1e-9)]


def test_tailp_sweep(ctx, oracle):
    worst, where, zeros, branches = 0.0, None, 0, 0
    for b, delta, m, tol in tailp_grid():
        got, want = ctx.tailp(b, delta, m, tol=tol), oracle.tailp(b, delta, m, tol=tol)
        e = tailp_error(got, want)
        if e > worst:
            worst, where = e, (b, delta, m, tol, got, want)
        zeros += want == 0.0
        lo, hi = x_range(b, delta, m)
        branches += lo <= 0.01 < hi
    rel = worst * TAILP_RTOL
    assert worst <= 1.0, f"largest tailp error {rel:.3g} (relative; absolute {TAILP_ATOL:g} where 0) at (b, delta, m, tol, got, want) = {where}"
    assert zeros >= 10 and branches >= 6, (zeros, branches)


# ---- htmaxp ------------------------------------------------------------------------------------------------------------
def htmaxp_seams(n, k):
    """prefix indices at which htmaxp's own blocks end (nb = int(n/k), CBS.cpp:77 rounding)"""
    nb = int(n / k)
    return [int(math.floor(n * (b / nb) + 0.5)) for b in range(1, nb)]


def htmaxp_rows(rng, n, k, count):
    """null rows, steps on the block seams, spikes of width <= k, shifts at both ends (wrap-around arcs), constant runs"""
    rows = []
    seams = htmaxp_seams(n, k) or [n // 2]
    for r in range(count):
        x = rng.normal(0, 0.2, n)
        kind = r % 6
        if kind == 1:
            s = int(rng.choice(seams))
            w = int(rng.integers(1, k + 1))
            a = max(0, s - int(rng.integers(0, w + 1)))
            x[a:a + w] += float(rng.choice([-1.5, 0.8, 2.5]))
        elif kind == 2:
            for _ in range(int(rng.integers(1, 4))):
                w = int(rng.integers(1, k + 1))
                a = int(rng.integers(0, max(1, n - w)))
                x[a:a + w] += float(rng.choice([-2.0, 1.0, 3.0]))
        elif kind == 3:
            w1, w2 = int(rng.integers(1, k + 1)), int(rng.integers(1, k + 1))
            x[:w1] += 1.2
            x[n - w2:] += float(rng.choice([1.2, 0.9, -0.5]))
        elif kind == 4:
            x = np.round(rng.normal(0, 1, n))  # integers: tied arc sums
            x[:int(rng.integers(0, n))] = 0.0
        elif kind == 5:
            x = np.repeat(rng.choice([-1.0, 0.0, 1.0], n // max(1, k // 2) + 1), max(1, k // 2))[:n]
        rows.append(f32(x) - float(np.mean(f32(x))))
    return np.stack(rows)


@pytest.mark.parametrize("k", KMAXES)
def test_htmaxp_bit_exact(ctx, oracle, k):
    """k_hscan against orc_htmaxp: the maximum over all arcs of al0..k markers (inside blocks, across seams, wrapping
    around the end) and htmaxp's per-block candidates, from n = k (one block) up to 147 726"""
    rng = np.random.default_rng(900 + k)
    ns = sorted({k, k + 1, 2 * k, 2 * k + 1, 2 * k + 2, 3 * k, 10 * k + 7} - {1}) + [50000, 147726]
    for al0 in (1, 2, 3, 5):
        if al0 > k:
            continue
        for n in ns:
            m = htmaxp_rows(rng, n, k, 24 if n < 50000 else 6)
            tss = float((m[0] * m[0]).sum())
            got = ctx.htmaxp(m, tss, k, al0)
            want = np.array([oracle.htmaxp(r, tss, k, al0) for r in m])
            bad = np.flatnonzero(got != want)
            assert not len(bad), (k, al0, n, bad[:5], got[bad[:3]], want[bad[:3]])


# ---- the pval1 boundary ------------------------------------------------------------------------------------------------
def boundary_clear(pval1, alpha, nperm, msg):
    """The decision that depends on pval1 (EX_TAILP, then nrejc) is the same for every value within TAILP_RTOL of the
    oracle's, so a last-bit difference of the device's tailp cannot change it.  Returns the relative change of pval1
    that would (alpha side, nrejc side) for the report."""
    def decide(p):
        return (True, 0) if p > alpha else (False, int((alpha - p) * nperm))
    want = decide(pval1)
    for q in (pval1 * (1 - TAILP_RTOL) - TAILP_ATOL, pval1 * (1 + TAILP_RTOL) + TAILP_ATOL):
        assert decide(q) == want, (f"pval1 = {pval1!r} is within the tailp tolerance of a decision boundary "
                                   f"(alpha = {alpha}, nperm = {nperm}): change the input", msg)
    rel_alpha = abs(alpha - pval1) / abs(pval1) if pval1 else math.inf
    rel_nrejc = math.inf
    if not want[0] and alpha - pval1 != alpha:  # else pval1 is below the rounding of alpha: nrejc = int(alpha * nperm)
        v = (alpha - pval1) * nperm
        rel_nrejc = min(v - math.floor(v), math.floor(v) + 1 - v) / nperm / abs(pval1)
    return rel_alpha, rel_nrejc


class Tally:
    def __init__(self):
        self.exits, self.tailp_exit, self.early, self.full_mid, self.short = {}, 0, 0, 0, 0  # see report()
        self.rel_alpha = self.rel_nrejc = math.inf
        self.tailp_worst = 0.0

    def hybrid_decision(self, ctx, oracle, n, kmax, ostat, exit_code, nrej, perms_run, alpha, nperm, tol, delta, msg):
        """pval1 at exactly this decision: device against oracle, and clear of both boundaries"""
        self.exits[exit_code] = self.exits.get(exit_code, 0) + 1
        self.short += n <= 2 * kmax
        b = math.sqrt(ostat)
        if b <= 0.1 or exit_code in (1, 2):  # pval1 not used (CBS.cpp:839-848)
            return
        got, want = ctx.tailp(b, delta, n, tol=tol), oracle.tailp(b, delta, n, tol=tol)
        e = tailp_error(got, want)
        assert e <= 1.0, ("tailp at a logged decision", msg, got, want)
        self.tailp_worst = max(self.tailp_worst, e * TAILP_RTOL)
        ra, rn = boundary_clear(want, alpha, nperm, msg)
        self.rel_alpha, self.rel_nrejc = min(self.rel_alpha, ra), min(self.rel_nrejc, rn)
        nrejc = int((alpha - want) * nperm) if want <= alpha else None
        self.tailp_exit += exit_code == 4
        self.early += exit_code == 3 and nrejc is not None and 0 < nrejc and nrej == nrejc + 1
        self.full_mid += exit_code == 0 and nrejc is not None and 0 < nrej <= nrejc and perms_run == nperm

    def report(self, what):
        print(f"{what}: exits {sorted(self.exits.items())}, EX_TAILP {self.tailp_exit}, early exits with nrejc > 0 {self.early}, "
              f"full runs with 0 < nrej <= nrejc {self.full_mid}, n <= 2 kmax {self.short}, "
              f"smallest relative pval1 margin to alpha {self.rel_alpha:.3g}, to an nrejc step {self.rel_nrejc:.3g}, "
              f"largest tailp error {self.tailp_worst:.3g}")


# ---- single fndcpt calls -----------------------------------------------------------------------------------------------
def decision_input(rng, kind, n):
    x = rng.normal(0, 0.2, n)
    if kind == "spike":  # short high arcs: the permutations run and usually end early
        for _ in range(int(rng.integers(1, 3))):
            w = int(rng.integers(1, max(2, min(n // 4, 8))))
            a = int(rng.integers(0, max(1, n - w)))
            x[a:a + w] += float(rng.choice([0.6, 1.0, 1.6]))
    elif kind == "weak":  # tailp > alpha on long segments
        x[n // 4: n // 2] += float(rng.choice([0.005, 0.02, 0.05]))
    elif kind == "step":  # t >= 7 shortcut
        x[n // 3:] += 1.5
    return f32(x)


def centred(x):
    cur = x - np.cumsum(x)[-1] / len(x)  # CBS.cpp:986-989, sequential sums
    return cur, float(np.cumsum(cur * cur)[-1])


def test_fndcpt_hybrid_single_calls(ctx, oracle):
    """cbs_gpu_fndcpt(hybrid) with a caller-owned engine already in use: n from 2 al0 through kmax <= n <= 2 kmax up to
    147 726, kmax 1..128, delta by default ((kmax+1)/n) and explicit.  Calls the reference leaves undefined are refused."""
    rng = np.random.default_rng(931)
    tally, refused = Tally(), 0
    cases = []
    for kmax in KMAXES:
        for n in sorted({4, kmax, kmax + 1, kmax + 2, kmax + 3, 2 * kmax - 1, 2 * kmax, 2 * kmax + 1, 300, 3000}):
            cases += [(kmax, n, kind) for kind in ("spike", "weak", "step", "null", "flat") if n >= 2]
    cases += [(kmax, n, kind) for kmax in (25, 128) for n in (20000, 147726) for kind in ("spike", "weak", "step")]
    for kmax, n, kind in cases:
        al0 = int(rng.choice([a for a in (1, 2, 3, 5) if a <= kmax and 2 * a <= n] or [1]))
        x = decision_input(rng, kind if kind != "flat" else "null", n)
        xc, tss = centred(x)
        if kind == "flat":  # t <= 0.1: the caller's tss is far larger than the segment's
            tss *= 1e6
        explicit = bool(rng.integers(0, 2))
        delta = float(rng.choice([0.01, 0.2, 0.45])) if explicit else (kmax + 1) / n
        nperm = int(rng.choice([100, 200])) if n > 20000 else int(rng.choice([100, 500]))
        alpha = float(rng.choice([0.01, 0.05]))
        p = Params(alpha=alpha, nperm=nperm, min_width=al0, hybrid=True, kmax=kmax, seed=9)
        eng, nxt = engine_after(oracle, 9, int(rng.integers(0, 3000)))
        msg = (kmax, n, kind, al0, delta)
        if n < kmax or delta >= 1.0:  # htmaxp without a block, or tailp NaN / -inf
            with pytest.raises(CbsGpuError) as e:
                ctx.fndcpt(xc, tss, p, delta=delta if explicit else 0.0, mt_next312=nxt)
            assert e.value.code == ERR_UNSUPPORTED and "hybrid fndcpt needs n >= hk and delta < 1" in str(e.value), msg
            refused += 1
            continue
        d0 = eng.draws
        want = oracle.fndcpt(xc, tss, nperm, alpha, eng, hybrid=True, al0=al0, hk=kmax, delta=delta)
        got = ctx.fndcpt(xc, tss, p, delta=delta if explicit else 0.0, mt_next312=nxt)
        assert got["ostat"] == want.ostat and got["iseg"] == tuple(want.iseg), msg
        assert (got["ncpt"], got["perms_run"], got["nrej"], got["exit_code"]) == \
            (want.ncpt, want.perms_run, want.nrej, want.exit_code), msg
        assert got["icpt"][:want.ncpt] == tuple(want.icpt)[:want.ncpt], msg
        assert got["draws"] == eng.draws - d0, msg
        tally.hybrid_decision(ctx, oracle, n, kmax, want.ostat, want.exit_code, want.nrej, want.perms_run, alpha, nperm,
                              1e-6, delta, msg)
    tally.report("fndcpt")
    assert {1, 2, 3, 4} <= set(tally.exits), tally.exits
    assert tally.short >= 40 and refused >= 20, (tally.short, refused)


# ---- split logs ----------------------------------------------------------------------------------------------------------
def short_unit(rng, n):
    """noise with a spike or a weak shift: decisions that exit early, on the tail probability or after all permutations"""
    x = rng.normal(0, 0.2, n)
    r = rng.random()
    if r < 0.4:
        w = int(rng.integers(1, max(2, n // 6)))
        a = int(rng.integers(0, max(1, n - w)))
        x[a:a + w] += float(rng.choice([-1.0, 0.5, 0.8, 1.5]))
    elif r < 0.7:
        a = int(rng.integers(0, n))
        x[a:int(rng.integers(a, n + 1))] += float(rng.choice([0.05, 0.15, 0.3]))
    return f32(x)


def long_unit(rng, n):
    """noise with steps of several sizes, short spikes and weak shifts at both ends"""
    x = rng.normal(0, 0.2, n)
    for _ in range(3):
        a = int(rng.integers(0, n))
        x[a:int(rng.integers(a, min(n, a + n // 3) + 1))] += float(rng.choice([-0.5, 0.1, 0.3, 0.6]))
    for _ in range(3):
        a = int(rng.integers(0, n - 10))
        x[a:a + int(rng.integers(1, 10))] += float(rng.choice([-1.2, 1.0]))
    x[:int(rng.integers(50, 3000))] += 0.05
    x[n - int(rng.integers(50, 3000)):] -= 0.05
    return f32(x)


# (mode, kmax, nmin, min_width, undo_prune)
SPLIT_CONFIGS = [("mt_chain", 1, 2, 2, False), ("philox", 1, 60, 3, True), ("mt_unit", 25, 26, 2, False),
                 ("mt_chain", 25, 200, 5, True), ("philox", 64, 100, 2, False), ("mt_unit", 64, 300, 3, False),
                 ("mt_chain", 128, 129, 3, False), ("philox", 128, 200, 2, True), ("mt_unit", 128, 400, 5, False)]


def run_split_batch(ctx, oracle, units, p, tally, first_batch=0):
    vals, off = pack(units)
    want = oracle.segment_units(vals, off, np.ones(len(units), np.int32), p, want_log=True)
    got = ctx.segment_batch(vals, off, gparams(p, record_splits=True, first_batch=first_batch))
    for u, w, _ in check_split_log(got, want, p, exact_draws=not p.rng_kind):
        n = w.hi - w.lo
        if p.nmin < n:  # use_hybrid (cbs_core.h new_task)
            tally.hybrid_decision(ctx, oracle, n, p.kmax, w.ostat, w.exit_code, w.nrej, w.perms_run, p.alpha, p.nperm,
                                  p.tol, (p.kmax + 1) / n, (u, w.lo, w.hi))


def test_split_logs_hybrid(ctx, oracle):
    """MT chain, MT unit and Philox; units of exactly nmin, nmin + 1 and up to 2 kmax markers beside 20 000- to 147 726-
    marker units; kmax 1..128 with nmin below and above 2 kmax, min_width 2/3/5, with and without undo_prune"""
    rng = np.random.default_rng(941)
    tally = Tally()
    for trial, (mode, kmax, nmin, mw, undo) in enumerate(SPLIT_CONFIGS):
        lens = [nmin, nmin, nmin + 1, nmin + 1, nmin + 2] + [int(v) for v in rng.integers(nmin + 1, max(nmin + 2, 2 * kmax + 1), 6)]
        lens += [int(v) for v in rng.integers(2 * mw, 3000, 6)]
        units = [short_unit(rng, n) for n in lens]
        units.insert(4, long_unit(rng, int(rng.choice([20000, 61003, 147726]))))
        units.insert(9, np.zeros(0))
        p = SegParams(nperm=int(rng.choice([100, 200, 500])), alpha=float(rng.choice([0.01, 0.05])), hybrid=True, kmax=kmax,
                      nmin=nmin, min_width=mw, undo_prune=undo, do_smooth=False, rng_kind=1 if mode == "philox" else 0,
                      chain=(mode == "mt_chain"), seed=int(rng.integers(1, 100)))
        run_split_batch(ctx, oracle, units, p, tally, first_batch=int(rng.choice([0, 16, 64])))
    tally.report("split logs")
    assert tally.tailp_exit >= 20 and tally.early >= 20 and tally.full_mid >= 5 and tally.short >= 20, vars(tally)


def test_split_log_past_2_20(ctx, oracle):
    """one 1 048 577-marker unit at kmax = 128 (rows past 2^20) beside short units, small nperm"""
    rng = np.random.default_rng(951)
    tally = Tally()
    n = (1 << 20) + 1
    big = f32(rng.normal(0, 0.2, n))
    big[300000:300040] += 1.0
    big[700000:900000] += 0.08
    big[:1500] += 0.1
    units = [short_unit(rng, m) for m in (129, 130, 200, 256)] + [big]
    p = SegParams(nperm=50, alpha=0.05, hybrid=True, kmax=128, nmin=129, do_smooth=False, rng_kind=0, chain=True, seed=3)
    run_split_batch(ctx, oracle, units, p, tally)
    tally.report("past 2^20")
    assert sum(tally.exits.values()) >= 5


# ---- undefined inputs are refused ----------------------------------------------------------------------------------------
def test_hybrid_refusals(ctx, oracle):
    """nmin <= kmax would let hybrid segments of kmax + 1 markers or fewer through, where the reference's htmaxp has no
    block or its tailp is NaN; nmin = kmax + 1 is accepted and equals the oracle"""
    rng = np.random.default_rng(961)
    x = short_unit(rng, 400)
    msg = "hybrid CBS needs nmin >= kmax + 1"
    for kmax, nmin in ((25, 0), (25, 23), (25, 25), (128, 127), (1, 1)):
        q = Params(hybrid=True, kmax=kmax, nmin=nmin, do_smooth=False)
        for call in (lambda: ctx.segment(x, q), lambda: ctx.segment_batch(x, np.array([0, 400]), q)):
            with pytest.raises(CbsGpuError) as e:
                call()
            assert e.value.code == ERR_UNSUPPORTED and msg in str(e.value), (kmax, nmin)
    for k in (5, 128):
        with pytest.raises(CbsGpuError) as e:
            ctx.htmaxp(np.zeros((1, k - 1)) + np.arange(k - 1), 1.0, k, 2)
        assert e.value.code == ERR_UNSUPPORTED, k
    tally = Tally()
    for kmax in (1, 25, 128):
        units = [short_unit(rng, n) for n in (kmax + 1, kmax + 2, kmax + 3, 2 * kmax + 2, 700)]
        p = SegParams(nperm=200, alpha=0.05, hybrid=True, kmax=kmax, nmin=kmax + 1, do_smooth=False, seed=kmax)
        run_split_batch(ctx, oracle, units, p, tally)


def test_cpp_shim_hybrid(oracle, tmp_path):
    """the refusals reach the C++ shim as std::runtime_error; a hybrid cbs_gpu::fndcpt with kmax <= n <= 2 kmax equals
    the oracle, engine position included"""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    exe = tmp_path / "hybrid_shim_test"
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), os.path.join(here, "cpp", "hybrid_shim_test.cpp"),
                    "-o", str(exe), "-L" + os.path.join(root, "genomic_b200"), "-l:libcbs_cuda.so",
                    "-L" + os.path.join(root, "oracle"), "-l:liboracle.so",
                    "-Wl,-rpath," + os.path.join(root, "genomic_b200"), "-Wl,-rpath," + os.path.join(root, "oracle")], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
