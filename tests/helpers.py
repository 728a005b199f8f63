"""Shared input builders for the parity tests."""
import ctypes as C

import numpy as np


def f32(x):
    return np.asarray(x, dtype=np.float64).astype(np.float32).astype(np.float64)


def make_unit(rng, n, kind):
    if kind == 0:  # pure null
        x = rng.normal(0, 0.2, n)
    elif kind == 1:  # a few steps
        x = rng.normal(0, 0.2, n)
        for _ in range(int(rng.integers(1, 4))):
            a = int(rng.integers(0, n))
            b = int(rng.integers(a, n + 1))
            x[a:b] += rng.choice([-0.4, 0.15, 0.3, 1.0])
    elif kind == 2:  # tie heavy: integers
        x = np.round(rng.normal(0, 1, n))
    elif kind == 3:  # outlier spikes
        x = rng.normal(0, 0.2, n)
        i = rng.integers(0, n, max(1, n // 100))
        x[i] += 3
    else:  # three-valued
        x = rng.integers(0, 3, n).astype(float)
    return f32(x)


def pack(units):
    off = np.concatenate([[0], np.cumsum([len(u) for u in units])]).astype(np.int64)
    vals = np.concatenate(units) if len(units) else np.zeros(0)
    return vals, off


def same_result(a_counts, a_len, a_means, b_counts, b_len, b_means):
    return (np.array_equal(a_counts, b_counts) and np.array_equal(a_len, b_len)
            and np.array_equal(a_means, b_means))


def equal_arrays(got, want):
    """np.array_equal, where `want` may also be a stored reference result known by its digest (tests/refgolden.py)."""
    from refgolden import Digest
    if isinstance(want, Digest):
        return want.matches(got)
    return np.array_equal(got, want)


def weighted_centre(x, w):
    """centred segment and weighted tss, each sum taken in order as segment_weighted does (CBS.cpp:1053-1063)"""
    avg = np.cumsum(w * x)[-1] / np.cumsum(w)[-1]
    cur = x - avg
    return cur, float(np.cumsum(w * cur * cur)[-1])


def untemper(y):
    """mt19937_64 output -> the raw state word it was tempered from"""
    y = int(y)
    M = (1 << 64) - 1
    y ^= y >> 43
    y ^= (y << 37) & 0xFFF7EEE000000000 & M
    z = y
    for _ in range(4):
        z = y ^ ((z << 17) & 0x71D67FFFEDA60000 & M)
    y = z
    z = y
    for _ in range(3):
        z = y ^ ((z >> 29) & 0x5555555555555555)
    return z


def engine_after(oracle, seed, skip):
    """an oracle engine that has already handed out `skip` draws, and the same engine as its next 312 raw words (the
    caller-owned engine state of the single-call entry points)"""
    eng = oracle.rng_mt(seed)
    oracle.lib.orc_rng_discard(C.byref(eng), skip)
    probe = oracle.rng_mt(seed)
    oracle.lib.orc_rng_discard(C.byref(probe), skip)
    outs = [oracle.lib.orc_rng_u64(C.byref(probe)) for _ in range(312)]
    return eng, np.array([untemper(v) for v in outs], dtype=np.uint64)


def gparams(p, **kw):
    """genomic_b200.Params carrying the options of an oracle SegParams; kw sets the device-only knobs or overrides"""
    from genomic_b200 import Params, RNG_MT19937_64, RNG_PHILOX
    args = dict(alpha=p.alpha, nperm=p.nperm, hybrid=p.hybrid, min_width=p.min_width, kmax=p.kmax, nmin=p.nmin, eta=p.eta,
                tol=p.tol, ibin=p.ibin, undo_prune=p.undo_prune, undo_prune_cutoff=p.undo_prune_cutoff, do_smooth=p.do_smooth,
                smooth_region=p.smooth_region, outlier_sd_scale=p.outlier_sd_scale, smooth_sd_scale=p.smooth_sd_scale,
                trim=p.trim, rng_mode=RNG_PHILOX if p.rng_kind else RNG_MT19937_64, chain=p.chain, seed=p.seed)
    args.update(kw)
    return Params(**args)


def check_edge_p(status, nrej, want_p, nperm, msg):
    """tpermp p-values of both boundaries: the device reports the rejection counts and the shortcut status"""
    for side in (0, 1):
        if want_p[side] < 0:
            continue  # not run
        got_p = 1.0 if status[side] == 1 else 0.0 if status[side] == 2 else nrej[side] / nperm
        assert got_p == want_p[side], (msg, side, status, nrej, want_p)


def check_split_log(got, want, p, exact_draws):
    """Every logged decision of the device equals the oracle's, matched by (unit, lo, hi): observed statistic and arc,
    change points, permutation counts, exit code and both edge p-values.  Returns the decisions that called fndcpt as
    (unit, oracle record, device record)."""
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    if p.hybrid:  # means of hybrid runs are compared to 1e-9 (DESIGN 2)
        assert np.allclose(got.means, want["means"], rtol=1e-9, atol=0)
    else:
        assert np.array_equal(got.means, want["means"])
    if exact_draws:
        assert np.array_equal(got.draws, want["draws"])
    assert len(got.splits) == len(want["log"])
    by_key = {(g["unit"], g["lo"], g["hi"]): g for g in got.splits}  # decisions are logged in order of completion
    assert len(by_key) == len(got.splits)
    called = []
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
        called.append((u, w, g))
    return called
