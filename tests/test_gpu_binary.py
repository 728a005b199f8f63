"""-m gpu: binary segmentation (ibin = true) through the device worklist against the oracle restatement (oracle/cbs_oracle.c,
pinned to the compiled reference for tmaxo(ibin=true)).  The permutations decide with the scan of binary.cuh: the decision
scan when the reject level Lstar lies above fac_max/4, the reference's ordered walk below it (DESIGN 4c)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from helpers import pack
from oracle.pyoracle import SegParams
import genomic_b200
from genomic_b200 import CbsGpuError, Params, RNG_MT19937_64, RNG_PHILOX
from genomic_b200.binding import ERR_UNSUPPORTED

pytestmark = pytest.mark.gpu


def gparams(p: SegParams, **kw) -> Params:
    return Params(alpha=p.alpha, nperm=p.nperm, min_width=p.min_width, ibin=True, undo_prune=p.undo_prune,
                  undo_prune_cutoff=p.undo_prune_cutoff, do_smooth=False, rng_mode=RNG_PHILOX if p.rng_kind else RNG_MT19937_64,
                  chain=p.chain, seed=p.seed, **kw)


def binary_unit(rng, n, kind):
    """0/1 data: piecewise Bernoulli, constant, alternating, sqrt(n)-periodic, very sparse"""
    if kind == 0:
        x = np.zeros(n)
        cuts = np.sort(rng.integers(0, n + 1, int(rng.integers(0, 4))))
        for a, b in zip(np.concatenate([[0], cuts]), np.concatenate([cuts, [n]])):
            x[a:b] = rng.random(b - a) < rng.choice([0.1, 0.3, 0.5, 0.8])
    elif kind == 1:
        x = np.full(n, float(rng.integers(0, 2)))
    elif kind == 2:
        x = (np.arange(n) % 2).astype(float)
        if n > 10:
            x[n // 3: n // 3 + max(2, n // 10)] = 1.0
    elif kind == 3:
        per = max(2, int(round(np.sqrt(n))))
        x = ((np.arange(n) // (per // 2 + 1)) % 2).astype(float)
    else:
        x = np.zeros(n)
        x[rng.integers(0, n, max(1, n // 500))] = 1.0
    return x.astype(float)


def check_split_log(got, want):
    assert len(got.splits) == len(want["log"])
    by_key = {(g["unit"], g["lo"], g["hi"]): g for g in got.splits}  # decisions are logged in order of completion
    assert len(by_key) == len(got.splits)
    for u, w in want["log"]:
        g = by_key[(u, w.lo, w.hi)]
        assert (g["called"], g["ncpt"]) == (w.called, w.ncpt), (u, w.lo, w.hi)
        if not w.called:
            continue
        assert g["ostat"] == w.ostat, (u, w.lo, w.hi)
        assert (g["iseg0"], g["iseg1"], g["perms_run"], g["nrej"], g["exit_code"]) == \
            (w.iseg0, w.iseg1, w.perms_run, w.nrej, w.exit_code), (u, w.lo, w.hi)
        if w.ncpt >= 1:
            assert g["icpt0"] == w.icpt0
        if w.ncpt == 2:
            assert g["icpt1"] == w.icpt1
        for side, want_p in ((0, w.edge_p0), (1, w.edge_p1)):
            if want_p >= 0:
                st, nrej = g[f"e_status{side}"], g[f"e_nrej{side}"]
                assert (1.0 if st == 1 else 0.0 if st == 2 else nrej / want["nperm"]) == want_p


def seq_tss(x):
    """tss of a pending segment as the reference computes it (CBS.cpp:986-989): sequential sums"""
    s = 0.0
    for v in x:
        s += v
    mean = s / len(x)
    t = 0.0
    for v in x:
        c = v - mean
        t += c * c
    return t


def reject_level(ostat, tss, n):
    """the smallest M with ostat*0.99999 <= M/(tss'/n), tss' = 1 when tss <= 1e-4 (cbs_core.h bin_reject_level)"""
    c = (1.0 if tss <= 0.0001 else tss) / n
    thresh = ostat * 0.99999
    m = max(thresh * c, 0.0)
    while m / c < thresh:
        m = np.nextafter(m, np.inf)
    while m > 0.0 and np.nextafter(m, 0.0) / c >= thresh:
        m = np.nextafter(m, 0.0)
    return m


def is_weak(lstar, n, al0):
    return not (lstar > 0.25 * (n / (al0 * (n - al0))))


@pytest.mark.parametrize("mode", ["mt_chain", "mt_unit", "philox"])
def test_binary_batch_matches_oracle(ctx, oracle, mode):
    rng = np.random.default_rng({"mt_chain": 301, "mt_unit": 302, "philox": 303}[mode])
    for trial in range(10):
        units = [binary_unit(rng, int(rng.integers(8, 6000)), int(rng.integers(0, 5))) for _ in range(int(rng.integers(1, 6)))]
        vals, off = pack(units)
        p = SegParams(nperm=int(rng.choice([50, 200, 1000])), alpha=float(rng.choice([0.01, 0.05])),
                      min_width=int(rng.choice([2, 3, 5])), ibin=True, undo_prune=bool(trial % 3 == 2), do_smooth=False,
                      rng_kind=1 if mode == "philox" else 0, chain=(mode == "mt_chain"), seed=int(rng.integers(1, 100)))
        check_batch(ctx, oracle, vals, off, p, first_batch=int(rng.choice([16, 64, 256])), max_batch=int(rng.choice([256, 2048])))


def check_batch(ctx, oracle, vals, off, p, **kw):
    lab = np.ones(len(off) - 1, np.int32)
    want = oracle.segment_units(vals, off, lab, p, want_log=True)
    want["nperm"] = p.nperm
    got = ctx.segment_batch(vals, off, gparams(p, record_splits=True, **kw))
    assert np.array_equal(got.seg_count, want["seg_count"])
    assert np.array_equal(got.lengths, want["lengths"])
    assert np.array_equal(got.means, want["means"])
    if p.rng_kind == 0:
        assert np.array_equal(got.draws, want["draws"])
    check_split_log(got, want)
    return got, want


def test_binary_weak_and_strong_reject_levels(ctx, oracle):
    """Permutations on both sides of the rule Lstar > fac_max/4 (decision scan) / Lstar <= fac_max/4 (ordered walk)."""
    rng = np.random.default_rng(311)
    units = []
    for n in (40, 60, 90, 150, 300, 800, 2000, 5000):
        units.append(binary_unit(rng, n, 0))
        units.append(binary_unit(rng, n, 4))
        x = np.zeros(n); x[rng.integers(0, n, 2)] = 1.0   # two ones: tiny statistics, weak levels
        units.append(x)
    vals, off = pack(units)
    p = SegParams(nperm=300, alpha=0.05, min_width=2, ibin=True, do_smooth=False, rng_kind=0, chain=False, seed=7)
    got, want = check_batch(ctx, oracle, vals, off, p)
    perms = {True: 0, False: 0}
    for u, w in want["log"]:
        if not w.called or w.perms_run == 0:
            continue
        seg = vals[off[u] + w.lo: off[u] + w.hi]
        lstar = reject_level(w.ostat, seq_tss(seg), w.hi - w.lo)
        perms[is_weak(lstar, w.hi - w.lo, p.min_width)] += w.perms_run
    assert perms[True] > 0 and perms[False] > 0, perms


def test_binary_tied_structures(ctx, oracle):
    """Heavily tied 0/1 patterns, where the observed location depends on the order of the reference's introsort."""
    rng = np.random.default_rng(321)
    units = []
    for n in (64, 100, 257, 1000, 2500, 4096):
        for kind in (1, 2, 3):
            units.append(binary_unit(rng, n, kind))
        x = np.tile([1.0, 1.0, 0.0, 0.0], n // 4 + 1)[:n]
        units.append(x)
    vals, off = pack(units)
    for al0 in (2, 3):
        p = SegParams(nperm=200, alpha=0.05, min_width=al0, ibin=True, do_smooth=False, rng_kind=0, chain=True, seed=3)
        check_batch(ctx, oracle, vals, off, p)
    for x in units[:8]:
        xc = x - x.mean()
        tss = float((xc * xc).sum())
        assert ctx.tmaxo(xc, tss, 2, True) == oracle.tmaxo(xc, tss, 2, True)


@pytest.mark.parametrize("mode", ["mt_unit", "philox"])
def test_binary_long_units(ctx, oracle, mode):
    rng = np.random.default_rng(331)
    a = (rng.random(70000) < 0.3).astype(float); a[30000:34000] = rng.random(4000) < 0.5
    b = (rng.random(147726) < 0.4).astype(float); b[100000:] = rng.random(47726) < 0.45
    vals, off = pack([a, b])
    p = SegParams(nperm=20, alpha=0.05, min_width=2, ibin=True, do_smooth=False, rng_kind=1 if mode == "philox" else 0,
                  chain=False, seed=4)
    check_batch(ctx, oracle, vals, off, p, first_batch=20, max_batch=20)


def untemper(y):
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
    eng = oracle.rng_mt(seed)
    oracle.lib.orc_rng_discard(C.byref(eng), skip)
    probe = oracle.rng_mt(seed)
    oracle.lib.orc_rng_discard(C.byref(probe), skip)
    outs = [oracle.lib.orc_rng_u64(C.byref(probe)) for _ in range(312)]
    return eng, np.array([untemper(v) for v in outs], dtype=np.uint64)


def test_binary_single_calls(ctx, oracle):
    rng = np.random.default_rng(341)
    for trial in range(6):
        x = binary_unit(rng, int(rng.integers(200, 3000)), trial % 5)
        p = SegParams(nperm=300, alpha=0.05, min_width=2, ibin=True, do_smooth=False, seed=9)
        eng, nxt = engine_after(oracle, 9, 777)
        wl, wm = oracle.segment(x, p, eng)
        gl, gm, draws = ctx.segment(x, gparams(p), mt_next312=nxt)
        assert np.array_equal(gl, wl) and np.array_equal(gm, wm), trial
        assert draws == eng.draws - 777
        xc = x - x.mean()
        tss = float((xc * xc).sum())
        for al0 in (2, 3):
            eng, nxt = engine_after(oracle, 5, 100)
            want = oracle.fndcpt(xc, tss, 500, 0.05, eng, ibin=True, al0=al0)
            got = ctx.fndcpt(xc, tss, Params(alpha=0.05, nperm=500, min_width=al0, ibin=True, seed=5), mt_next312=nxt)
            assert got["ostat"] == want.ostat and got["iseg"] == tuple(want.iseg), (trial, al0)
            assert (got["ncpt"], got["perms_run"], got["nrej"], got["exit_code"]) == \
                (want.ncpt, want.perms_run, want.nrej, want.exit_code), (trial, al0)
            assert got["icpt"][:want.ncpt] == tuple(want.icpt)[:want.ncpt]
            assert got["draws"] == eng.draws - 100, (trial, al0)


def test_binary_sub_batches(oracle, monkeypatch):
    rng = np.random.default_rng(351)
    units = [binary_unit(rng, n, k) for n, k in ((1500, 0), (2500, 4), (300, 2), (5200, 0), (900, 3), (3300, 0))]
    vals, off = pack(units)
    p = SegParams(nperm=300, alpha=0.05, min_width=2, ibin=True, do_smooth=False, rng_kind=0, chain=False, seed=11)
    c = genomic_b200.Context(0)
    try:
        whole = c.segment_batch(vals, off, gparams(p))
        monkeypatch.setenv("CBS_GPU_CHUNK_MARKERS", "4000")
        parts = c.segment_batch(vals, off, gparams(p))
        assert parts.rounds > whole.rounds  # it was split
        for f in ("seg_count", "lengths", "means", "draws"):
            assert np.array_equal(getattr(parts, f), getattr(whole, f)), f
        want = oracle.segment_units(vals, off, np.ones(len(units), np.int32), p)
        assert np.array_equal(whole.lengths, want["lengths"]) and np.array_equal(whole.means, want["means"])
    finally:
        c.close()


def test_binary_rejected_combinations(ctx):
    x = np.zeros(500); x[200:260] = 1.0
    w = np.ones(500)

    def unsupported(f):
        with pytest.raises(CbsGpuError) as e:
            f()
        assert e.value.code == ERR_UNSUPPORTED, e.value

    unsupported(lambda: ctx.segment(x, Params(ibin=True, hybrid=True, do_smooth=False)))
    unsupported(lambda: ctx.segment_batch(x, np.array([0, 500]), Params(ibin=True, hybrid=True, do_smooth=False)))
    unsupported(lambda: ctx.fndcpt(x - x.mean(), 1.0, Params(ibin=True, hybrid=True)))
    unsupported(lambda: ctx.segment_weighted(x, w, Params(ibin=True)))
    unsupported(lambda: ctx.segment_weighted_batch(x, w, np.array([0, 500]), Params(ibin=True)))
    unsupported(lambda: ctx.wfindcpt(x - x.mean(), w, 1.0, Params(ibin=True)))
    unsupported(lambda: ctx.htmaxp(np.stack([x - x.mean()]), 1.0, 10, 2, True))


def test_cpp_shim_binary(oracle, tmp_path):
    """cbs_gpu::segment(x, true, ...) and cbs_gpu::fndcpt(..., true, ...) of the C++ shim against liboracle, engine in/out"""
    here = os.path.dirname(os.path.abspath(__file__))
    root = os.path.dirname(here)
    exe = tmp_path / "binary_shim_test"
    subprocess.run(["g++", "-std=c++17", "-O1", "-I" + os.path.join(root, "include"), os.path.join(here, "cpp", "binary_shim_test.cpp"),
                    "-o", str(exe), "-L" + os.path.join(root, "genomic_b200"), "-l:libcbs_cuda.so",
                    "-L" + os.path.join(root, "oracle"), "-l:liboracle.so",
                    "-Wl,-rpath," + os.path.join(root, "genomic_b200"), "-Wl,-rpath," + os.path.join(root, "oracle")], check=True)
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
