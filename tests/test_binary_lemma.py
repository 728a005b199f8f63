"""The rule behind the decision scan of binary permutations (genomic_b200/csrc/binary.cuh k_scan_binary, DESIGN 4c), checked on
the oracle without a GPU: when the reject level Lstar exceeds fac_max/4, the reference's permutation statistic reaches the
threshold iff the seed arc or an arc inside the bands of a block pair whose bound reaches Lstar does, in any visiting order."""
import math

import numpy as np

from test_gpu_binary import is_weak, reject_level


def lround(v):
    return int(math.floor(v + 0.5))


def decision_by_rule(px, lstar, al0):
    """seed >= Lstar, or some arc of a pair with bsslim >= Lstar, inside its bands, with fac*(|d|-0.5)^2 >= Lstar"""
    n = len(px)
    rn = float(n)
    sx = np.concatenate([[0.0], np.cumsum(px)])          # np.cumsum adds sequentially, as the reference does
    nb = lround(math.sqrt(n)) if n >= 50 else 1
    bb = [lround(rn * (b / nb)) for b in range(nb + 1)]
    bmin, bmax, amin, amax = [], [], [], []
    for b in range(1, nb + 1):
        seg = sx[bb[b - 1] + 1: bb[b] + 1]
        bmin.append(seg.min()); bmax.append(seg.max())
        amin.append(bb[b - 1] + 1 + int(np.argmin(seg))); amax.append(bb[b - 1] + 1 + int(np.argmax(seg)))
    lo = min(bmin); hi = max(bmax)
    gmin, gimin = (lo, amin[bmin.index(lo)]) if lo < 0.0 else (0.0, n)
    gmax, gimax = (hi, amax[bmax.index(hi)]) if hi > 0.0 else (0.0, n)
    spread = gmax - gmin
    if spread <= 0.0:
        return False
    rj = float(abs(gimax - gimin))
    if rn / (rj * (rn - rj)) * ((spread - 0.5) * (spread - 0.5)) >= lstar:
        return True
    for bi in range(1, nb + 1):
        for bj in range(bi, nb + 1):
            ilo, ihi, jlo, jhi = bb[bi - 1] + 1, bb[bi], bb[bj - 1] + 1, bb[bj]
            lenhi = min(jhi - ilo, n - al0)
            lenlo = max(1 if bi == bj else jlo - ihi, al0)
            s1 = abs(bmax[bj - 1] - bmin[bi - 1]); s2 = abs(bmax[bi - 1] - bmin[bj - 1])
            smax = max(s1, s2)
            rlo, rhi = float(lenlo), float(lenhi)
            bsslim = rn / min(rlo * (rn - rlo), rhi * (rn - rhi)) * ((smax - 0.5) * (smax - 0.5))
            if not bsslim >= lstar:
                continue
            clen = abs(amax[bj - 1] - amin[bi - 1]) if s1 > s2 else abs(amin[bj - 1] - amax[bi - 1])
            lenmax = min(clen, n - clen)
            lengths = []
            if lenlo <= rn / 2 and lenlo <= lenmax:
                lengths += range(lenlo, lenmax + 1)
            if lenhi >= rn / 2 and lenhi >= n - lenmax:
                lengths += range(n - lenmax, lenhi + 1)
            for L in lengths:
                i = np.arange(ilo + max(0, jlo - ilo - L), ihi - max(0, ihi + L - jhi) + 1)
                if len(i) == 0:
                    continue
                d = np.abs(sx[i + L] - sx[i])
                rr = float(L)
                if np.any(rn / (rr * (rn - rr)) * ((d - 0.5) * (d - 0.5)) >= lstar):
                    return True
    return False


def test_decision_rule_matches_oracle_permutations(oracle):
    rng = np.random.default_rng(401)
    checked = agree = 0
    while checked < 1500:
        n = int(rng.integers(20, 700))
        al0 = int(rng.choice([2, 3, 5]))
        x = (rng.random(n) < rng.choice([0.05, 0.2, 0.5])).astype(float)
        if rng.random() < 0.5:
            a = int(rng.integers(0, n)); x[a: a + int(rng.integers(1, n))] = rng.random() < 0.5
        xc = x - x.mean()
        tss = float((xc * xc).sum())
        ostat = oracle.tmaxo(xc, tss, al0, True)[0]
        # thresholds around the observed value, as the permutations of a max-t test see them
        for scale in (1.0, 0.3):
            o = ostat * scale
            if not o > 0.0:
                continue
            lstar = reject_level(o, tss, n)
            if is_weak(lstar, n, al0):
                continue
            for _ in range(3):
                px = rng.permutation(xc)
                want = o * 0.99999 <= oracle.tmaxp(px, tss, al0, True)
                assert decision_by_rule(px, lstar, al0) == want, (n, al0, o)
                checked += 1
                agree += want
    assert 0 < agree < checked  # both outcomes occur
