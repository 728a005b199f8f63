"""Binary segmentation (ibin = true) on the B200: one run, written to profiles/binary_probe.json (or --out).

Cohort: the synthetic SNP6-shaped samples of genomic_b200.synth (23 chromosomes, SURVEY Appendix C sizes), made binary as
(value > 0), so that the copy-number steps of the synthetic data become steps of a Bernoulli rate.  nperm 10 000, alpha 0.01,
MT replay with one engine per unit (chain = 0), no smoothing.  Reported, with the card's name and power limit read in the
same run:
  * ms per sample at 1 and 16 samples per call, next to the same samples as continuous data (float32 values, ibin = false);
  * the share of max-t permutations that took the ordered walk (reject level Lstar <= fac_max/4), from the split log with
    each segment's tss recomputed on the host with sequential sums;
  * the scan time of round 0 (the observed scans of the 23 roots), from a call with nperm = 0 and per-launch events.
Timing: warm-up calls of every shape first, then the host clock around calls that end in a device synchronise."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import genomic_b200  # noqa: E402
from genomic_b200 import Params, RNG_MT19937_64, synth  # noqa: E402


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception as e:  # the measurement itself needs the device, the label does not
        return f"unknown ({e})"


def params(ibin, nperm=10000, **kw):
    return Params(nperm=nperm, alpha=0.01, ibin=ibin, do_smooth=False, rng_mode=RNG_MT19937_64, chain=False, seed=1, **kw)


def timed(ctx, vals, off, ids, p, reps):
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = ctx.segment_batch(vals, off, p, unit_ids=ids)  # returns after the device synchronised (results are on the host)
        ms.append((time.perf_counter() - t0) * 1e3)
    return ms, r


def seq_tss(x):
    """the reference's tss of a pending segment: sequential mean, centring, sequential sum of squares (np.cumsum adds in order)"""
    mean = np.cumsum(x)[-1] / len(x)
    c = x - mean
    return float(np.cumsum(c * c)[-1])


def reject_level(ostat, tss, n):
    c = (1.0 if tss <= 0.0001 else tss) / n
    thresh = ostat * 0.99999
    m = max(thresh * c, 0.0)
    while m / c < thresh:
        m = np.nextafter(m, np.inf)
    while m > 0.0 and np.nextafter(m, 0.0) / c >= thresh:
        m = np.nextafter(m, 0.0)
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "binary_probe.json"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink every chromosome (rehearsal only)")
    a = ap.parse_args()
    ctx = genomic_b200.Context(0)
    res = {"card": card(), "nperm": 10000, "alpha": 0.01, "rng": "mt replay, chain=0", "reps": a.reps}
    for spc in (1, 16):
        vals, off, lab, ids = synth.cohort(range(spc), scale=a.scale)
        bvals = (vals > 0).astype(np.float32)
        row = {"markers": int(off[-1])}
        for name, v, ibin in (("binary", bvals, True), ("continuous", vals, False)):
            timed(ctx, v, off, ids, params(ibin), 1)  # warm-up of this shape
            ms, r = timed(ctx, v, off, ids, params(ibin), a.reps)
            row[name] = {"ms_per_call": ms, "ms_per_sample_median": float(np.median(ms)) / spc, "segments": int(len(r.lengths)),
                         "perms_run": int(r.perms_run), "rounds": int(r.rounds)}
        res[f"samples_per_call_{spc}"] = row
    # fallback share, from the split log of one sample
    vals, off, lab, ids = synth.cohort([0], scale=a.scale)
    x = (vals > 0).astype(np.float64)
    r = ctx.segment_batch(x, off, params(True, record_splits=True), unit_ids=ids)
    weak = strong = 0
    for s in r.splits:
        if not s["called"] or s["perms_run"] == 0:
            continue
        n = s["hi"] - s["lo"]
        seg = x[off[s["unit"]] + s["lo"]: off[s["unit"]] + s["hi"]]
        lstar = reject_level(s["ostat"], seq_tss(seg), n)
        if lstar > 0.25 * (n / (2.0 * (n - 2.0))):
            strong += s["perms_run"]
        else:
            weak += s["perms_run"]
    res["ordered_walk_permutations"] = weak
    res["decision_scan_permutations"] = strong
    res["ordered_walk_share"] = weak / max(1, weak + strong)
    # round 0: observed scans of the 23 roots (nperm = 0: nothing else runs in the scan slot)
    ctx.set_profiling(events=True)
    obs = []
    for _ in range(1 + a.reps):
        ctx.segment_batch(x, off, params(True, nperm=0), unit_ids=ids)
        obs.append(ctx.last_kernel_ms()["scan"])
    ctx.set_profiling(events=False)
    res["observed_scan_round0_ms"] = obs[1:]
    res["observed_scan_round0_largest_unit"] = int(np.diff(off).max())
    ctx.close()
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
