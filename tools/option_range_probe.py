"""Wide smoothing windows and hybrid kmax above 128 on the GPU: time per call.

  python tools/option_range_probe.py [--reps 3] [--nperm 1000] [--out FILE]

* Smoothing: one SNP6-scale synthetic sample (genomic_b200.synth, 23 chromosomes, 1.8 M markers, sparse outliers),
  cbs_gpu_smooth with the chromosome labels at smooth_region 10 / 64 (k_sm_window) and 65 / 100 / 1000 (k_sm_run_*,
  k_sm_wide, k_sm_median).  Then the all-outliers input: 200 000 markers of alternating +-5 on a slow ramp with
  outlier_sd_scale 1e-6, so that every marker scans its whole window, at smooth_region 65 / 1000 / 10 000 / 10^6 (the
  last one wider than the input: every window is the whole vector, n^2 = 4e10 neighbour reads).
  Each smoothing configuration is reported twice: the whole call (host clock, copies included) and the device time of the
  smoothing kernels alone (CUDA events around every launch, cbs_gpu_set_profiling bit 0, summed by cbs_gpu_last_kernel_ms
  under "smooth": compaction, differences, sorts, trimmed SD and the window stage; the copies are not in it), in a
  separate pass so that the events do not slow the first.
* Hybrid segmentation of the same sample (unsmoothed values, one unit per chromosome, MT replay with one engine per unit,
  alpha 0.01, --nperm permutations) at kmax 25 / 128 (k_hscan<false>) and 129 / 500 / 1000 (k_hscan<true>), nmin =
  max(200, kmax + 1).
Each configuration: one warm-up call, then --reps calls timed with a host clock around the call (every call ends in a
device synchronise); the median is reported.  The card's name and power limit are read in the same process.  Writes one
JSON line to stdout (and to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 3) for t in ts]


def kernel_ms(ctx, fn, reps):
    """median over reps of the summed event time of the smoothing kernels of one call"""
    ctx.set_profiling(events=True)
    fn()
    ts = []
    for _ in range(reps):
        fn()
        ts.append(ctx.last_kernel_ms()["smooth"])
    ctx.set_profiling(False)
    return float(np.median(ts)), [round(t, 3) for t in ts]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--nperm", type=int, default=1000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import genomic_b200
    from genomic_b200 import Params, RNG_MT19937_64, synth
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()[0]
    ctx = genomic_b200.Context(0)
    vals, off, lab, ids = synth.cohort([0], scale=1.0, outliers=True)
    x = vals.astype(np.float64)
    chrom = np.repeat(lab, np.diff(off)).astype(np.int32)
    res = {"card": card, "markers": int(len(x)), "reps": a.reps, "smooth_ms": {}, "smooth_kernel_ms": {},
           "hybrid_ms_per_sample": {}}
    for r in (10, 64, 65, 100, 1000):
        res["smooth_ms"][f"snp6_R{r}"] = timed(lambda: ctx.smooth(x, chrom, r), a.reps)
        res["smooth_kernel_ms"][f"snp6_R{r}"] = kernel_ms(ctx, lambda: ctx.smooth(x, chrom, r), a.reps)
    n = 200000
    alt = np.where(np.arange(n) % 2 == 0, 5.0, -5.0) + 1e-3 * np.arange(n)
    one = np.ones(n, np.int32)
    for r in (65, 1000, 10000, 10 ** 6):
        res["smooth_ms"][f"all_outliers_200k_R{r}"] = timed(lambda: ctx.smooth(alt, one, r, outlier_sd_scale=1e-6), a.reps)
        res["smooth_kernel_ms"][f"all_outliers_200k_R{r}"] = kernel_ms(ctx, lambda: ctx.smooth(alt, one, r, outlier_sd_scale=1e-6), a.reps)
    for kmax in (25, 128, 129, 500, 1000):
        p = Params(nperm=a.nperm, alpha=0.01, hybrid=True, kmax=kmax, nmin=max(200, kmax + 1), do_smooth=False,
                   rng_mode=RNG_MT19937_64, chain=False, seed=1)
        segs = []
        res["hybrid_ms_per_sample"][f"kmax{kmax}"] = timed(lambda: segs.append(len(ctx.segment_batch(vals, off, p, unit_ids=ids).lengths)), a.reps)
        res["hybrid_ms_per_sample"][f"kmax{kmax}_segments"] = segs[-1]
    ctx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
