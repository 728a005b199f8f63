"""Long units on the GPU: read-depth-like samples in 100-bp bins.

  python tools/long_unit_probe.py [--samples 1] [--reps 2] [--nperm 10000] [--out FILE]

* Samples: 24 chromosomes at the GRCh38 lengths in 100-bp bins (2.49 M markers for chromosome 1, 30.9 M in all), a
  seeded log-ratio-like signal: noise, copy-number segments of 2 kb to 40 Mb, sparse outliers.  MT replay with one engine
  per unit (chain = 0), nperm 10 000, alpha 0.01, smoothing on.  Per sample: one warm-up call, `--reps` timed calls
  (host clock around the call, which ends in a device synchronise), then one call with every kernel serialised on one
  stream and event-timed (cbs_gpu_set_profiling bit 2 | bit 0) for the per-kernel split.
The card's name and power limit are read in the same process.  Writes one JSON line to stdout (and to --out)."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

GRCH38 = (248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422,
          135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167,
          46709983, 50818468, 156040895, 57227415)


def read_depth_sample(seed):
    rng = np.random.default_rng(seed)
    chunks, off = [], [0]
    for c, bp in enumerate(GRCH38):
        n = bp // 100
        x = rng.normal(0.0, 0.25, n)
        for _ in range(int(rng.integers(2, 12))):
            ln = int(min(n, np.exp(rng.uniform(np.log(20), np.log(400000)))))
            a = int(rng.integers(0, n - ln + 1))
            x[a:a + ln] += float(rng.choice([-1.0, -0.4, -0.2, 0.15, 0.3, 0.58]))
        k = rng.integers(0, n, n // 5000)
        x[k] += rng.normal(0, 2.0, len(k))
        chunks.append(x.astype(np.float32))
        off.append(off[-1] + n)
    return np.concatenate(chunks), np.asarray(off, dtype=np.int64)


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", type=int, default=1)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--nperm", type=int, default=10000)
    ap.add_argument("--out")
    args = ap.parse_args()
    import genomic_b200
    from genomic_b200 import Params, RNG_MT19937_64

    ctx = genomic_b200.Context(0)
    res = {"card": card(), "samples": []}

    def emit():
        line = json.dumps(res)
        if args.out:
            with open(args.out, "w") as f:
                f.write(line + "\n")
        return line

    # ---- whole samples ---------------------------------------------------------------------------------------------
    gp = Params(nperm=args.nperm, alpha=0.01, rng_mode=RNG_MT19937_64, chain=False, seed=1)
    for s in range(args.samples):
        vals, off = read_depth_sample(100 + s)
        ids = np.arange(len(off) - 1, dtype=np.uint64) + 24 * s
        t0 = time.perf_counter()
        r = ctx.segment_batch(vals, off, gp, unit_ids=ids)
        first = time.perf_counter() - t0
        secs = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            r = ctx.segment_batch(vals, off, gp, unit_ids=ids)
            secs.append(round(time.perf_counter() - t0, 3))
        ctx.set_profiling(events=True, serial=True)
        ctx.segment_batch(vals, off, gp, unit_ids=ids)
        split = {k: round(v, 1) for k, v in ctx.last_kernel_ms().items()}
        ctx.set_profiling()
        row = {"sample": s, "markers": int(off[-1]), "largest_unit": int(np.diff(off).max()), "first_call_s": round(first, 3),
               "call_s": secs, "segments": int(len(r.lengths)), "rounds": r.rounds, "perms_run": r.perms_run,
               "perm_elements": r.perm_elems, "serialised_kernel_ms": split}
        res["samples"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        emit()
    ctx.close()
    print(emit())


if __name__ == "__main__":
    main()
