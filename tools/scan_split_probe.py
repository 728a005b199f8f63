"""Where the scan time of the bench sample goes: observed rows (k_scan_obs) against permutation rows (k_scan_perm), and
what the shuffles cost when the observed scan runs beside them.

  python tools/scan_split_probe.py [--root TREE] [--reps 3] [--out FILE]

For each repetition, after two warm-up calls on one synthetic SNP6-scale sample (MT replay, nperm 10 000):
  * serialised: every kernel on one stream (as in bench.py's profile pass) with the per-round timeline
    (CBS_GPU_DEBUG_ROUNDS).  Where a round shows two scan launches, the earlier one is the observed scan; a lone scan
    launch is the observed scan if it starts where the round's prep ends (within 0.02 ms), else the permutation scan.  The
    timeline leaves out launches shorter than 0.05 ms, so the split covers slightly less than the scan total, which is
    printed next to it.
  * overlapped: the normal stream layout with event timing.  The shuffle kernels' summed event time there, set against the
    serialised one, is what running beside other kernels (the prep stream, and in this build the observed scan) costs them.
--root loads the package of another source tree (a build of the parent commit) for an A/B in the same session; in a tree
with a single scan kernel that launch holds both kinds of rows and is counted by the same rule.
Writes one JSON line to stdout (and to --out)."""
import argparse
import json
import os
import re
import sys
import tempfile

SHUF = ("perm", "shuf0", "shuf1", "shuf2", "shuf3")


def split_timeline(text):
    obs = perm = 0.0
    for line in text.splitlines():
        if not line.startswith("[round"):
            continue
        ent = [(k, float(a), float(d)) for k, a, d in re.findall(r" (\w+)=([\d.]+)\+([\d.]+)", line)]
        prep_end = [a + d for k, a, d in ent if k == "prep"]
        later = [a for k, a, d in ent if k in SHUF or k == "prefix"]
        first_later = min(later) if later else float("inf")
        scans = sorted((a, d) for k, a, d in ent if k == "scan")
        if len(scans) == 2:  # observed scan first (prep stream), permutation scan behind the chain
            obs += scans[0][1]
            perm += scans[1][1]
        elif scans:
            a, d = scans[0]
            if any(abs(a - e) < 0.02 for e in prep_end) or (not prep_end and a < first_later):
                obs += d
            else:
                perm += d
    return obs, perm


def call_with_stderr(fn):
    """run fn() with the process's stderr (fd 2, where the library writes its timeline) captured"""
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+b") as tmp:
        os.dup2(tmp.fileno(), 2)
        try:
            r = fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        tmp.seek(0)
        return r, tmp.read().decode(errors="replace")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--root", default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    sys.path.insert(0, os.path.abspath(args.root))
    import genomic_b200
    from genomic_b200 import Params, RNG_MT19937_64, synth

    ctx = genomic_b200.Context(0)
    vals, off, lab, ids = synth.cohort([0])
    gp = Params(nperm=10000, rng_mode=RNG_MT19937_64, chain=False, seed=1)
    for _ in range(2):
        ctx.segment_batch(vals, off, gp, unit_ids=ids)
    reps = []
    for _ in range(args.reps):
        os.environ["CBS_GPU_DEBUG_ROUNDS"] = "1"
        ctx.set_profiling(events=True, serial=True)
        _, text = call_with_stderr(lambda: ctx.segment_batch(vals, off, gp, unit_ids=ids))
        ser = ctx.last_kernel_ms()
        del os.environ["CBS_GPU_DEBUG_ROUNDS"]
        ctx.set_profiling(events=True)
        ctx.segment_batch(vals, off, gp, unit_ids=ids)
        ovl = ctx.last_kernel_ms()
        ctx.set_profiling()
        obs, perm = split_timeline(text)
        reps.append({"serialised_scan_ms": round(ser["scan"], 3), "serialised_scan_obs_ms": round(obs, 3),
                     "serialised_scan_perm_ms": round(perm, 3),
                     "serialised_shuffle_ms": round(sum(ser[k] for k in SHUF), 3),
                     "overlapped_shuffle_ms": round(sum(ovl[k] for k in SHUF), 3),
                     "overlapped_prefix_ms": round(ovl["prefix"], 3), "serialised_prefix_ms": round(ser["prefix"], 3)})
    ctx.close()
    line = json.dumps({"root": os.path.abspath(args.root), "reps": reps})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
