#!/usr/bin/env python
"""bench.py -- CBS markers*samples segmented per second (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo, N B200s of one node
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU code (oracle/_ref)

A "step" segments one batch of synthetic SNP6-scale input end to end (smoothing + CBS):
N=1 runs BASELINE.json configs[1] -- ONE synthetic sample, 1.8M markers over 23 chromosomes,
10k permutations, alpha 0.01, full-permutation p-values.  With N ranks every rank segments its own
sample(s) (weak scaling, the cohort shards by sample, no data-path collective) and the segment
tables are gathered at the end of the step.

One JSON line on rank 0.  `value` = device-resident input (float32 already in HBM when the timed
region starts); `e2e` = the same step through the C-ABI call with pinned HOST buffers (H2D copy of
the values and D2H of the segment table inside the timed region).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "cbs_markers_samples_per_sec"
UNIT = "markers*samples/s"
NPERM = 10000
ALPHA = 0.01


def workload_name(samples_per_gpu: int, scale: float) -> str:
    m = int(round(1800000 * scale))
    return (f"configs[1]: {samples_per_gpu} synthetic SNP6-scale sample(s) per GPU, {m} markers x 23 chromosomes, "
            f"nperm={NPERM}, alpha={ALPHA}, smoothing on, full-permutation p-values")


# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons during the timed region (B200_PROFILING.md recipe).  Sampled through NVML in a
    thread (nvidia_ml_py): a polling `nvidia-smi -lms` process contends for the driver with the ~500 kernel launches
    of a step and was measured to stretch single steps by up to 60 %; NVML queries do not.  Falls back to the
    nvidia-smi loop if NVML is not importable."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.sm, self.mx, self.reasons = [], [], set()
        self.stop_flag = False
        self.thread = None
        self.nvml = None

    def _nvml_loop(self):
        nv = self.nvml
        try:
            h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            names = (("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                     ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                     ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                     ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap))
            while not self.stop_flag:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.mx.append(mx)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for name, bit in names:
                    if r & bit:
                        self.reasons.add(name)
                time.sleep(0.1)
        except Exception:
            pass

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            # NVML indexes physical devices: honour CUDA_VISIBLE_DEVICES if it is a plain list of indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                self.gpu = int(vis.split(",")[self.gpu])
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "500", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.nvml is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": max(self.mx) if self.mx else None,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def read_peaks() -> dict:
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": float(d.get("hbm_gbs", 6650.0)), "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


# ---------------------------------------------------------------------------------------------
def cpu_reference_run(nperm: int, threads: int, sample: int = 0):
    """One step of the bench workload on the host: the reference's own lib/cbs (oracle/_ref, the unmodified sources) on ALL 23
    chromosomes of the synthetic sample -- smoothing + CBS per chromosome, one std::mt19937_64(1) per unit (what the GPU arm's
    MT replay reproduces), units handed out largest first to `threads` host threads.  Returns (markers, seconds, kind, threads)."""
    from genomic_b200 import synth
    from oracle.pyoracle import Oracle, Ref, SegParams
    vals, off, lab, _ = synth.cohort([sample], scale=1.0)
    p = SegParams(nperm=nperm, alpha=ALPHA, do_smooth=True, rng_kind=0, chain=False, seed=1)
    x = vals.astype(np.float64)
    if Ref.available():
        eng, kind = Ref(), "reference"
        threads = max(1, min(threads, len(off) - 1))  # a unit is the grain: no more threads than units can be busy
        t0 = time.perf_counter()
        eng.segment_units(x, off, lab, p, nthreads=threads)
        dt = time.perf_counter() - t0
    else:  # reference sources were never available on this box: time the C restatement instead
        eng, kind = Oracle(), "port"
        threads = 1
        t0 = time.perf_counter()
        eng.segment_units(x, off, lab, p)
        dt = time.perf_counter() - t0
    return int(off[-1]), dt, kind, threads


CPU_SAMPLE = ("the whole synthetic sample 0 (all 23 chromosomes, 1,800,000 markers): the workload of one step of this bench; "
              "chromosomes are handed to the host threads largest first, the longest chromosome bounds the wall time")
CPU_BUDGET_S = 200.0  # the reference arm stops adding steps when the next one would pass this


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return  # rank 0 alone runs and prints the reference arm
    threads = os.cpu_count() or 1
    times = []
    markers, kind, used = 0, "reference", threads
    # one step takes the reference about 100 s on 16 cores, so the requested warm-up is dropped (CPU code has none to do) and
    # steps are added only while they fit the time budget; `steps` in the line is the number actually timed
    while len(times) < max(1, args.steps):
        markers, dt, kind, used = cpu_reference_run(NPERM, threads, sample=0)
        times.append(dt)
        if sum(times) + dt > CPU_BUDGET_S:
            break
    total = sum(times)
    value = markers * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": 0, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(1, 1.0), "rng": "mt", "chain": False, "samples_per_gpu": 1,
                   "note": f"requested steps {args.steps} / warmup {args.warmup}; timed {len(times)} step(s) of ~{total / len(times):.0f} s "
                           f"within a {CPU_BUDGET_S:.0f} s budget"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": kind, "sample": CPU_SAMPLE},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, res, table: np.ndarray) -> None:
    """What one timed step hands its caller, as float64 .npy files, so that two builds can be compared output for output:
    this rank's BatchResult (segment offsets per unit, segment lengths and means, RNG draws consumed per unit) and the
    gathered segment table of all ranks (rows: global unit id, length, mean).  Past 64 MB in all, every array keeps the
    same share of its rows, chosen by a fixed seed."""
    arrays = {"seg_offsets": res.seg_offsets, "lengths": res.lengths, "means": res.means, "draws": res.draws,
              "segment_table": table}
    arrays = {k: np.asarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(out_dir, exist_ok=True)
    room = DUMP_LIMIT_BYTES - 4096  # .npy headers
    for name, a in arrays.items():
        if total > room:
            keep = int(len(a) * room // total)
            a = a[np.sort(np.random.default_rng(0).choice(len(a), keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ---------------------------------------------------------------------------------------------
def run_gpu_arm(args):
    import torch
    import genomic_b200
    from genomic_b200 import Params, RNG_MT19937_64, RNG_PHILOX, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    ctx = genomic_b200.Context(local_rank)  # raises if libcbs_cuda.so or the device is missing
    stream = torch.cuda.current_stream(dev)
    ctx.set_stream(stream.cuda_stream)

    S = args.samples_per_gpu
    from genomic_b200.shard import samples_of_rank
    my_samples = samples_of_rank(S * world, rank, world)  # global sample ids: results do not depend on the sharding
    vals, off, lab, ids = synth.cohort(my_samples, scale=args.scale)
    markers_rank = int(off[-1])
    rng_mode = RNG_PHILOX if args.rng == "philox" else RNG_MT19937_64
    gp = Params(alpha=ALPHA, nperm=NPERM, rng_mode=rng_mode, chain=False, seed=1, hybrid=bool(args.hybrid))

    host_pinned = torch.from_numpy(vals).pin_memory()
    d_vals = host_pinned.to(dev, non_blocking=False)
    l2_flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    from genomic_b200 import shard

    gather_cap = 64 * 24 * max(1, S)  # rows per rank of the one fixed-capacity all_gather (same on every rank)

    def gather_tables(res):
        """the only cross-GPU step: gather of the per-rank segment tables (ONE NCCL all_gather, one D2H copy)"""
        tab = shard.pack_table(res.seg_count, res.lengths, res.means, ids)
        gather_tables.last = shard.gather_tables(tab, dist, dev, capacity=gather_cap)
        return gather_tables.last.shape[0]

    local_done = {"ev": None}  # recorded when this rank's own samples are segmented, before the collective

    def mark_local():
        ev = torch.cuda.Event(enable_timing=True)
        ev.record(stream)
        local_done["ev"] = ev

    def step_device():
        r = ctx.segment_batch(None, off, gp, unit_ids=ids, device_ptr=d_vals.data_ptr(), dtype=genomic_b200.binding.F32)
        mark_local()
        gather_tables(r)
        return r

    def step_host():
        r = ctx.segment_batch(host_pinned.numpy(), off, gp, unit_ids=ids)
        mark_local()
        gather_tables(r)
        return r

    def timed(fn, steps, warmup, sample_clocks=False):
        for _ in range(warmup):
            fn()
        sampler = ClockSampler(local_rank) if sample_clocks else None
        per_step = []
        local = []
        last = None
        barrier()
        if sampler:
            sampler.start()
        for _ in range(steps):
            l2_flush.zero_()
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            e0.record(stream)
            last = fn()
            e1.record(stream)
            torch.cuda.synchronize(dev)
            per_step.append(e0.elapsed_time(e1))
            local.append(e0.elapsed_time(local_done["ev"]))
        barrier()
        clocks = sampler.stop() if sampler else None
        total_ms = float(sum(per_step))
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)  # max over ranks
        timed.last_steps = [round(x, 3) for x in per_step]  # this rank's per-step times (diagnostics)
        timed.last_local = [round(x, 3) for x in local]     # ... without the gather of the tables (the ranks' own work)
        return float(t.item()), last, clocks

    warm = max(args.warmup, 3) if not args.cohort_run else args.warmup
    total_ms, res, clocks = timed(step_device, args.steps, warm, sample_clocks=True)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, gather_tables.last)
    steps_device = timed.last_steps
    local_device = timed.last_local
    e2e_ms, res_h, _ = timed(step_host, args.steps, 0 if args.cohort_run else max(args.warmup, 3))
    steps_host = timed.last_steps
    launches_per_step = int(res.kernel_launches)
    full_table = gather_tables.last

    if args.cohort_run:
        # The north-star run (BASELINE configs[3]): a cohort sharded by sample over the ranks, timed end to end, with the
        # per-rank times (load balance) and the parity subset: the subset samples are segmented once more in ONE call on rank 0
        # (that call is what tests/test_gpu_fullsize.py::test_config4 compares with the compiled reference, log under profiles/)
        # and must agree row for row with what the sharded run produced for them.
        # per rank: the time of its own samples, taken BEFORE the collective (the step time is the same on every rank: the
        # all_gather waits for the slowest)
        rank_ms = torch.tensor([sum(local_device) / len(local_device)], device=dev, dtype=torch.float64)
        all_ms = [torch.zeros_like(rank_ms) for _ in range(world)]
        if dist is not None:
            dist.all_gather(all_ms, rank_ms)
        else:
            all_ms = [rank_ms]
        per_rank = [float(t.item()) for t in all_ms]
        if rank == 0:
            total = S * world
            subset = shard.parity_subset(total)
            sv, so, sl, sid = synth.cohort(subset, scale=args.scale)
            rs = ctx.segment_batch(sv, so, gp, unit_ids=sid)
            want = shard.pack_table(rs.seg_count, rs.lengths, rs.means, sid)
            keep = np.isin(full_table[:, 0], np.asarray(sid, dtype=np.float64))
            got = full_table[keep]
            order = np.lexsort((np.arange(len(got)), got[:, 0]))
            same = bool(got.shape == want.shape and np.array_equal(got[order], want))
            markers_total = markers_rank * world
            line = {
                "metric": METRIC, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
                "value": markers_total * args.steps / (total_ms * 1e-3), "ms_per_step": total_ms / args.steps,
                "e2e": {"value": markers_total * args.steps / (e2e_ms * 1e-3), "unit": UNIT, "ms_per_step": e2e_ms / args.steps,
                        "h2d_bytes_per_step": int(vals.nbytes) * world,
                        "d2h_bytes_per_step": int(len(res_h.lengths) * 12 + len(off) * 16) * world},
                "config": {"workload": workload_name(S, args.scale), "rng": args.rng, "chain": False, "samples": total,
                           "parallelism": f"sample-sharded x{world}, one all_gather of the segment tables"},
                "per_rank_local_ms_per_step": [round(x, 1) for x in per_rank],
                "max_over_mean_rank_time": max(per_rank) / (sum(per_rank) / len(per_rank)),
                "segments": int(full_table.shape[0]), "perms_run_rank0": int(res.perms_run), "rounds_rank0": int(res.rounds),
                "parity_subset": {"samples": subset, "rows": int(want.shape[0]), "sharded_equals_single_call": same,
                                  "reference": "the same single call equals the compiled reference bit for bit: "
                                               "tests/test_gpu_fullsize.py::test_config4_sixteen_sample_subset_vs_reference, "
                                               "profiles/r02_fullsize_slow.log"},
                "clocks": clocks, "higher_is_better": True, "scaling": "weak", "dtype": "f64", "data": "synthetic",
            }
            print(json.dumps(line), flush=True)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        ctx.close()
        return

    # Roofline inputs, kept OUT of the timed steps:
    #  (1) the same K steps once more with every kernel launch bracketed by CUDA events, ALL kernels on the one
    #      stream (the timed steps overlap independent kernels on side streams) -> per-kernel device time (sum over
    #      launches) on a serialised time base: the groups add up to the serialised step, none can exceed it;
    #  (2) one step with the scan kernel's work counters on (device atomics slow that kernel, so this
    #      step is never timed) -> arcs examined = the kernel's algorithmic work.
    ctx.set_profiling(events=True, serial=True)  # one stream: the per-kernel event times do not overlap
    kms = None
    prof_ms = 0.0
    for _ in range(args.steps):
        l2_flush.zero_()
        torch.cuda.synchronize(dev)
        p0 = time.perf_counter()
        step_device()
        torch.cuda.synchronize(dev)
        prof_ms += 1e3 * (time.perf_counter() - p0)
        k1 = ctx.last_kernel_ms()
        kms = k1 if kms is None else {k: kms[k] + v for k, v in k1.items()}
    kms = {k: v / args.steps for k, v in kms.items()}
    ctx.set_profiling(counters=True)
    res_c = step_device()
    arcs, slots = ctx.last_arc_evals()
    ctx.set_profiling()
    fp64_tinst = ctx.measure_fp64()

    markers_total = markers_rank * world
    value = markers_total * args.steps / (total_ms * 1e-3)
    e2e_value = markers_total * args.steps / (e2e_ms * 1e-3)

    if rank == 0:
        peaks = read_peaks()
        ksum = sum(kms.values()) or 1.0  # the serialised step: all kernels on one stream
        groups = {"scan": kms["scan"], "shuffle": kms["shuf0"] + kms["shuf1"] + kms["shuf2"] + kms["shuf3"] + kms["perm"],
                  "chain": kms["prefix"], "gen": kms["gen"], "prep": kms["prep"],
                  "edge": kms["edgeprep"] + kms["edgeperm"], "smooth": kms["smooth"], "sched": kms["sched"], "means": kms["means"]}
        dominant = max(groups, key=groups.get)
        elems = float(res_c.perm_elems)  # markers x permutations actually used by the decisions of one step
        # DRAM traffic per launch from the committed ncu --set full capture of one busy round (profiles/ncu_traffic.json, written
        # by tools/ncu_kernel_summary.py): dram__bytes_read.sum + dram__bytes_write.sum of the captured launch and the markers x
        # permutations that launch processed (the round's plan), hence measured bytes per element next to the algorithmic ones
        try:
            ncu = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
        except Exception:
            ncu = {}

        def traffic(kernel, alg_bytes_per_elem):
            k = ncu.get(kernel)
            if not k or "dram_read_bytes" not in k or not k.get("elements"):
                return None
            total = k["dram_read_bytes"] + k["dram_write_bytes"]
            return {"dram_bytes_per_launch": total, "launch_ms": k["ms"], "elements_in_launch": k["elements"],
                    "dram_bytes_per_element": total / k["elements"], "algorithmic_bytes_per_element": alg_bytes_per_elem,
                    "traffic_over_algorithmic": total / k["elements"] / alg_bytes_per_elem, "launches_captured": k["launches"],
                    "source": "profiles/ncu_traffic.json (" + ncu.get("_capture", "ncu --set full") + ")"}

        def hbm_roof(kernel, ms, bytes_per_elem, what, note):
            sec = ms * 1e-3
            gbs = bytes_per_elem * elems / sec / 1e9 if sec else None
            return {"bound": "hbm", "kernel": kernel, "achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                    "frac": gbs / peaks["hbm_gbs"] if gbs else None, "traffic": traffic(kernel.split("/")[0], bytes_per_elem),
                    "algorithmic_bytes": what, "ms_per_step": ms, "share_of_serialised_step": ms / ksum,
                    "time_base": "sum of the kernel's launches in a pass with every kernel on ONE stream (no overlap), CUDA events",
                    "peak_source": peaks["source"], "note": note}

        scan_s = kms["scan"] * 1e-3
        roof_scan = hbm_roof("k_scan", kms["scan"], 8.0, "8 B per marker per permutation: every prefix sum is read at least once",
                             "branch and bound: table-driven pruning discards most candidate arcs before any prefix sum is read; "
                             "the kernel is bound by the issue of the pruning tests, neither by HBM nor by the FP64 pipe")
        roof_scan["fp64"] = {"arcs_per_step": arcs, "slots_issued_per_step": slots, "peak_T_inst_per_s": fp64_tinst,
                             "achieved_T_inst_per_s": arcs / scan_s / 1e12 if scan_s else None,
                             "frac": (arcs / scan_s / 1e12 / fp64_tinst) if scan_s and fp64_tinst else None,
                             "note": "1 FP64-pipe instruction (DADD S_j - S_i) per arc actually examined; peak = DADD issue-rate "
                                     "microbenchmark on this GPU in this run (MEASURED_PEAKS.json has no FP64 figure)"}
        roof_chain = hbm_roof("k_chain", kms["prefix"], 16.0, "16 B per marker per permutation (read the permuted value, write S)",
                              "one dependent DADD chain per permutation (8 cycles per marker): latency bound unless thousands of "
                              "permutations are in flight")
        roof_shuffle = hbm_roof("k_shuffle/k_shuffle_cluster", groups["shuffle"], 16.0,
                                "16 B per marker per permutation (8 B gather + 8 B write, SURVEY 8d); the 8 B raw MT word per marker is extra",
                                "exact parallel Fisher-Yates replay, one CTA (or cluster) per permutation; last[] lives in shared "
                                "memory, so HBM only sees the MT words and the written row; bound by shared-memory latency and barriers")
        roofs = {"scan": roof_scan, "chain": roof_chain, "shuffle": roof_shuffle}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(S, args.scale) + (" [hybrid p-values]" if args.hybrid else ""), "rng": args.rng, "chain": False,
                       "samples_per_gpu": S, "l2": "256 MB buffer zeroed between timed steps; scratch arenas >> L2",
                       "parallelism": f"sample-sharded x{world}, final all_gather of segment tables"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(vals.nbytes) * world,
                    "d2h_bytes_per_step": int(len(res_h.lengths) * 12 + len(off) * 16) * world,
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "step_ms": {"device_resident": steps_device, "e2e": steps_host},
            "clocks": clocks,
            "kernel_ms_per_step_serialised": {k: round(v, 3) for k, v in kms.items()},
            "kernel_groups_ms_per_step_serialised": {k: round(v, 3) for k, v in groups.items()},
            "serialised_step_ms": {"kernels": round(ksum, 3), "wall": round(prof_ms / args.steps, 3),
                                   "note": "profile pass, all kernels on one stream; the timed steps above overlap independent kernels"},
            "dominant_kernel": dominant,
            "roofline": roofs.get(dominant, roof_scan),
            "roofline_scan": roof_scan, "roofline_chain": roof_chain, "roofline_shuffle": roof_shuffle,
            "segments": int(len(res.lengths)), "perms_run": int(res.perms_run), "perm_elements": int(res.perm_elems),
            "rounds": int(res.rounds),
        }
        if world == 1 and not args.no_cpu:
            m, dt, kind, used = cpu_reference_run(NPERM, os.cpu_count() or 1)
            line["cpu_baseline"] = {"value": m / dt, "unit": UNIT, "cores": used, "kind": kind, "seconds": round(dt, 1),
                                    "sample": CPU_SAMPLE}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rng", default="mt", choices=["mt", "philox"],
                    help="mt: bit-exact std::mt19937_64 replay (parity mode, default); philox: fast mode")
    ap.add_argument("--samples-per-gpu", type=int, default=1)
    ap.add_argument("--scale", type=float, default=1.0, help="shrink every chromosome (smoke runs only)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--cohort-run", action="store_true",
                    help="the north-star run: whole cohort (samples-per-gpu x gpus), per-rank times and the 16-sample parity subset; "
                         "no per-kernel profile passes, warm-up as given")
    ap.add_argument("--hybrid", action="store_true",
                    help="hybrid p-values (DNAcopy's default method, `cna segment --hybrid true`) instead of the CLI default; "
                         "not the headline configuration")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last device-resident timed step's results to DIR/<name>.npy (float64, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
