#!/usr/bin/env python
"""bench.py — the hot path of BASELINE.json on synthetic Nanopore-shaped reads.

  python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, sm_100a)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU path (oracle/_ref + oracle port)

A "step" is one pass of the hot path over one batch of reads:
    Assembler::findAlignmentCandidatesLowHash0 (all MinHash iterations)  ->  Assembler::computeAlignments (method 3)
on the BASELINE.json workload (configs[1]: 1 M synthetic Nanopore reads, N50 30 kb, ~30x, Nanopore-May2022.conf).
`value` = candidate read pairs found AND aligned per second (candidates / (LowHash time + alignment time)) with the marker
k-mer ids resident in HBM; the two halves are reported separately as lowhash_pairs_per_s and aligned_pairs_per_s.
`e2e` = the same through the reference-facing C-ABI calls with HOST buffers (7-byte CompressedMarker records, pinned):
host->device and device->host copies inside the timed region.
N > 1 (torchrun): the SAME read set is sharded by read id across the ranks (strong scaling): bucket all-to-all over
NCCL per LowHash iteration, all-gather of the k-mer ids, alignment of each rank's candidates.
One JSON line is printed by rank 0.
--dump-outputs DIR writes what the last timed step returned (see dump_outputs) as .npy files, so that two builds can be
compared output for output on the same seeded input.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# [MinHash] / [Align] values of the reference's configurations (conf/*.conf over the defaults of
# src/AssemblerOptions.cpp:327-489), the ones BASELINE.json's configs name.
MINHASH_DEFAULT = dict(m=4, hashFraction=0.01, minHashIterationCount=10, alignmentCandidatesPerRead=20.0,
                       log2MinHashBucketCount=0, minBucketSize=0, maxBucketSize=10, minFrequency=2)
ALIGN_DEFAULT = dict(alignMethod=3, k=10, maxSkip=30, maxDrift=30, maxTrim=30, minAlignedMarkerCount=100,
                     minAlignedFraction=0.4, matchScore=6, mismatchScore=-1, gapScore=-1, downsamplingFactor=0.1,
                     bandExtend=10, maxBand=1000, suppressContainments=0)
MINHASH_MAY2022 = dict(MINHASH_DEFAULT, minBucketSize=5, maxBucketSize=30, minFrequency=5)                  # conf/Nanopore-May2022.conf
ALIGN_MAY2022 = dict(ALIGN_DEFAULT, k=14, maxSkip=100, maxDrift=100, maxTrim=100, minAlignedMarkerCount=10,
                     minAlignedFraction=0.1, downsamplingFactor=0.05)
MINHASH_DEC2019 = dict(MINHASH_DEFAULT, minBucketSize=5, maxBucketSize=30, minFrequency=5)                  # conf/Nanopore-Dec2019.conf
ALIGN_DEC2019 = dict(ALIGN_DEFAULT, k=10, minAlignedFraction=0.4)
MINHASH_UL = dict(MINHASH_DEFAULT, minBucketSize=10, maxBucketSize=50, minFrequency=5)                      # conf/Nanopore-UL-May2022.conf
MINHASH_HIFI = dict(MINHASH_DEFAULT, hashFraction=0.05, minHashIterationCount=100, minFrequency=3,          # conf/HiFi-Oct2021.conf
                    minBucketSize=10, maxBucketSize=60)
ALIGN_HIFI = dict(ALIGN_DEFAULT, k=14, downsamplingFactor=0.05, minAlignedFraction=0.97, minAlignedMarkerCount=200,
                  maxSkip=6, maxDrift=4, maxTrim=2)

NANOPORE = dict(min_bases=10_000, drop=0.12, ins=0.05)
WORKLOADS = {
    # BASELINE.json configs[1]/[2]: 1M synthetic Nanopore reads (N50 30 kb, ~30x), Nanopore-May2022.conf
    "nanopore-may2022-1M": dict(NANOPORE, reads=1_000_000, n50=30_000, coverage=30.0, minhash=MINHASH_MAY2022, align=ALIGN_MAY2022),
    "nanopore-may2022-100k": dict(NANOPORE, reads=100_000, n50=30_000, coverage=30.0, minhash=MINHASH_MAY2022, align=ALIGN_MAY2022),
    "nanopore-may2022-10k": dict(NANOPORE, reads=10_000, n50=30_000, coverage=30.0, minhash=MINHASH_MAY2022, align=ALIGN_MAY2022),
    # configs[0]: 10k reads N50 20 kb, conf/Nanopore-Dec2019.conf (k = 10, default Align values, minAlignedFraction 0.4)
    "nanopore-dec2019-10k": dict(NANOPORE, reads=10_000, n50=20_000, coverage=20.0, minhash=MINHASH_DEC2019, align=ALIGN_DEC2019),
    # configs[3]: ultra-long, 200k reads N50 100 kb (>= 50 kb), conf/Nanopore-UL-May2022.conf; --align-method 4 for the Align4 run
    "nanopore-ul-200k": dict(min_bases=50_000, drop=0.12, ins=0.05, reads=200_000, n50=100_000, coverage=30.0,
                             minhash=MINHASH_UL, align=ALIGN_MAY2022),
    "nanopore-ul-20k": dict(min_bases=50_000, drop=0.12, ins=0.05, reads=20_000, n50=100_000, coverage=30.0,
                            minhash=MINHASH_UL, align=ALIGN_MAY2022),
    # configs[4]: HiFi, 2M reads N50 15 kb (>= 8 kb), low error, conf/HiFi-Oct2021.conf (hashFraction 0.05, 100 iterations)
    "hifi-2M": dict(min_bases=8_000, drop=0.004, ins=0.002, reads=2_000_000, n50=15_000, coverage=30.0,
                    minhash=MINHASH_HIFI, align=ALIGN_HIFI),
    "hifi-200k": dict(min_bases=8_000, drop=0.004, ins=0.002, reads=200_000, n50=15_000, coverage=30.0,
                      minhash=MINHASH_HIFI, align=ALIGN_HIFI),
}
CPU_SAMPLE_READS = int(os.environ.get("SHB_CPU_SAMPLE_READS", "20000"))   # bounded sample: same coverage, smaller genome
POLICY_SAMPLE_CANDIDATES = int(os.environ.get("SHB_POLICY_SAMPLE", "40000"))
M64 = (1 << 64) - 1


def synth_params(wl, reads=None, seed=1):
    """Marker-space read set of a workload (reads overrides the read count: the CPU sample keeps the coverage)."""
    from shasta_b200 import synth
    reads = reads or wl["reads"]
    mean_gap = 13.55
    mean_len = wl["n50"] * np.exp(-0.5 * 0.5 ** 2)          # log-normal: mean = N50 * exp(-sigma^2/2)
    span = mean_len / mean_gap
    genome_markers = int(max(reads * span / wl["coverage"], 4 * span))
    return synth.SynthParams(reads=reads, k=wl["align"]["k"], genome_markers=genome_markers, mean_gap=mean_gap, n50_bases=wl["n50"],
                             sigma=0.5, min_bases=wl["min_bases"], drop=wl["drop"], ins=wl["ins"], repeat_period=5000,
                             repeat_len=200, seed=seed)


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.rows = []
        self.proc = None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "500"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) >= 6 and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def cpu_reference_once(d, cores, minhash, align, keep=False):
    """The reference's CPU path on one read set: LowHash0 through the unmodified reference TUs (oracle/_ref) when they
    are present (else the oracle port), then computeAlignments through the oracle port (reference control flow
    restated + the SeqAn stand-in DP; 'not SeqAn', see DESIGN.md), one thread per core.
    Returns dict(candidates, lowhash_s, alignments, align_s, kind[, cand, rec, ctoc, cdata, ties])."""
    from oracle import bindings as B
    bp = B.LowHashParams(**minhash)
    if B.have_ref():
        c, _, _, sec_l = B.ref_lowhash0(d["toc"], d["data"], d["flags"], bp, threads=cores)
        kind = "reference"
    else:
        t0 = time.perf_counter()
        c, _, _ = B.oracle_lowhash0(d["toc"], d["data"], d["flags"], bp)
        sec_l = time.perf_counter() - t0
        kind = "port"
    oo = B.make_align_options(**{k: v for k, v in align.items() if k in B.ALIGN_DEFAULTS})
    t0 = time.perf_counter()
    rec, ctoc, cdata, ties = B.oracle_compute_alignments(d["toc"], d["kmer"], c, oo, threads=cores)
    sec_a = time.perf_counter() - t0
    out = dict(candidates=len(c), lowhash_s=sec_l, alignments=len(rec), align_s=sec_a, kind=kind)
    if keep:
        out.update(cand=c, rec=rec, ctoc=ctoc, cdata=cdata, ties=ties)
    return out


def policy_exposure(d, cand, align, cores):
    """How many candidate pairs are exposed to the (SeqAn-unpinned) tie-break rules of the DP at all: the oracle is run
    under all 8 policies of include/shb_dp_policy.h on a bounded slice of the sample's candidates; a pair is invariant
    when its stored result (kept or not, AlignmentData, compressed bytes) is the same under every policy."""
    from oracle import bindings as B
    cand = np.ascontiguousarray(cand[:POLICY_SAMPLE_CANDIDATES])
    oo = B.make_align_options(**{k: v for k, v in align.items() if k in B.ALIGN_DEFAULTS})
    default = B.default_dp_policy()
    keys = (cand[:, 0].astype(np.uint64) << np.uint64(33)) | (cand[:, 1].astype(np.uint64) << np.uint64(1)) | (cand[:, 2] & 1).astype(np.uint64)

    def per_candidate(rec, ctoc, cdata):
        # one 64-bit value per candidate: 0 = not stored, else a hash of its record and compressed bytes
        h = np.zeros(len(cand), np.uint64)
        if len(rec):
            rk = (rec[:, 0].astype(np.uint64) << np.uint64(33)) | (rec[:, 1].astype(np.uint64) << np.uint64(1)) | (rec[:, 2] & 1).astype(np.uint64)
            order = np.argsort(keys, kind="stable")                  # candidate keys are unique
            pos = order[np.searchsorted(keys[order], rk)]
            with np.errstate(over="ignore"):
                v = np.full(len(rec), 0xcbf29ce484222325, np.uint64)
                for k in range(16):
                    v = (v ^ rec[:, k].astype(np.uint64)) * np.uint64(0x100000001b3)
                csum = np.concatenate([np.zeros(1, np.uint64), np.cumsum(cdata.astype(np.uint64) * (np.arange(len(cdata), dtype=np.uint64) % np.uint64(251) + np.uint64(1)))])
                v ^= (csum[ctoc[1:].astype(np.int64)] - csum[ctoc[:-1].astype(np.int64)]) + (ctoc[1:] - ctoc[:-1]).astype(np.uint64) * np.uint64(0x9E3779B97F4A7C15)
            h[pos] = v | np.uint64(1)
        return h
    try:
        base = per_candidate(*B.oracle_compute_alignments(d["toc"], d["kmer"], cand, oo, threads=cores)[:3])
        differs = np.zeros(len(cand), bool)
        for policy in range(8):
            if policy == default:
                continue
            B.set_dp_policy(policy)
            differs |= per_candidate(*B.oracle_compute_alignments(d["toc"], d["kmer"], cand, oo, threads=cores)[:3]) != base
    finally:
        B.set_dp_policy(default)
    return {"candidates": int(len(cand)), "policy_invariant_fraction": float(1.0 - differs.mean()) if len(cand) else None,
            "policies": 8, "default_policy_bits": int(default)}


def run_reference(args, wl, rank):
    if rank != 0:
        return
    from shasta_b200 import synth
    # Bounded sample: the whole --steps K --warmup W run should end within a few minutes. One pass over the 20 000-read sample
    # takes ~25 s on the box's 128 threads (time is linear in the reads at fixed coverage), so the sample shrinks with K + W.
    budget_s, full_sample_s = 240.0, 25.0
    reads = int(CPU_SAMPLE_READS * min(1.0, budget_s / (max(1, args.steps + args.warmup) * full_sample_s)))
    p = synth_params(wl, reads=min(max(reads, 2000), wl["reads"]), seed=2)
    d = synth.generate(p)
    cores = effective_cpus()          # threads = the CPUs the container may use (quota), not the logical CPU count
    for _ in range(args.warmup):
        cpu_reference_once(d, cores, wl["minhash"], wl["align"])
    tl = ta = 0.0
    for _ in range(args.steps):
        r = cpu_reference_once(d, cores, wl["minhash"], wl["align"])
        tl += r["lowhash_s"]
        ta += r["align_s"]
    n, nal, kind = r["candidates"], r["alignments"], r["kind"]
    value = n * args.steps / (tl + ta)
    M = int(d["toc"][-1])
    sample = (f"{p.reads} synthetic reads ({M} markers both strands, {wl['coverage']}x, same generator/config), "
              f"{n} candidates, {nal} stored alignments; LowHash0 {tl / args.steps:.2f} s ({kind}), alignment {ta / args.steps:.2f} s (port)")
    line = {
        "impl": "reference", "metric": "candidate_pairs_found_and_aligned_per_s", "value": value, "unit": "pairs/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * (tl + ta) / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/i32", "data": "synthetic",
        "config": {"workload": args.workload, "minhash": wl["minhash"], "align": wl["align"], "sample": sample},
        "lowhash_pairs_per_s": n * args.steps / tl, "aligned_pairs_per_s": n * args.steps / ta,
        "cpu_baseline": {"value": value, "unit": "pairs/s", "cores": cores, "host_logical_cpus": os.cpu_count(), "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# The kernels that dominate the step (the banded / unbanded marker DPs) are bound by the integer ALU pipe, not by HBM or
# the tensor cores (profiles/README.md: ALU pipe 72 % busy at 72 % issue, DRAM a few percent), so next to the contract's
# `roofline` (the LowHash sweep, HBM by contract) the line carries the DP's own ceiling: the B200's integer ALU rate divided
# by the ALU-pipe instructions a DP cell needs (counted in the SASS of the wavefront kernel's unchecked block,
# profiles/r2_sass_banded1_unchecked_block.txt: ISETP x3, VIMNMX, VIADDMNMX per cell; the adds and the trace codes issue
# on the FMA pipe as IMADs). Informational: the cells counted include the padding of the band classes.
ALU_LANES_PER_SM = 64            # INT32 compare/select/min/max lanes per SM and clock (ncu: 2 warp instructions/clk/SM at 100 %)
SM_COUNT = 148
ALU_OPS_PER_CELL = 5             # k-mer equality test, max, add-max, 2 trace compares


def alignment_roofline(dp_cells, dp_ms, sm_mhz):
    """dp_cells: DP cells the kernels were asked to fill during the timed steps (band cells incl. the padding to the band
    class, plus the real cells of the trace-free stage 1); dp_ms: CUDA-event time of the DP launches of those steps
    (stage 1, stage 2, traceback and filter, as they overlap on their streams)."""
    if not dp_ms or not dp_cells:
        return None
    achieved = dp_cells / (1e-3 * dp_ms) / 1e9
    peak = SM_COUNT * ALU_LANES_PER_SM * (sm_mhz or 1965.0) * 1e6 / ALU_OPS_PER_CELL / 1e9
    return {"bound": "alu", "kernels": "bandedAlignKernel<C>, method3Stage1ForwardKernel<R> (+ tracebackKernel, filterStepsKernel overlapped)",
            "achieved": achieved, "peak": peak, "unit": "G cell updates/s", "frac": achieved / peak,
            "peak_source": "%d SMs x %d integer-ALU lanes x %.0f MHz / %d ALU operations per DP cell"
                           % (SM_COUNT, ALU_LANES_PER_SM, sm_mhz or 1965.0, ALU_OPS_PER_CELL)}


# Caps of what --dump-outputs writes, for all ranks together: 54.1 MB at most (64 MB is the bound).
DUMP_CANDIDATE_ROWS = 800_000         # 19.2 MB as float64
DUMP_STATS_ROWS = 500_000             # 12 MB as float64
DUMP_ALIGNMENT_ROWS = 80_000          # 10.24 MB as float64, and 0.64 MB of sizes
DUMP_COMPRESSED_BYTES = 3_000_000     # 12 MB as float32


def _sample_rows(n, cap, seed):
    """All row indices when n <= cap, else a fixed seeded sample of cap of them, in order."""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, cap, replace=False))


def dump_outputs(path, cand, stats=None, rec=None, ctoc=None, cdata=None, world=1):
    """Writes the outputs of one step as float64 (exact for their 32-bit fields and counts) and float32 (bytes) arrays:
      candidates.npy                 the LowHash0 candidates (readId0, readId1, isSameStrand), rows [n, 3]
      read_lowhash_statistics.npy    the per-read LowHash0 statistics (ReadLowHashStatistics), rows [R, 3]
      alignment_data.npy             the stored AlignmentData records, rows [n, 16]
      compressed_alignment_sizes.npy the compressed-alignment byte count of each of those records
      compressed_alignment_bytes.npy the compressed bytes of the first of those records, concatenated
      counts.npy                     total candidates and alignments
    Larger outputs are sampled: the same rows for the same counts. With `world` ranks each rank writes its own block of
    the candidates and alignments within 1/world of their caps; the statistics, the same on every rank, are passed by
    one rank only. All files together stay within the DUMP_* caps, 54.1 MB."""
    os.makedirs(path, exist_ok=True)
    ci = _sample_rows(len(cand), DUMP_CANDIDATE_ROWS // world, 1)
    np.save(os.path.join(path, "candidates.npy"), np.asarray(cand)[ci].astype(np.float64))
    counts = [len(cand)]
    if stats is not None:
        si = _sample_rows(len(stats), DUMP_STATS_ROWS, 3)
        np.save(os.path.join(path, "read_lowhash_statistics.npy"), np.asarray(stats)[si].astype(np.float64))
    if rec is not None:
        ai = _sample_rows(len(rec), DUMP_ALIGNMENT_ROWS // world, 2)
        ctoc = np.asarray(ctoc, np.int64)
        sizes = ctoc[1:][ai] - ctoc[:-1][ai]
        keep = int(np.searchsorted(np.cumsum(sizes), DUMP_COMPRESSED_BYTES // world, side="right"))
        data = [cdata[ctoc[i]:ctoc[i + 1]] for i in ai[:keep]]
        np.save(os.path.join(path, "alignment_data.npy"), np.asarray(rec)[ai].astype(np.float64))
        np.save(os.path.join(path, "compressed_alignment_sizes.npy"), sizes.astype(np.float64))
        np.save(os.path.join(path, "compressed_alignment_bytes.npy"),
                np.concatenate(data).astype(np.float32) if data else np.zeros(0, np.float32))
        counts.append(len(rec))
    np.save(os.path.join(path, "counts.npy"), np.array(counts, np.float64))


def effective_cpus():
    """Host CPUs this process can actually use: the affinity mask, capped by the container's CFS quota (cgroup v2 cpu.max or
    v1 cpu.cfs_quota_us / cpu.cfs_period_us). The pool's 1-GPU boxes show 128 logical CPUs under a quota of 16."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        try:
            quota = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if quota > 0:
                n = min(n, max(1, -(-quota // period)))
        except Exception:
            pass
    return n


def gpu_numa_cpus(torch, device_index):
    """(numa node, CPUs) of the NUMA node the GPU hangs off — what `numactl --cpunodebind` would be given — or (None, None)."""
    try:
        pr = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return None, None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        return node, cpus
    except Exception:
        return None, None


def _claim_stdout():
    """stdout carries exactly one JSON line. Libraries (NCCL prints its version banner) write to fd 1 directly, so fd 1
    is pointed at stderr for the whole run and the JSON line goes to a private copy of the original stdout."""
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w", buffering=1)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="nanopore-may2022-1M", choices=list(WORKLOADS))
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-align", action="store_true", help="LowHash0 only (profiling aid)")
    ap.add_argument("--align-method", type=int, default=3, choices=[3, 4],
                    help="3 = what Nanopore-May2022.conf selects (default); 4 = Align4, --Align.alignMethod 4")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (DIR/rank<r>/ with several GPUs)")
    args = ap.parse_args()
    wl = dict(WORKLOADS[args.workload])
    wl["align"] = dict(wl["align"], alignMethod=args.align_method)
    MINHASH, ALIGN = wl["minhash"], wl["align"]

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, wl, rank)
        return

    import torch
    import torch.distributed as dist
    from shasta_b200 import capi, synth
    from shasta_b200 import distributed as D

    torch.cuda.set_device(local_rank)
    # Process placement: the rank's host threads (and the memory they first touch: pinned marker buffer, result blocks) on the
    # CPUs of the GPU's own NUMA node, as `numactl --cpunodebind=<node of the GPU>` would do for a production process. The CPU
    # baseline / parity legs below run with the original mask (all host cores). SHB_BENCH_NO_AFFINITY=1 turns it off.
    affinity_all = os.sched_getaffinity(0)
    affinity_gpu, numa_node = None, None
    if not os.environ.get("SHB_BENCH_NO_AFFINITY"):
        numa_node, cpus = gpu_numa_cpus(torch, local_rank)
        if cpus and len(cpus & affinity_all) >= 8:
            affinity_gpu = cpus & affinity_all
            try:
                os.sched_setaffinity(0, affinity_gpu)
            except OSError:
                affinity_gpu = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum(x):
        t = torch.tensor([float(x)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    def allgather_floats(xs):
        """Every rank's values (one row per rank)."""
        t = torch.tensor([float(v) for v in xs], dtype=torch.float64, device="cuda")
        if world == 1:
            return [t.tolist()]
        parts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        return [q.tolist() for q in parts]

    def allsum_u64(x):
        """Sum of 64-bit digests over the ranks, mod 2^64 (gathered as two 32-bit halves: exact)."""
        x = int(x) & M64
        if world == 1:
            return x
        t = torch.tensor([x & 0xffffffff, x >> 32], dtype=torch.int64, device="cuda")
        parts = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(parts, t)
        return sum(int(q[0].item()) | (int(q[1].item()) << 32) for q in parts) & M64

    # ---- synthetic input, generated on the device; the same read set for every N (strong scaling) ----------------
    p = synth_params(wl, seed=1)
    R = p.reads
    ctx = capi.Context(local_rank)
    t0 = time.perf_counter()
    want_e2e = not args.no_e2e
    if world == 1:
        rb, re = 0, R
    else:
        _, span, _ = synth.read_windows(p)
        bounds = D.balanced_read_ranges(span, world)
        rb, re = bounds[rank], bounds[rank + 1]
    dm = capi.synth_generate_device(ctx, p, want_data7=want_e2e, read_begin=rb, read_end=re)
    M_local = dm.marker_count
    M = int(allsum(M_local))
    gen_s = time.perf_counter() - t0
    lparams = capi.make_lowhash_params(**MINHASH)
    aopts = capi.make_align_options(**ALIGN)
    ctx.set_markers_device(dm.toc, dm.kmer_ptr, dm.flags, keepalive=dm, read_begin=rb, read_end=re,
                           read_count_total=R, total_marker_count=M)
    if world > 1:
        # The library's own NCCL communicator (csrc/dist.cu); torch.distributed only ships the 128-byte id and does the
        # barriers / max-over-ranks of this script.
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(capi.dist_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, src=0)
        ctx.dist_init(world, rank, bytes(uid.cpu().numpy().tobytes()))

    stats_acc = {"sweep_ms": 0.0, "sweep_launches": 0, "launches": 0, "lowhash_s": 0.0, "align_s": 0.0, "gather_s": 0.0,
                 "dp_ms": 0.0, "dp_cells": 0, "dp_useful_cells": 0, "alignments": 0}
    last = {}

    def step(record, host_data7=None, keep_outputs=False):
        """One pass of the hot path. host_data7 != None: end-to-end mode, the marker records come from (pinned) host
        memory through shb_set_markers inside the timed region. keep_outputs: leave the step's outputs in last["outputs"]
        (only for the last step: held across steps they would keep the library from recycling its host result buffers)."""
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if host_data7 is not None:
            ctx.set_markers(dm.toc, host_data7, dm.flags, read_begin=rb, read_end=re, read_count_total=R, total_marker_count=M)
        if world == 1:
            cand, stats, _, res = ctx.lowhash0(lparams, want_stats=True)
            sweep_ms, sweep_launches, launches = res.sweepMs, res.sweepLaunches, res.kernelLaunches
        else:
            cand, stats, res = ctx.lowhash0_sharded(lparams, want_stats=True)
            if record:
                tm = ctx.dist_timing()
                for k in ("sweep", "partition", "exchange", "process", "final"):
                    stats_acc["sharded_" + k] = stats_acc.get("sharded_" + k, 0.0) + getattr(tm, k + "Seconds")
            sweep_ms, sweep_launches, launches = res.sweepMs, res.sweepLaunches, res.kernelLaunches
        last["candidate_digest"] = res.candidateDigest
        last["low_hashes"], last["pair_hits"] = res.lowHashCount, res.pairCount
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        nal = 0
        d2h = len(cand) * 12
        t2 = t1
        outputs = dict(cand=cand, stats=stats)
        if not args.no_align:
            t2 = time.perf_counter()
            if world > 1:           # gathers the k-mer ids of all ranks on the first call after the markers changed
                rec, ctoc, cdata, ares = capi.compute_alignments_sharded(ctx, cand, aopts)
                if record:
                    stats_acc["gather_once_s"] = ctx.dist_timing().gatherSeconds
            else:
                rec, ctoc, cdata, ares = capi.compute_alignments(ctx, cand, aopts)
            nal = len(rec)
            outputs.update(rec=rec, ctoc=ctoc, cdata=cdata)
            d2h += rec.nbytes + ctoc.nbytes + cdata.nbytes
            launches += ares.kernelLaunches
            last.update(alignment_data_digest=ares.alignmentDataDigest, compressed_digest=ares.compressedDigest,
                        skipped=ares.skippedCount, too_wide=ares.tooWideCount, workers=ares.workers)
            if record:
                stats_acc["dp_ms"] += ares.dpMs
                stats_acc["dp_cells"] += ares.dpCells
                stats_acc["dp_useful_cells"] += ares.dpUsefulCells
                stats_acc["align_copy_ms"] = stats_acc.get("align_copy_ms", 0.0) + ares.outputCopyMs
                stats_acc["align_lib_ms"] = stats_acc.get("align_lib_ms", 0.0) + ares.hostWallMs
        torch.cuda.synchronize()
        t3 = time.perf_counter()
        if record:
            stats_acc["sweep_ms"] += sweep_ms
            stats_acc["sweep_launches"] += sweep_launches
            stats_acc["launches"] += launches
            stats_acc["lowhash_s"] += t1 - t0
            stats_acc["gather_s"] += t2 - t1
            stats_acc["align_s"] += t3 - t2
            stats_acc["alignments"] = nal
        if keep_outputs:
            last["outputs"] = outputs
        stats_acc["last_d2h"] = d2h
        return cand, nal

    # ---- device-resident timing ----------------------------------------------------------------------------------
    for _ in range(args.warmup):
        cand, nal = step(False)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        ev0.record()
        t0 = time.perf_counter()
        for i in range(args.steps):
            cand, nal = step(True, keep_outputs=bool(args.dump_outputs) and i == args.steps - 1)
        ev1.record()
        barrier()
        wall = time.perf_counter() - t0
    wall = allmax(wall)
    if args.dump_outputs:
        outputs = last.pop("outputs")
        if rank != 0:
            outputs["stats"] = None         # all-reduced: every rank holds the same statistics
        dump_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, f"rank{rank}"), world=world, **outputs)
        del outputs
    total_cand = allsum(len(cand))
    total_al = allsum(nal)
    # Per-rank view of the timed steps (the aggregate keys below are maxima over the ranks, which do not add up): host-clock
    # time inside the LowHash0 call (includes waiting for slower ranks in its collectives), inside the alignment call, the DP
    # kernels' CUDA-event time, and the candidates each rank aligned.
    own_clocks = clocks.summary()
    per_rank = allgather_floats([1e3 * stats_acc["lowhash_s"] / args.steps, 1e3 * (stats_acc["align_s"] + stats_acc["gather_s"]) / args.steps,
                                 stats_acc["dp_ms"] / args.steps, len(cand), own_clocks.get("sm_mhz") or 0.0,
                                 1.0 if "sw_power_cap" in (own_clocks.get("reasons") or []) else 0.0])
    lowhash_s = allmax(stats_acc["lowhash_s"])
    align_s = allmax(stats_acc["align_s"] + stats_acc["gather_s"])
    value = total_cand * args.steps / wall
    # Order-independent digests of what the last timed step produced, summed over the ranks: equal for every N, and equal
    # to the digests of the CPU path's output on the same input (checked on the sample below and in tests/).
    digests = {"candidates": "%016x" % allsum_u64(last.get("candidate_digest", 0)),
               "alignment_data": "%016x" % allsum_u64(last.get("alignment_data_digest", 0)),
               "compressed_alignments": "%016x" % allsum_u64(last.get("compressed_digest", 0)),
               "definition": "include/shasta_b200.h: shb_digest_records / shb_digest_compressed (sum of per-record FNV-1a values mod 2^64)"}
    skipped_total, too_wide_total = int(allsum(last.get("skipped", 0))), int(allsum(last.get("too_wide", 0)))
    dp_cells_all, dp_useful_all, dp_ms_max = allsum(stats_acc["dp_cells"]), allsum(stats_acc["dp_useful_cells"]), allmax(stats_acc["dp_ms"])

    # ---- end to end through the reference-facing calls with host buffers ------------------------------------------------
    e2e = None
    if want_e2e:
        host = torch.empty(M_local * 7, dtype=torch.uint8, pin_memory=True)
        data7 = host.numpy()
        dm.data7_to_host(out=data7)
        e2e_steps = args.steps
        step(False, host_data7=data7)
        barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            c2, n2 = step(False, host_data7=data7)
        barrier()
        e2e_wall = allmax(time.perf_counter() - t0)
        assert allsum(len(c2)) == total_cand and allsum(n2) == total_al, "host-buffer path and device-resident path disagree"
        assert "%016x" % allsum_u64(last.get("alignment_data_digest", 0)) == digests["alignment_data"], "host-buffer path digest differs"
        if world == 1:
            assert np.array_equal(c2, cand)
        e2e = {"value": total_cand * e2e_steps / e2e_wall, "unit": "pairs/s",
               "h2d_bytes_per_step": int(allsum(M_local * 7 + dm.toc.nbytes + dm.flags.nbytes + (0 if args.no_align else len(c2) * 12))),
               "d2h_bytes_per_step": int(allsum(stats_acc["last_d2h"])), "steps": e2e_steps, "ms_per_step": 1e3 * e2e_wall / e2e_steps}
        del host, data7
        # restore the device-resident markers for anything that follows
        ctx.set_markers_device(dm.toc, dm.kmer_ptr, dm.flags, keepalive=dm, read_begin=rb, read_end=re,
                               read_count_total=R, total_marker_count=M)

    sweep_ms = allmax(stats_acc["sweep_ms"])
    if rank != 0:
        return

    # ---- roofline of the dominant LowHash kernel (hash sweep) -------------------------------------------------------
    iters = MINHASH["minHashIterationCount"]
    frac_h = MINHASH["hashFraction"]
    bytes_per_marker_iteration = 4.0 + 16.0 * frac_h                 # SURVEY.md section 8(d)
    launches = max(stats_acc["sweep_launches"], 1)
    iters_per_launch = iters * args.steps / launches
    alg_bytes_per_launch = M_local * bytes_per_marker_iteration * iters_per_launch
    avg_launch_s = 1e-3 * stats_acc["sweep_ms"] / launches
    achieved = alg_bytes_per_launch / avg_launch_s / 1e9
    peak, peak_src = measured_hbm_peak()
    traffic = None
    tp = os.path.join(ROOT, "profiles", "sweep_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            # measured on the 100k-read workload: scale per marker to this launch
            traffic = tj["dram_bytes_per_marker_per_launch"] * M_local
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "lowhashSweepKernel<%d>" % MINHASH["m"], "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "note": "achieved = ALGORITHMIC bytes (SURVEY 8d: M x (4 + 16 x hashFraction) per iteration, x iterations fused per "
                        "launch) / CUDA-event launch time: an algorithmic-equivalent bandwidth. One launch reads the k-mer ids once for "
                        "all its fused iterations, so the DRAM bytes actually moved (`traffic`) are a fraction of the algorithmic "
                        "bytes; the kernel is bound by integer instruction issue (3 dependent 64-bit multiplies per feature and "
                        "iteration), not by HBM.",
                "algorithmic_bytes_per_launch": alg_bytes_per_launch, "avg_launch_ms": 1e3 * avg_launch_s,
                "iterations_fused_per_launch": iters_per_launch, "sweep_share_of_step": 1e-3 * sweep_ms / wall,
                "alignment_gcups": (stats_acc["dp_cells"] / (1e-3 * stats_acc["dp_ms"]) / 1e9) if stats_acc["dp_ms"] else None}

    # ---- the reference's CPU path on a bounded sample, and the GPU path on that SAME sample: parity at bench scale ------
    cpu_baseline = None
    parity = None
    if not args.no_cpu_baseline and world == 1:
        ps = synth_params(wl, reads=min(CPU_SAMPLE_READS, wl["reads"]), seed=2)
        # Same generator as the numpy one (bit-identical), run on the device to save minutes of host time.
        dms = capi.synth_generate_device(ctx, ps, want_data7=True)
        d = {"toc": dms.toc, "data": dms.data7_to_host(), "flags": dms.flags, "kmer": dms.kmer_ids_to_host()}
        cores = effective_cpus()          # threads = the CPUs the container may use (quota), not the logical CPU count
        if affinity_gpu:
            os.sched_setaffinity(0, affinity_all)          # the CPU path gets every host core
        r = cpu_reference_once(d, cores, MINHASH, ALIGN, keep=True)
        n, sec_l, nalc, sec_a, kind = r["candidates"], r["lowhash_s"], r["alignments"], r["align_s"], r["kind"]
        Ms = int(d["toc"][-1])
        cpu_baseline = {"value": n / (sec_l + sec_a), "unit": "pairs/s", "cores": cores, "host_logical_cpus": os.cpu_count(), "kind": kind,
                        "sample": f"{ps.reads} synthetic reads ({Ms} markers both strands, same coverage/config), {n} candidates, "
                                  f"{nalc} stored alignments; LowHash0 {sec_l:.2f} s ({kind}: unmodified reference TUs), "
                                  f"alignment {sec_a:.2f} s (port: reference control flow + SeqAn stand-in DP)",
                        "lowhash_pairs_per_s": n / sec_l, "aligned_pairs_per_s": n / sec_a}
        # GPU on the sample, through the same C-ABI calls; every output compared with the CPU path's.
        sctx = capi.Context(local_rank)
        sctx.set_markers_device(dms.toc, dms.kmer_ptr, dms.flags, keepalive=dms)
        gc, gstats, _, gres = sctx.lowhash0(lparams, want_stats=True)
        parity = {"sample_reads": ps.reads, "candidates": int(len(gc)), "candidates_identical": bool(np.array_equal(gc, r["cand"]))}
        if not args.no_align:
            grec, gtoc, gdata, gares = capi.compute_alignments(sctx, gc, aopts)
            parity.update(alignments=int(len(grec)),
                          alignment_data_identical=bool(np.array_equal(grec, r["rec"])),
                          compressed_identical=bool(np.array_equal(gtoc, r["ctoc"]) and np.array_equal(gdata, r["cdata"])),
                          digests_match_cpu=bool(gares.alignmentDataDigest == capi.digest_records(r["rec"], 16)
                                                 and gares.compressedDigest == capi.digest_compressed(r["rec"], r["ctoc"], r["cdata"])
                                                 and gres.candidateDigest == capi.digest_candidates(r["cand"])))
            ties = r["ties"]
            parity["dp_tie_free_fraction"] = float(((ties & 6) == 0).mean()) if len(ties) else None
            parity["dp_tie_free_definition"] = ("fraction of the sample's candidate pairs none of whose DP paths passes through a cell with "
                                                "co-optimal predecessors or ends in a tied end cell (upper bound on the exposure to the "
                                                "SeqAn-unpinned tie-break rules)")
            parity["align4_component_tie_fraction"] = float((ties & 1).mean()) if len(ties) else None
            try:
                parity["policy_sweep"] = policy_exposure(d, r["cand"], ALIGN, cores)
            except Exception as e:            # informational: never lose the line over it
                parity["policy_sweep"] = {"error": str(e)}
        sctx.close()
        dms.free()
        ok = parity["candidates_identical"] and parity.get("alignment_data_identical", True) and parity.get("compressed_identical", True)
        assert ok, f"GPU and CPU paths disagree on the {ps.reads}-read sample: {parity}"

    useful = stats_acc["dp_useful_cells"]
    line = {
        "metric": "candidate_pairs_found_and_aligned_per_s", "value": value, "unit": "pairs/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64/i32", "data": "synthetic",
        "config": {"workload": args.workload, "reads": R, "markers": M, "minhash": MINHASH, "align": ALIGN,
                   "parallelism": ("reads sharded by id over %d GPUs (one process each, NCCL inside the library): bucket exchange per LowHash "
                                   "iteration overlapped with the bucket inspection, pair counts exchanged once, k-mer ids gathered once per "
                                   "marker set for the alignment of each rank's candidate block" % world)
                   if world > 1 else "single GPU",
                   "l2": "inputs (k-mer ids %.1f GB) larger than L2" % (4e-9 * M_local), "generation_s": gen_s,
                   "align_included": not args.no_align},
        "candidates": total_cand, "alignments": total_al, "skipped_candidates": skipped_total, "too_wide_candidates": too_wide_total,
        "digests": digests, "parity_on_cpu_sample": parity,
        "lowhash_work_per_step": {"low_hashes": last.get("low_hashes"), "pair_hits": last.get("pair_hits"),
                                  "note": "low hashes kept / candidate pair hits generated over all iterations (this rank's share when sharded)"},
        "lowhash_pairs_per_s": total_cand * args.steps / lowhash_s,
        "aligned_pairs_per_s": (total_cand * args.steps / align_s) if align_s else None,
        "lowhash_ms_per_step": 1e3 * lowhash_s / args.steps, "align_ms_per_step": 1e3 * align_s / args.steps,
        "marker_iterations_per_s": M * iters * args.steps / lowhash_s,
        "device_event_ms_per_step": ev0.elapsed_time(ev1) / args.steps,
        "sharded_lowhash_breakdown_ms_per_step": {k[8:]: 1e3 * v / args.steps for k, v in stats_acc.items() if k.startswith("sharded_")},
        "marker_gather_s_once_per_marker_set": stats_acc.get("gather_once_s"),
        "align_breakdown_ms_per_step": {"dp_kernels": stats_acc["dp_ms"] / args.steps,
                                        "result_copy_to_host": stats_acc.get("align_copy_ms", 0.0) / args.steps,
                                        "library_call": stats_acc.get("align_lib_ms", 0.0) / args.steps,
                                        "workers": last.get("workers")},
        "dp_cells": {"useful_per_step": useful / args.steps, "computed_per_step": stats_acc["dp_cells"] / args.steps,
                     "useful_g_per_s": (dp_useful_all / (1e-3 * dp_ms_max) / 1e9) if dp_ms_max else None,
                     "note": "useful = in-band, in-matrix cells (what the reference's DP fills) + the unbanded stage-1 cells; computed also "
                             "counts the padding of the band classes to multiples of 64 offsets and the two barrier offsets"},
        "per_rank_ms_per_step": {"lowhash_call": [round(r[0], 2) for r in per_rank], "alignment_call": [round(r[1], 2) for r in per_rank],
                                 "dp_kernels": [round(r[2], 2) for r in per_rank], "candidates": [int(r[3]) for r in per_rank],
                                 "sm_mhz": [r[4] for r in per_rank], "sw_power_cap_seen": [int(r[5]) for r in per_rank]},
        "host_placement": {"numa_node_of_gpu": numa_node, "cpus_bound": (len(affinity_gpu) if affinity_gpu else None),
                           "note": "timed legs run with the rank's threads bound to the CPUs of its GPU's NUMA node; the CPU legs use all host cores"},
        "gpu_launches": int(stats_acc["launches"]), "clocks": clocks.summary(),
        "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
    }
    try:
        line["alignment_roofline"] = alignment_roofline(stats_acc["dp_cells"], stats_acc["dp_ms"], (line["clocks"] or {}).get("sm_mhz"))
    except Exception:       # informational only: never let it cost the bench line
        line["alignment_roofline"] = None
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
