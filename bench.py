#!/usr/bin/env python
"""Benchmark of the FastSMC IBD hot path on B200 (BASELINE.json configs[1]: all-pairs decoding with hashing off,
1,000 synthetic haplotypes x 10,000 SNPs, 69-state decoding quantities; every pair is decoded over the whole sequence and
IBD segments with per-segment age estimates are called, as FastSMC::run does with hashing off).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over the whole job (499,500 haplotype pairs x 10,000 sites).
  value : pair-sites/s with the pair list resident in HBM (fsmc_plan_launch only inside the timed region)
  e2e   : the same through the C-ABI call fsmc_decode with HOST buffers: pair lists copied H2D and the segment records
          copied D2H inside the timed region
Under torchrun (N > 1) the SAME job is split over the N GPUs ("scaling": "strong"): the job's reference batches of 32 pairs
are independent once formed, so rank r decodes the r-th contiguous share of them (no collective on the data path; the
barrier and the max-over-ranks time are the only cross-rank operations); value = the job's pair-sites / the slowest rank's
device time.  `jobs_run` is the north star's jobs/jobInd partition on a hashing workload (cfg4 family): the J = 64 jobs of one
data set dealt to the N ranks from a shared counter, files to .ibd.gz, host and kernel seconds per rank.

--impl reference times the CPU restatement of the reference algorithm (oracle/, multi-threaded over batches, AVX2 lane
vectorisation like the reference's SIMD build) on a bounded sample of the same workload on the host cores.

--dump-outputs DIR writes the segment records of the last timed step of the headline run to DIR/segment_<field>.npy (see
dump_segments), so that two builds can be compared output for output on the same seeded inputs.

Data sets and output files go to a per-user directory under the system's temporary directory (WORK), never into the tree.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_HAPS, N_SITES, SPAN_BP, CHROM, SEED = 1000, 10_000, 30_000_000, 1, 20201117 + 2
DQ = os.path.join(ROOT, "data", "30-100-2000.decodingQuantities.gz")
DQ_159 = os.path.join(ROOT, "tests", "golden", "fastsmc_example", "example.decodingQuantities.gz")  # FASTSMC_EXAMPLE table
FLOPS_PER_PAIR_SITE_STATE = 35  # SURVEY.md §8(d) / App. A: 15 forward + 15 backward + 3 combine + 2 consume
NCU_NARROW_DRAM_BYTES_PER_PAIR_SITE = (6.072805e9 + 6.078759e9) / (37888 * 10000)  # profiles/r1_v4_decodeNarrow_s69_ncu_full.txt
NCU_DRAM_BYTES_PER_PAIR_SITE = (109.922461e9 + 109.458343e9) / (37888 * 10000)  # profiles/r1_v4_decodeFast_s69_ncu_full.txt
# profiles/r2_p2_decodeNarrowSparse_ncu_full.txt: 87.83 GB read + 101.53 GB written by one launch of decodeNarrowKernel<69, sparse>
# over cfg2 (blocks of 128 sites); refineKernel adds 75.8 GB per step (profiles/r2_final_refine_ncu_full.txt)
NCU_SPARSE_DRAM_BYTES_PER_PAIR_SITE = (87.827249e9 + 101.530119e9) / (499500 * 10000)
WORKLOAD = "cfg2: all-pairs, hashing off, 1000 haplotypes x 10000 SNPs, S=69 (30-100-2000), time=50, batchSize=32"
# per user: files another user's run left in a shared directory could not be overwritten
WORK = os.path.join(tempfile.gettempdir(), f"fsmc_bench_{os.getuid()}")


def dataset_root(rank):
    return f"{WORK}/r{rank}/cfg2_{N_HAPS}x{N_SITES}"


def make_dataset(rank):
    from fastsmc_b200 import synth
    root = dataset_root(rank)
    if not os.path.exists(root + ".hap.gz"):
        synth.dataset(root, N_HAPS, N_SITES, SPAN_BP, CHROM, SEED)
    return root


def all_pairs_in_reference_order(n_ind):
    """hapA, hapB of HMM::decodeAll's enumeration (ref: ASMC_SRC/SRC/HMM.cpp:325-357), vectorised."""
    a, b = [], []
    for i in range(n_ind):
        j = np.repeat(np.arange(i), 4)
        ih = np.tile(np.array([0, 0, 1, 1]), i)
        jh = np.tile(np.array([0, 1, 0, 1]), i)
        a.append(2 * j + jh)
        b.append(np.full(4 * i, 2 * i) + ih)
        a.append(np.array([2 * i]))
        b.append(np.array([2 * i + 1]))
    return np.concatenate(a).astype(np.uint32), np.concatenate(b).astype(np.uint32)


def rank_share(n_batches, world, rank):
    """Batches [lo, hi) of the job that `rank` decodes: contiguous, sizes differ by at most one."""
    return n_batches * rank // world, n_batches * (rank + 1) // world


def tiles_for(a, b, sites, world=1, rank=0):
    n = len(a)
    T = (n + 31) // 32
    A = np.zeros(T * 32, np.uint32)
    B = np.zeros(T * 32, np.uint32)
    A[:n], B[:n] = a, b
    tp = np.full(T, 32, np.int32)
    tp[-1] = n - 32 * (T - 1)
    lo, hi = rank_share(T, world, rank)
    A, B, tp = A.reshape(T, 32)[lo:hi], B.reshape(T, 32)[lo:hi], tp[lo:hi]
    T = hi - lo
    z, e = np.zeros(T, np.int32), np.full(T, sites, np.int32)
    return dict(hapA=np.ascontiguousarray(A), hapB=np.ascontiguousarray(B), tilePairs=np.ascontiguousarray(tp), tileFrom=z,
                tileTo=e, tileScanFrom=z, tileScanTo=e, rows=np.arange(int(tp.sum())))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (profiling recipe's clocks line)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc:
            self.proc.terminate()
            self.t.join(timeout=2)

    def summary(self):
        ok = [r for r in self.rows if len(r) == 7 and r[0].isdigit()]
        if not ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i] == "Active" for r in ok)]
        return {"sm_mhz": float(np.median([int(r[0]) for r in ok])), "sm_max_mhz": float(ok[0][1]),
                "power_w_max": max(float(r[2]) for r in ok), "samples": len(ok), "reasons": reasons}


REF_JOBS = 64  # the CPU arm cuts cfg2 into 64 jobs (reference jobs/jobInd) and runs one job per host core at a time


def reference_sample(cores):
    """One bounded sample of cfg2 on the reference's own CPU implementation: `cores` concurrent processes (the reference is
    single-threaded; its way to use many cores is one process per job, cpp_example/FastSMC_example_multiple_jobs.sh), each
    ASMC::FastSMC(params).run() of one of the REF_JOBS jobs of the data set, all 10,000 sites, same flags as the GPU arm.
    Returns (pair_sites, seconds of the slowest process's run(), kind, sample description).  Time excludes reading the
    data and preparing the model, as the GPU arm's does."""
    import re
    from oracle import pyoracle
    root = make_dataset(0)
    if pyoracle.reference_binary("avx") is None:
        return None
    procs = []
    # off-diagonal jobs only (job ids that are perfect squares are the diagonal jobs, a quarter of the pairs), so that the
    # concurrent processes carry equal work and the slowest one does not understate the CPU rate
    off_diagonal = [j for j in range(1, REF_JOBS + 1) if int(j ** 0.5) ** 2 != j]
    for k in range(cores):
        argv = pyoracle.reference_command("avx", root, DQ, f"{WORK}/ref_out_{k}", hashing=0, jobs=REF_JOBS,
                                          jobInd=off_diagonal[k % len(off_diagonal)], time=50, noConditionalAgeEstimates=1,
                                          batchSize=32)
        procs.append(subprocess.Popen(argv, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True))
    pairs, slowest = 0, 0.0
    for pr in procs:
        out, err = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError("reference build failed: " + err[-300:])
        slowest = max(slowest, json.loads(out.strip().splitlines()[-1])["run_s"])
        pairs += int(re.search(r"Decoded (\d+) pairs", out + err).group(1))
    sample = (f"{cores} concurrent processes of the reference (unmodified sources, -O3 -DAVX -mavx), each one job of cfg2 cut "
              f"into {REF_JOBS} jobs (jobs/jobInd): {pairs} pairs x {N_SITES} sites per step")
    return float(pairs) * N_SITES, slowest, "reference", sample


def port_sample(cores, n_pairs):
    from oracle import pyoracle
    pyoracle.build()
    _declare_sample(pyoracle)
    root = make_dataset(0)
    o = pyoracle.Oracle(root, DQ, f"{WORK}/ref_out", hashing=False, time=50, noConditionalAgeEstimates=True,
                        doPerPairMAP=True, doPerPairPosteriorMean=True, batchSize=32)
    t0 = time.time()
    ps = pyoracle.lib().fo_decode_sample(o._h, n_pairs, cores)
    return ps, time.time() - t0, "port", f"first {n_pairs} pairs of the job x {N_SITES} sites, {cores} threads (oracle port)"


def run_reference(args, rank, world):
    """CPU arm: the reference's own implementation (oracle/_ref/ref_fastsmc_avx, kind "reference"; the oracle port if that
    binary is absent) on all host cores, each step a bounded sample of cfg2."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    times, pair_sites, kind, sample = [], 0.0, "port", ""
    for it in range(args.warmup + args.steps):
        r = reference_sample(cores) or port_sample(cores, 32 * max(cores * 2, 16))
        if it >= args.warmup:
            times.append(r[1])
            pair_sites, kind, sample = r[0], r[2], r[3]
    ms = 1e3 * float(np.mean(times))
    value = pair_sites / (ms / 1e3)
    line = {"impl": "reference", "metric": "hmm_pair_sites_per_s", "value": value, "unit": "pair-sites/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": value, "unit": "pair-sites/s", "cores": cores, "kind": kind, "sample": sample,
                             "per_thread": value / cores},
            "e2e": {"value": value, "unit": "pair-sites/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def cpu_baseline():
    cores = os.cpu_count() or 1
    ps, dt, kind, sample = reference_sample(cores) or port_sample(cores, 64 * cores)
    return {"value": ps / dt, "unit": "pair-sites/s", "cores": cores, "kind": kind, "sample": sample + f", {dt:.1f} s",
            "per_thread": ps / dt / cores}


def dump_segments(directory, segments, tiles, prefix=""):
    """The segment records that a caller of the timed path receives, one DIR/<prefix>segment_<field>.npy per field, in the
    records' order (pair row, start site): the haplotype pair of the record's row (hapA, hapB), its sites and its level as
    float64 (exact), its scores (prob, postMean, mapTime) as the float32 the kernels write.  cfg2 gives ~4.6e5 records,
    ~28 MB in all."""
    os.makedirs(directory, exist_ok=True)
    row = segments["pair"].astype(np.int64)
    fields = {"hapA": tiles["hapA"].reshape(-1)[row], "hapB": tiles["hapB"].reshape(-1)[row]}
    fields.update({f: segments[f] for f in ("posStart", "posEnd", "mapState", "level", "prob", "postMean", "mapTime")})
    for name, v in fields.items():
        np.save(os.path.join(directory, f"{prefix}segment_{name}.npy"),
                v.astype(np.float32 if v.dtype == np.float32 else np.float64))


def max_over_ranks(value, world, device="cuda"):
    """Step time of the job = the slowest rank's (the only cross-rank operation of the benchmark)."""
    if world == 1:
        return float(value)
    import torch
    import torch.distributed as dist
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value, world, device="cuda"):
    if world == 1:
        return value
    import torch
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


JOBS_SAMPLES = int(os.environ.get("FSMC_BENCH_JOBS_SAMPLES", 12000))  # diploid samples of the cfg4-family data set
JOBS_SITES, JOBS_SPAN_BP, JOBS_CHROM, JOBS_J = 18022, 64_000_000, 20, 64   # chr20 array SNPs (SURVEY §8d config #4)


def jobs_run(asmc, rank, world, local, dist):
    """North-star partition (BASELINE.json configs[3] family): ONE data set, hashing + decoding with FastSMC_exe's default
    flags, cut into J = 64 jobs by the reference's jobs/jobInd geometry; the ranks take job indices from a shared counter
    (longest first) and each job is one ASMC::FastSMC(params, Data::forJob(whole, params)).run(), writing its own
    <out>.<jobInd>.<jobs>.FastSMC.ibd.gz.  No collective on the data path.  Returns (rank 0) the job-set wall time = slowest
    rank, and the host/kernel seconds per rank that explain it."""
    import torch
    from fastsmc_b200 import synth
    root = f"{WORK}/cfg4s_{JOBS_SAMPLES}x{JOBS_SITES}"
    if rank == 0 and not os.path.exists(root + ".hap.gz"):
        synth.dataset(root, 2 * JOBS_SAMPLES, JOBS_SITES, JOBS_SPAN_BP, JOBS_CHROM, SEED + 2)
    if dist:
        dist.barrier()
    p = asmc.DecodingParams()
    p.verbose = False
    p.inFileRoot, p.decodingQuantFile, p.outFileRoot = root, DQ, f"{WORK}/jobs_out/r{rank}"
    os.makedirs(f"{WORK}/jobs_out", exist_ok=True)
    p.decodingModeString, p.foldData, p.usingCSFS = "array", True, True
    p.FastSMC, p.hashing, p.batchSize, p.time, p.min_m = True, True, 32, 50, 1.5
    p.doPerPairMAP = p.doPerPairPosteriorMean = p.outputIbdSegmentLength = True
    p.useKnownSeed = True
    p.device = local
    p.jobs, p.jobInd = 1, 1
    p.validateParamsFastSMC()
    t0 = time.perf_counter()
    whole = asmc.Data(p)
    read_s = time.perf_counter() - t0
    p.jobs = JOBS_J
    order = asmc.pyASMC.jobOrder(JOBS_J)
    if dist:
        store = dist.distributed_c10d._get_default_store()
        key = "fsmc_jobs_next"
        def next_job():
            i = store.add(key, 1) - 1
            return order[i] if i < len(order) else 0
        dist.barrier()
    else:
        it = iter(order)
        def next_job():
            return next(it, 0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    # two host threads on the rank's GPU: one job's host stages overlap the other's kernels
    reports = asmc.pyASMC.runJobs(p, whole, next_job, [local, local])
    wall = time.perf_counter() - t0
    errors = [r.error for r in reports if r.error]
    if errors:
        raise RuntimeError("jobs_run: " + errors[0])
    mine = {"rank": rank, "jobs": len(reports), "wall_s": wall, "read_s": read_s,
            "pair_sites": sum(r.pairSites for r in reports), "candidates": sum(r.candidates for r in reports),
            "segments": sum(r.segments for r in reports),
            "decode_kernel_s": sum(r.kernelMs for r in reports) / 1e3, "seed_kernel_s": sum(r.seedMs for r in reports) / 1e3,
            "host_prepare_s": sum(r.prepareSeconds for r in reports), "host_prepare_cut_s": sum(r.cutSeconds for r in reports),
            "host_prepare_tables_s": sum(r.tablesSeconds for r in reports), "host_prepare_upload_s": sum(r.uploadSeconds for r in reports),
            "host_seed_call_s": sum(r.seedSeconds for r in reports),
            "host_order_s": sum(r.orderSeconds for r in reports), "host_decode_calls_s": sum(r.decodeSeconds for r in reports),
            "host_output_s": sum(r.outputSeconds for r in reports)}
    if dist:
        gathered = [None] * world
        dist.all_gather_object(gathered, mine)
    else:
        gathered = [mine]
    if rank != 0:
        return None
    slowest = max(gathered, key=lambda g: g["wall_s"])
    total_ps = sum(g["pair_sites"] for g in gathered)
    stages = {k: slowest[k] for k in ("decode_kernel_s", "seed_kernel_s", "host_prepare_s", "host_seed_call_s", "host_order_s",
                                      "host_decode_calls_s", "host_output_s")}
    host_stages = {k: v for k, v in stages.items() if k.startswith("host_")}
    return {"workload": f"cfg4 family: {JOBS_SAMPLES} synthetic diploid samples x {JOBS_SITES} chr20 array SNPs, hashing + decoding "
                        f"(min_m 1.5, time 50, FastSMC_exe default flags), J = {JOBS_J} jobs (jobs/jobInd) dealt to {world} GPU(s) "
                        "from a shared counter, 2 host threads per GPU, files -> per-job .ibd.gz",
            "scaling": "strong", "n_gpus": world, "wall_s": slowest["wall_s"], "pair_sites": total_ps,
            "pair_sites_per_s": total_ps / slowest["wall_s"], "candidates": sum(g["candidates"] for g in gathered),
            "segments": sum(g["segments"] for g in gathered), "read_s_per_rank": max(g["read_s"] for g in gathered),
            "host_cores": os.cpu_count(),
            "slowest_rank": slowest,
            "limiting_stage": max(host_stages, key=host_stages.get) if sum(host_stages.values()) > 2 * (stages["decode_kernel_s"] + stages["seed_kernel_s"]) else "kernels",
            "note": "stage seconds are summed over the rank's jobs (two jobs run concurrently, so they can exceed wall_s)",
            "per_rank": gathered}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-run", action="store_true", help="skip the one-off FastSMC.run() wall-clock measurement")
    ap.add_argument("--no-jobs-run", action="store_true", help="skip the jobs/jobInd-partitioned hashing run (jobs_run)")
    ap.add_argument("--no-states159", action="store_true", help="skip the 159-state legs (state-split kernels)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the segment records of the headline run's last timed step to DIR/segment_<field>.npy "
                         "(rank<r>_segment_<field>.npy per rank under torchrun)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    from fastsmc_b200 import _native as N, asmc

    # ---- host layer: data set -> Data -> model tables (the product's own code; the oracle is not involved) ----------
    if rank == 0:
        make_dataset(0)
    if world > 1:
        dist.barrier()
    root = dataset_root(0)
    p = asmc.DecodingParams()
    p.verbose = False
    p.inFileRoot, p.decodingQuantFile, p.outFileRoot = root, DQ, f"{WORK}/r{rank}/out"
    p.decodingModeString, p.foldData, p.usingCSFS = "array", True, True
    p.FastSMC, p.hashing, p.batchSize, p.time = True, False, 32, 50
    p.noConditionalAgeEstimates = p.doPerPairMAP = p.doPerPairPosteriorMean = p.outputIbdSegmentLength = True
    p.useKnownSeed = True
    p.device = local
    p.validateParamsFastSMC()
    data = asmc.Data(p)
    tables = asmc.pyASMC.prepareModelTables(data, p)
    S, L = tables["emission1"].shape[1], data.sites

    a, b = all_pairs_in_reference_order(len(data.IIDList))
    tiles = tiles_for(a, b, L, world, rank)  # this rank's share of the job's batches
    flags = N.CALL_SEGMENTS | N.SEG_AGE
    pair_sites = float(len(a)) * L                       # the whole job
    my_pair_sites = float(tiles["tilePairs"].sum()) * L  # this rank's share

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    class Lane:
        """One decode context with its own stream and a resident plan of this rank's share.  (Alternating the steps over
        two such lanes, so that the last tiles of one step share the GPU with the first tiles of the next, was measured
        and is slower: 348 vs 340 ms per step at N=1, and 393 vs 292 ms for the narrow kernel — two persistent kernels
        of 296 CTAs each do not interleave well.  One lane it is.)"""

        def __init__(self, model_tables):
            self.ctx = N.Context(local)
            # a real (non-default) torch stream: handle 0 would mean "the context's own stream" to fsmc_ctx_set_stream
            self.stream = torch.cuda.Stream(device=local)
            self.ctx.set_stream(self.stream.cuda_stream)
            self.ctx.set_model(**model_tables)
            self.ctx.set_haplotypes(data.hapBits, L)
            self.plan = self.ctx.plan(tiles, flags, segment_capacity=1 << 21)

        def close(self):
            self.plan.close()
            self.ctx.close()

    def timed_steps(lanes, sampler=None):
        """args.warmup untimed steps, then exactly args.steps steps alternating over the lanes; returns the device time in
        ms from the first launch to the end of the last kernel on either stream, and the lanes' collected results."""
        for k in range(max(args.warmup, len(lanes))):  # every lane at least once
            lanes[k % len(lanes)].plan.launch()
        barrier()
        for ln in lanes:
            ln.plan.collect()
        start = torch.cuda.Event(enable_timing=True)
        ends = [torch.cuda.Event(enable_timing=True) for _ in lanes]
        barrier()
        ctx_mgr = sampler if sampler is not None else ClockSampler(local)
        with ctx_mgr:
            start.record(lanes[0].stream)
            for ln in lanes[1:]:
                ln.stream.wait_event(start)
            for k in range(args.steps):
                lanes[k % len(lanes)].plan.launch()
            for ln, e in zip(lanes, ends):
                e.record(ln.stream)
            barrier()
        total = max(start.elapsed_time(e) for e in ends)
        used = lanes[:min(len(lanes), args.steps)]
        return total, [ln.plan.collect() for ln in used]

    # ---- value: pair list resident in HBM, kernels only ----------------------------------------------------------------
    lanes = [Lane(tables)]
    clocks = ClockSampler(local)
    rank0_ms, results = timed_steps(lanes, clocks)
    r = results[0]
    if args.dump_outputs:
        dump_segments(args.dump_outputs, r.segments, tiles, f"rank{rank}_" if world > 1 else "")
    per_step = [rank0_ms / args.steps]
    n_segments = int(r.stats.numSegments)
    scratch_bytes = int(r.stats.scratchBytes)
    launches_per_step = int(r.stats.kernelLaunches)
    sparse = {"on": bool(r.stats.sparseKernel), "block_sites": int(r.stats.checkpointSites), "items": int(r.stats.sparseItems),
              "checkpoint_bytes": int(r.stats.checkpointBytes)}
    ms_per_step = max_over_ranks(rank0_ms, world) / args.steps
    value = pair_sites / (ms_per_step / 1e3)
    n_segments = int(sum_over_ranks(n_segments, world))
    for ln in lanes:
        ln.plan.close()
    ctx = lanes[0].ctx   # the e2e leg below reuses the context

    # ---- the same job with FastSMC's command-line default age estimates (conditional on TMRCA < time, i.e.
    # noConditionalAgeEstimates off: only the states below the threshold are consumed -> decodeNarrowKernel) ------------
    cond_tables = dict(tables, age_threshold=tables["state_threshold"])
    lanes2 = [Lane(cond_tables)]
    narrow_total_ms, results2 = timed_steps(lanes2)
    narrow_rank0_ms = narrow_total_ms / args.steps
    narrow_ms = max_over_ranks(narrow_total_ms, world) / args.steps
    r2 = results2[0]
    narrow = {"value": pair_sites / (narrow_ms / 1e3), "unit": "pair-sites/s", "ms_per_step": narrow_ms,
              "kernel": "decodeNarrowKernel<69>" if r2.stats.narrowKernel else "decodeFastKernel<69>",
              "segments_per_step": int(sum_over_ranks(int(r2.stats.numSegments), world)), "scratch_bytes": int(r2.stats.scratchBytes),
              "flags": "as the headline run but age estimates conditional on TMRCA < time (FastSMC_exe default)"}
    for ln in lanes2:
        ln.close()

    # ---- cfg2 repeated with the 159-state table of FASTSMC_EXAMPLE (SURVEY 8(d) config #2), rank 0's first 2 048 batches,
    # both flag sets: the lane-split kernels (decode_lane.cuh) ------------------------------------------------------------
    states159 = None
    if rank == 0 and not args.no_states159:
        p.decodingQuantFile = DQ_159
        tables159 = asmc.pyASMC.prepareModelTables(data, p)
        p.decodingQuantFile = DQ
        S159 = tables159["emission1"].shape[1]
        sub = {k: (v[:2048] if k != "rows" else v) for k, v in tiles.items()}
        sub_pair_sites = float(sub["tilePairs"].sum()) * L
        states159 = {"workload": f"cfg2's first {len(sub['tilePairs'])} batches x {L} sites with the {S159}-state example table", "states": int(S159)}
        for label, age in (("all_state_ages", S159), ("default_flags", tables159["state_threshold"])):
            c159 = N.Context(local)
            st159 = torch.cuda.Stream(device=local)
            c159.set_stream(st159.cuda_stream)
            c159.set_model(**dict(tables159, age_threshold=age))
            c159.set_haplotypes(data.hapBits, L)
            pl = c159.plan(sub, flags, segment_capacity=1 << 20)
            pl.launch()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n159 = args.steps
            e0.record(st159)
            for _ in range(n159):
                pl.launch()
            e1.record(st159)
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / n159
            r159 = pl.collect()
            tf = sub_pair_sites / (ms / 1e3) * FLOPS_PER_PAIR_SITE_STATE * S159 / 1e12
            states159[label] = {"value": sub_pair_sites / (ms / 1e3), "unit": "pair-sites/s", "ms_per_step": ms,
                                "kernel": (f"decodeLaneKernel<{int(r159.stats.statesKernel)}, records>" if r159.stats.narrowKernel
                                           else f"decodeLaneWideKernel<{int(r159.stats.statesKernel)}>") + " (states cut across the lanes of a warp, "
                                          "8 pairs per warp, one 32-pair tile per CTA)",
                                "fp32_tflops": tf, "fp32_frac_nominal": tf / (torch.cuda.get_device_properties(local).multi_processor_count * 128 * 2 * 1.965e9 / 1e12)}
            pl.close()
            c159.close()

    # ---- e2e: fsmc_decode with host buffers -----------------------------------------------------------------------------
    for _ in range(2):
        ctx.decode(tiles, flags, segment_capacity=1 << 21)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        res = ctx.decode(tiles, flags, segment_capacity=1 << 21)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / args.steps
    e2e_s = max_over_ranks(e2e_s, world)
    h2d = sum(tiles[k].nbytes for k in ("hapA", "hapB", "tilePairs", "tileFrom", "tileTo", "tileScanFrom", "tileScanTo"))
    d2h = int(res.stats.numSegments) * N.SEGMENT_DTYPE.itemsize + 16
    e2e = {"value": pair_sites / e2e_s, "unit": "pair-sites/s", "h2d_bytes_per_step": int(h2d),
           "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * e2e_s,
           "call": "fsmc_decode (host pair lists in, host segment records out)"}

    # ---- one whole FastSMC.run(): read files, model preparation, decode, write .ibd.gz ------------------------------------
    ibd_wall = None
    if not args.no_e2e_run and rank == 0 and world == 1:
        t0 = time.perf_counter()
        f = asmc.FastSMC(p)
        f.run()
        ibd_wall = {"seconds": time.perf_counter() - t0, "segments": int(f.hmm().getNumberOfDetectedSegments()),
                    "decode_wall_s": f.hmm().getRunStats().decodeWallS, "output_wall_s": f.hmm().getRunStats().outputWallS,
                    "what": "FastSMC(params).run(): .hap.gz/.map/.samples + decoding quantities -> .ibd.gz"}
        del f

    jobs = None
    if not args.no_jobs_run:
        jobs = jobs_run(asmc, rank, world, local, dist if world > 1 else None)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"
        kernel_ms = float(np.mean(per_step))
        prop = torch.cuda.get_device_properties(local)
        fp32_peak = prop.multi_processor_count * 128 * 2 * 1.965e9 / 1e12
        fp32_achieved = my_pair_sites * FLOPS_PER_PAIR_SITE_STATE * S / (kernel_ms / 1e3) / 1e12
        if sparse["on"]:
            # decode_sparse.cuh: narrow sweeps + beta checkpoints + refinement of the IBD runs.  Algorithmic HBM bytes per
            # pair-site: 2 genotype bits, the narrow record written by the backward and read by the forward sweep
            # (2 x 16 B), one full beta vector (Spad floats) per block of `block_sites` sites
            bytes_per_pair_site = 0.25 + 32.0 + 4.0 * ((S + 3) // 4 * 4) / sparse["block_sites"]
            kernel_name = "decodeNarrowKernel<69, sparse> (+ refineKernel<69>, finalizeSegmentsKernel: ~6 % of the step)"
            ncu_bytes = NCU_SPARSE_DRAM_BYTES_PER_PAIR_SITE
            traffic_src = "ncu --set full capture of the kernel in this bench (profiles/r2_p2_decodeNarrowSparse_ncu_full.txt), scaled by pair-sites"
        else:
            # the backward sweep writes beta[S] floats and the forward sweep reads them back (8*S) + 2 genotype bits
            bytes_per_pair_site = 8.0 * S + 0.25
            kernel_name = "decodeFastKernel<69>"
            ncu_bytes = NCU_DRAM_BYTES_PER_PAIR_SITE
            traffic_src = "ncu --set full capture of a 37888-pair launch (profiles/r1_v4_decodeFast_s69_ncu_full.txt), scaled by pair-sites"
        achieved = my_pair_sites * bytes_per_pair_site / (kernel_ms / 1e3) / 1e9  # rank 0's launches
        hbm_roofline = {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                        "traffic": ncu_bytes * my_pair_sites, "traffic_source": traffic_src,
                        "algorithmic_bytes": bytes_per_pair_site * my_pair_sites, "peak_source": peak_src,
                        "algorithmic_bytes_per_pair_site": bytes_per_pair_site}
        fp32_roofline = {"bound": "fp32", "achieved": fp32_achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": fp32_achieved / fp32_peak, "traffic": ncu_bytes * my_pair_sites, "traffic_source": traffic_src,
                         "flops_per_pair_site": FLOPS_PER_PAIR_SITE_STATE * S,
                         "flops_source": "SURVEY.md 8(d): 35 x S algorithmic flops of the reference's recurrences per pair-site",
                         "peak_source": "SMs x 128 lanes x 2 x 1.965 GHz (nominal FP32 pipe; no tensor-core work on this path)"}
        # the kernel's binding roofline comes first: FP32 pipe for the sparse path, HBM for the kernel that streams beta
        roofline = dict(fp32_roofline if sparse["on"] else hbm_roofline, kernel=kernel_name, kernel_ms=kernel_ms)
        other = dict(hbm_roofline if sparse["on"] else fp32_roofline)
        line = {
            "metric": "hmm_pair_sites_per_s", "value": value, "unit": "pair-sites/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs": int(len(a)), "sites": int(L), "states": int(S),
                       "pair_sites_per_step": pair_sites, "pair_sites_per_step_rank0": my_pair_sites,
                       "segments_per_step": n_segments,
                       "flags": "segment length + per-segment posterior mean + MAP over ALL states (noConditionalAgeEstimates), "
                                "the reference's regression-test / FastSMC-constructor defaults",
                       "l2": f"no flush needed: each step streams {(scratch_bytes + sparse['checkpoint_bytes']) / 2**30:.0f} GiB of "
                             "backward-sweep records / checkpoints through HBM (>> 126 MB L2)", "parallelism": f"the job's {(len(a) + 31) // 32} reference batches dealt to {world} GPU(s) in contiguous shares; "
                                      "no collective on the data path"},
            "roofline": roofline, ("roofline_hbm" if sparse["on"] else "roofline_fp32"): other, "sparse_age_estimates": sparse,
            "default_flags": dict(narrow, roofline={"bound": "fp32", "achieved": my_pair_sites / (narrow_rank0_ms / 1e3) * FLOPS_PER_PAIR_SITE_STATE * S / 1e12,
                                                     "peak": fp32_peak, "unit": "TFLOP/s",
                                                     "frac": my_pair_sites / (narrow_rank0_ms / 1e3) * FLOPS_PER_PAIR_SITE_STATE * S / 1e12 / fp32_peak,
                                                     # DRAM bytes of one launch, from the ncu --set full capture
                                                     # profiles/r1_v4_decodeNarrow_s69_ncu_full.txt (12.15 GB for
                                                     # 37 888 pairs x 10 000 sites), scaled by pair-sites
                                                     "traffic": NCU_NARROW_DRAM_BYTES_PER_PAIR_SITE * my_pair_sites}),
            "e2e": e2e, "gpu_launches": launches_per_step * args.steps, "clocks": clocks.summary(),
            "ibd_wall": ibd_wall, "jobs_run": jobs, "states159": states159,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _declare_sample(pyoracle):
    import ctypes as C
    L = pyoracle.lib()
    L.fo_decode_sample.restype = C.c_double
    L.fo_decode_sample.argtypes = [C.c_void_p, C.c_long, C.c_int]


if __name__ == "__main__":
    main()
