"""FastSMC.run() writing the .bibd.gz against fastsmc_segments_cuda (segments left in HBM as torch tensors), on two
workloads: cfg2 (1 000 haplotypes x 10 000 SNPs, all pairs, hashing off) and cfg3's density with hashing (10 000 diploid
samples x 50 000 SNPs at UKBB chr1 array density).

    python tools/device_segments_probe.py [out.json] [reps] [cfg3_diploid]

Per path and repetition: wall time of the call (the tensor path ends with a device synchronise), decode kernel time (CUDA
events, HMM run statistics) and the bytes of decode outputs copied device -> host.  The two paths alternate after one
untimed run of each; the data set is loaded once (asmc.Data) and handed to both.  Both paths must give the same records.
"""
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from fastsmc_b200 import asmc, synth  # noqa: E402
from fastsmc_b200.cuda_results import fastsmc_segments_cuda  # noqa: E402

out_json = sys.argv[1] if len(sys.argv) > 1 else None
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
cfg3_dip = int(sys.argv[3]) if len(sys.argv) > 3 else 10_000
DQ = os.path.join(ROOT, "data", "30-100-2000.decodingQuantities.gz")
WORK = os.path.join(tempfile.gettempdir(), f"fsmc_segments_probe_{os.getuid()}")

if not torch.cuda.is_available():
    raise SystemExit("device_segments_probe: no CUDA device (timings are only meaningful on the GPU)")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()


def params(root, hashing, bit_cache):
    p = asmc.DecodingParams()
    p.verbose = False
    p.inFileRoot, p.decodingQuantFile, p.outFileRoot = root, DQ, root + ".out"
    p.decodingModeString, p.foldData, p.usingCSFS = "array", True, True
    p.FastSMC, p.hashing, p.batchSize, p.time = True, hashing, 32, 50
    p.min_m, p.gap = 1.5, 1
    p.doPerPairMAP = p.doPerPairPosteriorMean = p.outputIbdSegmentLength = True
    p.noConditionalAgeEstimates = False  # FastSMC_exe's default conditional age estimates
    p.useKnownSeed = True
    p.BIN_OUT = True
    p.hapBitCache = bit_cache
    p.validateParamsFastSMC()
    return p


def file_run(p, data):
    f = asmc.FastSMC(p, data)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    f.run()
    wall = time.perf_counter() - t0
    st = f.hmm().getRunStats()
    return dict(wall_s=wall, kernel_ms=st.kernelMs, d2h_bytes=st.d2hBytes, segments=st.segments,
                output_wall_s=st.outputWallS)


def tensor_run(p, data):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = fastsmc_segments_cuda(p, data)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return dict(wall_s=wall, kernel_ms=res.decode_kernel_ms, d2h_bytes=res.d2h_bytes, segments=res.n_segments), res


def records_match(p, res, limit=200_000):
    """The first `limit` records of the file against the tensors (start bp and score bits); the counts are compared in full."""
    r = asmc.BinaryDataReader(f"{p.outFileRoot}.1.1.FastSMC.bibd.gz")
    starts, scores = res.start_bp[:limit].cpu().numpy(), res.score[:limit].cpu().numpy()
    n = 0
    while n < min(limit, res.n_segments) and r.moreLinesInFile():
        line = r.getNextLine()
        if line.ibdStart != starts[n] or np.float32(line.ibdScore) != scores[n]:
            return False
        n += 1
    return n == min(limit, res.n_segments)


def workload(name, root, hashing, bit_cache):
    p = params(root, hashing, bit_cache)
    t0 = time.perf_counter()
    data = asmc.Data(p)
    rep = {"workload": name, "load_s": time.perf_counter() - t0, "file": [], "tensors": []}
    file_run(p, data)  # untimed: first launches, pooled contexts
    _, res = tensor_run(p, data)
    rep["first_records_match_file"] = records_match(p, res)
    del res
    for _ in range(reps):
        rep["file"].append(file_run(p, data))
        rep["tensors"].append(tensor_run(p, data)[0])
    print(json.dumps(rep, indent=1), flush=True)
    return rep


report = {"gpu": gpu[:1], "host_cores": os.cpu_count(), "workloads": []}
root2 = os.path.join(WORK, "cfg2_1000x10000")
if not os.path.exists(root2 + ".hap.gz"):
    synth.dataset(root2, 1000, 10_000, 30_000_000, 1, 20201117 + 2)  # bench.py's cfg2
report["workloads"].append(workload("cfg2: 1000 haplotypes x 10000 SNPs, all pairs, hashing off", root2, False, False))
root3 = os.path.join(WORK, f"cfg3_{cfg3_dip}x50000")
if not os.path.exists(root3 + ".hap.gz.fsmcbits"):
    synth.packed_dataset(root3, 2 * cfg3_dip, 50_000, 240_000_000, 1, 20201117 + 3)
report["workloads"].append(workload(f"cfg3 density: {cfg3_dip} diploid x 50000 SNPs, hashing", root3, True, True))
if out_json:
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    json.dump(report, open(out_json, "w"), indent=1)
