"""ASMC.decodePairs (results on the host) against decode_pairs_cuda (results left in HBM as torch tensors) at cfg5's site
count: synthetic diploid samples x 11 528 chr22 array SNPs, a fixed sample of haplotype pairs, per-pair posterior means.

    python tools/device_outputs_probe.py [out.json] [n_pairs] [n_diploid] [reps]

Per path and repetition: wall time of the call (ended by a device synchronise), kernel time of the decode calls (CUDA events,
HMM run statistics) and the bytes of decode outputs copied device -> host.  The two paths alternate; the first call of
each on a small sample is a warm-up and not reported.  Both paths must give bit-identical means and the same minima.
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from fastsmc_b200 import asmc, synth  # noqa: E402
from fastsmc_b200.cuda_results import decode_pairs_cuda  # noqa: E402

out_json = sys.argv[1] if len(sys.argv) > 1 else None
n_pairs = int(sys.argv[2]) if len(sys.argv) > 2 else 200_000
n_dip = int(sys.argv[3]) if len(sys.argv) > 3 else 2_000
reps = int(sys.argv[4]) if len(sys.argv) > 4 else 2
SITES, SPAN, CHROM, SEED = 11_528, 35_000_000, 22, 20201117 + 5
DQ = os.path.join(ROOT, "data", "30-100-2000.decodingQuantities.gz")
root = f"/tmp/fsmc_scale/device_outputs_{n_dip}"

if not torch.cuda.is_available():
    raise SystemExit("device_outputs_probe: no CUDA device (timings are only meaningful on the GPU)")
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
rep = {"n_diploid": n_dip, "sites": SITES, "pairs": n_pairs, "outputs": "per_pair_posterior_means", "gpu": gpu[:1],
       "host_cores": os.cpu_count()}
if not os.path.exists(root + ".hap.gz"):
    synth.dataset(root, 2 * n_dip, SITES, SPAN, CHROM, SEED)

# ASMC mode, array data, CSFS, no posterior sums over all pairs (ref: ASMC.cpp:28-50 without doPosteriorSums)
p = asmc.DecodingParams(root, DQ, root + ".out", 1, 1, "array", False, True, False, False, 0.0, False, False, False, "", False,
                        False)
p.verbose = False
p.useKnownSeed = True
m = asmc.ASMC(p)
hmm = m.hmm()

rng = np.random.default_rng(SEED)
H = 2 * n_dip
a = rng.integers(0, H, n_pairs).tolist()
b = ((np.array(a) + 1 + rng.integers(0, H - 1, n_pairs)) % H).tolist()


def host(a, b):
    s0 = hmm.getRunStats()
    k0, d0 = s0.kernelMs, s0.d2hBytes
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    m.decodePairs(a, b, False, False, True, False)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    s = hmm.getRunStats()
    return {"wall_s": wall, "kernel_ms": s.kernelMs - k0, "d2h_bytes": s.d2hBytes - d0}


def device(a, b):
    s0 = hmm.getRunStats()
    k0 = s0.kernelMs
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    res = decode_pairs_cuda(m, a, b, per_pair_posterior_means=True)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    return {"wall_s": wall, "kernel_ms": hmm.getRunStats().kernelMs - k0, "d2h_bytes": res.d2h_bytes}, res


host(a[:2048], b[:2048])  # warm-up: module loads, allocations, both kernels' first launches
device(a[:2048], b[:2048])
rep["host"], rep["device"] = [], []
for i in range(reps):
    rep["host"].append(host(a, b))
    d, res = device(a, b)
    rep["device"].append(d)
    del res
    torch.cuda.empty_cache()

# the two paths agree (last host call's results are still in the ASMC object)
r = m.get_ref_of_results()
d, res = device(a, b)
got = res.per_pair_posterior_means.cpu().numpy()
want = np.array(r.per_pair_posterior_means)
rep["bit_identical_means"] = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
rep["same_minima"] = bool(np.array_equal(res.min_posterior_means.cpu().numpy().view(np.uint32),
                                         np.array(r.min_posterior_means, np.float32).view(np.uint32)) and
                          np.array_equal(res.argmin_posterior_means.cpu().numpy(), np.array(r.argmin_posterior_means)))
# column minimum alone: the matrix is pairs x sites fp32 in HBM (larger than the 126 MB L2)
mat = res.per_pair_posterior_means
from fastsmc_b200.cuda_results import _context  # noqa: E402
ctx = _context(0)
side = torch.cuda.Stream()
ctx.set_stream(side.cuda_stream)
mn = torch.empty(SITES, device="cuda")
am = torch.empty(SITES, dtype=torch.int32, device="cuda")
torch.cuda.synchronize()
ctx.column_min(mat, mn, am)
ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
ev0.record(side)
for _ in range(10):
    ctx.column_min(mat, mn, am)
ev1.record(side)
torch.cuda.synchronize()
ctx.set_stream(None)
ms = ev0.elapsed_time(ev1) / 10
rep["column_min"] = {"ms": ms, "bytes": mat.numel() * 4, "bytes_per_s": mat.numel() * 4 / (ms / 1e3)}
best = lambda k, f: min(x[f] for x in rep[k])  # noqa: E731
rep["summary"] = {"host_wall_s": best("host", "wall_s"), "device_wall_s": best("device", "wall_s"),
                  "host_kernel_s": best("host", "kernel_ms") / 1e3, "device_kernel_s": best("device", "kernel_ms") / 1e3,
                  "host_d2h_bytes": rep["host"][0]["d2h_bytes"], "device_d2h_bytes": rep["device"][0]["d2h_bytes"]}
print(json.dumps(rep, indent=1))
if out_json:
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    json.dump(rep, open(out_json, "w"), indent=1)
