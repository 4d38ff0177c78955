#!/usr/bin/env python
"""Small decode requests through every production kernel family, sized for compute-sanitizer (racecheck / memcheck):

    compute-sanitizer --tool racecheck python tools/racecheck_probe.py

The mbarrier / bulk-copy ring protocols (decode_fast.cuh, decode_lane.cuh, decode_sparse.cuh) are what the tool checks;
the probe only asserts that every kernel ran and produced segments.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from fastsmc_b200 import _native as N, asmc, synth  # noqa: E402

DQ69 = os.path.join(ROOT, "data", "30-100-2000.decodingQuantities.gz")
EX = os.path.join(ROOT, "tests", "golden", "fastsmc_example", "example")


def context(root, dq, conditional):
    p = asmc.DecodingParams()
    p.verbose = False
    p.inFileRoot, p.decodingQuantFile, p.outFileRoot = root, dq, "/tmp/fsmc_racecheck/out"
    p.decodingModeString, p.foldData, p.usingCSFS = "array", True, True
    p.FastSMC, p.hashing, p.batchSize, p.time = True, False, 32, 50
    p.noConditionalAgeEstimates = not conditional
    p.doPerPairMAP = p.doPerPairPosteriorMean = p.outputIbdSegmentLength = True
    p.useKnownSeed = True
    p.validateParamsFastSMC()
    data = asmc.Data(p)
    tables = asmc.pyASMC.prepareModelTables(data, p)
    ctx = N.Context(0)
    ctx.set_model(**tables)
    ctx.set_haplotypes(data.hapBits, data.sites)
    return ctx, data


def main():
    os.makedirs("/tmp/fsmc_racecheck", exist_ok=True)
    root = "/tmp/fsmc_racecheck/syn"
    if not os.path.exists(root + ".hap.gz"):
        synth.dataset(root, 320, 640, 2_000_000, 1, 99)
    rng = np.random.default_rng(1)
    n_pairs = 5 * 32 + 7
    for label, r, dq, conditional in (
            ("wide69", root, DQ69, False), ("narrow69", root, DQ69, True),
            ("lane-wide159", EX, EX + ".decodingQuantities.gz", False),
            ("lane-narrow159", EX, EX + ".decodingQuantities.gz", True)):
        ctx, data = context(r, dq, conditional)
        H, L = data.hapBits.shape[0], min(data.sites, 640)
        a = rng.integers(0, H - 1, n_pairs).astype(np.uint32)
        b = (a + 1 + rng.integers(0, H - 1, n_pairs) % (H - 1 - a)).astype(np.uint32)
        nb = (n_pairs + 31) // 32
        win = np.array([[(7 * i) % 50, L - (11 * i) % 60] for i in range(nb)], np.int32)
        tiles = ctx.make_tiles(a, b, windows=win, sites=data.sites)
        res = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE, segment_capacity=1 << 16)
        res2 = ctx.decode(tiles, N.SITE_IBD | N.SITE_MEAN) if not conditional else ctx.decode(tiles, N.SITE_IBD)
        print(label, "segments", len(res.segments), "narrow", res.stats.narrowKernel, "tileWarps", res.stats.tileWarps,
              "states", res.stats.statesKernel, "ibd finite", bool(np.isfinite(res2.site_ibd).all()), flush=True)
        ctx.close()


if __name__ == "__main__":
    main()
