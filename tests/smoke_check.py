"""smoke(): one small invocation of the CUDA hot path on cuda:0, checked against the CPU oracle (test infrastructure)."""
import os
import tempfile

import numpy as np

from conftest import FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, REGRESSION_PARAMS, context_from_oracle


def run(verbose=False):
    from fastsmc_b200 import _native as N
    from oracle import pyoracle
    with tempfile.TemporaryDirectory() as tmp:
        o = pyoracle.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, os.path.join(tmp, "o"), hashing=True, **REGRESSION_PARAMS)
        n = o.run(os.path.join(tmp, "oracle.ibd.gz"))
    ints, floats = o.segments()
    batches, cands = o.batches(), o.candidates()
    ctx = context_from_oracle(o, pyoracle)
    tiles = ctx.make_tiles(cands[:, 0], cands[:, 1], windows=batches[:, 3:5], scan=batches[:, 1:3], sites=o.sites)
    for flags, exact in ((N.CALL_SEGMENTS | N.SEG_AGE | N.EXACT, True), (N.CALL_SEGMENTS | N.SEG_AGE, False)):
        r = ctx.decode(tiles, flags)
        seg = r.segments
        assert len(seg) == n, (len(seg), n)
        assert np.array_equal(seg["posStart"], ints[:, 4]) and np.array_equal(seg["posEnd"], ints[:, 5])
        if exact:
            assert np.array_equal(seg["prob"].view(np.uint32), floats[:, 0].copy().view(np.uint32))
        else:
            np.testing.assert_allclose(seg["prob"], floats[:, 0], rtol=1e-4)
            np.testing.assert_allclose(seg["postMean"], floats[:, 1], rtol=1e-4)
        if verbose:
            print(f"smoke: {len(seg)} segments match the oracle ({'exact' if exact else 'fast'} mode), "
                  f"kernel {r.stats.kernelMs:.2f} ms, {r.stats.pairSites / r.stats.kernelMs / 1e6:.2f} G pair-sites/s")
