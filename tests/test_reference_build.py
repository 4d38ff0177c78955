"""The oracle pinned to the REFERENCE ITSELF: the reference's own sources (HMM.cpp, FastSMC.cpp, HASHING/*, Data.cpp, ...)
compiled unmodified against the shim headers of oracle/shim (oracle/Makefile) write the same .ibd.gz as the oracle
restatement, line for line — in the NO_SSE flavour (exact 1/x) and in the reference's default AVX flavour (approximate
reciprocal), with hashing (seeding + boost node order + batching + caller) and without (job slice of the all-pairs
enumeration).  The reference's committed goldens were produced with an older libstdc++ (std::shuffle differs, SURVEY F11),
which is why this build is compared with the oracle and not with the golden files; the oracle reproduces those too
(test_oracle_golden.py).

The reference's sources are not part of this repository, so the reference build exists only where oracle/Makefile found a
reference checkout.  tests/golden/reference_build_outputs.json keeps, for every configuration below, the line count, the
SHA-256 and a sample of the lines of the .ibd.gz text on which the oracle and the reference build agreed; the oracle must
still write exactly that text.  Where the reference build is present its output is compared as well.
`python tests/test_reference_build.py` rewrites the record from the oracle (after a change the reference build confirms)."""
import gzip
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, GOLDEN, REGRESSION_PARAMS

RECORD = os.path.join(GOLDEN, "reference_build_outputs.json")
FLAVOURS = [("nosse", False), ("avx", True)]
JOBS = {"hashing": dict(hashing=True, jobs=1, jobInd=1), "hashing-job3of4": dict(hashing=True, jobs=4, jobInd=3),
        "allpairs-job8of25": dict(hashing=False, jobs=25, jobInd=8)}
DEFAULT_FLAGS = dict(hashing=True, noConditionalAgeEstimates=False)
SEEDING = {"skip0.13": dict(skip=0.13), "skip0.145-gap2": dict(skip=0.145, gap=2, min_m=2.5), "max_seeds20": dict(max_seeds=20),
           "max_seeds8-skip0.13": dict(max_seeds=8, skip=0.13)}
SAMPLED_LINES = 8


def _lines(path):
    with gzip.open(path, "rb") as f:
        return f.read().splitlines()


def _dense_dataset(directory):
    """Dense synthetic data (6 founders): a quarter to a half of the words are low complexity at the SEEDING thresholds,
    buckets of 20-60 haplotypes."""
    from fastsmc_b200 import synth
    root = os.path.join(str(directory), "dense")
    synth.dataset(root, 200, 1920, 3000 * 1920, 1, 11, founders=6)
    return root


def _dense_options(options):
    return dict(dict(hashing=True, min_m=2.0), **options)


def configurations(dense_root):
    """(test id, reference flavour, SIMD flavour of the oracle, data set, run options) of every test below."""
    for job, options in JOBS.items():
        for flavour, simd in FLAVOURS:
            yield f"test_oracle_equals_reference_build[{job}-{flavour}-{simd}]", flavour, simd, FASTSMC_EXAMPLE, options
    yield "test_reference_default_flags_conditional_age_estimates", "nosse", False, FASTSMC_EXAMPLE, DEFAULT_FLAGS
    for name, options in SEEDING.items():
        yield (f"test_oracle_equals_reference_build_with_skip_and_max_seeds[{name}]", "nosse", False, dense_root,
               _dense_options(options))


def _outputs(oracle_mod, directory, flavour, simd, in_root, options):
    """.ibd.gz lines of the oracle, and of the reference build of `flavour` (None where it is not built), for one run."""
    directory = str(directory)
    o = oracle_mod.Oracle(in_root, FASTSMC_EXAMPLE_DQ, os.path.join(directory, "orc"), shuffleFlavor=0, simdFlavor=simd,
                          **dict(REGRESSION_PARAMS, **options))
    path = os.path.join(directory, "oracle.ibd.gz")
    o.run(path)
    ref = None
    if oracle_mod.reference_binary(flavour) is not None:
        out = os.path.join(directory, "ref")
        oracle_mod.reference_run(flavour, in_root, FASTSMC_EXAMPLE_DQ, out, **options)
        ref = _lines(f"{out}.{options.get('jobInd', 1)}.{options.get('jobs', 1)}.FastSMC.ibd.gz")
    return _lines(path), ref


def _summary(lines):
    picked = np.unique(np.linspace(0, len(lines) - 1, SAMPLED_LINES).astype(int))
    return {"lines": len(lines), "sha256": hashlib.sha256(b"\n".join(lines)).hexdigest(),
            "sample": {str(i): lines[i].decode() for i in picked}}


def _check(oracle_mod, tmp_path, test_id, flavour, simd, in_root, options, min_lines):
    mine, ref = _outputs(oracle_mod, tmp_path, flavour, simd, in_root, options)
    want = json.load(open(RECORD))["outputs"][test_id]
    assert len(mine) == want["lines"] > min_lines
    for i, line in want["sample"].items():
        assert mine[int(i)].decode() == line, f"line {i}"
    assert _summary(mine)["sha256"] == want["sha256"]
    if ref is not None:
        assert mine == ref


@pytest.mark.parametrize("flavour,simd", FLAVOURS)
@pytest.mark.parametrize("job", list(JOBS))
def test_oracle_equals_reference_build(oracle_mod, tmp_path, request, flavour, simd, job):
    _check(oracle_mod, tmp_path, request.node.name, flavour, simd, FASTSMC_EXAMPLE, JOBS[job], 100)


def test_reference_default_flags_conditional_age_estimates(oracle_mod, tmp_path, request):
    """FastSMC_exe's default age estimates (conditional on TMRCA < time) through the reference build vs the oracle."""
    _check(oracle_mod, tmp_path, request.node.name, "nosse", False, FASTSMC_EXAMPLE, DEFAULT_FLAGS, 100)


@pytest.mark.parametrize("options", list(SEEDING.values()), ids=list(SEEDING))
def test_oracle_equals_reference_build_with_skip_and_max_seeds(oracle_mod, tmp_path, request, options):
    """The non-default seeding options (low-complexity word skipping, sub-hashing of oversized buckets; FastSMC.cpp:208-219,
    HASHING/SeedHash.hpp:56-69, 85-93) on dense synthetic data: reference build vs the oracle, whole .ibd.gz."""
    root = _dense_dataset(tmp_path)
    _check(oracle_mod, tmp_path, request.node.name, "nosse", False, root, _dense_options(options), 500)


if __name__ == "__main__":
    import tempfile
    from oracle import pyoracle
    pyoracle.build()
    outputs = {}
    with tempfile.TemporaryDirectory() as work:
        dense = _dense_dataset(work)
        for test_id, flavour, simd, in_root, options in configurations(dense):
            run = os.path.join(work, str(len(outputs)))
            os.makedirs(run)
            mine, ref = _outputs(pyoracle, run, flavour, simd, in_root, options)
            assert ref is None or mine == ref, test_id
            outputs[test_id] = _summary(mine)
    with open(RECORD, "w") as f:
        json.dump({"about": "FastSMC .ibd.gz text of the oracle (oracle/) for the configurations of "
                            "tests/test_reference_build.py, which the reference build wrote line for line when it was last "
                            "compared",
                   "outputs": outputs}, f, indent=1)
        f.write("\n")
