"""fastsmc_segments_cuda: FastSMC's IBD segments as CUDA tensors, record for record the run's own .bibd.gz (raw float32
values, so the comparison is bit for bit), and the C ABI underneath (fsmc_plan_collect_device)."""
import os

import numpy as np
import pytest

from conftest import DQ_69, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, REGRESSION_PARAMS, context_from_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def asmc():
    from fastsmc_b200 import asmc as mod
    return mod


def _params(asmc, root, dq, out, **kw):
    p = asmc.DecodingParams()
    p.verbose = False
    p.inFileRoot, p.decodingQuantFile, p.outFileRoot = root, dq, out
    p.decodingModeString, p.foldData, p.usingCSFS, p.FastSMC, p.hashing = "array", True, True, True, True
    for k, v in dict(REGRESSION_PARAMS, **kw).items():
        setattr(p, k, v)
    p.validateParamsFastSMC()
    return p


def _file_records(asmc, p):
    """FastSMC(p).run() with BIN_OUT: the records of the .bibd.gz, and the run's segment count."""
    p.BIN_OUT = True
    f = asmc.FastSMC(p)
    f.run()
    r = asmc.BinaryDataReader(f"{p.outFileRoot}.{p.jobInd}.{p.jobs}.FastSMC.bibd.gz")
    lines = []
    while r.moreLinesInFile():
        lines.append(r.getNextLine())
    return lines, f.hmm().getNumberOfDetectedSegments()


def _device(p):
    from fastsmc_b200.cuda_results import fastsmc_segments_cuda
    return fastsmc_segments_cuda(p)


def _host(res):
    return {name: (None if getattr(res, name) is None else getattr(res, name).cpu().numpy())
            for name in ("ind1", "hap1", "ind2", "hap2", "start_site", "end_site", "start_bp", "end_bp", "length_cm", "score",
                         "post_mean", "map_time")}


def _assert_same_records(lines, res, p):
    import torch
    torch.cuda.synchronize()
    h = _host(res)
    assert res.n_segments == len(lines) > 0
    assert all(v is None or len(v) == len(lines) for v in h.values())
    index = {(fam, iid): i for i, (fam, iid) in enumerate(zip(res.fam_ids, res.iids))}
    want_int = np.array([[index[l.ind1FamId, l.ind1Id], l.ind1Hap, index[l.ind2FamId, l.ind2Id], l.ind2Hap, l.ibdStart, l.ibdEnd]
                         for l in lines], np.int64)
    got_int = np.stack([h[k] for k in ("ind1", "hap1", "ind2", "hap2", "start_bp", "end_bp")], axis=1).astype(np.int64)
    bad = np.flatnonzero((want_int != got_int).any(axis=1))
    assert len(bad) == 0, f"{len(bad)} records differ, first {bad[0]}: {got_int[bad[0]]} vs {want_int[bad[0]]}"
    bits = lambda x: np.asarray(x, np.float32).view(np.uint32)  # noqa: E731
    assert np.array_equal(bits(h["length_cm"]), bits([l.lengthInCentimorgans for l in lines]))
    assert np.array_equal(bits(h["score"]), bits([l.ibdScore for l in lines]))
    if p.doPerPairPosteriorMean:
        assert np.array_equal(bits(h["post_mean"]), bits([l.postEst for l in lines]))
    else:
        assert h["post_mean"] is None
    if p.doPerPairMAP:
        assert np.array_equal(bits(h["map_time"]), bits([l.mapEst for l in lines]))
    else:
        assert h["map_time"] is None
    assert np.all(h["start_site"] <= h["end_site"])


def _no_files(directory):
    return not [f for f in os.listdir(directory) if "FastSMC" in f]


EXAMPLE_CASES = {"hashing": dict(hashing=True), "no_hashing_job7of9": dict(hashing=False, jobInd=7, jobs=9)}


@pytest.mark.parametrize("exact", [False, True], ids=["fma", "exact"])
@pytest.mark.parametrize("case", list(EXAMPLE_CASES))
def test_example_segments_equal_binary_file(asmc, tmp_path, case, exact):
    """The bundled FastSMC example (159 states, lane-split kernels) in the reference's regression configuration."""
    kw = dict(EXAMPLE_CASES[case], exactArithmetic=exact)
    dev_dir = tmp_path / "dev"
    dev_dir.mkdir()
    p = _params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(dev_dir / "out"), **kw)
    res = _device(p)
    assert _no_files(dev_dir)
    assert res.d2h_bytes == 0
    lines, count = _file_records(asmc, _params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(tmp_path / "file"), **kw))
    assert res.n_segments == count
    _assert_same_records(lines, res, p)


SYNTH_CASES = {
    # FastSMC_exe's default conditional age estimates: narrow kernel
    "default_flags": dict(hashing=False, noConditionalAgeEstimates=False),
    # all-state ages over whole-chromosome windows: sparse path (finalizeSegmentsKernel)
    "all_state_ages_long_windows": dict(hashing=False, noConditionalAgeEstimates=True),
    # all-state ages on hashing candidates: decodeFastKernel
    "all_state_ages_hashing": dict(hashing=True, noConditionalAgeEstimates=True, min_m=1.0),
}


@pytest.mark.parametrize("case", list(SYNTH_CASES))
def test_synthetic_69_state_segments_equal_binary_file(asmc, tmp_path, case):
    """69 states on synthetic data with 3e-5 Morgans between sites (a gap the bundled table has rows for).  The table's CSFS
    has 300 samples, so the data set needs at least 300 haplotypes."""
    from fastsmc_b200 import synth
    root = str(tmp_path / "syn")
    hashing = SYNTH_CASES[case]["hashing"]
    n_sites = 1920 if hashing else 3000
    synth.dataset(root, 400, n_sites, 3000 * n_sites, 1, 31 + n_sites, founders=6 if hashing else None)
    kw = SYNTH_CASES[case]
    p = _params(asmc, root, DQ_69, str(tmp_path / "dev"), **kw)
    res = _device(p)
    lines, count = _file_records(asmc, _params(asmc, root, DQ_69, str(tmp_path / "file"), **kw))
    assert res.n_segments == count
    _assert_same_records(lines, res, p)


def test_many_chunks_give_the_same_tensors(asmc, tmp_path, monkeypatch):
    """Chunks of two reference batches, one and two decode workers: many collects at growing offsets and several growths
    of the device columns give the tensors of the one-chunk run, and the file's records."""
    for case, kw in EXAMPLE_CASES.items():
        kw = dict(kw, noConditionalAgeEstimates=False)  # narrow kernel: two workers may run
        one = _host(_device(_params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(tmp_path / "one"), **kw)))
        monkeypatch.setenv("FSMC_FLUSH_BATCHES", "2")
        for workers in ("1", "2"):
            monkeypatch.setenv("FSMC_DECODE_WORKERS", workers)
            p = _params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(tmp_path / f"w{workers}"), **kw)
            res = _device(p)
            many = _host(res)
            for name, v in one.items():
                assert (v is None) == (many[name] is None)
                if v is not None:
                    assert np.array_equal(v.view(np.uint32), many[name].view(np.uint32)), (case, workers, name)
            lines, count = _file_records(asmc, _params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ,
                                                       str(tmp_path / f"file{workers}"), **kw))
            assert count > 100
            _assert_same_records(lines, res, p)
        monkeypatch.delenv("FSMC_FLUSH_BATCHES")
        monkeypatch.delenv("FSMC_DECODE_WORKERS")


def test_non_default_stream(asmc, tmp_path):
    import torch
    p = _params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(tmp_path / "a"))
    want = _host(_device(p))
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        res = _device(_params(asmc, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(tmp_path / "b")))
        assert res.score.device == torch.device("cuda", p.device)
    s.synchronize()
    got = _host(res)
    for name, v in want.items():
        assert (v is None) == (got[name] is None)
        if v is not None:
            assert np.array_equal(v.view(np.uint32), got[name].view(np.uint32)), name


# ---- C ABI ---------------------------------------------------------------------------------------------------------------


def test_collect_device_overflow_and_pointer_checks(oracle_mod, tmp_path):
    """fsmc_plan_collect_device: a count-only call, FSMC_E_OVERFLOW that leaves the plan collectable, rejected pointers, and
    columns equal to the host records of fsmc_decode translated like HMM::formatSegments."""
    import torch
    from fastsmc_b200 import _native
    o = oracle_mod.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, str(tmp_path / "o"), hashing=False, **REGRESSION_PARAMS)
    ctx = context_from_oracle(o, oracle_mod)
    gen, bp = o.positions()
    rng = np.random.default_rng(5)
    n = 200
    a = rng.integers(0, o.num_haps, n)
    b = (a + 1 + rng.integers(0, o.num_haps - 1, n)) % o.num_haps
    tiles = ctx.make_tiles(a, b, sites=o.sites)
    flags = _native.CALL_SEGMENTS | _native.SEG_AGE
    want = ctx.decode(tiles, flags).segments
    assert len(want) > 10

    plan = ctx.plan(tiles, flags, segment_capacity=4)  # too small: the library decodes the plan again with room
    plan.launch()
    with pytest.raises(_native.FastSMCError):
        plan.collect_device(None)  # no site positions yet
    ctx.set_site_positions(gen, bp)
    rc, st = plan.collect_device(None)
    assert rc == 0 and st.numSegments == len(want) and st.d2hBytes == 0

    dev = torch.device("cuda", 0)
    cols = {name: torch.full((len(want) + 3,), -7, dtype=getattr(torch, dt), device=dev) for name, dt in _native.SEGMENT_COLUMNS}
    rc, st = plan.collect_device(cols, offset=5)  # 5 + count > capacity
    assert rc == _native.E_OVERFLOW and st.numSegments == len(want)
    assert all(bool((t == -7).all()) for t in cols.values())  # nothing written

    host = np.zeros(len(want) + 3, np.int32)
    with pytest.raises(_native.FastSMCError, match="host memory"):
        plan.collect_device(dict(cols, start_bp=host.ctypes.data), capacity=len(want) + 3)
    if torch.cuda.device_count() > 1:
        other = torch.zeros(len(want) + 3, dtype=torch.int32, device="cuda:1")
        with pytest.raises(_native.FastSMCError, match="on device 1"):
            plan.collect_device(dict(cols, start_bp=other), capacity=len(want) + 3)

    rc, st = plan.collect_device(cols, offset=2)  # the plan is still collectable
    assert rc == 0 and st.numSegments == len(want) and st.d2hBytes == 0
    plan.close()
    torch.cuda.synchronize()
    h = {k: v.cpu().numpy() for k, v in cols.items()}
    pair_a = tiles["hapA"].reshape(-1)[want["pair"]]
    pair_b = tiles["hapB"].reshape(-1)[want["pair"]]
    s, e = want["posStart"], want["posEnd"]
    sl = slice(2, 2 + len(want))
    assert np.array_equal(h["ind1"][sl], pair_a // 2) and np.array_equal(h["hap1"][sl], 1 + pair_a % 2)
    assert np.array_equal(h["ind2"][sl], pair_b // 2) and np.array_equal(h["hap2"][sl], 1 + pair_b % 2)
    assert np.array_equal(h["start_site"][sl], s) and np.array_equal(h["end_site"][sl], e)
    assert np.array_equal(h["start_bp"][sl], bp[s]) and np.array_equal(h["end_bp"][sl], bp[e])
    cm = np.float32(100) * (gen[e] - gen[s])
    score = (want["prob"].astype(np.float64) / (e - s + 1).astype(np.float64)).astype(np.float32)
    for name, v in (("length_cm", cm), ("score", score), ("post_mean", want["postMean"]), ("map_time", want["mapTime"])):
        assert np.array_equal(h[name][sl].view(np.uint32), np.asarray(v, np.float32).view(np.uint32)), name
    assert all(bool((h[k][:2] == -7).all()) and bool((h[k][2 + len(want):] == -7).all()) for k in h)
