"""GPU parity of the decode kernels (through the C ABI) against the CPU oracle on the reference's example data."""
import numpy as np
import pytest

from conftest import FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, REGRESSION_PARAMS, context_from_oracle

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4  # north-star tolerance on per-site posterior mean TMRCA and IBD probability


@pytest.fixture(scope="module")
def example(oracle_mod):
    o = oracle_mod.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, "/tmp/fsmc_test", hashing=True, **REGRESSION_PARAMS)
    ctx = context_from_oracle(o, oracle_mod)
    return o, ctx


def _pairs(rng, n, num_haps):
    a = rng.integers(0, num_haps, n)
    b = rng.integers(0, num_haps, n)
    b = np.where(a == b, (b + 1) % num_haps, b)
    return a.astype(np.uint32), b.astype(np.uint32)


@pytest.mark.parametrize("generic", [False, True])
def test_per_site_outputs_exact_mode_bit_identical(example, generic):
    """FSMC_EXACT reproduces the oracle's per-site posterior mean, MAP and IBD probability bit for bit."""
    from fastsmc_b200 import _native as N
    o, ctx = example
    rng = np.random.default_rng(1)
    a, b = _pairs(rng, 40, o.num_haps)
    frm, to = 1000, 1700
    mean, mp, ibd = o.decode_summary(a, b, frm, to)
    tiles = ctx.make_tiles(a, b, windows=[[frm, to], [frm, to]], sites=o.sites)
    flags = N.SITE_MEAN | N.SITE_MAP | N.SITE_IBD | N.EXACT | (N.GENERIC_KERNEL if generic else 0)
    r = ctx.decode(tiles, flags)
    rows = tiles["rows"]
    assert r.stats.statesKernel == (0 if generic else 159)
    assert np.array_equal(r.site_mean[rows, :to - frm].view(np.uint32), mean.view(np.uint32))
    assert np.array_equal(r.site_ibd[rows, :to - frm].view(np.uint32), ibd.view(np.uint32))
    assert np.array_equal(r.site_map[rows, :to - frm], mp)


@pytest.mark.parametrize("generic", [False, True])
def test_per_site_outputs_fast_mode_within_tolerance(example, generic):
    from fastsmc_b200 import _native as N
    o, ctx = example
    rng = np.random.default_rng(2)
    a, b = _pairs(rng, 64, o.num_haps)
    frm, to = 0, 2500
    mean, mp, ibd = o.decode_summary(a, b, frm, to)
    tiles = ctx.make_tiles(a, b, windows=[[frm, to], [frm, to]], sites=o.sites)
    r = ctx.decode(tiles, N.SITE_MEAN | N.SITE_MAP | N.SITE_IBD | (N.GENERIC_KERNEL if generic else 0))
    rows = tiles["rows"]
    np.testing.assert_allclose(r.site_mean[rows, :to - frm], mean, rtol=REL_TOL)
    np.testing.assert_allclose(r.site_ibd[rows, :to - frm], ibd, rtol=REL_TOL, atol=1e-12)
    # MAP may differ only where the two largest posteriors are within tolerance of each other
    assert (r.site_map[rows, :to - frm] != mp).mean() < 1e-3


@pytest.mark.parametrize("generic", [False, True])
def test_full_posteriors_and_sum_over_pairs(example, generic):
    """FSMC_SITE_POSTERIOR: the whole posterior of every pair (what HMM::decode / decodePairs(per_pair_posteriors)
    return), bit-identical in exact mode.  FSMC_SUM_POSTERIOR: its sum over the real pairs of the call
    (augmentSumOverPairs, ref HMM.cpp:1044-1085), by genotype class with FSMC_SUM_BY_GENOTYPE; float atomics, so
    compared at 1e-5 relative."""
    from fastsmc_b200 import _native as N
    o, ctx = example
    rng = np.random.default_rng(5)
    a, b = _pairs(rng, 40, o.num_haps)  # 40 pairs: a full tile and a ragged one (padding lanes must not be summed)
    frm, to = 2000, 2300
    want = o.decode_posterior(a, b, frm, to)  # [pair][site][state]
    tiles = ctx.make_tiles(a, b, windows=[[frm, to], [frm, to]], sites=o.sites)
    kernel = N.GENERIC_KERNEL if generic else 0
    r = ctx.decode(tiles, N.SITE_POSTERIOR | N.SUM_POSTERIOR | N.EXACT | kernel)
    got = r.site_posterior[tiles["rows"], :, :to - frm].transpose(0, 2, 1)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    total = want.astype(np.float64).sum(axis=0).T  # [state][site]
    assert r.sum_posterior.shape == (1, o.states, o.sites)
    np.testing.assert_allclose(r.sum_posterior[0][:, frm:to], total, rtol=1e-5)
    assert not r.sum_posterior[0][:, :frm].any() and not r.sum_posterior[0][:, to:].any()
    np.testing.assert_allclose(r.sum_posterior[0][:, frm:to].sum(axis=0), len(a), rtol=1e-5)  # posteriors sum to 1

    # by genotype class of the pair at the site: 0 both major, 1 heterozygous, 2 both minor (folded alleles)
    haps = np.asarray(o.haplotypes())[:, frm:to].astype(bool)
    ha, hb = haps[a], haps[b]
    cls = np.where(ha ^ hb, 1, np.where(ha & hb, 2, 0))  # [pair][site]
    r3 = ctx.decode(tiles, N.SUM_POSTERIOR | N.SUM_BY_GENOTYPE | kernel)  # FMA arithmetic: 1e-4
    assert r3.sum_posterior.shape == (3, o.states, o.sites)
    for c in range(3):
        part = (want.astype(np.float64) * (cls == c)[:, :, None]).sum(axis=0).T
        np.testing.assert_allclose(r3.sum_posterior[c][:, frm:to], part, rtol=REL_TOL, atol=1e-7)


def _oracle_segments(o):
    ints, floats = o.segments()
    return ints, floats


@pytest.mark.parametrize("hashing", [True, False])
def test_segments_exact_mode_identical_to_oracle(oracle_mod, tmp_path, hashing):
    """Whole-job segment lists (golden G1 / G2 configurations): identical records in identical order."""
    from fastsmc_b200 import _native as N
    extra = dict(hashing=True) if hashing else dict(hashing=False, jobInd=7, jobs=9)
    o = oracle_mod.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, "/tmp/fsmc_test", **extra, **REGRESSION_PARAMS)
    n = o.run(str(tmp_path / "oracle.ibd.gz"))
    ints, floats = o.segments()
    batches = o.batches()
    ctx = context_from_oracle(o, oracle_mod)
    # rebuild the pair stream from the oracle's segment-independent batch list
    if hashing:
        cands = o.candidates()
        a, b = cands[:, 0], cands[:, 1]
    else:
        pytest.skip("covered by test_no_hashing_job_exact")
    tiles = ctx.make_tiles(a, b, windows=batches[:, 3:5], scan=batches[:, 1:3], sites=o.sites)
    r = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | N.EXACT)
    seg = r.segments
    assert len(seg) == n
    assert np.array_equal(seg["pair"], ints[:, 0] * 32 + ints[:, 1])
    assert np.array_equal(seg["posStart"], ints[:, 4])
    assert np.array_equal(seg["posEnd"], ints[:, 5])
    assert np.array_equal(seg["mapState"], ints[:, 6])
    assert np.array_equal(seg["prob"].view(np.uint32), floats[:, 0].copy().view(np.uint32))
    assert np.array_equal(seg["postMean"].view(np.uint32), floats[:, 1].copy().view(np.uint32))
    assert np.array_equal(seg["mapTime"].view(np.uint32), floats[:, 2].copy().view(np.uint32))


def test_segments_fast_mode_matches_oracle_within_tolerance(oracle_mod, tmp_path):
    from fastsmc_b200 import _native as N
    o = oracle_mod.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, "/tmp/fsmc_test", hashing=True, **REGRESSION_PARAMS)
    n = o.run(str(tmp_path / "oracle.ibd.gz"))
    ints, floats = o.segments()
    batches = o.batches()
    cands = o.candidates()
    ctx = context_from_oracle(o, oracle_mod)
    tiles = ctx.make_tiles(cands[:, 0], cands[:, 1], windows=batches[:, 3:5], scan=batches[:, 1:3], sites=o.sites)
    r = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE)
    seg = r.segments
    # boundaries may move only at sites whose IBD probability is within tolerance of a threshold;
    # on this data set none is, so the lists must coincide
    assert len(seg) == n
    assert np.array_equal(seg["pair"], ints[:, 0] * 32 + ints[:, 1])
    assert np.array_equal(seg["posStart"], ints[:, 4])
    assert np.array_equal(seg["posEnd"], ints[:, 5])
    np.testing.assert_allclose(seg["prob"], floats[:, 0], rtol=REL_TOL)
    np.testing.assert_allclose(seg["postMean"], floats[:, 1], rtol=REL_TOL)
    assert (seg["mapState"] != ints[:, 6]).mean() < 5e-3


def test_no_hashing_job_exact(oracle_mod, tmp_path):
    """Golden G2 configuration (hashing off, job 7 of 9): all-pairs tiles over the whole sequence."""
    from fastsmc_b200 import _native as N
    o = oracle_mod.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, "/tmp/fsmc_test", hashing=False, jobInd=7, jobs=9,
                          **REGRESSION_PARAMS)
    n = o.run(str(tmp_path / "oracle.ibd.gz"))
    ints, floats = o.segments()
    # pair stream: first record of each (batch, lane) is enough to recover hapA/hapB only for pairs with
    # segments, so re-enumerate the job's pairs exactly as HMM::decodeAll does (HMM.cpp:311-357)
    N_ind = o.num_haps // 2
    tot = 2 * N_ind * N_ind - N_ind
    lo, hi = tot * 6 // 9, tot * 7 // 9
    a, b = [], []
    idx = 0
    for i in range(N_ind):
        for j in range(i):
            for ih in (0, 1):
                for jh in (0, 1):
                    if lo <= idx < hi:
                        a.append(2 * j + jh)
                        b.append(2 * i + ih)
                    idx += 1
        if lo <= idx < hi:
            a.append(2 * i)
            b.append(2 * i + 1)
        idx += 1
    ctx = context_from_oracle(o, oracle_mod)
    tiles = ctx.make_tiles(np.array(a), np.array(b), sites=o.sites)
    r = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | N.EXACT)
    seg = r.segments
    assert len(seg) == n
    assert np.array_equal(seg["pair"], ints[:, 0] * 32 + ints[:, 1])
    assert np.array_equal(seg["posStart"], ints[:, 4])
    assert np.array_equal(seg["posEnd"], ints[:, 5])
    assert np.array_equal(seg["prob"].view(np.uint32), floats[:, 0].copy().view(np.uint32))
    assert np.array_equal(seg["postMean"].view(np.uint32), floats[:, 1].copy().view(np.uint32))
    assert np.array_equal(seg["mapState"], ints[:, 6])


# ---- 69-state decoding quantities (30-100-2000, the UKBB-style table of the synthetic benchmarks): this is the state
# count the production kernel (decode_fast.cuh) is specialised for --------------------------------------------------


@pytest.fixture(scope="module")
def synthetic69(oracle_mod, tmp_path_factory):
    from conftest import DQ_69
    from fastsmc_b200 import synth
    root = str(tmp_path_factory.mktemp("syn69") / "syn")
    synth.dataset(root, 400, 3000, 9_000_000, 1, 777)
    o = oracle_mod.Oracle(root, DQ_69, "/tmp/fsmc_test69", hashing=False, time=50, noConditionalAgeEstimates=True,
                          doPerPairMAP=True, doPerPairPosteriorMean=True, batchSize=32)
    ctx = context_from_oracle(o, oracle_mod)
    o.dataset_root = root  # for tests that open a second oracle on the same files
    return o, ctx


@pytest.fixture(params=[False, True], ids=["default", "one-warp"])
def one_warp(request):
    """Extra decode flags: none, or FSMC_ONE_WARP_KERNEL.  At 69 states both run one warp per tile (decode_fast.cuh)."""
    from fastsmc_b200 import _native as N
    return N.ONE_WARP_KERNEL if request.param else 0


def test_fast_kernel_per_site_outputs_69_states(synthetic69, one_warp):
    """Production kernel (FMA, rescaling every 4th site, bulk-copy ring): per-site posterior mean, IBD probability and MAP
    within the north-star tolerance of the oracle; ragged windows and a partially filled tile included."""
    from fastsmc_b200 import _native as N
    o, ctx = synthetic69
    rng = np.random.default_rng(5)
    a, b = _pairs(rng, 70, o.num_haps)  # 3 tiles, the last one with 6 pairs
    for frm, to in ((0, o.sites), (517, 1203), (2999, 3000), (0, 2)):
        mean, mp, ibd = o.decode_summary(a, b, frm, to)
        nb = (len(a) + 31) // 32
        tiles = ctx.make_tiles(a, b, windows=[[frm, to]] * nb, sites=o.sites)
        r = ctx.decode(tiles, N.SITE_MEAN | N.SITE_MAP | N.SITE_IBD | one_warp)
        assert r.stats.statesKernel == 69 and r.stats.tileWarps == 1
        rows = tiles["rows"]
        np.testing.assert_allclose(r.site_mean[rows, :to - frm], mean, rtol=REL_TOL)
        np.testing.assert_allclose(r.site_ibd[rows, :to - frm], ibd, rtol=REL_TOL, atol=1e-12)
        assert (r.site_map[rows, :to - frm] != mp).mean() < 2e-3


def test_fast_kernel_segments_69_states(synthetic69, tmp_path, one_warp):
    """Whole all-pairs job slice through the production kernel vs the oracle: same segments (a boundary may move only
    where the IBD probability is within tolerance of a threshold), sums and age estimates within 1e-4."""
    from fastsmc_b200 import _native as N
    o, ctx = synthetic69
    n = o.run(str(tmp_path / "oracle.ibd.gz"))
    ints, floats = o.segments()
    H = o.num_haps
    a, b = [], []
    for i in range(H // 2):
        for j in range(i):
            for ih in (0, 1):
                for jh in (0, 1):
                    a.append(2 * j + jh)
                    b.append(2 * i + ih)
        a.append(2 * i)
        b.append(2 * i + 1)
    tiles = ctx.make_tiles(np.array(a), np.array(b), sites=o.sites)
    r = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | one_warp, segment_capacity=1 << 20)
    seg = r.segments
    assert r.stats.statesKernel == 69 and r.stats.tileWarps == 1
    want = {(int(i[0]) * 32 + int(i[1]), int(i[4]), int(i[5])): f for i, f in zip(ints, floats)}
    got = {(int(s["pair"]), int(s["posStart"]), int(s["posEnd"])): s for s in seg}
    common = set(want) & set(got)
    # identical segment lists, except where the posterior is within tolerance of a threshold (checked site by site
    # against the oracle's per-site IBD probability for every pair whose lists differ)
    assert len(common) >= 0.995 * max(len(want), len(got)) and abs(len(seg) - n) <= 0.005 * n + 2
    from conftest import check_segments_up_to_threshold_ties
    check_segments_up_to_threshold_ties(o, seg, want.keys(), lambda p: (a[p], b[p]), REL_TOL)
    w = np.array([want[k] for k in sorted(common)])
    g = np.array([[got[k]["prob"], got[k]["postMean"], got[k]["mapTime"]] for k in sorted(common)])
    np.testing.assert_allclose(g[:, 0], w[:, 0], rtol=REL_TOL)
    np.testing.assert_allclose(g[:, 1], w[:, 1], rtol=REL_TOL)
    assert (g[:, 2] != w[:, 2]).mean() < 5e-3


def test_segment_records_do_not_depend_on_previous_buffer_contents(synthetic69):
    """fsmc_decode sorts the records into the caller's buffer; what the buffer held before the call must not matter.
    (A reused heap block holds the records of an earlier call: same pair numbering, other positions.)"""
    from fastsmc_b200 import _native as N
    o, ctx = synthetic69
    ia, ib = np.triu_indices(64, 1)
    tiles = ctx.make_tiles(ia.astype(np.uint32), ib.astype(np.uint32), sites=o.sites)
    flags = N.CALL_SEGMENTS | N.SEG_AGE
    clean = ctx.decode(tiles, flags, segment_capacity=1 << 16).segments.copy()
    assert len(clean) > 100
    # adversarial previous contents: every slot holds the record that belongs one slot further, moved to a later site
    stale = np.zeros(1 << 16, N.SEGMENT_DTYPE)
    stale[:len(clean) - 1] = clean[1:]
    stale["posStart"] += 1 << 20
    again = ctx.decode(tiles, flags, segment_capacity=1 << 16, segment_prefill=stale).segments
    assert again.tobytes() == clean.tobytes()
    key = clean["pair"].astype(np.int64) * (1 << 32) + clean["posStart"]
    assert (np.diff(key) > 0).all()  # sorted by (pair, start), every record once


def test_narrow_kernel_matches_oracle_and_wide_kernel(oracle_mod, synthetic69, one_warp):
    """FastSMC's default flags (age estimates conditional on TMRCA < time): the kernel that keeps only the states below
    the threshold and carries the normaliser by the scale-factor recurrence (decodeNarrowKernel) gives the oracle's
    segments and per-site IBD probabilities within 1e-4, over a 3 000-site window (750 rescalings)."""
    from conftest import DQ_69
    from fastsmc_b200 import _native as N
    o_wide, ctx_wide = synthetic69
    # a second oracle instance with conditional age estimates (ageThreshold == stateThreshold)
    root = o_wide.dataset_root
    o = oracle_mod.Oracle(root, DQ_69, "/tmp/fsmc_test69n", hashing=False, time=50, noConditionalAgeEstimates=False,
                          doPerPairMAP=True, doPerPairPosteriorMean=True, batchSize=32)
    ctx = context_from_oracle(o, oracle_mod)
    assert o.age_threshold == o.state_threshold
    rng = np.random.default_rng(11)
    a, b = _pairs(rng, 96, o.num_haps)
    # per-site IBD probability
    mean, mp, ibd = o.decode_summary(a, b, 0, o.sites, mean=False, map_=False)
    tiles = ctx.make_tiles(a, b, windows=[[0, o.sites]] * 3, sites=o.sites)
    r = ctx.decode(tiles, N.SITE_IBD | one_warp)
    assert r.stats.narrowKernel == 1 and r.stats.tileWarps == 1
    np.testing.assert_allclose(r.site_ibd[tiles["rows"]], ibd, rtol=REL_TOL, atol=1e-12)
    # segments with conditional age estimates: narrow vs the full-beta kernel (same arithmetic otherwise)
    rn = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | one_warp)
    rw = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | N.WIDE_KERNEL | one_warp)
    assert rn.stats.narrowKernel == 1 and rw.stats.narrowKernel == 0
    key = lambda s: (int(s["pair"]), int(s["posStart"]), int(s["posEnd"]))
    gn, gw = {key(s): s for s in rn.segments}, {key(s): s for s in rw.segments}
    common = sorted(set(gn) & set(gw))
    assert len(common) >= 0.95 * max(len(gn), len(gw)) > 10
    for f in ("prob", "postMean"):
        np.testing.assert_allclose([gn[k][f] for k in common], [gw[k][f] for k in common], rtol=REL_TOL)
    assert np.mean([gn[k]["mapState"] != gw[k]["mapState"] for k in common]) < 5e-3


# ---- 159 states (FASTSMC_EXAMPLE table): the lane-split kernels are the production path (4 warps per tile) ----------


@pytest.mark.parametrize("time", [50, 100, 140], ids=["time50-2quads", "time100-3quads", "time140-4quads"])
def test_lane_split_kernels_159_states(oracle_mod, tmp_path, time):
    """FastSMC's default flags on the example data (age estimates conditional on TMRCA < time) at 159 states: the lane-split
    kernels (decode_lane.cuh; records, and full beta rows with FSMC_WIDE_KERNEL) vs the oracle: same segments, per-segment
    values and per-site IBD probability within 1e-4, over ragged windows, a partially filled tile and a one-site window."""
    from fastsmc_b200 import _native as N
    params = dict(REGRESSION_PARAMS, noConditionalAgeEstimates=False, time=time)  # records of 2, 3 and 4 quads
    o = oracle_mod.Oracle(FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, "/tmp/fsmc_test159n", hashing=True, **params)
    assert o.age_threshold == o.state_threshold == time // 10
    n = o.run(str(tmp_path / "oracle.ibd.gz"))
    ints, floats = o.segments()
    batches = o.batches()
    cands = o.candidates()
    ctx = context_from_oracle(o, oracle_mod)
    tiles = ctx.make_tiles(cands[:, 0], cands[:, 1], windows=batches[:, 3:5], scan=batches[:, 1:3], sites=o.sites)
    for extra, narrow in ((0, 1), (N.WIDE_KERNEL, 0)):
        r = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | extra)
        assert r.stats.narrowKernel == narrow and r.stats.tileWarps == 4 and r.stats.statesKernel == 159
        seg = r.segments
        assert len(seg) == n
        assert np.array_equal(seg["pair"], ints[:, 0] * 32 + ints[:, 1])
        assert np.array_equal(seg["posStart"], ints[:, 4])
        assert np.array_equal(seg["posEnd"], ints[:, 5])
        np.testing.assert_allclose(seg["prob"], floats[:, 0], rtol=REL_TOL)
        np.testing.assert_allclose(seg["postMean"], floats[:, 1], rtol=REL_TOL)
        assert (seg["mapState"] != ints[:, 6]).mean() < 5e-3
    # per-site IBD probability over ragged windows, a partially filled tile and a single-site window
    rng = np.random.default_rng(3)
    a, b = _pairs(rng, 45, o.num_haps)
    for frm, to in ((0, o.sites), (311, 1999), (6759, 6760), (5, 7)):
        _, _, ibd = o.decode_summary(a, b, frm, to, mean=False, map_=False)
        t2 = ctx.make_tiles(a, b, windows=[[frm, to]] * 2, sites=o.sites)
        r = ctx.decode(t2, N.SITE_IBD)
        assert r.stats.narrowKernel == 1 and r.stats.tileWarps == 4
        np.testing.assert_allclose(r.site_ibd[t2["rows"], :to - frm], ibd, rtol=REL_TOL, atol=1e-12)


def test_one_warp_kernels_still_selectable_159(example):
    """FSMC_ONE_WARP_KERNEL keeps the register/shared-memory kernel of decode_kernels.cuh reachable (A/B checks)."""
    from fastsmc_b200 import _native as N
    o, ctx = example
    rng = np.random.default_rng(4)
    a, b = _pairs(rng, 32, o.num_haps)
    mean, mp, ibd = o.decode_summary(a, b, 100, 600)
    tiles = ctx.make_tiles(a, b, windows=[[100, 600]], sites=o.sites)
    r1 = ctx.decode(tiles, N.SITE_MEAN | N.SITE_IBD | N.ONE_WARP_KERNEL)
    r4 = ctx.decode(tiles, N.SITE_MEAN | N.SITE_IBD)
    assert r1.stats.tileWarps == 1 and r4.stats.tileWarps == 4
    for r in (r1, r4):
        np.testing.assert_allclose(r.site_mean[tiles["rows"], :500], mean, rtol=REL_TOL)
        np.testing.assert_allclose(r.site_ibd[tiles["rows"], :500], ibd, rtol=REL_TOL, atol=1e-12)


# ---- all-state age estimates without the beta round trip (decode_sparse.cuh) -------------------------------------------


def _all_pairs(H):
    a, b = [], []
    for i in range(H // 2):
        for j in range(i):
            for ih in (0, 1):
                for jh in (0, 1):
                    a.append(2 * j + jh)
                    b.append(2 * i + ih)
        a.append(2 * i)
        b.append(2 * i + 1)
    return np.array(a), np.array(b)


def _seg_key(s):
    return (int(s["pair"]), int(s["posStart"]), int(s["posEnd"]))


def test_sparse_age_estimates_match_oracle_and_dense_kernel(synthetic69, tmp_path, monkeypatch):
    """noConditionalAgeEstimates on whole-chromosome windows: narrow sweeps + checkpoints + refinement inside the IBD runs
    (sparseKernel) vs the oracle (1e-4) and vs the kernel that streams every beta row through HBM (same segments)."""
    from conftest import check_segments_up_to_threshold_ties
    from fastsmc_b200 import _native as N
    o, ctx = synthetic69
    n = o.run(str(tmp_path / "oracle.ibd.gz"))
    ints, floats = o.segments()
    a, b = _all_pairs(o.num_haps)
    tiles = ctx.make_tiles(a, b, sites=o.sites)
    flags = N.CALL_SEGMENTS | N.SEG_AGE
    want = {(int(i[0]) * 32 + int(i[1]), int(i[4]), int(i[5])): (f, int(i[6])) for i, f in zip(ints, floats)}
    dense = ctx.decode(tiles, flags | N.WIDE_KERNEL, segment_capacity=1 << 20)
    assert dense.stats.sparseKernel == 0 and dense.stats.narrowKernel == 0
    gd = {_seg_key(s): s for s in dense.segments}
    results = {}
    for label, env in (("default", {}), ("blocks of 8", {"FSMC_CKPT_SHIFT": "3"}), ("blocks of 32", {"FSMC_CKPT_SHIFT": "5"}),
                       ("item overflow", {"FSMC_ITEM_CAPACITY": "1000"})):
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        r = ctx.decode(tiles, flags, segment_capacity=1 << 20)
        for k in env:
            monkeypatch.delenv(k)
        st = r.stats
        assert st.sparseKernel == 1 and st.narrowKernel == 1 and st.sparseItems > len(r.segments) > 1000, label
        assert st.checkpointSites == {"blocks of 8": 8, "blocks of 32": 32}.get(label, 128)
        got = {_seg_key(s): s for s in r.segments}
        results[label] = got
        common = sorted(set(want) & set(got))
        assert len(common) >= 0.995 * max(len(want), len(got)) and abs(len(got) - n) <= 0.005 * n + 2, label
        if label == "default":
            check_segments_up_to_threshold_ties(o, r.segments, want.keys(), lambda p: (a[p], b[p]), REL_TOL)
        g = np.array([[got[k]["prob"], got[k]["postMean"], got[k]["mapTime"]] for k in common])
        w = np.array([want[k][0] for k in common])
        np.testing.assert_allclose(g[:, 0], w[:, 0], rtol=REL_TOL, err_msg=label)
        np.testing.assert_allclose(g[:, 1], w[:, 1], rtol=REL_TOL, err_msg=label)
        assert (g[:, 2] != w[:, 2]).mean() < 5e-3, label
        # and against the dense kernel
        both = sorted(set(gd) & set(got))
        assert len(both) >= 0.995 * max(len(gd), len(got))
        np.testing.assert_allclose([got[k]["postMean"] for k in both], [gd[k]["postMean"] for k in both], rtol=REL_TOL)
        assert np.mean([got[k]["mapState"] != gd[k]["mapState"] for k in both]) < 5e-3
    # the segment list itself does not depend on the block size or on the re-run
    assert set(results["default"]) == set(results["blocks of 8"]) == set(results["blocks of 32"]) == set(results["item overflow"])


def test_sparse_age_estimates_ragged_windows(synthetic69, monkeypatch):
    """Windows that start and end inside checkpoint blocks, scan windows narrower than the decode windows, a partially
    filled tile and windows shorter than a block: sparse path (forced) vs the dense kernel."""
    from fastsmc_b200 import _native as N
    o, ctx = synthetic69
    rng = np.random.default_rng(21)
    a, b = _pairs(rng, 32 * 39 + 5, o.num_haps)
    nb = (len(a) + 31) // 32
    win = np.array([[0, o.sites], [5, 37], [31, 33], [100, 2999], [1000, 1001], [777, 2222], [64, 96], [1, 3000]] * 5, np.int32)[:nb]
    scan = np.array([[0, o.sites], [6, 30], [31, 33], [500, 2500], [1000, 1001], [800, 2200], [64, 96], [33, 2990]] * 5, np.int32)[:nb]
    tiles = ctx.make_tiles(a, b, windows=win, scan=scan, sites=o.sites)
    flags = N.CALL_SEGMENTS | N.SEG_AGE
    dense = ctx.decode(tiles, flags | N.WIDE_KERNEL, segment_capacity=1 << 18)
    monkeypatch.setenv("FSMC_SPARSE", "1")
    sparse = ctx.decode(tiles, flags, segment_capacity=1 << 18)
    assert sparse.stats.sparseKernel == 1 and dense.stats.sparseKernel == 0
    gd, gs = {_seg_key(s): s for s in dense.segments}, {_seg_key(s): s for s in sparse.segments}
    both = sorted(set(gd) & set(gs))
    assert len(both) >= 0.99 * max(len(gd), len(gs)) and len(both) > 20
    for f in ("prob", "postMean"):
        np.testing.assert_allclose([gs[k][f] for k in both], [gd[k][f] for k in both], rtol=REL_TOL)
    assert np.mean([gs[k]["mapState"] != gd[k]["mapState"] for k in both]) < 1e-2


# ---- BASELINE.json configs[1] at its own shape: 1 000 haplotypes x 10 000 SNPs, S = 69 -----------------------------------


def test_cfg2_shape_batches_against_oracle(oracle_mod, tmp_path):
    """64 reference batches spread over cfg2's 15 610 (the last, partially filled one included), all 10 000 sites: the
    oracle's per-site posteriors vs (a) the per-site IBD probability of decodeNarrowKernel, (b) the segments of the sparse
    all-state path (the bench's headline) and of the narrow kernel (FastSMC_exe default flags): per-site levels equal
    except within 1e-4 of a threshold, segment scores within 1e-4, (c) posterior mean / MAP of the segments from the
    oracle's full posterior matrices for a sample of pairs."""
    import sys
    from concurrent.futures import ThreadPoolExecutor
    from conftest import DQ_69, ROOT
    from fastsmc_b200 import _native as N, synth
    sys.path.insert(0, ROOT)
    import bench
    root = str(tmp_path / "cfg2")
    synth.dataset(root, bench.N_HAPS, bench.N_SITES, bench.SPAN_BP, bench.CHROM, bench.SEED)
    kw = dict(hashing=False, time=50, doPerPairMAP=True, doPerPairPosteriorMean=True, batchSize=32)
    o = oracle_mod.Oracle(root, DQ_69, str(tmp_path / "o"), noConditionalAgeEstimates=True, **kw)
    o_cond = oracle_mod.Oracle(root, DQ_69, str(tmp_path / "oc"), noConditionalAgeEstimates=False, **kw)
    L = o.sites
    a_all, b_all = bench.all_pairs_in_reference_order(o.num_haps // 2)
    n_batches = (len(a_all) + 31) // 32
    assert n_batches == 15610 and len(a_all) % 32 == 12
    picked = np.unique(np.r_[np.linspace(0, n_batches - 1, 63).astype(int), n_batches - 1])
    idx = np.concatenate([np.arange(32 * t, min(32 * (t + 1), len(a_all))) for t in picked])
    a, b = a_all[idx], b_all[idx]
    # the oracle's per-site IBD probability of every picked pair (host threads; the oracle call releases the GIL)
    chunks = [np.arange(i, min(i + 32, len(a))) for i in range(0, len(a), 32)]
    with ThreadPoolExecutor(8) as pool:
        parts = list(pool.map(lambda c: o.decode_summary(a[c], b[c], 0, L, mean=False, map_=False)[2], chunks))
    ibd = np.concatenate(parts)
    thr = np.float32(o.probability_threshold) * np.array([1000, 100, 10, 1], np.float32)
    level = np.full(ibd.shape, -1, np.int8)
    for i in (3, 2, 1, 0):
        level[ibd >= thr[i]] = i
    ambiguous = np.zeros(ibd.shape, bool)
    for t in thr:
        ambiguous |= np.abs(ibd - t) <= REL_TOL * t

    def check_segments(ctx, label):
        tiles = ctx.make_tiles(a, b, sites=L)
        rows = tiles["rows"]
        row_of_pair = {int(r): i for i, r in enumerate(rows)}
        r = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE, segment_capacity=1 << 18)
        mine = np.full(ibd.shape, -1, np.int8)
        score_err = 0.0
        for s in r.segments:
            i = row_of_pair[int(s["pair"])]
            lo, hi = int(s["posStart"]), int(s["posEnd"]) + 1
            mine[i, lo:hi] = int(s["level"])
            if not ambiguous[i, max(lo - 1, 0):hi + 1].any():  # same segment in the oracle: compare the score
                want = float(ibd[i, lo:hi].astype(np.float64).sum())
                score_err = max(score_err, abs(float(s["prob"]) - want) / want)
        bad = (mine != level) & ~ambiguous
        assert not bad.any(), f"{label}: {int(bad.sum())} sites with a different level away from the thresholds"
        assert score_err < REL_TOL, label
        assert len(r.segments) > 1500
        return r, row_of_pair

    ctx = context_from_oracle(o, oracle_mod)
    r_sparse, row_of_pair = check_segments(ctx, "sparse")
    assert r_sparse.stats.sparseKernel == 1
    ctx_cond = context_from_oracle(o_cond, oracle_mod)
    r_narrow, _ = check_segments(ctx_cond, "narrow")
    assert r_narrow.stats.narrowKernel == 1 and r_narrow.stats.sparseKernel == 0
    tiles = ctx_cond.make_tiles(a, b, sites=L)
    site = ctx_cond.decode(tiles, N.SITE_IBD)
    assert site.stats.narrowKernel == 1
    np.testing.assert_allclose(site.site_ibd[tiles["rows"]], ibd, rtol=REL_TOL, atol=1e-12)

    # (c) age estimates: full posterior of the pairs that hold the 40 longest segments
    seg = r_sparse.segments
    longest = seg[np.argsort(seg["posEnd"] - seg["posStart"])[-40:]]
    exp_t, prior = o.vector("expectedTimes"), o.vector("initialStateProb")
    for s in longest:
        i = row_of_pair[int(s["pair"])]
        lo, hi = int(s["posStart"]), int(s["posEnd"]) + 1
        if ambiguous[i, max(lo - 1, 0):hi + 1].any():
            continue
        post = o.decode_posterior(a[i:i + 1], b[i:i + 1], 0, L)[0]  # [site][state]
        sums = post[lo:hi].astype(np.float64).sum(axis=0)
        want_mean = float((sums / sums.sum() * exp_t).sum())
        assert abs(float(s["postMean"]) - want_mean) <= REL_TOL * want_mean
        ratio = sums / prior
        best = int(np.argmax(ratio))
        assert int(s["mapState"]) == best or ratio[int(s["mapState"])] >= ratio[best] * (1 - 1e-3)


# ---- state counts other than 69 / 159: padded onto the specialised kernels -----------------------------------------------


@pytest.mark.parametrize("source,states,kernel_states", [("synthetic69", 40, 69), ("example", 100, 159), ("synthetic69", 68, 69)])
def test_other_state_counts_run_on_the_specialised_kernels(request, oracle_mod, source, states, kernel_states):
    """A decoding-quantities table with any number of states must not fall to the scalar-load kernel: the model is padded
    with probability-free states to 69 or 159.  Truncating a real table to its first `states` states gives a model with
    another state count (the recurrences do not care that it is no longer a proper transition matrix); the padded
    production kernels must agree with the any-S kernel (FSMC_GENERIC_KERNEL, itself checked against the oracle at 69 and
    159 states) within 1e-4: per-site outputs, segments with all-state and with conditional age estimates."""
    from conftest import model_from_oracle
    from fastsmc_b200 import _native as N
    o, _ = request.getfixturevalue(source)
    full = model_from_oracle(o, oracle_mod)
    cut = {k: (v[..., :states].copy() if isinstance(v, np.ndarray) and v.ndim >= 1 and v.shape[-1] == o.states else v)
           for k, v in full.items()}
    rng = np.random.default_rng(9)
    a, b = _pairs(rng, 75, o.num_haps)
    for age_threshold in (states, full["state_threshold"]):
        ctx = N.Context(0)
        ctx.set_model(**dict(cut, age_threshold=age_threshold))
        ctx.set_haplotypes(N.pack_haplotypes(o.haplotypes()), o.sites)
        nb = (len(a) + 31) // 32
        tiles = ctx.make_tiles(a, b, windows=[[3, min(o.sites, 2500)]] * nb, sites=o.sites)
        if age_threshold == states:
            fast = ctx.decode(tiles, N.SITE_MEAN | N.SITE_MAP | N.SITE_IBD)
            slow = ctx.decode(tiles, N.SITE_MEAN | N.SITE_MAP | N.SITE_IBD | N.GENERIC_KERNEL)
            assert fast.stats.statesKernel == kernel_states and slow.stats.statesKernel == 0
            rows, n = tiles["rows"], min(o.sites, 2500) - 3
            np.testing.assert_allclose(fast.site_mean[rows, :n], slow.site_mean[rows, :n], rtol=REL_TOL)
            np.testing.assert_allclose(fast.site_ibd[rows, :n], slow.site_ibd[rows, :n], rtol=REL_TOL, atol=1e-12)
            assert (fast.site_map[rows, :n] != slow.site_map[rows, :n]).mean() < 2e-3
        fast = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE, segment_capacity=1 << 16)
        slow = ctx.decode(tiles, N.CALL_SEGMENTS | N.SEG_AGE | N.GENERIC_KERNEL, segment_capacity=1 << 16)
        assert fast.stats.statesKernel == kernel_states and slow.stats.statesKernel == 0
        gf, gs = {_seg_key(s): s for s in fast.segments}, {_seg_key(s): s for s in slow.segments}
        both = sorted(set(gf) & set(gs))
        assert len(both) >= 0.98 * max(len(gf), len(gs)) and len(both) > 5
        for f in ("prob", "postMean"):
            np.testing.assert_allclose([gf[k][f] for k in both], [gs[k][f] for k in both], rtol=REL_TOL)
        assert np.mean([gf[k]["mapState"] != gs[k]["mapState"] for k in both]) < 2e-2
        ctx.close()


def test_posterior_sums_on_the_production_kernel(synthetic69):
    """FSMC_SUM_POSTERIOR[_BY_GENOTYPE] (ref: HMM.cpp:1044-1085): decodeFastKernel<69, SUM> (per-warp accumulators, static
    tile deal, ordered reduction) vs the any-S kernel's float atomics: same sums to rounding, and bit-identical from run
    to run."""
    from fastsmc_b200 import _native as N
    o, ctx = synthetic69
    rng = np.random.default_rng(17)
    a, b = _pairs(rng, 32 * 50 + 9, o.num_haps)
    tiles = ctx.make_tiles(a, b, sites=o.sites)
    for extra in (0, N.SUM_BY_GENOTYPE):
        fast = ctx.decode(tiles, N.SUM_POSTERIOR | extra)
        again = ctx.decode(tiles, N.SUM_POSTERIOR | extra)
        slow = ctx.decode(tiles, N.SUM_POSTERIOR | extra | N.GENERIC_KERNEL)
        assert fast.stats.statesKernel == 69 and slow.stats.statesKernel == 0
        assert fast.sum_posterior.shape == ((3 if extra else 1), o.states, o.sites)
        assert fast.sum_posterior.tobytes() == again.sum_posterior.tobytes()
        np.testing.assert_allclose(fast.sum_posterior, slow.sum_posterior, rtol=2e-4, atol=1e-6)
        # every pair contributes a distribution over the states at every site
        np.testing.assert_allclose(fast.sum_posterior.sum(axis=(0, 1)), len(a), rtol=1e-4)
