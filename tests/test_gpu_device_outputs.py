"""decode_pairs_cuda / fsmc_decode_device: ASMC.decodePairs outputs written by the decode kernels into CUDA tensors.

Every field must equal what ASMC.decodePairs returns for the same inputs, bit for bit (the sums of posteriors to 1e-5 where
the device adds them with float atomics); the host path's results must be left alone; nothing but O(1) statistics may cross
to the host.  The 69-state model runs through ASMC.decodePairs on the bundled ASMC example.  The bundled 159-state table only
holds the rows FastSMC mode needs (tests/golden/make_fixtures.py), so an ASMC-mode object cannot be built on it: the
159-state kernels (decodeLaneWideKernel, decodeTilesKernel<159>) are held to fsmc_decode, the call behind ASMC.decodePairs,
through the C ABI."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ASMC_EXAMPLE, DQ_69, FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, REGRESSION_PARAMS, context_from_oracle

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

HERE = os.path.dirname(os.path.abspath(__file__))
ALL = dict(per_pair_posteriors=True, sum_of_posteriors=True, per_pair_posterior_means=True, per_pair_MAPs=True)
SITE = dict(per_pair_posterior_means=True, per_pair_MAPs=True)
# name -> (data, decoding quantities, exactArithmetic, outputs, sums bit-identical)
CASES = {
    "fast69": (ASMC_EXAMPLE, DQ_69, False, dict(SITE, sum_of_posteriors=True), True),  # decodeFastKernel<SUM>
    "exact69": (ASMC_EXAMPLE, DQ_69, True, ALL, False),                                # decodeTilesKernel
    "posteriors69": (ASMC_EXAMPLE, DQ_69, False, dict(per_pair_posteriors=True), False),
}


def _asmc(root, dq, exact):
    from fastsmc_b200 import asmc
    p = asmc.DecodingParams(root, dq, "/tmp/fsmc_device_outputs", 1, 1, "array", False, True, False, False, 0.0, False,
                            False, False, "", False, False)
    p.useKnownSeed = True
    p.exactArithmetic = exact
    p.verbose = False
    return asmc.ASMC(p)


def _pairs(n, seed=0):
    """n pairs of the 300 haplotypes, with repeated pairs and a pair of a haplotype with itself."""
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 300, n).tolist()
    b = rng.integers(0, 300, n).tolist()
    if n > 6:
        a[5], b[5] = a[0], b[0]
        a[6], b[6] = a[3], a[3]
    return a, b


def _host(m, a, b, outputs):
    m.decodePairs(a, b, outputs.get("per_pair_posteriors", False), outputs.get("sum_of_posteriors", False),
                  outputs.get("per_pair_posterior_means", False), outputs.get("per_pair_MAPs", False))
    r = m.get_ref_of_results()
    out = dict(per_pair_indices=list(r.per_pair_indices))
    if outputs.get("per_pair_posteriors"):
        out["per_pair_posteriors"] = np.stack([np.array(x) for x in r.per_pair_posteriors])
    if outputs.get("sum_of_posteriors"):
        out["sum_of_posteriors"] = np.array(r.sum_of_posteriors).copy()
    if outputs.get("per_pair_posterior_means"):
        out["per_pair_posterior_means"] = np.array(r.per_pair_posterior_means).copy()
        out["min_posterior_means"] = np.array(r.min_posterior_means, np.float32)
        out["argmin_posterior_means"] = np.array(r.argmin_posterior_means, np.int32)
    if outputs.get("per_pair_MAPs"):
        out["per_pair_MAPs"] = np.array(r.per_pair_MAPs).copy()
        out["min_MAPs"] = np.array(r.min_MAPs, np.int32)
        out["argmin_MAPs"] = np.array(r.argmin_MAPs, np.int32)
    return out


def _same(got, want, name, sums_exact):
    got = got.cpu().numpy()
    assert got.shape == want.shape, name
    if name == "sum_of_posteriors" and not sums_exact:
        np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-30, err_msg=name)
    elif got.dtype == np.float32:
        assert np.array_equal(got.view(np.uint32), np.ascontiguousarray(want, np.float32).view(np.uint32)), name
    else:
        assert np.array_equal(got, want), name


def check_case(case, n=150, ids=False):
    """decode_pairs_cuda on a non-default stream vs ASMC.decodePairs, every field; the host results stay untouched."""
    from fastsmc_b200.cuda_results import decode_pairs_cuda
    root, dq, exact, outputs, sums_exact = CASES[case]
    m = _asmc(root, dq, exact)
    a, b = _pairs(n, seed=n)
    want = _host(m, a, b, outputs)
    if ids:
        a = [t[1] for t in want["per_pair_indices"]]
        b = [t[3] for t in want["per_pair_indices"]]
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        res = decode_pairs_cuda(m, a, b, **outputs)
        torch.cuda.current_stream().synchronize()
    assert res.d2h_bytes == 0
    assert [tuple(t) for t in res.per_pair_indices] == [tuple(t) for t in want["per_pair_indices"]]
    for name, w in want.items():
        if name != "per_pair_indices":
            t = getattr(res, name)
            assert t.device == torch.device("cuda", 0), name
            _same(t, w, name, sums_exact)
    r = m.get_ref_of_results()
    if outputs.get("per_pair_posterior_means"):
        assert np.array_equal(np.array(r.per_pair_posterior_means).view(np.uint32),
                              want["per_pair_posterior_means"].view(np.uint32))


@pytest.mark.parametrize("case", list(CASES))
def test_device_outputs_equal_decode_pairs(case):
    check_case(case)


def test_device_outputs_across_chunks():
    """One reference batch per chunk (FSMC_FLUSH_BATCHES=1): rows cross chunk boundaries; repeated pairs, string ids, and
    a single pair."""
    env = dict(os.environ, FSMC_FLUSH_BATCHES="1")
    code = (f"import sys; sys.path.insert(0, {HERE!r}); import test_gpu_device_outputs as t; "
            "t.check_case('exact69', n=200); t.check_case('fast69', n=150, ids=True); t.check_case('fast69', n=1)")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


# ---- C ABI: kernel choice, traffic, rejections ------------------------------------------------------------------------

# states -> (data, decoding quantities, oracle options, pairs per request)
MODELS = {69: (ASMC_EXAMPLE, DQ_69, dict(hashing=False, FastSMC=False, asmcMode=True, batchSize=64, useKnownSeed=True), 70),
          159: (FASTSMC_EXAMPLE, FASTSMC_EXAMPLE_DQ, dict(REGRESSION_PARAMS, hashing=True), 40)}
_MODEL_CACHE = {}


def _model(states):
    """(context, oracle) of a model: the oracle's tables are the inputs (conftest.context_from_oracle)."""
    if states not in _MODEL_CACHE:
        from oracle import pyoracle
        pyoracle.build()
        root, dq, kw, _ = MODELS[states]
        o = pyoracle.Oracle(root, dq, f"/tmp/fsmc_device_outputs_o{states}", **kw)
        _MODEL_CACHE[states] = (context_from_oracle(o, pyoracle), o)
    return _MODEL_CACHE[states]


def _tiles(ctx, o, n=70):
    a, b = _pairs(n, seed=3)
    return ctx.make_tiles(a, b, sites=o.sites, batch_size=64)


FLAG_SETS = {"mean_map": 0x4 | 0x8, "map_ibd": 0x8 | 0x10, "posterior_sum": 0x200 | 0x400, "sum": 0x400,
             "exact_all": 0x4 | 0x8 | 0x10 | 0x200 | 0x400 | 0x20, "ibd_wide": 0x10 | 0x80}
C_ABI_CASES = [(69, w) for w in FLAG_SETS] + [(159, w) for w in ("mean_map", "sum", "exact_all")]


@pytest.mark.parametrize("states,which", C_ABI_CASES)
def test_decode_device_same_kernel_and_values_as_decode(states, which):
    check_c_abi(states, which)


def check_c_abi(states, which):
    """fsmc_decode_device runs the kernel fsmc_decode runs for the same flags and writes the same rows (through a row
    table that reverses the pairs); fsmc_decode's d2hBytes is its output size, fsmc_decode_device's is 0."""
    ctx, o = _model(states)
    flags = FLAG_SETS[which]
    tiles = _tiles(ctx, o, MODELS[states][3])
    host = ctx.decode(tiles, flags)
    n, L, S = len(tiles["rows"]), o.sites, o.states
    rows = np.zeros(len(tiles["tilePairs"]) * 32, np.int64)
    rows[tiles["rows"]] = np.arange(n)[::-1]
    dev = torch.device("cuda", 0)
    t = dict(site_mean=torch.full((n, L), -1.0, device=dev) if flags & 0x4 else None,
             site_map=torch.full((n, L), -1, dtype=torch.int32, device=dev) if flags & 0x8 else None,
             site_ibd=torch.full((n, L), -1.0, device=dev) if flags & 0x10 else None,
             site_posterior=torch.full((n, S, L), -1.0, device=dev) if flags & 0x200 else None,
             sum_posterior=torch.full((1, S, L), 0.5, device=dev) if flags & 0x400 else None)
    w = np.linspace(0.5, 2.0, S).astype(np.float32)
    st = ctx.decode_device(tiles, flags, rows, n, L, state_weight=w, **t)
    torch.cuda.synchronize()
    for f in ("statesKernel", "narrowKernel", "sparseKernel", "tileWarps"):
        assert getattr(st, f) == getattr(host.stats, f), f
    assert st.d2hBytes == 0
    nlane = len(tiles["tilePairs"]) * 32
    out_bytes = sum(x.nbytes for x in (host.site_mean, host.site_map, host.site_ibd, host.site_posterior, host.sum_posterior)
                    if x is not None)
    assert host.stats.d2hBytes == out_bytes and nlane >= n
    order = tiles["rows"][::-1]  # device row r holds pair n-1-r
    for name, h in (("site_mean", host.site_mean), ("site_map", host.site_map), ("site_ibd", host.site_ibd)):
        if h is not None:
            got = t[name].cpu().numpy()
            assert np.array_equal(got, h[order]) if h.dtype != np.float32 else \
                np.array_equal(got.view(np.uint32), h[order].view(np.uint32)), name
    if host.site_posterior is not None:
        want = (host.site_posterior[order] * w[None, :, None]).astype(np.float32)
        assert np.array_equal(t["site_posterior"].cpu().numpy().view(np.uint32), want.view(np.uint32))
    if host.sum_posterior is not None:
        want = np.float32(0.5) + host.sum_posterior.astype(np.float64) * w[None, :, None]
        np.testing.assert_allclose(t["sum_posterior"].cpu().numpy(), want, rtol=1e-5)


def test_decode_device_rejections():
    """Host memory, memory of another device, a row table or stride too small for the outputs, segment calling, and a
    narrow-kernel request: each is refused before any kernel runs; the context keeps working."""
    from fastsmc_b200 import _native
    ctx, o = _model(69)
    tiles = _tiles(ctx, o)
    n, L = len(tiles["rows"]), o.sites
    rows = np.zeros(len(tiles["tilePairs"]) * 32, np.int64)
    rows[tiles["rows"]] = np.arange(n)
    dev = torch.device("cuda", 0)
    good = torch.empty((n, L), device=dev)
    bad = [
        (dict(site_mean=torch.empty((n, L))), 0x4, rows, n, L),                     # host tensor
        (dict(site_mean=torch.empty((n, L)).pin_memory()), 0x4, rows, n, L),        # page-locked host memory
        (dict(site_mean=good), 0x4, rows, n, L - 1),                                 # stride below the window
        (dict(site_mean=good), 0x4, rows, n - 1, L),                                 # a row outside numRows
        (dict(site_mean=torch.empty((n - 1, L), device=dev)), 0x4, rows, n, L),      # tensor smaller than numRows x stride
        (dict(site_mean=good), 0x4 | 0x1, rows, n, L),                               # segment calling
    ]
    if ctx.decode(tiles, 0x10).stats.narrowKernel:
        bad.append((dict(site_ibd=good), 0x10, rows, n, L))                         # the narrow kernel would run
    if torch.cuda.device_count() > 1:
        bad.append((dict(site_mean=torch.empty((n, L), device="cuda:1")), 0x4, rows, n, L))
    for kw, flags, r, nr, stride in bad:
        with pytest.raises((_native.FastSMCError, RuntimeError)):
            ctx.decode_device(tiles, flags, r, nr, stride, **kw)
    st = ctx.decode_device(tiles, 0x4, rows, n, L, site_mean=good)  # still usable
    torch.cuda.synchronize()
    assert st.statesKernel == 69


@pytest.mark.parametrize("dtype", ["float32", "int32"])
@pytest.mark.parametrize("shape", [(1, 7), (3, 1), (257, 33), (5000, 1001), (100003, 37)])
def test_column_min_first_row_of_minimum(shape, dtype):
    """fsmc_column_min_*: torch.min(dim=0) values, and the first row of the minimum (finaliseCalculations' rule) on
    matrices with planted ties; a padded leading dimension; NaN rows skipped unless in row 0."""
    from fastsmc_b200.cuda_results import _context
    rows, cols = shape
    g = torch.Generator().manual_seed(rows * 131 + cols)
    if dtype == "float32":
        m = torch.randint(0, 50, (rows, cols + 3), generator=g).float() / 7.0
    else:
        m = torch.randint(-20, 20, (rows, cols + 3), generator=g).to(torch.int32)
    m = m[:, :cols]  # leading dimension cols + 3
    if dtype == "float32" and rows > 2:
        m[1, 0] = float("nan")
        m[0, min(1, cols - 1)] = float("nan") if cols > 1 else m[0, 0]
    dev = m.cuda()
    mn = torch.empty(cols, dtype=m.dtype, device="cuda")
    am = torch.empty(cols, dtype=torch.int32, device="cuda")
    _context(0).column_min(dev, mn, am)
    torch.cuda.synchronize()
    x = m.numpy()
    # the reference loop (start at row 0, take a row only when strictly smaller): the first row of the minimum over row 0
    # and the later non-NaN rows; a NaN in row 0 stays (the values here are finite otherwise)
    skip = np.isnan(x) if dtype == "float32" else np.zeros(x.shape, bool)
    skip[0] = False
    xx = np.where(skip, np.inf, x) if dtype == "float32" else x
    want_i = np.argmin(np.where(np.isnan(xx), -np.inf, xx) if dtype == "float32" else xx, axis=0).astype(np.int32)
    if dtype == "float32":
        want_i[np.isnan(x[0])] = 0
    want_v = x[want_i, np.arange(cols)]
    got_v, got_i = mn.cpu().numpy(), am.cpu().numpy()
    assert np.array_equal(got_i, want_i)
    assert np.array_equal(got_v.view(np.uint32), want_v.view(np.uint32))
    finite = ~np.isnan(x).any(axis=0)
    tv, ti = torch.min(m, dim=0)
    assert np.array_equal(got_v[finite], tv.numpy()[finite])
