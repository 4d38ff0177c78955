"""ctypes binding of the C ABI in include/fastsmc_b200.h (libfastsmc_b200.so).

There is no CPU fallback: importing works without a GPU (so the symbols can be checked), but every
compute call needs a CUDA device and raises FastSMCError otherwise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfastsmc_b200.so")

TILE = 32

# flags (include/fastsmc_b200.h)
CALL_SEGMENTS = 0x1
SEG_AGE = 0x2
SITE_MEAN = 0x4
SITE_MAP = 0x8
SITE_IBD = 0x10
EXACT = 0x20
GENERIC_KERNEL = 0x40
WIDE_KERNEL = 0x80
ONE_WARP_KERNEL = 0x100
SITE_POSTERIOR = 0x200
SUM_POSTERIOR = 0x400
SUM_BY_GENOTYPE = 0x800

E_OVERFLOW = -4


class FastSMCError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"fastsmc_b200 error {code}: {msg}")
        self.code = code


class Model(C.Structure):
    _fields_ = [
        ("states", C.c_int32), ("sites", C.c_int32),
        ("initialStateProb", C.c_void_p), ("expectedTimes", C.c_void_p), ("columnRatios", C.c_void_p),
        ("emission1", C.c_void_p), ("emission0minus1", C.c_void_p), ("emission2minus0", C.c_void_p),
        ("numDistances", C.c_int32),
        ("D", C.c_void_p), ("B", C.c_void_p), ("U", C.c_void_p), ("RR", C.c_void_p),
        ("distanceRow", C.c_void_p),
        ("stateThreshold", C.c_int32), ("ageThreshold", C.c_int32), ("probabilityThreshold", C.c_float),
        ("modelTag", C.c_uint64),
    ]


class Request(C.Structure):
    _fields_ = [
        ("numTiles", C.c_int64),
        ("hapA", C.c_void_p), ("hapB", C.c_void_p), ("tilePairs", C.c_void_p),
        ("tileFrom", C.c_void_p), ("tileTo", C.c_void_p), ("tileScanFrom", C.c_void_p), ("tileScanTo", C.c_void_p),
        ("flags", C.c_uint32),
        ("segments", C.c_void_p), ("segmentCapacity", C.c_int64),
        ("siteMean", C.c_void_p), ("siteMap", C.c_void_p), ("siteIbd", C.c_void_p), ("siteStride", C.c_int64),
        ("sitePosterior", C.c_void_p), ("sumPosterior", C.c_void_p),
    ]


class Stats(C.Structure):
    _fields_ = [
        ("numSegments", C.c_int64), ("pairSites", C.c_double), ("kernelMs", C.c_float), ("totalMs", C.c_float),
        ("kernelLaunches", C.c_int32), ("statesKernel", C.c_int32), ("scratchBytes", C.c_int64),
        ("narrowKernel", C.c_int32), ("tileWarps", C.c_int32),
        ("sparseKernel", C.c_int32), ("checkpointSites", C.c_int32), ("sparseItems", C.c_int64), ("checkpointBytes", C.c_int64),
        ("d2hBytes", C.c_int64),
    ]


class DeviceOutputs(C.Structure):
    _fields_ = [
        ("laneRow", C.c_void_p), ("numRows", C.c_int64), ("siteStride", C.c_int64),
        ("siteMean_dev", C.c_void_p), ("siteMap_dev", C.c_void_p), ("siteIbd_dev", C.c_void_p),
        ("sitePosterior_dev", C.c_void_p), ("sumPosterior_dev", C.c_void_p), ("stateWeight", C.c_void_p),
    ]


SEGMENT_DTYPE = np.dtype([
    ("pair", np.uint32), ("posStart", np.int32), ("posEnd", np.int32), ("prob", np.float32),
    ("postMean", np.float32), ("mapTime", np.float32), ("mapState", np.int32), ("level", np.int32),
])

EXPORTS = [
    "fsmc_last_error", "fsmc_version", "fsmc_device_count", "fsmc_ctx_create", "fsmc_ctx_destroy",
    "fsmc_ctx_set_stream", "fsmc_set_model", "fsmc_set_haplotypes", "fsmc_decode", "fsmc_plan_create",
    "fsmc_plan_launch", "fsmc_plan_collect", "fsmc_plan_destroy", "fsmc_seed", "fsmc_query_kernel",
    "fsmc_decode_device", "fsmc_column_min_f32", "fsmc_column_min_i32",
]

_lib = None


def lib():
    """Load the native library; fail loudly if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise FastSMCError(-100, f"{LIB_PATH} is missing — run `python -m fastsmc_b200.build` (needs nvcc); "
                                     "there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.fsmc_last_error.restype = C.c_char_p
        L.fsmc_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        L.fsmc_ctx_destroy.argtypes = [C.c_void_p]
        L.fsmc_ctx_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        L.fsmc_set_model.argtypes = [C.c_void_p, C.POINTER(Model)]
        L.fsmc_set_haplotypes.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64]
        L.fsmc_decode.argtypes = [C.c_void_p, C.POINTER(Request), C.POINTER(Stats)]
        L.fsmc_plan_create.argtypes = [C.c_void_p, C.POINTER(Request), C.POINTER(C.c_void_p)]
        L.fsmc_plan_launch.argtypes = [C.c_void_p, C.c_void_p]
        L.fsmc_plan_collect.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(Request), C.POINTER(Stats)]
        L.fsmc_plan_destroy.argtypes = [C.c_void_p, C.c_void_p]
        L.fsmc_decode_device.argtypes = [C.c_void_p, C.POINTER(Request), C.POINTER(DeviceOutputs), C.POINTER(Stats)]
        for f in (L.fsmc_column_min_f32, L.fsmc_column_min_i32):
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]
        _lib = L
    return _lib


def _check(rc, allow=()):
    if rc != 0 and rc not in allow:
        raise FastSMCError(rc, lib().fsmc_last_error().decode())
    return rc


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def pack_haplotypes(haps):
    """[numHaps][sites] array of 0/1 -> [numHaps][ceil(sites/64)] uint64, bit s%64 of word s/64 = allele at site s."""
    haps = np.ascontiguousarray(haps, dtype=np.uint8)
    n, sites = haps.shape
    words = (sites + 63) // 64
    padded = np.zeros((n, words * 64), np.uint8)
    padded[:, :sites] = haps
    packed = np.packbits(padded.reshape(n, words, 64), axis=2, bitorder="little")
    return np.ascontiguousarray(packed).view(np.uint64).reshape(n, words)


class DecodeResult:
    def __init__(self, segments, site_mean, site_map, site_ibd, stats, site_posterior=None, sum_posterior=None):
        self.segments = segments
        self.site_mean = site_mean
        self.site_map = site_map
        self.site_ibd = site_ibd
        self.stats = stats
        self.site_posterior = site_posterior  # [pairs][states][siteStride]
        self.sum_posterior = sum_posterior    # [planes][states][sites]


class Context:
    """One GPU's decode context (fsmc_ctx)."""

    def __init__(self, device=0):
        self._h = C.c_void_p()
        _check(lib().fsmc_ctx_create(device, C.byref(self._h)))
        self.device = device
        self.states = 0
        self.sites = 0
        self.num_haps = 0
        self._keep = []

    def close(self):
        if getattr(self, "_h", None):
            lib().fsmc_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream):
        _check(lib().fsmc_ctx_set_stream(self._h, C.c_void_p(cuda_stream) if cuda_stream else None))

    def set_model(self, *, initial_state_prob, expected_times, column_ratios, emission1, emission0minus1,
                  emission2minus0, D, B, U, RR, distance_row, state_threshold, age_threshold, probability_threshold):
        e1, e0, e2 = _f32(emission1), _f32(emission0minus1), _f32(emission2minus0)
        L, S = e1.shape
        Dm, Bm, Um, Rm = _f32(D), _f32(B), _f32(U), _f32(RR)
        row = np.ascontiguousarray(distance_row, dtype=np.int32)
        pri, exp, col = _f32(initial_state_prob), _f32(expected_times), _f32(column_ratios)
        assert e0.shape == (L, S) and e2.shape == (L, S) and Dm.shape[1] == S and row.shape == (L,)
        m = Model(S, L, _p(pri), _p(exp), _p(col), _p(e1), _p(e0), _p(e2), Dm.shape[0], _p(Dm), _p(Bm), _p(Um), _p(Rm),
                  _p(row), int(state_threshold), int(age_threshold), float(probability_threshold))
        _check(lib().fsmc_set_model(self._h, C.byref(m)))
        self.states, self.sites = S, L

    def set_haplotypes(self, packed, sites):
        packed = np.ascontiguousarray(packed, dtype=np.uint64)
        assert packed.shape[1] == (sites + 63) // 64
        _check(lib().fsmc_set_haplotypes(self._h, _p(packed), packed.shape[0], sites))
        self.num_haps = packed.shape[0]

    # ---- request assembly
    @staticmethod
    def make_tiles(hap_a, hap_b, windows=None, scan=None, sites=None, batch_size=32):
        """Group a pair stream into tiles of <=32 pairs.

        hap_a, hap_b: per-pair haplotype indices, in reference submission order.
        windows / scan: per *batch* (batch_size consecutive pairs) (from,to) arrays; None = whole sequence.
        Returns dict of request arrays + index of each pair's row (tile*32+lane).
        """
        a = np.asarray(hap_a, dtype=np.uint32)
        b = np.asarray(hap_b, dtype=np.uint32)
        n = len(a)
        nb = (n + batch_size - 1) // batch_size
        if windows is None:
            windows = np.tile(np.array([[0, sites]], np.int32), (nb, 1))
        if scan is None:
            scan = windows
        windows = np.asarray(windows, np.int32).reshape(nb, 2)
        scan = np.asarray(scan, np.int32).reshape(nb, 2)
        tA, tB, tn, tf, tt, sf, stt, rows = [], [], [], [], [], [], [], np.empty(n, np.int64)
        tile = 0
        for bi in range(nb):
            lo, hi = bi * batch_size, min(n, (bi + 1) * batch_size)
            for s in range(lo, hi, TILE):
                e = min(hi, s + TILE)
                la = np.zeros(TILE, np.uint32)
                lb = np.zeros(TILE, np.uint32)
                la[:e - s] = a[s:e]
                lb[:e - s] = b[s:e]
                tA.append(la)
                tB.append(lb)
                tn.append(e - s)
                tf.append(windows[bi, 0])
                tt.append(windows[bi, 1])
                sf.append(scan[bi, 0])
                stt.append(scan[bi, 1])
                rows[s:e] = tile * TILE + np.arange(e - s)
                tile += 1
        z = np.zeros((0, TILE), np.uint32)
        return dict(hapA=np.ascontiguousarray(np.stack(tA) if tA else z), hapB=np.ascontiguousarray(np.stack(tB) if tB else z),
                    tilePairs=np.array(tn, np.int32), tileFrom=np.array(tf, np.int32), tileTo=np.array(tt, np.int32),
                    tileScanFrom=np.array(sf, np.int32), tileScanTo=np.array(stt, np.int32), rows=rows)

    def _request(self, tiles, flags, segment_capacity, site_stride, segment_prefill=None):
        T = len(tiles["tilePairs"])
        out = {}
        # uninitialised on purpose: the library never reads the caller's record buffer, and zero-filling capacity-sized
        # buffers would be host time inside every call
        seg = np.empty(max(segment_capacity, 1), SEGMENT_DTYPE) if flags & CALL_SEGMENTS else None
        if seg is not None and segment_prefill is not None:
            # previous contents of the caller's record buffer (the library must not depend on them)
            n = min(len(seg), len(segment_prefill))
            seg[:n] = segment_prefill[:n]
        stride = 0
        if flags & (SITE_MEAN | SITE_MAP | SITE_IBD | SITE_POSTERIOR):
            stride = site_stride or int((tiles["tileTo"] - tiles["tileFrom"]).max()) if T else 0
        mean = np.zeros((T * TILE, stride), np.float32) if flags & SITE_MEAN else None
        smap = np.zeros((T * TILE, stride), np.int32) if flags & SITE_MAP else None
        ibd = np.zeros((T * TILE, stride), np.float32) if flags & SITE_IBD else None
        post = np.zeros((T * TILE, self.states, stride), np.float32) if flags & SITE_POSTERIOR else None
        psum = (np.zeros((3 if flags & SUM_BY_GENOTYPE else 1, self.states, self.sites), np.float32)
                if flags & SUM_POSTERIOR else None)
        req = Request(T, _p(tiles["hapA"]), _p(tiles["hapB"]), _p(tiles["tilePairs"]), _p(tiles["tileFrom"]),
                      _p(tiles["tileTo"]), _p(tiles["tileScanFrom"]), _p(tiles["tileScanTo"]), flags,
                      _p(seg), segment_capacity if seg is not None else 0, _p(mean), _p(smap), _p(ibd), stride,
                      _p(post), _p(psum))
        out.update(seg=seg, mean=mean, smap=smap, ibd=ibd, post=post, psum=psum)
        return req, out

    def decode(self, tiles, flags, segment_capacity=1 << 20, site_stride=0, segment_prefill=None):
        """One-shot fsmc_decode with host buffers.  Grows the segment buffer and retries on overflow."""
        while True:
            req, out = self._request(tiles, flags, segment_capacity, site_stride, segment_prefill)
            stats = Stats()
            rc = _check(lib().fsmc_decode(self._h, C.byref(req), C.byref(stats)), allow=(E_OVERFLOW,))
            if rc == E_OVERFLOW:
                segment_capacity = int(stats.numSegments) + 1024
                continue
            seg = out["seg"][:stats.numSegments] if out["seg"] is not None else None
            return DecodeResult(seg, out["mean"], out["smap"], out["ibd"], stats, out["post"], out["psum"])

    # ---- device-resident outputs (torch tensors or anything with data_ptr() on this context's device)
    def decode_device(self, tiles, flags, lane_row, num_rows, site_stride, *, site_mean=None, site_map=None, site_ibd=None,
                      site_posterior=None, sum_posterior=None, state_weight=None):
        """fsmc_decode_device: the kernels write the given device buffers, row lane_row[tile*32+lane] of each.  The buffers'
        sizes are checked here (the C ABI sees raw pointers); where they lie is checked by the library."""
        T = len(tiles["tilePairs"])
        per_pair = site_stride * num_rows
        need = {"site_mean": (site_mean, per_pair), "site_map": (site_map, per_pair), "site_ibd": (site_ibd, per_pair),
                "site_posterior": (site_posterior, per_pair * self.states),
                "sum_posterior": (sum_posterior, (3 if flags & SUM_BY_GENOTYPE else 1) * self.states * self.sites)}
        for name, (t, n) in need.items():
            if t is not None and t.numel() < n:
                raise FastSMCError(-1, f"{name} has {t.numel()} elements, {n} needed")
            if t is not None and not t.is_contiguous():
                raise FastSMCError(-1, f"{name} is not contiguous")
        rows = np.ascontiguousarray(lane_row, dtype=np.int64)
        assert rows.shape == (T * TILE,)
        w = _f32(state_weight) if state_weight is not None else None
        req = Request(T, _p(tiles["hapA"]), _p(tiles["hapB"]), _p(tiles["tilePairs"]), _p(tiles["tileFrom"]),
                      _p(tiles["tileTo"]), _p(tiles["tileScanFrom"]), _p(tiles["tileScanTo"]), flags,
                      None, 0, None, None, None, 0, None, None)
        ptr = lambda t: t.data_ptr() if t is not None else None  # noqa: E731
        out = DeviceOutputs(_p(rows), int(num_rows), int(site_stride), ptr(site_mean), ptr(site_map), ptr(site_ibd),
                            ptr(site_posterior), ptr(sum_posterior), _p(w))
        stats = Stats()
        _check(lib().fsmc_decode_device(self._h, C.byref(req), C.byref(out), C.byref(stats)))
        return stats

    def column_min(self, m, out_min, out_argmin):
        """fsmc_column_min_f32 / _i32 of a 2-D row-major device tensor (float32 or int32) on the context's stream."""
        if m.dim() != 2 or m.stride(1) != 1 or out_min.numel() < m.shape[1] or out_argmin.numel() < m.shape[1]:
            raise FastSMCError(-1, "column_min: needs a row-major 2-D matrix and outputs of one value per column")
        rows, cols = m.shape
        f = lib().fsmc_column_min_f32 if m.dtype.is_floating_point else lib().fsmc_column_min_i32
        _check(f(self._h, m.data_ptr(), rows, cols, m.stride(0), out_min.data_ptr(), out_argmin.data_ptr()))

    # ---- split phase (device-resident inputs)
    def plan(self, tiles, flags, segment_capacity=1 << 20, site_stride=0):
        req, out = self._request(tiles, flags, segment_capacity, site_stride)
        h = C.c_void_p()
        _check(lib().fsmc_plan_create(self._h, C.byref(req), C.byref(h)))
        return Plan(self, h, req, out, tiles)


class Plan:
    def __init__(self, ctx, handle, req, out, tiles):
        self.ctx, self._h, self._req, self._out, self._tiles = ctx, handle, req, out, tiles

    def launch(self):
        _check(lib().fsmc_plan_launch(self.ctx._h, self._h))

    def collect(self):
        stats = Stats()
        _check(lib().fsmc_plan_collect(self.ctx._h, self._h, C.byref(self._req), C.byref(stats)))
        o = self._out
        seg = o["seg"][:stats.numSegments] if o["seg"] is not None else None
        return DecodeResult(seg, o["mean"], o["smap"], o["ibd"], stats, o["post"], o["psum"])

    def close(self):
        if self._h:
            lib().fsmc_plan_destroy(self.ctx._h, self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
