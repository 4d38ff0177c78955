"""ASMC.decodePairs results as CUDA tensors, written in place by the decode kernels.

    res = decode_pairs_cuda(asmc_obj, haps_a, haps_b, per_pair_posterior_means=True)
    res.per_pair_posterior_means   # torch.float32 [pairs][sites] on cuda:{params.device}

The fields carry the names of the reference's DecodePairsReturnStruct and the values ASMC.decodePairs returns, bit for bit
(the sums of posteriors to float rounding where the device adds them with atomics).  Nothing but O(1) statistics crosses
to the host: a user who keeps computing on the per-site outputs (minima over pairs, per-population averages, ...) does not
pay for moving pairs x sites values over PCIe and back.  All tensors are allocated by torch and written on
torch.cuda.current_stream(); read them after that stream (or a stream that waits on it) has reached them.
"""
import torch

from . import _native


class DecodePairsCudaResults:
    """Outputs of one decode_pairs_cuda call; tensors that were not asked for are None."""

    def __init__(self):
        self.per_pair_indices = []
        self.per_pair_posteriors = None      # float32 [pairs][states][sites], posterior * expectedTimes[state]
        self.sum_of_posteriors = None        # float32 [states][sites]
        self.per_pair_posterior_means = None  # float32 [pairs][sites]
        self.min_posterior_means = None      # float32 [sites]
        self.argmin_posterior_means = None   # int32 [sites]: first pair of the minimum
        self.per_pair_MAPs = None            # int32 [pairs][sites]
        self.min_MAPs = None                 # int32 [sites]
        self.argmin_MAPs = None              # int32 [sites]
        self.d2h_bytes = 0                   # decode outputs copied device -> host during the call (0)


_contexts = {}


def _context(device):
    """A library context per device for the column minima (the decode itself runs on the ASMC object's own context)."""
    if device not in _contexts:
        _contexts[device] = _native.Context(device)
    return _contexts[device]


def output_bytes(pairs, states, sites, *, per_pair_posteriors=False, sum_of_posteriors=False, per_pair_posterior_means=False,
                 per_pair_MAPs=False):
    """Device memory the requested outputs take."""
    n = 0
    if per_pair_posteriors:
        n += pairs * states * sites * 4
    if sum_of_posteriors:
        n += states * sites * 4
    if per_pair_posterior_means:
        n += pairs * sites * 4 + sites * 8
    if per_pair_MAPs:
        n += pairs * sites * 4 + sites * 8
    return n


def decode_pairs_cuda(asmc, haps_a, haps_b, *, per_pair_posteriors=False, sum_of_posteriors=False,
                      per_pair_posterior_means=False, per_pair_MAPs=False):
    """ASMC.decodePairs (haplotype indices or "<IID>#<1|2>" ids) with the results returned as CUDA tensors.

    Unlike ASMC.decodePairs this leaves the ASMC object's own results (get_ref_of_results) untouched.
    """
    haps_a, haps_b = list(haps_a), list(haps_b)
    if not haps_a or len(haps_a) != len(haps_b):
        raise ValueError(f"haps_a ({len(haps_a)}) and haps_b ({len(haps_b)}) must be non-empty and of equal length")
    hmm = asmc.hmm()
    rv = hmm.getDecodingReturnValues()
    S, L, n = int(rv.states), int(rv.sites), len(haps_a)
    dev = torch.device("cuda", hmm.getDevice())
    want = dict(per_pair_posteriors=per_pair_posteriors, sum_of_posteriors=sum_of_posteriors,
                per_pair_posterior_means=per_pair_posterior_means, per_pair_MAPs=per_pair_MAPs)
    need = output_bytes(n, S, L, **want)
    free, _ = torch.cuda.mem_get_info(dev)
    if need > free:
        raise MemoryError(f"decode_pairs_cuda: the requested outputs of {n} pairs x {L} sites ({S} states) take "
                          f"{need / 1e9:.2f} GB, {free / 1e9:.2f} GB of {dev} are free; decode fewer pairs per call")
    res = DecodePairsCudaResults()
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev)
        if per_pair_posteriors:
            res.per_pair_posteriors = torch.empty((n, S, L), dtype=torch.float32, device=dev)
        if sum_of_posteriors:
            res.sum_of_posteriors = torch.zeros((S, L), dtype=torch.float32, device=dev)  # the kernels add to it
        if per_pair_posterior_means:
            res.per_pair_posterior_means = torch.empty((n, L), dtype=torch.float32, device=dev)
        if per_pair_MAPs:
            res.per_pair_MAPs = torch.empty((n, L), dtype=torch.int32, device=dev)
        ptr = lambda t: t.data_ptr() if t is not None else 0  # noqa: E731
        before = hmm.getRunStats().d2hBytes
        res.per_pair_indices = asmc.decodePairsToDevice(
            haps_a, haps_b, per_pair_posteriors=ptr(res.per_pair_posteriors), sum_of_posteriors=ptr(res.sum_of_posteriors),
            per_pair_posterior_means=ptr(res.per_pair_posterior_means), per_pair_MAPs=ptr(res.per_pair_MAPs),
            stream=stream.cuda_stream)
        res.d2h_bytes = int(hmm.getRunStats().d2hBytes - before)
        if per_pair_posterior_means or per_pair_MAPs:
            ctx = _context(dev.index)
            ctx.set_stream(stream.cuda_stream)
            try:
                if per_pair_posterior_means:
                    res.min_posterior_means = torch.empty(L, dtype=torch.float32, device=dev)
                    res.argmin_posterior_means = torch.empty(L, dtype=torch.int32, device=dev)
                    ctx.column_min(res.per_pair_posterior_means, res.min_posterior_means, res.argmin_posterior_means)
                if per_pair_MAPs:
                    res.min_MAPs = torch.empty(L, dtype=torch.int32, device=dev)
                    res.argmin_MAPs = torch.empty(L, dtype=torch.int32, device=dev)
                    ctx.column_min(res.per_pair_MAPs, res.min_MAPs, res.argmin_MAPs)
            finally:
                ctx.set_stream(None)
    return res
