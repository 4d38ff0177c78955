// fastsmc_b200 — device-side ordering of the segment records of one decode call.
//
// The decode kernels append records with one atomic each, so they arrive in no particular order; the reference's
// order is (batch, pair in batch, site ascending) = ascending (pair index, first site).  A lane appends its own
// segments in ascending site order, so a STABLE sort by pair index restores the order: one radix sort of
// (pair, arrival index) and a gather, microseconds on the device, instead of a counting sort of the records on the
// host inside every fsmc_decode call.
#pragma once

#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/fastsmc_b200.h"

namespace fsmc
{

class SegmentSorter
{
public:
  SegmentSorter() = default;
  SegmentSorter(const SegmentSorter&) = delete;
  SegmentSorter& operator=(const SegmentSorter&) = delete;
  ~SegmentSorter();
  // Sorts in[0..n) by `pair` (stable) on `stream`; *out points at the sorted records (device memory owned by the
  // sorter, valid until the next call).  numPairs bounds the pair index (radix passes are limited to its bits).
  cudaError_t sort(const fsmc_segment* in, long long n, uint32_t numPairs, cudaStream_t stream, const fsmc_segment** out);

private:
  cudaError_t reserve(size_t n);
  void release();
  void* mTemp = nullptr;
  size_t mTempBytes = 0;
  uint32_t* mKeys = nullptr;  // [4][capacity]: keys, sorted keys, arrival indices, sorted indices
  fsmc_segment* mSorted = nullptr;
  size_t mCapacity = 0;
};

// The columns of fsmc_plan_collect_device from n sorted records: record i goes to index out.offset + i.  hapA / hapB are
// the plan's haplotypes per pair (tile * 32 + lane); gen / bp the site positions.
cudaError_t writeSegmentColumns(const fsmc_segment* sorted, long long n, const uint32_t* hapA, const uint32_t* hapB,
                                const float* gen, const int32_t* bp, const fsmc_device_segments& out, cudaStream_t stream);

}  // namespace fsmc
