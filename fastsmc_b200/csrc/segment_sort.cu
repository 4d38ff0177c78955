// fastsmc_b200 — see segment_sort.h.
#include "segment_sort.h"

#include <algorithm>
#include <cub/device/device_radix_sort.cuh>

namespace fsmc
{

namespace
{
__global__ void segmentKeysKernel(const fsmc_segment* __restrict__ in, const long long n, uint32_t* __restrict__ keys,
                                  uint32_t* __restrict__ index)
{
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    keys[i] = in[i].pair;
    index[i] = static_cast<uint32_t>(i);
  }
}

// one 32-byte record per pair of threads would be finer-grained; a record per thread as two 16-byte halves is enough
__global__ void segmentGatherKernel(const fsmc_segment* __restrict__ in, const uint32_t* __restrict__ index, const long long n,
                                    fsmc_segment* __restrict__ out)
{
  static_assert(sizeof(fsmc_segment) == 32, "records move as two 16-byte halves");
  const uint4* src = reinterpret_cast<const uint4*>(in);
  uint4* dst = reinterpret_cast<uint4*>(out);
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < 2 * n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    dst[i] = src[2ll * index[i >> 1] + (i & 1)];
  }
}

// HMM::toIbdSegment + the fields of HMM::formatSegments, one record per thread, with the writer's roundings
__global__ void segmentColumnsKernel(const fsmc_segment* __restrict__ in, const long long n, const uint32_t* __restrict__ hapA,
                                     const uint32_t* __restrict__ hapB, const float* __restrict__ gen,
                                     const int32_t* __restrict__ bp, const fsmc_device_segments out)
{
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const fsmc_segment g = in[i];
    const uint32_t a = hapA[g.pair], b = hapB[g.pair];
    const long long o = out.offset + i;
    out.ind1_dev[o] = static_cast<int32_t>(a / 2);
    out.hap1_dev[o] = 1 + static_cast<int32_t>(a % 2);
    out.ind2_dev[o] = static_cast<int32_t>(b / 2);
    out.hap2_dev[o] = 1 + static_cast<int32_t>(b % 2);
    out.startSite_dev[o] = g.posStart;
    out.endSite_dev[o] = g.posEnd;
    out.startBp_dev[o] = bp[g.posStart];
    out.endBp_dev[o] = bp[g.posEnd];
    out.lengthCm_dev[o] = __fmul_rn(100.f, __fsub_rn(gen[g.posEnd], gen[g.posStart]));
    const double sites = static_cast<double>(static_cast<unsigned>(g.posEnd - g.posStart) + 1u);
    out.score_dev[o] = __double2float_rn(__ddiv_rn(static_cast<double>(g.prob), sites));
    if (out.postMean_dev) {
      out.postMean_dev[o] = g.postMean;
    }
    if (out.mapTime_dev) {
      out.mapTime_dev[o] = g.mapTime;
    }
  }
}
}  // namespace

cudaError_t writeSegmentColumns(const fsmc_segment* sorted, const long long n, const uint32_t* hapA, const uint32_t* hapB,
                                const float* gen, const int32_t* bp, const fsmc_device_segments& out, cudaStream_t stream)
{
  if (n <= 0) {
    return cudaSuccess;
  }
  const int blocks = static_cast<int>(std::min<long long>((n + 255) / 256, 148 * 8));
  segmentColumnsKernel<<<blocks, 256, 0, stream>>>(sorted, n, hapA, hapB, gen, bp, out);
  return cudaGetLastError();
}

SegmentSorter::~SegmentSorter()
{
  release();
}

void SegmentSorter::release()
{
  cudaFree(mTemp);
  cudaFree(mKeys);
  cudaFree(mSorted);
  mTemp = nullptr;
  mKeys = nullptr;
  mSorted = nullptr;
  mTempBytes = 0;
  mCapacity = 0;
}

cudaError_t SegmentSorter::reserve(const size_t n)
{
  if (n <= mCapacity) {
    return cudaSuccess;
  }
  release();
  const size_t cap = n + n / 4 + 1024;
  cudaError_t e = cudaMalloc(&mKeys, 4 * cap * sizeof(uint32_t));
  if (e == cudaSuccess) {
    e = cudaMalloc(&mSorted, cap * sizeof(fsmc_segment));
  }
  if (e == cudaSuccess) {
    size_t bytes = 0;
    e = cub::DeviceRadixSort::SortPairs(nullptr, bytes, mKeys, mKeys, mKeys, mKeys, static_cast<int>(std::min<size_t>(cap, 0x7fffffff)));
    if (e == cudaSuccess) {
      e = cudaMalloc(&mTemp, bytes);
      mTempBytes = bytes;
    }
  }
  if (e != cudaSuccess) {
    release();
    return e;
  }
  mCapacity = cap;
  return cudaSuccess;
}

cudaError_t SegmentSorter::sort(const fsmc_segment* in, const long long n, const uint32_t numPairs, cudaStream_t stream,
                                const fsmc_segment** out)
{
  *out = in;
  if (n <= 1) {
    return cudaSuccess;
  }
  if (n > 0x7fffffffll) {
    return cudaErrorInvalidValue;
  }
  cudaError_t e = reserve(static_cast<size_t>(n));
  if (e != cudaSuccess) {
    return e;
  }
  uint32_t* keys = mKeys;
  uint32_t* keysOut = mKeys + mCapacity;
  uint32_t* index = mKeys + 2 * mCapacity;
  uint32_t* indexOut = mKeys + 3 * mCapacity;
  const int blocks = static_cast<int>(std::min<long long>((n + 255) / 256, 148 * 8));
  segmentKeysKernel<<<blocks, 256, 0, stream>>>(in, n, keys, index);
  int bits = 1;
  while (bits < 32 && (1ull << bits) < numPairs) {
    ++bits;
  }
  size_t bytes = mTempBytes;
  e = cub::DeviceRadixSort::SortPairs(mTemp, bytes, keys, keysOut, index, indexOut, static_cast<int>(n), 0, bits, stream);
  if (e != cudaSuccess) {
    return e;
  }
  segmentGatherKernel<<<blocks, 256, 0, stream>>>(in, indexOut, n, mSorted);
  *out = mSorted;
  return cudaGetLastError();
}

}  // namespace fsmc
