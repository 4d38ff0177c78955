// Column minimum and argmin of a row-major device matrix (fsmc_column_min_f32 / _i32), with the rule of
// DecodePairsReturnStruct::finaliseCalculations (ref: DecodePairsReturnStruct.hpp:105-118): row 0 is the start value, a
// later row replaces the current best only when strictly smaller.  So the result is the first row of the minimum, a NaN in
// row 0 is kept and NaNs in later rows are skipped.
//
// Pass 1: a block of 32 columns x 8 row groups reads a chunk of rows (a warp reads 128 contiguous bytes of a row); each
// thread scans its rows in ascending order, the 8 group results are combined in shared memory.  Pass 2 (only when the rows
// were cut into several chunks) combines the chunk results of each column.  Every combination compares (value, row), so the
// result does not depend on the order of the combinations: it is deterministic.
#pragma once

#include <cstdint>

namespace fsmc
{

constexpr int kColMinCols = 32;
constexpr int kColMinGroups = 8;

template <class T> __device__ __forceinline__ bool colMinIsNan(const T v)
{
  return v != v;  // false for every integer
}

// best = (v, row) of a partial scan, row < 0 = empty.  Takes `o` when it is the result of the sequential rule over both.
template <class T> __device__ __forceinline__ void colMinCombine(T& v, int& row, const T ov, const int orow)
{
  if (orow < 0 || (row == 0 && colMinIsNan(v))) {
    return;
  }
  if (row < 0 || (orow == 0 && colMinIsNan(ov)) || ov < v || (ov == v && orow < row)) {
    v = ov;
    row = orow;
  }
}

template <class T>
__global__ void __launch_bounds__(kColMinCols * kColMinGroups) columnMinPartialKernel(
    const T* __restrict__ m, const long long rows, const long long cols, const long long ld, const long long rowsPerChunk,
    T* __restrict__ outV, int* __restrict__ outRow)
{
  __shared__ T sv[kColMinGroups][kColMinCols];
  __shared__ int sr[kColMinGroups][kColMinCols];
  const int tx = threadIdx.x, ty = threadIdx.y;
  const long long col = static_cast<long long>(blockIdx.x) * kColMinCols + tx;
  const long long r0 = static_cast<long long>(blockIdx.y) * rowsPerChunk;
  const long long r1 = min(rows, r0 + rowsPerChunk);
  T best{};
  int arg = -1;
  if (col < cols) {
    constexpr int U = 8;  // loads in flight per thread
    long long r = r0 + ty;
    for (; r + (U - 1) * kColMinGroups < r1; r += U * kColMinGroups) {
      T x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        x[u] = __ldg(m + static_cast<size_t>(r + u * kColMinGroups) * ld + col);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const long long rr = r + u * kColMinGroups;
        if (arg < 0 ? (rr == 0 || !colMinIsNan(x[u])) : x[u] < best) {
          best = x[u];
          arg = static_cast<int>(rr);
        }
      }
    }
    for (; r < r1; r += kColMinGroups) {
      const T x = __ldg(m + static_cast<size_t>(r) * ld + col);
      if (arg < 0 ? (r == 0 || !colMinIsNan(x)) : x < best) {
        best = x;
        arg = static_cast<int>(r);
      }
    }
  }
  sv[ty][tx] = best;
  sr[ty][tx] = arg;
  __syncthreads();
  if (ty == 0 && col < cols) {
    for (int g = 1; g < kColMinGroups; ++g) {
      colMinCombine(best, arg, sv[g][tx], sr[g][tx]);
    }
    outV[static_cast<size_t>(blockIdx.y) * cols + col] = best;
    outRow[static_cast<size_t>(blockIdx.y) * cols + col] = arg;
  }
}

template <class T>
__global__ void columnMinCombineKernel(const T* __restrict__ partV, const int* __restrict__ partRow, const int chunks,
                                       const long long cols, T* __restrict__ outV, int* __restrict__ outRow)
{
  for (long long col = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; col < cols;
       col += static_cast<long long>(gridDim.x) * blockDim.x) {
    T best = partV[col];
    int arg = partRow[col];
    for (int c = 1; c < chunks; ++c) {
      colMinCombine(best, arg, partV[static_cast<size_t>(c) * cols + col], partRow[static_cast<size_t>(c) * cols + col]);
    }
    outV[col] = best;
    outRow[col] = arg;
  }
}

}  // namespace fsmc
