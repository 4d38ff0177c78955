// fastsmc_b200 — selection of the lane-split decode kernels (decode_lane.cuh).  The instantiations live in their own
// translation unit (lane_159.cu) so that the library's sources compile in parallel.
#pragma once

#include <cstddef>

#include "decode_fast.cuh"

namespace fsmc
{

typedef void (*FastKernelFn)(const FastModel, const DecodeArgs);

struct LaneChoice {
  FastKernelFn fn = nullptr;
  int warps = 0;          // warps per tile == warps per CTA
  size_t smemBytes = 0;   // dynamic shared memory per CTA
  int recordQuads = 0;    // 0 = wide (full beta rows in HBM)
  int Spad = 0;
};

// Lane-split kernels (lane_159.cu) at 159 states.  recordQuads: 1 to 4, records of ceil((stateThreshold + 1) / 4) quads
// (FastSMC_exe's default flags), or 0: full beta rows (per-site mean / MAP, age estimates over all states).  Returns
// fn == nullptr for any other value.  The kernels read the per-site laneAux table of the model (buildLaneAux159).
LaneChoice laneKernel159(int recordQuads);
size_t laneAuxFloats159();
void buildLaneAux159(int L, const float* rows, float* aux, int blocks, cudaStream_t st);

}  // namespace fsmc
