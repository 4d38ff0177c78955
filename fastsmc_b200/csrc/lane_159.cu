// fastsmc_b200 — lane-split decode kernel (decode_lane.cuh) for the 159-state decoding quantities (FASTSMC_EXAMPLE).
#include "decode_lane.cuh"
#include "lane_select.h"

namespace fsmc
{

constexpr int kLaneGroup = 4, kLaneDepth = 2;

template <int S, int RQ, int MINB> static LaneChoice makeLane()
{
  return LaneChoice{decodeLaneKernel<S, RQ, kLaneGroup, kLaneDepth, MINB>, kLaneQuarters,
                    LaneSmem<S, RQ, kLaneGroup, kLaneDepth>::kTotal, RQ, LaneGeom<S>::Spad};
}

template <int S, int MINB> static LaneChoice makeLaneWide()
{
  return LaneChoice{decodeLaneWideKernel<S, kLaneGroup, kLaneDepth, MINB>, kLaneQuarters,
                    LaneWideSmem<S, kLaneGroup, kLaneDepth>::kTotal, 0, LaneGeom<S>::Spad};
}

LaneChoice laneKernel159(const int recordQuads)
{
  switch (recordQuads) {
  case 0:
    return makeLaneWide<159, 3>();  // every state reaches the consumers: full beta rows through HBM
  case 1:
    return makeLane<159, 1, 3>();
  case 2:
    return makeLane<159, 2, 3>();
  case 3:
    return makeLane<159, 3, 3>();  // --time up to 140 generations with the example table
  case 4:
    return makeLane<159, 4, 3>();
  default:
    return {};
  }
}

size_t laneAuxFloats159()
{
  return LaneGeom<159>::kAuxFloats;
}

void buildLaneAux159(const int L, const float* rows, float* aux, const int blocks, cudaStream_t st)
{
  buildLaneAuxKernel<<<blocks, 256, 0, st>>>(LaneGeom<159>::Spad, L, rows, aux);
}

}  // namespace fsmc
