// fastsmc_b200 host layer — ASMC facade (per-site posterior mean TMRCA / MAP for chosen haplotype pairs) with the
// reference's interface (ref: ASMC_SRC/SRC/ASMC.hpp:44-68).
#pragma once

#include <string>
#include <vector>

#include "Data.hpp"
#include "DecodePairsReturnStruct.hpp"
#include "DecodingParams.hpp"
#include "HMM.hpp"

namespace ASMC
{

class ASMC
{
  DecodingParams mParams;
  Data mData;
  HMM mHmm;

public:
  explicit ASMC(DecodingParams params);
  ASMC(const std::string& inFileRoot, const std::string& decodingQuantFile, const std::string& outFileRoot = "");

  DecodingReturnValues decodeAllInJob();

  void decodePairs(const std::vector<unsigned long>& hapIndicesA, const std::vector<unsigned long>& hapIndicesB,
                   bool perPairPosteriors = false, bool sumOfPosteriors = false, bool perPairPosteriorMeans = false,
                   bool perPairMAPs = false);
  void decodePairs(const std::vector<std::string>& hapIdsA, const std::vector<std::string>& hapIdsB,
                   bool perPairPosteriors = false, bool sumOfPosteriors = false, bool perPairPosteriorMeans = false,
                   bool perPairMAPs = false);

  /// decodePairs with the outputs written by the kernels into caller-owned device memory of the decoding device (see
  /// HMM::DeviceOutputs; row r = pair r) on out.stream, without touching the results of decodePairs.  Returns
  /// per_pair_indices.  The minima over pairs are left to the caller (fsmc_column_min_f32 / _i32).
  using PairIndices = std::vector<std::tuple<unsigned long, std::string, unsigned long, std::string>>;
  PairIndices decodePairsToDevice(const std::vector<unsigned long>& hapIndicesA, const std::vector<unsigned long>& hapIndicesB,
                                  const HMM::DeviceOutputs& out);
  PairIndices decodePairsToDevice(const std::vector<std::string>& hapIdsA, const std::vector<std::string>& hapIdsB,
                                  const HMM::DeviceOutputs& out);

  DecodePairsReturnStruct getCopyOfResults();
  const DecodePairsReturnStruct& getRefOfResults();
  HMM& hmm() { return mHmm; }
  const Data& data() const { return mData; }
};

}  // namespace ASMC
