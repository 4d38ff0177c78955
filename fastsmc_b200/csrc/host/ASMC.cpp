// fastsmc_b200 host layer — see ASMC.hpp.
#include "ASMC.hpp"

#include <iostream>
#include <stdexcept>

#include "HmmUtils.hpp"

ASMC::ASMC::ASMC(DecodingParams params) : mParams{std::move(params)}, mData{mParams}, mHmm{mData, mParams} {}

// ref: ASMC.cpp:28-50 — array mode, CSFS on, posterior sums + per-pair means + MAP requested
ASMC::ASMC::ASMC(const std::string& inFileRoot, const std::string& decodingQuantFile, const std::string& outFileRoot)
    : mParams{inFileRoot, decodingQuantFile, outFileRoot.empty() ? inFileRoot : outFileRoot,
              1,          1,                 "array",
              false,      true,              false,
              false,      0.f,               false,
              true,       false,             "",
              false,      true,              true},
      mData{mParams}, mHmm{mData, mParams}
{
}

DecodingReturnValues ASMC::ASMC::decodeAllInJob()
{
  std::cout << "Decoding job " << mParams.jobInd << " of " << mParams.jobs << "\n\n";
  mHmm.decodeAll(mParams.jobs, mParams.jobInd);
  return mHmm.getDecodingReturnValues();
}

// ref: ASMC.cpp:80-100
void ASMC::ASMC::decodePairs(const std::vector<unsigned long>& hapIndicesA, const std::vector<unsigned long>& hapIndicesB,
                             bool perPairPosteriors, bool sumOfPosteriors, bool perPairPosteriorMeans, bool perPairMAPs)
{
  if (hapIndicesA.empty() || hapIndicesA.size() != hapIndicesB.size()) {
    throw std::runtime_error("Vector of A indices (" + std::to_string(hapIndicesA.size()) +
                             ") must be the same size as vector of B indices (" + std::to_string(hapIndicesB.size()) +
                             ").\n");
  }
  mHmm.getDecodePairsReturnStruct().initialise(hapIndicesA, hapIndicesB, mData.sites,
                                               mHmm.getDecodingQuantities().states, perPairPosteriors, sumOfPosteriors,
                                               perPairPosteriorMeans, perPairMAPs);
  mHmm.setStorePerPairPosteriorMean(perPairPosteriorMeans);
  mHmm.setStorePerPairMap(perPairMAPs);
  mHmm.setStorePerPairPosterior(perPairPosteriors);
  mHmm.setStoreSumOfPosterior(sumOfPosteriors);
  mHmm.decodeHapPairs(hapIndicesA, hapIndicesB);
  mHmm.finishDecoding();
  mHmm.getDecodePairsReturnStruct().finaliseCalculations();
}

namespace
{
// ref: ASMC.cpp:102-128 — ids of the form "<IID>#1" / "<IID>#2"
std::pair<std::vector<unsigned long>, std::vector<unsigned long>> hapIndicesOfIds(const Data& data, const std::vector<std::string>& hapIdsA,
                                                                                  const std::vector<std::string>& hapIdsB)
{
  if (hapIdsA.size() != hapIdsB.size()) {
    throw std::runtime_error("Vector of A IDs (" + std::to_string(hapIdsA.size()) +
                             ") must be the same size as vector of B IDs (" + std::to_string(hapIdsB.size()) + ").\n");
  }
  std::vector<unsigned long> a(hapIdsA.size()), b(hapIdsB.size());
  for (size_t i = 0; i < hapIdsA.size(); ++i) {
    const auto [idA, hapA] = asmc::combinedIdToIndPlusHap(hapIdsA[i]);
    const auto [idB, hapB] = asmc::combinedIdToIndPlusHap(hapIdsB[i]);
    a[i] = asmc::dipToHapId(asmc::getIndIdxFromIdString(data.IIDList, idA), hapA);
    b[i] = asmc::dipToHapId(asmc::getIndIdxFromIdString(data.IIDList, idB), hapB);
  }
  return {a, b};
}
}  // namespace

void ASMC::ASMC::decodePairs(const std::vector<std::string>& hapIdsA, const std::vector<std::string>& hapIdsB,
                             bool perPairPosteriors, bool sumOfPosteriors, bool perPairPosteriorMeans, bool perPairMAPs)
{
  const auto [a, b] = hapIndicesOfIds(mData, hapIdsA, hapIdsB);
  decodePairs(a, b, perPairPosteriors, sumOfPosteriors, perPairPosteriorMeans, perPairMAPs);
}

ASMC::ASMC::PairIndices ASMC::ASMC::decodePairsToDevice(const std::vector<unsigned long>& hapIndicesA,
                                                        const std::vector<unsigned long>& hapIndicesB, const HMM::DeviceOutputs& out)
{
  if (hapIndicesA.empty() || hapIndicesA.size() != hapIndicesB.size()) {
    throw std::runtime_error("Vector of A indices (" + std::to_string(hapIndicesA.size()) +
                             ") must be the same size as vector of B indices (" + std::to_string(hapIndicesB.size()) +
                             ").\n");
  }
  PairIndices indices(hapIndicesA.size());
  const unsigned long numHaps = mData.numLoadedHaplotypes();
  for (size_t i = 0; i < hapIndicesA.size(); ++i) {
    const unsigned long a = hapIndicesA[i], b = hapIndicesB[i];
    if (a >= numHaps || b >= numHaps) {
      throw std::runtime_error("haplotype index out of range");
    }
    indices[i] = std::make_tuple(a, asmc::indPlusHapToCombinedId(mData.IIDList.at(a / 2), 1 + a % 2), b,
                                 asmc::indPlusHapToCombinedId(mData.IIDList.at(b / 2), 1 + b % 2));
  }
  mHmm.decodeHapPairsToDevice(hapIndicesA, hapIndicesB, out);
  return indices;
}

ASMC::ASMC::PairIndices ASMC::ASMC::decodePairsToDevice(const std::vector<std::string>& hapIdsA, const std::vector<std::string>& hapIdsB,
                                                        const HMM::DeviceOutputs& out)
{
  const auto [a, b] = hapIndicesOfIds(mData, hapIdsA, hapIdsB);
  return decodePairsToDevice(a, b, out);
}

DecodePairsReturnStruct ASMC::ASMC::getCopyOfResults()
{
  return mHmm.getDecodePairsReturnStruct();
}

const DecodePairsReturnStruct& ASMC::ASMC::getRefOfResults()
{
  return mHmm.getDecodePairsReturnStruct();
}
