// fastsmc_b200 host layer — FastSMC facade with the reference's interface (ref: ASMC_SRC/SRC/FastSMC.hpp:42-53).
#pragma once

#include <string>
#include <vector>

#include "../../../include/fastsmc_b200.h"
#include "Data.hpp"
#include "DecodingParams.hpp"
#include "HMM.hpp"

namespace ASMC
{

class FastSMC
{
  DecodingParams mParams;
  Data mData;
  HMM mHmm;

public:
  explicit FastSMC(DecodingParams params);
  FastSMC(const std::string& inFileRoot, const std::string& outFileRoot);
  /// B200 build: run on data already in memory (synthetic workloads)
  FastSMC(DecodingParams params, Data data);

  /// Seeding (when hashing is on) -> batched decoding -> IBD segments written to
  /// <outFileRoot>.<jobInd>.<jobs>.FastSMC.{ibd,bibd}.gz (ref: FastSMC.cpp:41-238).
  void run();
  /// What run() does, with the segments left on the device (HMM::setDeviceSegments) instead of written to a file: same
  /// seeding, candidate order, chunks and records, in the file's order.  HMM::moveDeviceSegments hands them over.
  void runDeviceSegments();

  // ---- B200 build: introspection -------------------------------------------------------------------------------
  struct SeedingStats {
    fsmc_seed_stats device{};
    double seedWallS = 0.0;   // fsmc_seed call
    double orderWallS = 0.0;  // reference candidate order: device passes inside fsmc_seed, or the host replay (FSMC_HOST_ORDER)
    double submitWallS = 0.0; // decodeFromHashing calls of the ordered candidates (batching + decode submission)
    unsigned long candidates = 0;
  };
  const SeedingStats& getSeedingStats() const { return mSeedStats; }
  /// candidates handed to the HMM in the last run: (hapA, hapB, fromSite, toSite) in decodeFromHashing call order
  const std::vector<fsmc_match>& getCandidates() const { return mCandidates; }
  void setKeepCandidates(bool keep) { mKeepCandidates = keep; }
  HMM& hmm() { return mHmm; }
  const Data& data() const { return mData; }
  double getRunWallSeconds() const { return mRunWallS; }

private:
  SeedingStats mSeedStats;
  std::vector<fsmc_match> mCandidates;
  bool mKeepCandidates = false;
  double mRunWallS = 0.0;
  void seedAndDecode();
};

}  // namespace ASMC
