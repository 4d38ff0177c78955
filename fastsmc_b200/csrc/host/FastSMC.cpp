// fastsmc_b200 host layer — see FastSMC.hpp.
#include "FastSMC.hpp"

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <iostream>
#include <stdexcept>

#include "CandidateOrder.hpp"
#include "HmmUtils.hpp"

namespace
{
double now()
{
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}
}  // namespace

ASMC::FastSMC::FastSMC(DecodingParams params) : mParams{std::move(params)}, mData{mParams}, mHmm{mData, mParams} {}

ASMC::FastSMC::FastSMC(const std::string& inFileRoot, const std::string& outFileRoot)
    : mParams{inFileRoot, inFileRoot + ".decodingQuantities.gz", outFileRoot, true}, mData{mParams},
      mHmm{mData, mParams}
{
}

ASMC::FastSMC::FastSMC(DecodingParams params, Data data)
    : mParams{std::move(params)}, mData{std::move(data)}, mHmm{mData, mParams}
{
}

void ASMC::FastSMC::run()
{
  const double t0 = now();
  mHmm.decodeAll(mParams.jobs, mParams.jobInd);
  if (!mParams.hashing) {
    mHmm.closeIBDFile();  // ref: FastSMC.cpp:48-51
  } else {
    seedAndDecode();
  }
  mRunWallS = now() - t0;
  std::cout << "Inference done in " << mRunWallS << " seconds; " << mHmm.getNumberOfDetectedSegments()
            << " IBD segments detected." << std::endl;
}

void ASMC::FastSMC::runDeviceSegments()
{
  mHmm.setDeviceSegments(true);
  run();
}

// ref: FastSMC.cpp:53-235.  The reference streams the haps file a second time, filling a ring of 64-SNP words per
// haplotype and updating two hash maps word by word.  Here the packed haplotypes are already on the device; one
// fsmc_seed call returns every match interval of the job.
void ASMC::FastSMC::seedAndDecode()
{
  if (mParams.hashingWordSize != 64) {
    throw std::runtime_error("only 64-SNP hashing words are supported");
  }
  if (mParams.min_maf != 0.f || !mParams.haploid) {
    throw std::runtime_error("the B200 build does not support min_maf > 0 or diploid hashing "
                             "(gap, min_m, skip and max_seeds are free)");
  }
  if (mParams.max_seeds < 0) {
    throw std::runtime_error("max_seeds must be >= 0");
  }
  if (mParams.max_seeds > 0 && mParams.referenceCandidateOrder && std::getenv("FSMC_HOST_ORDER") != nullptr) {
    throw std::runtime_error("max_seeds > 0 needs the device candidate order (unset FSMC_HOST_ORDER)");
  }
  if (mParams.skip > 0.f && mParams.referenceCandidateOrder && std::getenv("FSMC_HOST_ORDER") != nullptr) {
    throw std::runtime_error("skip > 0 needs the device candidate order (unset FSMC_HOST_ORDER)");
  }
  const uint32_t H = static_cast<uint32_t>(mData.numLoadedHaplotypes());
  const int W = mData.sites / 64;
  const bool lastJob = mParams.jobInd == mParams.jobs;
  fsmc_seed_params sp{};
  sp.gap = mParams.gap;
  sp.minLengthCm = mParams.min_m;
  sp.geneticPositions = mData.geneticPositions.data();
  sp.globalHapId = mData.globalHapId.data();
  sp.loI = (mData.w_i - 1) * mData.windowSize;
  sp.hiI = mData.w_i * mData.windowSize;
  sp.loJ = (mData.w_j - 1) * mData.windowSize;
  sp.hiJ = mData.w_j * mData.windowSize;
  sp.lastJob = lastJob;
  sp.aboveDiag = mData.is_j_above_diag;
  // Reference candidate order (the default): computed on the device inside fsmc_seed, which then returns the candidates
  // only, in decodeFromHashing call order.  FSMC_HOST_ORDER=1 selects the round-1 host replay of the same order
  // (CandidateOrder.hpp; development / A-B checks): every interval comes back and is replayed on the host threads.
  static const bool hostOrder = std::getenv("FSMC_HOST_ORDER") != nullptr;
  const bool deviceOrder = mParams.referenceCandidateOrder && !hostOrder;
  sp.flipMask = mData.flipMask.data();
  sp.skip = mParams.skip;
  sp.maxSeeds = mParams.max_seeds;
  sp.readAhead = mParams.constReadAhead;
  sp.flags = deviceOrder ? FSMC_SEED_REFERENCE_ORDER
                         : (mParams.referenceCandidateOrder ? (FSMC_SEED_ALL_INTERVALS | FSMC_SEED_UNSORTED) : 0u);

  // not zero-filled: at biobank density the intervals are gigabytes, written once by the copy from the device
  candidate_order::RawArray<fsmc_match> buffer(std::max<size_t>(1u << 16, static_cast<size_t>(H) * 8));
  const double t0 = now();
  for (;;) {
    const int rc =
        fsmc_seed(mHmm.context(), &sp, buffer.data(), static_cast<int64_t>(buffer.size()), &mSeedStats.device);
    if (rc == FSMC_E_OVERFLOW) {
      buffer.reset(static_cast<size_t>(mSeedStats.device.numMatches) + 1024);
      continue;
    }
    if (rc != FSMC_OK) {
      throw std::runtime_error(std::string("fsmc_seed: ") + fsmc_last_error());
    }
    break;
  }
  struct Found {  // the filled part of the buffer
    const fsmc_match* p;
    size_t n;
    size_t size() const { return n; }
    const fsmc_match& operator[](const size_t i) const { return p[i]; }
  } const found{buffer.data(), static_cast<size_t>(mSeedStats.device.numMatches)};
  mSeedStats.seedWallS = now() - t0;

  mCandidates.clear();
  mSeedStats.candidates = 0;
  auto submit = [&](const fsmc_match& m) {
    // ref: HASHING/Match.hpp:46-51 — sites [64*start, 64*end + 63]
    const uint32_t from = static_cast<uint32_t>(m.startWord) * 64u, to = static_cast<uint32_t>(m.endWord) * 64u + 63u;
    mHmm.decodeFromHashing(m.hapA, m.hapB, from, to);
    ++mSeedStats.candidates;
    if (mKeepCandidates) {
      mCandidates.push_back(fsmc_match{m.hapA, m.hapB, static_cast<int32_t>(from), static_cast<int32_t>(to)});
    }
  };
  if (!mParams.referenceCandidateOrder || deviceOrder) {
    const double t1 = now();
    for (size_t i = 0; i < found.size(); ++i) {
      submit(found[i]);
    }
    mSeedStats.submitWallS = now() - t1;
    mSeedStats.orderWallS = deviceOrder ? mSeedStats.device.orderMs / 1e3 : 0.0;
  } else {
    const double t1 = now();
    auto rawWord = [&](const uint32_t h, const int w) {
      return mData.hapBits[static_cast<size_t>(h) * mData.wordsPerHap + w] ^ mData.flipMask[w];
    };
    auto longEnough = [&](const fsmc_match& m) {
      return asmc::cmBetween(m.startWord, m.endWord, mData.geneticPositions, 64) >= static_cast<double>(mParams.min_m);
    };
    candidate_order::replayReferenceOrderFast(found, H, W, mParams.gap, rawWord, longEnough,
                                              [&](const int64_t i) { submit(found[i]); });
    mSeedStats.orderWallS = now() - t1;
  }
  mHmm.finishFromHashing();
}
