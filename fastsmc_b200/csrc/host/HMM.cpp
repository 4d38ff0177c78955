// fastsmc_b200 host layer — see HMM.hpp.
#include "HMM.hpp"

#include <algorithm>
#include <atomic>
#include <thread>
#include <mutex>
#include <deque>
#include <condition_variable>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <limits>
#include <map>
#include <stdexcept>

#include <charconv>
#include <memory>

#include "../../../include/fastsmc_b200.h"
#include "HmmUtils.hpp"
#include "OutputPipeline.hpp"

namespace
{

double now()
{
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

void check(const int rc, const char* what)
{
  if (rc != FSMC_OK) {
    throw std::runtime_error(std::string(what) + ": " + fsmc_last_error());
  }
}

// printf("%.7g") is what the reference's ostream produces for floats at precision 7 (ref: HMM.cpp:1116-1141);
// std::to_chars with chars_format::general and a precision is specified to give the same characters, several times
// faster.
void appendG7(std::string& s, const double v)
{
  char buf[48];
  buf[0] = '\t';
  const auto r = std::to_chars(buf + 1, buf + sizeof buf, v, std::chars_format::general, 7);
  s.append(buf, static_cast<size_t>(r.ptr - buf));
}

void appendInt(std::string& s, const long v)
{
  char buf[24];
  const auto r = std::to_chars(buf, buf + sizeof buf, v);
  s.append(buf, static_cast<size_t>(r.ptr - buf));
}

}  // namespace

namespace
{
// Device contexts outlive the HMM that used them: the jobs of one data set (runJobs) create one HMM after the other on the
// same device, and a context's buffers (scratch slabs, seeding tables, sort buffers: grow-only) and its stream are what
// is expensive to set up.  A released context keeps its device memory until the process ends.
class ContextPool
{
public:
  fsmc_ctx* acquire(const int device)
  {
    {
      std::lock_guard<std::mutex> g(mLock);
      auto& idle = mIdle[device];
      if (!idle.empty()) {
        fsmc_ctx* ctx = idle.back();
        idle.pop_back();
        return ctx;
      }
    }
    fsmc_ctx* ctx = nullptr;
    check(fsmc_ctx_create(device, &ctx), "fsmc_ctx_create");
    return ctx;
  }
  void release(const int device, fsmc_ctx* ctx)
  {
    if (ctx) {
      std::lock_guard<std::mutex> g(mLock);
      mIdle[device].push_back(ctx);
    }
  }

private:
  std::mutex mLock;
  std::map<int, std::vector<fsmc_ctx*>> mIdle;
};
ContextPool& contextPool()
{
  static ContextPool* pool = new ContextPool;  // never destroyed: no CUDA calls during static destruction
  return *pool;
}
}  // namespace

struct HMM::GzOut {
  OutputPipeline writer;
  std::vector<std::string> idPrefix;  // "fam\tiid\t" per individual (text output)
  explicit GzOut(const std::string& path, const int level, const unsigned threads) : writer(path, level, threads) {}
};

// The segments of one decoded chunk, shared by the formatting tasks of the output pipeline.
struct HMM::SegmentBlock {
  std::vector<Pending> pend;         // the chunk's pairs
  std::vector<uint32_t> firstPair;   // tile -> index of its lane 0 in pend
  std::unique_ptr<fsmc_segment[]> seg;
  size_t count = 0;
};

HMM::HMM(Data _data, const DecodingParams& _decodingParams, int /*_scalingSkip*/)
    : data(std::move(_data)), m_decodingQuant(DecodingQuantities::cached(_decodingParams.decodingQuantFile)),
      decodingParams(_decodingParams)
{
  if (decodingParams.decodingSequence) {
    throw std::runtime_error("sequence mode is not supported by the B200 build (array mode only)");
  }
  if (!decodingParams.expectedCoalTimesFile.empty()) {
    // ref: HMM.cpp updateOutputStructures / readExpectedTimesFromIntervalsFile — not implemented: fail instead of silently
    // using the decoding quantities' expected times
    throw std::runtime_error("expectedCoalTimesFile is not supported by the B200 build (expected times come from the decoding quantities)");
  }
  m_batchSize = decodingParams.batchSize;
  sequenceLength = data.sites;
  const double tTables = now();
  {
    // The tables depend on the whole data set (allele counts, positions), the decoding quantities and a few options, not on
    // the job's sample subset: the jobs cut out of one data set build them once (Data::sharedObject) and pooled device
    // contexts that already hold them skip the upload (fsmc_model::modelTag).
    struct SharedModel {
      ModelTables tables;
      uint64_t tag = 0;
    };
    char opts[96];
    std::snprintf(opts, sizeof opts, "|%d%d%d%d|%.9g|%d|%d", int(decodingParams.foldData), int(decodingParams.usingCSFS),
                  int(decodingParams.decodingSequence), int(decodingParams.noConditionalAgeEstimates),
                  static_cast<double>(decodingParams.skipCSFSdistance), decodingParams.time, int(decodingParams.useKnownSeed));
    const std::string key = "HMM::ModelTables|" + decodingParams.decodingQuantFile + opts;
    const std::shared_ptr<const void> obj = data.sharedObject(key, [&]() -> std::shared_ptr<const void> {
      static std::atomic<uint64_t> nextTag{1};
      auto sm = std::make_shared<SharedModel>();
      sm->tables = buildModelTables(data, m_decodingQuant, decodingParams);
      sm->tag = nextTag++;
      return sm;
    });
    const SharedModel& sm = *static_cast<const SharedModel*>(obj.get());
    m_model = sm.tables;
    m_modelTag = sm.tag;
  }
  m_stats.tablesWallS = now() - tTables;
  stateThreshold = static_cast<unsigned>(m_model.stateThreshold);
  ageThreshold = static_cast<unsigned>(m_model.ageThreshold);
  probabilityThreshold = m_model.probabilityThreshold;
  m_decodingReturnValues.sites = data.sites;
  m_decodingReturnValues.states = m_decodingQuant.states;
  m_decodingReturnValues.siteWasFlippedDuringFolding = data.siteWasFlippedDuringFolding;
  // ref: HMM.cpp:271-279
  if (decodingParams.doPosteriorSums) {
    m_decodingReturnValues.sumOverPairs.resize(data.sites, m_decodingQuant.states);
  }
  if (decodingParams.doMajorMinorPosteriorSums) {
    m_decodingReturnValues.sumOverPairs00.resize(data.sites, m_decodingQuant.states);
    m_decodingReturnValues.sumOverPairs01.resize(data.sites, m_decodingQuant.states);
    m_decodingReturnValues.sumOverPairs11.resize(data.sites, m_decodingQuant.states);
  }
  // 8192 reference batches per kernel launch keep every SM busy; batch composition is unaffected because chunks
  // are cut at multiples of the batch size
  m_flushPairs = static_cast<size_t>(m_batchSize) * 8192;
  if (const char* e = std::getenv("FSMC_FLUSH_BATCHES")) {  // development: reference batches per decode call
    m_flushPairs = static_cast<size_t>(m_batchSize) * static_cast<size_t>(std::max(1, std::atoi(e)));
    m_perSiteChunkCap = m_flushPairs;
  }
  const double tUpload = now();
  uploadModel();
  m_stats.uploadWallS = now() - tUpload;
}

// ref: HMM.cpp:504-513
unsigned int HMM::getStateThreshold()
{
  unsigned int result = 0u;
  const std::vector<float>& disc = m_decodingQuant.discretization;
  while (disc[result] < static_cast<float>(decodingParams.time) && result < m_decodingQuant.states) {
    ++result;
  }
  return result;
}

// ref: HMM.cpp:159-256 (array mode).  Three tables e1, e0-e1, e2-e0 per site and state.
HMM::ModelTables HMM::buildModelTables(const Data& data, const DecodingQuantities& dq, const DecodingParams& decodingParams)
{
  ModelTables m_model;
  const int S = static_cast<int>(dq.states);
  const int L = data.sites;
  constexpr int precision = 2;
  constexpr float minGenetic = 1e-10f;
  m_model.states = S;
  m_model.sites = L;
  m_model.emission1.assign(static_cast<size_t>(L) * S, 0.f);
  m_model.emission0minus1.assign(static_cast<size_t>(L) * S, 0.f);
  m_model.emission2minus0.assign(static_cast<size_t>(L) * S, 0.f);

  std::vector<std::vector<int>> undist;
  if (decodingParams.usingCSFS) {
    undist = data.calculateUndistinguishedCounts(dq.CSFSSamples);
  }
  std::vector<uint8_t> useCsfs(L, 0);
  if (decodingParams.skipCSFSdistance < std::numeric_limits<float>::infinity() && L > 0) {
    useCsfs[0] = 1;
    float last = 0.f;
    for (int pos = 1; pos < L; ++pos) {
      if (data.geneticPositions[pos] - last >= decodingParams.skipCSFSdistance) {
        useCsfs[pos] = 1;
        last = data.geneticPositions[pos];
      }
    }
  }
  for (int pos = 0; pos < L; ++pos) {
    float* o1 = &m_model.emission1[static_cast<size_t>(pos) * S];
    float* o0 = &m_model.emission0minus1[static_cast<size_t>(pos) * S];
    float* o2 = &m_model.emission2minus0[static_cast<size_t>(pos) * S];
    if (!useCsfs[pos]) {
      const auto& T = decodingParams.decodingSequence ? dq.classicEmissionTable : dq.compressedEmissionTable;
      for (int k = 0; k < S; ++k) {
        o1[k] = T[1][k];
        o0[k] = T[0][k] - T[1][k];
        o2[k] = 0.f;
      }
      continue;
    }
    const int u0 = undist[pos][0], u1 = undist[pos][1], u2 = undist[pos][2];
    if (decodingParams.foldData) {
      const auto& T = dq.foldedAscertainedCSFSmap;
      for (int k = 0; k < S; ++k) {
        o1[k] = (u1 >= 0) ? T.at(u1)[1][k] : 0.f;
        o0[k] = T.at(u0)[0][k] - o1[k];
        o2[k] = (u2 >= 0) ? (T.at(u2)[0][k] - T.at(u0)[0][k]) : (0 - T.at(u0)[0][k]);
      }
    } else {
      const auto& T = dq.ascertainedCSFSmap;
      for (int k = 0; k < S; ++k) {
        o1[k] = (u1 >= 0) ? T.at(u1)[1][k] : 0.f;
        const float em0 = (u0 >= 0) ? T.at(u0)[0][k] : 0.f;
        o0[k] = em0 - o1[k];
        if (u2 >= 0) {
          const bool mono = (u2 == dq.CSFSSamples - 2);  // monomorphic derived is read from CSFS[0][0]
          o2[k] = T.at(mono ? 0 : u2)[mono ? 0 : 2][k] - em0;
        } else {
          o2[k] = 0 - em0;
        }
      }
    }
  }

  // The reference looks transition vectors up by exact float key at every site of every batch
  // (ref: HMM.cpp:753-756, 795-797, 907-909, 951-954).  Distances depend only on the site, so the key of every gap is
  // resolved once here and the distinct rows are packed densely for the device.
  std::map<float, int> rowOf;
  m_model.distanceRow.assign(L, 0);
  std::vector<float> keys;
  for (int pos = 1; pos < L; ++pos) {
    const float key =
        asmc::roundMorgans(data.geneticPositions[pos] - data.geneticPositions[pos - 1], precision, minGenetic);
    auto it = rowOf.find(key);
    if (it == rowOf.end()) {
      it = rowOf.emplace(key, static_cast<int>(keys.size())).first;
      keys.push_back(key);
    }
    m_model.distanceRow[pos] = it->second;
  }
  if (keys.empty()) {
    keys.push_back(minGenetic);
  }
  m_model.numDistances = static_cast<int>(keys.size());
  auto gather = [&](const std::unordered_map<float, std::vector<float>>& table, std::vector<float>& out) {
    out.assign(static_cast<size_t>(keys.size()) * S, 0.f);
    for (size_t r = 0; r < keys.size(); ++r) {
      const auto& row = table.at(keys[r]);  // throws std::out_of_range like the reference's .at()
      std::copy(row.begin(), row.begin() + S, out.begin() + r * S);
    }
  };
  gather(dq.Dvectors, m_model.D);
  gather(dq.Bvectors, m_model.B);
  gather(dq.Uvectors, m_model.U);
  gather(dq.rowRatioVectors, m_model.RR);
  // ref: HMM.cpp:504-513, 93-105
  unsigned st = 0u;
  while (dq.discretization[st] < static_cast<float>(decodingParams.time) && st < dq.states) {
    ++st;
  }
  float pT = 0.f;
  for (unsigned i = 0; i < st; ++i) {
    pT += dq.initialStateProb.at(i);
  }
  m_model.stateThreshold = static_cast<int>(st);
  m_model.ageThreshold = decodingParams.noConditionalAgeEstimates ? S : static_cast<int>(st);
  m_model.probabilityThreshold = pT;
  return m_model;
}

void HMM::uploadModel()
{
  uploadModelTo(m_ctx);
}

void HMM::uploadModelTo(fsmc_ctx*& ctx)
{
  fsmc_ctx*& m_ctx = ctx;  // the body below fills whichever context it is given
  m_ctx = contextPool().acquire(decodingParams.device);
  fsmc_model m{};
  m.states = m_model.states;
  m.sites = m_model.sites;
  m.initialStateProb = m_decodingQuant.initialStateProb.data();
  m.expectedTimes = m_decodingQuant.expectedTimes.data();
  m.columnRatios = m_decodingQuant.columnRatios.data();
  m.emission1 = m_model.emission1.data();
  m.emission0minus1 = m_model.emission0minus1.data();
  m.emission2minus0 = m_model.emission2minus0.data();
  m.numDistances = m_model.numDistances;
  m.D = m_model.D.data();
  m.B = m_model.B.data();
  m.U = m_model.U.data();
  m.RR = m_model.RR.data();
  m.distanceRow = m_model.distanceRow.data();
  m.stateThreshold = m_model.stateThreshold;
  m.ageThreshold = m_model.ageThreshold;
  m.probabilityThreshold = m_model.probabilityThreshold;
  m.modelTag = m_modelTag;
  check(fsmc_set_model(m_ctx, &m), "fsmc_set_model");
  check(fsmc_set_haplotypes(m_ctx, data.hapBits.data(), static_cast<int64_t>(data.numLoadedHaplotypes()), data.sites),
        "fsmc_set_haplotypes");
}

// ref: HMM.cpp:129-157
PairObservations HMM::makePairObs(int_least8_t iHap, unsigned int ind1, int_least8_t jHap, unsigned int ind2,
                                  const bool materialise)
{
  PairObservations p;
  p.iHap = iHap;
  p.jHap = jHap;
  p.iInd = ind1;
  p.jInd = ind2;
  if (materialise) {
    const unsigned long a = asmc::dipToHapId(ind1, iHap), b = asmc::dipToHapId(ind2, jHap);
    p.obsBits.resize(data.sites);
    p.homMinorBits.resize(data.sites);
    for (int s = 0; s < data.sites; ++s) {
      const bool x = data.allele(a, s), y = data.allele(b, s);
      p.obsBits[s] = x != y;
      p.homMinorBits[s] = x && y;
    }
  }
  return p;
}

// ref: HMM.cpp:296-303, 383-401
void HMM::openOutput(const int jobs, const int jobInd)
{
  const std::string path = decodingParams.outFileRoot + "." + std::to_string(jobInd) + "." + std::to_string(jobs) +
                           (decodingParams.BIN_OUT ? ".FastSMC.bibd.gz" : ".FastSMC.ibd.gz");
  m_out = std::make_unique<GzOut>(path, decodingParams.outputCompressionLevel,
                                  static_cast<unsigned>(std::max(0, decodingParams.outputThreads)));
  if (!decodingParams.BIN_OUT) {
    m_out->idPrefix.reserve(data.FamIDList.size());
    for (size_t i = 0; i < data.FamIDList.size(); ++i) {
      m_out->idPrefix.push_back(data.FamIDList[i] + '\t' + data.IIDList[i] + '\t');
    }
  }
  if (decodingParams.BIN_OUT) {
    auto& w = m_out->writer;
    w.write(&decodingParams.outputIbdSegmentLength, sizeof(bool));
    w.write(&decodingParams.doPerPairPosteriorMean, sizeof(bool));
    w.write(&decodingParams.doPerPairMAP, sizeof(bool));
    w.write(&data.chrNumber, sizeof(int));
    const unsigned nInd = static_cast<unsigned>(data.FamIDList.size());
    w.write(&nInd, sizeof(unsigned));
    for (unsigned i = 0; i < nInd; ++i) {
      unsigned len = static_cast<unsigned>(data.FamIDList[i].size());
      w.write(&len, sizeof(unsigned));
      w.write(data.FamIDList[i].data(), len);
      len = static_cast<unsigned>(data.IIDList[i].size());
      w.write(&len, sizeof(unsigned));
      w.write(data.IIDList[i].data(), len);
    }
  }
}

// ref: HMM.cpp:283-381
void HMM::decodeAll(const int jobs, const int jobInd)
{
  if (decodingParams.FastSMC) {
    openOutput(jobs, jobInd);
    if (decodingParams.hashing) {
      return;
    }
  }
  const uint64_t N = data.numLoadedIndividuals();
  const uint64_t totPairs = decodingParams.withinOnly ? N : 2 * N * N - N;
  const uint64_t lo = totPairs * static_cast<uint64_t>(jobInd - 1) / static_cast<uint64_t>(jobs);
  const uint64_t hi = totPairs * static_cast<uint64_t>(jobInd) / static_cast<uint64_t>(jobs);
  m_windowed = false;
  uint64_t idx = 0;
  const uint32_t L = static_cast<uint32_t>(data.sites);
  auto submit = [&](const uint32_t a, const uint32_t b) {
    if (lo <= idx && idx < hi) {
      m_pending.push_back(Pending{a, b, 0u, L});
      if (m_pending.size() >= m_flushPairs) {
        flushPending(false);
      }
    }
    ++idx;
  };
  // enumeration order of the reference: for i, for j < i, for iHap, for jHap: (jHap of j, iHap of i); then the
  // pair within individual i (ref: HMM.cpp:325-357)
  for (uint32_t i = 0; i < N && idx < hi; ++i) {
    if (!decodingParams.withinOnly) {
      if (idx + 4ull * i <= lo) {
        idx += 4ull * i;  // the whole row lies before the job's slice
      } else {
        for (uint32_t j = 0; j < i; ++j) {
          for (uint32_t ih = 0; ih < 2; ++ih) {
            for (uint32_t jh = 0; jh < 2; ++jh) {
              submit(2 * j + jh, 2 * i + ih);
            }
          }
        }
      }
    }
    submit(2 * i, 2 * i + 1);
  }
  finishDecoding();  // ref: HMM.cpp:359 (runLastBatch)
}

// ref: HMM.cpp:470-502
void HMM::decodeFromHashing(const unsigned int i, const unsigned int j, const unsigned int fromPosition,
                            const unsigned int toPosition)
{
  m_windowed = true;
  m_pending.push_back(Pending{i, j, fromPosition, toPosition});
  ++cpt;
  if (m_pending.size() >= m_flushPairs) {
    flushPending(false);
  }
}

void HMM::decodePair(const unsigned int i, const unsigned int j)
{
  // ref: HMM.cpp:413-440
  if (i != j) {
    for (uint32_t ih = 0; ih < 2; ++ih) {
      for (uint32_t jh = 0; jh < 2; ++jh) {
        decodeHapPair(2ul * i + ih, 2ul * j + jh);
      }
    }
  } else {
    decodeHapPair(2ul * i, 2ul * i + 1);
  }
}

void HMM::decodePairs(const std::vector<unsigned int>& individualsA, const std::vector<unsigned int>& individualsB)
{
  if (individualsA.size() != individualsB.size()) {
    throw std::runtime_error("vector of A indicies must be the same size as vector of B indicies");
  }
  for (size_t i = 0; i < individualsA.size(); ++i) {
    decodePair(individualsA[i], individualsB[i]);
  }
}

// ref: HMM.cpp:442-457
void HMM::decodeHapPair(const unsigned long i, const unsigned long j)
{
  const unsigned long numHaps = data.numLoadedHaplotypes();
  if (i >= numHaps || j >= numHaps) {
    throw std::runtime_error("haplotype index out of range");
  }
  m_windowed = false;
  const auto [iInd, iHap] = asmc::hapToDipId(i);
  const auto [jInd, jHap] = asmc::hapToDipId(j);
  m_observationsBatch.push_back(makePairObs(static_cast<int_least8_t>(iHap), static_cast<unsigned>(iInd),
                                            static_cast<int_least8_t>(jHap), static_cast<unsigned>(jInd)));
  if (static_cast<int>(m_observationsBatch.size()) == m_batchSize) {
    m_observationsBatch.clear();  // the reference's buffer empties when a batch is decoded (ref: HMM.cpp:589)
  }
  m_pendingRow.push_back(m_deviceOut ? m_deviceRowsQueued++ : m_decodePairsReturnStruct.getNumWritten() + m_pending.size());
  m_pending.push_back(Pending{static_cast<uint32_t>(i), static_cast<uint32_t>(j), 0u, static_cast<uint32_t>(data.sites)});
  // per-site outputs are pairs x sites floats: keep chunks small enough for host and device buffers
  // (full posterior matrices are states times larger)
  const size_t perPairFloats = std::max<size_t>(1, static_cast<size_t>(data.sites)) *
                               ((m_deviceOut ? m_deviceOut->perPairPosteriors != nullptr : m_storePerPairPosterior)
                                   ? static_cast<size_t>(m_decodingQuant.states) + 2
                                   : 2);
  size_t perSiteChunk = std::max<size_t>(static_cast<size_t>(m_batchSize),
                                         (size_t{1} << 29) / perPairFloats / m_batchSize * m_batchSize);
  if (m_perSiteChunkCap > 0) {
    perSiteChunk = std::min(perSiteChunk, m_perSiteChunkCap);
  }
  if (!decodingParams.FastSMC && m_pending.size() >= perSiteChunk) {
    flushPending(false);
  }
}

void HMM::decodeHapPairs(const std::vector<unsigned long>& hapsA, const std::vector<unsigned long>& hapsB)
{
  if (hapsA.size() != hapsB.size()) {
    throw std::runtime_error("vector of A indices must be the same size as vector of B indices");
  }
  m_pendingRow.clear();
  for (size_t i = 0; i < hapsA.size(); ++i) {
    decodeHapPair(hapsA[i], hapsB[i]);
  }
}

void HMM::finishDecoding()
{
  flushPending(true);
  drainDecodes();
  m_observationsBatch.clear();
}

void HMM::closeIBDFile()
{
  drainDecodes();
  if (m_out) {
    const double t0 = now();
    m_out->writer.close();
    m_stats.outputWallS += now() - t0;
    m_out.reset();
  }
}

void HMM::finishFromHashing()
{
  flushPending(true);
  drainDecodes();
  closeIBDFile();
}

// Decodes the pending pairs in whole reference batches (all of them when `all`).
void HMM::flushPending(const bool all)
{
  const size_t bs = static_cast<size_t>(m_batchSize);
  size_t n = all ? m_pending.size() : m_pending.size() / bs * bs;
  if (n == 0) {
    return;
  }
  const bool segments = decodingParams.FastSMC;
  const bool store = m_storePerPairPosteriorMean || m_storePerPairMAP || m_storePerPairPosterior || m_storeSumOfPosterior;
  if (segments) {
    runSegmentChunk(m_pending.data(), n);
  } else if (m_deviceOut) {
    runDeviceChunk(m_pending.data(), m_pendingRow.data(), n);
  } else {
    // ref: HMM.cpp:570-581 (addToBatch) — the sums over pairs and the per-pair outputs are independent consumers of the
    // same batch: both run when both are asked for
    if (store) {
      if (m_pendingRow.size() < n) {
        // pairs queued by decodeAll / decodePair while the store flags of an earlier ASMC::decodePairs are still set: the
        // return structure has no rows for them (the reference throws std::out_of_range from its .at() here)
        throw std::out_of_range("HMM: per-pair outputs are stored but the return structure was not initialised for these pairs");
      }
      runPerSiteChunk(m_pending.data(), m_pendingRow.data(), n);
    }
    if (decodingParams.doPosteriorSums || decodingParams.doMajorMinorPosteriorSums) {
      runPosteriorSumChunk(m_pending.data(), n);
    }
  }
  m_pendingRow.erase(m_pendingRow.begin(), m_pendingRow.begin() + static_cast<long>(std::min(n, m_pendingRow.size())));
  m_pending.erase(m_pending.begin(), m_pending.begin() + n);
}

namespace
{

// Tiles of one chunk: a reference batch of batchSize consecutive pairs shares one decode window and one scan
// window (ref: HMM.cpp:561-565, 1199-1204); batches wider than a warp become several tiles with the same windows.
struct TileSet {
  std::vector<uint32_t> hapA, hapB;
  std::vector<int32_t> pairs, from, to, scanFrom, scanTo;
  std::vector<uint32_t> firstPair;  // index into the chunk of lane 0 of each tile
};

template <class P>
TileSet buildTiles(const P* pend, const size_t n, const size_t batchSize, const bool windowed,
                   const std::vector<float>& gen, const int sites)
{
  TileSet t;
  for (size_t b0 = 0; b0 < n; b0 += batchSize) {
    const size_t b1 = std::min(n, b0 + batchSize);
    uint32_t lo = 0, hi = static_cast<uint32_t>(sites);
    if (windowed) {
      lo = std::numeric_limits<uint32_t>::max();
      hi = 0;
      for (size_t i = b0; i < b1; ++i) {
        lo = std::min(lo, pend[i].from);
        hi = std::max(hi, pend[i].to);
      }
    }
    const int from = static_cast<int>(asmc::getFromPosition(gen, lo));
    const int to = static_cast<int>(asmc::getToPosition(gen, hi));
    for (size_t s = b0; s < b1; s += FSMC_TILE) {
      const size_t e = std::min(b1, s + FSMC_TILE);
      const size_t base = t.hapA.size();
      t.hapA.resize(base + FSMC_TILE, 0u);
      t.hapB.resize(base + FSMC_TILE, 0u);
      for (size_t i = s; i < e; ++i) {
        t.hapA[base + (i - s)] = pend[i].hapA;
        t.hapB[base + (i - s)] = pend[i].hapB;
      }
      t.pairs.push_back(static_cast<int32_t>(e - s));
      t.from.push_back(from);
      t.to.push_back(to);
      t.scanFrom.push_back(static_cast<int32_t>(lo));
      t.scanTo.push_back(static_cast<int32_t>(hi));
      t.firstPair.push_back(static_cast<uint32_t>(s));
    }
  }
  return t;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------------
// Segment decoding is pipelined: the caller's thread (candidate order replay, pair enumeration) only cuts chunks and
// builds their tiles; decode workers, each with its own fsmc_ctx and stream, run fsmc_decode and hand the records to
// the output pipeline.  With two workers the host side of one chunk (copies, record checks, formatting hand-over)
// overlaps the kernel of the next.  Chunks complete strictly in submission order, so files and statistics are the
// same as with one synchronous call per chunk.  Two contexts are only used when the request runs the narrow kernel:
// the full-beta kernels size their scratch for the whole GPU.
// ---------------------------------------------------------------------------------------------------------------
struct HMM::ChunkJob {
  size_t seq = 0;
  TileSet tiles;
  std::vector<Pending> pend;
  std::shared_ptr<SegmentBlock> block;
  fsmc_decode_stats st{};
  double decodeWallS = 0.0;
};

struct HMM::DecodePipeline {
  std::mutex mutex;
  std::condition_variable cv;
  std::deque<std::unique_ptr<ChunkJob>> queue;
  size_t submitted = 0, completed = 0;
  bool stop = false;
  std::exception_ptr error;
  std::vector<std::thread> workers;
};

HMM::~HMM()
{
  if (m_pipeline) {
    {
      std::unique_lock<std::mutex> lock(m_pipeline->mutex);
      m_pipeline->cv.wait(lock, [&] { return m_pipeline->completed == m_pipeline->submitted; });
      m_pipeline->stop = true;
    }
    m_pipeline->cv.notify_all();
    for (auto& w : m_pipeline->workers) {
      w.join();
    }
  }
  contextPool().release(decodingParams.device, m_ctx2);
  contextPool().release(decodingParams.device, m_ctx);
}

void HMM::startDecodeWorkers()
{
  m_pipeline = std::make_unique<DecodePipeline>();
  const bool ages = decodingParams.doPerPairPosteriorMean || decodingParams.doPerPairMAP;
  // Two contexts only when the device layer says the request's kernel keeps its scratch small (narrow records): the
  // full-beta kernels and the checkpointed path size theirs from the free device memory, one context per device.
  fsmc_kernel_info info{};
  check(fsmc_query_kernel(m_ctx, FSMC_CALL_SEGMENTS | (ages ? FSMC_SEG_AGE : 0u) | (decodingParams.exactArithmetic ? FSMC_EXACT : 0u),
                          m_windowed ? 0.0 : static_cast<double>(data.sites), &info),
        "fsmc_query_kernel");
  int workers = info.largeScratch ? 1 : 2;
  if (const char* e = std::getenv("FSMC_DECODE_WORKERS")) {  // development / A-B runs
    workers = std::max(1, std::min(2, std::atoi(e)));
  }
  if (workers == 2) {
    uploadModelTo(m_ctx2);
  }
  for (int w = 0; w < workers; ++w) {
    fsmc_ctx* ctx = w == 0 ? m_ctx : m_ctx2;
    m_pipeline->workers.emplace_back([this, ctx] {
      DecodePipeline& p = *m_pipeline;
      for (;;) {
        std::unique_ptr<ChunkJob> job;
        {
          std::unique_lock<std::mutex> lock(p.mutex);
          p.cv.wait(lock, [&] { return p.stop || !p.queue.empty(); });
          if (p.queue.empty()) {
            return;
          }
          job = std::move(p.queue.front());
          p.queue.pop_front();
        }
        std::exception_ptr err;
        try {
          decodeChunk(*job, ctx);
        } catch (...) {
          err = std::current_exception();
        }
        std::unique_lock<std::mutex> lock(p.mutex);
        p.cv.wait(lock, [&] { return p.completed == job->seq; });  // chunks complete in submission order
        if (!err && !p.error) {
          lock.unlock();
          try {
            completeChunk(*job);
          } catch (...) {
            err = std::current_exception();
          }
          lock.lock();
        }
        if (err && !p.error) {
          p.error = err;
        }
        ++p.completed;
        lock.unlock();
        p.cv.notify_all();
      }
    });
  }
}

// Waits for every submitted chunk; rethrows the first error of a worker.
void HMM::drainDecodes()
{
  if (!m_pipeline) {
    return;
  }
  std::unique_lock<std::mutex> lock(m_pipeline->mutex);
  m_pipeline->cv.wait(lock, [&] { return m_pipeline->completed == m_pipeline->submitted; });
  if (m_pipeline->error) {
    const std::exception_ptr e = m_pipeline->error;
    m_pipeline->error = nullptr;
    std::rethrow_exception(e);
  }
}

void HMM::runSegmentChunk(const Pending* pend, const size_t n)
{
  if (!m_pipeline) {
    startDecodeWorkers();
  }
  auto job = std::make_unique<ChunkJob>();
  job->tiles = buildTiles(pend, n, static_cast<size_t>(m_batchSize), m_windowed, data.geneticPositions, data.sites);
  job->pend.assign(pend, pend + n);
  DecodePipeline& p = *m_pipeline;
  std::unique_lock<std::mutex> lock(p.mutex);
  // at most one chunk waiting behind the ones being decoded: bounds memory, keeps every worker fed
  p.cv.wait(lock, [&] { return p.submitted - p.completed <= p.workers.size() || p.error; });
  if (p.error) {
    const std::exception_ptr e = p.error;
    p.error = nullptr;
    std::rethrow_exception(e);
  }
  job->seq = p.submitted++;
  p.queue.push_back(std::move(job));
  lock.unlock();
  p.cv.notify_all();
}

// Runs on a decode worker, any order.
void HMM::decodeChunk(ChunkJob& job, fsmc_ctx* ctx)
{
  const TileSet& t = job.tiles;
  const size_t n = job.pend.size();
  const bool ages = decodingParams.doPerPairPosteriorMean || decodingParams.doPerPairMAP;
  fsmc_decode_request req{};
  req.numTiles = static_cast<int64_t>(t.pairs.size());
  req.hapA = t.hapA.data();
  req.hapB = t.hapB.data();
  req.tilePairs = t.pairs.data();
  req.tileFrom = t.from.data();
  req.tileTo = t.to.data();
  req.tileScanFrom = t.scanFrom.data();
  req.tileScanTo = t.scanTo.data();
  req.flags = FSMC_CALL_SEGMENTS | (ages ? FSMC_SEG_AGE : 0u) | (decodingParams.exactArithmetic ? FSMC_EXACT : 0u);
  // record buffer sized from the densest chunk seen so far (a retry after FSMC_E_OVERFLOW decodes the chunk again)
  size_t capacity =
      std::max<size_t>(1024, static_cast<size_t>(static_cast<double>(n) * m_segmentsPerPair.load() * 1.5) + 1024);
  job.block = std::make_shared<SegmentBlock>();
  for (;;) {
    job.block->seg.reset(new fsmc_segment[capacity]);
    req.segments = job.block->seg.get();
    req.segmentCapacity = static_cast<int64_t>(capacity);
    const double t0 = now();
    const int rc = fsmc_decode(ctx, &req, &job.st);
    job.decodeWallS += now() - t0;
    if (rc == FSMC_E_OVERFLOW) {
      capacity = static_cast<size_t>(job.st.numSegments) + 1024;
      continue;
    }
    check(rc, "fsmc_decode");
    break;
  }
  const double perPair = static_cast<double>(job.st.numSegments) / static_cast<double>(n);
  double seen = m_segmentsPerPair.load();
  while (perPair > seen && !m_segmentsPerPair.compare_exchange_weak(seen, perPair)) {
  }
}

// Runs on a decode worker, one chunk at a time, in submission order.
void HMM::completeChunk(ChunkJob& job)
{
  const size_t n = job.pend.size();
  const fsmc_decode_stats& st = job.st;
  m_stats.decodeWallS += job.decodeWallS;
  m_stats.decodeCalls += 1;
  m_stats.pairsDecoded += n;
  m_stats.batches += (n + m_batchSize - 1) / m_batchSize;
  m_stats.pairSites += st.pairSites;
  m_stats.kernelMs += st.kernelMs;
  m_stats.deviceMs += st.totalMs;

  const double t1 = now();
  const size_t count = static_cast<size_t>(st.numSegments);
  nbSegmentsDetected += count;
  m_stats.segments += count;
  std::shared_ptr<SegmentBlock> block = job.block;
  block->count = count;
  block->pend = std::move(job.pend);
  block->firstPair = std::move(job.tiles.firstPair);
  if (m_keepSegments) {
    m_segments.reserve(m_segments.size() + count);
    for (size_t i = 0; i < count; ++i) {
      m_segments.push_back(toIbdSegment(*block, i));
    }
  }
  if (m_out && count > 0) {
    // formatting + compression happen on the pipeline's threads, in blocks that become one gzip member each
    constexpr size_t kRecordsPerTask = size_t{1} << 15;
    for (size_t lo = 0; lo < count; lo += kRecordsPerTask) {
      const size_t hi = std::min(count, lo + kRecordsPerTask);
      m_out->writer.submit([this, block, lo, hi](std::string& out) { formatSegments(*block, lo, hi, out); });
    }
  }
  m_stats.outputWallS += now() - t1;
}

IbdSegment HMM::toIbdSegment(const SegmentBlock& block, const size_t i) const
{
  const fsmc_segment& g = block.seg[i];
  const Pending& pr = block.pend[block.firstPair[g.pair / FSMC_TILE] + (g.pair % FSMC_TILE)];
  IbdSegment s;
  // first haplotype of the pair is printed first (ref: HMM.cpp:483-486, 1116-1121)
  s.ind1 = pr.hapA / 2;
  s.hap1 = 1 + static_cast<int>(pr.hapA % 2);
  s.ind2 = pr.hapB / 2;
  s.hap2 = 1 + static_cast<int>(pr.hapB % 2);
  s.posStart = g.posStart;
  s.posEnd = g.posEnd;
  s.prob = g.prob;
  s.postMean = g.postMean;
  s.mapTime = g.mapTime;
  return s;
}

// ref: HMM.cpp:1110-1177.  Runs on the output pipeline's threads; reads only immutable members.
void HMM::formatSegments(const SegmentBlock& block, const size_t lo, const size_t hi, std::string& out) const
{
  const bool bin = decodingParams.BIN_OUT;
  out.reserve(out.size() + (hi - lo) * (bin ? 40 : 96));
  char chr[16];
  const size_t chrLen = static_cast<size_t>(std::to_chars(chr, chr + sizeof chr, data.chrNumber).ptr - chr);
  for (size_t i = lo; i < hi; ++i) {
    const IbdSegment s = toIbdSegment(block, i);
    const int bpStart = data.physicalPositions[s.posStart], bpEnd = data.physicalPositions[s.posEnd];
    const float cm = 100.f * (data.geneticPositions[s.posEnd] - data.geneticPositions[s.posStart]);
    const double score = s.prob / static_cast<double>(static_cast<unsigned>(s.posEnd - s.posStart) + 1u);
    if (!bin) {
      out += m_out->idPrefix[s.ind1];
      out += static_cast<char>('0' + s.hap1);
      out += '\t';
      out += m_out->idPrefix[s.ind2];
      out += static_cast<char>('0' + s.hap2);
      out += '\t';
      out.append(chr, chrLen);
      out += '\t';
      appendInt(out, bpStart);
      out += '\t';
      appendInt(out, bpEnd);
      if (decodingParams.outputIbdSegmentLength) {
        appendG7(out, static_cast<double>(cm));
      }
      appendG7(out, score);
      if (decodingParams.doPerPairPosteriorMean) {
        appendG7(out, static_cast<double>(s.postMean));
      }
      if (decodingParams.doPerPairMAP) {
        appendG7(out, static_cast<double>(s.mapTime));
      }
      out += '\n';
    } else {
      auto put = [&out](const void* p, const size_t nBytes) { out.append(static_cast<const char*>(p), nBytes); };
      const unsigned ind[2] = {s.ind1, s.ind2};
      const uint8_t hp[2] = {static_cast<uint8_t>(s.hap1), static_cast<uint8_t>(s.hap2)};
      const float scoreF = static_cast<float>(score);
      put(&ind[0], sizeof(unsigned));
      put(&hp[0], 1);
      put(&ind[1], sizeof(unsigned));
      put(&hp[1], 1);
      put(&bpStart, sizeof(int));
      put(&bpEnd, sizeof(int));
      if (decodingParams.outputIbdSegmentLength) {
        put(&cm, sizeof(float));
      }
      put(&scoreF, sizeof(float));
      if (decodingParams.doPerPairPosteriorMean) {
        put(&s.postMean, sizeof(float));
      }
      if (decodingParams.doPerPairMAP) {
        put(&s.mapTime, sizeof(float));
      }
    }
  }
}

// Per-site posterior mean / MAP for ASMC::decodePairs (ref: HMM.cpp:1360-1458)
void HMM::runPerSiteChunk(const Pending* pend, const unsigned long* rows, const size_t n)
{
  const TileSet t = buildTiles(pend, n, static_cast<size_t>(m_batchSize), false, data.geneticPositions, data.sites);
  const size_t T = t.pairs.size();
  const int L = data.sites;
  const int S = static_cast<int>(m_decodingQuant.states);
  fsmc_decode_request req{};
  req.numTiles = static_cast<int64_t>(T);
  req.hapA = t.hapA.data();
  req.hapB = t.hapB.data();
  req.tilePairs = t.pairs.data();
  req.tileFrom = t.from.data();
  req.tileTo = t.to.data();
  // the reference computes the MAP rows only under the posterior-mean flag (ref: HMM.cpp:1447-1449); both outputs
  // are produced here whenever either is stored
  req.flags = FSMC_SITE_MEAN | FSMC_SITE_MAP | (decodingParams.exactArithmetic ? FSMC_EXACT : 0u) |
              (m_storePerPairPosterior ? FSMC_SITE_POSTERIOR : 0u) | (m_storeSumOfPosterior ? FSMC_SUM_POSTERIOR : 0u);
  std::vector<float> mean(T * FSMC_TILE * static_cast<size_t>(L));
  std::vector<int32_t> map(T * FSMC_TILE * static_cast<size_t>(L));
  std::vector<float> post, postSum;
  req.siteMean = mean.data();
  req.siteMap = map.data();
  req.siteStride = L;
  if (m_storePerPairPosterior) {
    post.resize(T * FSMC_TILE * static_cast<size_t>(S) * static_cast<size_t>(L));
    req.sitePosterior = post.data();
  }
  if (m_storeSumOfPosterior) {
    postSum.resize(static_cast<size_t>(S) * static_cast<size_t>(L));
    req.sumPosterior = postSum.data();
  }
  fsmc_decode_stats st{};
  const double t0 = now();
  check(fsmc_decode(m_ctx, &req, &st), "fsmc_decode");
  m_stats.decodeWallS += now() - t0;
  m_stats.decodeCalls += 1;
  m_stats.pairsDecoded += n;
  m_stats.pairSites += st.pairSites;
  m_stats.kernelMs += st.kernelMs;
  m_stats.deviceMs += st.totalMs;
  m_stats.d2hBytes += static_cast<double>(st.d2hBytes);
  auto& out = m_decodePairsReturnStruct;
  for (size_t tile = 0; tile < T; ++tile) {
    for (int lane = 0; lane < t.pairs[tile]; ++lane) {
      const size_t p = t.firstPair[tile] + lane;
      const unsigned long row = rows[p];
      const size_t src = (tile * FSMC_TILE + lane) * static_cast<size_t>(L);
      const unsigned long a = pend[p].hapA, b = pend[p].hapB;
      out.perPairIndices.at(row) =
          std::make_tuple(a, asmc::indPlusHapToCombinedId(data.IIDList.at(a / 2), 1 + a % 2), b,
                          asmc::indPlusHapToCombinedId(data.IIDList.at(b / 2), 1 + b % 2));
      if (m_storePerPairPosteriorMean) {
        std::memcpy(out.perPairPosteriorMeans.row(static_cast<long>(row)), &mean[src], sizeof(float) * L);
      }
      if (m_storePerPairMAP) {
        std::memcpy(out.perPairMAPs.row(static_cast<long>(row)), &map[src], sizeof(int32_t) * L);
      }
      if (m_storePerPairPosterior) {
        // the reference stores posterior * expectedCoalTimes[k] (ref: HMM.cpp:1382-1386)
        auto& dst = out.perPairPosteriors.at(row);
        const float* srcPost = &post[(tile * FSMC_TILE + lane) * static_cast<size_t>(S) * L];
        for (int k = 0; k < S; ++k) {
          const float e = m_decodingQuant.expectedTimes[k];
          float* d = dst.row(k);
          for (int s2 = 0; s2 < L; ++s2) {
            d[s2] = srcPost[static_cast<size_t>(k) * L + s2] * e;
          }
        }
      }
      out.incrementNumWritten();
    }
  }
  if (m_storeSumOfPosterior) {
    // sum over pairs of posterior * expectedCoalTimes[k] (ref: HMM.cpp:1387-1389); the device sums the posteriors,
    // the weight is applied to the sum (equal to rounding)
    for (int k = 0; k < S; ++k) {
      const float e = m_decodingQuant.expectedTimes[k];
      float* d = out.sumOfPosteriors.row(k);
      for (int s2 = 0; s2 < L; ++s2) {
        d[s2] += postSum[static_cast<size_t>(k) * L + s2] * e;
      }
    }
  }
}

void HMM::decodeHapPairsToDevice(const std::vector<unsigned long>& hapsA, const std::vector<unsigned long>& hapsB,
                                 const DeviceOutputs& out)
{
  if (!m_pending.empty() || decodingParams.FastSMC) {
    throw std::runtime_error("HMM::decodeHapPairsToDevice: needs ASMC mode (no segment calling) and no pairs still queued");
  }
  check(fsmc_ctx_set_stream(m_ctx, out.stream), "fsmc_ctx_set_stream");
  m_deviceOut = &out;
  m_deviceRowsQueued = 0;
  try {
    decodeHapPairs(hapsA, hapsB);
    finishDecoding();
  } catch (...) {
    m_pending.clear();
    m_pendingRow.clear();
    m_deviceOut = nullptr;
    fsmc_ctx_set_stream(m_ctx, nullptr);
    throw;
  }
  m_deviceOut = nullptr;
  check(fsmc_ctx_set_stream(m_ctx, nullptr), "fsmc_ctx_set_stream");
}

// The outputs of runPerSiteChunk, written by the kernels into the caller's device rows (fsmc_decode_device)
void HMM::runDeviceChunk(const Pending* pend, const unsigned long* rows, const size_t n)
{
  const TileSet t = buildTiles(pend, n, static_cast<size_t>(m_batchSize), false, data.geneticPositions, data.sites);
  const size_t T = t.pairs.size();
  const DeviceOutputs& o = *m_deviceOut;
  fsmc_decode_request req{};
  req.numTiles = static_cast<int64_t>(T);
  req.hapA = t.hapA.data();
  req.hapB = t.hapB.data();
  req.tilePairs = t.pairs.data();
  req.tileFrom = t.from.data();
  req.tileTo = t.to.data();
  req.flags = (o.perPairPosteriorMeans ? FSMC_SITE_MEAN : 0u) | (o.perPairMAPs ? FSMC_SITE_MAP : 0u) |
              (o.perPairPosteriors ? FSMC_SITE_POSTERIOR : 0u) | (o.sumOfPosteriors ? FSMC_SUM_POSTERIOR : 0u) |
              (decodingParams.exactArithmetic ? FSMC_EXACT : 0u);
  std::vector<int64_t> laneRow(T * FSMC_TILE, 0);
  for (size_t tile = 0; tile < T; ++tile) {
    for (int lane = 0; lane < t.pairs[tile]; ++lane) {
      laneRow[tile * FSMC_TILE + lane] = static_cast<int64_t>(rows[t.firstPair[tile] + lane]);
    }
  }
  fsmc_device_outputs dev{};
  dev.laneRow = laneRow.data();
  dev.numRows = static_cast<int64_t>(m_deviceRowsQueued);
  dev.siteStride = data.sites;
  dev.siteMean_dev = o.perPairPosteriorMeans;
  dev.siteMap_dev = o.perPairMAPs;
  dev.sitePosterior_dev = o.perPairPosteriors;
  dev.sumPosterior_dev = o.sumOfPosteriors;
  // the reference stores posterior * expectedCoalTimes[k] (ref: HMM.cpp:1382-1389)
  dev.stateWeight = m_decodingQuant.expectedTimes.data();
  fsmc_decode_stats st{};
  const double t0 = now();
  check(fsmc_decode_device(m_ctx, &req, &dev, &st), "fsmc_decode_device");
  m_stats.decodeWallS += now() - t0;
  m_stats.decodeCalls += 1;
  m_stats.pairsDecoded += n;
  m_stats.pairSites += st.pairSites;
  m_stats.kernelMs += st.kernelMs;
  m_stats.deviceMs += st.totalMs;
  m_stats.d2hBytes += static_cast<double>(st.d2hBytes);
}

// Posterior sums over all pairs of the job for ASMC's decodeAll (ref: HMM.cpp:1044-1085, augmentSumOverPairs): the
// device sums the posteriors of a chunk per (site, state) and, for the major/minor sums, per genotype class of the
// pair at the site; chunks are added up here.  Float atomics: equal to the reference's sequential sums to rounding.
void HMM::runPosteriorSumChunk(const Pending* pend, const size_t n)
{
  const TileSet t = buildTiles(pend, n, static_cast<size_t>(m_batchSize), false, data.geneticPositions, data.sites);
  const int L = data.sites;
  const int S = static_cast<int>(m_decodingQuant.states);
  const bool byGenotype = decodingParams.doMajorMinorPosteriorSums;
  fsmc_decode_request req{};
  req.numTiles = static_cast<int64_t>(t.pairs.size());
  req.hapA = t.hapA.data();
  req.hapB = t.hapB.data();
  req.tilePairs = t.pairs.data();
  req.tileFrom = t.from.data();
  req.tileTo = t.to.data();
  req.flags = FSMC_SUM_POSTERIOR | (byGenotype ? FSMC_SUM_BY_GENOTYPE : 0u) | (decodingParams.exactArithmetic ? FSMC_EXACT : 0u);
  const size_t plane = static_cast<size_t>(S) * L;
  std::vector<float> sums((byGenotype ? 3 : 1) * plane);
  req.sumPosterior = sums.data();
  fsmc_decode_stats st{};
  const double t0 = now();
  check(fsmc_decode(m_ctx, &req, &st), "fsmc_decode");
  m_stats.decodeWallS += now() - t0;
  m_stats.decodeCalls += 1;
  m_stats.pairsDecoded += n;
  m_stats.batches += (n + m_batchSize - 1) / m_batchSize;
  m_stats.pairSites += st.pairSites;
  m_stats.kernelMs += st.kernelMs;
  m_stats.deviceMs += st.totalMs;
  auto& out = m_decodingReturnValues;
  auto addPlane = [&](RowMajorMatrix<float>& dst, const float* src) {
    for (int k = 0; k < S; ++k) {
      for (int pos = 0; pos < L; ++pos) {
        dst(pos, k) += src[static_cast<size_t>(k) * L + pos];
      }
    }
  };
  if (byGenotype) {
    addPlane(out.sumOverPairs00, &sums[0]);
    addPlane(out.sumOverPairs01, &sums[plane]);
    addPlane(out.sumOverPairs11, &sums[2 * plane]);
    if (decodingParams.doPosteriorSums) {
      for (int c = 0; c < 3; ++c) {
        addPlane(out.sumOverPairs, &sums[c * plane]);
      }
    }
  } else {
    addPlane(out.sumOverPairs, &sums[0]);
  }
}

// ref: HMM.cpp:1464-1495 — the whole posterior of one pair, [state][site - from]
std::vector<std::vector<float>> HMM::decode(const PairObservations& obs)
{
  return decode(obs, 0u, static_cast<unsigned>(data.sites));
}

std::vector<std::vector<float>> HMM::decode(const PairObservations& obs, const unsigned from, const unsigned to)
{
  if (from >= to || to > static_cast<unsigned>(data.sites)) {
    throw std::runtime_error("HMM::decode: window out of range");
  }
  const int S = static_cast<int>(m_decodingQuant.states);
  const int len = static_cast<int>(to - from);
  std::vector<uint32_t> hapA(FSMC_TILE, 0u), hapB(FSMC_TILE, 0u);
  hapA[0] = static_cast<uint32_t>(asmc::dipToHapId(obs.iInd, obs.iHap));
  hapB[0] = static_cast<uint32_t>(asmc::dipToHapId(obs.jInd, obs.jHap));
  const int32_t one = 1, f = static_cast<int32_t>(from), e = static_cast<int32_t>(to);
  fsmc_decode_request req{};
  req.numTiles = 1;
  req.hapA = hapA.data();
  req.hapB = hapB.data();
  req.tilePairs = &one;
  req.tileFrom = &f;
  req.tileTo = &e;
  const bool sums = decodingParams.doPosteriorSums;
  req.flags = FSMC_SITE_POSTERIOR | (decodingParams.exactArithmetic ? FSMC_EXACT : 0u);
  std::vector<float> post(static_cast<size_t>(FSMC_TILE) * S * len);
  req.sitePosterior = post.data();
  req.siteStride = len;
  check(fsmc_decode(m_ctx, &req, nullptr), "fsmc_decode");
  std::vector<std::vector<float>> out(static_cast<size_t>(S));
  for (int k = 0; k < S; ++k) {
    out[k].assign(post.begin() + static_cast<size_t>(k) * len, post.begin() + static_cast<size_t>(k + 1) * len);
    if (sums) {
      for (int pos = 0; pos < len; ++pos) {
        m_decodingReturnValues.sumOverPairs(static_cast<long>(from) + pos, k) += out[k][pos];
      }
    }
  }
  return out;
}

// ref: HMM.cpp:1532-1560
std::pair<std::vector<float>, std::vector<float>> HMM::decodeSummarize(const PairObservations& obs)
{
  const Pending p{static_cast<uint32_t>(asmc::dipToHapId(obs.iInd, obs.iHap)),
                  static_cast<uint32_t>(asmc::dipToHapId(obs.jInd, obs.jHap)), 0u, static_cast<uint32_t>(data.sites)};
  const TileSet t = buildTiles(&p, 1, 1, false, data.geneticPositions, data.sites);
  const int L = data.sites;
  fsmc_decode_request req{};
  req.numTiles = 1;
  req.hapA = t.hapA.data();
  req.hapB = t.hapB.data();
  req.tilePairs = t.pairs.data();
  req.tileFrom = t.from.data();
  req.tileTo = t.to.data();
  req.flags = FSMC_SITE_MEAN | FSMC_SITE_MAP | (decodingParams.exactArithmetic ? FSMC_EXACT : 0u);
  std::vector<float> mean(static_cast<size_t>(FSMC_TILE) * L);
  std::vector<int32_t> map(static_cast<size_t>(FSMC_TILE) * L);
  req.siteMean = mean.data();
  req.siteMap = map.data();
  req.siteStride = L;
  check(fsmc_decode(m_ctx, &req, nullptr), "fsmc_decode");
  std::pair<std::vector<float>, std::vector<float>> out;
  out.first.assign(mean.begin(), mean.begin() + L);
  out.second.resize(L);
  for (int s = 0; s < L; ++s) {
    out.second[s] = m_decodingQuant.expectedTimes[map[s]];
  }
  return out;
}
