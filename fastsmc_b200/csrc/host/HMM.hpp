// fastsmc_b200 host layer — the pairwise-coalescent HMM decoder, with the reference's public interface
// (ref: ASMC_SRC/SRC/HMM.hpp:172-299) over the CUDA kernels behind include/fastsmc_b200.h.
//
// What stays on the host: model preparation (emission tables with the reference's RNG sequence, transition-row
// lookup), the batching protocol (which pairs are decoded together and over which window, ref: HMM.cpp:470-636) and
// output formatting (ref: HMM.cpp:1110-1177).  What runs on the GPU: forward, backward, posterior, segment calling,
// per-segment age estimates and per-site summaries (ref: HMM.cpp:639-1041, 1087-1107, 1179-1458).
#pragma once

#include <atomic>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#include "Data.hpp"
#include "DecodePairsReturnStruct.hpp"
#include "DecodingParams.hpp"
#include "DecodingQuantities.hpp"

struct fsmc_ctx;

// A haplotype pair submitted for decoding (ref: HMM.hpp:36-51).  The reference materialises the XOR / AND bit
// vectors here; the kernels read the packed haplotypes directly, so only the indices are kept.  obsBits and
// homMinorBits are filled by HMM::makePairObs only when asked to (materialise = true).
struct PairObservations {
  int_least8_t iHap = 1;
  int_least8_t jHap = 1;
  unsigned int iInd = 0;
  unsigned int jInd = 0;
  std::vector<bool> obsBits;
  std::vector<bool> homMinorBits;
};

// ref: HMM.hpp:45-64.
struct DecodingReturnValues {
  /// sum of posteriors over all decoded pairs, sites x states (ref: HMM.hpp:52); filled when doPosteriorSums
  RowMajorMatrix<float> sumOverPairs;
  /// the same restricted to pairs that are both-major / heterozygous / both-minor at the site (doMajorMinorPosteriorSums)
  RowMajorMatrix<float> sumOverPairs00, sumOverPairs01, sumOverPairs11;
  int sites = 0;
  unsigned int states = 0;
  std::vector<bool> siteWasFlippedDuringFolding = {};
};

// One called IBD segment, ready for formatting.
struct IbdSegment {
  unsigned int ind1 = 0, ind2 = 0;  // indices into Data::FamIDList / IIDList
  int hap1 = 1, hap2 = 1;
  int posStart = 0, posEnd = 0;  // site indices, inclusive
  float prob = 0.f;              // sum of per-site IBD probabilities
  float postMean = 0.f;
  float mapTime = 0.f;
};

class HMM
{
public:
  HMM(Data _data, const DecodingParams& _decodingParams, int _scalingSkip = 1);
  ~HMM();
  HMM(const HMM&) = delete;
  HMM& operator=(const HMM&) = delete;

  /// Decodes every pair of the job when hashing is off (ref: HMM.cpp:283-381); with hashing on it only opens the
  /// output file, as the reference does.
  void decodeAll(int jobs, int jobInd);

  PairObservations makePairObs(int_least8_t iHap, unsigned int ind1, int_least8_t jHap, unsigned int ind2,
                               bool materialise = false);
  void decodePair(unsigned int i, unsigned int j);
  void decodeHapPair(unsigned long i, unsigned long j);
  void decodePairs(const std::vector<unsigned int>& individualsA, const std::vector<unsigned int>& individualsB);
  void decodeHapPairs(const std::vector<unsigned long>& individualsA, const std::vector<unsigned long>& individualsB);
  /// Queues haplotypes i, j (indices into the job's loaded haplotypes) with the match range [from, to]
  /// (ref: HMM.cpp:470-502).
  void decodeFromHashing(unsigned int i, unsigned int j, unsigned int fromPosition, unsigned int toPosition);

  /// Full posterior of one pair, states x sites (ref: HMM.cpp:1464-1530).
  std::vector<std::vector<float>> decode(const PairObservations& observations);
  std::vector<std::vector<float>> decode(const PairObservations& observations, unsigned from, unsigned to);
  /// (per-site posterior mean, per-site MAP expected time) of one pair (ref: HMM.cpp:1532-1560)
  std::pair<std::vector<float>, std::vector<float>> decodeSummarize(const PairObservations& observations);

  unsigned int getStateThreshold();
  const std::vector<PairObservations>& getBatchBuffer() { return m_observationsBatch; }
  const DecodingReturnValues& getDecodingReturnValues() { return m_decodingReturnValues; }
  DecodePairsReturnStruct& getDecodePairsReturnStruct() { return m_decodePairsReturnStruct; }
  void finishDecoding();
  void closeIBDFile();
  void finishFromHashing();
  const DecodingQuantities& getDecodingQuantities() const { return m_decodingQuant; }
  const Data& getData() const { return data; }

  void setStorePerPairPosteriorMean(bool v = true) { m_storePerPairPosteriorMean = v; }
  // the per-pair text writers of ASMC_exe (.perPairPosteriorMeans.gz / .perPairMAP.gz) are not part of this build: asking for
  // them fails loudly instead of silently producing no file (use ASMC::decodePairs and the returned arrays)
  void setWritePerPairPosteriorMean(bool v = true)
  {
    if (v) {
      throw std::runtime_error("writing .perPairPosteriorMeans.gz is not supported by the B200 build; use the stored per-pair outputs");
    }
    m_writePerPairPosteriorMean = v;
  }
  void setStorePerPairMap(bool v = true) { m_storePerPairMAP = v; }
  void setWritePerPairMap(bool v = true)
  {
    if (v) {
      throw std::runtime_error("writing .perPairMAP.gz is not supported by the B200 build; use the stored per-pair outputs");
    }
    m_writePerPairMAP = v;
  }
  void setStorePerPairPosterior(bool v = true) { m_storePerPairPosterior = v; }
  void setStoreSumOfPosterior(bool v = true) { m_storeSumOfPosterior = v; }

  /// Caller-owned device memory (of the decoding device) for decodeHapPairsToDevice; NULL = not computed.  Row r is the
  /// r-th pair of the call.  The values are those ASMC::decodePairs stores (posteriors times expectedTimes).
  struct DeviceOutputs {
    float* perPairPosteriors = nullptr;      // [pairs][states][sites]
    float* sumOfPosteriors = nullptr;        // [states][sites], added to
    float* perPairPosteriorMeans = nullptr;  // [pairs][sites]
    int32_t* perPairMAPs = nullptr;          // [pairs][sites]
    void* stream = nullptr;                  // cudaStream_t the work is enqueued on (NULL: the context's own stream)
  };
  /// The per-pair outputs of decodeHapPairs written by the kernels straight into `out`, chunk by chunk (the chunks of the
  /// host path, so the sums are added up in the same order).  Neither the return structure nor the posterior sums of
  /// decodeAll (DecodingReturnValues) are touched.
  void decodeHapPairsToDevice(const std::vector<unsigned long>& hapsA, const std::vector<unsigned long>& hapsB,
                              const DeviceOutputs& out);

  // ---- B200 build: model tables as handed to fsmc_set_model, and run statistics ---------------------------------
  struct ModelTables {
    int states = 0, sites = 0, numDistances = 0;
    std::vector<float> emission1, emission0minus1, emission2minus0;  // [sites][states]
    std::vector<float> D, B, U, RR;                                  // [numDistances][states]
    std::vector<int32_t> distanceRow;                                // [sites]
    int stateThreshold = 0, ageThreshold = 0;
    float probabilityThreshold = 0.f;
  };
  const ModelTables& getModelTables() const { return m_model; }
  uint64_t m_modelTag = 0;  // identity of m_model among the jobs of one data set (fsmc_model::modelTag)
  /// Host-only part of the constructor (no GPU needed): emission tables incl. the reference's RNG sequence
  /// (ref: HMM.cpp:159-256), per-site transition rows (SURVEY F10) and the IBD thresholds (ref: HMM.cpp:93-105).
  static ModelTables buildModelTables(const Data& data, const DecodingQuantities& dq, const DecodingParams& params);
  struct RunStats {
    unsigned long pairsDecoded = 0, batches = 0, segments = 0, decodeCalls = 0;
    double pairSites = 0.0;   // real pairs x window length, summed over batches
    double kernelMs = 0.0;    // device time inside the decode kernels
    double deviceMs = 0.0;    // device time of the fsmc_decode calls incl. their copies
    double decodeWallS = 0.0; // host wall time spent in fsmc_decode
    double outputWallS = 0.0; // host wall time formatting + compressing records
    double tablesWallS = 0.0; // constructor: decoding quantities + emission / transition tables on the host
    double uploadWallS = 0.0; // constructor: context creation, model and haplotype upload
    double d2hBytes = 0.0;    // decode outputs copied device -> host
  };
  const RunStats& getRunStats() const { return m_stats; }
  fsmc_ctx* context() { return m_ctx; }
  int getDevice() const { return decodingParams.device; }  // CUDA device of the decode context
  /// segments of the run are also kept in memory when this is set (tests, Python callers)
  void setKeepSegments(bool keep) { m_keepSegments = keep; }
  const std::vector<IbdSegment>& getSegments() const { return m_segments; }
  unsigned long getNumberOfDetectedSegments() const { return nbSegmentsDetected; }

private:
  struct Pending {
    uint32_t hapA, hapB, from, to;
  };
  struct GzOut;
  struct SegmentBlock;
  struct ChunkJob;
  struct DecodePipeline;

  Data data;
  DecodingQuantities m_decodingQuant;
  DecodingParams decodingParams;
  ModelTables m_model;
  fsmc_ctx* m_ctx = nullptr;
  fsmc_ctx* m_ctx2 = nullptr;  // second decode worker's context (narrow-kernel requests only)
  std::unique_ptr<DecodePipeline> m_pipeline;
  int m_batchSize = 64;
  long sequenceLength = 0;
  unsigned int stateThreshold = 0, ageThreshold = 0;
  float probabilityThreshold = 0.f;
  const int precision = 2;
  const float minGenetic = 1e-10f;

  std::vector<PairObservations> m_observationsBatch;  // mirrors the reference's partially filled batch
  std::vector<Pending> m_pending;
  std::vector<unsigned long> m_pendingRow;  // row of the return struct for each pending pair (decodePairs path)
  size_t m_flushPairs = 0;
  size_t m_perSiteChunkCap = 0;  // FSMC_FLUSH_BATCHES: also caps the per-site chunks of decodeHapPairs (0 = no cap)
  const DeviceOutputs* m_deviceOut = nullptr;  // set during decodeHapPairsToDevice
  unsigned long m_deviceRowsQueued = 0;        // pairs of that call queued so far
  bool m_windowed = false;  // pending pairs carry their own [from,to] (hashing) instead of [0, sites)

  DecodingReturnValues m_decodingReturnValues;
  DecodePairsReturnStruct m_decodePairsReturnStruct;
  bool m_storePerPairPosteriorMean = false, m_writePerPairPosteriorMean = false;
  bool m_storePerPairMAP = false, m_writePerPairMAP = false;
  bool m_storePerPairPosterior = false, m_storeSumOfPosterior = false;

  std::unique_ptr<GzOut> m_out;
  unsigned long cpt = 0, nbSegmentsDetected = 0;
  RunStats m_stats;
  bool m_keepSegments = false;
  std::vector<IbdSegment> m_segments;

  void uploadModel();
  void uploadModelTo(fsmc_ctx*& ctx);
  void startDecodeWorkers();
  void drainDecodes();
  void decodeChunk(ChunkJob& job, fsmc_ctx* ctx);
  void completeChunk(ChunkJob& job);
  void openOutput(int jobs, int jobInd);
  void flushPending(bool all);
  void runSegmentChunk(const Pending* pairs, size_t n);
  void runPerSiteChunk(const Pending* pairs, const unsigned long* rows, size_t n);
  void runPosteriorSumChunk(const Pending* pairs, size_t n);
  void runDeviceChunk(const Pending* pairs, const unsigned long* rows, size_t n);
  IbdSegment toIbdSegment(const SegmentBlock& block, size_t i) const;
  void formatSegments(const SegmentBlock& block, size_t lo, size_t hi, std::string& out) const;
  std::atomic<double> m_segmentsPerPair{4.0};  // densest chunk so far: sizes the next chunk's record buffer
};
