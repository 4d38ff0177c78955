// fastsmc_b200 — implementation of the C ABI declared in include/fastsmc_b200.h.
// Host side of the decode path: device buffers, model assembly, tile scheduling, launches.
#include <algorithm>
#include <atomic>
#include <cub/device/device_radix_sort.cuh>
#include <chrono>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <tuple>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

#include "column_min.cuh"
#include "decode_kernels.cuh"
#include "decode_fast.cuh"
#include "decode_sparse.cuh"
#include "seed_kernels.cuh"
#include "seed_order.h"
#include "host/SeedMapOrder.hpp"
#include "segment_sort.h"
#include "split_select.h"

namespace
{

thread_local std::string gLastError;

int fail(const int code, const char* fmt, ...)
{
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  gLastError = buf;
  return code;
}

#define FSMC_CUDA(expr)                                                                                  \
  do {                                                                                                   \
    const cudaError_t e_ = (expr);                                                                       \
    if (e_ != cudaSuccess) {                                                                             \
      return fail(e_ == cudaErrorMemoryAllocation ? FSMC_E_NOMEM : FSMC_E_CUDA, "%s failed: %s (%s:%d)", \
                  #expr, cudaGetErrorString(e_), __FILE__, __LINE__);                                    \
    }                                                                                                    \
  } while (0)

template <class T> struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  ~DevBuf() { release(); }
  void release()
  {
    if (p) {
      cudaFree(p);
      p = nullptr;
      n = 0;
    }
  }
  cudaError_t ensure(const size_t count)
  {
    if (count <= n && p) {
      return cudaSuccess;
    }
    release();
    const cudaError_t e = cudaMalloc(&p, std::max<size_t>(count, 1) * sizeof(T));
    if (e == cudaSuccess) {
      n = count;
    }
    return e;
  }
};

// Page-locked host staging buffer (grow-only): device-to-host copies of the segment records run at full PCIe rate
// and without the driver's pageable bounce copy.
template <class T> struct PinnedBuf {
  T* p = nullptr;
  size_t n = 0;
  ~PinnedBuf() { release(); }
  void release()
  {
    if (p) {
      cudaFreeHost(p);
      p = nullptr;
      n = 0;
    }
  }
  cudaError_t ensure(const size_t count)
  {
    if (count <= n && p) {
      return cudaSuccess;
    }
    release();
    const size_t want = std::max<size_t>(count + count / 4, 1);
    const cudaError_t e = cudaHostAlloc(reinterpret_cast<void**>(&p), want * sizeof(T), cudaHostAllocDefault);
    if (e == cudaSuccess) {
      n = want;
    }
    return e;
  }
};

}  // namespace

struct fsmc_plan;

struct SeedKey {
  int32_t gap;
  float minLengthCm;
  uint64_t genPosSum, globalIdSum, flipSum;  // checksums of the callers' arrays (contents, not addresses)
  float skip;
  uint32_t window[4];
  int32_t lastJob, aboveDiag;
  uint32_t flags;
  int32_t maxSeeds, readAhead;
};

struct fsmc_ctx {
  int device = 0;
  cudaStream_t ownStream = nullptr;
  cudaStream_t stream = nullptr;
  cudaDeviceProp prop{};
  bool hasModel = false, hasHaps = false;
  uint64_t modelTag = 0;  // fsmc_model::modelTag of the tables on the device (0 = untagged)
  fsmc::DeviceModel model{};
  // The production kernels are specialised for 69 and 159 states.  Any other state count runs on them too: the model is
  // padded to the next specialised count with states that carry no probability (prior, emissions and transition
  // coefficients 0: alpha stays 0 there, so every posterior is unchanged).  kernelModel = model when S is 69 or 159.
  fsmc::DeviceModel kernelModel{};
  DevBuf<float> kernelSiteRows;
  DevBuf<float> laneAux;  // kernelModel.laneAux
  DevBuf<float> bwdRows;  // kernelModel.bwdRows
  DevBuf<float> siteRows, prior, expTimes, colRatios;
  DevBuf<uint64_t> haps;
  long long numHaps = 0;
  DevBuf<float> scratch, accScratch;
  DevBuf<float> stageE1, stageE0, stageE2, stageD, stageB, stageU, stageR;  // fsmc_set_model staging
  DevBuf<int> stageRowIdx;
  DevBuf<float> sumScratch;  // decodeFastKernel<SUM>: [resident warp][planes][L][Spad]
  DevBuf<float> ckptBeta;  // sparse age estimates: beta checkpoints of every tile of the current plan (decode_sparse.cuh)
  std::vector<float> hostPrior, hostExpTimes, hostColRatios;
  long long sites = 0;
  // seeding scratch (fsmc_seed)
  DevBuf<uint64_t> seedKeysT;
  DevBuf<uint32_t> seedOwner, seedSlotCount, seedSlotGroup, seedSlotOf, seedRankOf, seedMembers, seedGroupSize,
      seedGroupMemberBase, seedGlobalId;
  DevBuf<unsigned long long> seedGroupPairBase, seedCounters, seedWordCounters, seedChunkBase;
  DevBuf<float> seedGenPos;
  DevBuf<fsmc_match> seedOut;
  DevBuf<uint32_t> seedRank;              // [W][H] seed-map iteration ranks (FSMC_SEED_REFERENCE_ORDER)
  DevBuf<unsigned char> seedLowComplexity; // [W] low-complexity flags (fsmc_seed_params.skip)
  // max_seeds > 0: registration keys (seed_kernels.cuh, nestedKeysKernels)
  DevBuf<uint32_t> seedRep0, seedCur;      // [W][H]
  DevBuf<unsigned char> seedDepth;         // [W][H]
  DevBuf<uint64_t> seedRegKeyT, seedRegKeys;  // [W][H], [H][W]
  fsmc::CandidateOrderer orderer;         // device-side reference candidate order (seed_order.h)
  const fsmc_match* orderedOut = nullptr; // its result, valid until the next fsmc_seed call
  bool seedCacheValid = false;  // seedOut holds every interval of the last fsmc_seed call (which overflowed the caller)
  SeedKey seedCacheKey{};
  fsmc_seed_stats seedCacheStats{};
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  // host staging of segment records and the per-pair counters of their counting sort (fsmc_plan_collect)
  PinnedBuf<fsmc_segment> segStage;
  std::vector<uint32_t> pairOffset, pairFirst;
  fsmc::SegmentSorter segmentSorter;  // device-side ordering of the records (segment_sort.h)
  // a destroyed plan is parked here so that the next fsmc_plan_create reuses its device buffers (fsmc_decode makes
  // one plan per call; cudaMalloc/cudaFree per call would serialise the device)
  fsmc_plan* sparePlan = nullptr;
  // (kernel, threads, dynamic shared memory) -> resident CTAs per SM: the attribute / occupancy queries of a plan are made
  // once per context, not once per call (they and cudaMemGetInfo were 10-90 ms of a 300 ms fsmc_decode call)
  std::map<std::tuple<const void*, int, size_t>, int> occupancy;
  DevBuf<uint32_t> colMinPart;  // fsmc_column_min_*: per-chunk (value, row) of every column
};

struct fsmc_plan {
  long long numTiles = 0;
  unsigned flags = 0;
  long long maxLen = 0;
  double pairSites = 0.0;
  long long segmentCapacity = 0;
  long long siteStride = 0;
  DevBuf<uint32_t> hapA, hapB;
  DevBuf<int> tilePairs, tileFrom, tileTo, scanFrom, scanTo, order;
  std::vector<int> hostOrder;  // source of the asynchronous copy into `order`
  DevBuf<fsmc_segment> segments;
  DevBuf<unsigned long long> counters;  // [0] segment count, [1] tile queue head
  DevBuf<float> siteMean, siteIbd, sitePosterior, sumPosterior;
  DevBuf<int> siteMap;
  // launch geometry
  int statesKernel = 0;
  int mode = 2;
  int threads = 128;
  int blocks = 0;
  size_t smemBytes = 0;
  long long scratchPerWarp = 0;
  bool launched = false;
  int launches = 0;
  bool fast = false;  // decodeFastKernel / decodeNarrowKernel (decode_fast.cuh)
  bool narrow = false;
  int tileWarps = 1;
  int tilesPerBlock = 1;  // tiles in flight per CTA (= scratch slabs per CTA)
  bool sumOnFast = false;  // posterior sums through per-warp accumulators (decodeFastKernel<SUM>)
  // sparse age estimates (decode_sparse.cuh)
  bool sparse = false;
  int ckptShift = 5;
  long long ckptSlots = 0;
  long long itemCapacity = 0;
  long long itemsFound = 0;
  DevBuf<long long> tileCkptBase;
  DevBuf<float> alphaScratch, itemAlpha, itemSums;
  DevBuf<fsmc::SparseItem> items;
  DevBuf<uint32_t> itemKeys;  // [4][itemCapacity]: keys, sorted keys, indices, sorted indices
  DevBuf<unsigned char> sortTemp;
  size_t sortTempBytes = 0;
  int refineBlocks = 0;
  size_t refineSmem = 0;
  // fsmc_decode_device: the kernels write the caller's device buffers at the rows of laneRow
  bool deviceOut = false;
  std::vector<uint32_t> hostLaneRow;
  std::vector<float> hostWeight;
  DevBuf<uint32_t> laneRow;
  DevBuf<float> stateWeight;  // [S]: the caller's weights, or ones
  float *outMean = nullptr, *outIbd = nullptr, *outPosterior = nullptr, *outSum = nullptr;
  int* outMap = nullptr;
};

namespace
{

using fsmc::DecodeArgs;
using fsmc::DeviceModel;

typedef void (*KernelFn)(const DeviceModel, const DecodeArgs);

struct KernelChoice {
  KernelFn fn;
  int statesKernel;
  int mode;
  int threads;
};

// Specialisations: the state counts of the decoding-quantity files shipped with the reference
// (69 = 30-100-2000 / UKBB, 159 = FASTSMC_EXAMPLE) get register-resident kernels; anything else
// runs on the generic shared-memory kernel.
KernelChoice chooseKernel(const int S, const unsigned flags)
{
  const bool exact = flags & FSMC_EXACT;
  const bool generic = flags & FSMC_GENERIC_KERNEL;
  if (!generic && S == 69) {
    return exact ? KernelChoice{fsmc::decodeTilesKernel<69, 0, true, 128, 2>, 69, 0, 128}
                 : KernelChoice{fsmc::decodeTilesKernel<69, 0, false, 128, 2>, 69, 0, 128};
  }
  if (!generic && S == 159) {
    return exact ? KernelChoice{fsmc::decodeTilesKernel<159, 1, true, 128, 1>, 159, 1, 128}
                 : KernelChoice{fsmc::decodeTilesKernel<159, 1, false, 128, 1>, 159, 1, 128};
  }
  return exact ? KernelChoice{fsmc::decodeTilesKernel<0, 2, true, 128, 1>, 0, 2, 128}
               : KernelChoice{fsmc::decodeTilesKernel<0, 2, false, 128, 1>, 0, 2, 128};
}

// The production kernel (decode_fast.cuh) exists for the state counts whose two state vectors fit the register file.
using fsmc::FastKernelFn;
constexpr int kFastDepth = 2, kFastRescale = 4;
struct FastChoice {
  FastKernelFn fn = nullptr;
  int Spad = 0;
  int threads = 0;
  bool acc = false;
  bool narrow = false;      // decodeNarrowKernel: sT+1 floats per pair-site in HBM instead of S
  int recordQuads = 0;
  int splitWarps = 0;       // > 0: decodeSplitKernel, one tile per CTA of this many warps (decode_split.cuh)
  size_t splitSmem = 0;
  bool sparse = false;      // decodeNarrowKernel<SPARSE> + refineKernel (decode_sparse.cuh)
  bool sum = false;         // decodeFastKernel<SUM>: per-warp accumulators of the posterior sums
};

// FSMC_SPLIT=0 forces the one-warp-per-tile kernels, FSMC_SPLIT=1 the state-split kernels wherever one exists
// (development / A-B measurements); unset = the faster of the two as measured on B200.
int splitPreference()
{
  const char* e = std::getenv("FSMC_SPLIT");
  return e && *e ? std::atoi(e) : -1;
}
// Without per-segment age estimates 8 warps (2 CTAs of 4) fit an SM; the accumulators of FSMC_SEG_AGE cost 8.6 KB of
// shared memory per warp, which leaves room for 7 warps (1 CTA).
// preferSparse: the request's scan windows are long (all-pairs decoding): IBD runs cover a small part of them
FastChoice chooseFastKernel(const DeviceModel& m, const unsigned flags, const bool preferSparse = false)
{
  const int S = m.S;
  // full posterior matrices are produced by decodeTilesKernel only; sums over pairs also by decodeFastKernel<69, SUM>
  if ((flags & (FSMC_EXACT | FSMC_GENERIC_KERNEL | FSMC_SITE_POSTERIOR)) || S > fsmc::kMaxParamStates) {
    return {};
  }
  if (flags & FSMC_SUM_POSTERIOR) {
    if (S == 69 && !(flags & FSMC_CALL_SEGMENTS)) {
      FastChoice fc{fsmc::decodeFastKernel<69, kFastDepth, kFastRescale, false, 128, 2, true>, 72, 128, false};
      fc.sum = true;
      return fc;
    }
    return {};
  }
  const bool acc = (flags & FSMC_SEG_AGE) && (flags & FSMC_CALL_SEGMENTS);
  // only states below the IBD time threshold are looked at: no beta round trip needed
  const bool narrow = !(flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP | FSMC_WIDE_KERNEL)) && (!acc || m.ageThreshold <= m.stateThreshold) &&
                      m.stateThreshold + 1 <= 4 * fsmc::kNarrowMaxQuads;
  const int rqWanted = narrow ? (m.stateThreshold + 1 + 3) / 4 : 0;
  const int pref = (flags & FSMC_ONE_WARP_KERNEL) ? 0 : splitPreference();
  const bool trySplit = pref == 1 || (pref == -1 && S == 159);
  if (trySplit && (S == 69 || S == 159) && m.stateThreshold <= 32) {
    fsmc::SplitChoice sc{};
    static const bool laneOff = [] { const char* e = std::getenv("FSMC_LANE"); return e && *e == '0'; }();  // A/B runs
    if (S == 159 && m.laneAux && !laneOff) {
      sc = fsmc::laneKernel159(rqWanted);  // states cut across the lanes of a warp (decode_lane.cuh)
    }
    if (!sc.fn) {
      sc = S == 69 ? fsmc::splitKernel69(rqWanted, acc) : fsmc::splitKernel159(rqWanted, acc);
    }
    if (!sc.fn && narrow) {
      sc = S == 69 ? fsmc::splitKernel69(0, acc) : fsmc::splitKernel159(0, acc);  // no such record width: full rows
    }
    if (sc.fn) {
      FastChoice fc{sc.fn, sc.Spad, sc.warps * 32, sc.acc, sc.recordQuads > 0, sc.recordQuads};
      fc.splitWarps = sc.warps;
      fc.splitSmem = sc.smemBytes;
      return fc;
    }
  }
  // all-state age estimates of sparse IBD runs: narrow sweeps + checkpoints, full posteriors only inside the runs
  const bool sparse = preferSparse && S == 69 && acc && m.ageThreshold > m.stateThreshold &&
                      !(flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP | FSMC_WIDE_KERNEL)) && m.stateThreshold + 1 <= 4 * fsmc::kNarrowMaxQuads;
  if (sparse) {
    const int rq = (m.stateThreshold + 1 + 3) / 4;
    FastKernelFn fn = rq == 1   ? fsmc::decodeNarrowKernel<69, 1, 4, kFastDepth, 128, 2, 1>
                      : rq == 2 ? fsmc::decodeNarrowKernel<69, 2, 2, kFastDepth, 128, 2, 1>
                      : rq == 3 ? fsmc::decodeNarrowKernel<69, 3, 2, kFastDepth, 128, 2, 1>
                                : fsmc::decodeNarrowKernel<69, 4, 2, kFastDepth, 128, 2, 1>;
    if (const char* e = std::getenv("FSMC_SPARSE_VARIANT")) {  // development: A/B of code-size variants
      const int v = std::atoi(e);
      if (rq == 1 && v == 65) fn = fsmc::decodeNarrowKernel<69, 1, 4, kFastDepth, 128, 2, 65>;  // groups fully unrolled
    }
    FastChoice fc{fn, 72, 128, false, true, rq};
    fc.sparse = true;
    return fc;
  }
  if (S == 69 && narrow) {
    // 2 CTAs x 4 warps per SM at 255 registers: measured 12.2e9 pair-sites/s vs 10.1e9 at 3 CTAs / 168 registers (spills)
    const int rq = (m.stateThreshold + 1 + 3) / 4;
    // ring slots hold 4 window positions when two CTAs of that size fit an SM (records of 4 floats), else 2
    FastKernelFn fn = rq == 1   ? fsmc::decodeNarrowKernel<69, 1, 4, kFastDepth, 128, 2>
                      : rq == 2 ? fsmc::decodeNarrowKernel<69, 2, 2, kFastDepth, 128, 2>
                      : rq == 3 ? fsmc::decodeNarrowKernel<69, 3, 2, kFastDepth, 128, 2>
                                : fsmc::decodeNarrowKernel<69, 4, 2, kFastDepth, 128, 2>;
    if (const char* e = std::getenv("FSMC_SPARSE_VARIANT")) {
      if (rq == 1 && std::atoi(e) == 65) fn = fsmc::decodeNarrowKernel<69, 1, 4, kFastDepth, 128, 2, 64>;
    }
    return FastChoice{fn, 72, 128, false, true, rq};
  }
  if (S == 69) {
    return acc ? FastChoice{fsmc::decodeFastKernel<69, kFastDepth, kFastRescale, true, 128, 2>, 72, 128, true}
               : FastChoice{fsmc::decodeFastKernel<69, kFastDepth, kFastRescale, false, 128, 2>, 72, 128, false};
  }
  return {};
}
bool sparsePreferred(const double meanScanSites)
{
  if (const char* e = std::getenv("FSMC_SPARSE")) {
    return std::atoi(e) != 0;
  }
  return meanScanSites >= 2000.0;
}

size_t fastSmemBytes(const FastChoice& fc, const int S)
{
  if (fc.splitWarps > 0) {
    return fc.splitSmem;
  }
  const size_t warps = fc.threads / 32;
  if (fc.narrow) {
    const size_t group = fc.recordQuads == 1 ? 4 : 2;
    const size_t slot = group * static_cast<size_t>(fsmc::kBwdArrays) * fc.Spad * 4 + (group + 1) * static_cast<size_t>(fc.recordQuads) * 32 * 16;
    return warps * kFastDepth * slot + warps * kFastDepth * sizeof(uint64_t);
  }
  return warps * (kFastDepth * (static_cast<size_t>(fc.Spad) * 32 * 4 + static_cast<size_t>(fsmc::kRowArrays) * fc.Spad * 4) +
                  0 * static_cast<size_t>(S)) +
         warps * 2 * kFastDepth * sizeof(uint64_t);
}

size_t sumPosteriorCount(const DeviceModel& m, const unsigned flags)
{
  return static_cast<size_t>((flags & FSMC_SUM_BY_GENOTYPE) ? 3 : 1) * static_cast<size_t>(m.S) * static_cast<size_t>(m.L);
}

size_t smemPerWarp(const DeviceModel& m, const int mode, const unsigned flags)
{
  const bool age = (flags & FSMC_SEG_AGE) && (flags & FSMC_CALL_SEGMENTS);
  const size_t rows = (age ? m.ageThreshold : 0) + (mode >= 1 ? m.S : 0) + (mode == 2 ? m.S : 0);
  return rows * 32 * sizeof(float);
}

}  // namespace

extern "C" {

const char* fsmc_last_error(void)
{
  return gLastError.c_str();
}

int fsmc_version(void)
{
  return 100;
}

int fsmc_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

int fsmc_ctx_create(const int device, fsmc_ctx** out)
{
  if (!out) {
    return fail(FSMC_E_INVALID, "fsmc_ctx_create: out is NULL");
  }
  *out = nullptr;
  int n = 0;
  FSMC_CUDA(cudaGetDeviceCount(&n));
  if (device < 0 || device >= n) {
    return fail(FSMC_E_INVALID, "fsmc_ctx_create: device %d out of range (%d visible)", device, n);
  }
  FSMC_CUDA(cudaSetDevice(device));
  auto* ctx = new fsmc_ctx;
  ctx->device = device;
  cudaError_t e = cudaGetDeviceProperties(&ctx->prop, device);
  if (e == cudaSuccess) {
    e = cudaStreamCreateWithFlags(&ctx->ownStream, cudaStreamNonBlocking);
  }
  for (int i = 0; i < 4 && e == cudaSuccess; ++i) {
    e = cudaEventCreate(&ctx->ev[i]);
  }
  if (e != cudaSuccess) {
    delete ctx;
    return fail(FSMC_E_CUDA, "fsmc_ctx_create: %s", cudaGetErrorString(e));
  }
  ctx->stream = ctx->ownStream;
  *out = ctx;
  return FSMC_OK;
}

int fsmc_ctx_destroy(fsmc_ctx* ctx)
{
  if (!ctx) {
    return FSMC_OK;
  }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (auto& e : ctx->ev) {
    if (e) {
      cudaEventDestroy(e);
    }
  }
  if (ctx->ownStream) {
    cudaStreamDestroy(ctx->ownStream);
  }
  delete ctx->sparePlan;
  delete ctx;
  return FSMC_OK;
}

int fsmc_ctx_set_stream(fsmc_ctx* ctx, void* cuda_stream)
{
  if (!ctx) {
    return fail(FSMC_E_INVALID, "fsmc_ctx_set_stream: ctx is NULL");
  }
  ctx->stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : ctx->ownStream;
  return FSMC_OK;
}

int fsmc_set_model(fsmc_ctx* ctx, const fsmc_model* mdl)
{
  if (!ctx || !mdl) {
    return fail(FSMC_E_INVALID, "fsmc_set_model: NULL argument");
  }
  const int S = mdl->states, L = mdl->sites;
  if (S < 2 || L < 1 || mdl->numDistances < 1 || !mdl->initialStateProb || !mdl->expectedTimes ||
      !mdl->columnRatios || !mdl->emission1 || !mdl->emission0minus1 || !mdl->emission2minus0 || !mdl->D ||
      !mdl->B || !mdl->U || !mdl->RR || !mdl->distanceRow) {
    return fail(FSMC_E_INVALID, "fsmc_set_model: bad sizes or NULL table (states=%d sites=%d)", S, L);
  }
  if (mdl->stateThreshold < 0 || mdl->stateThreshold > S || mdl->ageThreshold < 0 || mdl->ageThreshold > S) {
    return fail(FSMC_E_INVALID, "fsmc_set_model: thresholds out of range");
  }
  for (int s = 1; s < L; ++s) {
    if (mdl->distanceRow[s] < 0 || mdl->distanceRow[s] >= mdl->numDistances) {
      return fail(FSMC_E_INVALID, "fsmc_set_model: distanceRow[%d]=%d out of range", s, mdl->distanceRow[s]);
    }
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  const int Spad = (S + 3) / 4 * 4;
  cudaStream_t st = ctx->stream;
  auto setThresholds = [&](DeviceModel& dm) {
    dm.stateThreshold = mdl->stateThreshold;
    dm.ageThreshold = mdl->ageThreshold;
    // the reference compares against `N * probabilityThreshold` with an int N promoted to float
    dm.thr[0] = 1000 * mdl->probabilityThreshold;
    dm.thr[1] = 100 * mdl->probabilityThreshold;
    dm.thr[2] = 10 * mdl->probabilityThreshold;
    dm.thr[3] = mdl->probabilityThreshold;
  };
  if (mdl->modelTag != 0 && ctx->hasModel && ctx->modelTag == mdl->modelTag && ctx->model.S == S && ctx->model.L == L) {
    // the same tables as the ones this context holds (the jobs of one data set): keep the device rows
    setThresholds(ctx->model);
    setThresholds(ctx->kernelModel);
    return FSMC_OK;
  }
  ctx->hasModel = false;
  ctx->modelTag = 0;

  // staging copies of the caller's tables, gathered into per-site rows on the device.  The staging buffers belong to the
  // context (grow-only): cudaFree synchronises the whole device, which stalls the other host thread of a GPU that runs
  // the jobs of a data set two at a time.
  DevBuf<float>&e1 = ctx->stageE1, &e0 = ctx->stageE0, &e2 = ctx->stageE2, &D = ctx->stageD, &B = ctx->stageB, &U = ctx->stageU,
  &R = ctx->stageR;
  DevBuf<int>& rowIdx = ctx->stageRowIdx;
  const size_t nE = static_cast<size_t>(L) * S, nT = static_cast<size_t>(mdl->numDistances) * S;
  FSMC_CUDA(e1.ensure(nE));
  FSMC_CUDA(e0.ensure(nE));
  FSMC_CUDA(e2.ensure(nE));
  FSMC_CUDA(D.ensure(nT));
  FSMC_CUDA(B.ensure(nT));
  FSMC_CUDA(U.ensure(nT));
  FSMC_CUDA(R.ensure(nT));
  FSMC_CUDA(rowIdx.ensure(L));
  FSMC_CUDA(ctx->siteRows.ensure(static_cast<size_t>(L) * fsmc::kRowArrays * Spad));
  FSMC_CUDA(ctx->prior.ensure(Spad));
  FSMC_CUDA(ctx->expTimes.ensure(Spad));
  FSMC_CUDA(ctx->colRatios.ensure(Spad));
  FSMC_CUDA(cudaMemcpyAsync(e1.p, mdl->emission1, nE * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(e0.p, mdl->emission0minus1, nE * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(e2.p, mdl->emission2minus0, nE * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(D.p, mdl->D, nT * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(B.p, mdl->B, nT * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(U.p, mdl->U, nT * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(R.p, mdl->RR, nT * sizeof(float), cudaMemcpyHostToDevice, st));
  FSMC_CUDA(cudaMemcpyAsync(rowIdx.p, mdl->distanceRow, L * sizeof(int), cudaMemcpyHostToDevice, st));
  std::vector<float> pad(Spad, 0.f);
  auto upPad = [&](float* dst, const float* src) {
    std::fill(pad.begin(), pad.end(), 0.f);
    std::copy(src, src + S, pad.begin());
    return cudaMemcpyAsync(dst, pad.data(), Spad * sizeof(float), cudaMemcpyHostToDevice, st);
  };
  ctx->hostPrior.assign(mdl->initialStateProb, mdl->initialStateProb + S);
  ctx->hostExpTimes.assign(mdl->expectedTimes, mdl->expectedTimes + S);
  ctx->hostColRatios.assign(mdl->columnRatios, mdl->columnRatios + S);
  FSMC_CUDA(upPad(ctx->prior.p, mdl->initialStateProb));
  FSMC_CUDA(cudaStreamSynchronize(st));
  FSMC_CUDA(upPad(ctx->expTimes.p, mdl->expectedTimes));
  FSMC_CUDA(cudaStreamSynchronize(st));
  FSMC_CUDA(upPad(ctx->colRatios.p, mdl->columnRatios));
  FSMC_CUDA(cudaStreamSynchronize(st));

  const int threads = 256;
  const int blocks = std::max(1, ctx->prop.multiProcessorCount * 8);
  fsmc::buildSiteRowsKernel<<<blocks, threads, 0, st>>>(S, Spad, L, e1.p, e0.p, e2.p, D.p, B.p, U.p, R.p, rowIdx.p,
                                                         ctx->siteRows.p);
  FSMC_CUDA(cudaGetLastError());
  FSMC_CUDA(cudaStreamSynchronize(st));

  DeviceModel& m = ctx->model;
  m.S = S;
  m.Spad = Spad;
  m.L = L;
  m.siteRows = ctx->siteRows.p;
  m.prior = ctx->prior.p;
  m.expTimes = ctx->expTimes.p;
  m.colRatios = ctx->colRatios.p;
  setThresholds(m);
  m.haps = ctx->haps.p;
  m.wordsPerHap = ctx->hasHaps ? (ctx->sites + 63) / 64 : 0;
  ctx->kernelModel = m;
  const int Sk = S <= 69 ? 69 : (S <= 159 ? 159 : 0);
  if (Sk != 0 && Sk != S) {
    const int SpadK = (Sk + 3) / 4 * 4;
    FSMC_CUDA(ctx->kernelSiteRows.ensure(static_cast<size_t>(L) * fsmc::kRowArrays * SpadK));
    fsmc::buildSiteRowsKernel<<<blocks, threads, 0, st>>>(S, SpadK, L, e1.p, e0.p, e2.p, D.p, B.p, U.p, R.p, rowIdx.p,
                                                           ctx->kernelSiteRows.p);
    FSMC_CUDA(cudaGetLastError());
    FSMC_CUDA(cudaStreamSynchronize(st));
    ctx->kernelModel.S = Sk;
    ctx->kernelModel.Spad = SpadK;
    ctx->kernelModel.siteRows = ctx->kernelSiteRows.p;
  }
  ctx->model.laneAux = nullptr;
  ctx->kernelModel.laneAux = nullptr;
  ctx->model.bwdRows = nullptr;
  ctx->kernelModel.bwdRows = nullptr;
  if (ctx->kernelModel.S == 69) {
    FSMC_CUDA(ctx->bwdRows.ensure(static_cast<size_t>(L) * fsmc::kBwdArrays * ctx->kernelModel.Spad));
    fsmc::buildBackwardRowsKernel<<<blocks, threads, 0, st>>>(ctx->kernelModel.Spad, L, ctx->kernelModel.siteRows, ctx->bwdRows.p);
    FSMC_CUDA(cudaGetLastError());
    FSMC_CUDA(cudaStreamSynchronize(st));
    ctx->kernelModel.bwdRows = ctx->bwdRows.p;
  }
  if (ctx->kernelModel.S == 159) {
    FSMC_CUDA(ctx->laneAux.ensure(static_cast<size_t>(L) * fsmc::laneAuxFloats159()));
    fsmc::buildLaneAux159(L, ctx->kernelModel.siteRows, ctx->laneAux.p, blocks, st);
    FSMC_CUDA(cudaGetLastError());
    FSMC_CUDA(cudaStreamSynchronize(st));
    ctx->kernelModel.laneAux = ctx->laneAux.p;
  }
  ctx->hasModel = true;
  ctx->modelTag = mdl->modelTag;
  return FSMC_OK;
}

int fsmc_set_haplotypes(fsmc_ctx* ctx, const uint64_t* bits, const int64_t numHaps, const int64_t sites)
{
  if (!ctx || !bits || numHaps < 1 || sites < 1) {
    return fail(FSMC_E_INVALID, "fsmc_set_haplotypes: bad argument");
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  const long long words = (sites + 63) / 64;
  const size_t n = static_cast<size_t>(numHaps) * words;
  FSMC_CUDA(ctx->haps.ensure(n));
  FSMC_CUDA(cudaMemcpyAsync(ctx->haps.p, bits, n * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  FSMC_CUDA(cudaStreamSynchronize(ctx->stream));
  ctx->model.haps = ctx->haps.p;
  ctx->model.wordsPerHap = words;
  ctx->kernelModel.haps = ctx->haps.p;
  ctx->kernelModel.wordsPerHap = words;
  ctx->numHaps = numHaps;
  ctx->sites = sites;
  ctx->hasHaps = true;
  ctx->seedCacheValid = false;
  return FSMC_OK;
}

int fsmc_query_kernel(fsmc_ctx* ctx, const uint32_t flags, const double meanScanSites, fsmc_kernel_info* out)
{
  if (!ctx || !out) {
    return fail(FSMC_E_INVALID, "fsmc_query_kernel: NULL argument");
  }
  if (!ctx->hasModel) {
    return fail(FSMC_E_STATE, "fsmc_query_kernel: set the model first");
  }
  const DeviceModel& m = ctx->model;
  const FastChoice fc = chooseFastKernel(ctx->kernelModel, flags, sparsePreferred(meanScanSites));
  const KernelChoice kc = chooseKernel(m.S, flags);
  out->statesKernel = fc.fn ? ctx->kernelModel.S : kc.statesKernel;
  out->narrowKernel = fc.narrow ? 1 : 0;
  out->sparseKernel = fc.sparse ? 1 : 0;
  out->tileWarps = fc.splitWarps > 0 ? fc.splitWarps : 1;
  out->largeScratch = (!fc.fn || !fc.narrow || fc.sparse) ? 1 : 0;
  return FSMC_OK;
}

namespace
{
// cudaFuncSetAttribute(max dynamic shared memory) + resident CTAs per SM, cached per context
cudaError_t residentBlocks(fsmc_ctx* ctx, const void* fn, const int threads, const size_t smem, int* blocksPerSm)
{
  const auto key = std::make_tuple(fn, threads, smem);
  const auto it = ctx->occupancy.find(key);
  if (it != ctx->occupancy.end()) {
    *blocksPerSm = it->second;
    return cudaSuccess;
  }
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, static_cast<int>(smem));
  if (e != cudaSuccess) {
    return e;
  }
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocksPerSm, fn, threads, smem);
  if (e == cudaSuccess) {
    ctx->occupancy[key] = *blocksPerSm;
  }
  return e;
}
}  // namespace

namespace
{
// memory of the context's device (cudaMalloc'd or managed), not host memory or another device's
int checkDevicePtr(const fsmc_ctx* ctx, const void* p, const char* what)
{
  cudaPointerAttributes at{};
  const cudaError_t e = cudaPointerGetAttributes(&at, p);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(FSMC_E_INVALID, "%s is not a CUDA pointer (%s)", what, cudaGetErrorString(e));
  }
  if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged) {
    return fail(FSMC_E_INVALID, "fsmc_decode_device: %s is host memory, device memory of device %d is needed", what, ctx->device);
  }
  if (at.device != ctx->device) {
    return fail(FSMC_E_INVALID, "fsmc_decode_device: %s is on device %d, the context on device %d", what, at.device, ctx->device);
  }
  return FSMC_OK;
}
}  // namespace

// fsmc_plan_create; with `dev`, the outputs are the caller's device buffers (fsmc_decode_device) and none is allocated
static int planCreate(fsmc_ctx* ctx, const fsmc_decode_request* req, const fsmc_device_outputs* dev, fsmc_plan** out)
{
  if (!ctx || !req || !out) {
    return fail(FSMC_E_INVALID, "fsmc_plan_create: NULL argument");
  }
  *out = nullptr;
  if (!ctx->hasModel || !ctx->hasHaps) {
    return fail(FSMC_E_STATE, "fsmc_plan_create: set the model and the haplotypes first");
  }
  static const bool tracePlan = std::getenv("FSMC_TRACE_PLAN") != nullptr;  // development: host time of the phases below
  auto tMark = std::chrono::steady_clock::now();
  auto mark = [&](const char* what) {
    if (tracePlan) {
      const auto now = std::chrono::steady_clock::now();
      std::fprintf(stderr, "  plan_create %s %.2f ms\n", what, std::chrono::duration<double, std::milli>(now - tMark).count());
      tMark = now;
    }
  };
  const long long T = req->numTiles;
  if (T < 0 || T > (1ll << 26)) {
    return fail(FSMC_E_INVALID, "fsmc_plan_create: numTiles=%lld out of range", T);
  }
  const unsigned flags = req->flags;
  const bool seg = flags & FSMC_CALL_SEGMENTS;
  const bool siteOut = flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP | FSMC_SITE_IBD | FSMC_SITE_POSTERIOR);
  if ((flags & FSMC_SUM_BY_GENOTYPE) && !(flags & FSMC_SUM_POSTERIOR)) {
    return fail(FSMC_E_INVALID, "fsmc_plan_create: FSMC_SUM_BY_GENOTYPE needs FSMC_SUM_POSTERIOR");
  }
  if (T > 0 && (!req->hapA || !req->hapB || !req->tilePairs || !req->tileFrom || !req->tileTo ||
                (seg && (!req->tileScanFrom || !req->tileScanTo)))) {
    return fail(FSMC_E_INVALID, "fsmc_plan_create: NULL input array");
  }
  const DeviceModel& m = ctx->model;
  if (ctx->sites != m.L) {
    return fail(FSMC_E_STATE, "fsmc_plan_create: the haplotypes have %lld sites, the model %d", static_cast<long long>(ctx->sites), m.L);
  }
  long long maxLen = 0;
  double pairSites = 0.0, scanSites = 0.0;
  for (long long t = 0; t < T; ++t) {
    const int n = req->tilePairs[t], f = req->tileFrom[t], e = req->tileTo[t];
    if (n < 1 || n > FSMC_TILE || f < 0 || e > m.L || e <= f) {
      return fail(FSMC_E_INVALID, "fsmc_plan_create: tile %lld has pairs=%d window=[%d,%d) (sites=%d)", t, n, f, e,
                  m.L);
    }
    if (seg && (req->tileScanFrom[t] < f || req->tileScanTo[t] > e)) {
      return fail(FSMC_E_INVALID, "fsmc_plan_create: tile %lld scan window [%d,%d) outside decode window [%d,%d)", t,
                  req->tileScanFrom[t], req->tileScanTo[t], f, e);
    }
    for (int l = 0; l < n; ++l) {
      if (req->hapA[t * 32 + l] >= ctx->numHaps || req->hapB[t * 32 + l] >= ctx->numHaps) {
        return fail(FSMC_E_INVALID, "fsmc_plan_create: tile %lld lane %d haplotype index out of range", t, l);
      }
    }
    maxLen = std::max<long long>(maxLen, e - f);
    pairSites += static_cast<double>(n) * (e - f);
    scanSites += seg ? static_cast<double>(req->tileScanTo[t] - req->tileScanFrom[t]) : 0.0;
  }
  const long long siteStride = dev ? dev->siteStride : req->siteStride;
  if (siteOut && siteStride < maxLen) {
    return fail(FSMC_E_INVALID, "fsmc_plan_create: siteStride=%lld < longest window %lld", siteStride, maxLen);
  }
  if (dev) {
    if (seg) {
      return fail(FSMC_E_INVALID, "fsmc_decode_device: FSMC_CALL_SEGMENTS is not supported (segments go to the host: fsmc_decode)");
    }
    if (dev->numRows < 1 || dev->numRows > 0x7fffffffll) {
      return fail(FSMC_E_INVALID, "fsmc_decode_device: numRows=%lld out of range [1, 2^31)", static_cast<long long>(dev->numRows));
    }
    const struct {
      unsigned flag;
      const void* p;
      const char* name;
    } outs[] = {{FSMC_SITE_MEAN, dev->siteMean_dev, "siteMean_dev"},
                {FSMC_SITE_MAP, dev->siteMap_dev, "siteMap_dev"},
                {FSMC_SITE_IBD, dev->siteIbd_dev, "siteIbd_dev"},
                {FSMC_SITE_POSTERIOR, dev->sitePosterior_dev, "sitePosterior_dev"},
                {FSMC_SUM_POSTERIOR, dev->sumPosterior_dev, "sumPosterior_dev"}};
    for (const auto& o : outs) {
      if (!(flags & o.flag)) {
        continue;
      }
      if (!o.p) {
        return fail(FSMC_E_INVALID, "fsmc_decode_device: %s is NULL but its flag is set", o.name);
      }
      const int rc = checkDevicePtr(ctx, o.p, o.name);
      if (rc != FSMC_OK) {
        return rc;
      }
    }
    if (siteOut && T > 0) {
      if (!dev->laneRow) {
        return fail(FSMC_E_INVALID, "fsmc_decode_device: laneRow is NULL");
      }
      for (long long t = 0; t < T; ++t) {
        for (int l = 0; l < req->tilePairs[t]; ++l) {
          const int64_t r = dev->laneRow[t * 32 + l];
          if (r < 0 || r >= dev->numRows) {
            return fail(FSMC_E_INVALID, "fsmc_decode_device: laneRow[%lld]=%lld outside [0, numRows=%lld)", t * 32 + l,
                        static_cast<long long>(r), static_cast<long long>(dev->numRows));
          }
        }
      }
    }
  }
  if (seg && req->segmentCapacity < 0) {
    return fail(FSMC_E_INVALID, "fsmc_plan_create: negative segmentCapacity");
  }

  FSMC_CUDA(cudaSetDevice(ctx->device));
  fsmc_plan* plan = ctx->sparePlan ? ctx->sparePlan : new fsmc_plan;
  ctx->sparePlan = nullptr;
  struct Guard {
    fsmc_plan*& p;
    bool keep = false;
    ~Guard()
    {
      if (!keep) {
        delete p;
        p = nullptr;
      }
    }
  } guard{plan};

  plan->numTiles = T;
  plan->flags = flags;
  plan->maxLen = maxLen;
  plan->pairSites = pairSites;
  plan->segmentCapacity = seg ? req->segmentCapacity : 0;
  plan->siteStride = siteOut ? siteStride : 0;
  plan->deviceOut = dev != nullptr;

  // longest-window-first launch order (dynamic queue → LPT schedule); stable, so equal windows keep input order
  std::vector<int>& order = plan->hostOrder;
  order.resize(T);
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](const int x, const int y) {
    return (req->tileTo[x] - req->tileFrom[x]) > (req->tileTo[y] - req->tileFrom[y]);
  });

  mark("validate + order");
  cudaStream_t st = ctx->stream;
  const size_t nLane = static_cast<size_t>(T) * 32;
  FSMC_CUDA(plan->hapA.ensure(nLane));
  FSMC_CUDA(plan->hapB.ensure(nLane));
  FSMC_CUDA(plan->tilePairs.ensure(T));
  FSMC_CUDA(plan->tileFrom.ensure(T));
  FSMC_CUDA(plan->tileTo.ensure(T));
  FSMC_CUDA(plan->order.ensure(T));
  FSMC_CUDA(plan->counters.ensure(2));
  if (T > 0) {
    FSMC_CUDA(cudaMemcpyAsync(plan->hapA.p, req->hapA, nLane * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaMemcpyAsync(plan->hapB.p, req->hapB, nLane * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaMemcpyAsync(plan->tilePairs.p, req->tilePairs, T * sizeof(int), cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaMemcpyAsync(plan->tileFrom.p, req->tileFrom, T * sizeof(int), cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaMemcpyAsync(plan->tileTo.p, req->tileTo, T * sizeof(int), cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaMemcpyAsync(plan->order.p, order.data(), T * sizeof(int), cudaMemcpyHostToDevice, st));
  }
  if (seg) {
    FSMC_CUDA(plan->scanFrom.ensure(T));
    FSMC_CUDA(plan->scanTo.ensure(T));
    FSMC_CUDA(plan->segments.ensure(plan->segmentCapacity));
    if (T > 0) {
      FSMC_CUDA(cudaMemcpyAsync(plan->scanFrom.p, req->tileScanFrom, T * sizeof(int), cudaMemcpyHostToDevice, st));
      FSMC_CUDA(cudaMemcpyAsync(plan->scanTo.p, req->tileScanTo, T * sizeof(int), cudaMemcpyHostToDevice, st));
    }
  }
  const size_t nSite = nLane * static_cast<size_t>(plan->siteStride);
  if (dev) {
    plan->outMean = dev->siteMean_dev;
    plan->outMap = dev->siteMap_dev;
    plan->outIbd = dev->siteIbd_dev;
    plan->outPosterior = dev->sitePosterior_dev;
    plan->outSum = dev->sumPosterior_dev;
    plan->hostLaneRow.assign(nLane, 0u);
    if (siteOut) {
      for (long long t = 0; t < T; ++t) {
        for (int l = 0; l < req->tilePairs[t]; ++l) {
          plan->hostLaneRow[t * 32 + l] = static_cast<uint32_t>(dev->laneRow[t * 32 + l]);
        }
      }
    }
    plan->hostWeight.assign(m.S, 1.f);
    if (dev->stateWeight) {
      std::copy(dev->stateWeight, dev->stateWeight + m.S, plan->hostWeight.begin());
    }
    FSMC_CUDA(plan->laneRow.ensure(nLane));
    FSMC_CUDA(plan->stateWeight.ensure(m.S));
    if (T > 0) {
      FSMC_CUDA(cudaMemcpyAsync(plan->laneRow.p, plan->hostLaneRow.data(), nLane * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    }
    FSMC_CUDA(cudaMemcpyAsync(plan->stateWeight.p, plan->hostWeight.data(), m.S * sizeof(float), cudaMemcpyHostToDevice, st));
  } else if (flags & FSMC_SITE_MEAN) {
    FSMC_CUDA(plan->siteMean.ensure(nSite));
  }
  if (!dev && (flags & FSMC_SITE_MAP)) {
    FSMC_CUDA(plan->siteMap.ensure(nSite));
  }
  if (!dev && (flags & FSMC_SITE_IBD)) {
    FSMC_CUDA(plan->siteIbd.ensure(nSite));
  }
  if (!dev && (flags & FSMC_SITE_POSTERIOR)) {
    FSMC_CUDA(plan->sitePosterior.ensure(nSite * static_cast<size_t>(ctx->model.S)));
  }
  if (!dev && (flags & FSMC_SUM_POSTERIOR)) {
    FSMC_CUDA(plan->sumPosterior.ensure(sumPosteriorCount(ctx->model, flags)));
  }
  plan->launched = false;
  plan->launches = 0;
  mark("buffers + uploads");

  // ---- launch geometry --------------------------------------------------------------------------
  const KernelChoice kc = chooseKernel(m.S, flags);
  // Sparse age estimates pay off when IBD runs cover a small part of the scan windows: whole-chromosome windows
  // (all-pairs decoding, hashing off).  The windows of hashing candidates lie mostly inside runs: dense kernel.
  // FSMC_SPARSE=0/1 overrides the window-length rule (development / tests).
  const bool preferSparse = T > 0 && sparsePreferred(scanSites / static_cast<double>(T));
  const FastChoice fc = chooseFastKernel(ctx->kernelModel, flags, preferSparse);
  plan->fast = fc.fn != nullptr;
  plan->sparse = fc.sparse;
  plan->statesKernel = plan->fast ? ctx->kernelModel.S : kc.statesKernel;
  plan->narrow = fc.narrow;
  plan->tileWarps = fc.splitWarps > 0 ? fc.splitWarps : 1;
  plan->mode = kc.mode;
  if (dev && (fc.narrow || fc.sparse)) {
    return fail(FSMC_E_INVALID, "fsmc_decode_device: flags 0x%x run a narrow kernel, which has no caller rows: set FSMC_SITE_MEAN, "
                "FSMC_SITE_MAP or FSMC_WIDE_KERNEL", flags);
  }
  // tiles in flight per CTA: one per warp, except for the state-split kernels (one tile per CTA)
  int warpsPerBlock = fc.splitWarps > 0 ? 1 : (plan->fast ? fc.threads : kc.threads) / 32;
  const size_t smemLimit = ctx->prop.sharedMemPerBlockOptin;
  int blocksPerSm = 0;
  if (plan->fast) {
    plan->threads = fc.threads;
    plan->smemBytes = fastSmemBytes(fc, ctx->kernelModel.S);
    FSMC_CUDA(residentBlocks(ctx, reinterpret_cast<const void*>(fc.fn), plan->threads, plan->smemBytes, &blocksPerSm));
  } else {
    const size_t perWarp = smemPerWarp(m, kc.mode, flags);
    while (warpsPerBlock > 1 && perWarp * warpsPerBlock > smemLimit) {
      warpsPerBlock /= 2;
    }
    if (perWarp * warpsPerBlock > smemLimit) {
      return fail(FSMC_E_INVALID, "fsmc_plan_create: %d states need %zu bytes of shared memory per warp (limit %zu)", m.S,
                  perWarp, smemLimit);
    }
    plan->threads = warpsPerBlock * 32;
    plan->smemBytes = perWarp * warpsPerBlock;
    FSMC_CUDA(residentBlocks(ctx, reinterpret_cast<const void*>(kc.fn), plan->threads, plan->smemBytes, &blocksPerSm));
  }
  if (blocksPerSm < 1) {
    return fail(FSMC_E_CUDA, "fsmc_plan_create: kernel does not fit on an SM (threads=%d smem=%zu)", plan->threads,
                plan->smemBytes);
  }
  long long blocks = static_cast<long long>(ctx->prop.multiProcessorCount) * blocksPerSm;
  blocks = std::min<long long>(blocks, (T + warpsPerBlock - 1) / warpsPerBlock);
  blocks = std::max<long long>(blocks, 1);

  plan->sumOnFast = fc.sum;
  if (fc.sum) {
    // private accumulators of the posterior sums, one per resident warp (allocated before the slabs are sized)
    const size_t perWarp = sumPosteriorCount(m, flags) / static_cast<size_t>(m.S) * static_cast<size_t>(fc.Spad);
    FSMC_CUDA(ctx->sumScratch.ensure(static_cast<size_t>(blocks) * warpsPerBlock * perWarp));
  }

  // backward-sweep scratch: one slab of maxLen*S*32 floats per resident warp.  Shrink the grid if
  // the slabs would not fit in 85% of the free memory.
  plan->scratchPerWarp = maxLen * (plan->fast ? (fc.narrow ? fc.recordQuads * 4 : fc.Spad) : m.S) * 32;
  const size_t slabBytes = static_cast<size_t>(plan->scratchPerWarp) * sizeof(float);
  // (the context's buffer already holds the full grid's slabs: nothing to size, no driver query)
  if (slabBytes > 0 && ctx->scratch.n < static_cast<size_t>(blocks) * warpsPerBlock * static_cast<size_t>(plan->scratchPerWarp)) {
    size_t freeB = 0, totalB = 0;
    FSMC_CUDA(cudaMemGetInfo(&freeB, &totalB));
    const size_t have = ctx->scratch.n * sizeof(float);
    const size_t budget = static_cast<size_t>(0.85 * static_cast<double>(freeB + have));
    long long maxWarps = static_cast<long long>(budget / slabBytes);
    if (maxWarps < 1) {
      return fail(FSMC_E_NOMEM, "fsmc_plan_create: a window of %lld sites needs a %zu-byte slab, %zu bytes free", maxLen,
                  slabBytes, freeB);
    }
    blocks = std::min<long long>(blocks, std::max<long long>(1, maxWarps / warpsPerBlock));
    if (blocks * warpsPerBlock > maxWarps) {
      return fail(FSMC_E_NOMEM, "fsmc_plan_create: not enough device memory for one block's scratch");
    }
    FSMC_CUDA(ctx->scratch.ensure(static_cast<size_t>(blocks) * warpsPerBlock * plan->scratchPerWarp));
  }

  plan->blocks = static_cast<int>(blocks);
  plan->tilesPerBlock = warpsPerBlock;
  mark("geometry + scratch");

  if (plan->sparse) {
    // ---- checkpoints, items and the refine pass (decode_sparse.cuh) -------------------------------------------------
    const size_t vecFloats = static_cast<size_t>(fc.Spad) * 32;
    // budget for the checkpoints: 45 % of what is free, or what the context already holds if that is more (then the
    // driver is not asked at all: cudaMemGetInfo costs milliseconds)
    double budget = static_cast<double>(ctx->ckptBeta.n * sizeof(float));
    bool asked = false;
    auto askBudget = [&]() -> cudaError_t {
      if (!asked) {
        size_t freeB = 0, totalB = 0;
        const cudaError_t e = cudaMemGetInfo(&freeB, &totalB);
        if (e != cudaSuccess) {
          return e;
        }
        budget = std::max(budget, 0.45 * static_cast<double>(freeB + ctx->ckptBeta.n * sizeof(float)));
        asked = true;
      }
      return cudaSuccess;
    };
    // blocks of 128 sites (measured on cfg2: 385 ms per step with blocks of 32 sites, 340 ms with 128: every block boundary
    // inside an IBD run costs the warp an item, and every block a checkpoint); coarser when the checkpoints of the whole
    // request would not fit
    int shift = 7;
    if (const char* e = std::getenv("FSMC_CKPT_SHIFT")) {
      shift = std::max(2, std::min(10, std::atoi(e)));
    }
    std::vector<long long> base(static_cast<size_t>(T) + 1, 0);
    for (;; ++shift) {
      long long slots = 0;
      for (long long t = 0; t < T; ++t) {
        base[t] = slots;
        slots += ((req->tileTo[t] - req->tileFrom[t] - 1) >> shift) + 1;  // blocks count from the window's first site
      }
      base[T] = slots;
      if (static_cast<double>(slots) * vecFloats * sizeof(float) <= budget || shift >= 12) {
        break;
      }
      if (!asked) {
        FSMC_CUDA(askBudget());
        --shift;  // try the same block size again with the real budget
      }
    }
    plan->ckptShift = shift;
    plan->ckptSlots = base[T];
    FSMC_CUDA(ctx->ckptBeta.ensure(static_cast<size_t>(plan->ckptSlots) * vecFloats));
    FSMC_CUDA(plan->tileCkptBase.ensure(static_cast<size_t>(T) + 1));
    FSMC_CUDA(cudaMemcpyAsync(plan->tileCkptBase.p, base.data(), (static_cast<size_t>(T) + 1) * sizeof(long long),
                              cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaStreamSynchronize(st));  // `base` goes out of scope
    FSMC_CUDA(plan->alphaScratch.ensure(static_cast<size_t>(blocks) * warpsPerBlock * vecFloats));
    FSMC_CUDA(plan->counters.ensure(4));
    // items: one per (run, block).  Start from one item per 512 pair-sites (all-pairs data sets have one per ~1500);
    // fsmc_plan_collect re-runs the request with a larger buffer if that was not enough.
    if (plan->itemCapacity == 0) {
      plan->itemCapacity = std::max<long long>(1 << 16, static_cast<long long>(pairSites / 512.0));
    }
    if (const char* e = std::getenv("FSMC_ITEM_CAPACITY")) {  // tests: force the overflow / re-run path
      plan->itemCapacity = std::max<long long>(1, std::atoll(e));
    }
    plan->itemCapacity = std::min<long long>(plan->itemCapacity, 0x7ffffff0ll);
    // refine pass geometry
    auto refineFn = fsmc::refineKernel<69, fsmc::kRefineDepth, kFastRescale, 128, 2>;
    plan->refineSmem = 4 * (fsmc::kRefineDepth * (vecFloats * 4 + static_cast<size_t>(fsmc::kRowArrays) * fc.Spad * 4)) +
                       4 * 2 * fsmc::kRefineDepth * sizeof(uint64_t);
    int perSm = 0;
    FSMC_CUDA(residentBlocks(ctx, reinterpret_cast<const void*>(refineFn), 128, plan->refineSmem, &perSm));
    if (perSm < 1) {
      return fail(FSMC_E_CUDA, "fsmc_plan_create: refine kernel does not fit on an SM (smem=%zu)", plan->refineSmem);
    }
    plan->refineBlocks = ctx->prop.multiProcessorCount * perSm;
    const size_t refineScratch = static_cast<size_t>(plan->refineBlocks) * 4 * (size_t{1} << shift) * vecFloats;
    FSMC_CUDA(ctx->scratch.ensure(std::max<size_t>(refineScratch, static_cast<size_t>(blocks) * static_cast<size_t>(warpsPerBlock) * static_cast<size_t>(plan->scratchPerWarp))));
    mark("sparse buffers");
  }
  guard.keep = true;
  *out = plan;
  return FSMC_OK;
}

int fsmc_plan_create(fsmc_ctx* ctx, const fsmc_decode_request* req, fsmc_plan** out)
{
  return planCreate(ctx, req, nullptr, out);
}

namespace
{
// item buffers of a sparse plan, (re)sized to plan->itemCapacity
int allocateItems(fsmc_plan* plan, const int Spad)
{
  const size_t cap = static_cast<size_t>(plan->itemCapacity);
  FSMC_CUDA(plan->items.ensure(cap));
  FSMC_CUDA(plan->itemAlpha.ensure(cap * Spad));
  FSMC_CUDA(plan->itemSums.ensure(cap * Spad));
  FSMC_CUDA(plan->itemKeys.ensure(4 * cap));
  size_t bytes = 0;
  uint32_t* k = plan->itemKeys.p;
  FSMC_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, bytes, k, k, k, k, static_cast<int>(cap)));
  FSMC_CUDA(plan->sortTemp.ensure(bytes));
  plan->sortTempBytes = bytes;
  return FSMC_OK;
}
}  // namespace

int fsmc_plan_launch(fsmc_ctx* ctx, fsmc_plan* plan)
{
  if (!ctx || !plan) {
    return fail(FSMC_E_INVALID, "fsmc_plan_launch: NULL argument");
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const DeviceModel& m = plan->fast ? ctx->kernelModel : ctx->model;  // the specialised kernels see the padded model
  FSMC_CUDA(cudaEventRecord(ctx->ev[1], st));
  plan->launches = 0;
  if (plan->numTiles > 0) {
    FSMC_CUDA(cudaMemsetAsync(plan->counters.p, 0, (plan->sparse ? 4 : 2) * sizeof(unsigned long long), st));
    DecodeArgs a{};
    if (plan->sparse) {
      const int rc = allocateItems(plan, m.Spad);
      if (rc != FSMC_OK) {
        return rc;
      }
      a.ckptShift = plan->ckptShift;
      a.tileCkptBase = plan->tileCkptBase.p;
      a.ckptBeta = ctx->ckptBeta.p;
      a.alphaScratch = plan->alphaScratch.p;
      a.items = plan->items.p;
      a.itemAlpha = plan->itemAlpha.p;
      a.itemSums = plan->itemSums.p;
      a.itemCount = plan->counters.p + 2;
      a.itemCapacity = plan->itemCapacity;
      a.itemOrder = plan->itemKeys.p + 3 * static_cast<size_t>(plan->itemCapacity);
      a.refineCounter = plan->counters.p + 3;
    }
    a.hapA = plan->hapA.p;
    a.hapB = plan->hapB.p;
    a.tilePairs = plan->tilePairs.p;
    a.tileFrom = plan->tileFrom.p;
    a.tileTo = plan->tileTo.p;
    a.tileScanFrom = plan->scanFrom.p;
    a.tileScanTo = plan->scanTo.p;
    a.order = plan->order.p;
    a.numTiles = plan->numTiles;
    a.flags = plan->flags;
    a.segments = plan->segments.p;
    a.segmentCount = plan->counters.p;
    a.segmentCapacity = plan->segmentCapacity;
    const bool dev = plan->deviceOut;
    a.siteMean = dev ? plan->outMean : plan->siteMean.p;
    a.siteMap = dev ? plan->outMap : plan->siteMap.p;
    a.siteIbd = dev ? plan->outIbd : plan->siteIbd.p;
    a.sitePosterior = dev ? plan->outPosterior : plan->sitePosterior.p;
    a.sumPosterior = dev ? plan->outSum : plan->sumPosterior.p;
    a.laneRow = dev ? plan->laneRow.p : nullptr;
    a.stateWeight = dev ? plan->stateWeight.p : nullptr;
    const int sumPlanes = (plan->flags & FSMC_SUM_BY_GENOTYPE) ? 3 : 1;
    const int sumWarps = plan->blocks * plan->tilesPerBlock;
    if (plan->flags & FSMC_SUM_POSTERIOR) {
      if (!dev) {  // the caller's sums are added to
        FSMC_CUDA(cudaMemsetAsync(plan->sumPosterior.p, 0, sumPosteriorCount(ctx->model, plan->flags) * sizeof(float), st));
      }
      if (plan->sumOnFast) {
        a.sumScratch = ctx->sumScratch.p;
        FSMC_CUDA(cudaMemsetAsync(ctx->sumScratch.p, 0, static_cast<size_t>(sumWarps) * sumPlanes * m.L * m.Spad * sizeof(float), st));
      }
    }
    a.siteStride = plan->siteStride;
    a.scratch = ctx->scratch.p;
    a.scratchPerWarp = plan->scratchPerWarp;
    a.tileCounter = plan->counters.p + 1;
    a.accScratch = nullptr;
    if (plan->fast) {
      fsmc::FastModel fm{};
      fm.base = m;
      std::copy(ctx->hostColRatios.begin(), ctx->hostColRatios.end(), fm.colRatios);
      std::copy(ctx->hostExpTimes.begin(), ctx->hostExpTimes.end(), fm.expTimes);
      std::copy(ctx->hostPrior.begin(), ctx->hostPrior.end(), fm.prior);
      const FastChoice fc = chooseFastKernel(m, plan->flags, plan->sparse);
      fc.fn<<<plan->blocks, plan->threads, plan->smemBytes, st>>>(fm, a);
      if (plan->sumOnFast) {
        fsmc::sumScratchReduceKernel<<<ctx->prop.multiProcessorCount * 8, 256, 0, st>>>(ctx->sumScratch.p, sumWarps, sumPlanes, m.L,
                                                                                        ctx->model.S, m.Spad, a.sumPosterior,
                                                                                        a.stateWeight);
        plan->launches += 1;
      }
      if (plan->sparse) {
        // items by block, full posteriors inside the items, age estimates of the segments
        const long long cap = plan->itemCapacity;
        uint32_t* keys = plan->itemKeys.p;
        uint32_t* keysOut = keys + cap;
        uint32_t* index = keys + 2 * cap;
        uint32_t* indexOut = keys + 3 * cap;
        const int kb = static_cast<int>(std::min<long long>((cap + 255) / 256, ctx->prop.multiProcessorCount * 8ll));
        fsmc::itemKeysKernel<<<kb, 256, 0, st>>>(a.items, a.itemCount, cap, a.tileFrom, plan->ckptShift, keys, index);
        size_t bytes = plan->sortTempBytes;
        FSMC_CUDA(cub::DeviceRadixSort::SortPairs(plan->sortTemp.p, bytes, keys, keysOut, index, indexOut, static_cast<int>(cap), 0, 32, st));
        DecodeArgs r = a;
        r.scratchPerWarp = (1ll << plan->ckptShift) * m.Spad * 32;
        fsmc::refineKernel<69, fsmc::kRefineDepth, kFastRescale, 128, 2><<<plan->refineBlocks, 128, plan->refineSmem, st>>>(fm, r);
        fsmc::finalizeSegmentsKernel<<<ctx->prop.multiProcessorCount * 8, 256, 0, st>>>(m, a.segments, a.segmentCount, a.segmentCapacity,
                                                                                          a.items, a.itemSums, a.itemCount, cap);
        plan->launches += 4;
      }
    } else {
      const KernelChoice kc = chooseKernel(m.S, plan->flags);
      kc.fn<<<plan->blocks, plan->threads, plan->smemBytes, st>>>(m, a);
    }
    FSMC_CUDA(cudaGetLastError());
    plan->launches += 1;
  }
  FSMC_CUDA(cudaEventRecord(ctx->ev[2], st));
  plan->launched = true;
  return FSMC_OK;
}

namespace
{
void fillStats(fsmc_ctx* ctx, const fsmc_plan* plan, long long found, int64_t d2h, fsmc_decode_stats* stats);
}  // namespace

int fsmc_plan_collect(fsmc_ctx* ctx, fsmc_plan* plan, const fsmc_decode_request* out, fsmc_decode_stats* stats)
{
  if (!ctx || !plan || !out) {
    return fail(FSMC_E_INVALID, "fsmc_plan_collect: NULL argument");
  }
  if (!plan->launched) {
    return fail(FSMC_E_STATE, "fsmc_plan_collect: plan was not launched");
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const unsigned flags = plan->flags;
  unsigned long long counters[4] = {0, 0, 0, 0};
  for (;;) {
    if (plan->numTiles > 0) {
      FSMC_CUDA(cudaMemcpyAsync(counters, plan->counters.p, (plan->sparse ? 4 : 2) * sizeof(unsigned long long),
                                cudaMemcpyDeviceToHost, st));
    }
    FSMC_CUDA(cudaStreamSynchronize(st));
    plan->itemsFound = static_cast<long long>(counters[2]);
    if (!plan->sparse || plan->itemsFound <= plan->itemCapacity) {
      break;
    }
    // more run pieces than item slots: run the request again with enough of them (the launch re-allocates)
    if (plan->itemsFound >= 0x7ffffff0ll) {
      return fail(FSMC_E_NOMEM, "fsmc_plan_collect: %lld run pieces in one request; decode fewer tiles per call", plan->itemsFound);
    }
    plan->itemCapacity = std::min<long long>(plan->itemsFound + plan->itemsFound / 8 + 1024, 0x7ffffff0ll);
    const int rc = fsmc_plan_launch(ctx, plan);
    if (rc != FSMC_OK) {
      return rc;
    }
  }
  const long long found = static_cast<long long>(counters[0]);
  const long long stored = std::min<long long>(found, plan->segmentCapacity);
  int rc = FSMC_OK;
  int64_t d2h = 0;
  if (flags & FSMC_CALL_SEGMENTS) {
    if (stored > 0) {
      if (!out->segments || out->segmentCapacity < stored) {
        return fail(FSMC_E_INVALID, "fsmc_plan_collect: segment buffer missing or smaller than at plan creation");
      }
      // reference order = ascending (pair, first site): stable sort by pair on the device (a lane appends its
      // segments in ascending site order), then one copy into pinned staging
      const fsmc_segment* sorted = nullptr;
      FSMC_CUDA(ctx->segmentSorter.sort(plan->segments.p, stored, static_cast<uint32_t>(plan->numTiles * 32), st, &sorted));
      FSMC_CUDA(ctx->segStage.ensure(static_cast<size_t>(stored)));
      FSMC_CUDA(cudaMemcpyAsync(ctx->segStage.p, sorted, stored * sizeof(fsmc_segment), cudaMemcpyDeviceToHost, st));
      d2h += stored * static_cast<int64_t>(sizeof(fsmc_segment));
    }
  }
  const size_t nSite = static_cast<size_t>(plan->numTiles) * 32 * static_cast<size_t>(plan->siteStride);
  if ((flags & FSMC_SITE_MEAN) && nSite) {
    if (!out->siteMean) {
      return fail(FSMC_E_INVALID, "fsmc_plan_collect: siteMean is NULL");
    }
    FSMC_CUDA(cudaMemcpyAsync(out->siteMean, plan->siteMean.p, nSite * sizeof(float), cudaMemcpyDeviceToHost, st));
    d2h += nSite * sizeof(float);
  }
  if ((flags & FSMC_SITE_MAP) && nSite) {
    if (!out->siteMap) {
      return fail(FSMC_E_INVALID, "fsmc_plan_collect: siteMap is NULL");
    }
    FSMC_CUDA(cudaMemcpyAsync(out->siteMap, plan->siteMap.p, nSite * sizeof(int), cudaMemcpyDeviceToHost, st));
    d2h += nSite * sizeof(int);
  }
  if ((flags & FSMC_SITE_IBD) && nSite) {
    if (!out->siteIbd) {
      return fail(FSMC_E_INVALID, "fsmc_plan_collect: siteIbd is NULL");
    }
    FSMC_CUDA(cudaMemcpyAsync(out->siteIbd, plan->siteIbd.p, nSite * sizeof(float), cudaMemcpyDeviceToHost, st));
    d2h += nSite * sizeof(float);
  }
  if ((flags & FSMC_SITE_POSTERIOR) && nSite) {
    if (!out->sitePosterior) {
      return fail(FSMC_E_INVALID, "fsmc_plan_collect: sitePosterior is NULL");
    }
    FSMC_CUDA(cudaMemcpyAsync(out->sitePosterior, plan->sitePosterior.p,
                              nSite * static_cast<size_t>(ctx->model.S) * sizeof(float), cudaMemcpyDeviceToHost, st));
    d2h += nSite * static_cast<size_t>(ctx->model.S) * sizeof(float);
  }
  if (flags & FSMC_SUM_POSTERIOR) {
    if (!out->sumPosterior) {
      return fail(FSMC_E_INVALID, "fsmc_plan_collect: sumPosterior is NULL");
    }
    FSMC_CUDA(cudaMemcpyAsync(out->sumPosterior, plan->sumPosterior.p, sumPosteriorCount(ctx->model, flags) * sizeof(float),
                              cudaMemcpyDeviceToHost, st));
    d2h += sumPosteriorCount(ctx->model, flags) * sizeof(float);
  }
  FSMC_CUDA(cudaEventRecord(ctx->ev[3], st));
  FSMC_CUDA(cudaStreamSynchronize(st));
  if (stored > 0) {
    // the records arrive sorted by pair (device radix sort); copy them out and check the order, sites included
    const fsmc_segment* in = ctx->segStage.p;
    const size_t nPairs = static_cast<size_t>(plan->numTiles) * 32;
    std::memcpy(out->segments, in, static_cast<size_t>(stored) * sizeof(fsmc_segment));
    bool ordered = true;
    for (long long i = 0; i < stored; ++i) {
      if (in[i].pair >= nPairs) {
        return fail(FSMC_E_CUDA, "fsmc_plan_collect: corrupt segment record (pair %u of %zu)", in[i].pair, nPairs);
      }
      if (i > 0 && (in[i - 1].pair > in[i].pair || (in[i - 1].pair == in[i].pair && in[i - 1].posStart > in[i].posStart))) {
        ordered = false;
      }
    }
    if (!ordered) {  // never taken by the kernels of this library (one lane emits a pair's segments in site order)
      std::stable_sort(out->segments, out->segments + stored, [](const fsmc_segment& x, const fsmc_segment& y) {
        return x.pair != y.pair ? x.pair < y.pair : x.posStart < y.posStart;
      });
    }
  }
  if (found > plan->segmentCapacity) {
    rc = fail(FSMC_E_OVERFLOW, "fsmc_plan_collect: %lld segments found, capacity %lld", found, plan->segmentCapacity);
  }
  fillStats(ctx, plan, found, d2h, stats);
  plan->launched = false;
  return rc;
}

namespace
{
void fillStats(fsmc_ctx* ctx, const fsmc_plan* plan, const long long found, const int64_t d2h, fsmc_decode_stats* stats)
{
  if (stats) {
    stats->numSegments = found;
    stats->pairSites = plan->pairSites;
    stats->kernelMs = 0.f;
    stats->totalMs = 0.f;
    cudaEventElapsedTime(&stats->kernelMs, ctx->ev[1], ctx->ev[2]);
    if (cudaEventElapsedTime(&stats->totalMs, ctx->ev[0], ctx->ev[3]) != cudaSuccess) {
      cudaGetLastError();
      stats->totalMs = 0.f;
    }
    stats->kernelLaunches = plan->launches;
    stats->statesKernel = plan->statesKernel;
    stats->narrowKernel = plan->narrow ? 1 : 0;
    stats->tileWarps = plan->tileWarps;
    stats->scratchBytes = static_cast<int64_t>(plan->scratchPerWarp) * sizeof(float) * plan->blocks * plan->tilesPerBlock;
    stats->sparseKernel = plan->sparse ? 1 : 0;
    stats->sparseItems = plan->sparse ? plan->itemsFound : 0;
    stats->checkpointBytes = plan->sparse ? plan->ckptSlots * static_cast<int64_t>(ctx->kernelModel.Spad) * 32 * 4 : 0;
    stats->checkpointSites = plan->sparse ? (1 << plan->ckptShift) : 0;
    stats->d2hBytes = d2h;
  }
}
}  // namespace

int fsmc_plan_destroy(fsmc_ctx* ctx, fsmc_plan* plan)
{
  if (ctx) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (plan && !ctx->sparePlan) {
      ctx->sparePlan = plan;  // keeps its device buffers for the next plan
      return FSMC_OK;
    }
  }
  delete plan;
  return FSMC_OK;
}


int fsmc_seed(fsmc_ctx* ctx, const fsmc_seed_params* sp, fsmc_match* out, const int64_t capacity,
              fsmc_seed_stats* stats)
{
  if (!ctx || !sp || capacity < 0 || (capacity > 0 && !out)) {
    return fail(FSMC_E_INVALID, "fsmc_seed: NULL argument or negative capacity");
  }
  if (!ctx->hasHaps) {
    return fail(FSMC_E_STATE, "fsmc_seed: set the haplotypes first");
  }
  if (!sp->geneticPositions || !sp->globalHapId || sp->gap < 0) {
    return fail(FSMC_E_INVALID, "fsmc_seed: geneticPositions / globalHapId missing or negative gap");
  }
  if (sp->maxSeeds < 0 || (sp->maxSeeds > 0 && (sp->readAhead < 1 || sp->readAhead > 127))) {
    return fail(FSMC_E_INVALID, "fsmc_seed: maxSeeds must be >= 0 and, when set, readAhead in [1, 127]");
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const uint32_t H = static_cast<uint32_t>(ctx->numHaps);
  const int L = static_cast<int>(ctx->sites);
  const int W = L / 64;  // a trailing partial word is never hashed
  const bool refOrder = sp->flags & FSMC_SEED_REFERENCE_ORDER;
  // A call that overflowed the caller's buffer leaves its result on the device; the retry with a larger buffer and the
  // same inputs only copies it out.  "Same inputs" = same scalar parameters and same CONTENTS of the two arrays (a
  // checksum, not their addresses: a caller may reuse a buffer for other data).
  auto checksum = [](const void* p, const size_t bytes) {
    uint64_t h = 1469598103934665603ull;
    const unsigned char* c = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < bytes; ++i) {
      h = (h ^ c[i]) * 1099511628211ull;
    }
    return h;
  };
  SeedKey key;
  std::memset(&key, 0, sizeof key);
  key.gap = sp->gap;
  key.minLengthCm = sp->minLengthCm;
  key.genPosSum = checksum(sp->geneticPositions, sizeof(float) * static_cast<size_t>(L));
  key.globalIdSum = checksum(sp->globalHapId, sizeof(uint32_t) * H);
  key.flipSum = (refOrder && sp->flipMask) ? checksum(sp->flipMask, sizeof(uint64_t) * static_cast<size_t>(std::max(W, 0))) : 0;
  key.skip = sp->skip;
  key.window[0] = sp->loI;
  key.window[1] = sp->hiI;
  key.window[2] = sp->loJ;
  key.window[3] = sp->hiJ;
  key.lastJob = sp->lastJob;
  key.aboveDiag = sp->aboveDiag;
  key.flags = sp->flags;
  key.maxSeeds = sp->maxSeeds;
  key.readAhead = sp->readAhead;
  const bool cacheHit = ctx->seedCacheValid && std::memcmp(&key, &ctx->seedCacheKey, sizeof key) == 0 &&
                        capacity >= ctx->seedCacheStats.numMatches;
  if (!cacheHit) {
    ctx->seedCacheValid = false;
    ctx->orderedOut = nullptr;
    uint32_t C = 64;
    while (C < 2u * H) {
      C <<= 1;
    }
    const size_t maxGroups = H / 2 + 2;
    // Words are independent, so a launch handles a batch of them (blockIdx.y = word in the batch), each with its own
    // slice of the scratch tables: at small sample counts the per-word kernels are a few microseconds of work and the
    // pass would otherwise be bound by launch latency (5 launches per word).  The batch is as large as 2 GiB of tables
    // allow, up to 64 words.
    const size_t perWordBytes = static_cast<size_t>(C) * 12 + static_cast<size_t>(H) * 12 + maxGroups * 16 + 40;
    const int WB = static_cast<int>(std::max<size_t>(1, std::min<size_t>({64, static_cast<size_t>(std::max(W, 1)),
                                                                         (size_t{2} << 30) / perWordBytes})));
    FSMC_CUDA(ctx->seedKeysT.ensure(static_cast<size_t>(std::max(W, 1)) * H));
    FSMC_CUDA(ctx->seedOwner.ensure(static_cast<size_t>(WB) * C));
    FSMC_CUDA(ctx->seedSlotCount.ensure(static_cast<size_t>(WB) * C));
    FSMC_CUDA(ctx->seedSlotGroup.ensure(static_cast<size_t>(WB) * C));
    FSMC_CUDA(ctx->seedSlotOf.ensure(static_cast<size_t>(WB) * H));
    FSMC_CUDA(ctx->seedRankOf.ensure(static_cast<size_t>(WB) * H));
    FSMC_CUDA(ctx->seedMembers.ensure(static_cast<size_t>(WB) * H));
    FSMC_CUDA(ctx->seedGroupSize.ensure(static_cast<size_t>(WB) * maxGroups));
    FSMC_CUDA(ctx->seedGroupMemberBase.ensure(static_cast<size_t>(WB) * maxGroups));
    FSMC_CUDA(ctx->seedGroupPairBase.ensure(static_cast<size_t>(WB) * (maxGroups + 1)));
    FSMC_CUDA(ctx->seedWordCounters.ensure(static_cast<size_t>(WB) * 4));
    FSMC_CUDA(ctx->seedChunkBase.ensure(static_cast<size_t>(WB) + 2));
    FSMC_CUDA(ctx->seedCounters.ensure(8));
    FSMC_CUDA(ctx->seedGenPos.ensure(L));
    FSMC_CUDA(ctx->seedGlobalId.ensure(H));
    // device-side interval buffer: at least 16 Mi intervals (256 MiB) whatever the caller's capacity, so that an
    // under-sized first call does not have to be recomputed.  In reference-order mode every interval of the job is
    // needed on the device (the caller's capacity only counts candidates): an eighth of the free memory to begin with.
    size_t freeB = 0, totalB = 0;
    FSMC_CUDA(cudaMemGetInfo(&freeB, &totalB));
    const long long avail = static_cast<long long>((freeB + ctx->seedOut.n * sizeof(fsmc_match)) / sizeof(fsmc_match));
    long long devCap = refOrder ? std::max<long long>(1ll << 20, std::min<long long>(avail / 8, 0x7ffffff0ll))
                                : std::max<long long>(capacity, std::min<long long>(1ll << 24, avail / 4));
    FSMC_CUDA(ctx->seedOut.ensure(static_cast<size_t>(devCap)));
    FSMC_CUDA(cudaMemcpyAsync(ctx->seedGenPos.p, sp->geneticPositions, sizeof(float) * L, cudaMemcpyHostToDevice, st));
    FSMC_CUDA(cudaMemcpyAsync(ctx->seedGlobalId.p, sp->globalHapId, sizeof(uint32_t) * H, cudaMemcpyHostToDevice, st));

    fsmc::SeedArgs a{};
    a.haps = ctx->haps.p;
    a.wordsPerHap = ctx->model.wordsPerHap;
    a.keysT = ctx->seedKeysT.p;
    a.H = H;
    a.W = W;
    a.L = L;
    a.gap = sp->gap;
    a.minLengthCm = sp->minLengthCm;
    a.genPos = ctx->seedGenPos.p;
    a.globalId = ctx->seedGlobalId.p;
    a.loI = sp->loI;
    a.hiI = sp->hiI;
    a.loJ = sp->loJ;
    a.hiJ = sp->hiJ;
    a.lastJob = sp->lastJob;
    a.aboveDiag = sp->aboveDiag;
    a.flags = sp->flags | (refOrder ? FSMC_SEED_ALL_INTERVALS : 0u);
    a.owner = ctx->seedOwner.p;
    a.slotCount = ctx->seedSlotCount.p;
    a.slotGroup = ctx->seedSlotGroup.p;
    a.C = C;
    a.slotOf = ctx->seedSlotOf.p;
    a.rankOf = ctx->seedRankOf.p;
    a.groupSize = ctx->seedGroupSize.p;
    a.groupMemberBase = ctx->seedGroupMemberBase.p;
    a.groupPairBase = ctx->seedGroupPairBase.p;
    a.members = ctx->seedMembers.p;
    a.maxGroups = static_cast<uint32_t>(maxGroups);
    a.wordCounters = ctx->seedWordCounters.p;
    a.batchChunkBase = ctx->seedChunkBase.p;
    a.counters = ctx->seedCounters.p;

    int launches = 0;
    FSMC_CUDA(cudaEventRecord(ctx->ev[1], st));
    const int sms = ctx->prop.multiProcessorCount;
    if (W > 0) {
      const dim3 tb(32, 8), tg((H + 31) / 32, (W + 31) / 32);
      fsmc::transposeWordsKernel<<<tg, tb, 0, st>>>(a.haps, a.wordsPerHap, H, W, ctx->seedKeysT.p);
      ++launches;
    }
    // reference order: the seed map's iteration ranks (host threads, SeedMapOrder.hpp) are computed from the transposed
    // words while the device runs the pair kernels
    std::vector<uint64_t> hostKeys;
    std::vector<uint32_t> hostRank;
    std::thread rankThread;
    double rankMs = 0.0;
    const bool useSkip = sp->skip > 0.f;
    if ((refOrder || useSkip) && W > 0) {
      hostKeys.resize(static_cast<size_t>(W) * H);
      FSMC_CUDA(cudaMemcpyAsync(hostKeys.data(), ctx->seedKeysT.p, hostKeys.size() * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
      FSMC_CUDA(cudaStreamSynchronize(st));
    }
    a.lowComplexity = nullptr;
    if (useSkip && W > 0) {
      // ref: FastSMC.cpp:208-219 — float(#distinct words) / float(#haplotypes) > skip, else the word is skipped
      std::vector<unsigned char> lc(static_cast<size_t>(W), 0);
      const float skip = sp->skip;
      candidate_order::parallelForWords(W, 0, [&](const int w) {
        std::vector<uint64_t> keys(hostKeys.begin() + static_cast<size_t>(w) * H, hostKeys.begin() + static_cast<size_t>(w + 1) * H);
        std::sort(keys.begin(), keys.end());
        const size_t distinct = static_cast<size_t>(std::unique(keys.begin(), keys.end()) - keys.begin());
        lc[w] = !(static_cast<float>(static_cast<int>(distinct)) / static_cast<float>(H) > skip);
      });
      FSMC_CUDA(ctx->seedLowComplexity.ensure(static_cast<size_t>(W)));
      FSMC_CUDA(cudaMemcpyAsync(ctx->seedLowComplexity.p, lc.data(), lc.size(), cudaMemcpyHostToDevice, st));
      FSMC_CUDA(cudaStreamSynchronize(st));
      a.lowComplexity = ctx->seedLowComplexity.p;
    }
    if (refOrder && W > 0) {
      const uint64_t* flip = sp->flipMask;
      const int maxSeeds = sp->maxSeeds, readAhead = sp->readAhead;
      rankThread = std::thread([&hostKeys, &hostRank, &rankMs, flip, H, W, maxSeeds, readAhead] {
        const auto t0 = std::chrono::steady_clock::now();
        hostRank = candidate_order::seedGroupRanks(
            H, W, [&](const uint32_t h, const int w) { return hostKeys[static_cast<size_t>(w) * H + h] ^ (flip ? flip[w] : 0ull); }, 0,
            maxSeeds, readAhead);
        rankMs = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      });
    }
    struct Joiner {
      std::thread& t;
      ~Joiner()
      {
        if (t.joinable()) {
          t.join();
        }
      }
    } joiner{rankThread};
    // max_seeds > 0: registration keys of every (word, haplotype) replace the words (seed_kernels.cuh)
    a.nested = 0;
    a.maxDepth = 0;
    if (sp->maxSeeds > 0 && W > 0) {
      const size_t WH = static_cast<size_t>(W) * H;
      FSMC_CUDA(ctx->seedRep0.ensure(WH));
      FSMC_CUDA(ctx->seedCur.ensure(WH));
      FSMC_CUDA(ctx->seedDepth.ensure(WH));
      FSMC_CUDA(ctx->seedRegKeyT.ensure(WH));
      FSMC_CUDA(ctx->seedRegKeys.ensure(WH));
      fsmc::NestArgs na{};
      na.H = H;
      na.W = W;
      na.C = C;
      na.maxSeeds = sp->maxSeeds;
      na.readAhead = sp->readAhead;
      na.owner = a.owner;
      na.slotCount = a.slotCount;
      na.slotOf = a.slotOf;
      na.rep0 = ctx->seedRep0.p;
      na.cur = ctx->seedCur.p;
      na.depth = ctx->seedDepth.p;
      na.pending = ctx->seedCounters.p + 7;
      na.regKeyT = ctx->seedRegKeyT.p;
      for (int level = 0; level < sp->readAhead; ++level) {
        FSMC_CUDA(cudaMemsetAsync(na.pending, 0, sizeof(unsigned long long), st));
        na.level = level;
        for (int w0 = 0; w0 < W; w0 += WB) {
          const unsigned nw = static_cast<unsigned>(std::min(WB, W - w0));
          const long long perWordCap = std::max<long long>(1, sms * 8ll / nw);
          const unsigned hapBlocks = static_cast<unsigned>(std::min<long long>((H + 255ll) / 256, perWordCap));
          a.wordBase = na.wordBase = w0;
          a.wordsInBatch = static_cast<int>(nw);
          FSMC_CUDA(cudaMemsetAsync(a.owner, 0, sizeof(uint32_t) * C * nw, st));
          FSMC_CUDA(cudaMemsetAsync(a.slotCount, 0, sizeof(uint32_t) * C * nw, st));
          if (level == 0) {
            fsmc::groupInsertKernel<<<dim3(hapBlocks, nw), 256, 0, st>>>(a);
            fsmc::nestLevel0Kernel<<<dim3(hapBlocks, nw), 256, 0, st>>>(na);
          } else {
            fsmc::nestInsertKernel<<<dim3(hapBlocks, nw), 256, 0, st>>>(na);
            fsmc::nestFinishKernel<<<dim3(hapBlocks, nw), 256, 0, st>>>(na);
          }
          launches += 2;
        }
        unsigned long long pending = 0;
        FSMC_CUDA(cudaMemcpyAsync(&pending, na.pending, sizeof pending, cudaMemcpyDeviceToHost, st));
        FSMC_CUDA(cudaStreamSynchronize(st));
        if (pending == 0) {
          break;
        }
      }
      fsmc::nestEmitKernel<<<sms * 4, 256, 0, st>>>(na);
      const dim3 tb(32, 8), tg((H + 31) / 32, (W + 31) / 32);
      fsmc::transposeKeysBackKernel<<<tg, tb, 0, st>>>(ctx->seedRegKeyT.p, H, W, ctx->seedRegKeys.p);
      launches += 2;
      FSMC_CUDA(cudaGetLastError());
      a.keysT = ctx->seedRegKeyT.p;
      a.haps = ctx->seedRegKeys.p;
      a.wordsPerHap = W;
      a.nested = 1;
      a.maxDepth = sp->readAhead - 1;
    }
    unsigned long long counters[8] = {0};
    for (int attempt = 0; attempt < 2; ++attempt) {
      a.out = ctx->seedOut.p;
      a.capacity = devCap;
      FSMC_CUDA(cudaMemsetAsync(ctx->seedCounters.p, 0, 8 * sizeof(unsigned long long), st));
      for (int w0 = 0; w0 < W; w0 += WB) {
        const unsigned nw = static_cast<unsigned>(std::min(WB, W - w0));
        // grid.x: enough CTAs per word to cover it, but no more than ~8 CTAs per SM over the whole batch
        const long long perWordCap = std::max<long long>(1, sms * 8ll / nw);
        const unsigned hapBlocks = static_cast<unsigned>(std::min<long long>((H + 255ll) / 256, perWordCap));
        const unsigned slotBlocks = static_cast<unsigned>(std::min<long long>((C + 255ll) / 256, perWordCap));
        a.wordBase = w0;
        a.wordsInBatch = static_cast<int>(nw);
        FSMC_CUDA(cudaMemsetAsync(a.owner, 0, sizeof(uint32_t) * C * nw, st));
        FSMC_CUDA(cudaMemsetAsync(a.slotCount, 0, sizeof(uint32_t) * C * nw, st));
        FSMC_CUDA(cudaMemsetAsync(a.wordCounters, 0, sizeof(unsigned long long) * 4 * nw, st));
        fsmc::groupInsertKernel<<<dim3(hapBlocks, nw), 256, 0, st>>>(a);
        fsmc::groupCompactKernel<<<dim3(slotBlocks, nw), 256, 0, st>>>(a);
        fsmc::groupScanKernel<<<nw, 1024, 0, st>>>(a);
        fsmc::groupScatterKernel<<<dim3(hapBlocks, nw), 256, 0, st>>>(a);
        fsmc::batchChunksKernel<<<1, 32, 0, st>>>(a);
        if (a.nested) {
          fsmc::pairExtendKernel<true><<<sms * 8, fsmc::kPairBlockThreads, 0, st>>>(a);
        } else {
          fsmc::pairExtendKernel<false><<<sms * 8, fsmc::kPairBlockThreads, 0, st>>>(a);
        }
        launches += 6;
      }
      FSMC_CUDA(cudaGetLastError());
      FSMC_CUDA(cudaMemcpyAsync(counters, ctx->seedCounters.p, sizeof counters, cudaMemcpyDeviceToHost, st));
      FSMC_CUDA(cudaStreamSynchronize(st));
      if (!refOrder || static_cast<long long>(counters[3]) <= devCap) {
        break;
      }
      // reference order needs every interval on the device: run the pass again with a buffer of the right size
      devCap = static_cast<long long>(counters[3]) + 1024;
      if (devCap >= 0x7fffffffll) {
        return fail(FSMC_E_NOMEM, "fsmc_seed: %llu intervals in one job exceed the 2^31 limit of the device ordering; use more jobs",
                    counters[3]);
      }
      FSMC_CUDA(ctx->seedOut.ensure(static_cast<size_t>(devCap)));
    }
    FSMC_CUDA(cudaEventRecord(ctx->ev[2], st));
    FSMC_CUDA(cudaStreamSynchronize(st));
    fsmc_seed_stats& cs = ctx->seedCacheStats;
    cs = fsmc_seed_stats{};
    cs.numMatches = static_cast<int64_t>(counters[3]);
    cs.numIntervals = cs.numMatches;
    cs.pairVisits = static_cast<int64_t>(counters[4]);
    cs.numStarts = static_cast<int64_t>(counters[5]);
    cs.numWords = W;
    cs.kernelLaunches = launches;
    cs.kernelMs = 0.f;
    cudaEventElapsedTime(&cs.kernelMs, ctx->ev[1], ctx->ev[2]);
    // every packed word read and written once by the transpose, read once by the grouping pass; slot table cleared
    // and probed; three per-haplotype bookkeeping words; 16 bytes per emitted interval
    cs.bytesRead = static_cast<int64_t>(W) * (static_cast<int64_t>(H) * (8 + 8 + 8 + 12) + static_cast<int64_t>(C) * 12) +
                   16 * cs.numMatches;
    if (refOrder) {
      if (rankThread.joinable()) {
        rankThread.join();
      }
      cs.rankHostMs = static_cast<float>(rankMs);
      FSMC_CUDA(ctx->seedRank.ensure(std::max<size_t>(hostRank.size(), 1)));
      if (!hostRank.empty()) {
        FSMC_CUDA(cudaMemcpyAsync(ctx->seedRank.p, hostRank.data(), hostRank.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
      }
      fsmc::OrderStats os;
      long long numCandidates = 0;
      const cudaError_t e = ctx->orderer.order(ctx->seedOut.p, static_cast<long long>(counters[3]), H, W, L, sp->gap, sp->minLengthCm,
                                               ctx->seedGenPos.p, ctx->seedRank.p, st, &ctx->orderedOut, &numCandidates, &os);
      if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(e == cudaErrorMemoryAllocation ? FSMC_E_NOMEM : FSMC_E_CUDA, "fsmc_seed: device candidate ordering failed: %s",
                    cudaGetErrorString(e));
      }
      cs.numMatches = numCandidates;
      cs.maxLiveNodes = os.maxLive;
      cs.orderEpochs = os.epochs;
      cs.orderMs = os.deviceMs;
      ctx->seedCacheValid = true;
    } else {
      ctx->seedCacheValid = cs.numMatches <= devCap;  // everything found is on the device
    }
    ctx->seedCacheKey = key;
  }  // !cacheHit
  const long long found = static_cast<long long>(ctx->seedCacheStats.numMatches);
  if (stats) {
    *stats = ctx->seedCacheStats;
  }
  if (found > capacity) {
    return fail(FSMC_E_OVERFLOW, "fsmc_seed: %lld intervals found, capacity %lld", found, static_cast<long long>(capacity));
  }
  ctx->seedCacheValid = false;  // consumed by this call
  const long long stored = found;
  if (stored > 0 && refOrder) {
    FSMC_CUDA(cudaMemcpyAsync(out, ctx->orderedOut, stored * sizeof(fsmc_match), cudaMemcpyDeviceToHost, st));
    FSMC_CUDA(cudaStreamSynchronize(st));
  } else if (stored > 0 && (sp->flags & FSMC_SEED_UNSORTED)) {
    FSMC_CUDA(cudaMemcpyAsync(out, ctx->seedOut.p, stored * sizeof(fsmc_match), cudaMemcpyDeviceToHost, st));
    FSMC_CUDA(cudaStreamSynchronize(st));
    for (long long i = 0; i < stored; ++i) {
      if (out[i].endWord < out[i].startWord || out[i].startWord < 0 || out[i].endWord >= static_cast<int>(ctx->sites / 64)) {
        return fail(FSMC_E_CUDA, "fsmc_seed: corrupt match record (words %d..%d)", out[i].startWord, out[i].endWord);
      }
    }
  } else if (stored > 0) {
    // canonical candidate order (endWord, hapA, hapB): counting sort by end word from a staging copy into the
    // caller's buffer, then every end-word bucket is sorted by pair on its own host thread
    std::vector<fsmc_match> stage(static_cast<size_t>(stored));
    FSMC_CUDA(cudaMemcpyAsync(stage.data(), ctx->seedOut.p, stored * sizeof(fsmc_match), cudaMemcpyDeviceToHost, st));
    FSMC_CUDA(cudaStreamSynchronize(st));
    std::vector<size_t> begin(static_cast<size_t>(W) + 2, 0);
    for (const fsmc_match& mt : stage) {
      if (mt.endWord < 0 || mt.endWord >= W) {
        return fail(FSMC_E_CUDA, "fsmc_seed: corrupt match record (end word %d of %d)", mt.endWord, W);
      }
      ++begin[static_cast<size_t>(mt.endWord) + 1];
    }
    for (int w = 0; w < W; ++w) {
      begin[w + 1] += begin[w];
    }
    {
      std::vector<size_t> cursor(begin.begin(), begin.begin() + W);
      for (const fsmc_match& mt : stage) {
        out[cursor[mt.endWord]++] = mt;
      }
    }
    std::atomic<int> nextBucket{0};
    auto sortBuckets = [&] {
      for (int w = nextBucket++; w < W; w = nextBucket++) {
        std::sort(out + begin[w], out + begin[w + 1], [](const fsmc_match& x, const fsmc_match& y) {
          return x.hapA != y.hapA ? x.hapA < y.hapA : x.hapB < y.hapB;
        });
      }
    };
    const unsigned nThreads = stored < (1 << 16) ? 1u : std::min(32u, std::max(1u, std::thread::hardware_concurrency()));
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < nThreads; ++t) {
      pool.emplace_back(sortBuckets);
    }
    sortBuckets();
    for (auto& th : pool) {
      th.join();
    }
  }
  return FSMC_OK;
}

int fsmc_decode(fsmc_ctx* ctx, const fsmc_decode_request* req, fsmc_decode_stats* stats)
{
  if (!ctx || !req) {
    return fail(FSMC_E_INVALID, "fsmc_decode: NULL argument");
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  FSMC_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
  static const bool trace = std::getenv("FSMC_TRACE") != nullptr;  // development: host time of the call's phases
  const auto t0 = std::chrono::steady_clock::now();
  fsmc_plan* plan = nullptr;
  int rc = fsmc_plan_create(ctx, req, &plan);
  if (rc != FSMC_OK) {
    return rc;
  }
  const auto t1 = std::chrono::steady_clock::now();
  rc = fsmc_plan_launch(ctx, plan);
  const auto t2 = std::chrono::steady_clock::now();
  if (rc == FSMC_OK) {
    rc = fsmc_plan_collect(ctx, plan, req, stats);
  }
  const auto t3 = std::chrono::steady_clock::now();
  const std::string keep = gLastError;
  fsmc_plan_destroy(ctx, plan);
  gLastError = keep;
  if (trace) {
    const auto ms = [](auto a, auto b) { return std::chrono::duration<double, std::milli>(b - a).count(); };
    std::fprintf(stderr, "fsmc_decode tiles=%lld create %.2f ms launch %.2f ms collect %.2f ms (kernel %.2f ms) destroy %.2f ms\n",
                 static_cast<long long>(req->numTiles), ms(t0, t1), ms(t1, t2), ms(t2, t3), stats ? stats->kernelMs : 0.f,
                 ms(t3, std::chrono::steady_clock::now()));
  }
  return rc;
}

int fsmc_decode_device(fsmc_ctx* ctx, const fsmc_decode_request* req, const fsmc_device_outputs* out, fsmc_decode_stats* stats)
{
  if (!ctx || !req || !out) {
    return fail(FSMC_E_INVALID, "fsmc_decode_device: NULL argument");
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  FSMC_CUDA(cudaEventRecord(ctx->ev[0], ctx->stream));
  fsmc_plan* plan = nullptr;
  int rc = planCreate(ctx, req, out, &plan);
  if (rc != FSMC_OK) {
    return rc;
  }
  rc = fsmc_plan_launch(ctx, plan);
  if (rc == FSMC_OK) {
    const cudaError_t e = cudaEventRecord(ctx->ev[3], ctx->stream);
    const cudaError_t e2 = e == cudaSuccess ? cudaStreamSynchronize(ctx->stream) : e;
    if (e2 != cudaSuccess) {
      rc = fail(FSMC_E_CUDA, "fsmc_decode_device: %s", cudaGetErrorString(e2));
    } else {
      fillStats(ctx, plan, 0, 0, stats);
    }
  }
  plan->launched = false;
  const std::string keep = gLastError;
  fsmc_plan_destroy(ctx, plan);
  gLastError = keep;
  return rc;
}

}  // extern "C"

namespace
{
template <class T>
int columnMin(fsmc_ctx* ctx, const char* name, const T* m, const int64_t rows, const int64_t cols, const int64_t ld, T* minOut,
              int32_t* argOut)
{
  if (!ctx || !m || !minOut || !argOut) {
    return fail(FSMC_E_INVALID, "%s: NULL argument", name);
  }
  if (rows < 1 || rows > 0x7fffffffll || cols < 1 || ld < cols) {
    return fail(FSMC_E_INVALID, "%s: rows=%lld cols=%lld ld=%lld (need 1 <= rows < 2^31, 1 <= cols <= ld)", name,
                static_cast<long long>(rows), static_cast<long long>(cols), static_cast<long long>(ld));
  }
  for (const auto& [p, what] : {std::make_pair(static_cast<const void*>(m), "m_dev"), std::make_pair(static_cast<const void*>(minOut), "min_dev"),
                                std::make_pair(static_cast<const void*>(argOut), "argmin_dev")}) {
    const int rc = checkDevicePtr(ctx, p, what);
    if (rc != FSMC_OK) {
      return rc;
    }
  }
  FSMC_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // rows are cut into chunks until the grid has about 16 blocks of 256 threads per SM
  const long long colBlocks = (cols + fsmc::kColMinCols - 1) / fsmc::kColMinCols;
  const long long want = (16ll * ctx->prop.multiProcessorCount + colBlocks - 1) / colBlocks;
  const long long chunks = std::max(1ll, std::min<long long>({want, static_cast<long long>((rows + 255) / 256), 65535ll}));
  const long long rowsPerChunk = (rows + chunks - 1) / chunks;
  const dim3 block(fsmc::kColMinCols, fsmc::kColMinGroups);
  const dim3 grid(static_cast<unsigned>(colBlocks), static_cast<unsigned>(chunks));
  if (chunks == 1) {
    fsmc::columnMinPartialKernel<T><<<grid, block, 0, st>>>(m, rows, cols, ld, rowsPerChunk, minOut, argOut);
  } else {
    FSMC_CUDA(ctx->colMinPart.ensure(2 * static_cast<size_t>(chunks) * cols));
    T* partV = reinterpret_cast<T*>(ctx->colMinPart.p);
    int* partRow = reinterpret_cast<int*>(ctx->colMinPart.p + static_cast<size_t>(chunks) * cols);
    fsmc::columnMinPartialKernel<T><<<grid, block, 0, st>>>(m, rows, cols, ld, rowsPerChunk, partV, partRow);
    const int cb = static_cast<int>(std::min<long long>((cols + 255) / 256, 8ll * ctx->prop.multiProcessorCount));
    fsmc::columnMinCombineKernel<T><<<cb, 256, 0, st>>>(partV, partRow, static_cast<int>(chunks), cols, minOut, argOut);
  }
  FSMC_CUDA(cudaGetLastError());
  return FSMC_OK;
}
}  // namespace

extern "C" {

int fsmc_column_min_f32(fsmc_ctx* ctx, const float* m_dev, const int64_t rows, const int64_t cols, const int64_t ld, float* min_dev,
                        int32_t* argmin_dev)
{
  return columnMin(ctx, "fsmc_column_min_f32", m_dev, rows, cols, ld, min_dev, argmin_dev);
}

int fsmc_column_min_i32(fsmc_ctx* ctx, const int32_t* m_dev, const int64_t rows, const int64_t cols, const int64_t ld,
                        int32_t* min_dev, int32_t* argmin_dev)
{
  return columnMin(ctx, "fsmc_column_min_i32", m_dev, rows, cols, ld, min_dev, argmin_dev);
}

}  // extern "C"
