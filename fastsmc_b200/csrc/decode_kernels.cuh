// fastsmc_b200 — sm_100a kernels for the batched pairwise-coalescent HMM (ASMC/FastSMC decode).
//
// One warp owns one TILE: 32 haplotype pairs (lane = pair) that share a decode window, i.e. one
// reference batch (ref: ASMC_SRC/SRC/HMM.cpp:555-636).  The warp makes two sweeps over the window:
//
//   sweep 1 (backward, ref HMM.cpp:882-1041): beta[pos][k] for every site, rescaled to sum 1 at
//            every site, streamed to a per-warp HBM slab laid out [pos][k][lane] so that each
//            (pos,k) row is one coalesced 128-byte line;
//   sweep 2 (forward, ref HMM.cpp:725-879) : alpha[pos][k] kept on chip only; at every site the
//            posterior alpha*beta/sum (ref HMM.cpp:669-692) is formed in registers and consumed at
//            once by the segment caller (ref HMM.cpp:1179-1357), the per-site posterior-mean / MAP
//            reducers (ref HMM.cpp:1378-1409) and the IBD-probability threshold.  Per-site
//            posteriors never reach HBM.
//
// The backward sweep runs first so that the consumers see sites in ascending order, the order in
// which the reference accumulates per-segment sums; with FSMC_EXACT (unfused multiply/add in the
// reference's NO_SSE operation order) every output is then bit-identical to the reference.
//
// State vectors live in registers when the state count is a compile-time constant (fully unrolled
// linear-time recurrences), in shared memory ([k][lane], conflict-free) otherwise.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/fastsmc_b200.h"

namespace fsmc
{

constexpr int kRowArrays = 8;  // per-site table row: E_homMajor, E_het, E_homMinor, D, B, U, RR, U shifted by one state (each Spad floats)
constexpr int kBwdArrays = 10;  // per-site backward row of the narrow kernel, emission folded in (buildBackwardRowsKernel)
constexpr unsigned kFull = 0xffffffffu;

struct DeviceModel {
  int S;       // states
  int Spad;    // S rounded up to a multiple of 4 (float4 loads)
  int L;       // sites
  const float* siteRows;   // [L][kRowArrays][Spad]
  const float* bwdRows;    // [L][kBwdArrays][Spad] backward rows with the emission folded in; 69-state models only
  const float* laneAux;    // [L][Spad + 16] suffix products of RR inside the state quarters (decode_lane.cuh); 159-state models only
  const float* prior;      // [Spad] initialStateProb
  const float* expTimes;   // [Spad] expectedTimes
  const float* colRatios;  // [Spad] columnRatios
  int stateThreshold;
  int ageThreshold;
  float thr[4];            // 1000*pT, 100*pT, 10*pT, pT  (ref HMM.cpp:1226,1254,1281,1308)
  const uint64_t* haps;    // [numHaps][wordsPerHap]
  long long wordsPerHap;
};

// One piece of an IBD run inside one checkpoint block: sites [first, last] of pair `pair`.  The pieces of a run are
// chained through `prev` (the segment record points at the last one).
struct SparseItem {
  uint32_t pair;
  int32_t block;
  int32_t first, last;
  int32_t prev;
};

struct DecodeArgs {
  const uint32_t* hapA;
  const uint32_t* hapB;
  const int* tilePairs;
  const int* tileFrom;
  const int* tileTo;
  const int* tileScanFrom;
  const int* tileScanTo;
  const int* order;  // tiles in launch order (longest window first)
  long long numTiles;
  unsigned flags;
  fsmc_segment* segments;
  unsigned long long* segmentCount;
  long long segmentCapacity;
  float* siteMean;
  int* siteMap;
  float* siteIbd;
  long long siteStride;
  float* sitePosterior;        // [pair][S][siteStride]
  float* sumPosterior;         // [planes][S][L]
  float* scratch;              // beta slabs
  long long scratchPerWarp;    // floats per warp slab
  float* accScratch;           // fast kernel: per-warp [S][32] per-state segment sums
  unsigned long long* tileCounter;
  // ---- sparse age estimates (decode_sparse.cuh): all-state per-segment sums without the beta round trip ------------
  int ckptShift;                    // checkpoint block = 2^ckptShift sites, aligned to absolute site numbers
  const long long* tileCkptBase;    // [numTiles] first checkpoint slot of each tile
  float* ckptBeta;                  // [slot][Spad/4][32][4] beta at the last site of every block of every tile
  float* alphaScratch;              // [resident warp][Spad/4][32][4] alpha at the first site of the block being swept
  SparseItem* items;                // pieces of IBD runs, one per (run, block)
  float* itemAlpha;                 // [item][Spad] alpha at the first site of the item's block (or of the window)
  float* itemSums;                  // [item][Spad] per-state posterior sums over the item's sites (refine pass)
  unsigned long long* itemCount;
  long long itemCapacity;
  const uint32_t* itemOrder;        // items sorted by block (refine pass)
  unsigned long long* refineCounter;
  // ---- sums of posteriors over pairs on the production kernel: private accumulators per resident warp ------------------
  float* sumScratch;                // [warp][planes][L][Spad]
  // ---- fsmc_decode_device: caller-owned outputs --------------------------------------------------------------------
  const uint32_t* laneRow;          // [numTiles*32] output row of pair tile*32+lane; NULL = the pair number
  const float* stateWeight;         // [S] posterior rows are multiplied by it; sums are added to the output times it
};

// ---- arithmetic: EXACT = separate IEEE multiply and add (never contracted), else FMA ------------
template <bool EXACT> __device__ __forceinline__ float mulAdd(float a, float b, float c)
{
  if constexpr (EXACT) {
    return __fadd_rn(__fmul_rn(a, b), c);
  } else {
    return fmaf(a, b, c);
  }
}
// a*b + c*d  (two rounded products, then the sum, in EXACT mode)
template <bool EXACT> __device__ __forceinline__ float mulMulAdd(float a, float b, float c, float d)
{
  if constexpr (EXACT) {
    return __fadd_rn(__fmul_rn(a, b), __fmul_rn(c, d));
  } else {
    return fmaf(a, b, c * d);
  }
}

// ---- state-vector storage -----------------------------------------------------------------------
template <int N> struct RegVec {
  float v[N];
  __device__ __forceinline__ float get(int k) const { return v[k]; }
  __device__ __forceinline__ void set(int k, float x) { v[k] = x; }
};
struct SmemVec {
  float* p;  // already offset by the lane; element k at p[k*32]
  __device__ __forceinline__ float get(int k) const { return p[k * 32]; }
  __device__ __forceinline__ void set(int k, float x) { p[k * 32] = x; }
};

__device__ __forceinline__ float4 ldg4(const float* p)
{
  return __ldg(reinterpret_cast<const float4*>(p));
}
__device__ __forceinline__ float elem(const float4& v, int j)
{
  return j == 0 ? v.x : (j == 1 ? v.y : (j == 2 ? v.z : v.w));
}

// Visit states k < limit (limit is warp-uniform).  For register-resident vectors the loop is fully
// unrolled; groups of 8 states are skipped with a uniform branch when limit is small (the IBD
// state threshold is typically a handful of states).
template <int S_T, class F> __device__ __forceinline__ void forStatesBelow(const int limit, F&& f)
{
  if constexpr (S_T > 0) {
#pragma unroll
    for (int g = 0; g < (S_T + 7) / 8; ++g) {
      if (8 * g < limit) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int k = 8 * g + j;
          if (k < S_T && k < limit) {
            f(k);
          }
        }
      }
    }
  } else {
    for (int k = 0; k < limit; ++k) {
      f(k);
    }
  }
}

// Genotype class of this lane's pair at one site: 0 = both major, 1 = heterozygous, 2 = both minor.
// ref HMM.cpp:647-652 (obsIsZero = !xor, obsIsTwo = and) folded into a 3-way table select.
struct PairBits {
  const uint64_t* a;
  const uint64_t* b;
  uint64_t x = 0, t = 0;
  long long word = -1;
  __device__ __forceinline__ int cls(int site)
  {
    const long long w = site >> 6;
    if (w != word) {
      const uint64_t wa = __ldg(a + w), wb = __ldg(b + w);
      x = wa ^ wb;
      t = wa & wb;
      word = w;
    }
    const int bit = site & 63;
    return ((x >> bit) & 1ull) ? 1 : (((t >> bit) & 1ull) ? 2 : 0);
  }
};

// -------------------------------------------------------------------------------------------------
// sweep 1: backward.  ref HMM.cpp:882-940 (driver), 943-1041 (step), HmmUtils.cpp:102-151 (scaling)
// -------------------------------------------------------------------------------------------------
template <int S_T, bool EXACT, class VecA, class VecC>
__device__ __forceinline__ void sweepBackward(const DeviceModel& m, PairBits& bits, const int from, const int len,
                                              VecA& b, VecC& c, float* __restrict__ beta /* slab + lane */)
{
  const int S = S_T ? S_T : m.S;
  const int SQ = (S_T ? (S_T + 3) / 4 : m.Spad / 4);
  const int Spad = SQ * 4;
  const size_t plane = static_cast<size_t>(S) * 32;

  // beta at the last site: ones, rescaled (sum of S ones is exactly S)
  {
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      sum = __fadd_rn(sum, 1.0f);
    }
    const float sc = 1.0f / sum;
    float* out = beta + static_cast<size_t>(len - 1) * plane;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const float v = __fmul_rn(1.0f, sc);
      b.set(k, v);
      out[k * 32] = v;
    }
  }

  for (int p = len - 2; p >= 0; --p) {
    const int site = from + p + 1;  // emission of pos+1, transition for the gap (pos, pos+1)
    const float* row = m.siteRows + static_cast<size_t>(site) * kRowArrays * Spad;
    const float* E = row + bits.cls(site) * Spad;
    const float* Dr = row + 3 * Spad;
    const float* Br = row + 4 * Spad;
    const float* Ur = row + 5 * Spad;
    const float* Rr = row + 6 * Spad;

    // vec = beta(pos+1) * emission(pos+1)      (ref HMM.cpp:957-964), in place in b
#pragma unroll
    for (int q = 0; q < SQ; ++q) {
      const float4 e4 = ldg4(E + 4 * q);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int k = 4 * q + j;
        if (k < S) {
          b.set(k, __fmul_rn(b.get(k), elem(e4, j)));
        }
      }
    }
    // BU[k] = U[k]*vec[k+1] + RR[k]*BU[k+1], BU[S-1] = 0      (ref HMM.cpp:986-990)
    {
      float bu = 0.f;
#pragma unroll
      for (int q = SQ - 1; q >= 0; --q) {
        const float4 u4 = ldg4(Ur + 4 * q);
        const float4 r4 = ldg4(Rr + 4 * q);
#pragma unroll
        for (int j = 3; j >= 0; --j) {
          const int k = 4 * q + j;
          if (k == S - 1) {
            c.set(k, 0.f);
          } else if (k < S - 1) {
            bu = mulMulAdd<EXACT>(elem(u4, j), b.get(k + 1), elem(r4, j), bu);
            c.set(k, bu);
          }
        }
      }
    }
    // beta(pos)[k] = (BL + D[k]*vec[k]) + BU[k],  BL += B[k-1]*vec[k-1]     (ref HMM.cpp:1008-1016)
    float sum = 0.f;
    {
      float bl = 0.f, bPrev = 0.f, vPrev = 0.f;
#pragma unroll
      for (int q = 0; q < SQ; ++q) {
        const float4 d4 = ldg4(Dr + 4 * q);
        const float4 b4 = ldg4(Br + 4 * q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = 4 * q + j;
          if (k < S) {
            const float v = b.get(k);
            if (k) {
              bl = mulAdd<EXACT>(bPrev, vPrev, bl);
            }
            const float nb = __fadd_rn(mulAdd<EXACT>(elem(d4, j), v, bl), c.get(k));
            c.set(k, nb);
            sum = __fadd_rn(sum, nb);
            bPrev = elem(b4, j);
            vPrev = v;
          }
        }
      }
    }
    // rescale to sum 1 and stream out
    const float sc = 1.0f / sum;
    float* out = beta + static_cast<size_t>(p) * plane;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const float v = __fmul_rn(c.get(k), sc);
      b.set(k, v);
      out[k * 32] = v;
    }
  }
}

// -------------------------------------------------------------------------------------------------
// segment emission.  ref HMM.cpp:1110-1177 (record), 1087-1107 (posterior mean / MAP of the sums)
// -------------------------------------------------------------------------------------------------
template <bool EXACT>
__device__ __noinline__ void emitSegment(const DeviceModel& m, const DecodeArgs& a, const uint32_t pair, const int start,
                                         const int end, const float prob, const int level,
                                         const float* acc /* smem + lane, stride 32 */, const bool age,
                                         const int lastItem = -1 /* sparse age estimates: chain of the run's items */)
{
  fsmc_segment s;
  s.pair = pair;
  s.posStart = start;
  s.posEnd = end;
  s.prob = prob;
  s.level = level;
  s.postMean = 0.f;
  s.mapTime = 0.f;
  s.mapState = lastItem;  // replaced by finalizeSegmentsKernel (decode_sparse.cuh) when >= 0
  if (age) {
    const int n = m.ageThreshold;
    float tot = 0.f;
    for (int k = 0; k < n; ++k) {
      tot = __fadd_rn(tot, acc[k * 32]);
    }
    const float norm = 1.f / tot;
    float mean = 0.f;
    int best = 0;
    float bestRatio = acc[0] / __ldg(m.prior);
    for (int k = 0; k < n; ++k) {
      const float x = acc[k * 32];
      mean = __fadd_rn(mean, __fmul_rn(__fmul_rn(norm, x), __ldg(m.expTimes + k)));
      const float r = x / __ldg(m.prior + k);
      if (bestRatio < r) {
        bestRatio = r;
        best = k;
      }
    }
    s.postMean = mean;
    s.mapState = best;
    s.mapTime = __ldg(m.expTimes + best);
  }
  const unsigned long long idx = atomicAdd(a.segmentCount, 1ull);
  if (static_cast<long long>(idx) < a.segmentCapacity) {
    a.segments[idx] = s;
  }
}

// Per-lane run-length state of the segment caller (ref HMM.cpp:1182-1186: the four isIBD* flags are
// mutually exclusive, so one `level` suffices).
struct CallerState {
  int level = -1;
  int start = 0;
  float prob = 0.f;
};

// -------------------------------------------------------------------------------------------------
// sweep 2: forward + fused posterior consumers.
// -------------------------------------------------------------------------------------------------
template <int S_T, bool EXACT, class VecA, class VecC>
__device__ __forceinline__ void sweepForward(const DeviceModel& m, const DecodeArgs& args, PairBits& bits,
                                             const int from, const int len, const int scanFrom, const int scanTo,
                                             const uint32_t pair, const uint32_t outRow, const bool laneActive, VecA& a, VecC& c,
                                             const float* __restrict__ beta, float* acc /* smem + lane */)
{
  const int S = S_T ? S_T : m.S;
  const int SQ = (S_T ? (S_T + 3) / 4 : m.Spad / 4);
  const int Spad = SQ * 4;
  const size_t plane = static_cast<size_t>(S) * 32;
  const unsigned flags = args.flags;
  const bool wantSeg = flags & FSMC_CALL_SEGMENTS;
  const bool wantAge = (flags & FSMC_SEG_AGE) && wantSeg;
  const int sT = m.stateThreshold;
  const int nAcc = m.ageThreshold;
  const bool lane0 = (threadIdx.x & 31) == 0;
  CallerState cs;

  for (int p = 0; p < len; ++p) {
    const int site = from + p;
    const float* row = m.siteRows + static_cast<size_t>(site) * kRowArrays * Spad;
    const float* E = row + bits.cls(site) * Spad;
    float sum = 0.f;

    if (p == 0) {
      // alpha(from)[k] = prior[k] * emission      (ref HMM.cpp:736-743)
#pragma unroll
      for (int q = 0; q < SQ; ++q) {
        const float4 e4 = ldg4(E + 4 * q);
        const float4 p4 = ldg4(m.prior + 4 * q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = 4 * q + j;
          if (k < S) {
            const float v = __fmul_rn(elem(p4, j), elem(e4, j));
            c.set(k, v);
            sum = __fadd_rn(sum, v);
          }
        }
      }
    } else {
      const float* Dr = row + 3 * Spad;
      const float* Br = row + 4 * Spad;
      const float* Ur = row + 5 * Spad;
      // alphaC[k] = sum_{j>=k} alpha(pos-1)[j]      (ref HMM.cpp:799-814)
      {
        float run = 0.f;
#pragma unroll
        for (int k = S - 1; k >= 0; --k) {
          run = (k == S - 1) ? a.get(k) : __fadd_rn(run, a.get(k));
          c.set(k, run);
        }
      }
      // ref HMM.cpp:816-830
      float au = 0.f, uPrev = 0.f, crPrev = 0.f, aPrev = 0.f;
#pragma unroll
      for (int q = 0; q < SQ; ++q) {
        const float4 e4 = ldg4(E + 4 * q);
        const float4 d4 = ldg4(Dr + 4 * q);
        const float4 b4 = ldg4(Br + 4 * q);
        const float4 u4 = ldg4(Ur + 4 * q);
        const float4 r4 = ldg4(m.colRatios + 4 * q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = 4 * q + j;
          if (k < S) {
            const float ak = a.get(k);
            if (k) {
              au = mulMulAdd<EXACT>(uPrev, aPrev, crPrev, au);
            }
            float term = mulAdd<EXACT>(elem(d4, j), ak, au);
            if (k < S - 1) {
              term = mulAdd<EXACT>(elem(b4, j), c.get(k + 1), term);
            }
            const float v = __fmul_rn(elem(e4, j), term);
            c.set(k, v);
            sum = __fadd_rn(sum, v);
            uPrev = elem(u4, j);
            crPrev = elem(r4, j);
            aPrev = ak;
          }
        }
      }
    }
    // rescale alpha(pos) to sum 1 (ref HmmUtils.cpp:102-151), then q = alpha*beta (ref HMM.cpp:672-680)
    const float sc = 1.0f / sum;
    const float* bp = beta + static_cast<size_t>(p) * plane;
    float qsum = 0.f;
#pragma unroll
    for (int k = 0; k < S; ++k) {
      const float al = __fmul_rn(c.get(k), sc);
      a.set(k, al);
      const float q = __fmul_rn(al, bp[k * 32]);
      c.set(k, q);
      qsum = __fadd_rn(qsum, q);
    }
    const float r = 1.0f / qsum;  // ref HMM.cpp:681-685 (NO_SSE: exact reciprocal)
    // posterior[k] = c[k] * r from here on (ref HMM.cpp:686-692)

    // ---- per-site reducers (ref HMM.cpp:1378-1409) ------------------------------------------
    if (flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP)) {
      float mean = 0.f, best = 0.f;
      int arg = 0;
#pragma unroll
      for (int q = 0; q < SQ; ++q) {
        const float4 t4 = ldg4(m.expTimes + 4 * q);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int k = 4 * q + j;
          if (k < S) {
            const float post = __fmul_rn(c.get(k), r);
            mean = mulAdd<EXACT>(post, elem(t4, j), mean);
            if (best < post) {
              best = post;
              arg = k;
            }
          }
        }
      }
      if (laneActive) {
        if (flags & FSMC_SITE_MEAN) {
          args.siteMean[static_cast<size_t>(outRow) * args.siteStride + p] = mean;
        }
        if (flags & FSMC_SITE_MAP) {
          args.siteMap[static_cast<size_t>(outRow) * args.siteStride + p] = arg;
        }
      }
    }

    // ---- full posteriors and their sum over pairs (ref HMM.cpp:1372-1389, 1044-1085) ----------
    if (flags & (FSMC_SITE_POSTERIOR | FSMC_SUM_POSTERIOR)) {
      float* postRow = args.sitePosterior + static_cast<size_t>(outRow) * S * args.siteStride + p;
      // plane of the sum this lane's pair contributes to: its genotype class at the site, or the only plane
      const int plane = (flags & FSMC_SUM_BY_GENOTYPE) ? bits.cls(site) : 0;
      const int nPlanes = (flags & FSMC_SUM_BY_GENOTYPE) ? 3 : 1;
#pragma unroll
      for (int k = 0; k < S; ++k) {
        const float post = __fmul_rn(c.get(k), r);
        // fsmc_decode_device: weighted rows and sums (the host's posterior * expectedTimes[k], one rounding)
        const float w = args.stateWeight ? __ldg(args.stateWeight + k) : 1.f;
        if ((flags & FSMC_SITE_POSTERIOR) && laneActive) {
          postRow[static_cast<size_t>(k) * args.siteStride] = args.stateWeight ? __fmul_rn(post, w) : post;
        }
        if (flags & FSMC_SUM_POSTERIOR) {
          for (int pl = 0; pl < nPlanes; ++pl) {
            float v = (laneActive && plane == pl) ? post : 0.f;
#pragma unroll
            for (int d = 16; d > 0; d >>= 1) {
              v += __shfl_xor_sync(kFull, v, d);
            }
            if (lane0 && v != 0.f) {
              atomicAdd(args.sumPosterior + (static_cast<size_t>(pl) * S + k) * m.L + site, args.stateWeight ? __fmul_rn(v, w) : v);
            }
          }
        }
      }
    }

    const bool inScan = wantSeg && site >= scanFrom && site < scanTo;
    if ((flags & FSMC_SITE_IBD) || inScan) {
      // IBD probability = sum_{k<stateThreshold} posterior[k], ascending k (ref HMM.cpp:1206-1224)
      float ibd = 0.f;
      forStatesBelow<S_T>(sT, [&](const int k) { ibd = __fadd_rn(ibd, __fmul_rn(c.get(k), r)); });
      if ((flags & FSMC_SITE_IBD) && laneActive) {
        args.siteIbd[static_cast<size_t>(outRow) * args.siteStride + p] = ibd;
      }

      if (inScan) {
        // ---- segment caller (ref HMM.cpp:1226-1354) -------------------------------------------
        int now = -1;
        if (ibd >= m.thr[0]) {
          now = 0;
        } else if (ibd >= m.thr[1]) {
          now = 1;
        } else if (ibd >= m.thr[2]) {
          now = 2;
        } else if (ibd >= m.thr[3]) {
          now = 3;
        }
        if (!laneActive) {
          now = -1;
        }
        const bool changed = now != cs.level;
        if (changed && cs.level >= 0) {
          // the run that ended at site-1; its sums do not include this site (prev_sum_posterior_per_state)
          emitSegment<EXACT>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, acc, wantAge);
        }
        if (wantAge && __any_sync(kFull, now >= 0)) {
          // per-state sums of the current run: restart with this site's posterior on a new run,
          // accumulate otherwise (ref HMM.cpp:1209-1218,1229,1257,1284,1311)
          forStatesBelow<S_T>(nAcc, [&](const int k) {
            if (now >= 0) {
              const float post = __fmul_rn(c.get(k), r);
              acc[k * 32] = changed ? post : __fadd_rn(acc[k * 32], post);
            }
          });
        }
        if (now >= 0) {
          if (changed) {
            cs.start = site;
            cs.prob = ibd;
          } else {
            cs.prob = __fadd_rn(cs.prob, ibd);
          }
          if (site == scanTo - 1) {
            emitSegment<EXACT>(m, args, pair, cs.start, site, cs.prob, now, acc, wantAge);
            cs.prob = 0.f;
          }
        } else {
          cs.prob = 0.f;
        }
        cs.level = now;
      }
    }
  }
}

// -------------------------------------------------------------------------------------------------
// kernel: persistent warps pulling tiles from a global queue (longest window first).
// MODE 0: alpha/beta and the scan vector in registers (S_T > 0)
// MODE 1: first vector in registers, scan vector in shared memory (large S_T)
// MODE 2: both in shared memory, any S at run time (S_T == 0)
// -------------------------------------------------------------------------------------------------
template <int S_T, int MODE, bool EXACT, int THREADS, int MIN_BLOCKS>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) decodeTilesKernel(const DeviceModel m, const DecodeArgs args)
{
  extern __shared__ float smem[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int kWarps = blockDim.x >> 5;  // may be fewer than THREADS/32 when shared memory limits the block
  const int S = S_T ? S_T : m.S;
  const bool wantAge = (args.flags & FSMC_SEG_AGE) && (args.flags & FSMC_CALL_SEGMENTS);

  // shared-memory carve-up per warp: [acc (ageThreshold rows, if wanted)] [scan vector] [first vector]
  const int accRows = wantAge ? m.ageThreshold : 0;
  const int rowsPerWarp = accRows + (MODE >= 1 ? S : 0) + (MODE == 2 ? S : 0);
  float* mine = smem + static_cast<size_t>(warp) * rowsPerWarp * 32 + lane;
  float* acc = mine;
  float* beta = args.scratch + (static_cast<size_t>(blockIdx.x) * kWarps + warp) * args.scratchPerWarp + lane;

  for (;;) {
    unsigned long long t = 0;
    if (lane == 0) {
      t = atomicAdd(args.tileCounter, 1ull);
    }
    t = __shfl_sync(kFull, t, 0);
    if (static_cast<long long>(t) >= args.numTiles) {
      break;
    }
    const int tile = args.order ? args.order[t] : static_cast<int>(t);
    const int nPairs = args.tilePairs[tile];
    const int from = args.tileFrom[tile];
    const int len = args.tileTo[tile] - from;
    const int scanFrom = (args.flags & FSMC_CALL_SEGMENTS) ? args.tileScanFrom[tile] : 0;
    const int scanTo = (args.flags & FSMC_CALL_SEGMENTS) ? args.tileScanTo[tile] : 0;
    const bool laneActive = lane < nPairs;
    const int srcLane = laneActive ? lane : nPairs - 1;  // padding repeats the last pair (ref HMM.cpp:616-619)
    const uint32_t pair = static_cast<uint32_t>(tile) * 32u + static_cast<uint32_t>(lane);
    const uint32_t outRow = args.laneRow ? __ldg(args.laneRow + pair) : pair;  // output row (fsmc_decode_device)
    PairBits bits;
    bits.a = m.haps + static_cast<size_t>(args.hapA[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    bits.b = m.haps + static_cast<size_t>(args.hapB[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;

    if constexpr (MODE == 0) {
      RegVec<S_T> v0, v1;
      sweepBackward<S_T, EXACT>(m, bits, from, len, v0, v1, beta);
      sweepForward<S_T, EXACT>(m, args, bits, from, len, scanFrom, scanTo, pair, outRow, laneActive, v0, v1, beta, acc);
    } else if constexpr (MODE == 1) {
      RegVec<S_T> v0;
      SmemVec v1{mine + static_cast<size_t>(accRows) * 32};
      sweepBackward<S_T, EXACT>(m, bits, from, len, v0, v1, beta);
      sweepForward<S_T, EXACT>(m, args, bits, from, len, scanFrom, scanTo, pair, outRow, laneActive, v0, v1, beta, acc);
    } else {
      SmemVec v1{mine + static_cast<size_t>(accRows) * 32};
      SmemVec v0{mine + static_cast<size_t>(accRows + S) * 32};
      sweepBackward<0, EXACT>(m, bits, from, len, v0, v1, beta);
      sweepForward<0, EXACT>(m, args, bits, from, len, scanFrom, scanTo, pair, outRow, laneActive, v0, v1, beta, acc);
    }
    __syncwarp();
  }
}

// -------------------------------------------------------------------------------------------------
// model assembly: gather the distance-keyed transition rows and the three emission classes into one
// contiguous row per site: [E_homMajor | E_het | E_homMinor | D | B | U | RR | Us], each Spad floats; Us[k] = U[k-1]
// (the packed backward step multiplies U[k-1] vec[k] for two neighbouring states at once, decode_fast.cuh).
// E_homMajor = e1 + e0m1, E_het = e1, E_homMinor = (e1 + e0m1) + e2m0 are bit-identical to the
// reference's e1 + e0m1*isZero + e2m0*isTwo for the three genotype classes (ref HMM.cpp:827-828).
// -------------------------------------------------------------------------------------------------
static __global__ void buildSiteRowsKernel(const int S, const int Spad, const int L, const float* __restrict__ e1,
                                    const float* __restrict__ e0m1, const float* __restrict__ e2m0,
                                    const float* __restrict__ D, const float* __restrict__ B,
                                    const float* __restrict__ U, const float* __restrict__ RR,
                                    const int* __restrict__ distRow, float* __restrict__ rows)
{
  const long long total = static_cast<long long>(L) * Spad;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int site = static_cast<int>(i / Spad);
    const int k = static_cast<int>(i % Spad);
    float* out = rows + static_cast<size_t>(site) * kRowArrays * Spad + k;
    float v[kRowArrays] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (k < S) {
      const size_t e = static_cast<size_t>(site) * S + k;
      const float hm = __fadd_rn(e1[e], e0m1[e]);
      v[0] = hm;
      v[1] = e1[e];
      v[2] = __fadd_rn(hm, e2m0[e]);
      if (site > 0) {
        const size_t t = static_cast<size_t>(distRow[site]) * S + k;
        v[3] = D[t];
        v[4] = B[t];
        v[5] = U[t];
        v[6] = RR[t];
        if (k > 0) {
          v[7] = U[t - 1];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kRowArrays; ++j) {
      out[static_cast<size_t>(j) * Spad] = v[j];
    }
  }
}

// The narrow kernel's backward rows (decode_fast.cuh), from the rows above: the emission of each genotype class c is
// multiplied into the coefficients once per site, so that the backward step never multiplies beta by it.
//   backward row of site s: [UsE_0..2 | DE_0..2 | BE_0..2 | RR],  UsE_c = Us_s E_s[c], DE_c = D_s E_s[c], BE_c = B_s E_s[c]
static __global__ void buildBackwardRowsKernel(const int Spad, const int L, const float* __restrict__ rows,
                                               float* __restrict__ bwd)
{
  const long long total = static_cast<long long>(L) * Spad;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int site = static_cast<int>(i / Spad);
    const int k = static_cast<int>(i % Spad);
    const float* r = rows + static_cast<size_t>(site) * kRowArrays * Spad + k;
    const float D = r[3 * Spad], B = r[4 * Spad], Us = r[7 * Spad];
    float* b = bwd + static_cast<size_t>(site) * kBwdArrays * Spad + k;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float e = r[c * Spad];
      b[c * Spad] = __fmul_rn(Us, e);
      b[(3 + c) * Spad] = __fmul_rn(D, e);
      b[(6 + c) * Spad] = __fmul_rn(B, e);
    }
    b[9 * Spad] = r[6 * Spad];  // RR
  }
}

}  // namespace fsmc
