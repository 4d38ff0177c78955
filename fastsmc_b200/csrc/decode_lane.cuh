// fastsmc_b200 — lane-split decode kernel for sm_100a (159 states, FastSMC_exe's default flags).
//
// At 159 states a lane cannot hold two state vectors (decode_fast.cuh), and cutting the states across the WARPS of a CTA
// (decode_split.cuh) costs three CTA barriers per step and four different instruction streams per CTA: the profiler shows
// `no_instruction` and `barrier` as its first two stalls (profiles/r1_v19_decodeSplit_s159_ncu_full.txt).  Here the states
// are cut across the LANES of a warp instead: a warp decodes 8 pairs, lane = (quarter g of the state range, pair p), so
//   * every lane runs the same instructions (one body for the whole kernel: the sweeps stream from the instruction cache),
//   * the four quarters of a scan meet through warp shuffles, not through shared memory and barriers,
//   * a lane holds 2 x 40 states: ~110 registers, 16 warps per SM.
//
// A scan over the states (ref: HMM.cpp:787-879, 943-1041) is a first-order linear recurrence c[k+1] = m[k] c[k] + v[k].
// Each quarter runs it from a zero carry-in (pass 1); the true carry-in of a quarter follows from the four local results
// and the quarters' aggregate multipliers (a handful of FMAs after the shuffles); pass 2 adds carry-in x (product of the
// multipliers from the quarter's first state to k) to every state.  The multipliers of the forward AU scan are the
// column ratios (site-independent: prefix products in shared memory, once per CTA); those of the backward BU scan are the
// per-site RR coefficients: their suffix products inside each quarter come with the site's row (laneAux table, built by
// buildLaneAuxKernel).  The two plain sums (suffix sums of alpha, BL) have multiplier 1.
//
// One 32-pair tile (= one reference batch, HMM.cpp:694-716) is one CTA of 4 warps that share the coefficient ring
// (cp.async.bulk on mbarriers, one CTA barrier per group of G sites).  Records (beta below the IBD time threshold + the
// scale divisor, decodeNarrowKernel's scheme) are written and read by the quarter-0 lanes directly.
#pragma once

#include "decode_fast.cuh"

namespace fsmc
{

constexpr int kLaneQuarters = 4;
constexpr int kLaneAuxExtra = 16;  // per site: {RR, suffix product of RR, U} at the quarter boundaries, 4 floats per quarter

template <int S_T> struct LaneGeom {
  static constexpr int SQ = (S_T + 3) / 4;
  static constexpr int Spad = SQ * 4;
  static constexpr int SEG = Spad / kLaneQuarters;  // states per lane
  static constexpr int SEGQ = SEG / 4;
  static constexpr int kAuxFloats = Spad + kLaneAuxExtra;
  static_assert(Spad % (4 * kLaneQuarters) == 0, "whole quads per quarter");
  static_assert(S_T > Spad - SEG, "the last quarter holds real states");
};

// laneAux[site] = [ Rp[Spad] | boundary[4][4] ]:  Rp[k] = prod of RR over the states from k to the one before the last of
// k's quarter (1 at the quarter's last state); boundary[q] = { RR[last of q], Rp[first of q], U[last of q], 0 }.
static __global__ void buildLaneAuxKernel(const int Spad, const int L, const float* __restrict__ rows, float* __restrict__ aux)
{
  const int SEG = Spad / kLaneQuarters;
  const int auxFloats = Spad + kLaneAuxExtra;
  const long long total = static_cast<long long>(L) * kLaneQuarters;
  for (long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; t < total;
       t += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int site = static_cast<int>(t / kLaneQuarters), q = static_cast<int>(t % kLaneQuarters);
    const float* row = rows + static_cast<size_t>(site) * kRowArrays * Spad;
    const float* RR = row + 6 * Spad + q * SEG;
    const float* U = row + 5 * Spad + q * SEG;
    float* out = aux + static_cast<size_t>(site) * auxFloats;
    float p = 1.f;
    out[q * SEG + SEG - 1] = 1.f;
    for (int i = SEG - 2; i >= 0; --i) {
      p *= RR[i];
      out[q * SEG + i] = p;
    }
    float* bd = out + Spad + 4 * q;
    bd[0] = RR[SEG - 1];
    bd[1] = p;
    bd[2] = U[SEG - 1];
    bd[3] = 0.f;
  }
}

template <int S_T, int RQ, int G, int DEPTH> struct LaneSmem {
  using Geo = LaneGeom<S_T>;
  static constexpr size_t kCoefBytes = static_cast<size_t>(kRowArrays) * Geo::Spad * 4;
  static constexpr size_t kAuxBytes = static_cast<size_t>(Geo::kAuxFloats) * 4;
  static constexpr size_t kSlotBytes = G * (kCoefBytes + kAuxBytes);
  static constexpr size_t kConstOff = DEPTH * kSlotBytes;  // colRatios | prefix products | prior | quarter products
  static constexpr size_t kConstBytes = (3 * static_cast<size_t>(Geo::Spad) + 16) * 4;
  static constexpr size_t kParkOff = kConstOff + kConstBytes;  // per warp [4 RQ][32] floats: a segment's per-state sums
  static constexpr size_t kParkBytes = static_cast<size_t>(kLaneQuarters) * 4 * RQ * 32 * 4;
  static constexpr size_t kBarOff = (kParkOff + kParkBytes + 15) / 16 * 16;
  static constexpr size_t kTileOff = kBarOff + DEPTH * sizeof(uint64_t);
  static constexpr size_t kTotal = kTileOff + 16;
};

__device__ __forceinline__ float pick4(const int g, const float v0, const float v1, const float v2, const float v3)
{
  return g == 0 ? v0 : (g == 1 ? v1 : (g == 2 ? v2 : v3));
}

// ---- forward step.  x = alpha(p-1) (kept), y = unscaled alpha(p); returns sum_k x[k] over ALL states (ref: HMM.cpp:799-830)
template <int S> __device__ __forceinline__ float forwardLane(float (&x)[LaneGeom<S>::SEG], float (&y)[LaneGeom<S>::SEG],
                                                              const float* row, const int cls, const float* sCr,
                                                              const float* sCpre, const float* sCq, const int g, const int pl)
{
  using Geo = LaneGeom<S>;
  constexpr int SEGQ = Geo::SEGQ, Spad = Geo::Spad;
  const float4* E = reinterpret_cast<const float4*>(row + cls * Spad) + g * SEGQ;
  const float4* Dr = reinterpret_cast<const float4*>(row + 3 * Spad) + g * SEGQ;
  const float4* Br = reinterpret_cast<const float4*>(row + 4 * Spad) + g * SEGQ;
  const float4* Ur = reinterpret_cast<const float4*>(row + 5 * Spad) + g * SEGQ;
  const float4* Cr = reinterpret_cast<const float4*>(sCr) + g * SEGQ;
  const float4* Cp = reinterpret_cast<const float4*>(sCpre) + g * SEGQ;
  // pass 1: both scans from a zero carry-in.  y = AU'[k] + D[k] x[k] + B[k] (suffix sum inside the quarter)
  float au = 0.f;
#pragma unroll
  for (int q = 0; q < SEGQ; ++q) {
    const float4 d4 = Dr[q], u4 = Ur[q], c4 = Cr[q];
#pragma unroll
    for (int jp = 0; jp < 2; ++jp) {
      const int i = 4 * q + 2 * jp;
      const float2 xx = pk(x[i], x[i + 1]);
      const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), xx);
      const float au0 = au;
      const float au1 = fmaf(f4(c4, 2 * jp), au0, t.x);  // AU[k+1] = U[k] x[k] + colRatio[k] AU[k]
      au = fmaf(f4(c4, 2 * jp + 1), au1, t.y);
      const float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), xx, pk(au0, au1));
      y[i] = w.x;
      y[i + 1] = w.y;
    }
  }
  float run = 0.f;
#pragma unroll
  for (int q = SEGQ - 1; q >= 0; --q) {
    const float4 b4 = Br[q];
#pragma unroll
    for (int jp = 1; jp >= 0; --jp) {
      const int i = 4 * q + 2 * jp;
      const float s1 = run;
      const float s0 = s1 + x[i + 1];
      run = s0 + x[i];
      const float2 w = __ffma2_rn(pk(f4(b4, 2 * jp), f4(b4, 2 * jp + 1)), pk(s0, s1), pk(y[i], y[i + 1]));
      y[i] = w.x;
      y[i + 1] = w.y;
    }
  }
  // carries: AU entering quarter g, and the sum of x over the quarters above g
  const float a0 = __shfl_sync(kFull, au, pl), a1 = __shfl_sync(kFull, au, 8 + pl), a2 = __shfl_sync(kFull, au, 16 + pl);
  const float t0 = __shfl_sync(kFull, run, pl), t1 = __shfl_sync(kFull, run, 8 + pl), t2 = __shfl_sync(kFull, run, 16 + pl),
              t3 = __shfl_sync(kFull, run, 24 + pl);
  const float in2 = fmaf(sCq[1], a0, a1);
  const float in3 = fmaf(sCq[2], in2, a2);
  const float carryA = pick4(g, 0.f, a0, in2, in3);
  const float carryR = pick4(g, (t1 + t2) + t3, t2 + t3, t3, 0.f);
  // pass 2: alpha(p)[k] = E[k] (y[k] + prefix[k] carryA + B[k] carryR)
  const float2 cA = pk(carryA, carryA), cR = pk(carryR, carryR);
#pragma unroll
  for (int q = 0; q < SEGQ; ++q) {
    const float4 e4 = E[q], b4 = Br[q], p4 = Cp[q];
#pragma unroll
    for (int jp = 0; jp < 2; ++jp) {
      const int i = 4 * q + 2 * jp;
      float2 w = __ffma2_rn(pk(f4(p4, 2 * jp), f4(p4, 2 * jp + 1)), cA, pk(y[i], y[i + 1]));
      w = __ffma2_rn(pk(f4(b4, 2 * jp), f4(b4, 2 * jp + 1)), cR, w);
      w = __fmul2_rn(pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)), w);
      y[i] = w.x;
      y[i + 1] = w.y;
    }
  }
  return (t0 + t1) + (t2 + t3);
}

// ---- backward step.  x = beta(p+1) on entry (becomes beta * emission), y = unscaled beta(p) (ref: HMM.cpp:957-1016)
template <int S> __device__ __forceinline__ void backwardLane(float (&x)[LaneGeom<S>::SEG], float (&y)[LaneGeom<S>::SEG],
                                                              const float* row, const float* aux, const int cls, const int g,
                                                              const int pl)
{
  using Geo = LaneGeom<S>;
  constexpr int SEGQ = Geo::SEGQ, SEG = Geo::SEG, Spad = Geo::Spad;
  const float4* E = reinterpret_cast<const float4*>(row + cls * Spad) + g * SEGQ;
  const float4* Dr = reinterpret_cast<const float4*>(row + 3 * Spad) + g * SEGQ;
  const float4* Br = reinterpret_cast<const float4*>(row + 4 * Spad) + g * SEGQ;
  const float4* Rr = reinterpret_cast<const float4*>(row + 6 * Spad) + g * SEGQ;
  const float4* Us = reinterpret_cast<const float4*>(row + 7 * Spad) + g * SEGQ;  // Us[k] = U[k-1]
  const float4* Rp = reinterpret_cast<const float4*>(aux) + g * SEGQ;
  const float4* bd = reinterpret_cast<const float4*>(aux + Spad);
  // pass 1: vec = beta(p+1) * emission(p+1) in place; y = BL'[k] + D[k] vec[k] + BU'[k] with both scans from zero
  float bl = 0.f;
#pragma unroll
  for (int q = 0; q < SEGQ; ++q) {
    const float4 e4 = E[q], d4 = Dr[q], b4 = Br[q];
#pragma unroll
    for (int jp = 0; jp < 2; ++jp) {
      const int i = 4 * q + 2 * jp;
      const float2 v = __fmul2_rn(pk(x[i], x[i + 1]), pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)));
      x[i] = v.x;
      x[i + 1] = v.y;
      const float bl0 = bl;
      const float bl1 = fmaf(f4(b4, 2 * jp), v.x, bl0);  // BL[k+1] = BL[k] + B[k] vec[k]
      bl = fmaf(f4(b4, 2 * jp + 1), v.y, bl1);
      const float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), v, pk(bl0, bl1));
      y[i] = w.x;
      y[i + 1] = w.y;
    }
  }
  float bu = 0.f, above = 0.f;  // BU' of the state above, and U[k] vec[k+1] for the state k reached next
#pragma unroll
  for (int q = SEGQ - 1; q >= 0; --q) {
    const float4 u4 = Us[q], r4 = Rr[q];
#pragma unroll
    for (int jp = 1; jp >= 0; --jp) {
      const int i = 4 * q + 2 * jp;
      const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), pk(x[i], x[i + 1]));
      // BU[k] = U[k] vec[k+1] + RR[k] BU[k+1]; at the quarter's last state both inputs are the carry (0 here)
      const float b1 = i + 1 == SEG - 1 ? 0.f : fmaf(f4(r4, 2 * jp + 1), bu, above);
      const float b0 = fmaf(f4(r4, 2 * jp), b1, t.y);
      bu = b0;
      above = t.x;
      const float2 w = __fadd2_rn(pk(y[i], y[i + 1]), pk(b0, b1));
      y[i] = w.x;
      y[i + 1] = w.y;
    }
  }
  // carries: BL entering quarter g; X = true BU at the quarter's last state, from the quarters above
  const float l0 = __shfl_sync(kFull, bl, pl), l1 = __shfl_sync(kFull, bl, 8 + pl), l2 = __shfl_sync(kFull, bl, 16 + pl);
  const float u1 = __shfl_sync(kFull, bu, 8 + pl), u2 = __shfl_sync(kFull, bu, 16 + pl), u3 = __shfl_sync(kFull, bu, 24 + pl);
  const float v1 = __shfl_sync(kFull, x[0], 8 + pl), v2 = __shfl_sync(kFull, x[0], 16 + pl), v3 = __shfl_sync(kFull, x[0], 24 + pl);
  const float4 q0 = bd[0], q1 = bd[1], q2 = bd[2];  // {RR[last], Rp[first], U[last]} of quarters 0..2
  const float x2 = fmaf(q2.x, u3, q2.z * v3);       // (the top quarter's own carry is 0: BU[S-1] = 0)
  const float bu2 = fmaf(q2.y, x2, u2);
  const float x1 = fmaf(q1.x, bu2, q1.z * v2);
  const float bu1 = fmaf(q1.y, x1, u1);
  const float x0 = fmaf(q0.x, bu1, q0.z * v1);
  const float carryL = pick4(g, 0.f, l0, l0 + l1, (l0 + l1) + l2);
  const float carryX = pick4(g, x0, x1, x2, 0.f);
  // pass 2
  const float2 cL = pk(carryL, carryL), cX = pk(carryX, carryX);
#pragma unroll
  for (int q = 0; q < SEGQ; ++q) {
    const float4 p4 = Rp[q];
#pragma unroll
    for (int jp = 0; jp < 2; ++jp) {
      const int i = 4 * q + 2 * jp;
      const float2 w = __ffma2_rn(pk(f4(p4, 2 * jp), f4(p4, 2 * jp + 1)), cX, __fadd2_rn(pk(y[i], y[i + 1]), cL));
      y[i] = w.x;
      y[i + 1] = w.y;
    }
  }
  if (Geo::Spad > S && g == kLaneQuarters - 1) {
#pragma unroll
    for (int i = SEG - (Geo::Spad - S); i < SEG; ++i) {
      y[i] = 0.f;  // padding states carry nothing (their BL would leak into the scale factor)
    }
  }
}

template <int SEG> __device__ __forceinline__ float sumLane(const float (&a)[SEG])
{
  float2 s01 = pk(0.f, 0.f), s23 = pk(0.f, 0.f);
#pragma unroll
  for (int i = 0; i < SEG; i += 4) {
    s01 = __fadd2_rn(s01, pk(a[i], a[i + 1]));
    s23 = __fadd2_rn(s23, pk(a[i + 2], a[i + 3]));
  }
  float s = (s01.x + s01.y) + (s23.x + s23.y);
  s += __shfl_xor_sync(kFull, s, 8);
  s += __shfl_xor_sync(kFull, s, 16);
  return s;
}

template <int SEG> __device__ __forceinline__ void scaleLane(float (&a)[SEG], const float sc)
{
#pragma unroll
  for (int i = 0; i < SEG; i += 2) {
    const float2 v = __fmul2_rn(pk(a[i], a[i + 1]), pk(sc, sc));
    a[i] = v.x;
    a[i + 1] = v.y;
  }
}

// PairBits with the haplotype indices instead of row pointers (registers limit this kernel's occupancy)
struct LaneBits {
  uint32_t ha, hb;
  uint64_t x = 0, t = 0;
  int word = -1;
  __device__ __forceinline__ int cls(const DeviceModel& m, const int site)
  {
    const int w = site >> 6;
    if (w != word) {
      const uint64_t wa = __ldg(m.haps + static_cast<size_t>(ha) * m.wordsPerHap + w);
      const uint64_t wb = __ldg(m.haps + static_cast<size_t>(hb) * m.wordsPerHap + w);
      x = wa ^ wb;
      t = wa & wb;
      word = w;
    }
    const int bit = site & 63;
    return ((x >> bit) & 1ull) ? 1 : (((t >> bit) & 1ull) ? 2 : 0);
  }
};

template <int S_T, int RQ, int G, int DEPTH, int MIN_BLOCKS>
__global__ void __launch_bounds__(kLaneQuarters * 32, MIN_BLOCKS) decodeLaneKernel(const __grid_constant__ FastModel fm,
                                                                                 const __grid_constant__ DecodeArgs args)
{
  using Geo = LaneGeom<S_T>;
  using SM = LaneSmem<S_T, RQ, G, DEPTH>;
  constexpr int S = S_T, Spad = Geo::Spad, SEG = Geo::SEG, SEGQ = Geo::SEGQ;
  constexpr int NR = 4 * RQ - 1;  // beta entries of a record; entry NR is the scale divisor
  constexpr size_t kRowFloats = static_cast<size_t>(kRowArrays) * Spad;
  constexpr size_t kAuxFloats = Geo::kAuxFloats;
  constexpr uint32_t kCoefBytes = static_cast<uint32_t>(SM::kCoefBytes), kAuxBytes = static_cast<uint32_t>(SM::kAuxBytes);
  static_assert(NR <= SEG && G % 2 == 0, "records come from quarter 0; the two state vectors swap roles every step");

  extern __shared__ __align__(128) unsigned char smemRaw[];
  // (grid constants: emitSegment takes the model by reference; a by-value copy would live in local memory and every
  // threshold test of the consumers would be a local load)
  const DeviceModel& m = fm.base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 3, pl = lane & 7;
  const int K0 = g * SEG;
  float* sCr = reinterpret_cast<float*>(smemRaw + SM::kConstOff);
  float* sCpre = sCr + Spad;
  float* sPrior = sCpre + Spad;
  float* sCq = sPrior + Spad;
  float* park = reinterpret_cast<float*>(smemRaw + SM::kParkOff) + static_cast<size_t>(warp) * 4 * RQ * 32 + lane;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smemRaw + SM::kBarOff);
  volatile long long* tileSlot = reinterpret_cast<volatile long long*>(smemRaw + SM::kTileOff);
  auto coefArea = [&](const int slot) { return reinterpret_cast<float*>(smemRaw + static_cast<size_t>(slot) * SM::kSlotBytes); };
  auto auxArea = [&](const int slot) {
    return reinterpret_cast<float*>(smemRaw + static_cast<size_t>(slot) * SM::kSlotBytes + static_cast<size_t>(G) * kCoefBytes);
  };
  const bool leader = threadIdx.x == 0;
  for (int k = threadIdx.x; k < Spad; k += blockDim.x) {
    sCr[k] = k < S ? fm.colRatios[k < S ? k : 0] : 0.f;
    sPrior[k] = k < S ? fm.prior[k < S ? k : 0] : 0.f;
  }
  if (leader) {
    for (int i = 0; i < DEPTH; ++i) {
      mbarInit(&bars[i], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x < kLaneQuarters) {
    float c = 1.f;
    for (int i = 0; i < SEG; ++i) {
      sCpre[threadIdx.x * SEG + i] = c;
      c *= sCr[threadIdx.x * SEG + i];
    }
    sCq[threadIdx.x] = c;
  }
  __syncthreads();
  uint32_t parity = 0;

  const unsigned flags = args.flags;
  const bool wantSeg = flags & FSMC_CALL_SEGMENTS;
  const bool wantAge = (flags & FSMC_SEG_AGE) && wantSeg;
  const int sT = m.stateThreshold;
  float4* slab = reinterpret_cast<float4*>(args.scratch + static_cast<long long>(blockIdx.x) * args.scratchPerWarp);

  for (long long it = 0;; ++it) {
    if (leader) {
      tileSlot[it & 1] = static_cast<long long>(atomicAdd(args.tileCounter, 1ull));
    }
    __syncthreads();
    const long long t = tileSlot[it & 1];
    if (t >= args.numTiles) {
      break;
    }
    const int tile = args.order ? args.order[t] : static_cast<int>(t);
    const int nPairs = args.tilePairs[tile];
    const int from = args.tileFrom[tile];
    const int len = args.tileTo[tile] - from;
    const int scanFrom = wantSeg ? args.tileScanFrom[tile] : 0;
    const int scanTo = wantSeg ? args.tileScanTo[tile] : 0;
    const int pairInTile = warp * 8 + pl;
    const bool laneActive = pairInTile < nPairs;
    const int srcPair = laneActive ? pairInTile : nPairs - 1;
    const uint32_t pair = static_cast<uint32_t>(tile) * 32u + static_cast<uint32_t>(pairInTile);
    LaneBits bits;
    bits.ha = args.hapA[static_cast<size_t>(tile) * 32 + srcPair];
    bits.hb = args.hapB[static_cast<size_t>(tile) * 32 + srcPair];
    // record of window position p, quad q of this lane's pair: [p][q][pair in tile]
    auto recAt = [&](const int p, const int q) { return slab + (static_cast<size_t>(p) * RQ + q) * 32 + pairInTile; };

    float a[SEG], c[SEG];
    // per-state sums of the lane's current run: in this lane's column of the warp's parking area (emitSegment reads them
    // there with a stride of 32 floats); registers are what limits this kernel's occupancy
    if (g == 0) {
#pragma unroll
      for (int k = 0; k < NR; ++k) {
        park[k * 32] = 0.f;
      }
    }
    // (beta^[k < sT], 0.., scale divisor) of window position p: quarter-0 lanes only
    auto storeRecord = [&](const float (&v)[SEG], const int p, const float divisor) {
      if (g == 0) {
#pragma unroll
        for (int q = 0; q < RQ; ++q) {
          float w[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int k = 4 * q + i;
            w[i] = k == NR ? divisor : (k < sT ? v[k] : 0.f);
          }
          *recAt(p, q) = make_float4(w[0], w[1], w[2], w[3]);
        }
      }
    };

    // ---- sweep 1: backward.  Step j handles window position len-2-j with the coefficient row of len-1-j -------------
    {
      const int steps = len - 1;
      const int nGroups = (steps + G - 1) / G;
      auto prefetch = [&](const int gi) {  // rows of the steps [j0, j1): window positions [len-j1, len-j0), ascending
        const int j0 = gi * G, j1 = min(steps, j0 + G);
        const int slot = gi % DEPTH;
        const uint32_t n = static_cast<uint32_t>(j1 - j0);
        mbarExpectTx(&bars[slot], n * (kCoefBytes + kAuxBytes));
        bulkLoad(coefArea(slot), m.siteRows + static_cast<size_t>(from + len - j1) * kRowFloats, n * kCoefBytes, &bars[slot]);
        bulkLoad(auxArea(slot), m.laneAux + static_cast<size_t>(from + len - j1) * kAuxFloats, n * kAuxBytes, &bars[slot]);
      };
      if (leader) {
        for (int gi = 0; gi < DEPTH && gi < nGroups; ++gi) {
          prefetch(gi);
        }
      }
#pragma unroll
      for (int i = 0; i < SEG; ++i) {
        a[i] = K0 + i < S ? 1.f : 0.f;  // beta at the last site: all ones (any positive scale is equivalent)
      }
      storeRecord(a, len - 1, 1.0f);
      for (int gi = 0; gi < nGroups; ++gi) {
        const int slot = gi % DEPTH;
        const int j0 = gi * G;
        const int n = min(G, steps - j0);
        const float* coef = coefArea(slot);
        const float* aux = auxArea(slot);
        mbarWait(&bars[slot], (parity >> slot) & 1u);
        parity ^= 1u << slot;
        auto step = [&](const int i, float (&x)[SEG], float (&y)[SEG]) {
          const int p = len - 2 - (j0 + i);
          const int cls = bits.cls(m, from + p + 1);
          backwardLane<S>(x, y, coef + static_cast<size_t>(n - 1 - i) * kRowFloats, aux + static_cast<size_t>(n - 1 - i) * kAuxFloats,
                          cls, g, pl);
          float divisor = 1.0f;
          if (i == G - 1) {  // last step of a full group
            divisor = sumLane<SEG>(y);
            scaleLane<SEG>(y, 1.0f / divisor);
          }
          storeRecord(y, p, divisor);
        };
#pragma unroll 1
        for (int i = 0; i < G; i += 2) {
          if (i < n) {
            step(i, a, c);
          }
          if (i + 1 < n) {
            step(i + 1, c, a);
          }
        }
        __syncthreads();  // every warp is done with the slot
        if (leader && gi + DEPTH < nGroups) {
          prefetch(gi + DEPTH);
        }
      }
      if (!(steps & 1)) {  // beta^ of the first site ended in a; the forward sweep wants it in c
#pragma unroll
        for (int k = 0; k < SEG; ++k) {
          c[k] = a[k];
        }
      }
    }

    // ---- sweep 2: forward + consumers (quarter-0 lanes) --------------------------------------------------------------
    {
      const int nGroups = (len + G - 1) / G;
      auto prefetch = [&](const int gi) {
        const int p0 = gi * G;
        const uint32_t n = static_cast<uint32_t>(min(G, len - p0));
        const int slot = gi % DEPTH;
        mbarExpectTx(&bars[slot], n * (kCoefBytes + kAuxBytes));
        bulkLoad(coefArea(slot), m.siteRows + static_cast<size_t>(from + p0) * kRowFloats, n * kCoefBytes, &bars[slot]);
        bulkLoad(auxArea(slot), m.laneAux + static_cast<size_t>(from + p0) * kAuxFloats, n * kAuxBytes, &bars[slot]);
      };
      if (leader) {
        for (int gi = 0; gi < DEPTH && gi < nGroups; ++gi) {
          prefetch(gi);
        }
      }
      CallerState cs;
      float Z = 1.f, bPrev = 1.f;

      // consumers of window position p (quarter-0 lanes); v = alpha^(p)
      auto consume = [&](const int p, const float (&v)[SEG], const float4 (&rec)[RQ]) {
        const int site = from + p;
        float q[4 * RQ];  // alpha^[k] beta^[k] for k < sT (0 above); q[NR] = b_p
#pragma unroll
        for (int qq = 0; qq < RQ; ++qq) {
          const float4 r4 = rec[qq];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            q[4 * qq + i] = f4(r4, i);
          }
        }
        bPrev = q[NR];
        float ibdRaw = 0.f;
#pragma unroll
        for (int k = 0; k < NR; ++k) {
          q[k] *= v[k];
          ibdRaw += q[k];
        }
        const float r = 1.0f / Z;
        const float ibd = ibdRaw * r;
        if ((flags & FSMC_SITE_IBD) && laneActive) {
          args.siteIbd[static_cast<size_t>(pair) * args.siteStride + p] = ibd;
        }
        const bool inScan = wantSeg && site >= scanFrom && site < scanTo;
        if (inScan) {
          int now = ibd >= m.thr[0] ? 0 : (ibd >= m.thr[1] ? 1 : (ibd >= m.thr[2] ? 2 : (ibd >= m.thr[3] ? 3 : -1)));
          if (!laneActive) {
            now = -1;
          }
          const bool changed = now != cs.level;
          const bool ending = changed && cs.level >= 0;
          const bool closing = now >= 0 && site == scanTo - 1;
          const float rr = now >= 0 ? r : 0.f;
          const float keep = changed ? 0.f : 1.f;
          if (ending) {
            emitSegment<false>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, park, wantAge);
          }
          if (wantAge && (now >= 0 || changed)) {
            // per-state sums of the current run (ref: HMM.cpp:1209-1218); a run that just ended leaves zeros
#pragma unroll
            for (int k = 0; k < NR; ++k) {
              park[k * 32] = fmaf(q[k], rr, keep * park[k * 32]);
            }
          }
          if (closing) {
            emitSegment<false>(m, args, pair, changed ? site : cs.start, site, changed ? ibd : cs.prob + ibd, now, park, wantAge);
          }
          cs.prob = (now >= 0 && !closing) ? (changed ? ibd : cs.prob + ibd) : 0.f;
          cs.start = (now >= 0 && changed) ? site : cs.start;
          cs.level = now;
        }
      };

      for (int gi = 0; gi < nGroups; ++gi) {
        const int slot = gi % DEPTH;
        const int p0 = gi * G;
        const int n = min(G, len - p0);
        const float* coef = coefArea(slot);
        mbarWait(&bars[slot], (parity >> slot) & 1u);
        parity ^= 1u << slot;
        auto step = [&](const int i, float (&x)[SEG], float (&y)[SEG]) {
          const int p = p0 + i;
          const int cls = bits.cls(m, from + p);
          float4 rec[RQ];  // this position's record: in flight while the step is computed
#pragma unroll
          for (int qq = 0; qq < RQ; ++qq) {
            rec[qq] = *recAt(p, qq);
          }
          const float total = forwardLane<S>(x, y, coef + static_cast<size_t>(i) * kRowFloats, cls, sCr, sCpre, sCq, g, pl);
          float sc = 1.0f;
          if (i == G - 1) {
            sc = 1.0f / total;  // sum of alpha^(p-1): keeps alpha in range (any positive scale is equivalent)
            scaleLane<SEG>(y, sc);
          }
          if (g == 0) {
            Z *= bPrev * sc;  // Z_p = Z_{p-1} * b_{p-1} / a_p
            consume(p, y, rec);
          }
        };
#pragma unroll 1
        for (int i = 0; i < G; i += 2) {
          if (i == 0 && gi == 0) {
            // p = 0: alpha^(0) = prior * emission into a; the one exact normaliser Z_0 = sum_k alpha^(0)[k] beta^(0)[k]
            const int cls = bits.cls(m, from);
            float4 rec[RQ];
#pragma unroll
            for (int qq = 0; qq < RQ; ++qq) {
              rec[qq] = *recAt(0, qq);
            }
            const float4* E = reinterpret_cast<const float4*>(coef + cls * Spad) + g * SEGQ;
            const float4* P = reinterpret_cast<const float4*>(sPrior) + g * SEGQ;
            float2 z01 = pk(0.f, 0.f), z23 = pk(0.f, 0.f);
#pragma unroll
            for (int q = 0; q < SEGQ; ++q) {
              const float4 e4 = E[q], p4 = P[q];
              const float2 lo = __fmul2_rn(pk(p4.x, p4.y), pk(e4.x, e4.y)), hi = __fmul2_rn(pk(p4.z, p4.w), pk(e4.z, e4.w));
              a[4 * q] = lo.x;
              a[4 * q + 1] = lo.y;
              a[4 * q + 2] = hi.x;
              a[4 * q + 3] = hi.y;
              z01 = __ffma2_rn(lo, pk(c[4 * q], c[4 * q + 1]), z01);
              z23 = __ffma2_rn(hi, pk(c[4 * q + 2], c[4 * q + 3]), z23);
            }
            float z = (z01.x + z01.y) + (z23.x + z23.y);
            z += __shfl_xor_sync(kFull, z, 8);
            z += __shfl_xor_sync(kFull, z, 16);
            if (g == 0) {
              Z = z;
              consume(0, a, rec);
            }
          } else if (i < n) {
            step(i, c, a);
          }
          if (i + 1 < n) {
            step(i + 1, a, c);
          }
        }
        __syncthreads();  // every warp is done with the slot
        if (leader && gi + DEPTH < nGroups) {
          prefetch(gi + DEPTH);
        }
      }
    }
  }
}

}  // namespace fsmc

namespace fsmc
{

// -------------------------------------------------------------------------------------------------------------------
// decodeLaneWideKernel: the same lane-split sweeps when every state reaches the consumers (per-site posterior mean / MAP,
// per-segment age estimates over all states: `noConditionalAgeEstimates`).  Full beta rows stream through HBM: a lane
// writes its own 40 states per site ([pos][state quad][pair in tile][4]: the 8 lanes of a quarter write 128 contiguous
// bytes) and reads them back in the forward sweep into the registers of the dead alpha(p-1).  The posterior's
// normaliser, mean and argmax are reduced across the four quarters with shuffles; every lane of a pair runs the
// run-length state machine of the segment caller on the same numbers, quarter 0 emits.  The per-state sums of a run
// (FSMC_SEG_AGE) live in shared memory, [state][pair in tile] — emitSegment's layout — and are touched only while a
// pair of the warp is inside a run.
// -------------------------------------------------------------------------------------------------------------------
template <int S_T, int G, int DEPTH> struct LaneWideSmem {
  using Base = LaneSmem<S_T, 1, G, DEPTH>;
  using Geo = LaneGeom<S_T>;
  static constexpr size_t kExpOff = Base::kTotal;                                     // expected times [Spad]
  static constexpr size_t kAccOff = (kExpOff + static_cast<size_t>(Geo::Spad) * 4 + 127) / 128 * 128;  // [Spad][32]
  static constexpr size_t kTotal = kAccOff + static_cast<size_t>(Geo::Spad) * 32 * 4;
};

template <int S_T, int G, int DEPTH, int MIN_BLOCKS>
__global__ void __launch_bounds__(kLaneQuarters * 32, MIN_BLOCKS) decodeLaneWideKernel(const __grid_constant__ FastModel fm,
                                                                                     const __grid_constant__ DecodeArgs args)
{
  using Geo = LaneGeom<S_T>;
  using SM = LaneSmem<S_T, 1, G, DEPTH>;
  using SMW = LaneWideSmem<S_T, G, DEPTH>;
  constexpr int S = S_T, Spad = Geo::Spad, SEG = Geo::SEG, SEGQ = Geo::SEGQ, SQ = Geo::SQ;
  constexpr size_t kRowFloats = static_cast<size_t>(kRowArrays) * Spad;
  constexpr size_t kAuxFloats = Geo::kAuxFloats;
  constexpr uint32_t kCoefBytes = static_cast<uint32_t>(SM::kCoefBytes), kAuxBytes = static_cast<uint32_t>(SM::kAuxBytes);
  static_assert(G % 2 == 0, "the two state vectors swap roles every step");

  extern __shared__ __align__(128) unsigned char smemRaw[];
  const DeviceModel& m = fm.base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 3, pl = lane & 7;
  const int K0 = g * SEG;
  float* sCr = reinterpret_cast<float*>(smemRaw + SM::kConstOff);
  float* sCpre = sCr + Spad;
  float* sPrior = sCpre + Spad;
  float* sCq = sPrior + Spad;
  float* sExp = reinterpret_cast<float*>(smemRaw + SMW::kExpOff);
  float* sAcc = reinterpret_cast<float*>(smemRaw + SMW::kAccOff);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smemRaw + SM::kBarOff);
  volatile long long* tileSlot = reinterpret_cast<volatile long long*>(smemRaw + SM::kTileOff);
  auto coefArea = [&](const int slot) { return reinterpret_cast<float*>(smemRaw + static_cast<size_t>(slot) * SM::kSlotBytes); };
  auto auxArea = [&](const int slot) {
    return reinterpret_cast<float*>(smemRaw + static_cast<size_t>(slot) * SM::kSlotBytes + static_cast<size_t>(G) * kCoefBytes);
  };
  const bool leader = threadIdx.x == 0;
  for (int k = threadIdx.x; k < Spad; k += blockDim.x) {
    sCr[k] = k < S ? fm.colRatios[k < S ? k : 0] : 0.f;
    sPrior[k] = k < S ? fm.prior[k < S ? k : 0] : 0.f;
    sExp[k] = k < S ? fm.expTimes[k < S ? k : 0] : 0.f;
  }
  if (leader) {
    for (int i = 0; i < DEPTH; ++i) {
      mbarInit(&bars[i], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x < kLaneQuarters) {
    float c = 1.f;
    for (int i = 0; i < SEG; ++i) {
      sCpre[threadIdx.x * SEG + i] = c;
      c *= sCr[threadIdx.x * SEG + i];
    }
    sCq[threadIdx.x] = c;
  }
  __syncthreads();
  uint32_t parity = 0;

  const unsigned flags = args.flags;
  const bool wantSeg = flags & FSMC_CALL_SEGMENTS;
  const bool wantAge = (flags & FSMC_SEG_AGE) && wantSeg;
  const bool wantSite = flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP);
  const int sT = m.stateThreshold;
  const int nAcc = m.ageThreshold;
  float4* slab = reinterpret_cast<float4*>(args.scratch + static_cast<long long>(blockIdx.x) * args.scratchPerWarp);

  for (long long it = 0;; ++it) {
    if (leader) {
      tileSlot[it & 1] = static_cast<long long>(atomicAdd(args.tileCounter, 1ull));
    }
    __syncthreads();
    const long long t = tileSlot[it & 1];
    if (t >= args.numTiles) {
      break;
    }
    const int tile = args.order ? args.order[t] : static_cast<int>(t);
    const int nPairs = args.tilePairs[tile];
    const int from = args.tileFrom[tile];
    const int len = args.tileTo[tile] - from;
    const int scanFrom = wantSeg ? args.tileScanFrom[tile] : 0;
    const int scanTo = wantSeg ? args.tileScanTo[tile] : 0;
    const int pairInTile = warp * 8 + pl;
    const bool laneActive = pairInTile < nPairs;
    const int srcPair = laneActive ? pairInTile : nPairs - 1;
    const uint32_t pair = static_cast<uint32_t>(tile) * 32u + static_cast<uint32_t>(pairInTile);
    const uint32_t outRow = args.laneRow ? __ldg(args.laneRow + pair) : pair;  // output row (fsmc_decode_device)
    PairBits bits;
    bits.a = m.haps + static_cast<size_t>(args.hapA[static_cast<size_t>(tile) * 32 + srcPair]) * m.wordsPerHap;
    bits.b = m.haps + static_cast<size_t>(args.hapB[static_cast<size_t>(tile) * 32 + srcPair]) * m.wordsPerHap;
    const float* rowBase = m.siteRows + static_cast<size_t>(from) * kRowFloats;
    const float* auxBase = fm.base.laneAux + static_cast<size_t>(from) * kAuxFloats;
    // this lane's part of the beta row of window position p: quads [g SEGQ, (g+1) SEGQ) of [p][quad][pair in tile]
    auto betaAt = [&](const int p, const int q) { return slab + (static_cast<size_t>(p) * SQ + g * SEGQ + q) * 32 + pairInTile; };
    auto storeBeta = [&](const float (&v)[SEG], const int p) {
#pragma unroll
      for (int q = 0; q < SEGQ; ++q) {
        *betaAt(p, q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
      }
    };
    float* accCol = sAcc + static_cast<size_t>(K0) * 32 + pairInTile;  // [state K0 + i][pair]: entry i at accCol[i * 32]

    float a[SEG], c[SEG];
    if (wantAge) {
#pragma unroll
      for (int i = 0; i < SEG; ++i) {
        accCol[i * 32] = 0.f;
      }
    }

    // ---- sweep 1: backward ---------------------------------------------------------------------------------------------
    {
      const int steps = len - 1;
      const int nGroups = (steps + G - 1) / G;
      auto prefetch = [&](const int gi) {
        const int j0 = gi * G, j1 = min(steps, j0 + G);
        const int slot = gi % DEPTH;
        const uint32_t n = static_cast<uint32_t>(j1 - j0);
        mbarExpectTx(&bars[slot], n * (kCoefBytes + kAuxBytes));
        bulkLoad(coefArea(slot), rowBase + static_cast<size_t>(len - j1) * kRowFloats, n * kCoefBytes, &bars[slot]);
        bulkLoad(auxArea(slot), auxBase + static_cast<size_t>(len - j1) * kAuxFloats, n * kAuxBytes, &bars[slot]);
      };
      if (leader) {
        for (int gi = 0; gi < DEPTH && gi < nGroups; ++gi) {
          prefetch(gi);
        }
      }
#pragma unroll
      for (int i = 0; i < SEG; ++i) {
        a[i] = K0 + i < S ? 1.f : 0.f;
      }
      storeBeta(a, len - 1);
      for (int gi = 0; gi < nGroups; ++gi) {
        const int slot = gi % DEPTH;
        const int j0 = gi * G;
        const int n = min(G, steps - j0);
        const float* coef = coefArea(slot);
        const float* aux = auxArea(slot);
        mbarWait(&bars[slot], (parity >> slot) & 1u);
        parity ^= 1u << slot;
        auto step = [&](const int i, float (&x)[SEG], float (&y)[SEG]) {
          const int p = len - 2 - (j0 + i);
          const int cls = bits.cls(from + p + 1);
          backwardLane<S>(x, y, coef + static_cast<size_t>(n - 1 - i) * kRowFloats, aux + static_cast<size_t>(n - 1 - i) * kAuxFloats,
                          cls, g, pl);
          if (i == G - 1) {
            scaleLane<SEG>(y, 1.0f / sumLane<SEG>(y));
          }
          storeBeta(y, p);
        };
#pragma unroll 1
        for (int i = 0; i < G; i += 2) {
          if (i < n) {
            step(i, a, c);
          }
          if (i + 1 < n) {
            step(i + 1, c, a);
          }
        }
        __syncthreads();
        if (leader && gi + DEPTH < nGroups) {
          prefetch(gi + DEPTH);
        }
      }
    }

    // ---- sweep 2: forward + fused consumers (ref: HMM.cpp:725-879, 669-692, 1179-1357, 1378-1409) ------------------------
    {
      const int nGroups = (len + G - 1) / G;
      auto prefetch = [&](const int gi) {
        const int p0 = gi * G;
        const uint32_t n = static_cast<uint32_t>(min(G, len - p0));
        const int slot = gi % DEPTH;
        mbarExpectTx(&bars[slot], n * (kCoefBytes + kAuxBytes));
        bulkLoad(coefArea(slot), rowBase + static_cast<size_t>(p0) * kRowFloats, n * kCoefBytes, &bars[slot]);
        bulkLoad(auxArea(slot), auxBase + static_cast<size_t>(p0) * kAuxFloats, n * kAuxBytes, &bars[slot]);
      };
      if (leader) {
        for (int gi = 0; gi < DEPTH && gi < nGroups; ++gi) {
          prefetch(gi);
        }
      }
      CallerState cs;

      // consumers of window position p: v = alpha(p) (this lane's states); w = the dead vector, receives beta, then alpha*beta
      auto consume = [&](const int p, const float (&v)[SEG], float (&w)[SEG]) {
        const int site = from + p;
        float2 z01 = pk(0.f, 0.f), z23 = pk(0.f, 0.f);
#pragma unroll
        for (int q = 0; q < SEGQ; ++q) {
          const float4 b4 = *betaAt(p, q);
          const float2 lo = __fmul2_rn(pk(v[4 * q], v[4 * q + 1]), pk(b4.x, b4.y));
          const float2 hi = __fmul2_rn(pk(v[4 * q + 2], v[4 * q + 3]), pk(b4.z, b4.w));
          w[4 * q] = lo.x;
          w[4 * q + 1] = lo.y;
          w[4 * q + 2] = hi.x;
          w[4 * q + 3] = hi.y;
          z01 = __fadd2_rn(z01, lo);
          z23 = __fadd2_rn(z23, hi);
        }
        float z = (z01.x + z01.y) + (z23.x + z23.y);
        z += __shfl_xor_sync(kFull, z, 8);
        z += __shfl_xor_sync(kFull, z, 16);
        const float r = 1.0f / z;  // ref HMM.cpp:681-685
        const bool inScan = wantSeg && site >= scanFrom && site < scanTo;
        const bool wantIbd = (flags & FSMC_SITE_IBD) || inScan;
        if (wantSite) {
          float mean = 0.f, best = 0.f;
          int arg = K0;
#pragma unroll
          for (int i = 0; i < SEG; ++i) {
            mean = fmaf(w[i], sExp[K0 + i], mean);
            if (best < w[i]) {  // first maximum, as the reference's ascending scan
              best = w[i];
              arg = K0 + i;
            }
          }
#pragma unroll
          for (int d = 8; d <= 16; d <<= 1) {
            mean += __shfl_xor_sync(kFull, mean, d);
            const float ob = __shfl_xor_sync(kFull, best, d);
            const int oa = __shfl_xor_sync(kFull, arg, d);
            if (ob > best || (ob == best && oa < arg)) {
              best = ob;
              arg = oa;
            }
          }
          if (g == 0 && laneActive) {
            if (flags & FSMC_SITE_MEAN) {
              args.siteMean[static_cast<size_t>(outRow) * args.siteStride + p] = mean * r;
            }
            if (flags & FSMC_SITE_MAP) {
              args.siteMap[static_cast<size_t>(outRow) * args.siteStride + p] = best > 0.f ? arg : 0;
            }
          }
        }
        if (wantIbd) {
          float ibdRaw = 0.f;
          forStatesBelow<SEG>(sT, [&](const int k) { ibdRaw += w[k]; });  // meaningful in quarter 0 (sT <= SEG)
          const float ibd = __shfl_sync(kFull, ibdRaw, pl) * r;
          if ((flags & FSMC_SITE_IBD) && g == 0 && laneActive) {
            args.siteIbd[static_cast<size_t>(outRow) * args.siteStride + p] = ibd;
          }
          if (inScan) {
            // every lane of a pair runs the same run-length state machine on the same numbers; quarter 0 emits
            int now = ibd >= m.thr[0] ? 0 : (ibd >= m.thr[1] ? 1 : (ibd >= m.thr[2] ? 2 : (ibd >= m.thr[3] ? 3 : -1)));
            if (!laneActive) {
              now = -1;
            }
            const bool changed = now != cs.level;
            const bool ending = changed && cs.level >= 0;  // the run that ended at site-1 is written now
            const bool closing = now >= 0 && site == scanTo - 1;
            if (__any_sync(kFull, ending)) {
              __syncwarp();  // the sums of the four quarters are in shared memory
              if (g == 0 && ending) {
                emitSegment<false>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, sAcc + pairInTile, wantAge);
              }
              __syncwarp();
            }
            if (wantAge && __any_sync(kFull, now >= 0 || changed)) {
              // per-state sums of the current run (ref: HMM.cpp:1209-1218,1229,1257,1284,1311)
              if (now >= 0 || changed) {
                const float rr = now >= 0 ? r : 0.f;
                const float keep = changed ? 0.f : 1.f;
#pragma unroll
                for (int i = 0; i < SEG; ++i) {
                  if (K0 + i < nAcc) {
                    accCol[i * 32] = fmaf(w[i], rr, keep * accCol[i * 32]);
                  }
                }
              }
            }
            if (__any_sync(kFull, closing)) {
              __syncwarp();
              if (g == 0 && closing) {
                emitSegment<false>(m, args, pair, changed ? site : cs.start, site, changed ? ibd : cs.prob + ibd, now,
                                   sAcc + pairInTile, wantAge);
              }
              __syncwarp();
            }
            cs.prob = (now >= 0 && !closing) ? (changed ? ibd : cs.prob + ibd) : 0.f;
            cs.start = (now >= 0 && changed) ? site : cs.start;
            cs.level = now;
          }
        }
      };

      for (int gi = 0; gi < nGroups; ++gi) {
        const int slot = gi % DEPTH;
        const int p0 = gi * G;
        const int n = min(G, len - p0);
        const float* coef = coefArea(slot);
        mbarWait(&bars[slot], (parity >> slot) & 1u);
        parity ^= 1u << slot;
        auto step = [&](const int i, float (&x)[SEG], float (&y)[SEG]) {
          const int p = p0 + i;
          const int cls = bits.cls(from + p);
          const float total = forwardLane<S>(x, y, coef + static_cast<size_t>(i) * kRowFloats, cls, sCr, sCpre, sCq, g, pl);
          if (i == G - 1) {
            scaleLane<SEG>(y, 1.0f / total);
          }
          consume(p, y, x);
        };
#pragma unroll 1
        for (int i = 0; i < G; i += 2) {
          if (i == 0 && gi == 0) {
            // p = 0: alpha(from)[k] = prior[k] * emission  (ref HMM.cpp:736-743)
            const int cls = bits.cls(from);
            const float4* E = reinterpret_cast<const float4*>(coef + cls * Spad) + g * SEGQ;
            const float4* P = reinterpret_cast<const float4*>(sPrior) + g * SEGQ;
#pragma unroll
            for (int q = 0; q < SEGQ; ++q) {
              const float4 e4 = E[q], p4 = P[q];
              const float2 lo = __fmul2_rn(pk(p4.x, p4.y), pk(e4.x, e4.y)), hi = __fmul2_rn(pk(p4.z, p4.w), pk(e4.z, e4.w));
              a[4 * q] = lo.x;
              a[4 * q + 1] = lo.y;
              a[4 * q + 2] = hi.x;
              a[4 * q + 3] = hi.y;
            }
            consume(0, a, c);
          } else if (i < n) {
            step(i, c, a);
          }
          if (i + 1 < n) {
            step(i + 1, a, c);
          }
        }
        __syncthreads();
        if (leader && gi + DEPTH < nGroups) {
          prefetch(gi + DEPTH);
        }
      }
    }
  }
}

}  // namespace fsmc
