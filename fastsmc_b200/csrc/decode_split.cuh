// fastsmc_b200 — state-split decode kernels for sm_100a: one 32-pair tile per CTA, the state vector cut into NW
// contiguous segments, one warp per segment (lane = pair in every warp).
//
// Why: with one warp per tile (decode_fast.cuh) a lane holds two whole state vectors, which caps the SM at 8 warps
// at S=69 (255 registers) and does not fit at all at S=159 (the FASTSMC_EXAMPLE table).  Cutting the states across
// NW warps divides the register footprint by NW, so twice (or four times) as many warps are resident and the
// dependent-FMA chains of the recurrences are hidden by other warps instead of by nothing.
//
// The linear-time transition recurrences (ref: HMM.cpp:787-879, 943-1041) are two first-order scans over the states in
// opposite directions (forward: AU ascending, suffix sums descending; backward: BL ascending, BU descending).  A scan
// crosses a segment boundary with one carried scalar per lane, so a step is a pipeline of NW stages: in stage s warp s
// runs its piece of the ascending scan and warp NW-1-s its piece of the descending one; carries travel through shared
// memory, stages are separated by a CTA barrier.  Each warp therefore touches each of its states exactly twice per
// step, the second time completing it — the same instructions as the one-warp kernel, no fix-up arithmetic.
//
// Rescaling (only there to keep fp32 in range: the posterior is invariant to the scale of alpha and of beta) uses a
// normaliser that is one site old, so that it can ride on the next step's carry exchange instead of costing a barrier.
//
// Two variants, as in decode_fast.cuh:
//   RQ == 0  "wide":   full beta rows stream through HBM (each warp copies its own segment with cp.async.bulk); all
//                      states reach the consumers (per-site mean / MAP, age estimates over all states);
//   RQ  > 0  "narrow": only beta[k < stateThreshold] and the scale divisor are kept per pair-site (4*RQ floats); the
//                      posterior normaliser is carried by the scale-factor recurrence (see decodeNarrowKernel).
#pragma once

#include "decode_fast.cuh"

namespace fsmc
{

template <int S_T, int NW> struct SplitGeom {
  static constexpr int SQ = (S_T + 3) / 4;
  static constexpr int Spad = SQ * 4;
  static constexpr int SEGQ = (SQ + NW - 1) / NW;  // quads per warp
  static constexpr int SEG = SEGQ * 4;             // states per warp
  static_assert(NW >= 2 && NW % 2 == 0, "segments pair up: warp g runs the ascending scan first iff g < NW/2");
  static_assert(SEGQ * NW == SQ, "the state quads must divide evenly among the warps");
};

// exchange area in shared memory: [parity][kind][warp or boundary][lane]
enum SplitKind { kXAsc = 0, kXDesc, kXVec, kXPart, kXIbd, kXMean, kXBest, kXArg, kXKinds };
template <int NW> struct SplitXch {
  float v[2][kXKinds][NW][32];
};

__device__ __forceinline__ void ctaBarrier()
{
  asm volatile("bar.sync 0;" ::: "memory");
}

// ---- one forward step: x = alpha(p-1) (kept), y = unscaled alpha(p).  ref: HMM.cpp:799-830 -------------------------
// Warps below the middle run the AU scan first (y = AU + D x) and complete y in the suffix-sum pass; warps above the
// middle take the suffix sums first and complete y in the AU pass.  Returns sum_k x[k] on warp 0.
template <int S, int NW, int GID, class F>
__device__ __forceinline__ float forwardSplit(const float* __restrict__ colRatios, float (&x)[SplitGeom<S, NW>::SEG],
                                              float (&y)[SplitGeom<S, NW>::SEG], const float* row, const int cls,
                                              float (*xc)[NW][32], const int lane, F&& afterFirstBarrier)
{
  using G = SplitGeom<S, NW>;
  constexpr int SEGQ = G::SEGQ, SEG = G::SEG, Spad = G::Spad, K0 = GID * SEG, Q0 = GID * SEGQ;
  constexpr bool LOWER = GID < NW / 2;
  const float4* E = reinterpret_cast<const float4*>(row + cls * Spad) + Q0;
  const float4* Dr = reinterpret_cast<const float4*>(row + 3 * Spad) + Q0;
  const float4* Br = reinterpret_cast<const float4*>(row + 4 * Spad) + Q0;
  const float4* Ur = reinterpret_cast<const float4*>(row + 5 * Spad) + Q0;
  float total = 0.f;
#pragma unroll
  for (int s = 0; s < NW; ++s) {
    if (s == GID) {
      float au = GID == 0 ? 0.f : xc[kXAsc][GID - 1][lane];
#pragma unroll
      for (int q = 0; q < SEGQ; ++q) {
        const float4 d4 = Dr[q], u4 = Ur[q];
        float4 e4 = make_float4(0.f, 0.f, 0.f, 0.f), b4 = e4;
        if (!LOWER) {
          e4 = E[q];
          b4 = Br[q];
        }
#pragma unroll
        for (int jp = 0; jp < 2; ++jp) {
          const int i = 4 * q + 2 * jp, k = K0 + i;
          if (k + 1 < S) {
            // two neighbouring states per packed instruction; only the AU chain itself is scalar (decode_fast.cuh)
            const float2 xx = pk(x[i], x[i + 1]);
            const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), xx);
            const float au0 = au;
            const float au1 = fmaf(colRatios[k], au0, t.x);  // AU[k+1] = U[k] x[k] + colRatio[k] AU[k]
            au = fmaf(colRatios[k + 1], au1, t.y);
            float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), xx, pk(au0, au1));  // AU[k] + D[k] x[k]
            if (!LOWER) {
              // (the last state's suffix sum is 0, so its B term adds nothing)
              w = __fmul2_rn(pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)),
                             __ffma2_rn(pk(f4(b4, 2 * jp), f4(b4, 2 * jp + 1)), pk(y[i], y[i + 1]), w));
            }
            y[i] = w.x;
            y[i + 1] = w.y;
          } else {
            if (k < S) {
              const float t = fmaf(f4(d4, 2 * jp), x[i], au);
              y[i] = LOWER ? t : f4(e4, 2 * jp) * (k < S - 1 ? fmaf(f4(b4, 2 * jp), y[i], t) : t);
              au = fmaf(colRatios[k < S ? k : 0], au, f4(u4, 2 * jp) * x[i]);
            } else {
              y[i] = 0.f;
            }
            y[i + 1] = 0.f;
          }
        }
      }
      if (GID < NW - 1) {
        xc[kXAsc][GID][lane] = au;
      }
    }
    if (s == NW - 1 - GID) {
      float run = GID == NW - 1 ? 0.f : xc[kXDesc][GID][lane];
#pragma unroll
      for (int q = SEGQ - 1; q >= 0; --q) {
        float4 e4 = make_float4(0.f, 0.f, 0.f, 0.f), b4 = e4;
        if (LOWER) {
          e4 = E[q];
          b4 = Br[q];
        }
#pragma unroll
        for (int jp = 1; jp >= 0; --jp) {
          const int i = 4 * q + 2 * jp, k = K0 + i;
          if (k + 1 < S) {
            const float s1 = run;  // sum_{j>k+1} x[j]
            const float s0 = s1 + x[i + 1];
            run = s0 + x[i];
            if (LOWER) {
              // E (AU + D x + B sum_{j>k} x[j])
              const float2 w = __fmul2_rn(pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)),
                                          __ffma2_rn(pk(f4(b4, 2 * jp), f4(b4, 2 * jp + 1)), pk(s0, s1), pk(y[i], y[i + 1])));
              y[i] = w.x;
              y[i + 1] = w.y;
            } else {
              y[i] = s0;
              y[i + 1] = s1;
            }
          } else if (k < S) {
            if (LOWER) {
              y[i] = f4(e4, 2 * jp) * fmaf(f4(b4, 2 * jp), run, y[i]);
            } else {
              y[i] = run;
            }
            run += x[i];
          }
        }
      }
      if (GID > 0) {
        xc[kXDesc][GID - 1][lane] = run;
      } else {
        total = run;
      }
    }
    if (s < NW - 1) {
      ctaBarrier();
      if (s == 0) {
        afterFirstBarrier();
      }
    }
  }
  return total;
}

// ---- one backward step: x = beta(p+1) on entry (becomes vec = beta * emission), y = unscaled beta(p) ----------------
// ref: HMM.cpp:957-1016.  Warps below the middle run the BL scan first, warps above it the BU scan.
template <int S, int NW, int GID, class F>
__device__ __forceinline__ void backwardSplit(float (&x)[SplitGeom<S, NW>::SEG], float (&y)[SplitGeom<S, NW>::SEG],
                                              const float* row, const int cls, float (*xc)[NW][32], const int lane,
                                              F&& afterFirstBarrier)
{
  using G = SplitGeom<S, NW>;
  constexpr int SEGQ = G::SEGQ, SEG = G::SEG, Spad = G::Spad, K0 = GID * SEG, Q0 = GID * SEGQ;
  constexpr bool LOWER = GID < NW / 2;
  const float4* E = reinterpret_cast<const float4*>(row + cls * Spad) + Q0;
  const float4* Dr = reinterpret_cast<const float4*>(row + 3 * Spad) + Q0;
  const float4* Br = reinterpret_cast<const float4*>(row + 4 * Spad) + Q0;
  const float4* Us = reinterpret_cast<const float4*>(row + 7 * Spad) + Q0;  // U shifted by one state
  const float4* Rr = reinterpret_cast<const float4*>(row + 6 * Spad) + Q0;
#pragma unroll
  for (int s = 0; s < NW; ++s) {
    if (s == GID) {
      float bl = GID == 0 ? 0.f : xc[kXAsc][GID - 1][lane];
#pragma unroll
      for (int q = 0; q < SEGQ; ++q) {
        const float4 d4 = Dr[q], b4 = Br[q];
        float4 e4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (LOWER) {
          e4 = E[q];
        }
#pragma unroll
        for (int jp = 0; jp < 2; ++jp) {
          const int i = 4 * q + 2 * jp, k = K0 + i;
          if (k + 1 < S) {
            float2 v = pk(x[i], x[i + 1]);
            if (LOWER) {
              v = __fmul2_rn(v, pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)));  // vec = beta(p+1) * emission(p+1)
              x[i] = v.x;
              x[i + 1] = v.y;
            }
            const float bl0 = bl;
            const float bl1 = fmaf(f4(b4, 2 * jp), v.x, bl0);  // BL[k+1] = BL[k] + B[k] vec[k]
            bl = fmaf(f4(b4, 2 * jp + 1), v.y, bl1);
            float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), v, pk(bl0, bl1));  // BL[k] + D[k] vec[k]
            if (!LOWER) {
              w = __fadd2_rn(w, pk(y[i], y[i + 1]));
            }
            y[i] = w.x;
            y[i + 1] = w.y;
          } else if (k < S) {
            if (LOWER) {
              x[i] *= f4(e4, 2 * jp);
              y[i] = fmaf(f4(d4, 2 * jp), x[i], bl);
            } else {
              y[i] = fmaf(f4(d4, 2 * jp), x[i], bl) + y[i];
            }
            bl = fmaf(f4(b4, 2 * jp), x[i], bl);
          }
        }
      }
      if (GID < NW - 1) {
        xc[kXAsc][GID][lane] = bl;
      }
    }
    if (s == NW - 1 - GID) {
      float bu = GID == NW - 1 ? 0.f : xc[kXDesc][GID][lane];
      // U[k] vec[k+1] for the state k the BU chain reaches next; across the warp boundary: vec of the next warp's first state
      float above = 0.f;
      if (GID < NW - 1) {
        above = Us[SEGQ].x * xc[kXVec][GID][lane];  // Us[k] = U[k-1]
      }
#pragma unroll
      for (int q = SEGQ - 1; q >= 0; --q) {
        const float4 u4 = Us[q], r4 = Rr[q];
        float4 e4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (!LOWER) {
          e4 = E[q];
        }
#pragma unroll
        for (int jp = 1; jp >= 0; --jp) {
          const int i = 4 * q + 2 * jp, k = K0 + i;
          if (k + 1 < S) {
            float2 v = pk(x[i], x[i + 1]);
            if (!LOWER) {
              v = __fmul2_rn(v, pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)));
              x[i] = v.x;
              x[i + 1] = v.y;
            }
            const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), v);  // U[k-1] vec[k]
            float b1 = 0.f;  // BU[S-1] = 0
            if (k + 1 < S - 1) {
              b1 = fmaf(f4(r4, 2 * jp + 1), bu, above);  // BU[k] = U[k] vec[k+1] + RR[k] BU[k+1]
            }
            const float b0 = fmaf(f4(r4, 2 * jp), b1, t.y);
            bu = b0;
            above = t.x;
            if (LOWER) {
              const float2 w = __fadd2_rn(pk(y[i], y[i + 1]), pk(b0, b1));
              y[i] = w.x;
              y[i + 1] = w.y;
            } else {
              y[i] = b0;
              y[i + 1] = b1;
            }
          } else {
            if (k < S) {
              if (!LOWER) {
                x[i] *= f4(e4, 2 * jp);
              }
              above = f4(u4, 2 * jp) * x[i];
              float b0 = 0.f;
              if (k < S - 1) {
                b0 = fmaf(f4(r4, 2 * jp), bu, above);
              }
              bu = b0;
              if (LOWER) {
                y[i] += b0;
              } else {
                y[i] = b0;
              }
            } else {
              x[i] = 0.f;
              y[i] = 0.f;
            }
            x[i + 1] = 0.f;
            y[i + 1] = 0.f;
          }
        }
      }
      if (GID > 0) {
        xc[kXDesc][GID - 1][lane] = bu;
        xc[kXVec][GID - 1][lane] = x[0];
      }
    }
    if (s < NW - 1) {
      ctaBarrier();
      if (s == 0) {
        afterFirstBarrier();
      }
    }
  }
}

template <int S, int NW, int GID> __device__ __forceinline__ float sumSegment(const float (&a)[SplitGeom<S, NW>::SEG])
{
  constexpr int SEG = SplitGeom<S, NW>::SEG, K0 = GID * SEG;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
  for (int i = 0; i < SEG; i += 4) {
    if (K0 + i < S) s0 += a[i];
    if (K0 + i + 1 < S) s1 += a[i + 1];
    if (K0 + i + 2 < S) s2 += a[i + 2];
    if (K0 + i + 3 < S) s3 += a[i + 3];
  }
  return (s0 + s1) + (s2 + s3);
}

template <int NW> __device__ __forceinline__ float sumParts(const float (*part)[32], const int lane)
{
  float t = part[0][lane];
#pragma unroll
  for (int g = 1; g < NW; ++g) {
    t += part[g][lane];
  }
  return t;
}

// Shared-memory carve-up of one CTA (bytes); used by the kernel and by the host for the launch configuration.
template <int S_T, int NW, int RQ, int GRP, int DEPTH> struct SplitSmem {
  using G = SplitGeom<S_T, NW>;
  static constexpr size_t kCoefBytes = static_cast<size_t>(kRowArrays) * G::Spad * 4;
  static constexpr size_t kBetaBytes = static_cast<size_t>(G::SQ) * 32 * 16;  // wide: one site of beta, all warps
  static constexpr size_t kRecBytes = static_cast<size_t>(RQ) * 32 * 16;      // narrow: one record
  static constexpr size_t kSlotBytes = RQ == 0 ? kCoefBytes + kBetaBytes : GRP * kCoefBytes + (GRP + 1) * kRecBytes;
  static constexpr size_t kRing = DEPTH * kSlotBytes;
  static constexpr size_t kXchOff = (kRing + 127) / 128 * 128;
  static constexpr size_t kBarOff = kXchOff + sizeof(SplitXch<NW>);
  static constexpr size_t kNumBars = DEPTH * (1 + NW);  // coefficient slot full; per-warp beta part full
  static constexpr size_t kTileOff = kBarOff + kNumBars * sizeof(uint64_t);
  static constexpr size_t kTotal = kTileOff + 16;
};

// -------------------------------------------------------------------------------------------------------------------
// The per-warp body.  GID (the warp's segment) is a compile-time constant, so that every state index, padding test and
// colRatio operand is static; the kernel switches on the warp index once.
// -------------------------------------------------------------------------------------------------------------------
template <int S_T, int NW, int RQ, bool ACC, int GRP, int DEPTH, int GID>
__device__ __forceinline__ void splitBody(const FastModel& fm, const DecodeArgs& args, unsigned char* smemRaw)
{
  using G = SplitGeom<S_T, NW>;
  using SM = SplitSmem<S_T, NW, RQ, GRP, DEPTH>;
  constexpr int S = S_T, SEG = G::SEG, SEGQ = G::SEGQ, Spad = G::Spad, K0 = GID * SEG, Q0 = GID * SEGQ;
  constexpr bool NARROW = RQ > 0;
  constexpr int NR = NARROW ? 4 * RQ - 1 : 0;
  constexpr size_t kRowFloats = static_cast<size_t>(kRowArrays) * Spad;
  constexpr uint32_t kCoefBytes = static_cast<uint32_t>(SM::kCoefBytes);
  constexpr uint32_t kRecBytes = static_cast<uint32_t>(SM::kRecBytes);
  constexpr size_t kRecFloats = static_cast<size_t>(RQ) * 32 * 4;
  constexpr uint32_t kPartBytes = SEGQ * 32 * 16;  // wide: this warp's part of a beta row
  constexpr size_t kBetaFloats = static_cast<size_t>(G::SQ) * 32 * 4;
  static_assert(!NARROW || (GRP % 2 == 0 && NR <= SEG), "narrow: even groups; the record states live in warp 0");
  static_assert(NARROW || GRP == 1, "wide: one window position per ring slot");

  const DeviceModel m = fm.base;
  const int lane = threadIdx.x & 31;
  SplitXch<NW>* xch = reinterpret_cast<SplitXch<NW>*>(smemRaw + SM::kXchOff);
  uint64_t* coefBar = reinterpret_cast<uint64_t*>(smemRaw + SM::kBarOff);
  uint64_t* betaBar = coefBar + DEPTH + GID * DEPTH;
  volatile long long* tileSlot = reinterpret_cast<volatile long long*>(smemRaw + SM::kTileOff);
  auto coefArea = [&](const int slot) { return reinterpret_cast<float*>(smemRaw + static_cast<size_t>(slot) * SM::kSlotBytes); };
  // wide: beta row of the slot (all warps, [quad][lane][4]); narrow: the slot's records
  auto dataArea = [&](const int slot) {
    return reinterpret_cast<float4*>(smemRaw + static_cast<size_t>(slot) * SM::kSlotBytes + static_cast<size_t>(GRP) * kCoefBytes);
  };
  const bool leader = GID == 0 && lane == 0;
  if (leader) {
    for (int i = 0; i < static_cast<int>(SM::kNumBars); ++i) {
      mbarInit(&coefBar[i], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  ctaBarrier();
  uint32_t coefParity = 0, betaParity = 0;  // bit i = parity the next wait on slot i expects
  int xp = 0;                               // exchange-area parity, flips every step

  const unsigned flags = args.flags;
  const bool wantSeg = flags & FSMC_CALL_SEGMENTS;
  const bool wantAge = (NARROW || ACC) && (flags & FSMC_SEG_AGE) && wantSeg;
  const bool wantSite = !NARROW && (flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP));
  const int sT = m.stateThreshold;
  const int nAcc = m.ageThreshold;
  float* slab = args.scratch + static_cast<long long>(blockIdx.x) * args.scratchPerWarp;

  for (long long it = 0;; ++it) {
    if (leader) {
      tileSlot[it & 1] = static_cast<long long>(atomicAdd(args.tileCounter, 1ull));
    }
    ctaBarrier();
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
    const bool laneActive = lane < nPairs;
    const int srcLane = laneActive ? lane : nPairs - 1;
    const uint32_t pair = static_cast<uint32_t>(tile) * 32u + static_cast<uint32_t>(lane);
    // output row (fsmc_decode_device); the narrow kernels write pair-numbered rows only
    const uint32_t outRow = (!NARROW && args.laneRow) ? __ldg(args.laneRow + pair) : pair;
    PairBits bits;
    bits.a = m.haps + static_cast<size_t>(args.hapA[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    bits.b = m.haps + static_cast<size_t>(args.hapB[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    const float* rowBase = m.siteRows + static_cast<size_t>(from) * kRowFloats;

    float a[SEG], c[SEG];
    constexpr int NACC = NARROW ? (GID == 0 ? NR : 1) : (ACC ? SEG : 1);
    float acc[NACC];
#pragma unroll
    for (int k = 0; k < NACC; ++k) {
      acc[k] = 0.f;
    }

    if constexpr (NARROW) {
      // =============================================================================================================
      // narrow, sweep 1: backward.  Step j handles window position len-2-j with the coefficient row of len-1-j; ring
      // slots hold GRP consecutive positions (one bulk copy and one mbarrier wait per group).
      // =============================================================================================================
      auto stageRecord = [&](const float (&v)[SEG], float4* out, const float divisor) {
#pragma unroll
        for (int q = 0; q < RQ; ++q) {
          float w[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int k = 4 * q + i;
            w[i] = k == NR ? divisor : (k < sT ? v[k < SEG ? k : 0] : 0.f);
          }
          out[q * 32 + lane] = make_float4(w[0], w[1], w[2], w[3]);
        }
      };
      {
        const int steps = len - 1;
        const int nGroups = (steps + GRP - 1) / GRP;
        auto prefetch = [&](const int g) {  // rows of steps [g GRP, g GRP + n): window positions [len-j1, len-j0)
          const int j0 = g * GRP, j1 = min(steps, j0 + GRP);
          const int slot = g % DEPTH;
          const uint32_t bytes = static_cast<uint32_t>(j1 - j0) * kCoefBytes;
          mbarExpectTx(&coefBar[slot], bytes);
          bulkLoad(coefArea(slot), rowBase + static_cast<size_t>(len - j1) * kRowFloats, bytes, &coefBar[slot]);
        };
        if (leader) {
          for (int g = 0; g < DEPTH && g < nGroups; ++g) {
            prefetch(g);
          }
        }
#pragma unroll
        for (int i = 0; i < SEG; ++i) {
          a[i] = K0 + i < S ? 1.f : 0.f;
        }
        if (nGroups == 0 && GID == 0) {
          stageRecord(a, dataArea(0), 1.0f);  // single-site window: only the all-ones record
          fenceProxyAsync();
          __syncwarp();
          if (lane == 0) {
            bulkStore(slab, dataArea(0), kRecBytes);
            bulkCommit();
          }
        }
        for (int g = 0; g < nGroups; ++g) {
          const int slot = g % DEPTH;
          const int j0 = g * GRP;
          const int n = min(GRP, steps - j0);
          const float* coef = coefArea(slot);
          float4* stage = dataArea(slot);
          if (leader) {
            bulkWaitRead<DEPTH - 1>();  // the store that last read this slot's staging records has drained them
          }
          mbarWait(&coefBar[slot], (coefParity >> slot) & 1u);
          coefParity ^= 1u << slot;
          if (GID == 0) {
            __syncwarp();
            if (g == 0) {
              stageRecord(a, stage + static_cast<size_t>(n) * RQ * 32, 1.0f);  // position len-1
            }
          }
          auto step = [&](const int i, float (&x)[SEG], float (&y)[SEG]) {
            const int p = len - 2 - (j0 + i);
            const int cls = bits.cls(from + p + 1);
            backwardSplit<S, NW, GID>(x, y, coef + static_cast<size_t>(n - 1 - i) * kRowFloats, cls, xch->v[xp], lane, [&] {
              // every warp has left the previous group: its coefficient slot can be refilled
              if (leader && i == 0 && g > 0 && g - 1 + DEPTH < nGroups) {
                prefetch(g - 1 + DEPTH);
              }
            });
            float divisor = 1.0f;
            if (n == GRP && i == GRP - 1) {
              divisor = sumParts<NW>(xch->v[xp ^ 1][kXPart], lane);  // sum of the previous step's beta
              const float sc = 1.0f / divisor;
#pragma unroll
              for (int k = 0; k < SEG; ++k) {
                y[k] *= sc;
              }
            }
            if (n == GRP && i == GRP - 2) {
              xch->v[xp][kXPart][GID][lane] = sumSegment<S, NW, GID>(y);
            }
            if (GID == 0) {
              stageRecord(y, stage + static_cast<size_t>(n - 1 - i) * RQ * 32, divisor);
            }
            xp ^= 1;
          };
          // (not unrolled: one copy of the step pair per sweep keeps the four warps' bodies in the instruction cache)
#pragma unroll 1
          for (int i = 0; i < GRP; i += 2) {
            if (i < n) {
              step(i, a, c);
            }
            if (i + 1 < n) {
              step(i + 1, c, a);
            }
          }
          if (GID == 0) {
            fenceProxyAsync();
            __syncwarp();
            if (lane == 0) {
              const int j1 = j0 + n;
              bulkStore(slab + static_cast<size_t>(len - 1 - j1) * kRecFloats, stage,
                        static_cast<uint32_t>(n + (g == 0 ? 1 : 0)) * kRecBytes);
              bulkCommit();
            }
          }
        }
        if (!(steps & 1)) {  // beta^ of the first site ended in a; the forward sweep wants it in c
#pragma unroll
          for (int k = 0; k < SEG; ++k) {
            c[k] = a[k];
          }
        }
        if (leader) {
          bulkWaitAll<0>();
        }
        ctaBarrier();  // records are in HBM and every warp is done with the ring
      }

      // =============================================================================================================
      // narrow, sweep 2: forward + consumers (warp 0 holds the states below the threshold)
      // =============================================================================================================
      {
        const int nGroups = (len + GRP - 1) / GRP;
        auto prefetch = [&](const int g) {
          const int p0 = g * GRP;
          const uint32_t n = static_cast<uint32_t>(min(GRP, len - p0));
          const int slot = g % DEPTH;
          mbarExpectTx(&coefBar[slot], n * (kCoefBytes + kRecBytes));
          bulkLoad(coefArea(slot), rowBase + static_cast<size_t>(p0) * kRowFloats, n * kCoefBytes, &coefBar[slot]);
          bulkLoad(dataArea(slot), slab + static_cast<size_t>(p0) * kRecFloats, n * kRecBytes, &coefBar[slot]);
        };
        if (leader) {
          for (int g = 0; g < DEPTH && g < nGroups; ++g) {
            prefetch(g);
          }
        }
        CallerState cs;
        float Z = 1.f, bPrev = 1.f;

        // consumers of window position p (warp 0 only); v = alpha^(p); rec = this position's record
        auto consume = [&](const int p, const float (&v)[SEG], float4* rec) {
          const int site = from + p;
          float q[4 * RQ];  // alpha^[k] beta^[k] for k < sT (0 above); q[NR] = b_p
#pragma unroll
          for (int qq = 0; qq < RQ; ++qq) {
            const float4 r4 = rec[qq * 32 + lane];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              q[4 * qq + i] = f4(r4, i);
            }
          }
          bPrev = q[NR];
          float ibdRaw = 0.f;
#pragma unroll
          for (int k = 0; k < NR; ++k) {
            q[k] *= v[k < SEG ? k : 0];
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
            if (__any_sync(kFull, ending || closing)) {
              float* park = reinterpret_cast<float*>(rec) + lane;  // drained record: [k][32], k < NR
              __syncwarp();
              if (wantAge) {
#pragma unroll
                for (int k = 0; k < NR; ++k) {
                  park[k * 32] = acc[k < NACC ? k : 0];
                }
                __syncwarp();
              }
              if (ending) {
                emitSegment<false>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, park, wantAge);
              }
              __syncwarp();
              if (wantAge) {
#pragma unroll
                for (int k = 0; k < NR; ++k) {
                  acc[k < NACC ? k : 0] = fmaf(q[k], rr, keep * acc[k < NACC ? k : 0]);
                  park[k * 32] = acc[k < NACC ? k : 0];
                }
                __syncwarp();
              }
              if (closing) {
                emitSegment<false>(m, args, pair, changed ? site : cs.start, site, changed ? ibd : cs.prob + ibd, now, park, wantAge);
              }
              __syncwarp();
            } else if (wantAge) {
#pragma unroll
              for (int k = 0; k < NR; ++k) {
                acc[k < NACC ? k : 0] = fmaf(q[k], rr, keep * acc[k < NACC ? k : 0]);
              }
            }
            cs.prob = (now >= 0 && !closing) ? (changed ? ibd : cs.prob + ibd) : 0.f;
            cs.start = (now >= 0 && changed) ? site : cs.start;
            cs.level = now;
          }
        };

        for (int g = 0; g < nGroups; ++g) {
          const int slot = g % DEPTH;
          const int p0 = g * GRP;
          const int n = min(GRP, len - p0);
          const float* coef = coefArea(slot);
          float4* recs = dataArea(slot);
          mbarWait(&coefBar[slot], (coefParity >> slot) & 1u);
          coefParity ^= 1u << slot;
          auto step = [&](const int i, float (&x)[SEG], float (&y)[SEG]) {
            const int p = p0 + i;
            const int cls = bits.cls(from + p);
            const float total = forwardSplit<S, NW, GID>(fm.colRatios, x, y, coef + static_cast<size_t>(i) * kRowFloats, cls,
                                                         xch->v[xp], lane, [&] {
                                                           if (leader && i == 0 && g > 0 && g - 1 + DEPTH < nGroups) {
                                                             prefetch(g - 1 + DEPTH);
                                                           }
                                                         });
            const bool scaled = n == GRP && (GRP > 2 || g > 0);
            float sc = 1.0f;
            if (scaled && i == GRP - 1) {
              sc = 1.0f / xch->v[xp ^ 1][kXPart][0][lane];  // sum of alpha two sites back (published by warp 0)
#pragma unroll
              for (int k = 0; k < SEG; ++k) {
                y[k] *= sc;
              }
            }
            if (GID == 0) {
              if (scaled && i == GRP - 2) {
                xch->v[xp][kXPart][0][lane] = total;
              }
              Z *= bPrev * sc;  // Z_p = Z_{p-1} * b_{p-1} / a_p
              consume(p, y, recs + static_cast<size_t>(i) * RQ * 32);
            }
            xp ^= 1;
          };
          if (g == 0) {
            // p = 0: alpha^(0) = prior * emission into a; the one exact normaliser Z_0 = sum_k alpha^(0)[k] beta^(0)[k]
            const int cls = bits.cls(from);
            const float4* E = reinterpret_cast<const float4*>(coef + cls * Spad) + Q0;
            float z0 = 0.f, z1 = 0.f, z2 = 0.f, z3 = 0.f;
#pragma unroll
            for (int q = 0; q < SEGQ; ++q) {
              const float4 e4 = E[q];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int k = K0 + 4 * q + i;
                a[4 * q + i] = k < S ? fm.prior[k < S ? k : 0] * f4(e4, i) : 0.f;
              }
              z0 = fmaf(a[4 * q], c[4 * q], z0);
              z1 = fmaf(a[4 * q + 1], c[4 * q + 1], z1);
              z2 = fmaf(a[4 * q + 2], c[4 * q + 2], z2);
              z3 = fmaf(a[4 * q + 3], c[4 * q + 3], z3);
            }
            xch->v[xp][kXPart][GID][lane] = (z0 + z1) + (z2 + z3);
            ctaBarrier();
            if (GID == 0) {
              Z = sumParts<NW>(xch->v[xp][kXPart], lane);
              consume(0, a, recs);
            }
            xp ^= 1;
          } else {
            step(0, c, a);
          }
#pragma unroll 1
          for (int i = 1; i < GRP; i += 2) {
            if (i < n) {
              step(i, a, c);
            }
            if (i + 1 < GRP && i + 1 < n) {
              step(i + 1, c, a);
            }
          }
        }
        ctaBarrier();  // every warp is done with the ring before the next tile refills it
      }
    } else {
      // =============================================================================================================
      // wide, sweep 1: backward.  Every warp streams its own part of each beta row to the tile's slab.
      // =============================================================================================================
      float4* myPartOf = nullptr;
      (void)myPartOf;
      auto betaPart = [&](const int slot) { return dataArea(slot) + static_cast<size_t>(Q0) * 32; };
      auto storeRow = [&](const float (&v)[SEG], const int p, const int bslot) {
        if (lane == 0) {
          bulkWaitRead<DEPTH - 1>();  // the copy that last read this staging slot has drained it
        }
        __syncwarp();
        float4* out = betaPart(bslot);
#pragma unroll
        for (int q = 0; q < SEGQ; ++q) {
          out[q * 32 + lane] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        }
        fenceProxyAsync();
        __syncwarp();
        if (lane == 0) {
          bulkStore(slab + static_cast<size_t>(p) * kBetaFloats + static_cast<size_t>(Q0) * 128, out, kPartBytes);
          bulkCommit();
        }
      };
      {
        const int steps = len - 1;
        auto prefetchCoef = [&](const int j) {  // row of window position len-1-j into slot j % DEPTH
          uint64_t* bar = &coefBar[j % DEPTH];
          mbarExpectTx(bar, kCoefBytes);
          bulkLoad(coefArea(j % DEPTH), rowBase + static_cast<size_t>(len - 1 - j) * kRowFloats, kCoefBytes, bar);
        };
        if (leader) {
          for (int j = 0; j < DEPTH && j < steps; ++j) {
            prefetchCoef(j);
          }
        }
#pragma unroll
        for (int i = 0; i < SEG; ++i) {
          a[i] = K0 + i < S ? 1.f : 0.f;  // beta at the last site: all ones (any positive scale is equivalent)
        }
        storeRow(a, len - 1, 0);
        auto step = [&](const int j, float (&x)[SEG], float (&y)[SEG]) {
          const int p = len - 2 - j;
          const int slot = j % DEPTH;
          const int cls = bits.cls(from + p + 1);
          mbarWait(&coefBar[slot], (coefParity >> slot) & 1u);
          coefParity ^= 1u << slot;
          backwardSplit<S, NW, GID>(x, y, coefArea(slot), cls, xch->v[xp], lane, [&] {
            if (leader && j > 0 && j - 1 + DEPTH < steps) {
              prefetchCoef(j - 1 + DEPTH);  // every warp has left step j-1
            }
          });
          if ((p & 3) == 0 && j > 0) {
            const float sc = 1.0f / sumParts<NW>(xch->v[xp ^ 1][kXPart], lane);  // sum of beta(p+1), before its own scaling
#pragma unroll
            for (int k = 0; k < SEG; ++k) {
              y[k] *= sc;
            }
          }
          if ((p & 3) == 1) {
            xch->v[xp][kXPart][GID][lane] = sumSegment<S, NW, GID>(y);
          }
          storeRow(y, p, (j + 1) % DEPTH);
          xp ^= 1;
        };
        int j = 0;
        for (; j + 1 < steps; j += 2) {
          step(j, a, c);
          step(j + 1, c, a);
        }
        if (j < steps) {
          step(j, a, c);
        }
        if (lane == 0) {
          bulkWaitAll<0>();  // this warp's beta parts are in global memory
        }
        ctaBarrier();  // ... and so are everybody else's; the coefficient ring is idle
      }

      // =============================================================================================================
      // wide, sweep 2: forward + fused consumers (ref: HMM.cpp:725-879, 669-692, 1179-1357, 1378-1409)
      // =============================================================================================================
      {
        auto prefetchCoef = [&](const int p) {
          uint64_t* bar = &coefBar[p % DEPTH];
          mbarExpectTx(bar, kCoefBytes);
          bulkLoad(coefArea(p % DEPTH), rowBase + static_cast<size_t>(p) * kRowFloats, kCoefBytes, bar);
        };
        auto prefetchBeta = [&](const int p) {
          if (lane == 0) {
            const int slot = p % DEPTH;
            mbarExpectTx(&betaBar[slot], kPartBytes);
            bulkLoad(betaPart(slot), slab + static_cast<size_t>(p) * kBetaFloats + static_cast<size_t>(Q0) * 128, kPartBytes,
                     &betaBar[slot]);
          }
        };
        for (int p = 0; p < DEPTH && p < len; ++p) {
          if (leader) {
            prefetchCoef(p);
          }
          prefetchBeta(p);
        }
        CallerState cs;

        // consumers of window position p: v = alpha(p) (this warp's states); w = the dead vector, receives alpha*beta
        auto consume = [&](const int p, const float (&v)[SEG], float (&w)[SEG]) {
          const int site = from + p;
          const int slot = p % DEPTH;
          mbarWait(&betaBar[slot], (betaParity >> slot) & 1u);
          betaParity ^= 1u << slot;
          const float4* B4 = betaPart(slot);
          float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f;
#pragma unroll
          for (int q = 0; q < SEGQ; ++q) {
            const float4 b4 = B4[q * 32 + lane];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              w[4 * q + i] = v[4 * q + i] * f4(b4, i);  // padding states: alpha is 0
            }
            q0 += w[4 * q];
            q1 += w[4 * q + 1];
            q2 += w[4 * q + 2];
            q3 += w[4 * q + 3];
          }
          float (*xc)[NW][32] = xch->v[xp];
          xc[kXPart][GID][lane] = (q0 + q1) + (q2 + q3);
          const bool inScan = wantSeg && site >= scanFrom && site < scanTo;
          const bool wantIbd = (flags & FSMC_SITE_IBD) || inScan;
          if (GID == 0 && wantIbd) {
            float ibdRaw = 0.f;
            forStatesBelow<SEG>(sT, [&](const int k) { ibdRaw += w[k]; });
            xc[kXIbd][0][lane] = ibdRaw;
          }
          if (wantSite) {
            float mean = 0.f, best = 0.f;
            int arg = K0;
#pragma unroll
            for (int k = 0; k < SEG; ++k) {
              if (K0 + k < S) {
                mean = fmaf(w[k], fm.expTimes[K0 + k < S ? K0 + k : 0], mean);
                if (best < w[k]) {
                  best = w[k];
                  arg = K0 + k;
                }
              }
            }
            xc[kXMean][GID][lane] = mean;
            xc[kXBest][GID][lane] = best;
            xc[kXArg][GID][lane] = __int_as_float(arg);
          }
          ctaBarrier();
          const float r = 1.0f / sumParts<NW>(xc[kXPart], lane);  // ref HMM.cpp:681-685
          if (wantSite && GID == 0 && laneActive) {
            if (flags & FSMC_SITE_MEAN) {
              args.siteMean[static_cast<size_t>(outRow) * args.siteStride + p] = sumParts<NW>(xc[kXMean], lane) * r;
            }
            if (flags & FSMC_SITE_MAP) {
              float best = 0.f;
              int arg = 0;
#pragma unroll
              for (int g = 0; g < NW; ++g) {
                const float b = xc[kXBest][g][lane];
                if (best < b) {  // first maximum, as the reference's ascending scan
                  best = b;
                  arg = __float_as_int(xc[kXArg][g][lane]);
                }
              }
              args.siteMap[static_cast<size_t>(outRow) * args.siteStride + p] = arg;
            }
          }
          if (wantIbd) {
            const float ibd = xc[kXIbd][0][lane] * r;
            if ((flags & FSMC_SITE_IBD) && GID == 0 && laneActive) {
              args.siteIbd[static_cast<size_t>(outRow) * args.siteStride + p] = ibd;
            }
            if (inScan) {
              // every warp runs the same run-length state machine on the same numbers; warp 0 emits
              int now = ibd >= m.thr[0] ? 0 : (ibd >= m.thr[1] ? 1 : (ibd >= m.thr[2] ? 2 : (ibd >= m.thr[3] ? 3 : -1)));
              if (!laneActive) {
                now = -1;
              }
              const bool changed = now != cs.level;
              const bool ending = changed && cs.level >= 0;  // the run that ended at site-1 is written now
              const bool closing = now >= 0 && site == scanTo - 1;
              float* park = reinterpret_cast<float*>(dataArea(slot)) + lane;  // this site's drained beta row: [k][32]
              auto parkAcc = [&] {
                __syncwarp();  // this warp has read its part of the beta row
                if constexpr (ACC) {
#pragma unroll
                  for (int k = 0; k < SEG; ++k) {
                    park[(K0 + k) * 32] = acc[k];
                  }
                }
                ctaBarrier();
              };
              if (__any_sync(kFull, ending)) {
                if (wantAge) {
                  parkAcc();
                }
                if (GID == 0 && ending) {
                  emitSegment<false>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, park, wantAge);
                }
                if (wantAge) {
                  ctaBarrier();
                }
              }
              if constexpr (ACC) {
                if (wantAge && __any_sync(kFull, now >= 0)) {
                  // per-state sums of the current run (ref: HMM.cpp:1209-1218,1229,1257,1284,1311)
                  const float rr = now >= 0 ? r : 0.f;
                  const float keep = changed ? 0.f : 1.f;
                  forStatesBelow<SEG>(nAcc - K0, [&](const int k) { acc[k] = fmaf(w[k], rr, keep * acc[k]); });
                }
              }
              if (__any_sync(kFull, closing)) {
                if (wantAge) {
                  parkAcc();
                }
                if (GID == 0 && closing) {
                  emitSegment<false>(m, args, pair, changed ? site : cs.start, site, changed ? ibd : cs.prob + ibd, now, park,
                                     wantAge);
                }
                if (wantAge) {
                  ctaBarrier();
                }
              }
              cs.prob = (now >= 0 && !closing) ? (changed ? ibd : cs.prob + ibd) : 0.f;
              cs.start = (now >= 0 && changed) ? site : cs.start;
              cs.level = now;
            }
          }
          __syncwarp();  // this warp's part of the beta slot is drained
          if (p + DEPTH < len) {
            prefetchBeta(p + DEPTH);
          }
          xp ^= 1;
        };

        // p = 0: alpha(from)[k] = prior[k] * emission  (ref HMM.cpp:736-743)
        {
          const int cls = bits.cls(from);
          mbarWait(&coefBar[0], coefParity & 1u);
          coefParity ^= 1u;
          const float4* E = reinterpret_cast<const float4*>(coefArea(0) + cls * Spad) + Q0;
#pragma unroll
          for (int q = 0; q < SEGQ; ++q) {
            const float4 e4 = E[q];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int k = K0 + 4 * q + i;
              a[4 * q + i] = k < S ? fm.prior[k < S ? k : 0] * f4(e4, i) : 0.f;
            }
          }
          consume(0, a, c);  // its barrier also tells the leader that slot 0's coefficients are drained
          if (leader && DEPTH < len) {
            prefetchCoef(DEPTH);
          }
        }
        auto step = [&](const int p, float (&x)[SEG], float (&y)[SEG]) {
          const int slot = p % DEPTH;
          const int cls = bits.cls(from + p);
          mbarWait(&coefBar[slot], (coefParity >> slot) & 1u);
          coefParity ^= 1u << slot;
          const float total = forwardSplit<S, NW, GID>(fm.colRatios, x, y, coefArea(slot), cls, xch->v[xp], lane, [&] {
            if (leader && p > 1 && p - 1 + DEPTH < len) {
              prefetchCoef(p - 1 + DEPTH);  // every warp has left step p-1
            }
          });
          if ((p & 3) == 0) {
            const float sc = 1.0f / xch->v[xp ^ 1][kXDesc][NW - 1][lane];  // sum of alpha(p-2), published by warp 0
#pragma unroll
            for (int k = 0; k < SEG; ++k) {
              y[k] *= sc;
            }
          }
          if (GID == 0 && (p & 3) == 3) {
            xch->v[xp][kXDesc][NW - 1][lane] = total;  // (slot NW-1 of the descending carries is otherwise unused)
          }
          consume(p, y, x);
        };
        int p = 1;
        for (; p + 1 < len; p += 2) {
          step(p, a, c);
          step(p + 1, c, a);
        }
        if (p < len) {
          step(p, a, c);
        }
        ctaBarrier();  // every warp is done with the rings before the next tile refills them
      }
    }
  }
}

template <int S_T, int NW, int RQ, bool ACC, int GRP, int DEPTH, int MIN_BLOCKS>
__global__ void __launch_bounds__(NW * 32, MIN_BLOCKS) decodeSplitKernel(const FastModel fm, const DecodeArgs args)
{
  extern __shared__ __align__(128) unsigned char smemRaw[];
  const int warp = threadIdx.x >> 5;
  if constexpr (NW == 2) {
    if (warp == 0) {
      splitBody<S_T, NW, RQ, ACC, GRP, DEPTH, 0>(fm, args, smemRaw);
    } else {
      splitBody<S_T, NW, RQ, ACC, GRP, DEPTH, 1>(fm, args, smemRaw);
    }
  } else {
    static_assert(NW == 4, "two or four warps per tile");
    switch (warp) {
    case 0:
      splitBody<S_T, NW, RQ, ACC, GRP, DEPTH, 0>(fm, args, smemRaw);
      break;
    case 1:
      splitBody<S_T, NW, RQ, ACC, GRP, DEPTH, 1>(fm, args, smemRaw);
      break;
    case 2:
      splitBody<S_T, NW, RQ, ACC, GRP, DEPTH, 2>(fm, args, smemRaw);
      break;
    default:
      splitBody<S_T, NW, RQ, ACC, GRP, DEPTH, 3>(fm, args, smemRaw);
      break;
    }
  }
}

}  // namespace fsmc
