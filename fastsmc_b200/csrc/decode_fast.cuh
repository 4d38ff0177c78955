// fastsmc_b200 — the production decode kernel for sm_100a (FMA arithmetic; results within 1e-4 of the reference).
//
// Same two sweeps per 32-pair tile as decode_kernels.cuh (backward sweep streams beta to a per-warp HBM slab, forward
// sweep keeps alpha on chip and consumes the posterior at once), rebuilt around the three things the first kernel
// stalled on (profiles/r1_v1_*: 24 % issue-slot utilisation, 3.3 warps stalled on the long scoreboard per issue):
//
//  1. every HBM access of the sweeps is a bulk asynchronous copy (cp.async.bulk, the non-tensor TMA path) through a
//     per-warp shared-memory ring completed on mbarriers: one elected lane issues one 9 KB copy per site instead of
//     69 scalar loads/stores per lane, and the copy for site p+DEPTH is in flight while site p is computed.  beta rows
//     are laid out [state/4][lane][4] so that a lane moves four states per 128-bit shared-memory access;
//  2. the per-site coefficient row (three emission classes, D, B, U, RR: 2 KB) is prefetched into the same ring, so
//     the recurrences read their coefficients with warp-broadcast LDS.128 instead of waiting on L2;
//  3. the per-site rescaling to sum 1 (ref: HmmUtils.cpp:102-151, two instructions per state per sweep) is done every
//     fourth site only: the posterior alpha*beta/sum(alpha*beta) is invariant to the scale of alpha and of beta, so
//     scaling exists only to keep fp32 in range.  The forward sweep gets its normaliser for free from the suffix sums.
//     The combine step is a dot product (one FMA per state); per-state posteriors are formed only for lanes inside an
//     IBD segment or when per-site summaries are requested.
//
// State vectors stay in registers (fully unrolled linear-time recurrences, ref: HMM.cpp:787-879, 943-1041); the small
// site-independent vectors (columnRatios, expectedTimes) are kernel parameters, i.e. constant-bank operands.
#pragma once

#include "decode_kernels.cuh"

namespace fsmc
{

constexpr int kMaxParamStates = 160;

struct FastModel {
  DeviceModel base;
  float colRatios[kMaxParamStates];
  float expTimes[kMaxParamStates];
  float prior[kMaxParamStates];
};

// ---- bulk async copy / mbarrier primitives (PTX ISA: cp.async.bulk, mbarrier) -----------------------------------
__device__ __forceinline__ uint32_t smemPtr(const void* p)
{
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbarInit(uint64_t* bar, const uint32_t count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smemPtr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbarExpectTx(uint64_t* bar, const uint32_t bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smemPtr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarWait(uint64_t* bar, const uint32_t parity)
{
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smemPtr(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulkLoad(void* smemDst, const void* gmemSrc, const uint32_t bytes, uint64_t* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smemPtr(smemDst)),
               "l"(gmemSrc), "r"(bytes), "r"(smemPtr(bar))
               : "memory");
}
__device__ __forceinline__ void bulkStore(void* gmemDst, const void* smemSrc, const uint32_t bytes)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmemDst), "r"(smemPtr(smemSrc)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulkCommit()
{
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int N> __device__ __forceinline__ void bulkWaitRead()
{
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N> __device__ __forceinline__ void bulkWaitAll()
{
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void fenceProxyAsync()
{
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ float f4(const float4& v, const int j)
{
  return j == 0 ? v.x : (j == 1 ? v.y : (j == 2 ? v.z : v.w));
}


// ---- the two recurrences on register-resident state vectors; coefficient row in shared memory ---------------------
// row = [E(hom-major) | E(het) | E(hom-minor) | D | B | U | RR], each Spad floats (buildSiteRowsKernel).
// Both steps read one vector and write the OTHER one ("ping-pong"): every element's last read is the instruction that
// overwrites its partner, so the unrolled site loop (two sites per trip, roles swapped) needs no register moves at its
// back edge (the in-place form cost 77 MOVs per warp-site, profiles/r1_v3_*).

// x: beta(p+1) on entry (destroyed); y: unscaled beta(p) on return.  ref: HMM.cpp:957-1016
//
// The step is two first-order recurrences in opposite directions (BU descending, BL ascending), each a chain of S
// dependent FMAs.  With two warps per scheduler a single chain leaves the FMA pipe idle for most of its 4-cycle
// latency, so the state range is cut in the middle and the two chains always run at the same time on different halves:
//   phase A: BU over the upper half (descending)  ||  BL over the lower half (ascending), partial results parked in y
//   phase B: BU over the lower half (descending)  ||  BL over the upper half (ascending), each completing y
// Same operations on the same operands as the one-chain-at-a-time form (bit-identical), same instruction count.
#ifndef FSMC_PACKED_FP32
#define FSMC_PACKED_FP32 1
#endif
// Packed fp32 (FFMA2 / FMUL2 / FADD2 of sm_100: two lanes of arithmetic per issue slot, same rounding as the scalar
// instructions).  The kernels are issue-bound, not pipe-bound, so every operation of a step that is NOT on one of the two
// dependent chains is done for two neighbouring states (2m, 2m+1) at once: per state a step is 2 chain FMAs + 4 halves of
// packed instructions = 4 issue slots instead of 6, with the same operations on the same operands (bit-identical).
__device__ __forceinline__ float2 pk(const float a, const float b)
{
  return make_float2(a, b);
}

template <int S> __device__ __forceinline__ void backwardStep(float (&x)[S], float (&y)[S], const float* row, const int cls)
{
  constexpr int SQ = (S + 3) / 4, Spad = SQ * 4, QM = (SQ + 1) / 2;
  static_assert(4 * QM < S - 1, "the lower half lies below the last state");
  const float4* E = reinterpret_cast<const float4*>(row + cls * Spad);
  const float4* Dr = reinterpret_cast<const float4*>(row + 3 * Spad);
  const float4* Br = reinterpret_cast<const float4*>(row + 4 * Spad);
  const float4* Rr = reinterpret_cast<const float4*>(row + 6 * Spad);
  const float4* Us = reinterpret_cast<const float4*>(row + 7 * Spad);  // U shifted by one state: Us[k] = U[k-1]
  float bu = 0.f, bl = 0.f;
  float above = 0.f;  // U[k] vec[k+1] for the state k the BU chain reaches next
  // phase A
#pragma unroll
  for (int i = 0; i < QM; ++i) {
    const int qu = SQ - 1 - i;
    if (qu >= QM) {
      const float4 e4 = E[qu], u4 = Us[qu], r4 = Rr[qu];
#pragma unroll
      for (int jp = 1; jp >= 0; --jp) {
        const int k = 4 * qu + 2 * jp, k1 = k + 1;
        if (k1 < S) {
          // vec = beta(p+1) * emission(p+1), in place; then U[k-1] vec[k]
          const float2 v = __fmul2_rn(pk(x[k], x[k1]), pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)));
          x[k] = v.x;
          x[k1] = v.y;
          const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), v);
          if (k1 == S - 1) {
            y[k1] = 0.f;  // BU[S-1] = 0
          } else {
            bu = fmaf(f4(r4, 2 * jp + 1), bu, above);  // BU[k] = U[k] vec[k+1] + RR[k] BU[k+1]
            y[k1] = bu;
          }
          bu = fmaf(f4(r4, 2 * jp), bu, t.y);
          y[k] = bu;
          above = t.x;
        } else if (k < S) {
          x[k] *= f4(e4, 2 * jp);
          above = f4(u4, 2 * jp) * x[k];
          if (k == S - 1) {
            y[k] = 0.f;
          } else {
            bu = fmaf(f4(r4, 2 * jp), bu, above);
            y[k] = bu;
          }
        }
      }
    }
    {
      const int ql = i;
      const float4 e4 = E[ql], d4 = Dr[ql], b4 = Br[ql];
#pragma unroll
      for (int jp = 0; jp < 2; ++jp) {
        const int k = 4 * ql + 2 * jp, k1 = k + 1;
        const float2 v = __fmul2_rn(pk(x[k], x[k1]), pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)));
        x[k] = v.x;
        x[k1] = v.y;
        const float bl0 = bl;
        const float bl1 = fmaf(f4(b4, 2 * jp), v.x, bl0);  // BL[k+1] = BL[k] + B[k] vec[k]
        bl = fmaf(f4(b4, 2 * jp + 1), v.y, bl1);
        const float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), v, pk(bl0, bl1));  // BL[k] + D[k] vec[k]
        y[k] = w.x;
        y[k1] = w.y;
      }
    }
  }
  // phase B
#pragma unroll
  for (int i = 0; i < QM; ++i) {
    {
      const int ql = QM - 1 - i;
      const float4 u4 = Us[ql], r4 = Rr[ql];
#pragma unroll
      for (int jp = 1; jp >= 0; --jp) {
        const int k = 4 * ql + 2 * jp, k1 = k + 1;
        const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), pk(x[k], x[k1]));
        const float b1 = fmaf(f4(r4, 2 * jp + 1), bu, above);
        const float b0 = fmaf(f4(r4, 2 * jp), b1, t.y);
        bu = b0;
        above = t.x;
        const float2 w = __fadd2_rn(pk(y[k], y[k1]), pk(b0, b1));
        y[k] = w.x;
        y[k1] = w.y;
      }
    }
    const int qu = QM + i;
    if (qu < SQ) {
      const float4 d4 = Dr[qu], b4 = Br[qu];
#pragma unroll
      for (int jp = 0; jp < 2; ++jp) {
        const int k = 4 * qu + 2 * jp, k1 = k + 1;
        if (k1 < S) {
          const float bl0 = bl;
          const float bl1 = fmaf(f4(b4, 2 * jp), x[k], bl0);
          bl = fmaf(f4(b4, 2 * jp + 1), x[k1], bl1);
          const float2 w = __fadd2_rn(__ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), pk(x[k], x[k1]), pk(bl0, bl1)),
                                      pk(y[k], y[k1]));
          y[k] = w.x;
          y[k1] = w.y;
        } else if (k < S) {
          y[k] = fmaf(f4(d4, 2 * jp), x[k], bl) + y[k];
        }
      }
    }
  }
}

template <int S> __device__ __forceinline__ float sumStates(const float (&a)[S])
{
  // four partial sums over the states k % 4, as two packed accumulators
  float2 s01 = pk(0.f, 0.f), s23 = pk(0.f, 0.f);
#pragma unroll
  for (int k = 0; k < S; k += 4) {
    if (k + 1 < S) {
      s01 = __fadd2_rn(s01, pk(a[k], a[k + 1]));
    } else {
      s01.x += a[k];
    }
    if (k + 3 < S) {
      s23 = __fadd2_rn(s23, pk(a[k + 2], a[k + 3]));
    } else if (k + 2 < S) {
      s23.x += a[k + 2];
    }
  }
  return (s01.x + s01.y) + (s23.x + s23.y);
}

template <int S> __device__ __forceinline__ void scaleStates(float (&a)[S], const float sc)
{
#pragma unroll
  for (int k = 0; k < S; k += 2) {
    if (k + 1 < S) {
      const float2 v = __fmul2_rn(pk(a[k], a[k + 1]), pk(sc, sc));
      a[k] = v.x;
      a[k + 1] = v.y;
    } else {
      a[k] *= sc;
    }
  }
}

// x: alpha(p-1) on entry; y: unscaled alpha(p) on return.  Returns sum_k alpha(p-1)[k], the normaliser of the previous
// site, for free.  ref: HMM.cpp:799-830.  Two chains (AU ascending, the suffix sums of x descending) run at the same
// time on different halves of the state range, like backwardStep:
//   phase A: y[k] = AU[k] + D[k] x[k] over the lower half  ||  y[k] = sum_{j>k} x[j] over the upper half
//   phase B: y[k] = E[k] (AU[k] + D[k] x[k] + B[k] y[k]) over the upper half  ||  y[k] = E[k] (y[k] + B[k] run) over the lower
template <int S>
__device__ __forceinline__ float forwardStep(const float* colRatios, float (&x)[S], float (&y)[S], const float* row, const int cls)
{
  constexpr int SQ = (S + 3) / 4, Spad = SQ * 4, QM = (SQ + 1) / 2;
  static_assert(4 * QM < S, "the upper half holds the last state");
  const float4* E = reinterpret_cast<const float4*>(row + cls * Spad);
  const float4* Dr = reinterpret_cast<const float4*>(row + 3 * Spad);
  const float4* Br = reinterpret_cast<const float4*>(row + 4 * Spad);
  const float4* Ur = reinterpret_cast<const float4*>(row + 5 * Spad);
  float au = 0.f, run = 0.f;
  // phase A
#pragma unroll
  for (int i = 0; i < QM; ++i) {
    {
      const int ql = i;
      const float4 d4 = Dr[ql], u4 = Ur[ql];
#pragma unroll
      for (int jp = 0; jp < 2; ++jp) {
        const int k = 4 * ql + 2 * jp, k1 = k + 1;
        const float2 xx = pk(x[k], x[k1]);
        const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), xx);
        const float au0 = au;
        const float au1 = fmaf(colRatios[k], au0, t.x);  // AU[k+1] = U[k] x[k] + colRatio[k] AU[k]
        au = fmaf(colRatios[k1], au1, t.y);
        const float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), xx, pk(au0, au1));  // AU[k] + D[k] x[k]
        y[k] = w.x;
        y[k1] = w.y;
      }
    }
    const int qu = SQ - 1 - i;
    if (qu >= QM) {
#pragma unroll
      for (int j = 3; j >= 0; --j) {
        const int k = 4 * qu + j;
        if (k < S) {
          y[k] = run;
          run += x[k];
        }
      }
    }
  }
  // phase B
#pragma unroll
  for (int i = 0; i < QM; ++i) {
    const int qu = QM + i;
    if (qu < SQ) {
      const float4 d4 = Dr[qu], u4 = Ur[qu], e4 = E[qu], b4 = Br[qu];
#pragma unroll
      for (int jp = 0; jp < 2; ++jp) {
        const int k = 4 * qu + 2 * jp, k1 = k + 1;
        if (k1 < S) {
          const float2 xx = pk(x[k], x[k1]);
          const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), xx);
          const float au0 = au;
          const float au1 = fmaf(colRatios[k], au0, t.x);
          au = fmaf(colRatios[k1], au1, t.y);
          const float2 tt = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), xx, pk(au0, au1));
          // (the last state's suffix sum is 0: its B term adds nothing, as in the reference's special case)
          const float2 w = __fmul2_rn(pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)),
                                      __ffma2_rn(pk(f4(b4, 2 * jp), f4(b4, 2 * jp + 1)), pk(y[k], y[k1]), tt));
          y[k] = w.x;
          y[k1] = w.y;
        } else if (k < S) {
          y[k] = f4(e4, 2 * jp) * fmaf(f4(d4, 2 * jp), x[k], au);  // k == S-1 (S odd)
        }
      }
    }
    {
      const int ql = QM - 1 - i;
      const float4 e4 = E[ql], b4 = Br[ql];
#pragma unroll
      for (int jp = 1; jp >= 0; --jp) {
        const int k = 4 * ql + 2 * jp, k1 = k + 1;
        const float s1 = run;  // sum_{j>k1} x[j]
        const float s0 = s1 + x[k1];
        run = s0 + x[k];
        const float2 w = __fmul2_rn(pk(f4(e4, 2 * jp), f4(e4, 2 * jp + 1)),
                                    __ffma2_rn(pk(f4(b4, 2 * jp), f4(b4, 2 * jp + 1)), pk(s0, s1), pk(y[k], y[k1])));
        y[k] = w.x;
        y[k1] = w.y;
      }
    }
  }
  return run;
}

// ---- the backward step on the narrow kernel's backward rows (buildBackwardRowsKernel) -----------------------------------
// The emission is part of the coefficients, so the packed multiply v = beta * E per pair of states goes: 7 issue slots and
// 4 LDS.128 per two states instead of 8 and 5.  Same phases and chains as backwardStep; the products round differently
// ((U E) x instead of U (E x): fp32, within the fast mode's 1e-4).
// x: beta(p+1) on entry (kept); y: unscaled beta(p) on return.  row = backward row of site p+1.
template <int S>
__device__ __forceinline__ void backwardStepFolded(const float (&x)[S], float (&y)[S], const float* row, const int cls)
{
  constexpr int SQ = (S + 3) / 4, Spad = SQ * 4, QM = (SQ + 1) / 2;
  static_assert(4 * QM < S - 1, "the lower half lies below the last state");
  const float4* UsE = reinterpret_cast<const float4*>(row + cls * Spad);  // Us[k] E[k] = U[k-1] E[k]
  const float4* DE = reinterpret_cast<const float4*>(row + (3 + cls) * Spad);
  const float4* BE = reinterpret_cast<const float4*>(row + (6 + cls) * Spad);
  const float4* Rr = reinterpret_cast<const float4*>(row + 9 * Spad);
  float bu = 0.f, bl = 0.f;
  float above = 0.f;  // U[k] E[k+1] x[k+1] for the state k the BU chain reaches next
  // phase A
#pragma unroll
  for (int i = 0; i < QM; ++i) {
    const int qu = SQ - 1 - i;
    if (qu >= QM) {
      const float4 u4 = UsE[qu], r4 = Rr[qu];
#pragma unroll
      for (int jp = 1; jp >= 0; --jp) {
        const int k = 4 * qu + 2 * jp, k1 = k + 1;
        if (k1 < S) {
          const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), pk(x[k], x[k1]));
          if (k1 == S - 1) {
            y[k1] = 0.f;  // BU[S-1] = 0
          } else {
            bu = fmaf(f4(r4, 2 * jp + 1), bu, above);  // BU[k] = U[k] E[k+1] x[k+1] + RR[k] BU[k+1]
            y[k1] = bu;
          }
          bu = fmaf(f4(r4, 2 * jp), bu, t.y);
          y[k] = bu;
          above = t.x;
        } else if (k < S) {
          above = f4(u4, 2 * jp) * x[k];
          if (k == S - 1) {
            y[k] = 0.f;
          } else {
            bu = fmaf(f4(r4, 2 * jp), bu, above);
            y[k] = bu;
          }
        }
      }
    }
    {
      const int ql = i;
      const float4 d4 = DE[ql], b4 = BE[ql];
#pragma unroll
      for (int jp = 0; jp < 2; ++jp) {
        const int k = 4 * ql + 2 * jp, k1 = k + 1;
        const float bl0 = bl;
        const float bl1 = fmaf(f4(b4, 2 * jp), x[k], bl0);  // BL[k+1] = BL[k] + B[k] E[k] x[k]
        bl = fmaf(f4(b4, 2 * jp + 1), x[k1], bl1);
        const float2 w = __ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), pk(x[k], x[k1]), pk(bl0, bl1));
        y[k] = w.x;
        y[k1] = w.y;
      }
    }
  }
  // phase B
#pragma unroll
  for (int i = 0; i < QM; ++i) {
    {
      const int ql = QM - 1 - i;
      const float4 u4 = UsE[ql], r4 = Rr[ql];
#pragma unroll
      for (int jp = 1; jp >= 0; --jp) {
        const int k = 4 * ql + 2 * jp, k1 = k + 1;
        const float2 t = __fmul2_rn(pk(f4(u4, 2 * jp), f4(u4, 2 * jp + 1)), pk(x[k], x[k1]));
        const float b1 = fmaf(f4(r4, 2 * jp + 1), bu, above);
        const float b0 = fmaf(f4(r4, 2 * jp), b1, t.y);
        bu = b0;
        above = t.x;
        const float2 w = __fadd2_rn(pk(y[k], y[k1]), pk(b0, b1));
        y[k] = w.x;
        y[k1] = w.y;
      }
    }
    const int qu = QM + i;
    if (qu < SQ) {
      const float4 d4 = DE[qu], b4 = BE[qu];
#pragma unroll
      for (int jp = 0; jp < 2; ++jp) {
        const int k = 4 * qu + 2 * jp, k1 = k + 1;
        if (k1 < S) {
          const float bl0 = bl;
          const float bl1 = fmaf(f4(b4, 2 * jp), x[k], bl0);
          bl = fmaf(f4(b4, 2 * jp + 1), x[k1], bl1);
          const float2 w = __fadd2_rn(__ffma2_rn(pk(f4(d4, 2 * jp), f4(d4, 2 * jp + 1)), pk(x[k], x[k1]), pk(bl0, bl1)),
                                      pk(y[k], y[k1]));
          y[k] = w.x;
          y[k1] = w.y;
        } else if (k < S) {
          y[k] = fmaf(f4(d4, 2 * jp), x[k], bl) + y[k];
        }
      }
    }
  }
}

// One item per lane with `pred` (decode_sparse.cuh): slots from one atomic per warp, the descriptor, and alpha at the block's
// first site (copied from the warp's scratch, column `lane`).  Returns the lane's new chain head.  Out of line on purpose:
// it runs at a few percent of the sites, and inlined into the unrolled site loop it slowed every site down (the loop no
// longer streamed from the instruction cache: 413 ms instead of 329 ms per cfg2 step).
static __device__ __noinline__ int emitSparseItems(SparseItem* items, float* itemAlpha, unsigned long long* itemCount,
                                            const long long capacity, const bool pred, const uint32_t pair, const int block,
                                            const int first, const int last, int chain, const float4* alphaStart,
                                            const int lane, const int SQ)
{
  const unsigned mask = __ballot_sync(kFull, pred);
  if (!mask) {
    return chain;
  }
  unsigned long long base = 0;
  if (lane == 0) {
    base = atomicAdd(itemCount, static_cast<unsigned long long>(__popc(mask)));
  }
  base = __shfl_sync(kFull, base, 0);
  if (pred) {
    const long long slot = static_cast<long long>(base) + __popc(mask & ((1u << lane) - 1u));
    if (slot < capacity) {
      items[slot] = SparseItem{pair, block, first, last, chain};
      float4* dst = reinterpret_cast<float4*>(itemAlpha + static_cast<size_t>(slot) * SQ * 4);
      for (int q = 0; q < SQ; ++q) {
        dst[q] = alphaStart[q * 32 + lane];
      }
    }
    chain = static_cast<int>(slot);
  }
  return chain;
}

// -------------------------------------------------------------------------------------------------------------------
// decodeNarrowKernel: the same sweeps WITHOUT the beta round trip, for requests that only look at the states below the
// IBD time threshold (segment calling, per-site IBD probability, and age estimates conditioned on TMRCA < threshold,
// which is FastSMC's default: ageThreshold == stateThreshold, ref: HMM.cpp:101-105).
//
// What the consumers need at site t is  sum_{k<sT} alpha_t[k] beta_t[k] / Z_t  with  Z_t = sum_k alpha_t[k] beta_t[k]
// over ALL states.  For scaled vectors alpha^ = alpha/A_t, beta^ = beta/B_t the full dot product telescopes:
// Z_t = P(data)/(A_t B_t), hence Z_{t+1} = Z_t * b_t / a_{t+1} with a, b the per-site scale divisors that the sweeps
// apply anyway.  Z is computed exactly once (at the first site, where the backward sweep ends with all of beta in
// registers) and carried by that recurrence, so the backward sweep only has to leave a record of 4*RQ floats per
// pair-site in HBM (beta^[k < sT], zero padding, and b_t in the last slot) instead of S: 16 bytes instead of 276 at
// S=69, sT<=3.  The kernel becomes issue-bound.
// -------------------------------------------------------------------------------------------------------------------
constexpr int kNarrowMaxQuads = 4;  // record = up to 16 floats: sT <= 15
constexpr int kNarrowGroup = 4;     // window positions per ring slot (one bulk copy and one barrier per group)

// Ring slot of one warp: G coefficient rows (backward rows in the backward sweep, the smaller 8-array rows in the forward
// sweep) followed by G+1 records (the extra record is the all-ones beta of the window's last site, which rides with the
// first group of the backward sweep).  RQ = 1, G = 4: 112.7 KB per CTA of 4 warps at DEPTH 2, two CTAs per SM.
template <int S_T, int RQ, int G> struct NarrowSlot {
  static constexpr int SQ = (S_T + 3) / 4, Spad = SQ * 4;
  static constexpr uint32_t kCoefBytes = kBwdArrays * Spad * 4;
  static constexpr uint32_t kRecBytes = RQ * 32 * 16;
  static constexpr uint32_t kBytes = G * kCoefBytes + (G + 1) * kRecBytes;
};

// Site loop: positions are handled in groups of G.  Per group the elected lane waits once on the slot's mbarrier,
// and issues one bulk copy per array (coefficient rows are contiguous over consecutive sites, and so are the records
// of consecutive positions in the slab), so the per-site cost outside the recurrences is the genotype class lookup,
// the record (RQ shared-memory accesses) and the segment caller.  Rescaling happens at the last step of every full
// group, i.e. every G-th site.
//
// SPARSE (decode_sparse.cuh): age estimates over ALL states without a beta round trip.  The window is cut into blocks of
// 2^ckptShift positions (counted from the window's first site; a multiple of the group size G, so block boundaries are
// group boundaries in both sweeps and the per-site code is that of the plain kernel).  The backward sweep leaves a full
// beta vector at the last position of every block (checkpoints, 4*Spad/2^ckptShift bytes per pair-site), the forward sweep
// keeps alpha of the position before the current block in a per-warp scratch that stays in L2 and records every piece of
// an IBD run (one item per run and block) together with that alpha.  The refine pass recomputes the full posterior only
// inside those pieces.
template <int S_T, int RQ, int G, int DEPTH, int THREADS, int MIN_BLOCKS, int SPARSE_V = 0>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) decodeNarrowKernel(const FastModel fm, const DecodeArgs args)
{
  constexpr bool SPARSE = (SPARSE_V & 1) != 0;
  constexpr bool kSkipFwd = (SPARSE_V & 2) != 0, kSkipBwd = (SPARSE_V & 4) != 0;  // timing experiments only
  // One copy of each step pair per sweep: the site loops stream from the instruction cache.  Fully unrolled over the group
  // (bit 64, kept for A/B runs) the kernel is ~100 KB of straight-line code and `no_instruction` is its first stall
  // (profiles/r2_p1_decodeNarrowSparse_packed_unrolled_ncu_full.txt: 1.61 warps per issue; 346 -> 294 ms per cfg2 step without the unrolling).
  constexpr int kGroupUnroll = (SPARSE_V & 64) ? G / 2 : 1;
  constexpr bool kSkipAlpha = (SPARSE_V & 8) != 0, kSkipBoundaryItems = (SPARSE_V & 16) != 0, kSkipRunItems = (SPARSE_V & 32) != 0;
  constexpr int S = S_T;
  constexpr int SQ = (S + 3) / 4;
  constexpr int Spad = SQ * 4;
  constexpr int NR = 4 * RQ - 1;                     // beta entries of a record; entry NR is the scale divisor
  using Slot = NarrowSlot<S_T, RQ, G>;
  constexpr uint32_t kRecBytes = Slot::kRecBytes;
  constexpr uint32_t kCoefBytes = Slot::kCoefBytes;
  constexpr size_t kRecFloats = static_cast<size_t>(RQ) * 32 * 4;
  constexpr size_t kRowFloats = static_cast<size_t>(kRowArrays) * Spad;  // forward sweep: the 8-array rows
  constexpr uint32_t kRowBytes = static_cast<uint32_t>(kRowFloats) * 4;
  constexpr size_t kBwdFloats = static_cast<size_t>(kBwdArrays) * Spad;  // backward sweep: the folded rows
  constexpr int kWarps = THREADS / 32;
  constexpr size_t kWarpBytes = static_cast<size_t>(DEPTH) * Slot::kBytes;
  static_assert(S >= 4 * kNarrowMaxQuads && RQ >= 1 && RQ <= kNarrowMaxQuads, "record quads index the state vector");
  static_assert(G % 2 == 0, "the two state vectors swap roles every step");

  extern __shared__ __align__(128) unsigned char smemRaw[];
  const DeviceModel m = fm.base;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  unsigned char* mine = smemRaw + static_cast<size_t>(warp) * kWarpBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smemRaw + static_cast<size_t>(kWarps) * kWarpBytes) + warp * DEPTH;
  auto coefArea = [&](const int slot) { return reinterpret_cast<float*>(mine + static_cast<size_t>(slot) * Slot::kBytes); };
  auto recArea = [&](const int slot) {
    return reinterpret_cast<float4*>(mine + static_cast<size_t>(slot) * Slot::kBytes + static_cast<size_t>(G) * kCoefBytes);
  };
  if (lane == 0) {
    for (int i = 0; i < DEPTH; ++i) {
      mbarInit(&bars[i], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  uint32_t parity = 0;  // bit i = parity the next wait on slot i expects

  const unsigned flags = args.flags;
  const bool wantSeg = flags & FSMC_CALL_SEGMENTS;
  const bool wantAge = !SPARSE && (flags & FSMC_SEG_AGE) && wantSeg;  // SPARSE: the refine pass computes the age estimates
  const int sT = m.stateThreshold;  // <= NR by the host's kernel choice
  const long long warpGlobal = static_cast<long long>(blockIdx.x) * kWarps + warp;
  float* slab = args.scratch + warpGlobal * args.scratchPerWarp;
  constexpr size_t kVecFloats = static_cast<size_t>(SQ) * 32 * 4;  // one state vector of the warp, [quad][lane][4]
  const int ckShift = SPARSE ? args.ckptShift : 0;
  const int ckMask = (1 << ckShift) - 1;
  float4* alphaStart = SPARSE ? reinterpret_cast<float4*>(args.alphaScratch + warpGlobal * kVecFloats) : nullptr;

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
    const int scanFrom = wantSeg ? args.tileScanFrom[tile] : 0;
    const int scanTo = wantSeg ? args.tileScanTo[tile] : 0;
    const bool laneActive = lane < nPairs;
    const int srcLane = laneActive ? lane : nPairs - 1;
    const uint32_t pair = static_cast<uint32_t>(tile) * 32u + static_cast<uint32_t>(lane);
    PairBits bits;
    bits.a = m.haps + static_cast<size_t>(args.hapA[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    bits.b = m.haps + static_cast<size_t>(args.hapB[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    const float* rowBase = m.siteRows + static_cast<size_t>(from) * kRowFloats;
    // SPARSE: checkpoint slot of block b (window positions [b << ckShift, ...)) of this tile = ckptSlot0 + b
    const long long ckptSlot0 = SPARSE ? args.tileCkptBase[tile] : 0;
    // full state vector of the warp -> [quad][lane][4] in global memory (coalesced 512-byte rows)
    auto storeVector = [&](const float (&v)[S], float4* dst) {
#pragma unroll
      for (int q = 0; q < SQ; ++q) {
        dst[q * 32 + lane] = make_float4(v[4 * q], 4 * q + 1 < S ? v[4 * q + 1] : 0.f, 4 * q + 2 < S ? v[4 * q + 2] : 0.f,
                                         4 * q + 3 < S ? v[4 * q + 3] : 0.f);
      }
    };
    auto storeCheckpoint = [&](const float (&v)[S], const int p) {  // beta of window position p, the last of its block
      storeVector(v, reinterpret_cast<float4*>(args.ckptBeta + static_cast<size_t>(ckptSlot0 + (p >> ckShift)) * kVecFloats));
    };

    float a[S], c[S];
    float acc[NR];
#pragma unroll
    for (int k = 0; k < NR; ++k) {
      acc[k] = 0.f;
    }

    // (beta^[k < sT], 0.., scale divisor) of one window position into a staging record
    auto stageRecord = [&](const float (&v)[S], float4* out, const float divisor) {
#pragma unroll
      for (int q = 0; q < RQ; ++q) {
        float w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int k = 4 * q + i;
          w[i] = k == NR ? divisor : (k < sT ? v[k] : 0.f);
        }
        out[q * 32 + lane] = make_float4(w[0], w[1], w[2], w[3]);
      }
    };

    // ---- sweep 1: backward.  Step j handles window position len-2-j with the coefficient row of len-1-j ------------
    {
      const int steps = len - 1;
      // groups of G steps; SPARSE: the first group is shortened so that every later group starts at a window position
      // p with p % G == G - 1 — then the last position of every checkpoint block is the top of a group
      const int first = SPARSE ? min(steps, (len % G) ? (len % G) : G) : G;
      const int nGroups = steps <= 0 ? 0 : 1 + (max(steps - first, 0) + G - 1) / G;
      auto groupBegin = [&](const int g) { return g == 0 ? 0 : first + (g - 1) * G; };
      auto prefetch = [&](const int g) {  // rows of the group's steps [j0, j1): window positions [len-j1, len-j0), ascending
        if (lane == 0) {
          const int j0 = groupBegin(g), j1 = min(steps, j0 + (g == 0 ? first : G));
          const int slot = g % DEPTH;
          const uint32_t bytes = static_cast<uint32_t>(j1 - j0) * kCoefBytes;
          mbarExpectTx(&bars[slot], bytes);
          bulkLoad(coefArea(slot), m.bwdRows + static_cast<size_t>(from + len - j1) * kBwdFloats, bytes, &bars[slot]);
        }
      };
      for (int g = 0; g < DEPTH && g < nGroups; ++g) {
        prefetch(g);
      }
#pragma unroll
      for (int k = 0; k < S; ++k) {
        a[k] = 1.f;
      }
      if constexpr (SPARSE) {
        storeCheckpoint(a, len - 1);  // the window's last block ends at its last position (beta = ones)
      }
      if (nGroups == 0) {
        // single-site window: only the all-ones record
        stageRecord(a, recArea(0), 1.0f);
        fenceProxyAsync();
        __syncwarp();
        if (lane == 0) {
          bulkStore(slab, recArea(0), kRecBytes);
          bulkCommit();
        }
      }
      for (int g = 0; g < nGroups; ++g) {
        const int slot = g % DEPTH;
        const int j0 = groupBegin(g);
        const int n = min(g == 0 ? first : G, steps - j0);
        const float* coef = coefArea(slot);
        float4* stage = recArea(slot);
        if constexpr (SPARSE && !kSkipBwd) {
          // a = beta of window position len-1-j0, the top of this group: the last position of a block?
          if (g > 0 && ((len - 1 - j0) & ckMask) == ckMask) {
            storeCheckpoint(a, len - 1 - j0);
          }
        }
        if (lane == 0) {
          bulkWaitRead<DEPTH - 1>();  // the store that last read this slot's staging records has drained them
        }
        mbarWait(&bars[slot], (parity >> slot) & 1u);
        parity ^= 1u << slot;
        __syncwarp();
        if (g == 0) {
          stageRecord(a, stage + static_cast<size_t>(n) * RQ * 32, 1.0f);  // position len-1
        }
        auto step = [&](const int i, float (&x)[S], float (&y)[S], const bool rescale) {
          const int p = len - 2 - (j0 + i);
          const int cls = bits.cls(from + p + 1);
          backwardStepFolded<S>(x, y, coef + static_cast<size_t>(n - 1 - i) * kBwdFloats, cls);
          float divisor = 1.0f;
          if (rescale) {
            divisor = sumStates<S>(y);
            scaleStates<S>(y, 1.0f / divisor);
          }
          stageRecord(y, stage + static_cast<size_t>(n - 1 - i) * RQ * 32, divisor);
        };
        // The kernel is bound by instruction supply: per-SITE sparse bookkeeping made "no instruction" its first stall
        // (profiles/r2_v4_decodeNarrowSparse_ncu_full.txt), which is why that bookkeeping lives at the group tops.
#pragma unroll(kGroupUnroll)
        for (int i = 0; i < G; i += 2) {
          if (i < n) {
            step(i, a, c, false);
          }
          if (i + 1 < n) {
            step(i + 1, c, a, i + 1 == G - 1);
          }
        }
        fenceProxyAsync();
        __syncwarp();  // every lane is done with the coefficient rows and has staged its records
        if (lane == 0) {
          const int j1 = j0 + n;
          bulkStore(slab + static_cast<size_t>(len - 1 - j1) * kRecFloats, stage,
                    static_cast<uint32_t>(n + (g == 0 ? 1 : 0)) * kRecBytes);
          bulkCommit();
        }
        if (g + DEPTH < nGroups) {
          prefetch(g + DEPTH);
        }
        if (SPARSE && g == 0 && (n & 1)) {
          // a shortened first group of odd size left its result in c: the groups read a
#pragma unroll
          for (int k = 0; k < S; ++k) {
            a[k] = c[k];
          }
        }
      }
      // where beta^ of the first site ended: the steps after the first group alternate a -> c -> a (the first group ends
      // in a: even size, or copied above)
      const int rest = SPARSE ? max(steps - first, 0) : steps;
      if (rest & 1) {
        // in c
      } else {
#pragma unroll
        for (int k = 0; k < S; ++k) {
          c[k] = a[k];
        }
      }
      if (lane == 0) {
        bulkWaitAll<0>();
      }
      __syncwarp();
    }

    // ---- sweep 2: forward + consumers ---------------------------------------------------------------------------------
    {
      const int nGroups = (len + G - 1) / G;
      auto prefetch = [&](const int g) {
        if (lane == 0) {
          const int p0 = g * G;
          const uint32_t n = static_cast<uint32_t>(min(G, len - p0));
          const int slot = g % DEPTH;
          mbarExpectTx(&bars[slot], n * (kRowBytes + kRecBytes));
          bulkLoad(coefArea(slot), rowBase + static_cast<size_t>(p0) * kRowFloats, n * kRowBytes, &bars[slot]);
          bulkLoad(recArea(slot), slab + static_cast<size_t>(p0) * kRecFloats, n * kRecBytes, &bars[slot]);
        }
      };
      for (int g = 0; g < DEPTH && g < nGroups; ++g) {
        prefetch(g);
      }
      CallerState cs;
      float Z = 1.f, bPrev = 1.f;
      // SPARSE: the open piece of the lane's current run (sites pieceStart.. in the current block) and the chain of the
      // run's earlier pieces
      bool runOpen = false;
      int pieceStart = 0, chain = -1;
      auto emitItems = [&](const bool pred, const int block, const int first, const int last) {
        chain = emitSparseItems(args.items, args.itemAlpha, args.itemCount, args.itemCapacity, pred, pair, block, first, last, chain,
                                alphaStart, lane, SQ);
      };

      // consumers of window position p; v = alpha^(p); rec = this position's record (parking area once drained)
      auto consume = [&](const int p, const float (&v)[S], float4* rec) {
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
          if constexpr (SPARSE && !kSkipFwd) {
            if (__any_sync(kFull, ending || closing)) {
              // the run's last piece, then the record; the refine pass fills in the age estimates from the chain
              if constexpr (!kSkipRunItems) {
                emitItems(ending && runOpen && pieceStart <= site - 1, (p - 1) >> ckShift, pieceStart, site - 1);
              }
              if (ending) {
                emitSegment<false>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, nullptr, false, chain);
                chain = -1;
                runOpen = false;
              }
              if (now >= 0 && changed) {
                runOpen = true;
                pieceStart = site;
              }
              if constexpr (!kSkipRunItems) {
                emitItems(closing, p >> ckShift, pieceStart, site);
              }
              if (closing) {
                emitSegment<false>(m, args, pair, changed ? site : cs.start, site, changed ? ibd : cs.prob + ibd, now, nullptr,
                                   false, chain);
                chain = -1;
                runOpen = false;
              }
            } else if (now >= 0 && changed) {
              runOpen = true;
              pieceStart = site;
            }
          } else if (__any_sync(kFull, ending || closing)) {
            // rare: a run ends at site-1 and/or the scan window closes on a live run
            float* park = reinterpret_cast<float*>(rec) + lane;  // drained record: [k][32], k < NR
            __syncwarp();
            if (wantAge) {
#pragma unroll
              for (int k = 0; k < NR; ++k) {
                park[k * 32] = acc[k];
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
                acc[k] = fmaf(q[k], rr, keep * acc[k]);
                park[k * 32] = acc[k];
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
              acc[k] = fmaf(q[k], rr, keep * acc[k]);
            }
          }
          cs.prob = (now >= 0 && !closing) ? (changed ? ibd : cs.prob + ibd) : 0.f;
          cs.start = (now >= 0 && changed) ? site : cs.start;
          cs.level = now;
        }
      };

      for (int g = 0; g < nGroups; ++g) {
        const int slot = g % DEPTH;
        const int p0 = g * G;
        const int n = min(G, len - p0);
        const float* coef = coefArea(slot);
        float4* recs = recArea(slot);
        mbarWait(&bars[slot], (parity >> slot) & 1u);
        parity ^= 1u << slot;
        if constexpr (SPARSE && !kSkipFwd) {
          if (g > 0 && (p0 & ckMask) == 0) {
            // a block begins with this group; c = alpha of the position before it.  A run that continues into the block
            // leaves the piece of the block that just ended (with the alpha that was parked when that block began), then
            // the new block's alpha is parked.  Same lanes write and read the scratch: no synchronisation needed.
            if constexpr (!kSkipBoundaryItems) {
              if (__any_sync(kFull, runOpen)) {
                emitItems(runOpen, (p0 - 1) >> ckShift, pieceStart, from + p0 - 1);
              }
            }
            pieceStart = from + p0;
            if constexpr (!kSkipAlpha) {
              storeVector(c, alphaStart);
            }
          }
        }
        auto step = [&](const int i, float (&x)[S], float (&y)[S], const bool rescale) {
          const int p = p0 + i;
          const int cls = bits.cls(from + p);
          const float total = forwardStep<S>(fm.colRatios, x, y, coef + static_cast<size_t>(i) * kRowFloats, cls);
          float sc = 1.0f;
          if (rescale) {
            sc = 1.0f / total;
            scaleStates<S>(y, sc);
          }
          Z *= bPrev * sc;  // Z_p = Z_{p-1} * b_{p-1} / a_p
          consume(p, y, recs + static_cast<size_t>(i) * RQ * 32);
        };
#pragma unroll(kGroupUnroll)
        for (int i = 0; i < G; i += 2) {
          if (i == 0 && g == 0) {
            // p = 0: alpha^(0) = prior * emission into a; the one exact normaliser Z_0 = sum_k alpha^(0)[k] beta^(0)[k]
            const int cls = bits.cls(from);
            const float4* E = reinterpret_cast<const float4*>(coef + cls * Spad);
            float z0 = 0.f, z1 = 0.f, z2 = 0.f, z3 = 0.f;
#pragma unroll
            for (int q = 0; q < SQ; ++q) {
              const float4 e4 = E[q];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const int k = 4 * q + j;
                if (k < S) {
                  a[k] = fm.prior[k] * f4(e4, j);
                }
              }
              z0 = fmaf(a[4 * q], c[4 * q], z0);
              if (4 * q + 1 < S) z1 = fmaf(a[4 * q + 1], c[4 * q + 1], z1);
              if (4 * q + 2 < S) z2 = fmaf(a[4 * q + 2], c[4 * q + 2], z2);
              if (4 * q + 3 < S) z3 = fmaf(a[4 * q + 3], c[4 * q + 3], z3);
            }
            Z = (z0 + z1) + (z2 + z3);
            consume(0, a, recs);
          } else if (i < n) {
            step(i, c, a, false);
          }
          if (i + 1 < n) {
            step(i + 1, a, c, i + 1 == G - 1);
          }
        }
        __syncwarp();  // the slot is drained (its records double as the parking area above)
        if (g + DEPTH < nGroups) {
          prefetch(g + DEPTH);
        }
      }
    }
    __syncwarp();
  }
}

// -------------------------------------------------------------------------------------------------------------------
// decodeFastKernel: all states reach the consumers (per-site posterior mean / MAP, age estimates over all states):
// the backward sweep streams full beta rows through HBM.
// S_T   : states (compile time), DEPTH: ring depth, RESCALE: sites between rescalings (power of two)
// ACC   : keep per-state segment accumulators (FSMC_SEG_AGE) in registers
// -------------------------------------------------------------------------------------------------------------------
// SUM   : FSMC_SUM_POSTERIOR[_BY_GENOTYPE] (ref: HMM.cpp:1044-1085 augmentSumOverPairs).  Every resident warp adds the
//         posteriors of its tiles into a PRIVATE [plane][site][state] accumulator in global memory (plain read-add-write,
//         no atomics; the 32 pairs of a tile are first added up through the drained beta slot in shared memory), tiles are
//         dealt to the warps statically, and sumScratchReduceKernel adds the warps' accumulators in a fixed order: the
//         result does not depend on scheduling.
template <int S_T, int DEPTH, int RESCALE, bool ACC, int THREADS, int MIN_BLOCKS, bool SUM = false>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS) decodeFastKernel(const FastModel fm, const DecodeArgs args)
{
  constexpr int S = S_T;
  constexpr int SQ = (S + 3) / 4;
  constexpr int Spad = SQ * 4;
  constexpr uint32_t kBetaBytes = SQ * 32 * 16;           // one site of beta for 32 lanes
  constexpr uint32_t kCoefBytes = kRowArrays * Spad * 4;  // one site's coefficient row
  constexpr size_t kBetaFloats = static_cast<size_t>(SQ) * 32 * 4;
  constexpr int kWarps = THREADS / 32;
  constexpr size_t kWarpBytes = static_cast<size_t>(DEPTH) * (kBetaBytes + kCoefBytes);

  extern __shared__ __align__(128) unsigned char smemRaw[];
  const DeviceModel m = fm.base;  // a copy: taking the address of a kernel parameter would move all of fm to local memory
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  unsigned char* mine = smemRaw + static_cast<size_t>(warp) * kWarpBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smemRaw + static_cast<size_t>(kWarps) * kWarpBytes) +
                   warp * 2 * DEPTH;  // [0,DEPTH): beta slot full, [DEPTH,2*DEPTH): coefficient slot full
  auto betaSlot = [&](const int i) { return reinterpret_cast<float4*>(mine + static_cast<size_t>(i) * kBetaBytes); };
  auto coefSlot = [&](const int i) {
    return reinterpret_cast<const float*>(mine + static_cast<size_t>(DEPTH) * kBetaBytes + static_cast<size_t>(i) * kCoefBytes);
  };
  if (lane == 0) {
    for (int i = 0; i < 2 * DEPTH; ++i) {
      mbarInit(&bars[i], 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  uint32_t betaParity = 0, coefParity = 0;  // bit i = parity the next wait on slot i expects

  const unsigned flags = args.flags;
  const bool wantSeg = flags & FSMC_CALL_SEGMENTS;
  const bool wantAge = ACC && (flags & FSMC_SEG_AGE) && wantSeg;
  const bool wantSite = flags & (FSMC_SITE_MEAN | FSMC_SITE_MAP);
  const int sT = m.stateThreshold;
  const int nAcc = m.ageThreshold;
  const long long warpGlobal = static_cast<long long>(blockIdx.x) * kWarps + warp;
  float* slab = args.scratch + warpGlobal * args.scratchPerWarp;  // beta rows of this warp
  const int sumPlanes = SUM && (flags & FSMC_SUM_BY_GENOTYPE) ? 3 : 1;
  float* sumMine = SUM ? args.sumScratch + static_cast<size_t>(warpGlobal) * sumPlanes * m.L * Spad : nullptr;
  const long long totalWarps = static_cast<long long>(gridDim.x) * kWarps;

  for (long long turn = 0;; ++turn) {
    unsigned long long t = 0;
    if constexpr (SUM) {
      t = static_cast<unsigned long long>(warpGlobal + turn * totalWarps);  // static deal: reproducible sums
    } else {
      if (lane == 0) {
        t = atomicAdd(args.tileCounter, 1ull);
      }
      t = __shfl_sync(kFull, t, 0);
    }
    if (static_cast<long long>(t) >= args.numTiles) {
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
    const uint32_t outRow = args.laneRow ? __ldg(args.laneRow + pair) : pair;  // output row (fsmc_decode_device)
    PairBits bits;
    bits.a = m.haps + static_cast<size_t>(args.hapA[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    bits.b = m.haps + static_cast<size_t>(args.hapB[static_cast<size_t>(tile) * 32 + srcLane]) * m.wordsPerHap;
    const float* rowBase = m.siteRows + static_cast<size_t>(from) * kRowArrays * Spad;  // row of window position 0

    float a[S], c[S];
    float acc[ACC ? S : 1];  // per-state posterior sums of the lane's current IBD run (FSMC_SEG_AGE)
#pragma unroll
    for (int k = 0; k < (ACC ? S : 1); ++k) {
      acc[k] = 0.f;
    }

    // stage the beta row of window position p and hand it to the copy engine
    auto storeRow = [&](const float (&v)[S], const int p, const int bslot) {
      if (lane == 0) {
        bulkWaitRead<DEPTH - 1>();  // the copy that last read this staging slot has drained it
      }
      __syncwarp();
      float4* out = betaSlot(bslot);
#pragma unroll
      for (int q = 0; q < SQ; ++q) {
        out[q * 32 + lane] = make_float4(v[4 * q], 4 * q + 1 < S ? v[4 * q + 1] : 0.f, 4 * q + 2 < S ? v[4 * q + 2] : 0.f,
                                         4 * q + 3 < S ? v[4 * q + 3] : 0.f);
      }
      fenceProxyAsync();
      __syncwarp();
      if (lane == 0) {
        bulkStore(slab + static_cast<size_t>(p) * kBetaFloats, out, kBetaBytes);
        bulkCommit();
      }
    };

    // =============================================================================================================
    // sweep 1: backward (ref: HMM.cpp:882-1041).  Step j = 0 .. len-2 handles p = len-2-j with the row of p+1.
    // =============================================================================================================
    {
      auto prefetchCoef = [&](const int j) {  // row of window position len-1-j into slot j % DEPTH
        if (lane == 0) {
          uint64_t* bar = &bars[DEPTH + j % DEPTH];
          mbarExpectTx(bar, kCoefBytes);
          bulkLoad(const_cast<float*>(coefSlot(j % DEPTH)), rowBase + static_cast<size_t>(len - 1 - j) * kRowArrays * Spad,
                   kCoefBytes, bar);
        }
      };
      const int steps = len - 1;
      for (int j = 0; j < DEPTH && j < steps; ++j) {
        prefetchCoef(j);
      }
#pragma unroll
      for (int k = 0; k < S; ++k) {
        a[k] = 1.f;  // beta at the last site: all ones (any positive scale is equivalent)
      }
      storeRow(a, len - 1, 0);
      auto step = [&](const int j, float (&x)[S], float (&y)[S]) {
        const int p = len - 2 - j;
        const int slot = j % DEPTH;
        const int cls = bits.cls(from + p + 1);
        mbarWait(&bars[DEPTH + slot], (coefParity >> slot) & 1u);
        coefParity ^= 1u << slot;
        backwardStep<S>(x, y, coefSlot(slot), cls);
        __syncwarp();  // every lane is done with the coefficient slot
        if (j + DEPTH < steps) {
          prefetchCoef(j + DEPTH);
        }
        if ((p & (RESCALE - 1)) == 0) {
          scaleStates<S>(y, 1.0f / sumStates<S>(y));
        }
        storeRow(y, p, (j + 1) % DEPTH);
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
        bulkWaitAll<0>();  // all beta rows are in global memory before the forward sweep reads them back
      }
      __syncwarp();
    }

    // =============================================================================================================
    // sweep 2: forward + fused consumers (ref: HMM.cpp:725-879, 669-692, 1179-1357, 1378-1409)
    // =============================================================================================================
    {
      auto prefetch = [&](const int p) {
        if (lane == 0) {
          const int slot = p % DEPTH;
          mbarExpectTx(&bars[slot], kBetaBytes);
          bulkLoad(betaSlot(slot), slab + static_cast<size_t>(p) * kBetaFloats, kBetaBytes, &bars[slot]);
          mbarExpectTx(&bars[DEPTH + slot], kCoefBytes);
          bulkLoad(const_cast<float*>(coefSlot(slot)), rowBase + static_cast<size_t>(p) * kRowArrays * Spad, kCoefBytes,
                   &bars[DEPTH + slot]);
        }
      };
      for (int p = 0; p < DEPTH && p < len; ++p) {
        prefetch(p);
      }
      CallerState cs;

      // consumers of window position p: v = alpha(p); w = the other (dead) vector, receives q[k] = alpha[k] beta[k]
      auto consume = [&](const int p, const float (&v)[S], float (&w)[S]) {
        const int site = from + p;
        const int slot = p % DEPTH;
        mbarWait(&bars[slot], (betaParity >> slot) & 1u);
        betaParity ^= 1u << slot;
        const float4* B4 = betaSlot(slot);
        float q0 = 0.f, q1 = 0.f, q2 = 0.f, q3 = 0.f, ibdRaw = 0.f;
#pragma unroll
        for (int q = 0; q < SQ; ++q) {
          const float4 b4 = B4[q * 32 + lane];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int k = 4 * q + i;
            if (k < S) {
              w[k] = v[k] * f4(b4, i);
            }
          }
          q0 += w[4 * q];
          if (4 * q + 1 < S) q1 += w[4 * q + 1];
          if (4 * q + 2 < S) q2 += w[4 * q + 2];
          if (4 * q + 3 < S) q3 += w[4 * q + 3];
        }
        const float r = 1.0f / ((q0 + q1) + (q2 + q3));  // ref HMM.cpp:681-685

        if (wantSite) {
          float mean = 0.f, best = 0.f;
          int arg = 0;
#pragma unroll
          for (int k = 0; k < S; ++k) {
            mean = fmaf(w[k], fm.expTimes[k], mean);
            if (best < w[k]) {
              best = w[k];
              arg = k;
            }
          }
          if (laneActive) {
            if (flags & FSMC_SITE_MEAN) {
              args.siteMean[static_cast<size_t>(outRow) * args.siteStride + p] = mean * r;
            }
            if (flags & FSMC_SITE_MAP) {
              args.siteMap[static_cast<size_t>(outRow) * args.siteStride + p] = arg;
            }
          }
        }

        if constexpr (SUM) {
          // posteriors of the tile's 32 pairs -> [state][pair] in the drained beta slot, then lane l adds up states
          // l, l+32, l+64 (reading the pairs rotated by its lane number: conflict-free) and updates the warp's accumulator
          float* stage = reinterpret_cast<float*>(betaSlot(slot));
          const int cls = bits.cls(site);
          const unsigned het = __ballot_sync(kFull, cls == 1), minor = __ballot_sync(kFull, cls == 2);
          const float rr = laneActive ? r : 0.f;
          __syncwarp();  // every lane has read its beta quads
#pragma unroll
          for (int k = 0; k < S; ++k) {
            stage[k * 32 + lane] = w[k] * rr;
          }
          __syncwarp();
          const bool byGenotype = sumPlanes == 3;
#pragma unroll
          for (int j = 0; j < (S + 31) / 32; ++j) {
            const int k = lane + 32 * j;
            if (k < S) {
              float s0 = 0.f, s1 = 0.f, s2 = 0.f;
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                const int src = (i + lane) & 31;
                const float v = stage[k * 32 + src];
                if (byGenotype) {
                  const bool h = (het >> src) & 1u, mn = (minor >> src) & 1u;
                  s0 += (h || mn) ? 0.f : v;
                  s1 += h ? v : 0.f;
                  s2 += mn ? v : 0.f;
                } else {
                  s0 += v;
                }
              }
              float* row = sumMine + static_cast<size_t>(site) * Spad + k;
              row[0] += s0;
              if (byGenotype) {
                row[static_cast<size_t>(m.L) * Spad] += s1;
                row[2 * static_cast<size_t>(m.L) * Spad] += s2;
              }
            }
          }
        }

        const bool inScan = wantSeg && site >= scanFrom && site < scanTo;
        if ((flags & FSMC_SITE_IBD) || inScan) {
          forStatesBelow<S_T>(sT, [&](const int k) { ibdRaw += w[k]; });
          const float ibd = ibdRaw * r;
          if ((flags & FSMC_SITE_IBD) && laneActive) {
            args.siteIbd[static_cast<size_t>(outRow) * args.siteStride + p] = ibd;
          }
          if (inScan) {
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
            const bool ending = changed && cs.level >= 0;  // the run that ended at site-1 is written now
            const bool closing = now >= 0 && site == scanTo - 1;
            float* park = reinterpret_cast<float*>(betaSlot(slot)) + lane;  // this site's drained beta slot: [k][32]
            if (__any_sync(kFull, ending)) {
              __syncwarp();  // every lane has read its beta quads: the slot becomes the parking area (racecheck: WAR)
              if (wantAge) {
                // rare: park the per-state sums (through site-1) for emitSegment
#pragma unroll
                for (int k = 0; k < (ACC ? S : 1); ++k) {
                  park[k * 32] = acc[k];
                }
                __syncwarp();
              }
              if (ending) {
                emitSegment<false>(m, args, pair, cs.start, site - 1, cs.prob, cs.level, park, wantAge);
              }
              __syncwarp();
            }
            if constexpr (ACC) {
              if (wantAge && __any_sync(kFull, now >= 0)) {
                // per-state sums of the current run: restart on a new run, accumulate otherwise
                // (ref: HMM.cpp:1209-1218,1229,1257,1284,1311)
                const float rr = now >= 0 ? r : 0.f;
                const float keep = changed ? 0.f : 1.f;
                forStatesBelow<S_T>(nAcc, [&](const int k) { acc[k] = fmaf(w[k], rr, keep * acc[k]); });
              }
            }
            if (__any_sync(kFull, closing)) {
              __syncwarp();
              if (wantAge) {
#pragma unroll
                for (int k = 0; k < (ACC ? S : 1); ++k) {
                  park[k * 32] = acc[k];
                }
                __syncwarp();
              }
              if (closing) {
                emitSegment<false>(m, args, pair, changed ? site : cs.start, site, changed ? ibd : cs.prob + ibd, now, park,
                                   wantAge);
              }
              __syncwarp();
            }
            if (now >= 0) {
              cs.prob = changed ? ibd : cs.prob + ibd;
              if (changed) {
                cs.start = site;
              }
              if (closing) {
                cs.prob = 0.f;
              }
            } else {
              cs.prob = 0.f;
            }
            cs.level = now;
          }
        }
        __syncwarp();  // both slots of this position are drained (the beta slot doubles as the parking area above)
        if (p + DEPTH < len) {
          prefetch(p + DEPTH);
        }
      };

      // p = 0: alpha(from)[k] = prior[k] * emission  (ref HMM.cpp:736-743)
      {
        const int cls = bits.cls(from);
        mbarWait(&bars[DEPTH], coefParity & 1u);
        coefParity ^= 1u;
        const float4* E = reinterpret_cast<const float4*>(coefSlot(0) + cls * Spad);
#pragma unroll
        for (int q = 0; q < SQ; ++q) {
          const float4 e4 = E[q];
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int k = 4 * q + i;
            if (k < S) {
              a[k] = fm.prior[k] * f4(e4, i);
            }
          }
        }
        consume(0, a, c);
      }
      auto step = [&](const int p, float (&x)[S], float (&y)[S]) {
        const int slot = p % DEPTH;
        const int cls = bits.cls(from + p);
        mbarWait(&bars[DEPTH + slot], (coefParity >> slot) & 1u);
        coefParity ^= 1u << slot;
        const float total = forwardStep<S>(fm.colRatios, x, y, coefSlot(slot), cls);
        if ((p & (RESCALE - 1)) == 0) {
          scaleStates<S>(y, 1.0f / total);
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
    }
    __syncwarp();
  }
}

// out[(plane * S + k) * L + site] = sum over warps of scratch[warp][plane][site][k], warps in ascending order;
// with a weight vector (fsmc_decode_device): out[...] += sum * weight[k] instead
static __global__ void sumScratchReduceKernel(const float* __restrict__ scratch, const int warps, const int planes, const int L,
                                              const int S, const int Spad, float* __restrict__ out,
                                              const float* __restrict__ weight = nullptr)
{
  const long long total = static_cast<long long>(planes) * L * Spad;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int k = static_cast<int>(i % Spad);
    if (k >= S) {
      continue;
    }
    const long long site = (i / Spad) % L;
    const long long plane = i / Spad / L;
    float sum = 0.f;
    for (int w = 0; w < warps; ++w) {
      sum += scratch[static_cast<size_t>(w) * total + i];
    }
    float* o = out + (plane * S + k) * L + site;
    *o = weight ? __fadd_rn(*o, __fmul_rn(sum, weight[k])) : sum;
  }
}

}  // namespace fsmc
