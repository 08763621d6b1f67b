// fll_pair.cu — K4 for large batches: the band-edge FLL (MS/Models/Band-Edge Filter.cs:102-129,185-195) with two lanes
// per stream, 16 streams per warp.
//
// The two-warp kernel (fll_duo.cu) spreads one stream over 8 lanes and two warps to shorten the per-sample recurrence;
// that costs ~44 warp instructions per stream and sample, and from ~4096 streams on the issue slots, not the latency,
// set its time.  This kernel spends ~21 issue slots per stream and sample, so it takes over from 5120 streams (the
// measured crossover is in FllEngine::process_dev).
//   * taps: kernel parameters, copied once to shared memory and read with broadcast LDS.128 (two taps each);
//   * ring of past outputs: shared memory, 2N rows — every sample is written at `pos` and `pos + N`, so the
//     chronological window is the N slots after `pos` with compile-time offsets (no modulo, no index arithmetic);
//   * input / output: staged through shared memory in rounds of 32 samples, coalesced row reads and writes.
// State layout in device memory is the generic one (ring [N][C] + head, (phase, freq)), so calls may alternate between
// this kernel and the others.  sin/cos and the phase wrap are short-range forms (|phase| < 64; the launcher sends a
// caller-set |phase| >= 32 to the two-warp kernel).  Compiled with --fmad=false.
#include "loops.cuh"

namespace qpsk {

namespace {

constexpr int kLaneBlock = 32;            // samples per staged round

// packed (I, Q) arithmetic with every product and sum rounded on its own, as RyuJIT emits them:
//   product  fma.rn.f32x2 with an addend of -0 loaded at run time: fma(x, g, -0) == round(x*g) exactly, and ptxas cannot
//            contract it into the add that follows (it does contract mul.rn.f32x2 + add.rn.f32x2 into one FFMA2);
//   sum      add.rn.f32x2 / sub.rn.f32x2 (FADD2, the subtraction as an operand negation).
// One FFMA2, two FMUL and four FADD2 per tap instead of four FMUL and eight FADD: the same 12 FP32-pipe cycles, 7 issue
// slots instead of 12 — and this kernel runs one warp per scheduler, i.e. it is bound by its own issue stream.
__device__ float2 g_lane_neg_zero2 = {-0.0f, -0.0f};
__device__ __forceinline__ float2 lane_add2(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}
__device__ __forceinline__ float2 lane_sub2(float2 a, float2 b) {
  float2 d;
  asm("sub.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}

template <int N>
struct LaneTaps {
  float i[N], q[N];                       // reversed lower-filter taps (rev[k] = lower[N-1-k])
};

// remainderf(phase, 2 pi) for |phase| < 1e5, as in fll_duo.cu (exact fp64 quotient, exact remainder; a zero keeps the
// sign of phase like Math.IEEERemainder)
__device__ __forceinline__ float lane_wrap_phase(float phase) {
  const double c = (double)kTwoPiF;
  const double pd = (double)phase;
  const double n = rint(pd * (1.0 / c));
  const double r = fma(-n, c, pd);
  return (r == 0.0) ? copysignf(0.f, phase) : (float)r;
}

// ---------------------------------------------------------------------------------------------------------------------
// fll_pair_kernel: TWO lanes per stream, 16 streams per warp.  One lane per stream would leave 512 warps for 592
// warp schedulers at 16384 streams — one in-order warp per scheduler, bound by its own issue stream and every stall in
// it.  Here lane 2s + h of a warp owns the SIMD-lane partials 4h .. 4h+3 of stream s (ComplexDotWindow's eight partial
// sums, FIRFilter.cs:165-192): half the taps per lane, twice the warps (two per scheduler at 16384 streams), and the
// ordered horizontal sum ((((0 + L0) + L1) + ...) + L7) crosses the pair once — lane 2s sums L0..L3, hands the four values
// over with shuffles, lane 2s+1 adds L4..L7 and the scalar tail, and the error goes back with one more shuffle, so both
// lanes carry identical (phase, freq).  Same roundings in the same order as fll_group_kernel (loops.cu); same state layout
// in device memory.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int kPairStreams = 16;
constexpr int kPairPitch = 17;            // float2 row pitch of the staging tiles (odd)
constexpr int kPairRing = 18;             // float2 row pitch of the output ring (see fll_pair_kernel)

// One tap of both band-edge filters on window element v (the four sums of loops.cuh, same roundings): lo += P + D, up += P - D
// with P = a*(vI, vQ), D = ((-b)*vQ, b*vI).
__device__ __forceinline__ void pair_tap(float2 v, float a, float bq, float2 nz, float2& lo, float2& up) {
  const float2 Pp = ffma2(v, make_float2(a, a), nz);
  const float2 Dd = make_float2(__fmul_rn(-bq, v.y), __fmul_rn(bq, v.x));
  lo = lane_add2(lo, lane_add2(Pp, Dd));
  up = lane_add2(up, lane_sub2(Pp, Dd));
}
__device__ __forceinline__ float2 sel2(bool c, float2 a, float2 b) { return make_float2(c ? a.x : b.x, c ? a.y : b.y); }

// Software pipeline (one in-order warp per scheduler has nothing else to hide the recurrence behind): while the chain of
// sample n runs — phase -> sin/cos -> rotate -> newest tap -> error -> phase — the warp accumulates window n+1 over every
// element that is already in the ring (all but out[n] and out[n+1]), in the same basic block, so that ptxas interleaves the
// two streams.  Window n+1's elements N-2 (= out[n]) and N-1 (= out[n+1]) are each the LAST addition of their SIMD-lane
// partial (or the last two tail elements), so adding them late keeps the reference's order of additions.  The loop body
// is branch-free (lane roles, the phase wrap and the clamps are selects) for the same reason.
template <int N>
__global__ void __launch_bounds__(32)
    fll_pair_kernel(const FllParams P, const __grid_constant__ LaneTaps<N> T, float2* ring_g, int* head_g, float2* pf_g, int C,
                    const float2* __restrict__ x, float2* __restrict__ y, long long L, long long ldx, long long ldy) {
  constexpr int nVec = N - (N & 7);
  constexpr int kTail = N & 7;
  static_assert(nVec >= 8 && (kTail == 0 || kTail >= 2), "the two newest elements are both in the last block or both in the tail");
  constexpr bool kNewInVec = kTail == 0;               // N % 8 == 0: elements N-2, N-1 are partials 6, 7 (the odd lane's j = 2, 3)
  // + 2 rows: the odd lane's (unused) look at the slots of elements still to come.  Row pitch 18 float2 = 36 words: the two
  // lanes of a pair read rows four apart (4 * 36 = 144 = 16 mod 32 banks), so the even lanes of a half-warp use banks 0-15
  // and the odd lanes 16-31 — with the natural pitch of 16 they collide on every window load (173 M conflicts per call in ncu)
  __shared__ float2 ring[2 * N + 2][kPairRing];
  __shared__ float2 xin[2][kLaneBlock][kPairPitch];
  __shared__ float2 yout[kLaneBlock][kPairPitch];
  __shared__ __align__(16) float4 tap4[(N + 1) / 2];
  const int lane = threadIdx.x;
  const int st = lane >> 1;
  const bool odd = (lane & 1) != 0;
  const int h = lane & 1;
  for (int k = lane; k < (N + 1) / 2; k += 32)
    tap4[k] = make_float4(T.i[2 * k], T.q[2 * k], (2 * k + 1 < N) ? T.i[2 * k + 1] : 0.f, (2 * k + 1 < N) ? T.q[2 * k + 1] : 0.f);
  const int c0 = blockIdx.x * kPairStreams;
  const int c = c0 + st;
  const bool live = c < C;
  const int cc = live ? c : C - 1;        // idle pairs shadow the last stream (their results are dropped)
  {
    const int head = head_g[cc];
    for (int j = h; j < N; j += 2) {      // the pair shares the copy
      int k = head + j;
      if (k >= N) k -= N;
      const float2 v = ring_g[(long long)k * C + cc];
      ring[j][st] = v;
      ring[j + N][st] = v;
    }
  }
  const int rows = (C - c0 < kPairStreams) ? (C - c0) : kPairStreams;
  auto stage = [&](int buf, long long n0) {            // lane l fetches sample n0 + l of every stream of the CTA (cp.async)
    const int blk = (int)((L - n0 < kLaneBlock) ? (L - n0) : kLaneBlock);
    if (lane < blk) {
#pragma unroll 8
      for (int r = 0; r < kPairStreams; ++r) {
        const int ch = c0 + (r < rows ? r : rows - 1);
        const unsigned dst = (unsigned)__cvta_generic_to_shared(&xin[buf][lane][r]);
        asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(x + (long long)ch * ldx + n0 + lane) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  if (L > 0) stage(0, 0);
  __syncwarp();
  const float2 pf = pf_g[cc];
  float phase = pf.x, freq = pf.y;
  float2 nz;
  asm volatile("ld.volatile.global.v2.f32 {%0, %1}, [%2];" : "=f"(nz.x), "=f"(nz.y) : "l"(&g_lane_neg_zero2));
  // The pair's ODD lane carries the recurrence (its partial sums end with the newest outputs); the even lane runs the same
  // instructions on its own copy of (phase, freq), which nothing reads — no broadcast of the error sits on the chain.
  // sin/cos: the short-range form of the two-warp kernel (sincos_f32arg_rq: |phase| < 64, see FllEngine::process_dev).
  const SinCosF SKF = sincos_f_load_consts();
  int pos = 0;

  // window element i of the window starting at slot `wb`, this lane's share of block b: elements b + 4h + j
  // taps of element i: tap4[i >> 1].{x,y} (even i) / .{z,w} (odd i)
#define PAIR_TAP_OF(i, A, B)                                  \
  const float4 t4_##A = tap4[(i) >> 1];                       \
  const float A = ((i) & 1) ? t4_##A.z : t4_##A.x, B = ((i) & 1) ? t4_##A.w : t4_##A.y;

  // partial sums of the CURRENT window over everything but its newest element (prologue: all N-1 old outputs are in the ring)
  float2 clo[4], cup[4];
  float2 ctail[kTail > 2 ? kTail - 2 : 1];             // old tail elements nVec .. N-3 of the current window
  float2 vprev = ring[N - 1][st];                      // out[n-1]: the newest output so far (slot pos + N - 1 with pos = 0)
  {
    const float2* win = &ring[1 + 4 * h][st];
#pragma unroll
    for (int l = 0; l < 4; ++l) clo[l] = cup[l] = make_float2(0.f, 0.f);
#pragma unroll
    for (int b = 0; b < nVec; b += 8) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (kNewInVec && b == nVec - 8 && j == 3) continue;   // slot of the element still to come (the odd lane's)
        const float2 v = win[(b + j) * kPairRing];
        const float4 t4 = tap4[(b >> 1) + 2 * h + (j >> 1)];
        pair_tap(v, (j & 1) ? t4.z : t4.x, (j & 1) ? t4.w : t4.y, nz, clo[j], cup[j]);
      }
    }
    if (kNewInVec) {
      // the even lane's j = 3 of the last block is element N-5 (old); the odd lane's is the newest, added in the loop
      const float2 v = ring[1 + (nVec - 8) + 3][st];     // element nVec - 5 (even lane's view)
      const float4 t4 = tap4[((nVec - 8) >> 1) + 1];
      float2 l3 = clo[3], u3 = cup[3];
      pair_tap(v, t4.z, t4.w, nz, l3, u3);
      clo[3] = sel2(odd, clo[3], l3);
      cup[3] = sel2(odd, cup[3], u3);
    }
#pragma unroll
    for (int i = nVec; i < N - 2; ++i) ctail[i - nVec] = ring[1 + i][st];
  }

  int buf = 0;
  for (long long n0 = 0; n0 < L; n0 += kLaneBlock, buf ^= 1) {
    const int blk = (int)((L - n0 < kLaneBlock) ? (L - n0) : kLaneBlock);
    if (n0 + kLaneBlock < L) stage(buf ^ 1, n0 + kLaneBlock);         // next round in flight during this one
    else asm volatile("cp.async.commit_group;" ::: "memory");
    asm volatile("cp.async.wait_group 1;" ::: "memory");
    __syncwarp();
    for (int sidx = 0; sidx < blk; ++sidx) {
      const float2 in = xin[buf][sidx][st];
      const int wb = pos + 1;                          // slot of window n's element 0; window n+1 starts one slot later
      // ---- window n+1, elements 0 .. N-3 (slots wb+1 .. wb+N-2: all written in earlier iterations) ----
      float2 nlo[4], nup[4];
#pragma unroll
      for (int l = 0; l < 4; ++l) nlo[l] = nup[l] = make_float2(0.f, 0.f);
      const float2* win1 = &ring[wb + 1 + 4 * h][st];
      float2 vE = make_float2(0.f, 0.f);               // even lane's element N-5 of window n+1 (slot shared with the odd lane's N-1)
      float2 vD = make_float2(0.f, 0.f);               // even lane's element N-6 (odd lane: N-2 = out[n], not in the ring yet)
#pragma unroll
      for (int b = 0; b < nVec; b += 8) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (kNewInVec && b == nVec - 8 && j >= 2) {  // the odd lane's elements N-2 / N-1: deferred for BOTH lanes
            const float2 v = win1[(b + j) * kPairRing];   // (the even lane's value is its real, old element; the odd lane's is stale)
            if (j == 2) vD = v; else vE = v;
            continue;
          }
          const float2 v = win1[(b + j) * kPairRing];
          const float4 t4 = tap4[(b >> 1) + 2 * h + (j >> 1)];
          pair_tap(v, (j & 1) ? t4.z : t4.x, (j & 1) ? t4.w : t4.y, nz, nlo[j], nup[j]);
        }
      }
      float2 ntail[kTail > 2 ? kTail - 2 : 1];
#pragma unroll
      for (int i = nVec; i < N - 2; ++i) ntail[i - nVec] = ring[wb + 1 + i][st];
      // ---- chain of sample n ----
      // MathF.Cos/Sin(phase) :108-109 and the rotation :111-112 with phase = r + q*pi/2 and the exact factor j^q applied to
      // the input sample while the polynomials run: out = (in * j^q) * (cos r + j sin r) — the same two products per
      // component as in.x*cos - in.y*sin / in.x*sin + in.y*cos (signs are exact, a + b == b + a); see fll_duo.cu
      float sr, cr;
      unsigned q;
      sincos_f32arg_rq((double)phase, SKF, &sr, &cr, &q);
      const bool qodd = (q & 1u) != 0;
      const unsigned fx = ((q + 1u) & 2u) << 30;       // sign of the first component: quadrants 1, 2
      const unsigned fy = (q & 2u) << 30;              // sign of the second: quadrants 2, 3
      const float ax = __uint_as_float(__float_as_uint(qodd ? in.y : in.x) ^ fx);
      const float ay = __uint_as_float(__float_as_uint(qodd ? in.x : in.y) ^ fy);
      const float oI = ax * cr - ay * sr;
      const float oQ = ax * sr + ay * cr;
      // the odd lane's output is the stream's; the even lane needs it only where it shares the odd lane's instructions
      const float2 vnew = make_float2(oI, oQ);
      if (kNewInVec) {
        // window n: its last element (N-1 = out[n]) closes the odd lane's partial 3; the even lane's partial 3 is complete
        const float4 t4 = tap4[((nVec - 8) >> 1) + 2 * 1 + 1];        // taps N-2, N-1 of the odd lane
        float2 l3 = clo[3], u3 = cup[3];
        pair_tap(vnew, t4.z, t4.w, nz, l3, u3);
        clo[3] = sel2(odd, l3, clo[3]);
        cup[3] = sel2(odd, u3, cup[3]);
      }
      // lanes 0..3 summed by the even lane, handed over, lanes 4..7 added by the odd lane (:176-180): both lanes run both
      // passes (no divergence), each keeps the one that is its own
      float2 sLo = make_float2(0.f, 0.f), sUp = make_float2(0.f, 0.f);
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        sLo = lane_add2(sLo, clo[l]);
        sUp = lane_add2(sUp, cup[l]);
      }
      float2 aLo = make_float2(__shfl_xor_sync(0xffffffffu, sLo.x, 1), __shfl_xor_sync(0xffffffffu, sLo.y, 1));
      float2 aUp = make_float2(__shfl_xor_sync(0xffffffffu, sUp.x, 1), __shfl_xor_sync(0xffffffffu, sUp.y, 1));
#pragma unroll
      for (int l = 0; l < 4; ++l) {                    // meaningful on the odd lane: (even lane's sum + L4) + L5 ...
        aLo = lane_add2(aLo, clo[l]);
        aUp = lane_add2(aUp, cup[l]);
      }
      if (!kNewInVec) {                                // scalar tail (:183-192): old elements, then out[n-1], then out[n]
#pragma unroll
        for (int i = nVec; i < N - 2; ++i) {
          PAIR_TAP_OF(i, ta, tb)
          pair_tap(ctail[i - nVec], ta, tb, nz, aLo, aUp);
        }
        {
          PAIR_TAP_OF(N - 2, ta, tb)
          pair_tap(vprev, ta, tb, nz, aLo, aUp);
        }
        {
          PAIR_TAP_OF(N - 1, ta, tb)
          pair_tap(vnew, ta, tb, nz, aLo, aUp);
        }
      }
      const float powUpper = aUp.x * aUp.x + aUp.y * aUp.y;            // :118
      const float powLower = aLo.x * aLo.x + aLo.y * aLo.y;            // :119
      const float error = powLower - powUpper;                         // :121 (the odd lane's is the stream's)
      freq += P.beta * error;                            // :124
      const float p1 = phase + (freq + P.alpha * error); // :125
      const float pw = lane_wrap_phase(p1);
      phase = (p1 > kTwoPiF || p1 < -kTwoPiF) ? pw : p1; // :185-189
      freq = (freq > P.max_freq) ? P.max_freq : ((freq < P.min_freq) ? P.min_freq : freq);   // :191-195
      // ---- window n+1 becomes the current one: out[n] is its element N-2 ----
      if (kNewInVec) {
        // the odd lane's j = 2 (element N-2 = out[n]); the even lane's j = 2, 3 are its old elements N-6, N-5 (vD, vE)
        const float4 t4 = tap4[((nVec - 8) >> 1) + 2 * h + 1];
        pair_tap(sel2(odd, vnew, vD), t4.x, t4.y, nz, nlo[2], nup[2]);
        float2 l3 = nlo[3], u3 = nup[3];
        pair_tap(vE, t4.z, t4.w, nz, l3, u3);
        nlo[3] = sel2(odd, nlo[3], l3);
        nup[3] = sel2(odd, nup[3], u3);
      }
#pragma unroll
      for (int l = 0; l < 4; ++l) {
        clo[l] = nlo[l];
        cup[l] = nup[l];
      }
#pragma unroll
      for (int i = 0; i < (kTail > 2 ? kTail - 2 : 1); ++i) ctail[i] = ntail[i];
      vprev = vnew;
      if (odd) {
        yout[sidx][st] = vnew;
        ring[pos][st] = vnew;                          // over the oldest sample, and its mirror
        ring[pos + N][st] = vnew;
      }
      pos = (pos + 1 == N) ? 0 : pos + 1;
      __syncwarp();                                    // the next iteration's window loads see both copies
    }
    if (lane < blk) {                     // flush: lane l writes sample n0 + l of every live stream
#pragma unroll 8
      for (int r = 0; r < kPairStreams; ++r)
        if (r < rows) y[(long long)(c0 + r) * ldy + n0 + lane] = yout[lane][r];
    }
    __syncwarp();
  }
#undef PAIR_TAP_OF
  if (live) {
    for (int j = h; j < N; j += 2) ring_g[(long long)j * C + c] = ring[pos + j][st];   // oldest first from slot `pos`
    if (odd) {
      head_g[c] = 0;
      pf_g[c] = make_float2(phase, freq);
    }
  }
}

template <int N>
int fll_pair_launch_n(const FllParams& P, const std::vector<float>& lower, float2* ring, int* head, float2* pf, int C,
                      const float2* x, float2* y, long long L, long long ldx, long long ldy, cudaStream_t s) {
  LaneTaps<N> T;
  for (int k = 0; k < N; ++k) {
    T.i[k] = lower[2 * (size_t)(N - 1 - k)];
    T.q[k] = lower[2 * (size_t)(N - 1 - k) + 1];
  }
  fll_pair_kernel<N><<<(C + kPairStreams - 1) / kPairStreams, 32, 0, s>>>(P, T, ring, head, pf, C, x, y, L, ldx, ldy);
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}

}  // namespace

bool fll_pair_supported(int n_taps) { return n_taps == 40 || n_taps == 10; }

int fll_pair_launch(const FllParams& P, const std::vector<float>& lower, float2* ring, int* head, float2* pf, int C,
                    const float2* x, float2* y, long long L, long long ldx, long long ldy, cudaStream_t s) {
  switch (P.n_taps) {
    case 40: return fll_pair_launch_n<40>(P, lower, ring, head, pf, C, x, y, L, ldx, ldy, s);   // QPSKDeModulator.cs:35
    case 10: return fll_pair_launch_n<10>(P, lower, ring, head, pf, C, x, y, L, ldx, ldy, s);   // testFullDemodChain.cs:24
    default: return QPSK_ERR_UNSUPPORTED;
  }
}

}  // namespace qpsk
