// fll_duo.cu — K4, the band-edge FLL (MS/Models/Band-Edge Filter.cs:102-129,185-195) for N = 8*K + TAIL taps,
// 8 <= N <= 55: two warps per four streams, the per-sample recurrence alone on one of them.
//
// Why two warps.  With a few thousand streams there is about one FLL warp per warp scheduler, and a lone warp
// issues in order: every instruction that is not on the loop-carried chain
//      phase -> sin/cos -> rotate -> newest tap term -> |lo|^2-|up|^2 -> freq -> phase
// still delays it.  So the work is split by what it depends on:
//   * CHAIN warp (8 lanes per stream = the 8 SIMD lanes of the reference's Vector<float> dot product,
//     FIRFilter.cs:165-180): sin/cos, rotation, and only the terms that involve the newest output out[n];
//   * SIDE warp (same lane <-> (stream, SIMD lane) mapping): everything that depends only on outputs at least 8
//     samples old — the first K-1 elements of every lane partial — plus all global I/O (input prefetch, output
//     flush, state load/store).  It runs one batch (4 samples) ahead and hands results over through shared memory
//     with mbarriers; its latencies never touch the chain.
//
// Order of additions (bit-identical to ComplexDotWindow, FIRFilter.cs:165-192):
//   window n, SIMD lane l:   L_l(n) = (((0 + e_{l}) + e_{l+8}) + ...) + e_{l+8(K-1)},  e_i = tap_rev[i] (x) out[n-(N-1)+i]
//   horizontal sum:          P_7(n) = ((((((0 + L_0) + L_1) + ...) + L_6) + L_7
//   scalar tail (:183-192):  acc(n) = (P_7(n) + e_{8K}) + ... + e_{N-1}                      (TAIL = N % 8 elements)
// The last vector element of lane l in window m is out[m-TAIL-7+l], so at step n (out[n] just computed) GPU lane g
// finishes L_g of window m = n+TAIL+7-g and extends that window's prefix  P_g(m) = P_{g-1}(m) + L_g(m)  with the value
// lane g-1 produced one step earlier (handed over through shared memory, read before the rotation is known): the
// horizontal sum is a systolic pipeline across the 8 lanes and across time, and nothing but register arithmetic
// follows the rotation.  TAIL == 0: every lane also plays lane 7's role for the current window (acc(n) = P_6(n) +
// L_7(n)), redundantly, so the loop state (phase, freq) stays uniform in the group without a broadcast on the chain.
// TAIL > 0: the tail elements are TAIL more pipeline stages, T_j = T_{j-1} + e_{8K+j}, that every lane runs in registers
// from lane 7's prefix of the previous step; the last stage closes window n.
#include "loops.cuh"

#include <type_traits>

namespace qpsk {

namespace {

constexpr int kDuoStreams = 4;            // streams per warp pair
// ring slots per stream: a power of two >= N + 16 (64 up to 48 taps, 128 up to 55); rows are RING + 2 float2 long
// (16-byte aligned, the four streams' rows 4 banks apart)
constexpr int kDuoBatch = 4;              // samples per hand-over
constexpr int kDuoSuper = 16;             // samples per global-memory transaction and stream
constexpr int kDuoXStride = kDuoSuper + 2;

__device__ __forceinline__ uint32_t duo_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void duo_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(duo_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void duo_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(duo_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void duo_mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(duo_smem_u32(bar)), "r"(parity)
        : "memory");
  } while (!ok);
}

// shared-memory accesses by 32-bit address + compile-time offset.  The chain warp's addresses are pinned in
// registers (duo_pin): left to itself ptxas recomputes each of them from %tid inside every step (~12 integer
// instructions per sample on a warp whose issue slots are the bottleneck).
__device__ __forceinline__ uint32_t duo_pin(uint32_t v) {
  uint32_t r;
  asm volatile("mov.u32 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}
template <int OFF>
__device__ __forceinline__ float4 duo_lds128(uint32_t a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4+%5];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a), "n"(OFF) : "memory");
  return v;
}
template <int OFF>
__device__ __forceinline__ float2 duo_lds64(uint32_t a) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2+%3];" : "=f"(v.x), "=f"(v.y) : "r"(a), "n"(OFF) : "memory");
  return v;
}
template <int OFF>
__device__ __forceinline__ void duo_sts128(uint32_t a, float4 v) {
  asm volatile("st.shared.v4.f32 [%0+%1], {%2, %3, %4, %5};" ::"r"(a), "n"(OFF), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
template <int OFF>
__device__ __forceinline__ void duo_sts64(uint32_t a, float2 v) {
  asm volatile("st.shared.v2.f32 [%0+%1], {%2, %3};" ::"r"(a), "n"(OFF), "f"(v.x), "f"(v.y) : "memory");
}

// side-warp wait: try_wait with a suspend-time hint, so the waiting warp sleeps in hardware until the phase completes
// (or ~2 us pass) instead of spinning through the issue slots of a chain warp on the same scheduler
__device__ __forceinline__ void duo_mbar_wait_sleepy(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(duo_smem_u32(bar)), "r"(parity), "r"(2000u)
        : "memory");
  } while (!ok);
}
__device__ __forceinline__ bool duo_mbar_test(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(duo_smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}

template <int RING>
struct DuoSmem {
  float2 ring[kDuoStreams * (RING + 2)];                // past outputs, slot = sample index & (RING - 1)
  float4 lp[2][kDuoBatch][32];                          // per batch parity: stale lane partials (loI, loQ, upI, upQ)
  float2 xq[2][kDuoStreams * kDuoXStride];              // input samples, one super-batch per slot
  uint64_t lp_full[2];                                  // side -> chain: batch's partials (and inputs) are in place
  uint64_t out_full[2];                                 // chain -> side: batch's outputs are in the ring
  float consts[4];                                      // beta, alpha, max_freq, min_freq
  float4 exch[kDuoStreams * 9];                         // chain warp: lane prefixes of the previous step
  uint32_t opaque[32];                                  // chain warp: see a_ex_out
};

// the four sums of one window element: (loI, loQ, upI, upQ) += tap (x) v, the reference's products and order
// (Band-Edge Filter.cs:115-116 through FIRFilter.cs:165-192; upper = conj(lower) shares the four products)
__device__ __forceinline__ void duo_acc(float4& a, float ta, float tb, float vx, float vy) {
  const float p1 = ta * vx, p2 = tb * vy, p3 = ta * vy, p4 = tb * vx;
  a.x = a.x + (p1 - p2);
  a.y = a.y + (p3 + p4);
  a.z = a.z + (p1 + p2);
  a.w = a.w + (p3 - p4);
}

// The rare wrap phase = IEEERemainder(phase, 2*pi_f32) (Band-Edge Filter.cs:185-189) in five instructions instead of
// the inlined remainderf (~80, four copies per batch).  With c = fl32(2*pi) = 13176795 * 2^-21 (odd mantissa) and
// |phase| > c an fp32 phase is an even multiple of 2^-22 while every tie point (m + 1/2) c is an odd one, so
// phase / c stays >= 3.8e-8 away from a tie and n = rint(phase * (1/c)) in fp64 is the exact quotient for
// |n| < 2^20; phase - n*c is then exact in fp64 and (IEEE remainders are representable) in fp32.  A zero result
// keeps the sign of phase, like remainderf / Math.IEEERemainder.  Checked against remainderf on the host
// (tools/sincos_check.cpp).  The launcher keeps |phase| < 1e5 for this kernel.
__device__ __forceinline__ float duo_wrap_phase(float phase, double pd) {
  const double c = (double)kTwoPiF;
  const double n = rint(pd * (1.0 / c));
  const double r = fma(-n, c, pd);
  return (r == 0.0) ? copysignf(0.f, phase) : (float)r;
}

template <int K, int TAIL, int PAIRS>
__global__ void __launch_bounds__(64 * PAIRS)
    fll_duo_kernel(const FllParams P, const float* __restrict__ taps, float2* ring_g, int* head_g, float2* pf_g, int C,
                   const float2* __restrict__ x, float2* __restrict__ y, long long L, long long ldx, long long ldy) {
  constexpr int N = 8 * K + TAIL;                           // 8-lane vector part + scalar tail (FIRFilter.cs:165-192)
  constexpr int kDuoRing = (N + 16 <= 64) ? 64 : 128;
  constexpr int kDuoRingStride = kDuoRing + 2;
  // warm-up batches (even, so that batch parity stays b & 1): the prefix of window 0 starts TAIL + 7 steps early
  constexpr int WB = (TAIL <= 1) ? 2 : 4;
  static_assert(4 * WB >= TAIL + 7, "warm-up too short");
  __shared__ __align__(16) DuoSmem<kDuoRing> smem[PAIRS];
  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // warps 0..PAIRS-1 are the chain warps, PAIRS..2*PAIRS-1 their side warps: with PAIRS = 4 (warps go to the four
  // schedulers round robin) every scheduler holds one chain warp and one side warp of the CTA
  const int pair = warp % PAIRS;
  const bool is_chain = warp < PAIRS;
  DuoSmem<kDuoRing>& S = smem[pair];
  const int sl = lane >> 3;                                 // stream slot in the pair
  const int g = lane & 7;                                   // reference SIMD lane
  const int c_raw = (blockIdx.x * PAIRS + pair) * kDuoStreams + sl;
  const bool live = c_raw < C;
  const int c = live ? c_raw : C - 1;                       // idle groups shadow the last stream, no stores
  float2* myring = S.ring + sl * kDuoRingStride;
  const long long nB = (L + kDuoBatch - 1) / kDuoBatch;     // batches of real samples; batches -WB..-1 are the warm-up

  if (lane == 0 && is_chain) {
    duo_mbar_init(&S.lp_full[0], 1);
    duo_mbar_init(&S.lp_full[1], 1);
    duo_mbar_init(&S.out_full[0], 1);
    duo_mbar_init(&S.out_full[1], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  if (!is_chain) {
    // =========================================== SIDE warp ===========================================
    float ta[K > 1 ? K - 1 : 1], tb[K > 1 ? K - 1 : 1];
#pragma unroll
    for (int k = 0; k < K - 1; ++k) {
      ta[k] = taps[g + 8 * k];
      tb[k] = taps[N + g + 8 * k];
    }
    // history: chronological element j (oldest first) of the saved ring goes to sample index j - N
    {
      const int head = head_g[c];
      for (int j = g; j < N; j += 8) {
        int slot = head + j;
        if (slot >= N) slot -= N;
        myring[(j - N) & (kDuoRing - 1)] = ring_g[(long long)slot * C + c];
      }
    }
    __syncwarp();
    const float2* xc = x + (long long)c * ldx;
    float2* yc = y + (long long)c * ldy;
    // input prefetch registers: super-batch sb holds samples [16 sb, 16 sb + 16); lane g loads g and g + 8
    float2 xr0 = make_float2(0.f, 0.f), xr1 = make_float2(0.f, 0.f);
    if (g < L) xr0 = xc[g];
    if (g + 8 < L) xr1 = xc[g + 8];
    long long flushed = 0;
    for (long long b = -WB; b < nB; ++b) {
      // chain finished batch b-2 (its phase index on barrier b & 1 is (b - 2 + WB) / 2)
      if (b >= 2 - WB) duo_mbar_wait_sleepy(&S.out_full[b & 1], (uint32_t)(((b - 2 + WB) >> 1) & 1));
      if (b >= 0 && (b & 3) == 0) {
        const long long sb = b >> 2;
        float2* q = S.xq[sb & 1] + sl * kDuoXStride;
        q[g] = xr0;
        q[g + 8] = xr1;
        const long long i0 = (sb + 1) * kDuoSuper + g;
        if (i0 < L) xr0 = xc[i0];
        if (i0 + 8 < L) xr1 = xc[i0 + 8];
      }
      if ((b & 3) == 1 && b >= 5) {
        // outputs through sample 4(b-2)+3 = 16 sb - 1 are final: flush [16(sb-1), 16 sb)
        const long long f0 = ((b >> 2) - 1) * kDuoSuper;
        if (live) {
          yc[f0 + g] = myring[(int)(f0 + g) & (kDuoRing - 1)];
          yc[f0 + g + 8] = myring[(int)(f0 + g + 8) & (kDuoRing - 1)];
        }
        flushed = f0 + kDuoSuper;
      }
      // stale partials for the steps n = 4b + j: elements k = 0..K-2 of this lane's window, out[n - 8(K-1-k)]
      float4 acc[kDuoBatch];
#pragma unroll
      for (int j = 0; j < kDuoBatch; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < K - 1; ++k) {
        const int s0 = (int)(4 * b - 8 * (K - 1 - k)) & (kDuoRing - 1);        // multiple of 4
        const float4 v01 = *reinterpret_cast<const float4*>(myring + s0);
        const float4 v23 = *reinterpret_cast<const float4*>(myring + s0 + 2);
        duo_acc(acc[0], ta[k], tb[k], v01.x, v01.y);
        duo_acc(acc[1], ta[k], tb[k], v01.z, v01.w);
        duo_acc(acc[2], ta[k], tb[k], v23.x, v23.y);
        duo_acc(acc[3], ta[k], tb[k], v23.z, v23.w);
      }
#pragma unroll
      for (int j = 0; j < kDuoBatch; ++j) S.lp[b & 1][j][lane] = acc[j];
      __syncwarp();
      if (lane == 0) duo_mbar_arrive(&S.lp_full[b & 1]);
    }
    // the chain's last batch
    {
      const long long bl = nB - 1;
      duo_mbar_wait_sleepy(&S.out_full[bl & 1], (uint32_t)(((bl + WB) >> 1) & 1));
    }
    if (live) {
      for (long long i = flushed + g; i < L; i += 8) yc[i] = myring[(int)i & (kDuoRing - 1)];
      // state: chronological ring, oldest at slot 0 = where the next output goes
      for (int j = g; j < N; j += 8) ring_g[(long long)j * C + c] = myring[(int)(L - N + j) & (kDuoRing - 1)];
      if (g == 0) head_g[c] = 0;
    }
    return;
  }

  // =========================================== CHAIN warp ===========================================
  const float tA = taps[g + 8 * (K - 1)], tB = taps[N + g + 8 * (K - 1)];   // tap of this lane's newest element
  const float nA = taps[8 * K - 1], nBq = taps[N + 8 * K - 1];                // lane 7's newest element (TAIL == 0: out[n] in window n)
  // scalar tail (TAIL > 0): window m adds  tail_j (x) out[m-TAIL+1+j], j = 0..TAIL-1, after the lane sum.  At step n stage j
  // extends window n+TAIL-1-j with out[n]: T_j = T_{j-1}(previous step) + tail_j (x) out[n], T_{-1} = lane 7's prefix of
  // the previous step; every lane runs all stages (register arithmetic only), the last one closes window n.
  float tTa[TAIL > 0 ? TAIL : 1], tTb[TAIL > 0 ? TAIL : 1];
  float4 Tt[TAIL > 0 ? TAIL : 1];
#pragma unroll
  for (int j = 0; j < (TAIL > 0 ? TAIL : 1); ++j) {
    tTa[j] = (TAIL > 0) ? taps[8 * K + j] : 0.f;
    tTb[j] = (TAIL > 0) ? taps[N + 8 * K + j] : 0.f;
    Tt[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  const SinCosF SK = sincos_f_load_consts();
  const float2 pf = pf_g[c];
  float phase = pf.x, freq = pf.y;
  double pd = (double)phase;
  // loop constants in registers: ptxas re-issues constant-bank loads inside the step (a dependent LDC each), so they
  // take a detour through shared memory with a volatile load it cannot rematerialise
  float beta, alpha, max_freq, min_freq;
  {
    if (lane == 0) {
      S.consts[0] = P.beta;
      S.consts[1] = P.alpha;
      S.consts[2] = P.max_freq;
      S.consts[3] = P.min_freq;
    }
    __syncwarp();
    const uint32_t a = duo_smem_u32(S.consts);
    asm volatile("ld.volatile.shared.f32 %0, [%1];" : "=f"(beta) : "r"(a));
    asm volatile("ld.volatile.shared.f32 %0, [%1+4];" : "=f"(alpha) : "r"(a));
    asm volatile("ld.volatile.shared.f32 %0, [%1+8];" : "=f"(max_freq) : "r"(a));
    asm volatile("ld.volatile.shared.f32 %0, [%1+12];" : "=f"(min_freq) : "r"(a));
  }
  // Prefix hand-over between neighbouring lanes: lane g stores its new prefix in slot g+1 of its stream's row and
  // reads slot g (lane g-1's value of the previous step; slot 0 stays zero: "aLo = 0; aLo += lane 0", :176-180) and
  // slot 7 (lane 6's: P_6 of the current window).  One STS.128 + two LDS.128 per step instead of eight SHFL.
  float4* const ex_row = S.exch + sl * 9;
  if (g == 0) ex_row[0] = make_float4(0.f, 0.f, 0.f, 0.f);
  ex_row[g + 1] = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncwarp();
  const uint32_t a_ex = duo_pin(duo_smem_u32(ex_row + g));          // lane g-1's prefix
  // this lane's slot: the address takes a round trip through shared memory (volatile load), so ptxas cannot relate
  // it to a_ex and has to keep every prefix store ahead of the following loads (see step)
  uint32_t a_ex_out;
  {
    S.opaque[lane] = duo_smem_u32(ex_row + g + 1);
    __syncwarp();
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(a_ex_out) : "r"(duo_smem_u32(&S.opaque[lane])));
  }
  const uint32_t a_p6 = duo_pin(duo_smem_u32(ex_row + (TAIL == 0 ? 7 : 8)));   // lane 6's prefix (TAIL > 0: lane 7's)
  const uint32_t a_lp0 = duo_pin(duo_smem_u32(&S.lp[0][0][lane]));
  const uint32_t a_l70 = duo_pin(duo_smem_u32(&S.lp[0][0][sl * 8 + 7]));
  const uint32_t a_xq0 = duo_pin(duo_smem_u32(S.xq[0] + sl * kDuoXStride));
  const uint32_t a_ring0 = duo_pin(duo_smem_u32(myring));
  const bool writer = duo_pin((uint32_t)(g == 7)) != 0;
  constexpr int kLpBatchBytes = kDuoBatch * 32 * 16;                // lp[1] - lp[0]
  constexpr int kXqSlotBytes = kDuoStreams * kDuoXStride * 8;       // xq[1] - xq[0]
  // one sample step; WARM: warm-up (the output is read back from the ring, no loop update).  Every shared-memory
  // address is a per-batch base plus a compile-time offset.
  auto step = [&](auto warm_tag, auto j_tag, uint32_t a_lp, uint32_t a_l7, uint32_t a_xq, uint32_t a_rn) {
    constexpr bool WARM = decltype(warm_tag)::value;
    constexpr int J = decltype(j_tag)::value;
    // No __syncwarp between a step's prefix store and the next step's loads (it costs ~55 cycles per sample here).
    // What it would guarantee holds anyway: the warp is converged (the only branch of a step reconverges before the
    // store) and one warp's shared-memory accesses are performed in issue order; the store and load addresses sit in
    // separately pinned registers, so ptxas cannot prove them disjoint and keeps the store first.
    // known before the rotation: stale partials, previous-step prefixes of the neighbours
    const float4 lpo = duo_lds128<J * 512>(a_lp);
    const float4 Pin = duo_lds128<0>(a_ex);
    float oI, oQ;
    float4 P6, L7;
    if (WARM) {
      const float2 o = duo_lds64<J * 8>(a_rn);               // outputs of earlier calls
      oI = o.x;
      oQ = o.y;
    } else {
      P6 = duo_lds128<0>(a_p6);
      if (TAIL == 0) L7 = duo_lds128<J * 512>(a_l7);
      const float2 in = duo_lds64<J * 8>(a_xq);
      // MathF.Cos/Sin(phase) :108-109 and the rotation :111-112, with phase = r + q*pi/2 and the exact factor j^q
      // applied to the input sample while the polynomials run:  out = (in * j^q) * (cos r + j sin r).  Same two
      // products per component as in.x*cos - in.y*sin / in.x*sin + in.y*cos (signs are exact, a + b == b + a).
      float sr, cr;
      unsigned q;
      sincos_f32arg_rq(pd, SK, &sr, &cr, &q);
      const bool odd = (q & 1u) != 0;
      const unsigned fx = ((q + 1u) & 2u) << 30;             // sign of the first component: quadrants 1, 2
      const unsigned fy = (q & 2u) << 30;                    // sign of the second: quadrants 2, 3
      const float ax = __uint_as_float(__float_as_uint(odd ? in.y : in.x) ^ fx);
      const float ay = __uint_as_float(__float_as_uint(odd ? in.x : in.y) ^ fy);
      oI = ax * cr - ay * sr;
      oQ = ax * sr + ay * cr;
    }
    // this lane's newest element completes L_g of window n+7-g; extend that window's prefix
    float4 Lg = lpo;
    duo_acc(Lg, tA, tB, oI, oQ);
    float4 Pn;
    Pn.x = Pin.x + Lg.x;
    Pn.y = Pin.y + Lg.y;
    Pn.z = Pin.z + Lg.z;
    Pn.w = Pin.w + Lg.w;
    float aLoI = 0.f, aLoQ = 0.f, aUpI = 0.f, aUpQ = 0.f;
    if (TAIL > 0) {
      // tail stages, newest window last; warm-up steps run them too (they fill the pipeline)
      float4 P7;
      if constexpr (WARM) P7 = duo_lds128<0>(a_p6);
      else P7 = P6;
#pragma unroll
      for (int j = TAIL - 1; j >= 1; --j) {
        float4 v = Tt[j - 1];
        duo_acc(v, tTa[j], tTb[j], oI, oQ);
        Tt[j] = v;
      }
      float4 v0 = P7;
      duo_acc(v0, tTa[0], tTb[0], oI, oQ);
      Tt[0] = v0;
      aLoI = Tt[TAIL - 1].x; aLoQ = Tt[TAIL - 1].y; aUpI = Tt[TAIL - 1].z; aUpQ = Tt[TAIL - 1].w;
    }
    if (!WARM) {
      if (TAIL == 0) {
        // lane 7's role for the current window, on every lane: acc = P_6(n) + L_7(n)
        duo_acc(L7, nA, nBq, oI, oQ);
        aLoI = P6.x + L7.x; aLoQ = P6.y + L7.y; aUpI = P6.z + L7.z; aUpQ = P6.w + L7.w;
      }
      const float powUpper = aUpI * aUpI + aUpQ * aUpQ;      // :118
      const float powLower = aLoI * aLoI + aLoQ * aLoQ;      // :119
      const float error = powLower - powUpper;               // :121
      freq += beta * error;                                  // :124
      phase += freq + alpha * error;                         // :125
      // converted before the wrap test resolves (the wrap is rare); volatile so the two conversions are not merged
      // into one after the branch
      asm volatile("cvt.f64.f32 %0, %1;" : "=d"(pd) : "f"(phase));
      if (writer) duo_sts64<J * 8>(a_rn, make_float2(oI, oQ));
      if (phase > kTwoPiF || phase < -kTwoPiF) {             // :185-189
        phase = duo_wrap_phase(phase, pd);
        asm volatile("cvt.f64.f32 %0, %1;" : "=d"(pd) : "f"(phase));
      }
      freq = (freq > max_freq) ? max_freq : ((freq < min_freq) ? min_freq : freq);   // :191-195
    }
    duo_sts128<0>(a_ex_out, Pn);
  };
  auto batch_done = [&](long long b) {
    __syncwarp();
    if (lane == 0) duo_mbar_arrive(&S.out_full[b & 1]);
  };
  auto batch_wait = [&](long long b) { duo_mbar_wait(&S.lp_full[b & 1], (uint32_t)(((b + WB) >> 1) & 1)); };
  // non-blocking probe of a later batch's barrier, issued mid-batch so that its latency hides under the chain
  auto batch_probe = [&](long long b) { return duo_mbar_test(&S.lp_full[b & 1], (uint32_t)(((b + WB) >> 1) & 1)); };
  bool ready = false;
  using J0 = std::integral_constant<int, 0>;
  using J1 = std::integral_constant<int, 1>;
  using J2 = std::integral_constant<int, 2>;
  using J3 = std::integral_constant<int, 3>;
  auto batch = [&](auto warm_tag, long long b, int ns) {
    if (!ready) batch_wait(b);
    const uint32_t par = (uint32_t)(b & 1);
    const uint32_t a_lp = duo_pin(a_lp0 + par * kLpBatchBytes), a_l7 = duo_pin(a_l70 + par * kLpBatchBytes);
    const uint32_t a_xq = duo_pin(a_xq0 + (uint32_t)((b >> 2) & 1) * kXqSlotBytes + (uint32_t)(b & 3) * (kDuoBatch * 8));
    const uint32_t a_rn = duo_pin(a_ring0 + ((uint32_t)(4 * b) & (kDuoRing - 1)) * 8);
    step(warm_tag, J0{}, a_lp, a_l7, a_xq, a_rn);
    if (ns > 1) step(warm_tag, J1{}, a_lp, a_l7, a_xq, a_rn);
    ready = batch_probe(b + 1);                              // (a barrier never used again just reads "not ready")
    if (ns > 2) step(warm_tag, J2{}, a_lp, a_l7, a_xq, a_rn);
    if (ns > 3) step(warm_tag, J3{}, a_lp, a_l7, a_xq, a_rn);
    batch_done(b);
  };
  // warm-up: fills the prefix (and tail) pipeline from the outputs of earlier calls (steps -4*WB..-1)
  for (long long b = -WB; b < 0; ++b) batch(std::true_type{}, b, kDuoBatch);
  const long long nFull = L / kDuoBatch;
  for (long long b = 0; b < nFull; ++b) batch(std::false_type{}, b, kDuoBatch);
  if (nFull < nB) batch(std::false_type{}, nFull, (int)(L - 4 * nFull));
  if (live && g == 0) pf_g[c] = make_float2(phase, freq);
}

template <int K, int PAIRS>
int launch_duo_tail(int tail, const FllParams& P, const float* taps, float2* ring, int* head, float2* pf, int C, const float2* x,
                    float2* y, long long L, long long ldx, long long ldy, cudaStream_t s) {
  const int per_cta = PAIRS * kDuoStreams;
  const int blocks = (C + per_cta - 1) / per_cta;
  switch (tail) {
#define QPSK_DUO_CASE(TT) \
  case TT: fll_duo_kernel<K, TT, PAIRS><<<blocks, 64 * PAIRS, 0, s>>>(P, taps, ring, head, pf, C, x, y, L, ldx, ldy); break;
    QPSK_DUO_CASE(0) QPSK_DUO_CASE(1) QPSK_DUO_CASE(2) QPSK_DUO_CASE(3) QPSK_DUO_CASE(4) QPSK_DUO_CASE(5) QPSK_DUO_CASE(6)
    QPSK_DUO_CASE(7)
#undef QPSK_DUO_CASE
    default: return QPSK_ERR_UNSUPPORTED;
  }
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}
template <int PAIRS>
int launch_duo(int n_taps, const FllParams& P, const float* taps, float2* ring, int* head, float2* pf, int C, const float2* x,
               float2* y, long long L, long long ldx, long long ldy, cudaStream_t s) {
  const int tail = n_taps & 7;
  switch (n_taps >> 3) {
    case 1: return launch_duo_tail<1, PAIRS>(tail, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
    case 2: return launch_duo_tail<2, PAIRS>(tail, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
    case 3: return launch_duo_tail<3, PAIRS>(tail, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
    case 4: return launch_duo_tail<4, PAIRS>(tail, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
    case 5: return launch_duo_tail<5, PAIRS>(tail, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
    case 6: return launch_duo_tail<6, PAIRS>(tail, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
    default: return QPSK_ERR_UNSUPPORTED;
  }
}

}  // namespace

bool fll_duo_supported(int n_taps) { return n_taps >= 8 && n_taps <= 55; }

int fll_duo_launch(const FllParams& P, const float* taps, float2* ring, int* head, float2* pf, int C, const float2* x,
                   float2* y, long long L, long long ldx, long long ldy, cudaStream_t s) {
  // measured on a B200 (tools/fll_only.py, 40 taps): up to ~1300 streams one pair per CTA spreads the chain warps
  // over all SMs (356 cycles per sample at 1024 streams against 421); beyond that four pairs per CTA, one chain and
  // one side warp per scheduler, keep two chain warps off the same scheduler (4096 streams: 580 against 724)
  if (C <= 1280) return launch_duo<1>(P.n_taps, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
  return launch_duo<4>(P.n_taps, P, taps, ring, head, pf, C, x, y, L, ldx, ldy, s);
}

}  // namespace qpsk
