// demod.cu — K5: QPSKDeModulator on the GPU (MS/QPSKDeModulator.cs:11-456), batched over independent
// channels.  Compiled with --fmad=false (see loops.cuh).
//
// Chain per call (DeModulate :345-425):  [feed-forward AGC (opt-in, agc.cu; not in the reference)] ->
// [FLL (opt-in; the call at :359 is commented out upstream)] ->
// RRC matched filter (FirEngine, fir.cu) -> [fractionally spaced CMA equalizer (opt-in, eq.cu; not in the reference)] ->
// Mueller-Muller (loops.cu) -> [CMA equalizer (opt-in, eq.cu; not in the reference)] -> decode kernel: Costas + decision + differential decode -> bits -> TSC exact-match strip (:413-422).
// DeModulateBytes (:169-259): the bits then feed the per-channel framer kernel (8 bit-offset marker
// hunt, MSB-first packing into a bounded ring, end-marker search).
// All loop / framer state lives in device memory per channel and persists across calls, so arbitrary
// chunking of a stream gives the same output as the reference object would.
// Every call runs one loop over time chunks (DemodEngine::bits_dev): the front end of a chunk (front_chunk: host copy ->
// AGC -> FLL -> matched filter), then its symbol stage.  Long fused calls pipeline the chunks over a side stream; a single
// launch is the one-chunk case of the same loop, on the caller's stream.
#include <functional>
#include <memory>
#include <string>

#include "agc.cuh"
#include "eq.cuh"
#include "fir.cuh"
#include "loops.cuh"

namespace qpsk {

struct DiffState {
  int have_prev;
  float prevI, prevQ;
  int pad;
};

// ---------------------------------------------------------------------------------------------
// decode: Costas -> sign decision -> (differential) bits, one thread per channel (:374-408)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32)
    decode_kernel(const CostasParams P, CostasState* cst_g, DiffState* dst_g, int C, const float2* __restrict__ sym,
                  long long ld_sym, const int* __restrict__ n_sym, int diff, uint8_t* __restrict__ bits, long long ld_bits,
                  long long* n_bits) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const SinCosK K = sincos_load_consts();
  CostasState S = cst_g[c];
  DiffState D = dst_g[c];
  const float2* sc = sym + (long long)c * ld_sym;
  uchar2* bc = reinterpret_cast<uchar2*>(bits + (long long)c * ld_bits);
  const int n = n_sym[c];
  long long nb = 0;
  for (int k = 0; k < n; ++k) {
    const float2 in = sc[k];
    float rI, rQ;
    costas_step(P, K, S, in.x, in.y, rI, rQ);              // :378
    const float dI = (rI >= 0.f) ? 1.f : -1.f;             // GetSign (CostasLoopQpsk.cs:52-56)
    const float dQ = (rQ >= 0.f) ? 1.f : -1.f;
    unsigned char b0, b1;
    if (diff) {
      if (!D.have_prev) {                                  // :390-395 first symbol ever: reference only
        D.prevI = dI; D.prevQ = dQ; D.have_prev = 1;
        continue;
      }
      const float deltaI = dI * D.prevI + dQ * D.prevQ;    // :397
      const float deltaQ = dQ * D.prevI - dI * D.prevQ;    // :398
      D.prevI = dI; D.prevQ = dQ;
      if (fabsf(deltaI) >= fabsf(deltaQ)) {                // AppendDeltaBits :320-337
        if (deltaI >= 0.f) { b0 = 0; b1 = 0; } else { b0 = 1; b1 = 1; }
      } else {
        if (deltaQ >= 0.f) { b0 = 0; b1 = 1; } else { b0 = 1; b1 = 0; }
      }
    } else {                                               // AppendDecisionBits :304-318
      if (dI < 0.f) { b0 = 0; b1 = (dQ < 0.f) ? 0 : 1; }
      else { b0 = 1; b1 = (dQ >= 0.f) ? 1 : 0; }
    }
    bc[nb >> 1] = make_uchar2(b0, b1);
    nb += 2;
  }
  cst_g[c] = S;
  dst_g[c] = D;
  n_bits[c] = nb;
}

// ---------------------------------------------------------------------------------------------
// symsync_decode_kernel: Mueller-Muller -> Costas -> decision -> bits fused, 32 channels per CTA of two
// warps working as a pipeline, one thread per channel in each:
//   warp 0  stages the matched-filter samples of its 32 channels through shared memory in rounds of
//           kSsBlock samples (cp.async, double-buffered: the next round's loads fly while this one is
//           processed, and the interpolator's data-dependent 4-sample reads hit shared memory), runs the
//           Mueller-Muller recurrence and leaves the round's symbols in a shared queue;
//   warp 1  runs Costas + decision + differential decode on the previous round's symbols.
// The two recurrences are independent (MM never looks at the Costas output), so a round costs
// max(MM, Costas) instead of their sum.  Every round is one MuellerMuller.Process() call on
// [carried samples | block]: the reference loop is chunk-invariant (MuellerMuller.cs:122-133), so the
// symbols are those of the one-shot call.  Requires the unlimited-room case (sps - 0.1 > 1).
// ---------------------------------------------------------------------------------------------
constexpr int kSsBlock = 32;
constexpr int kSsCarry = 4;
// a channel's row of a round: [kSsCarry slots for the samples carried over from the previous round, right-aligned | the
// round's kSsBlock samples | 1 pad] — carried samples and block are contiguous, so the interpolator's four samples are four
// unconditional loads at (row + kSsCarry - carried + index).  Odd pitch (float2): rows of different lanes fall in different banks.
constexpr int kSsPitch = kSsCarry + kSsBlock + 1;
constexpr int kSsSymCap = kSsBlock + 4;  // symbols one round can emit (advance >= 0.9 samples)

__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

struct SsSmem {
  float2 raw[2][32 * kSsPitch];
  int nsymq[2][32];
};

// a ? x : y on doubles as an explicit selp (two SELs, never a branch)
__device__ __forceinline__ double sel_f64(bool a, double x, double y) {
  double r;
  asm("{\n.reg .pred p;\nsetp.ne.u32 p, %3, 0;\nselp.f64 %0, %1, %2, p;\n}" : "=d"(r) : "d"(x), "d"(y), "r"((unsigned)a));
  return r;
}

// ---- matched filter fused into the symbol-stage kernel (MFW > 0) --------------------------------------------------
// MFW extra warps run the RRC matched filter (ComplexFIRFilter.Filter :80-91 as called at QPSKDeModulator.cs:360) in the
// reference's own summation order — ComplexDotWindow's 8 lane partials, lanes added 0..7, then the N mod 8 tail, every
// product and sum rounded separately (FIRFilter.cs:165-192; the same arithmetic as fir_exact_real_kernel, bit for bit) —
// one round AHEAD of the Mueller-Muller warp, from a shared-memory ring of the last 128 RAW input samples per channel.
// The chain then reads each input sample from HBM once (8 B / sample, the fused-ideal traffic of SURVEY §8d) and the
// filtered samples never leave the SM: no matched-filter launch, no [channels][samples] scratch round trip.
// raw samples kept per channel: the round being filtered, N-1 samples of history before it and the round in flight —
// 96 slots (3 rounds) while N - 1 <= 32, else 128; rows are ring_n + 1 float2 apart (odd pitch: the 32 channels of a warp
// fall in different banks)
constexpr int kMfMaxTaps = 65;
struct MfTaps {
  float rev[kMfMaxTaps + 7];              // rev[i] = h[N-1-i]: window element i (oldest first) meets tap rev[i]
  int n_taps;
};
struct MfArgs {
  const float2* hist_in;                  // [C][HL] delay line of the FirEngine (newest last)
  float2* hist_out;
  int HL;
};
__device__ float2 g_neg_zero2 = {-0.0f, -0.0f};
// products rounded on their own: fma(x, g, -0) == round(x*g) exactly (the -0 addend changes neither value nor sign), and
// with the addend loaded at run time ptxas cannot contract the product into the add that follows (it does contract
// mul.rn.f32x2 feeding add.rn.f32x2 into one FFMA2, which would round once where the reference rounds twice)
__device__ __forceinline__ float2 mul2_rounded(float2 x, float2 g, float2 nz) { return ffma2(x, g, nz); }
__device__ __forceinline__ float2 add2_rn(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}

// One output through the reference's full complex product (hq = +0): the path for outputs whose real-tap reduction came
// out non-finite — an infinite SAMPLE makes the reference's hq*x terms NaN (0 * Inf), which the reduction does not model
// (see fir_exact_real_kernel).  Out of line: it practically never runs.
__device__ __noinline__ float2 mf_output_full(const float2* __restrict__ ring_ch, int ring_n, const MfTaps& T, int fmod) {
  const int N = T.n_taps;
  const int n_vec = N & ~7;
  float lI[8], lQ[8];
  for (int l = 0; l < 8; ++l) lI[l] = lQ[l] = 0.f;
  const float hq = 0.f;
  for (int i = 0; i < n_vec; ++i) {
    const float2 xv = ring_ch[(fmod + i) % ring_n];
    const float hi = T.rev[i];
    lI[i & 7] = __fadd_rn(lI[i & 7], __fsub_rn(__fmul_rn(hi, xv.x), __fmul_rn(hq, xv.y)));
    lQ[i & 7] = __fadd_rn(lQ[i & 7], __fadd_rn(__fmul_rn(hi, xv.y), __fmul_rn(hq, xv.x)));
  }
  float aI = 0.f, aQ = 0.f;
  for (int l = 0; l < 8; ++l) {
    aI = __fadd_rn(aI, lI[l]);
    aQ = __fadd_rn(aQ, lQ[l]);
  }
  for (int i = n_vec; i < N; ++i) {
    const float2 xv = ring_ch[(fmod + i) % ring_n];
    const float hi = T.rev[i];
    aI = __fadd_rn(aI, __fsub_rn(__fmul_rn(hi, xv.x), __fmul_rn(hq, xv.y)));
    aQ = __fadd_rn(aQ, __fadd_rn(__fmul_rn(hi, xv.y), __fmul_rn(hq, xv.x)));
  }
  return make_float2(aI, aQ);
}

// outputs j0 .. j1-1 (< blk) of round q for this lane's channel: sample n = 32q + j, window element i = raw[n-(N-1)+i].
// Four outputs per pass (32 independent lane partials: the warp runs alone on its scheduler, so the parallelism has to come
// from inside the thread).  All register arrays keep compile-time indices; the ring wrap is resolved once per block of
// eight taps (warp-uniform branch), so the common case loads with immediate offsets.  NB >= 0: the filter has exactly NB
// blocks of eight taps (+ a tail of < 8) and its taps sit in registers `tg` (the modem's usual 17 / 21 taps: NB = 2);
// NB < 0: any length, taps read from the constant bank.
constexpr int kMfR = 4;
constexpr int kMfRegTaps = 31;                    // taps held in registers by the NB = 1..3 variants
template <int NB>
__device__ __forceinline__ void mf_round(const float2* __restrict__ ring_ch, int ring_n, const MfTaps& T,
                                         const float (&tg)[kMfRegTaps], float2 nz, int q, int j0, int j1, int blk,
                                         float2* __restrict__ out_ch) {
  const int N = T.n_taps;
  const int n_vec = (NB >= 0) ? 8 * NB : (N & ~7);
  const int n_tail = N - n_vec;                   // 0..7
  for (int j = j0; j < j1 && j < blk; j += kMfR) {
    const int first = q * kSsBlock + j - (N - 1);
    int bmod = first % ring_n;                      // slot of window element 0 (first may be negative)
    if (bmod < 0) bmod += ring_n;
    const int fmod = bmod;
    float2 lp[kMfR][8];
#pragma unroll
    for (int r = 0; r < kMfR; ++r)
#pragma unroll
      for (int l = 0; l < 8; ++l) lp[r][l] = make_float2(0.f, 0.f);
    float2 wv[8 + kMfR - 1];
    // window elements bmod + k0 .. bmod + k1 - 1 into DST[k0 .. k1)
#define QPSK_MF_LOAD(DST, K0, K1)                                                             \
    if (bmod + (K1) <= ring_n) {                                                              \
      _Pragma("unroll") for (int k = (K0); k < (K1); ++k) DST[k] = ring_ch[bmod + k];          \
    } else {                                                                                  \
      _Pragma("unroll") for (int k = (K0); k < (K1); ++k) {                                    \
        const int idx = bmod + k;                                                             \
        DST[k] = ring_ch[idx >= ring_n ? idx - ring_n : idx];                                 \
      }                                                                                       \
    }
#define QPSK_MF_BLOCK(TAP)                                                                    \
    {                                                                                         \
      QPSK_MF_LOAD(wv, kMfR - 1, 8 + kMfR - 1)                                                \
      bmod += 8;                                                                              \
      if (bmod >= ring_n) bmod -= ring_n;                                                     \
      _Pragma("unroll") for (int l = 0; l < 8; ++l) {                                          \
        const float g = TAP(l);                                                               \
        const float2 gg = make_float2(g, g);                                                  \
        _Pragma("unroll") for (int r = 0; r < kMfR; ++r)                                       \
            lp[r][l] = add2_rn(lp[r][l], mul2_rounded(wv[l + r], gg, nz));                    \
      }                                                                                       \
      _Pragma("unroll") for (int k = 0; k < kMfR - 1; ++k) wv[k] = wv[8 + k];                  \
    }
    QPSK_MF_LOAD(wv, 0, kMfR - 1)
    if constexpr (NB >= 0) {
#pragma unroll
      for (int b = 0; b < NB; ++b) {
#define QPSK_TAP_REG(l) tg[8 * b + (l)]
        QPSK_MF_BLOCK(QPSK_TAP_REG)
#undef QPSK_TAP_REG
      }
    } else {
      for (int ib = 0; ib < n_vec; ib += 8) {
#define QPSK_TAP_LDC(l) T.rev[ib + (l)]
        QPSK_MF_BLOCK(QPSK_TAP_LDC)
#undef QPSK_TAP_LDC
      }
    }
#undef QPSK_MF_BLOCK
    // tail window: elements n_vec .. N-1 (+ kMfR-1); loaded in full (slots past the window hold other samples of the ring
    // and meet no tap) before the dependent lane sums start
    float2 tw[7 + kMfR - 1];
    QPSK_MF_LOAD(tw, 0, 7 + kMfR - 1)
#undef QPSK_MF_LOAD
    float2 acc[kMfR];
#pragma unroll
    for (int r = 0; r < kMfR; ++r) {
      acc[r] = make_float2(0.f, 0.f);
#pragma unroll
      for (int l = 0; l < 8; ++l) acc[r] = add2_rn(acc[r], lp[r][l]);            // lanes 0..7 (:176-180)
    }
#pragma unroll
    for (int i = 0; i < 7; ++i) {                                                  // scalar tail (:183-192)
      if (i >= n_tail) break;                                                      // warp-uniform
      float g;
      if constexpr (NB >= 0) g = tg[8 * NB + i]; else g = T.rev[n_vec + i];
      const float2 gg = make_float2(g, g);
#pragma unroll
      for (int r = 0; r < kMfR; ++r) acc[r] = add2_rn(acc[r], mul2_rounded(tw[i + r], gg, nz));
    }
    bool bad = false;
#pragma unroll
    for (int r = 0; r < kMfR; ++r)
      bad |= !(fabsf(acc[r].x) <= 3.402823466e+38f) || !(fabsf(acc[r].y) <= 3.402823466e+38f);
    if (bad) {
#pragma unroll
      for (int r = 0; r < kMfR; ++r)
        if (!(fabsf(acc[r].x) <= 3.402823466e+38f) || !(fabsf(acc[r].y) <= 3.402823466e+38f)) {
          int fm = fmod + r;
          if (fm >= ring_n) fm -= ring_n;
          acc[r] = mf_output_full(ring_ch, ring_n, T, fm);
        }
    }
#pragma unroll
    for (int r = 0; r < kMfR; ++r)
      if (j + r < blk) out_ch[j + r] = acc[r];
  }
}

// DENSE: compiled for four resident CTAs per SM (a 128-register cap: some spills in the filter warps) — the choice when
// the batch has more 32-channel CTAs than three per SM can hold, where one wave beats two
template <bool DIFF, int MFW, bool DENSE = false>
__global__ void __launch_bounds__(64 + 32 * MFW, MFW == 2 ? (DENSE ? 4 : 3) : (MFW == 4 ? 2 : 1))
    symsync_decode_kernel(const MmParams MP, MmState* mm_g, const float2* __restrict__ q_in, float2* __restrict__ q_out,
                          long long qcap, const CostasParams CP, CostasState* cst_g, DiffState* dst_g, int C,
                          const float2* __restrict__ x, long long L, long long ldx, uint8_t* __restrict__ bits,
                          long long ld_bits, long long* n_bits, int* n_sym_g, int append, const __grid_constant__ MfTaps MT,
                          const MfArgs MA, const int ring_n, const int sym_pitch) {
  // MFW > 0: x is the RAW input (or the FLL output) and MFW extra warps run the matched filter one round ahead; MFW == 0:
  // x is the matched-filter output (MT / MA unused).
  // append != 0: this launch continues a call split into time chunks (DemodEngine::bits_dev): bits and counts go on
  // from where the previous chunk left them.  A chunk boundary on a multiple of kSsBlock samples is exactly a round
  // boundary of the single launch (same carried samples, same rebased base_index), so the split is bit-neutral.
  constexpr bool diff = DIFF;
  __shared__ SsSmem sm;
  // dynamic shared memory: the symbol queues [2][32][sym_pitch] (sym_pitch - 1 = most symbols one round can emit at this
  // samples-per-symbol rate), then — MFW > 0 — the raw-sample ring [32][ring_n + 1]
  extern __shared__ __align__(16) float2 dyn_smem[];
  float2* const symq0 = dyn_smem;
  float2* const mf_ring = dyn_smem + 2 * 32 * sym_pitch;
  const int ring_pitch = ring_n + 1;
  const int lane = threadIdx.x & 31;
  const int role = threadIdx.x >> 5;                // 0: symbol sync, 1: Costas + decode, 2..: matched filter
  const int c0 = blockIdx.x * 32;
  const int c_raw = c0 + lane;
  const bool live = c_raw < C;
  const int c = live ? c_raw : C - 1;
  const int rounds = (int)((L + kSsBlock - 1) / kSsBlock);

  // role 0 state
  MmState S;
  int carried = 0, n_sym = 0;
  // role 1 state
  const SinCosK SK = sincos_load_consts();
  const double magic = ld_const_pinned(&kSinCosMagic);
  CostasState K;
  DiffState D;
  long long nb = (append && role == 1) ? n_bits[c] : 0;
  uchar2* bc = reinterpret_cast<uchar2*>(bits + (long long)c * ld_bits);

  auto stage = [&](int r) {                          // lane i copies sample 32r+i of every channel of the CTA
    const long long n0 = (long long)r * kSsBlock;
    const int blk = (int)((L - n0) < kSsBlock ? (L - n0) : kSsBlock);
    // MFW == 0: straight into the round's double buffer; MFW > 0: into the raw ring (slot = sample index mod 128)
    float2* dst = (MFW > 0) ? (mf_ring + (int)((n0 + lane) % ring_n)) : (sm.raw[r & 1] + kSsCarry + lane);
    const int pitch = (MFW > 0) ? ring_pitch : kSsPitch;
    if (lane < blk) {
#pragma unroll 8
      for (int j = 0; j < 32; ++j) {
        int ch = c0 + j;
        if (ch >= C) ch = C - 1;
        cp_async8(dst + j * pitch, x + (long long)ch * ldx + n0 + lane);
      }
    }
    cp_async_commit();
  };
  constexpr int kAhead = (MFW > 0) ? 2 : 1;          // rounds the staging runs ahead of the Mueller-Muller warp
  float2 nz = make_float2(0.f, 0.f);
  if (MFW > 0 && role >= 2) {
    asm volatile("ld.volatile.global.v2.f32 {%0, %1}, [%2];" : "=f"(nz.x), "=f"(nz.y) : "l"(&g_neg_zero2));
  }
  const int mf_per = (MFW > 0) ? (kSsBlock / (MFW > 0 ? MFW : 1)) : 0;   // outputs per matched-filter warp and round
  // the filter's taps in registers when there are few enough (NB = 1..3 blocks of eight + tail)
  float tg[kMfRegTaps];
  const int mf_nb = (MFW > 0 && MT.n_taps >= 8 && MT.n_taps <= kMfRegTaps) ? (MT.n_taps >> 3) : -1;
  if (MFW > 0 && role >= 2) {
#pragma unroll
    for (int i = 0; i < kMfRegTaps; ++i) tg[i] = MT.rev[i];
  }
  auto mf_dispatch = [&](int q, int blk_q) {
    const float2* rc = mf_ring + lane * ring_pitch;
    float2* oc = sm.raw[q & 1] + lane * kSsPitch + kSsCarry;
    const int j0 = (role - 2) * mf_per, j1 = (role - 1) * mf_per;
    switch (mf_nb) {
      case 1: mf_round<1>(rc, ring_n, MT, tg, nz, q, j0, j1, blk_q, oc); break;
      case 2: mf_round<2>(rc, ring_n, MT, tg, nz, q, j0, j1, blk_q, oc); break;
      case 3: mf_round<3>(rc, ring_n, MT, tg, nz, q, j0, j1, blk_q, oc); break;
      default: mf_round<-1>(rc, ring_n, MT, tg, nz, q, j0, j1, blk_q, oc); break;
    }
  };

  // The Costas warp (which has the slack) also stages the samples: round r+1 is requested at the top of round r and
  // waited for before the barrier that ends it, so the Mueller-Muller warp finds its round in shared memory.
  if (role == 0) {
    S = mm_g[c];
    if (append) n_sym = n_sym_g[c];
    carried = S.queued;                              // host guarantees <= kSsCarry
    for (int i = 0; i < carried; ++i) sm.raw[0][lane * kSsPitch + kSsCarry - carried + i] = q_in[(long long)c * qcap + i];
  } else if (role == 1) {
    if (rounds > 0) stage(0);
    if (MFW > 0 && rounds > 1) stage(1);
    K = cst_g[c];
    D = dst_g[c];
    cp_async_wait<0>();
  } else {
    // the filter's delay line: samples -1 .. -(N-1) of this call are the newest entries of the FirEngine history
    for (int k = 1; k < MT.n_taps; ++k)
      if ((k - 1) % MFW == role - 2)
        mf_ring[lane * ring_pitch + (ring_n - k)] = MA.hist_in[(long long)c * MA.HL + MA.HL - k];
  }
  __syncthreads();
  if (MFW > 0) {
    if (role >= 2 && rounds > 0) {
      const int blk0 = (int)(L < kSsBlock ? L : kSsBlock);
      mf_dispatch(0, blk0);
    }
    __syncthreads();
  }
  // Mueller-Muller loop registers.  The previous decision is +-1 and only ever multiplies (:78), so it is kept as a
  // sign; the previous sample is kept widened (it only appears as (double)dec * prevSample, :79).
  bool prevNegI = S.prevDI < 0.f, prevNegQ = S.prevDQ < 0.f;
  double prevSI_d = (double)S.prevSI, prevSQ_d = (double)S.prevSQ;
  bool has_prev = S.has_prev != 0;

  // 1 / (largest advance per symbol), rounded down a little: the counted loop below must stay conservative
  const double inv_max_adv = (1.0 / (MP.sps + 0.1000001)) * (1.0 - 1e-12);
  for (int r = 0; r <= rounds; ++r) {
    if (role == 0) {
      if (r < rounds) {
        const long long n0 = (long long)r * kSsBlock;
        const int blk = (int)((L - n0) < kSsBlock ? (L - n0) : kSsBlock);
        // logical buffer [carried samples | block] = row + kSsCarry - carried .. (one contiguous run)
        const float2* vbuf = sm.raw[r & 1] + lane * kSsPitch + (kSsCarry - carried);
        const int count = carried + blk;
        const double limit_d = (double)(count - 2);  // loop test in fp64: base + 2 < count  <=>  base_d < count - 2
        float2* sq = symq0 + ((r & 1) * 32 + lane) * sym_pitch;
        int ns = 0;
        double base_d = (double)S.base_index;        // == (double)baseIndex exactly; floor() keeps it integral
        // One pass = one symbol (MuellerMuller.cs:62-120); the loop-carried chain is mu -> interpolator -> error ->
        // loop filter -> newTime -> floor -> mu.  Off that chain: +-1 factors are sign flips (exact), both clamp tests
        // read the unclamped value (:87-89: 0.1 > -0.1, so the second test cannot fire after the first), floor()
        // yields (double)baseIndex directly (no F2I -> I2F round trip), and the loop test reads the fp64 base.  The
        // post-advance break (:118-119, base + 1 >= count) implies the loop test fails, so one test serves both.
        const double adv_hi = MP.sps + 0.1, adv_lo = MP.sps + (-0.1);            // sps + clamp(corr) at the two rails
        auto one_symbol = [&]() {
          float ci, cq;
          mm_interp_lin(vbuf, S.base_index, S.mu, ci, cq);
          const bool posI = ci >= 0.f, posQ = cq >= 0.f;     // GetSignQpsk :194-198
          const double ci_d = (double)ci, cq_d = (double)cq;
          // branch-free (one basic block per symbol, so ptxas can interleave the independent work with the chain):
          // without a previous symbol the error terms are computed and discarded (:72-97)
          const double term1 = flip_sign_if(ci_d, prevNegI) + flip_sign_if(cq_d, prevNegQ);       // :78
          const double term2 = flip_sign_if(prevSI_d, !posI) + flip_sign_if(prevSQ_d, !posQ);     // :79
          const double e = term1 - term2;
          const double integ = S.integral + MP.ki * e;       // :83
          const double corr = MP.kp * e + integ;             // :84
          // clamp (:87-89), advance (:91, :96) and newTime (:113) with the selects moved to the end: the three
          // possible advances sps + 0.1, sps - 0.1, sps do not depend on the error, so their newTime candidates
          // are formed early and the two compares run beside the adds of the unclamped candidate — same operations
          // on the selected path, ~20 cycles less on the loop-carried chain
          const double bm = base_d + S.mu;
          const double nt_c = bm + (MP.sps + corr);
          const bool hi = corr > 0.1, lo = corr < -0.1;
          // selp through inline PTX: left to itself the compiler folds the candidates back into bm + select(advance)
          // and branches on the compares
          const double nt_cl = sel_f64(hi, bm + adv_hi, sel_f64(lo, bm + adv_lo, nt_c));
          const double newTime = sel_f64(has_prev, nt_cl, bm + MP.sps);
          S.integral = has_prev ? integ : S.integral;
          has_prev = true;
          prevSI_d = ci_d; prevSQ_d = cq_d; prevNegI = !posI; prevNegQ = !posQ;
          // floor (:114) by a round-down add of 2^52 (0 <= newTime < 2^31): one DADD.RM instead of FRND.F64.FLOOR on
          // the XU pipe, and the integer index is the low word of the same sum (no F2I in front of the next LDS)
          const double fl52 = __dadd_rd(newTime, 4503599627370496.0);
          S.base_index = __double2loint(fl52);       // :114
          base_d = fl52 - 4503599627370496.0;        // == floor(newTime), exact
          S.mu = newTime - base_d;                   // :115
          sq[ns++] = make_float2(ci, cq);
        };
        // The loop test reads the newest base, i.e. it closes the dependency chain through floor -> compare -> branch.
        // Every symbol advances time by at most sps + 0.1 (:87-91), so the first n_safe passes are known to satisfy it
        // and run as a counted loop whose branch resolves early; only the last one or two passes are tested.
        const double span_d = limit_d - (base_d + S.mu);
        const double q = span_d * inv_max_adv;       // (a product instead of a ~60-instruction fp64 division per round)
        int n_safe = (q > 1.0) ? (int)q - 1 : 0;       // conservative: floor(q) - 1 full advances certainly fit
        for (int j = 0; j < n_safe; ++j) one_symbol();
        while (base_d < limit_d) one_symbol();       // :62
        n_sym += ns;
        sm.nsymq[r & 1][lane] = ns;
        // drop consumed samples, keep at least the last three (:123-129)
        const int consumed = min(max(0, S.base_index - 1), max(0, count - 3));
        const int remain = count - consumed;         // <= 3 here (4 slots)
        // ... into the carry slots of the NEXT round's row, right-aligned against its block (the filter warps / cp.async
        // only write the block part of that row)
        float2* nrow = sm.raw[(r + 1) & 1] + lane * kSsPitch + (kSsCarry - remain);
#pragma unroll
        for (int i = 0; i < kSsCarry; ++i)
          if (i < remain) nrow[i] = vbuf[consumed + i];
        carried = remain;
        S.base_index -= consumed;
      }
    } else if (role == 1) {
      if (r + kAhead < rounds) stage(r + kAhead);    // in flight during this round's Costas work
    } else if (r + 1 < rounds) {
      // matched filter of round r+1 (its raw samples landed before the barrier that ended round r-1)
      const long long n1 = (long long)(r + 1) * kSsBlock;
      const int blk1 = (int)((L - n1) < kSsBlock ? (L - n1) : kSsBlock);
      mf_dispatch(r + 1, blk1);
    }
    if (role == 1 && r >= 1) {
      // ---- Costas + decision + differential decode (QPSKDeModulator.cs:374-408) on round r-1 ----
      // One basic block per symbol: the Costas recurrence is the critical chain; the decisions, the differential
      // decode (pure predicate logic on the four sign bits: d*conj(d_prev) of two unit-corner symbols is one of
      // 2, 2j, -2, -2j, so the float products of :397-398 reduce to XORs of signs, bit for bit) and the predicated
      // bit store hang off it and are scheduled into its latency shadows.  The |theta| >= 1e5 case of costas_step
      // cannot be tested inside the block without splitting it: it is accumulated in `wild` and, should it ever fire,
      // the round is replayed from the saved state through the exact (branching) step.
      const int b = (r - 1) & 1;
      const int ns = sm.nsymq[b][lane];
      const float2* sq = symq0 + (b * 32 + lane) * sym_pitch;
      const CostasState K0 = K;
      const DiffState D0 = D;
      const long long nb0 = nb;
      bool wild = false;
      // decisions as sign bits: bit 0 = I is -1, bit 1 = Q is -1; `prev` holds the previous symbol's pair
      unsigned prev = (D.prevI < 0.f ? 1u : 0u) | (D.prevQ < 0.f ? 2u : 0u);
      const bool skipFirst = diff && !D.have_prev;       // the first symbol ever is only the reference (:390-395)
      // The two output bits as a function of idx = cur | prev << 2, one 16-entry table per bit.  Differential
      // (AppendDeltaBits :320-337 on delta = d * conj(d_prev), :397-398): the four float products are +-1, so
      // deltaI = +-2 iff the I and Q sign changes agree (then bits 00 / 11), else deltaQ = +-2 (bits 01 / 10).
      // Absolute (AppendDecisionBits :304-318): b0 = (dI >= 0), b1 = (dQ >= 0).
      constexpr unsigned kB0 = DIFF ? 0x3A5Cu : 0x5555u;   // enumerated from the float formulas (tests compare with the
      constexpr unsigned kB1 = DIFF ? 0x53CAu : 0x3333u;   // unfused decode_kernel, which keeps them)
      // Idle lanes shadow channel C-1 on identical inputs, so their stores duplicate the owner's bytes: no `live`
      // predicate (and no branch around the store).  When the very first symbol is only a reference, its bits land on
      // slot 0 and are overwritten by the next symbol's (the pointer is held for one pass).
      uchar2* p = bc + (nb >> 1);
      bool hold = skipFirst;
      float2 nxt = sq[0];
#pragma unroll 2
      for (int k = 0; k < ns; ++k) {
        const float2 in = nxt;
        nxt = sq[k + 1];                                 // row pitch >= symbols per round + 1: in bounds for every k < ns
        float rI, rQ;
        unsigned sI, sQ;
        costas_step_fast2(CP, SK, magic, K, in.x, in.y, rI, rQ, sI, sQ, wild);
        const unsigned cur = (sI >> 31) | (sQ >> 30);
        const unsigned idx = cur | (prev << 2);
        prev = cur;
        *p = make_uchar2((unsigned char)((kB0 >> idx) & 1u), (unsigned char)((kB1 >> idx) & 1u));
        p += hold ? 0 : 1;
        hold = false;
      }
      const int stored = ns - ((skipFirst && ns > 0) ? 1 : 0);
      nb += 2LL * stored;
      const bool pNegI = (prev & 1u) != 0, pNegQ = (prev & 2u) != 0;
      if (diff && ns > 0) { D.have_prev = 1; D.prevI = pNegI ? -1.f : 1.f; D.prevQ = pNegQ ? -1.f : 1.f; }
      if (wild) {                                         // never in practice; exactness for any input
        K = K0; D = D0; nb = nb0;
        for (int k = 0; k < ns; ++k) {
          const float2 in = sq[k];
          float rI, rQ;
          costas_step(CP, SK, K, in.x, in.y, rI, rQ);
          const float dI = (rI >= 0.f) ? 1.f : -1.f;
          const float dQ = (rQ >= 0.f) ? 1.f : -1.f;
          unsigned char b0, b1;
          if (diff) {
            if (!D.have_prev) {
              D.prevI = dI; D.prevQ = dQ; D.have_prev = 1;
              continue;
            }
            const float deltaI = dI * D.prevI + dQ * D.prevQ;
            const float deltaQ = dQ * D.prevI - dI * D.prevQ;
            D.prevI = dI; D.prevQ = dQ;
            if (fabsf(deltaI) >= fabsf(deltaQ)) {
              if (deltaI >= 0.f) { b0 = 0; b1 = 0; } else { b0 = 1; b1 = 1; }
            } else {
              if (deltaQ >= 0.f) { b0 = 0; b1 = 1; } else { b0 = 1; b1 = 0; }
            }
          } else {
            if (dI < 0.f) { b0 = 0; b1 = (dQ < 0.f) ? 0 : 1; }
            else { b0 = 1; b1 = (dQ >= 0.f) ? 1 : 0; }
          }
          if (live) bc[nb >> 1] = make_uchar2(b0, b1);
          nb += 2;
        }
      }
    }
    if (role == 1) cp_async_wait<0>();               // the next round's samples have landed
    __syncthreads();                                 // hand the round's symbol queue over / free the other one
  }
  if (role == 0) {
    S.has_prev = has_prev ? 1 : 0;
    S.prevSI = (float)prevSI_d; S.prevSQ = (float)prevSQ_d;   // exact: they were widened floats
    S.prevDI = prevNegI ? -1.f : 1.f; S.prevDQ = prevNegQ ? -1.f : 1.f;
  }
  if (live) {
    if (role == 0) {
      for (int i = 0; i < carried; ++i) q_out[(long long)c * qcap + i] = sm.raw[rounds & 1][lane * kSsPitch + kSsCarry - carried + i];
      S.queued = carried;
      mm_g[c] = S;
      n_sym_g[c] = n_sym;
    } else if (role == 1) {
      cst_g[c] = K;
      dst_g[c] = D;
      n_bits[c] = nb;
    } else {
      // the delay line after this call: the last HL samples of (history ++ x), as FirEngine keeps it
      for (int i = role - 2; i < MA.HL; i += (MFW > 0 ? MFW : 1)) {
        const long long m = L - MA.HL + i;
        MA.hist_out[(long long)c * MA.HL + i] = (m < 0) ? MA.hist_in[(long long)c * MA.HL + MA.HL + m] : x[(long long)c * ldx + m];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// TSC strip: rx.IndexOf(tsc) then Substring (:413-422), one warp per channel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
    tsc_strip_kernel(const uint8_t* __restrict__ raw, long long ld_raw, const long long* __restrict__ n_raw,
                     const uint8_t* __restrict__ tsc, int T, uint8_t* __restrict__ out, long long ld_out, long long* n_out,
                     int C) {
  const int c = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (c >= C) return;
  const int lane = threadIdx.x & 31;
  const uint8_t* r = raw + (long long)c * ld_raw;
  const long long n = n_raw[c];
  long long first = -1;
  for (long long base = 0; base + T <= n; base += 32) {
    const long long idx = base + lane;
    bool ok = idx + T <= n;
    for (int j = 0; ok && j < T; ++j) ok = (r[idx + j] == tsc[j]);
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m) {
      first = base + (__ffs(m) - 1);
      break;
    }
  }
  uint8_t* o = out + (long long)c * ld_out;
  long long len = 0;
  if (first >= 0) {
    const long long start = first + T;
    len = n - start;
    for (long long i = lane; i < len; i += 32) o[i] = r[start + i];
  }
  if (lane == 0) n_out[c] = len;
}

// Same, with the channel's bits staged in shared memory first (coalesced 16-byte loads), so the search
// and the shifted copy read shared memory; used when a channel's raw bits fit (the usual burst sizes).
__global__ void __launch_bounds__(128)
    tsc_strip_smem_kernel(const uint8_t* __restrict__ raw, long long ld_raw, const long long* __restrict__ n_raw,
                          const uint8_t* __restrict__ tsc, int T, uint8_t* __restrict__ out, long long ld_out, long long* n_out,
                          int C, int row_bytes, int words_per_row) {
  extern __shared__ __align__(16) uint8_t sm_bits[];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c = blockIdx.x * (blockDim.x >> 5) + w;
  if (c >= C) return;
  uint8_t* row = sm_bits + (size_t)w * row_bytes;
  uint8_t* pat = sm_bits + (size_t)(blockDim.x >> 5) * row_bytes + (size_t)w * ((T + 15) & ~15);
  // packed-bit rows behind the patterns (words_per_row == 0: not provisioned, byte search)
  uint32_t* words = words_per_row > 0
                        ? reinterpret_cast<uint32_t*>(sm_bits + (size_t)(blockDim.x >> 5) * (row_bytes + ((T + 15) & ~15)))
                        : nullptr;
  const uint8_t* r = raw + (long long)c * ld_raw;
  const int n = (int)n_raw[c];
  // rows are 16-byte aligned when ld_raw is a multiple of 16 and the base is; otherwise byte loads
  if ((((uintptr_t)r) & 15) == 0) {
    const uint4* r4 = reinterpret_cast<const uint4*>(r);
    uint4* row4 = reinterpret_cast<uint4*>(row);
    for (int i = lane; i < (n + 15) / 16; i += 32) row4[i] = r4[i];
  } else {
    for (int i = lane; i < n; i += 32) row[i] = r[i];
  }
  for (int i = lane; i < T; i += 32) pat[i] = tsc[i];
  __syncwarp();
  int first = -1;
  // Bit-parallel search (T <= 64, the usual 64-bit TSC): the row's 0/1 bytes are packed 32 per word (`words`, behind the
  // patterns in shared memory), the pattern into two words, and position 32k + lane is tested with two funnel shifts and
  // two masked compares — about 12 instructions per 32 positions instead of a byte loop with early exit per position.
  // Same result: the first position whose T bytes equal the pattern (a pattern byte other than 0/1 never matches a
  // bit, so such patterns keep the byte loop).
  bool searched = false;
  if (T >= 1 && T <= 64 && words != nullptr) {
    uint32_t* W = words + (size_t)w * words_per_row;
    bool binary = true;
    for (int i = lane; i < T; i += 32) binary &= pat[i] <= 1;
    binary = __all_sync(0xffffffffu, binary);
    if (binary) {
      const int ng = (n + 31) >> 5;                          // 32-byte groups; bytes at and beyond n are masked off
      const uint32_t* rw = reinterpret_cast<const uint32_t*>(row);
      for (int k = lane; k < ng; k += 32) {
        uint32_t bits = 0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const int bidx = 32 * k + 4 * q;
          uint32_t v = (bidx < n) ? rw[8 * k + q] : 0u;      // bytes b0..b3 (0/1) -> bits 0..3
          if (bidx + 4 > n) v &= (n - bidx >= 1 ? 0xFFu : 0u) | (n - bidx >= 2 ? 0xFF00u : 0u) | (n - bidx >= 3 ? 0xFF0000u : 0u);
          bits |= ((v * 0x01020408u) >> 24) << (4 * q);
        }
        W[k] = bits;
      }
      if (lane < 2) W[ng + lane] = 0u;
      uint32_t p_lo = 0, p_hi = 0;
      for (int i = 0; i < T; ++i) {
        const uint32_t b = pat[i];
        if (i < 32) p_lo |= b << i; else p_hi |= b << (i - 32);
      }
      const uint32_t m_lo = (T >= 32) ? 0xFFFFFFFFu : ((1u << T) - 1u);
      const uint32_t m_hi = (T <= 32) ? 0u : ((T >= 64) ? 0xFFFFFFFFu : ((1u << (T - 32)) - 1u));
      __syncwarp();
      for (int k = 0; 32 * k + T <= n; ++k) {
        const uint32_t a = W[k], b = W[k + 1], c2 = W[k + 2];
        const uint32_t lo = __funnelshift_r(a, b, lane), hi = __funnelshift_r(b, c2, lane);
        const bool ok = (32 * k + lane + T <= n) && ((((lo ^ p_lo) & m_lo) | ((hi ^ p_hi) & m_hi)) == 0u);
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (m) {
          first = 32 * k + (__ffs(m) - 1);
          break;
        }
      }
      searched = true;
    }
  }
  for (int base = 0; !searched && base + T <= n; base += 32) {
    const int idx = base + lane;
    bool ok = idx + T <= n;
    for (int j = 0; ok && j < T; ++j) ok = (row[idx + j] == pat[j]);
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m) {
      first = base + (__ffs(m) - 1);
      break;
    }
  }
  uint8_t* o = out + (long long)c * ld_out;
  int len = 0;
  if (first >= 0) {
    const int start = first + T;
    len = n - start;
    if (len >= 64) {
      // shifted copy, 16 bytes per lane and pass: up to 15 head bytes bring the output to a 16-byte boundary, then five
      // aligned shared-memory words are funnel-shifted into four output words (the staged row is 16-byte aligned and
      // the words around the payload lie inside the CTA's shared memory; only bytes below n enter the result)
      const int head = (int)((16 - (((uintptr_t)o) & 15)) & 15);
      if (lane < head) o[lane] = row[start + lane];
      const int st2 = start + head, len2 = len - head;
      const int sh = (st2 & 3) * 8;
      const uint32_t* rw = reinterpret_cast<const uint32_t*>(row) + (st2 >> 2);
      uint4* o16 = reinterpret_cast<uint4*>(o + head);
      const int nq = len2 >> 4;
      for (int i = lane; i < nq; i += 32) {
        const uint32_t* w = rw + 4 * i;
        const uint32_t w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
        const uint32_t w4 = sh ? w[4] : 0u;
        o16[i] = make_uint4(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh), __funnelshift_r(w2, w3, sh),
                            __funnelshift_r(w3, w4, sh));
      }
      for (int i = 16 * nq + lane; i < len2; i += 32) o[head + i] = row[st2 + i];
    } else if ((((uintptr_t)o) & 3) == 0) {
      uint32_t* o4 = reinterpret_cast<uint32_t*>(o);
      const int nw = len >> 2;
      for (int i = lane; i < nw; i += 32) {
        const uint8_t* sp = row + start + 4 * i;
        o4[i] = (uint32_t)sp[0] | ((uint32_t)sp[1] << 8) | ((uint32_t)sp[2] << 16) | ((uint32_t)sp[3] << 24);
      }
      for (int i = 4 * nw + lane; i < len; i += 32) o[i] = row[start + i];
    } else {
      for (int i = lane; i < len; i += 32) o[i] = row[start + i];
    }
  }
  if (lane == 0) n_out[c] = len;
}

// ---------------------------------------------------------------------------------------------
// framer (DeModulateBytes :169-259), one warp per channel: the byte packing, the eight bit-offset marker hunts, the
// ring append, the end-marker search and the payload copy are each spread over the 32 lanes; the decisions (which
// offset wins, where the frame ends, overflow -> reset) are the reference's, taken warp-uniformly.
// ---------------------------------------------------------------------------------------------
struct FramerState {
  int in_frame;
  int pack_byte;
  int pack_bits;
  int carry_len;
  long long ring_count;
};

struct FramerArgs {
  FramerState* st;
  uint8_t* carry;       // [C][carry_cap] bits 0/1
  int carry_cap;
  uint8_t* ring;        // [C][ring_cap] payload bytes of the current frame
  long long ring_cap;
  uint8_t* pk;          // [C][pk_ld] scratch: candidate bits packed MSB-first at offset 0
  long long pk_ld;
  const uint8_t* rx;    // [C][ld_rx] bits 0/1 of this call
  long long ld_rx;
  const long long* n_rx;
  const uint8_t* markers;  // start | end
  int ns, ne;
  uint8_t* payload;     // [C][payload_cap]
  long long payload_cap;
  long long* n_payload; // [C] full payload length (may exceed payload_cap: truncated copy)
  int C;
};

constexpr int kFramerWarps = 4;           // channels per CTA

__device__ __forceinline__ void framer_reset(FramerState& S) {   // ResetFramer :159-167
  S.in_frame = 0; S.pack_byte = 0; S.pack_bits = 0; S.carry_len = 0; S.ring_count = 0;
}

// byte i of the packed candidate read at bit offset o: pk[i] holds candidate bits 8i .. 8i+7, MSB first, and the
// byte after the last packed one is zero (BitsToBytes at offset o, HelperFunctions.cs:32-52, without re-packing)
__device__ __forceinline__ int framer_pk_byte(const uint8_t* pk, long long i, int o) {
  const int hi = pk[i], lo = pk[i + 1];
  return ((hi << o) | (lo >> (8 - o))) & 0xFF;
}

// RingIndexOf :133-149, positions spread over the lanes; the lowest matching index wins
__device__ __forceinline__ long long framer_ring_index_of(const uint8_t* ring, long long ring_count, const uint8_t* pat, int np,
                                                          long long from, int lane) {
  if (np == 0) return 0;
  if (ring_count < np) return -1;
  const long long last = ring_count - np;
  for (long long base = (from > 0 ? from : 0); base <= last; base += 32) {
    const long long i = base + lane;
    bool ok = i <= last;
    if (ok) {
      for (int j = 0; j < np; ++j)
        if (ring[i + j] != pat[j]) { ok = false; break; }
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (m) return base + (__ffs(m) - 1);
  }
  return -1;
}

// RingCopyOut :151-157 + the length the caller sees
__device__ __forceinline__ void framer_emit(const FramerArgs& a, int c, const uint8_t* ring, long long end_at, int lane) {
  uint8_t* out = a.payload + (long long)c * a.payload_cap;
  const long long ncopy = end_at < a.payload_cap ? end_at : a.payload_cap;
  for (long long i = lane; i < ncopy; i += 32) out[i] = ring[i];
  if (lane == 0) a.n_payload[c] = end_at;
}

__global__ void __launch_bounds__(32 * kFramerWarps) framer_kernel(const FramerArgs a) {
  const int lane = threadIdx.x & 31;
  const int c = blockIdx.x * kFramerWarps + (threadIdx.x >> 5);
  if (c >= a.C) return;                                          // warp-uniform
  const long long n_rx = a.n_rx[c];
  if (lane == 0) a.n_payload[c] = 0;
  if (n_rx == 0) return;                                         // :179-180
  FramerState S = a.st[c];
  uint8_t* ring = a.ring + (long long)c * a.ring_cap;
  const uint8_t* rx = a.rx + (long long)c * a.ld_rx;
  const uint8_t* sm = a.markers;
  const uint8_t* em = a.markers + a.ns;
  __syncwarp();                                                  // every lane has read the state before lane 0 rewrites it
  if (!S.in_frame) {
    uint8_t* carry = a.carry + (long long)c * a.carry_cap;
    const int cl = S.carry_len;
    const long long cand_len = cl + n_rx;                        // :185
    // pack the candidate bits once (offset 0); byte i at bit offset o is a shift of two neighbours
    uint8_t* pk = a.pk + (long long)c * a.pk_ld;
    const long long nb0 = (cand_len + 7) >> 3;
    for (long long i = lane; i < nb0; i += 32) {
      int v = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const long long k = 8 * i + j;
        int bit = 0;
        if (k < cand_len) bit = (k < cl) ? carry[k] : rx[k - cl];
        v = (v << 1) | bit;
      }
      pk[i] = (uint8_t)v;
    }
    if (lane == 0) pk[nb0] = 0;
    __syncwarp();
    // one pass over the byte positions: first[o] = lowest byte index at which the start marker sits at bit offset o
    // (IndexOf of BitsToBytes(candidate, o), :187-196); the lowest offset that has one wins, as in the reference's loop
    long long first[8];
#pragma unroll
    for (int o = 0; o < 8; ++o) first[o] = -1;
    const long long n_pos = ((cand_len >> 3) >= a.ns) ? (cand_len >> 3) - a.ns + 1 : 0;   // positions valid at offset 0
    for (long long base = 0; base < n_pos; base += 32) {
      const long long i = base + lane;
      unsigned hit = 0;
      if (i < n_pos) {
#pragma unroll
        for (int o = 0; o < 8; ++o) {
          // offset o has nB = (cand_len - o) >> 3 bytes (none when fewer than 8 bits are usable, :190)
          if (i + a.ns > ((cand_len - o) >> 3)) continue;
          bool ok = true;
          for (int j = 0; j < a.ns; ++j)
            if (framer_pk_byte(pk, i + j, o) != sm[j]) { ok = false; break; }
          if (ok) hit |= 1u << o;
        }
      }
      if (!__any_sync(0xffffffffu, hit != 0)) continue;
#pragma unroll
      for (int o = 0; o < 8; ++o) {
        const unsigned m = __ballot_sync(0xffffffffu, (hit >> o) & 1u);
        if (m && first[o] < 0) first[o] = base + (__ffs(m) - 1);
      }
      if (first[0] >= 0) break;                                  // nothing can beat offset 0
    }
    int o_win = -1;
    long long s = -1;
#pragma unroll
    for (int o = 7; o >= 0; --o)
      if (first[o] >= 0) { o_win = o; s = first[o]; }
    if (o_win >= 0) {
      const long long marker_end = o_win + 8 * (s + a.ns);       // :198
      S.in_frame = 1;                                            // :202-207
      // AppendBitsToRing(candidate, marker_end) :210-211: whole bytes are the offset-o bytes after the marker
      const long long total = cand_len - marker_end;
      const long long appended = total >> 3;
      const int rem = (int)(total & 7);
      if (appended > a.ring_cap) {                               // RingTryWriteByte fails :96-104 -> :212-217
        framer_reset(S);
        if (lane == 0) a.st[c] = S;
        return;
      }
      for (long long j = lane; j < appended; j += 32) ring[j] = (uint8_t)framer_pk_byte(pk, s + a.ns + j, o_win);
      S.ring_count = appended;
      S.pack_bits = rem;
      S.pack_byte = rem ? (framer_pk_byte(pk, s + a.ns + appended, o_win) >> (8 - rem)) : 0;
      __syncwarp();
      const long long end_at = framer_ring_index_of(ring, S.ring_count, em, a.ne, S.ring_count - (appended + a.ne), lane);   // :220
      if (end_at >= 0) {
        framer_emit(a, c, ring, end_at, lane);
        framer_reset(S);
      }
      if (lane == 0) a.st[c] = S;
      return;                                                    // :226 / :229
    }
    // no start marker: keep a tail so it can span calls (:233-235); the bits come back out of the packed copy
    const long long keep = cand_len < (long long)(a.ns * 8 + 7) ? cand_len : (long long)(a.ns * 8 + 7);
    const long long src0 = cand_len - keep;
    for (long long i = lane; i < keep; i += 32) {
      const long long k = src0 + i;
      carry[i] = (uint8_t)((pk[k >> 3] >> (7 - (int)(k & 7))) & 1);
    }
    S.carry_len = (int)keep;
    if (lane == 0) a.st[c] = S;
    return;
  }
  // already inside a frame (:238-258): the bit stream is the pending pack bits followed by this call's bits
  const int nb_old = S.pack_bits, pb_old = S.pack_byte;
  const long long total = nb_old + n_rx;
  const long long appended = total >> 3;
  auto stream_bit = [&](long long q) -> int { return (q < nb_old) ? ((pb_old >> (nb_old - 1 - (int)q)) & 1) : (int)rx[q - nb_old]; };
  if (S.ring_count + appended > a.ring_cap) {                    // RingTryWriteByte fails :96-104 -> :241-246
    framer_reset(S);
    if (lane == 0) a.st[c] = S;
    return;
  }
  for (long long j = lane; j < appended; j += 32) {
    int v = 0;
#pragma unroll
    for (int t = 0; t < 8; ++t) v = (v << 1) | stream_bit(8 * j + t);
    ring[S.ring_count + j] = (uint8_t)v;
  }
  int pb = 0;
  for (long long q = 8 * appended; q < total; ++q) pb = (pb << 1) | stream_bit(q);
  S.pack_byte = pb;
  S.pack_bits = (int)(total & 7);
  S.ring_count += appended;
  __syncwarp();
  const long long end_at = framer_ring_index_of(ring, S.ring_count, em, a.ne, S.ring_count - (appended + a.ne), lane);
  if (end_at >= 0) {
    framer_emit(a, c, ring, end_at, lane);
    framer_reset(S);
  }
  if (lane == 0) a.st[c] = S;
}

__global__ void bits_to_chars_kernel(const uint8_t* in, char* out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = in[i] ? '1' : '0';
}

// ---------------------------------------------------------------------------------------------
// DemodEngine
// ---------------------------------------------------------------------------------------------
constexpr int kMaxMarkerBytes = 256;

// samples still in HOST memory: the chain then runs as a pipeline over time chunks — the copy of chunk t+1 (and, for CS16,
// its widening to cf32) is in flight on the side stream while the chain works on chunk t
struct HostSrc {
  const void* p = nullptr;      // [channels][ld] complex samples: float2, or int16 pairs when cs16
  int64_t ld = 0;               // complex samples between consecutive channels
  bool cs16 = false;
  float scale = 1.0f;           // cf32 = (float)int16 * scale
  bool pageable = false;        // the driver does not know the memory as page-locked: chunks go through h_bounce
};
int cs16_to_cf32_launch(const int16_t* d_in, long long ld_in, float scale, float2* d_out, long long ld_out, long long L, int channels,
                        cudaStream_t s);   // stream.cu

struct DemodEngine {
  int channels = 1;
  int device = 0;              // every entry point selects it (handles own their device, qpskcuda.h)
  bool diff = true, has_tsc = false, use_fll = false;
  std::string tsc;
  double sps = 0.0;
  int int_sps = 0;             // fs / rs when rs divides fs, else 0 (the fractionally spaced stage needs an integer rate)
  FirEngine mf;
  FllEngine fll;
  MmEngine mm;
  CostasEngine costas;
  std::unique_ptr<EqEngine> eq;    // opt-in CMA stage between MM and Costas (qpsk_demod_set_equalizer); null = off
  // opt-in T/sps-spaced CMA stage between the matched filter and MM (qpsk_demod_set_fractional_equalizer); null = off
  std::unique_ptr<EqEngine> fse;
  int64_t fse_drop = 0;            // outputs the stage still discards: the same for every channel (every call feeds all L)
  // opt-in feed-forward AGC ahead of everything else (qpsk_demod_set_agc); null = off.  It writes t_agc, which the
  // unchanged path then reads in place of the input.
  std::unique_ptr<AgcEngine> agc;
  int64_t agc_drop = 0;            // AGC outputs still to discard (W-1 once per stream), the same for every channel
  DevBuf<float2> t_fll, t_rrc, t_sym, t_eq, t_fse, t_agc;
  DevBuf<int> d_nsym, d_neq, d_ncon;   // d_ncon: symbol counts of qpsk_demod_constellation
  DevBuf<uint8_t> d_raw, d_tsc, d_bits, d_markers, d_carry, d_ring, d_pk, d_payload;
  DevBuf<long long> d_nraw, d_nbits, d_npayload;
  DevBuf<DiffState> d_diff;
  DevBuf<FramerState> d_framer;
  DevBuf<float2> h_in, h_out;       // device staging for the host entry points
  DevBuf<int16_t> h_cs16;           // CS16 staging ([channels][2*ld] int16)
  std::vector<uint8_t> markers_host;
  std::vector<long long> last_np;   // payload lengths of the last host framer call (qpsk_demod_last_payload)
  long long ring_cap = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t side = nullptr;               // front-end stream of the time-chunk pipeline
  cudaStream_t copy = nullptr;               // host-source calls: the PCIe copies (and the CS16 widening) of the chunks
  cudaEvent_t ev_in = nullptr;
  std::vector<cudaEvent_t> ev_chunk, ev_copy;
  // page-locked landing zone of the host entry points' results: a 2-D device-to-host copy into PAGEABLE caller memory goes
  // row by row through the driver's bounce buffer (2048 rows of ~540 bytes: 0.3-0.8 ms, a third of a DeModulateBytes call);
  // one contiguous copy into this buffer and a memcpy per row cost ~0.1 ms
  uint8_t* h_land = nullptr;
  size_t h_land_bytes = 0;
  int landing(size_t bytes) {
    if (bytes <= h_land_bytes) return QPSK_OK;
    if (h_land) cudaFreeHost(h_land);
    h_land = nullptr;
    h_land_bytes = 0;
    QPSK_CUDA_TRY(cudaHostAlloc((void**)&h_land, bytes, cudaHostAllocPortable));
    h_land_bytes = bytes;
    return QPSK_OK;
  }
  // The result tail of the host entry points: the per-channel counts d_n[C] to n[C], then the rows `ld_dev` bytes apart on
  // the device to rows `cap` bytes apart in caller memory, in one copy as wide as the widest row that fits (a row's bytes
  // past its own count are unspecified, like the rest of the caller's buffer).  A row is `bits` bits per count; one
  // longer than `cap` bytes is not copied and makes the call QPSK_ERR_CAPACITY, its count still reported.  `prep` runs on
  // `s` first, when there is a row to copy.  Synchronises `s`.
  template <typename Count>
  int fetch_results(const Count* d_n, int64_t* n, int bits, void* out, int64_t cap, const void* dev, size_t ld_dev,
                    cudaStream_t s, const std::function<int()>& prep = nullptr) {
    std::vector<Count> h((size_t)channels);
    QPSK_CUDA_TRY(cudaMemcpyAsync(h.data(), d_n, sizeof(Count) * channels, cudaMemcpyDeviceToHost, s));
    QPSK_CUDA_TRY(cudaStreamSynchronize(s));
    int st = QPSK_OK;
    long long widest = 0;
    for (int c = 0; c < channels; ++c) {
      n[c] = h[(size_t)c];
      const long long bytes = ((long long)h[(size_t)c] * bits + 7) / 8;
      if (bytes > cap) st = QPSK_ERR_CAPACITY;
      else if (bytes > widest) widest = bytes;
    }
    if (widest == 0) return st;
    if (!out) return QPSK_ERR_NULL;
    if (prep) QPSK_TRY(prep());
    const size_t width = (size_t)widest;
    QPSK_TRY(landing(width * (size_t)channels));
    QPSK_CUDA_TRY(cudaMemcpy2DAsync(h_land, width, dev, ld_dev, width, (size_t)channels, cudaMemcpyDeviceToHost, s));
    QPSK_CUDA_TRY(cudaStreamSynchronize(s));
    for (int c = 0; c < channels; ++c) memcpy((uint8_t*)out + (size_t)c * (size_t)cap, h_land + (size_t)c * width, width);
    return st;
  }

  ~DemodEngine() {
    if (stream) cudaStreamDestroy(stream);
    if (side) cudaStreamDestroy(side);
    if (copy) cudaStreamDestroy(copy);
    if (h_land) cudaFreeHost(h_land);
    if (h_bounce) cudaFreeHost(h_bounce);
    if (ev_in) cudaEventDestroy(ev_in);
    for (cudaEvent_t e : ev_chunk) cudaEventDestroy(e);
    for (cudaEvent_t e : ev_copy) cudaEventDestroy(e);
  }

  int init(int fs, int rs, float alpha, int span, double sym_bw, double costas_bw, double cfo_bw, int diff_in,
           const char* tsc_in, int use_fll_in, int64_t max_frame_bytes, int channels_in) {
    if (channels_in <= 0) return QPSK_ERR_RANGE;
    if (rs == 0) return QPSK_ERR_RANGE;                        // DivideByZeroException upstream
    QPSK_TRY(ensure_device());
    device = current_device();
    channels = channels_in;
    diff = diff_in != 0;
    use_fll = use_fll_in != 0;
    has_tsc = !blank_or_null(tsc_in);                          // :21
    if (has_tsc) tsc = tsc_in;
    sps = (double)fs / (double)rs;
    int_sps = (fs % rs == 0) ? fs / rs : 0;
    QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    const std::vector<double> h = design_rrc((double)span, (double)alpha, fs, rs);   // :28-32
    const std::vector<float> iq = real_taps_as_iq(h);
    QPSK_TRY(mf.init(iq.data(), (int)iq.size(), channels));
    // demodulated bits are compared bit for bit with the reference: the matched filter defaults to the reference's own
    // summation order (FIRFilter.cs:165-192); QPSK_FIR_FAST (FMA accumulation, ~1e-7 relative) is the opt-in
    mf.mode = QPSK_FIR_EXACT;
    QPSK_TRY(fll.init((float)(fs / rs), alpha, 40, (float)cfo_bw, channels));        // :35 (integer division)
    double kp, ki;
    mm_gains(sym_bw, &kp, &ki);                                // :39-55
    QPSK_TRY(mm.init(sps, kp, ki, channels));
    QPSK_TRY(costas.init((double)rs, (double)rs / costas_bw, 0.707, channels));      // :56
    QPSK_TRY(d_nsym.alloc((size_t)channels));
    QPSK_TRY(d_nraw.alloc((size_t)channels));
    QPSK_TRY(d_nbits.alloc((size_t)channels));
    QPSK_TRY(d_npayload.alloc((size_t)channels));
    QPSK_TRY(d_diff.alloc((size_t)channels));
    QPSK_TRY(d_framer.alloc((size_t)channels));
    QPSK_TRY(d_diff.zero(stream));
    QPSK_TRY(d_framer.zero(stream));
    if (has_tsc) {
      std::vector<uint8_t> t;
      for (char ch : tsc) t.push_back((uint8_t)(ch == '0' ? 0 : (ch == '1' ? 1 : 2)));
      QPSK_TRY(d_tsc.alloc(t.size()));
      QPSK_CUDA_TRY(cudaMemcpyAsync(d_tsc.p, t.data(), t.size(), cudaMemcpyHostToDevice, stream));
      QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    }
    ring_cap = max_frame_bytes > 0 ? max_frame_bytes : (1LL << 20);
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    return QPSK_OK;
  }

  // most symbols one call can emit: every symbol advances time by >= sps - 0.1 (MuellerMuller.cs:87-89)
  long long symbols_bound(int64_t L) const {
    if (sps - 0.1 <= 1.0) return L;
    long long b = (long long)((double)(L + 4) / (sps - 0.1)) + 2;
    return b < L ? b : L;
  }
  long long bits_bound(int64_t L) const { return 2 * symbols_bound(L); }

  // switches an opt-in stage once both streams are idle: off (`on` false), or a fresh one set up by init(stage)
  template <typename E, typename Init>
  int replace_stage(std::unique_ptr<E>& stage, bool on, Init init) {
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    if (side) QPSK_CUDA_TRY(cudaStreamSynchronize(side));
    if (!on) {
      stage.reset();
      return QPSK_OK;
    }
    std::unique_ptr<E> e(new (std::nothrow) E());
    if (!e) return QPSK_ERR_NOMEM;
    QPSK_TRY(init(*e));
    stage = std::move(e);
    return QPSK_OK;
  }
  // opt-in equalizer stage: n_taps 0 = off; otherwise a fresh equalizer (spike taps, zero window, discard count D)
  int set_equalizer(int n_taps, float mu, float modulus) {
    if (n_taps != 0) QPSK_TRY(eq_check_params(n_taps, mu, modulus, 1));
    return replace_stage(eq, n_taps != 0, [&](EqEngine& e) {
      QPSK_TRY(e.init(n_taps, mu, modulus, 1, channels));
      return d_neq.ensure((size_t)channels);
    });
  }
  // opt-in fractionally spaced stage, update stride S = fs / rs: n_taps 0 = off; otherwise a fresh equalizer (spike taps,
  // zero window, sample counter 0, discard count D)
  int set_fractional_equalizer(int n_taps, float mu, float modulus) {
    if (n_taps != 0) {
      if (int_sps < 2 || int_sps > kEqMaxSps) return QPSK_ERR_UNSUPPORTED;
      QPSK_TRY(eq_check_params(n_taps, mu, modulus, int_sps));
    }
    return replace_stage(fse, n_taps != 0, [&](EqEngine& e) {
      QPSK_TRY(e.init(n_taps, mu, modulus, int_sps, channels));
      fse_drop = (n_taps - 1) / 2;
      return QPSK_OK;
    });
  }
  // opt-in AGC stage: window 0 = off; otherwise a fresh AGC (zero history, discard count W-1)
  int set_agc(int window, float ref, float max_gain) {
    if (window != 0) QPSK_TRY(agc_check_params(window, ref, max_gain));
    return replace_stage(agc, window != 0, [&](AgcEngine& a) {
      QPSK_TRY(a.init(window, ref, max_gain, channels));
      agc_drop = window - 1;
      return QPSK_OK;
    });
  }

  // Time-chunk pipeline of bits_dev (FLL path): number of chunks for an L-sample call.  Short calls stay on one stream: the
  // split costs two launches and a warm-up per chunk.  The channel count does not matter: a single stream gains as much as
  // a full batch (1.10 -> 0.84 ms for 4196 samples), because the FLL and the symbol stages are each latency-bound on their
  // own warps.
  int pipeline_chunks(int64_t L) const {
    // six chunks while the FLL is latency-bound (1.22 -> 1.15 ms per step at 2048 channels: a shorter exposed tail); four once
    // it is issue-bound and every extra launch pair costs more than the tail it hides (8192 channels: 2.22 against 2.32 ms)
    int n = channels <= 4096 ? 6 : 4;
    if (L < 2048) n = 1;
    while (n > 1 && L < (int64_t)n * 8 * kSsBlock) --n;
    return n;
  }
  // host-source calls: chunks of >= 8 MiB of samples, at most 6 — every chunk is a 2-D copy of `channels` row pieces, and short
  // pieces cost PCIe efficiency (2048 channels x 4380 samples, Gsample/s end to end at 1 / 2 / 4 / 6 / 8 / 16 chunks: cf32 4.25 /
  // 4.91 / 5.11 / 5.13 / 5.07 / 4.96, CS16 6.03 / 7.00 / 7.47 / 7.39 / 7.17 / 6.69)
  int host_chunks(int64_t L, bool cs16) const {
    const double bytes = (double)L * channels * (cs16 ? 4.0 : 8.0);
    int n = (int)(bytes / (8.0 * 1024 * 1024));
    if (n > 6) n = 6;
    if (n < 1) n = 1;
    while (n > 1 && L < (int64_t)n * 8 * kSsBlock) --n;
    return n;
  }
  // copy (and widen) samples [n0, n0+len) of every channel from the host source into h_in, on stream `st`.  Pageable
  // sources: an asynchronous copy on them blocks the calling thread in the driver's own staging; the row pieces are gathered
  // into a page-locked mirror of the block by the host copy pool instead (common.cuh) and leave from there.
  int stage_host_chunk(const HostSrc& hs, int64_t n0, int64_t len, int64_t ld, cudaStream_t st) {
    const size_t esz = hs.cs16 ? 4 : 8;                      // bytes per complex sample on the host
    const char* src = (const char*)hs.p + (size_t)n0 * esz;
    size_t spitch = (size_t)hs.ld * esz;
    if (hs.pageable && h_bounce) {
      char* mirror = (char*)h_bounce + (size_t)n0 * esz;
      host_parallel_copy_rows(mirror, spitch, src, spitch, (size_t)len * esz, (size_t)channels);
      src = mirror;
    }
    if (!hs.cs16) {
      QPSK_CUDA_TRY(cudaMemcpy2DAsync(h_in.p + n0, (size_t)ld * 8, src, spitch, (size_t)len * 8, (size_t)channels,
                                      cudaMemcpyHostToDevice, st));
      return QPSK_OK;
    }
    QPSK_CUDA_TRY(cudaMemcpy2DAsync(h_cs16.p + 2 * n0, (size_t)ld * 4, src, spitch, (size_t)len * 4, (size_t)channels,
                                    cudaMemcpyHostToDevice, st));
    return cs16_to_cf32_launch(h_cs16.p + 2 * n0, ld, hs.scale, h_in.p + n0, ld, len, channels, st);
  }
  // page-locked mirror of a pageable host block (up to 512 MiB; larger blocks stay on the driver's pageable path)
  void* h_bounce = nullptr;
  size_t h_bounce_bytes = 0;
  int ensure_bounce(size_t bytes) {
    if (bytes > ((size_t)512 << 20)) {
      if (h_bounce) cudaFreeHost(h_bounce);
      h_bounce = nullptr;
      h_bounce_bytes = 0;
      return QPSK_OK;
    }
    if (bytes <= h_bounce_bytes) return QPSK_OK;
    if (h_bounce) cudaFreeHost(h_bounce);
    h_bounce = nullptr;
    h_bounce_bytes = 0;
    QPSK_CUDA_TRY(cudaHostAlloc(&h_bounce, bytes, cudaHostAllocPortable));
    h_bounce_bytes = bytes;
    return QPSK_OK;
  }
  int ensure_pipeline(int chunks, bool from_host) {
    if (!side) QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&side, cudaStreamNonBlocking));
    if (from_host && !copy) QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    if (!ev_in) QPSK_CUDA_TRY(cudaEventCreateWithFlags(&ev_in, cudaEventDisableTiming));
    while ((int)ev_chunk.size() < chunks) {
      cudaEvent_t e = nullptr;
      QPSK_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ev_chunk.push_back(e);
    }
    while (from_host && (int)ev_copy.size() < chunks) {
      cudaEvent_t e = nullptr;
      QPSK_CUDA_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
      ev_copy.push_back(e);
    }
    return QPSK_OK;
  }

  // the fused MM -> Costas -> decode kernel applies when no call can run out of output room and the MM
  // queue holds at most kSsCarry samples (always true once every call has had room)
  bool can_fuse() const { return !eq && !fse && (sps - 0.1 > 1.0) && mm.q_bound <= kSsCarry; }
  // ... and it takes the matched filter in as well (MFW extra warps, see symsync_decode_kernel) when the filter runs in
  // the reference's summation order (the demodulator's default), has real taps and at most 65 of them.
  bool can_fuse_mf() const {
    // a lone CTA gains nothing from the fusion (the separate filter launch costs ~5 us) and its rounds run ~10 % slower
    // with the filter warps on board: one radio stream (qpsk_stream_*, per-call DeModulateBytes) keeps the separate kernel
    if (channels < 32) return false;
    return mf.mode == QPSK_FIR_EXACT && mf.real_taps && mf.n_taps <= kMfMaxTaps && mf.n_taps >= 1;
  }
  // matched-filter warps per 32-channel CTA.  One round costs a Mueller-Muller warp ~340 cycles per symbol; the filter
  // needs ~70 issue slots per tap for the round's 32 outputs.  Two filter warps while the estimate below fits in 60 % of a
  // round, else four.
  int mf_warps() const {
    const double round_cycles = 340.0 * (double)kSsBlock / sps;
    const double mf_slots = 110.0 * mf.n_taps;       // issue slots for the 32 outputs of one round (~3.4 per tap and output)
    return (mf_slots <= 0.6 * round_cycles) ? 2 : 4;
  }

  // one launch of the symbol-stage kernel over `len` samples at `xin` (matched-filter output, or — with_mf — its input)
  int launch_symsync(const float2* xin, int64_t len, int64_t ldin, uint8_t* raw, long long ld_raw, long long* n_raw, int append,
                     bool with_mf, cudaStream_t s) {
    MfTaps mt;
    memset(&mt, 0, sizeof mt);
    MfArgs ma;
    ma.hist_in = nullptr; ma.hist_out = nullptr; ma.HL = 0;
    const int grid = (channels + 31) / 32;
    // most symbols one round of kSsBlock samples (+ the carried ones) can emit: every symbol advances >= sps - 0.1
    int sym_cap = (int)((double)(kSsBlock + kSsCarry) / (sps - 0.1)) + 2;
    if (sym_cap > kSsSymCap) sym_cap = kSsSymCap;
    const int sym_pitch = (sym_cap + 1) | 1;         // + 1: the decode loop reads one slot ahead; odd: bank spread
    const int ring_n = (mf.n_taps - 1 <= 32) ? 96 : 128;
    const size_t symq_bytes = (size_t)2 * 32 * sym_pitch * sizeof(float2);
#define QPSK_SS_ARGS mm.P, mm.d_state.p, mm.d_queue[mm.qcur].p, mm.d_queue[mm.qcur ^ 1].p, mm.qcap, costas.P, costas.d_state.p, \
                     d_diff.p, channels, xin, len, ldin, raw, ld_raw, n_raw, d_nsym.p, append, mt, ma, ring_n, sym_pitch
    if (!with_mf) {
      if (diff) symsync_decode_kernel<true, 0><<<grid, 64, symq_bytes, s>>>(QPSK_SS_ARGS);
      else symsync_decode_kernel<false, 0><<<grid, 64, symq_bytes, s>>>(QPSK_SS_ARGS);
    } else {
      const int N = mf.n_taps;
      mt.n_taps = N;
      for (int i = 0; i < N; ++i) mt.rev[i] = mf.taps_iq[2 * (N - 1 - i)];
      ma.hist_in = mf.hist[mf.cur].p; ma.hist_out = mf.hist[mf.cur ^ 1].p; ma.HL = mf.HL;
      const size_t smem = symq_bytes + (size_t)32 * (ring_n + 1) * sizeof(float2);
      const int w = mf_warps();
      decltype(&symsync_decode_kernel<false, 4>) kern;
      if (w == 4) kern = diff ? symsync_decode_kernel<true, 4> : symsync_decode_kernel<false, 4>;
      else if (grid > 3 * device_sm_count()) kern = diff ? symsync_decode_kernel<true, 2, true> : symsync_decode_kernel<false, 2, true>;
      else kern = diff ? symsync_decode_kernel<true, 2> : symsync_decode_kernel<false, 2>;
      QPSK_TRY(allow_max_dynamic_smem((const void*)kern));
      kern<<<grid, 64 + 32 * w, smem, s>>>(QPSK_SS_ARGS);
      mf.cur ^= 1;                                   // the kernel left the advanced delay line in the other buffer
    }
#undef QPSK_SS_ARGS
    QPSK_LAUNCH_CHECK();
    mm.qcur ^= 1;
    mm.q_bound = 4;
    return QPSK_OK;
  }

  // What one call runs and the sizes it works in, fixed before its first launch.  Every route runs the same loop over
  // `chunks` time chunks (front_chunk, then the symbol stage of the chunk); a single launch is the one-chunk case.
  struct CallPlan {
    bool fused = false;          // the symbol stage is symsync_decode_kernel (else FSE -> MM -> EQ -> decode_kernel)
    bool fuse_mf = false;        // ... with the matched filter inside it
    bool from_host = false;      // samples staged from `hs` into h_in chunk by chunk
    int chunks = 1;
    HostSrc hs;
    int64_t ld = 0;              // pitch of every scratch row of the call
    int64_t agc_dc = 0;          // leading samples of the call the AGC discards
    long long sym_ld = 1;        // symbol rows
  };
  // refuses nothing: the callers check their arguments first, and the plan only sizes scratch and picks the route
  int plan(CallPlan& p, int64_t L, const HostSrc* hs, bool fused) {
    p.fused = fused;
    p.fuse_mf = fused && can_fuse_mf();
    p.from_host = hs != nullptr && hs->p != nullptr;
    p.chunks = (fused && use_fll) ? pipeline_chunks(L) : 1;
    if (fused && p.from_host) p.chunks = std::max(p.chunks, host_chunks(L, hs->cs16));
    p.ld = L + (L & 1);
    p.agc_dc = agc ? std::min(agc_drop, L) : 0;
    // a single launch sizes the symbol rows from the samples it keeps: Mueller-Muller's room rule reads that size (and
    // with it how many symbols a call leaves queued for the next one)
    p.sym_ld = std::max(1LL, symbols_bound(p.chunks > 1 ? L : L - p.agc_dc));
    const size_t rows = (size_t)p.ld * channels;
    if (p.from_host) {
      p.hs = *hs;
      p.hs.pageable = host_ptr_is_pageable(hs->p);
      QPSK_TRY(h_in.ensure(rows));
      if (hs->cs16) QPSK_TRY(h_cs16.ensure(2 * rows));
      if (p.hs.pageable) QPSK_TRY(ensure_bounce((size_t)channels * (size_t)hs->ld * (hs->cs16 ? 4 : 8)));
    }
    if (agc) QPSK_TRY(t_agc.ensure(rows));
    if (use_fll) QPSK_TRY(t_fll.ensure(rows));
    if (!p.fuse_mf) QPSK_TRY(t_rrc.ensure(rows));
    if (!fused) {
      QPSK_TRY(t_sym.ensure((size_t)p.sym_ld * channels));
      if (fse) QPSK_TRY(t_fse.ensure(rows));
      if (eq) QPSK_TRY(t_eq.ensure((size_t)p.sym_ld * channels));
    }
    if (p.chunks > 1) QPSK_TRY(ensure_pipeline(p.chunks, p.from_host));
    return QPSK_OK;
  }

  // The front end of time chunk t, samples [n0, n0 + len) of the call: staged from the host (from_host) -> AGC -> its
  // discard -> FLL -> matched filter (unless the symbol stage runs it).  The AGC writes the chunk's outputs from column n0
  // of t_agc, so the kept ones sit at n0 + skip; the FLL and the filter write theirs from column n0.  x / ldx (the call's
  // device source) come back pointing at what the symbol stage reads, len as the number of samples kept.  In the
  // pipeline it runs on the side stream and the host copies on the copy stream, and the caller's stream waits for it.
  int front_chunk(const CallPlan& p, int t, int64_t n0, int64_t& len, const float2*& x, int64_t& ldx, cudaStream_t s) {
    const bool pipe = p.chunks > 1;
    cudaStream_t fs = pipe ? side : s;
    if (p.from_host) {
      QPSK_TRY(stage_host_chunk(p.hs, n0, len, p.ld, pipe ? copy : s));   // pageable source: the host gathers the chunk first
      if (pipe) {
        QPSK_CUDA_TRY(cudaEventRecord(ev_copy[(size_t)t], copy));
        QPSK_CUDA_TRY(cudaStreamWaitEvent(side, ev_copy[(size_t)t], 0));
      }
      x = h_in.p;
      ldx = p.ld;
    }
    x += n0;
    if (agc) {
      QPSK_TRY(agc->process_dev(x, len, ldx, t_agc.p + n0, p.ld, fs));
      const int64_t skip = p.agc_dc > n0 ? std::min(p.agc_dc - n0, len) : 0;
      agc_drop -= skip;
      len -= skip;
      x = t_agc.p + n0 + skip;
      ldx = p.ld;
    }
    if (len > 0 && use_fll) {
      QPSK_TRY(fll.process_dev(x, t_fll.p + n0, len, ldx, p.ld, fs));   // the call at :359
      x = t_fll.p + n0;
      ldx = p.ld;
    }
    if (len > 0 && !p.fuse_mf) {
      QPSK_TRY(mf.filter_dev(x, t_rrc.p + n0, len, ldx, p.ld, fs));     // :360
      x = t_rrc.p + n0;
      ldx = p.ld;
    }
    if (pipe) {
      QPSK_CUDA_TRY(cudaEventRecord(ev_chunk[(size_t)t], side));
      QPSK_CUDA_TRY(cudaStreamWaitEvent(s, ev_chunk[(size_t)t], 0));
    }
    return QPSK_OK;
  }

  // [FSE ->] MM [-> EQ] over the matched-filter output of an unfused call (one chunk, len samples at x / ldx): the
  // symbols Costas reads, sym [C][sym_ld], and their counts
  int symbols(const CallPlan& p, const float2* x, int64_t len, int64_t ldx, const float2*& sym, const int*& nsym,
              cudaStream_t s) {
    int64_t mm_n = len;
    if (fse) {
      // every channel takes len samples, so every channel discards the same dc: MM takes len - dc samples of each row
      QPSK_TRY(fse->process_dev(x, t_fse.p, len, ldx, p.ld, nullptr, nullptr, true, s));
      const int64_t dc = std::min(fse_drop, len);
      fse_drop -= dc;
      x = t_fse.p;
      ldx = p.ld;
      mm_n = len - dc;
    }
    QPSK_TRY(mm.process_dev(x, mm_n, ldx, t_sym.p, 2 * len, p.sym_ld, d_nsym.p, s));   // :364-367
    sym = t_sym.p;
    nsym = d_nsym.p;
    if (eq) {
      QPSK_TRY(eq->process_dev(t_sym.p, t_eq.p, p.sym_ld, p.sym_ld, p.sym_ld, d_nsym.p, d_neq.p, true, s));
      sym = t_eq.p;
      nsym = d_neq.p;
    }
    return QPSK_OK;
  }

  // DeModulate: bits (bytes 0/1) to out [C][ld_out], counts to n_out[C]
  // hs != nullptr: the samples are in host memory (x / ldx ignored): staged into h_in chunk by chunk
  int bits_dev(const float2* x, int64_t L, int64_t ldx, uint8_t* out, int64_t ld_out, long long* n_out, cudaStream_t s,
               const HostSrc* hs = nullptr) {
    if (L == 0) {
      QPSK_CUDA_TRY(cudaMemsetAsync(n_out, 0, sizeof(long long) * channels, s));   // :350-351
      return QPSK_OK;
    }
    // every check comes BEFORE the first stage that advances state (AGC history, FLL ring, matched-filter delay line, MM
    // queue, loop state): a refused call must leave the stream where it was
    if (ld_out < 2 * std::max(1LL, symbols_bound(L))) return QPSK_ERR_CAPACITY;
    // uchar2 stores; with a TSC the symbol stage writes the engine's own 16-byte rows
    if (!has_tsc && ((reinterpret_cast<uintptr_t>(out) & 1) || (ld_out & 1))) return QPSK_ERR_ARG;
    CallPlan p;
    QPSK_TRY(plan(p, L, hs, can_fuse()));
    uint8_t* raw = out;
    long long ld_raw = ld_out;
    long long* n_raw = n_out;
    if (has_tsc) {
      ld_raw = (2 * p.sym_ld + 15) & ~15LL;
      QPSK_TRY(d_raw.ensure((size_t)ld_raw * channels));
      raw = d_raw.p;
      n_raw = d_nraw.p;
    }
    if (p.chunks > 1) {
      // the time-chunk pipeline: the front end of chunk t+1 on the side stream while the symbol stage of chunk t runs on
      // the caller's.  Every stage carries its state from chunk to chunk exactly (AGC history, FLL ring/phase, MF delay
      // line, MM queue, Costas, differential reference), so the split changes nothing but the schedule.
      QPSK_CUDA_TRY(cudaEventRecord(ev_in, s));
      QPSK_CUDA_TRY(cudaStreamWaitEvent(side, ev_in, 0));     // inputs (and the previous call) are complete
      // the PCIe copies run on a stream of their own: chunk t+1 crosses the bus while the FLL (side stream) works on chunk t
      // and the symbol stage (caller's stream) on chunk t-1.  On the side stream they would queue behind the FLL launches:
      // copy and FLL would take turns (3.3 ms per step where 1.3 + tail is possible).
      if (p.from_host) QPSK_CUDA_TRY(cudaStreamWaitEvent(copy, ev_in, 0));
    }
    // equal chunks except a half-size last one: the FLL on the side stream is the critical resource throughout, so what is
    // left exposed at the end is the last chunk's symbol stage.  One chunk: the whole call.
    const int chunks = p.chunks;
    const int64_t step = ((2 * L + 2 * chunks - 2) / (2 * chunks - 1) + kSsBlock - 1) / kSsBlock * kSsBlock;
    bool launched = false;
    int t = 0;
    for (int64_t n0 = 0; n0 < L; n0 += step, ++t) {
      int64_t len = std::min(step, L - n0);
      const float2* y = x;
      int64_t ldy = ldx;
      QPSK_TRY(front_chunk(p, t, n0, len, y, ldy, s));
      if (len == 0) continue;
      if (p.fused) {
        QPSK_TRY(launch_symsync(y, len, ldy, raw, ld_raw, n_raw, launched ? 1 : 0, p.fuse_mf, s));
      } else {
        const float2* sym;
        const int* nsym;
        QPSK_TRY(symbols(p, y, len, ldy, sym, nsym, s));
        decode_kernel<<<(channels + 31) / 32, 32, 0, s>>>(costas.P, costas.d_state.p, d_diff.p, channels, sym, p.sym_ld, nsym,
                                                          diff ? 1 : 0, raw, ld_raw, n_raw);
        QPSK_LAUNCH_CHECK();
      }
      launched = true;
    }
    if (!launched) {                                 // the AGC discarded every sample of the call
      if (chunks == 1) {
        QPSK_CUDA_TRY(cudaMemsetAsync(n_out, 0, sizeof(long long) * channels, s));
        return QPSK_OK;
      }
      QPSK_CUDA_TRY(cudaMemsetAsync(n_raw, 0, sizeof(long long) * channels, s));
    }
    if (has_tsc) {
      const int T = (int)tsc.size();
      const long long row_bytes = (ld_raw + 15) & ~15LL;
      const int words_per_row = (int)((row_bytes + 31) / 32 + 4);          // packed bits of a row + two zero words
      const size_t smem = (size_t)4 * (row_bytes + ((T + 15) & ~15)) + (size_t)4 * words_per_row * sizeof(uint32_t);
      if (smem <= 160 * 1024 && (ld_raw & 15) == 0) {
        QPSK_TRY(allow_max_dynamic_smem((const void*)tsc_strip_smem_kernel));
        tsc_strip_smem_kernel<<<(channels + 3) / 4, 128, smem, s>>>(raw, ld_raw, n_raw, d_tsc.p, T, out, ld_out, n_out, channels,
                                                                   (int)row_bytes, words_per_row);
      } else {
        tsc_strip_kernel<<<(channels + 3) / 4, 128, 0, s>>>(raw, ld_raw, n_raw, d_tsc.p, T, out, ld_out, n_out, channels);
      }
      QPSK_LAUNCH_CHECK();
    }
    return QPSK_OK;
  }

  // symbols after Costas (:447-452) to out [C][ld_out], counts to n_out[C]; hs as for bits_dev
  int constellation_dev(const float2* x, int64_t L, int64_t ldx, float2* out, int64_t ld_out, int* n_out, cudaStream_t s,
                        const HostSrc* hs = nullptr) {
    if (L == 0) {
      QPSK_CUDA_TRY(cudaMemsetAsync(n_out, 0, sizeof(int) * channels, s));
      return QPSK_OK;
    }
    if (ld_out < std::max(1LL, symbols_bound(L))) return QPSK_ERR_CAPACITY;   // refuse before any stage consumes the samples
    CallPlan p;
    QPSK_TRY(plan(p, L, hs, false));
    int64_t len = L;
    QPSK_TRY(front_chunk(p, 0, 0, len, x, ldx, s));
    if (len == 0) {                                  // the AGC discarded every sample of the call
      QPSK_CUDA_TRY(cudaMemsetAsync(n_out, 0, sizeof(int) * channels, s));
      return QPSK_OK;
    }
    const float2* sym;
    const int* nsym;
    QPSK_TRY(symbols(p, x, len, ldx, sym, nsym, s));
    QPSK_TRY(costas.process_dev(sym, out, p.sym_ld, p.sym_ld, ld_out, nsym, s));   // :447-452
    QPSK_CUDA_TRY(cudaMemcpyAsync(n_out, nsym, sizeof(int) * channels, cudaMemcpyDeviceToDevice, s));
    return QPSK_OK;
  }

  int upload_markers(const uint8_t* sm, int64_t ns, const uint8_t* em, int64_t ne, cudaStream_t s) {
    std::vector<uint8_t> m(sm, sm + ns);
    m.insert(m.end(), em, em + ne);
    if (m != markers_host || !d_markers.p) {
      QPSK_CUDA_TRY(cudaStreamSynchronize(s));
      QPSK_TRY(d_markers.ensure(m.size()));
      markers_host = m;
      QPSK_CUDA_TRY(cudaMemcpyAsync(d_markers.p, markers_host.data(), markers_host.size(), cudaMemcpyHostToDevice, s));
    }
    return QPSK_OK;
  }

  // DeModulateBytes: payload bytes to payload [C][cap], full lengths to n_payload[C]
  int bytes_dev(const float2* x, int64_t L, int64_t ldx, const uint8_t* sm, int64_t ns, const uint8_t* em, int64_t ne,
                uint8_t* payload, int64_t cap, long long* n_payload, cudaStream_t s, const HostSrc* hs = nullptr) {
    if (ns == 0 || ne == 0) return QPSK_ERR_ARG;               // :174-175
    if (!sm || !em) return QPSK_ERR_NULL;
    if (ns > kMaxMarkerBytes || ne > kMaxMarkerBytes) return QPSK_ERR_UNSUPPORTED;
    const long long ldb = bits_bound(L) + 2;
    QPSK_TRY(d_bits.ensure((size_t)ldb * channels));
    QPSK_TRY(bits_dev(x, L, ldx, d_bits.p, ldb, d_nbits.p, s, hs));
    return frame_dev(d_bits.p, ldb, d_nbits.p, sm, ns, em, ne, payload, cap, n_payload, s);
  }

  // the framer of DeModulateBytes (:182-259) over bits [C][ldb] (one 0/1 byte each), n_bits[C] of them per channel
  int frame_dev(const uint8_t* bits, long long ldb, const long long* n_bits, const uint8_t* sm, int64_t ns, const uint8_t* em,
                int64_t ne, uint8_t* payload, int64_t cap, long long* n_payload, cudaStream_t s) {
    if (ns == 0 || ne == 0) return QPSK_ERR_ARG;               // :174-175
    if (!sm || !em) return QPSK_ERR_NULL;
    if (ns > kMaxMarkerBytes || ne > kMaxMarkerBytes) return QPSK_ERR_UNSUPPORTED;
    QPSK_TRY(upload_markers(sm, ns, em, ne, s));
    const int carry_cap = kMaxMarkerBytes * 8 + 8;
    if (!d_carry.p) {
      QPSK_TRY(d_carry.alloc((size_t)carry_cap * channels));
      QPSK_TRY(d_ring.alloc((size_t)ring_cap * channels));
    }
    const long long pk_ld = ((carry_cap + ldb) >> 3) + 4;
    QPSK_TRY(d_pk.ensure((size_t)pk_ld * channels));
    FramerArgs a;
    a.st = d_framer.p; a.carry = d_carry.p; a.carry_cap = carry_cap; a.ring = d_ring.p; a.ring_cap = ring_cap;
    a.pk = d_pk.p; a.pk_ld = pk_ld; a.rx = bits; a.ld_rx = ldb; a.n_rx = n_bits; a.markers = d_markers.p;
    a.ns = (int)ns; a.ne = (int)ne; a.payload = payload; a.payload_cap = cap; a.n_payload = n_payload; a.C = channels;
    framer_kernel<<<(channels + kFramerWarps - 1) / kFramerWarps, 32 * kFramerWarps, 0, s>>>(a);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }
};

}  // namespace qpsk

using namespace qpsk;

struct qpsk_demod {
  DemodEngine eng;
};

extern "C" {

int qpsk_demod_create_batch(int sample_rate, int symbol_rate, float rrc_alpha, int rrc_span, double symbol_sync_bw,
                            double costas_loop_bw, double cfo_loop_bw, int differential, const char* tsc_bits, int use_fll,
                            int64_t max_frame_bytes, int channels, qpsk_demod** out) {
  if (!out) return QPSK_ERR_NULL;
  *out = nullptr;
  qpsk_demod* d = new (std::nothrow) qpsk_demod();
  if (!d) return QPSK_ERR_NOMEM;
  int st = d->eng.init(sample_rate, symbol_rate, rrc_alpha, rrc_span, symbol_sync_bw, costas_loop_bw, cfo_loop_bw, differential,
                       tsc_bits, use_fll, max_frame_bytes, channels);
  if (st != QPSK_OK) { delete d; return st; }
  *out = d;
  return QPSK_OK;
}
int qpsk_demod_create(int sample_rate, int symbol_rate, float rrc_alpha, int rrc_span, double symbol_sync_bw,
                      double costas_loop_bw, double cfo_loop_bw, int differential, const char* tsc_bits, int use_fll,
                      int64_t max_frame_bytes, qpsk_demod** out) {
  return qpsk_demod_create_batch(sample_rate, symbol_rate, rrc_alpha, rrc_span, symbol_sync_bw, costas_loop_bw, cfo_loop_bw,
                                 differential, tsc_bits, use_fll, max_frame_bytes, 1, out);
}
int qpsk_demod_destroy(qpsk_demod* d) {
  if (d) {
    if (d->eng.stream) cudaStreamSynchronize(d->eng.stream);
    delete d;
  }
  return QPSK_OK;
}
int qpsk_demod_set_fir_mode(qpsk_demod* d, int mode) {
  if (!d) return QPSK_ERR_NULL;
  if (mode != QPSK_FIR_FAST && mode != QPSK_FIR_EXACT) return QPSK_ERR_RANGE;
  // FAST inside the modem = the tap-sequential FMA kernel: chunk-invariant bit for bit (the time-chunk pipeline relies on it)
  d->eng.mf.mode = mode == QPSK_FIR_FAST ? QPSK_FIR_FMA : mode;
  return QPSK_OK;
}
int qpsk_demod_set_equalizer(qpsk_demod* d, int n_taps, float mu, float modulus) {
  if (!d) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(d->eng.device));
  return d->eng.set_equalizer(n_taps, mu, modulus);
}
int qpsk_demod_set_agc(qpsk_demod* d, int window, float ref, float max_gain) {
  if (!d) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(d->eng.device));
  return d->eng.set_agc(window, ref, max_gain);
}
int qpsk_demod_equalizer_taps(qpsk_demod* d, float* taps_iq, int64_t cap_floats) {
  if (!d || !taps_iq) return QPSK_ERR_NULL;
  DemodEngine& e = d->eng;
  if (!e.eq) return QPSK_ERR_ARG;
  const int64_t need = (int64_t)e.channels * 2 * e.eq->P.n_taps;
  if (cap_floats < need) return QPSK_ERR_CAPACITY;
  QPSK_TRY(ensure_device(e.device));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaMemcpy(taps_iq, e.eq->d_taps.p, (size_t)need * 4, cudaMemcpyDeviceToHost));
  return QPSK_OK;
}
int qpsk_demod_set_fractional_equalizer(qpsk_demod* d, int n_taps, float mu, float modulus) {
  if (!d) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(d->eng.device));
  return d->eng.set_fractional_equalizer(n_taps, mu, modulus);
}
int qpsk_demod_fractional_equalizer_taps(qpsk_demod* d, float* taps_iq, int64_t cap_floats) {
  if (!d || !taps_iq) return QPSK_ERR_NULL;
  DemodEngine& e = d->eng;
  if (!e.fse) return QPSK_ERR_ARG;
  const int64_t need = (int64_t)e.channels * 2 * e.fse->P.n_taps;
  if (cap_floats < need) return QPSK_ERR_CAPACITY;
  QPSK_TRY(ensure_device(e.device));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaMemcpy(taps_iq, e.fse->d_taps.p, (size_t)need * 4, cudaMemcpyDeviceToHost));
  return QPSK_OK;
}

static int demod_check_in(qpsk_demod* d, const void* in, int64_t n_floats) {
  if (!d) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;              // :347-348
  if (n_floats > 0 && !in) return QPSK_ERR_NULL;
  return QPSK_OK;
}

int qpsk_demod_bits(qpsk_demod* d, const float* iq_in, int64_t n_floats, char* bits_out, int64_t cap, int64_t* n_bits) {
  QPSK_TRY(demod_check_in(d, iq_in, n_floats));
  if (!n_bits) return QPSK_ERR_NULL;
  DemodEngine& e = d->eng;
  for (int c = 0; c < e.channels; ++c) n_bits[c] = 0;
  if (n_floats == 0) return QPSK_OK;                         // :350-351
  QPSK_TRY(ensure_device(d->eng.device));
  cudaStream_t s = e.stream;
  const int64_t L = n_floats >> 1;
  const long long ldb = (e.bits_bound(L) + 2 + 15) & ~15LL;
  QPSK_TRY(e.d_bits.ensure((size_t)ldb * e.channels));
  HostSrc hs;
  hs.p = iq_in; hs.ld = L; hs.cs16 = false;
  QPSK_TRY(e.bits_dev(nullptr, L, 0, e.d_bits.p, ldb, e.d_nbits.p, s, &hs));
  // bytes 0/1 -> '0'/'1' on the device before the rows come back
  return e.fetch_results(e.d_nbits.p, n_bits, 8, bits_out, cap, e.d_bits.p, (size_t)ldb, s, [&] {
    const long long tot = ldb * e.channels;
    long long blocks = (tot + 255) / 256;
    const long long capb = 32LL * device_sm_count();
    if (blocks > capb) blocks = capb;
    bits_to_chars_kernel<<<(int)blocks, 256, 0, s>>>(e.d_bits.p, reinterpret_cast<char*>(e.d_bits.p), tot);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  });
}

int qpsk_demod_bits_packed(qpsk_demod* d, const float* iq_in, int64_t n_floats, uint8_t* packed_out, int64_t cap_bytes,
                           int64_t* n_bits) {
  QPSK_TRY(demod_check_in(d, iq_in, n_floats));
  if (!n_bits) return QPSK_ERR_NULL;
  if (cap_bytes < 0) return QPSK_ERR_RANGE;
  DemodEngine& e = d->eng;
  for (int c = 0; c < e.channels; ++c) n_bits[c] = 0;
  if (n_floats == 0) return QPSK_OK;                         // :350-351
  QPSK_TRY(ensure_device(d->eng.device));
  cudaStream_t s = e.stream;
  const int64_t L = n_floats >> 1;
  const long long ldb = (e.bits_bound(L) + 2 + 7) & ~7LL;    // 8-byte aligned rows for the pack kernel's wide loads
  QPSK_TRY(e.d_bits.ensure((size_t)ldb * e.channels));
  HostSrc hs;
  hs.p = iq_in; hs.ld = L; hs.cs16 = false;
  QPSK_TRY(e.bits_dev(nullptr, L, 0, e.d_bits.p, ldb, e.d_nbits.p, s, &hs));
  const long long ldp = ldb / 8;
  QPSK_TRY(e.d_pk.ensure((size_t)ldp * e.channels));
  QPSK_TRY(qpsk_pack_bits_dev(e.d_bits.p, ldb, (const int64_t*)e.d_nbits.p, ldb, e.channels, e.d_pk.p, ldp, s));
  return e.fetch_results(e.d_nbits.p, n_bits, 1, packed_out, cap_bytes, e.d_pk.p, (size_t)ldp, s);
}

// host samples -> payload bytes: the chain runs as a pipeline over time chunks (HostSrc), the payloads come back in one
// 2-D copy whose width is the longest payload of the call
static int demod_bytes_host(qpsk_demod* d, const HostSrc& hs, int64_t L, const uint8_t* start_marker, int64_t n_start,
                            const uint8_t* end_marker, int64_t n_end, uint8_t* payload_out, int64_t cap, int64_t* n_bytes) {
  DemodEngine& e = d->eng;
  cudaStream_t s = e.stream;
  // device payload rows: what one call can complete is bounded by the framer ring, and by `cap` when the caller gave less
  const int64_t pcap = cap > 0 ? (cap < e.ring_cap ? cap : e.ring_cap) : 1;
  QPSK_TRY(e.d_payload.ensure((size_t)pcap * e.channels));
  QPSK_TRY(e.bytes_dev(nullptr, L, 0, start_marker, n_start, end_marker, n_end, e.d_payload.p, pcap, e.d_npayload.p, s, &hs));
  // a frame longer than `cap` stays in the ring: qpsk_demod_last_payload
  const int st = e.fetch_results(e.d_npayload.p, n_bytes, 8, payload_out, cap, e.d_payload.p, (size_t)pcap, s);
  e.last_np.assign(n_bytes, n_bytes + e.channels);
  return st;
}

int qpsk_demod_bytes(qpsk_demod* d, const float* iq_in, int64_t n_floats, const uint8_t* start_marker, int64_t n_start,
                     const uint8_t* end_marker, int64_t n_end, uint8_t* payload_out, int64_t cap, int64_t* n_bytes) {
  if (!d || !n_bytes) return QPSK_ERR_NULL;
  if (n_start == 0 || n_end == 0) return QPSK_ERR_ARG;       // :174-175 (checked before the samples)
  QPSK_TRY(demod_check_in(d, iq_in, n_floats));
  DemodEngine& e = d->eng;
  for (int c = 0; c < e.channels; ++c) n_bytes[c] = 0;
  if (n_floats == 0) return QPSK_OK;
  if (cap < 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device(d->eng.device));
  HostSrc hs;
  hs.p = iq_in; hs.ld = n_floats >> 1; hs.cs16 = false;
  return demod_bytes_host(d, hs, n_floats >> 1, start_marker, n_start, end_marker, n_end, payload_out, cap, n_bytes);
}

// the same call on CS16 samples (interleaved int16 I, Q — the format SaveAsCs16 writes, HelperFunctions.cs:75-106, and SDR
// drivers deliver): widened on the device as (float)v * scale, so PCIe carries 4 bytes per complex sample instead of 8
int qpsk_demod_bytes_cs16(qpsk_demod* d, const int16_t* iq_in, int64_t n_int16, float scale, const uint8_t* start_marker,
                          int64_t n_start, const uint8_t* end_marker, int64_t n_end, uint8_t* payload_out, int64_t cap,
                          int64_t* n_bytes) {
  if (!d || !n_bytes) return QPSK_ERR_NULL;
  if (n_start == 0 || n_end == 0) return QPSK_ERR_ARG;
  QPSK_TRY(demod_check_in(d, iq_in, n_int16));
  DemodEngine& e = d->eng;
  for (int c = 0; c < e.channels; ++c) n_bytes[c] = 0;
  if (n_int16 == 0) return QPSK_OK;
  if (cap < 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device(d->eng.device));
  HostSrc hs;
  hs.p = iq_in; hs.ld = n_int16 >> 1; hs.cs16 = true; hs.scale = scale;
  return demod_bytes_host(d, hs, n_int16 >> 1, start_marker, n_start, end_marker, n_end, payload_out, cap, n_bytes);
}

int qpsk_demod_last_payload(qpsk_demod* d, uint8_t* payload_out, int64_t cap, int64_t* n_bytes) {
  if (!d || !n_bytes) return QPSK_ERR_NULL;
  if (cap < 0) return QPSK_ERR_RANGE;
  DemodEngine& e = d->eng;
  QPSK_TRY(ensure_device(e.device));
  int st = QPSK_OK;
  for (int c = 0; c < e.channels; ++c) {
    const long long n = (size_t)c < e.last_np.size() ? e.last_np[(size_t)c] : 0;
    n_bytes[c] = n;
    if (n == 0) continue;
    if (n > cap) { st = QPSK_ERR_CAPACITY; continue; }
    if (!payload_out) return QPSK_ERR_NULL;
    // a completed frame stays at the head of the channel's ring until the next framer call starts a new one
    // (ResetFramer :159-167 clears the counters, not the bytes)
    QPSK_CUDA_TRY(cudaMemcpy(payload_out + (size_t)c * cap, e.d_ring.p + (size_t)c * (size_t)e.ring_cap, (size_t)n,
                             cudaMemcpyDeviceToHost));
  }
  return st;
}

int qpsk_demod_frame_bits(qpsk_demod* d, const uint8_t* bits, int64_t bits_stride, const int64_t* n_bits,
                          const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                          uint8_t* payload_out, int64_t cap, int64_t* n_bytes) {
  if (!d || !n_bytes || !n_bits) return QPSK_ERR_NULL;
  if (n_start == 0 || n_end == 0) return QPSK_ERR_ARG;       // :174-175
  if (bits_stride < 0 || cap < 0) return QPSK_ERR_RANGE;
  DemodEngine& e = d->eng;
  long long max_bits = 0;
  for (int c = 0; c < e.channels; ++c) {
    n_bytes[c] = 0;
    if (n_bits[c] < 0 || n_bits[c] > bits_stride) return QPSK_ERR_RANGE;
    if (n_bits[c] > max_bits) max_bits = n_bits[c];
  }
  if (max_bits == 0) return QPSK_OK;                         // :179-180 for every channel
  if (!bits) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(d->eng.device));
  cudaStream_t s = e.stream;
  const long long ldb = max_bits;
  QPSK_TRY(e.d_bits.ensure((size_t)ldb * e.channels));
  QPSK_CUDA_TRY(cudaMemcpy2DAsync(e.d_bits.p, (size_t)ldb, bits, (size_t)bits_stride, (size_t)max_bits, (size_t)e.channels,
                                  cudaMemcpyHostToDevice, s));
  QPSK_CUDA_TRY(cudaMemcpyAsync(e.d_nbits.p, n_bits, sizeof(long long) * e.channels, cudaMemcpyHostToDevice, s));
  const int64_t pcap = cap > 0 ? cap : 1;
  QPSK_TRY(e.d_payload.ensure((size_t)pcap * e.channels));
  QPSK_TRY(e.frame_dev(e.d_bits.p, ldb, e.d_nbits.p, start_marker, n_start, end_marker, n_end, e.d_payload.p, pcap, e.d_npayload.p, s));
  const int st = e.fetch_results(e.d_npayload.p, n_bytes, 8, payload_out, cap, e.d_payload.p, (size_t)pcap, s);
  e.last_np.assign(n_bytes, n_bytes + e.channels);
  return st;
}

int qpsk_demod_constellation(qpsk_demod* d, const float* iq_in, int64_t n_floats, float* sym_iq_out, int64_t cap_floats,
                             int64_t* n_sym) {
  QPSK_TRY(demod_check_in(d, iq_in, n_floats));
  if (!n_sym) return QPSK_ERR_NULL;
  DemodEngine& e = d->eng;
  for (int c = 0; c < e.channels; ++c) n_sym[c] = 0;
  if (n_floats == 0) return QPSK_OK;
  QPSK_TRY(ensure_device(d->eng.device));
  cudaStream_t s = e.stream;
  const int64_t L = n_floats >> 1;
  const long long lds = std::max(1LL, e.symbols_bound(L));
  QPSK_TRY(e.h_out.ensure((size_t)lds * e.channels));
  QPSK_TRY(e.d_ncon.ensure((size_t)e.channels));
  HostSrc hs;
  hs.p = iq_in; hs.ld = L; hs.cs16 = false;
  QPSK_TRY(e.constellation_dev(nullptr, L, 0, e.h_out.p, lds, e.d_ncon.p, s, &hs));
  return e.fetch_results(e.d_ncon.p, n_sym, 64, sym_iq_out, cap_floats * 4, e.h_out.p, (size_t)lds * 8, s);
}

int qpsk_demod_device(const qpsk_demod* d, int* ordinal) {
  if (!d || !ordinal) return QPSK_ERR_NULL;
  *ordinal = d->eng.device;
  return QPSK_OK;
}

int qpsk_demod_channels(const qpsk_demod* d, int* channels) {
  if (!d || !channels) return QPSK_ERR_NULL;
  *channels = d->eng.channels;
  return QPSK_OK;
}

int qpsk_demod_bits_dev(qpsk_demod* d, const float* d_in, int64_t n_floats, int64_t in_stride_floats, uint8_t* d_bits,
                        int64_t bits_cap, int64_t* d_n_bits, void* stream) {
  QPSK_TRY(demod_check_in(d, d_in, n_floats));
  if (!d_bits || !d_n_bits) return QPSK_ERR_NULL;
  if (in_stride_floats & 1) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(d->eng.device));
  DemodEngine& e = d->eng;
  cudaStream_t s = stream ? (cudaStream_t)stream : e.stream;
  return e.bits_dev((const float2*)d_in, n_floats >> 1, in_stride_floats >> 1, d_bits, bits_cap, (long long*)d_n_bits, s);
}

int qpsk_demod_bits_bound(qpsk_demod* d, int64_t n_floats, int64_t* bits_cap) {
  if (!d || !bits_cap) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  long long b = d->eng.bits_bound(n_floats >> 1);
  if (b < 2) b = 2;
  *bits_cap = b + (b & 1);
  return QPSK_OK;
}

int qpsk_demod_bytes_dev(qpsk_demod* d, const float* d_in, int64_t n_floats, int64_t in_stride_floats,
                         const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                         uint8_t* d_payload, int64_t payload_cap, int64_t* d_n_bytes, void* stream) {
  if (!d) return QPSK_ERR_NULL;
  if (n_start == 0 || n_end == 0) return QPSK_ERR_ARG;
  QPSK_TRY(demod_check_in(d, d_in, n_floats));
  if (!d_payload || !d_n_bytes) return QPSK_ERR_NULL;
  if (in_stride_floats & 1) return QPSK_ERR_ARG;
  if (payload_cap <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device(d->eng.device));
  DemodEngine& e = d->eng;
  cudaStream_t s = stream ? (cudaStream_t)stream : e.stream;
  if (n_floats == 0) {
    QPSK_CUDA_TRY(cudaMemsetAsync(d_n_bytes, 0, sizeof(int64_t) * e.channels, s));
    return QPSK_OK;
  }
  return e.bytes_dev((const float2*)d_in, n_floats >> 1, in_stride_floats >> 1, start_marker, n_start, end_marker, n_end,
                     d_payload, payload_cap, (long long*)d_n_bytes, s);
}

int qpsk_demod_frame_bits_dev(qpsk_demod* d, const uint8_t* d_bits, int64_t bits_stride, const int64_t* d_n_bits,
                              const uint8_t* start_marker, int64_t n_start, const uint8_t* end_marker, int64_t n_end,
                              uint8_t* d_payload, int64_t payload_cap, int64_t* d_n_bytes, void* stream) {
  if (!d) return QPSK_ERR_NULL;
  if (n_start == 0 || n_end == 0) return QPSK_ERR_ARG;       // :174-175
  if (!d_bits || !d_n_bits || !d_payload || !d_n_bytes) return QPSK_ERR_NULL;
  if (bits_stride < 0) return QPSK_ERR_RANGE;
  if (payload_cap <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device(d->eng.device));
  DemodEngine& e = d->eng;
  cudaStream_t s = stream ? (cudaStream_t)stream : e.stream;
  return e.frame_dev(d_bits, bits_stride, (const long long*)d_n_bits, start_marker, n_start, end_marker, n_end, d_payload,
                     payload_cap, (long long*)d_n_bytes, s);
}

int qpsk_demod_constellation_dev(qpsk_demod* d, const float* d_in, int64_t n_floats, int64_t in_stride_floats, float* d_sym,
                                 int64_t sym_stride_floats, int* d_n_sym, void* stream) {
  QPSK_TRY(demod_check_in(d, d_in, n_floats));
  if (!d_sym || !d_n_sym) return QPSK_ERR_NULL;
  if ((in_stride_floats & 1) || (sym_stride_floats & 1)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(d->eng.device));
  DemodEngine& e = d->eng;
  cudaStream_t s = stream ? (cudaStream_t)stream : e.stream;
  return e.constellation_dev((const float2*)d_in, n_floats >> 1, in_stride_floats >> 1, (float2*)d_sym, sym_stride_floats >> 1,
                             d_n_sym, s);
}

int qpsk_demod_loop_state(qpsk_demod* d, double* costas_theta, double* costas_freq, double* mm_mu, double* mm_integral,
                          float* fll_phase, float* fll_freq) {
  if (!d) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(d->eng.device));
  DemodEngine& e = d->eng;
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaDeviceSynchronize());
  const size_t C = (size_t)e.channels;
  std::vector<CostasState> cs(C);
  std::vector<MmState> ms(C);
  std::vector<float2> pf(C);
  QPSK_CUDA_TRY(cudaMemcpy(cs.data(), e.costas.d_state.p, C * sizeof(CostasState), cudaMemcpyDeviceToHost));
  QPSK_CUDA_TRY(cudaMemcpy(ms.data(), e.mm.d_state.p, C * sizeof(MmState), cudaMemcpyDeviceToHost));
  QPSK_CUDA_TRY(cudaMemcpy(pf.data(), e.fll.d_pf.p, C * sizeof(float2), cudaMemcpyDeviceToHost));
  for (size_t c = 0; c < C; ++c) {
    if (costas_theta) costas_theta[c] = cs[c].theta;
    if (costas_freq) costas_freq[c] = cs[c].freq;
    if (mm_mu) mm_mu[c] = ms[c].mu;
    if (mm_integral) mm_integral[c] = ms[c].integral;
    if (fll_phase) fll_phase[c] = pf[c].x;
    if (fll_freq) fll_freq[c] = pf[c].y;
  }
  return QPSK_OK;
}

int qpsk_demod_in_frame(qpsk_demod* d, int* in_frame) {
  if (!d || !in_frame) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(d->eng.device));
  DemodEngine& e = d->eng;
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  std::vector<FramerState> fs((size_t)e.channels);
  QPSK_CUDA_TRY(cudaMemcpy(fs.data(), e.d_framer.p, fs.size() * sizeof(FramerState), cudaMemcpyDeviceToHost));
  for (int c = 0; c < e.channels; ++c) in_frame[c] = fs[(size_t)c].in_frame;
  return QPSK_OK;
}

}  // extern "C"
