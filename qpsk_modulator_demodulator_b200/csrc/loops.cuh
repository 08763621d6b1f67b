// loops.cuh — the serial feedback loops, one thread per independent stream, recurrences kept exactly
// sequential and in the reference's precisions.  This translation unit family is compiled with
// --fmad=false: RyuJIT never fuses a*b+c, so every product and sum below rounds separately.
//
//   FllParams/FllEngine    FLLBandEdgeFilter.Process   MS/Models/Band-Edge Filter.cs:102-129,185-195
//   MmState/mm_*           MuellerMuller.Process       MS/Models/MuellerMuller.cs:52-136,160-198
//   CostasState/costas_step CostasLoopQpsk.Process     MS/Models/CostasLoopQpsk.cs:63-92
#pragma once
#include "handle.cuh"
#include "design.h"

namespace qpsk {

// ---------------------------------------------------------------------------------------------
// FLL
// ---------------------------------------------------------------------------------------------
struct FllParams {
  float beta, alpha, max_freq, min_freq;
  int n_taps;
};

// The two band-edge filters see the same input and upper = conj(lower) (Band-Edge Filter.cs:176-178),
// so one ring of past outputs and the four products a*xI, b*xQ, a*xQ, b*xI serve both; sums keep
// ComplexDotWindow's order (8 lane partials over the chronological window, lanes 0..7, scalar
// tail: FIRFilter.cs:165-192).  (-b)*x == -(b*x) and p - (-q) == p + q exactly, so sharing the
// products is bit-neutral.  Every FLL kernel takes the lower-filter taps reversed (rev[i] = lower[N-1-i]).

// ---------------------------------------------------------------------------------------------
// Mueller-Muller
// ---------------------------------------------------------------------------------------------
struct MmState {
  double mu, integral;
  float prevSI, prevSQ, prevDI, prevDQ;
  int base_index;
  int has_prev;
  int queued;  // complex samples carried in the queue
  int pad;
};

struct MmParams {
  double sps, kp, ki;
};

// logical buffer = [queue(0..queued) | incoming]
struct MmView {
  const float2* queue;
  const float2* in;
  int queued;
  __device__ __forceinline__ float2 at(int k) const { return (k < queued) ? queue[k] : in[k - queued]; }
};

// CubicLagrange4 (MuellerMuller.cs:160-190): fp32, mu cast to float, products/sums left to right
__device__ __forceinline__ void mm_interp(const MmView& v, int n, double mu, float& oI, float& oQ) {
  const float2 xm1 = v.at(n - 1), x0 = v.at(n), x1 = v.at(n + 1), x2 = v.at(n + 2);
  const float t = (float)mu;
  const float tm1 = t - 1.f, tm2 = t - 2.f, tp1 = t + 1.f;
  const float sixth = 1.f / 6.f, half = 1.f / 2.f;
  const float c_m1 = -(t * tm1 * tm2) * sixth;
  const float c_0 = (tp1 * tm1 * tm2) * half;
  const float c_1 = -(tp1 * t * tm2) * half;
  const float c_2 = (tp1 * t * tm1) * sixth;
  oI = c_m1 * xm1.x + c_0 * x0.x + c_1 * x1.x + c_2 * x2.x;
  oQ = c_m1 * xm1.y + c_0 * x0.y + c_1 * x1.y + c_2 * x2.y;
}

// the same on a contiguous buffer (symsync_decode_kernel keeps [carried | block] in one run): four unconditional loads
__device__ __forceinline__ void mm_interp_lin(const float2* __restrict__ b, int n, double mu, float& oI, float& oQ) {
  const float2 xm1 = b[n - 1], x0 = b[n], x1 = b[n + 1], x2 = b[n + 2];
  const float t = (float)mu;
  const float tm1 = t - 1.f, tm2 = t - 2.f, tp1 = t + 1.f;
  const float sixth = 1.f / 6.f, half = 1.f / 2.f;
  const float c_m1 = -(t * tm1 * tm2) * sixth;
  const float c_0 = (tp1 * tm1 * tm2) * half;
  const float c_1 = -(tp1 * t * tm2) * half;
  const float c_2 = (tp1 * t * tm1) * sixth;
  oI = c_m1 * xm1.x + c_0 * x0.x + c_1 * x1.x + c_2 * x2.x;
  oQ = c_m1 * xm1.y + c_0 * x0.y + c_1 * x1.y + c_2 * x2.y;
}

// One pass of the `while` body (:62-120).  Returns false when the loop must stop *before* emitting
// (output full, :101-102).  `stop_after` is set when the post-advance break (:118-119) fires.
__device__ __forceinline__ bool mm_symbol(const MmParams& P, MmState& S, const MmView& v, int buf_count, bool room,
                                          float& currI, float& currQ, bool& stop_after) {
  mm_interp(v, S.base_index, S.mu, currI, currQ);
  const float decI = (currI >= 0.f) ? 1.f : -1.f;   // GetSignQpsk :194-198
  const float decQ = (currQ >= 0.f) ? 1.f : -1.f;
  double advance;
  if (S.has_prev) {
    const double term1 = (double)S.prevDI * currI + (double)S.prevDQ * currQ;   // :78
    const double term2 = (double)decI * S.prevSI + (double)decQ * S.prevSQ;     // :79
    const double e = term1 - term2;
    S.integral += P.ki * e;                          // :83
    double corr = P.kp * e + S.integral;             // :84
    if (corr > 0.1) corr = 0.1;                      // :87-89
    if (corr < -0.1) corr = -0.1;
    advance = P.sps + corr;
  } else {
    S.has_prev = 1;
    advance = P.sps;
  }
  if (!room) return false;                           // :101-102 (loop state already touched)
  S.prevSI = currI; S.prevSQ = currQ; S.prevDI = decI; S.prevDQ = decQ;
  const double newTime = S.base_index + S.mu + advance;   // :113
  S.base_index = (int)floor(newTime);
  S.mu = newTime - S.base_index;
  stop_after = (S.base_index + 1 >= buf_count);      // :118-119
  return true;
}

// ---------------------------------------------------------------------------------------------
// Costas
// ---------------------------------------------------------------------------------------------
struct CostasState {
  double theta, freq;
};
struct CostasParams {
  double alpha, beta;
};

// flip the sign of x when `neg` (exact: what multiplying by -1.0 does)
__device__ __forceinline__ double flip_sign_if(double x, bool neg) {
  return __hiloint2double(__double2hiint(x) ^ (neg ? (int)0x80000000u : 0), __double2loint(x));
}

// One CostasLoopQpsk.Process step (:63-92).  This is a loop-carried dependency chain of ~30 fp64 operations with
// nothing to overlap it with (one stream per thread), so everything that is not arithmetic on the value path has been
// moved off it, without changing a single rounding:
//   * sin/cos through sincos_fast_f64_k (constants in registers, quadrant fix-up by select / sign-bit XOR); the
//     |theta| >= 1e5 case (never reached: theta is wrapped every step, :89-91) re-evaluates with sincos() afterwards;
//   * the decisions sign((float)mi), sign((float)mq) (:76-80) are taken on the fp64 values: (float)m >= 0 exactly when
//     m >= -2^-150 (smaller magnitudes round to +-0 and -0.0f >= 0) — this removes an F2F -> FSETP -> FSEL -> F2F chain;
//   * est = +-1.0, so est*m is an exact sign flip: pe = (+-mq) - (+-mi) (:82);
//   * both wrap candidates theta -+ 2*pi are formed speculatively and selected (:89-91).
// |x| >= bound (or NaN) tested on the high word with an integer compare (4-cycle ALU instead of a DSETP on the
// fp64 pipe); `bound_hi` = high word of a bound whose low word is zero
__device__ __forceinline__ bool abs_ge_hi(double x, int bound_hi) { return (__double2hiint(x) & 0x7fffffff) >= bound_hi; }

// the straight-line part: valid while |theta| < 1e5 and both mixer outputs are finite and not in the band where the
// fp32 rounding decides the sign (`wild` reports otherwise and the caller replays through costas_step_exact).
// sgnI/sgnQ: bit 31 set when the decision on the fp32 output is -1, i.e. when !(out >= 0).
__device__ __forceinline__ void costas_step_fast(const CostasParams& P, const SinCosK& K, CostasState& S, float inI, float inQ,
                                                 float& outI, float& outQ, unsigned& sgnI, unsigned& sgnQ, bool& wild) {
  wild |= abs_ge_hi(S.theta, 0x40F86A00);                    // |theta| >= 1e5 or NaN
  double s, c;
  sincos_fast_f64_k(S.theta, K, &s, &c);
  const double dI = (double)inI, dQ = (double)inQ;
  const double mi = dI * c + dQ * s;                         // :72
  const double mq = dQ * c - dI * s;                         // :73
  outI = (float)mi;
  outQ = (float)mq;
  // GetSign of the fp32 outputs (:52-56, :76-80) from the fp64 values: (float)m >= 0 exactly when m >= -2^-150
  // (smaller magnitudes round to +-0 and -0.0f >= 0).  Outside (-2^-149, -0] that is the sign bit of m; that sliver,
  // Inf and NaN take the replay path, so one AND per output is all that sits on the chain.
  const int hi_i = __double2hiint(mi), hi_q = __double2hiint(mq);
  const unsigned ui = (unsigned)hi_i, uq = (unsigned)hi_q;
  wild |= (ui - 0x80000000u < 0x36A00000u) | ((ui & 0x7fffffffu) >= 0x7ff00000u) |      // -2^-149 < mi <= -0, Inf, NaN
          (uq - 0x80000000u < 0x36A00000u) | ((uq & 0x7fffffffu) >= 0x7ff00000u);
  sgnI = (unsigned)hi_i & 0x80000000u;
  sgnQ = (unsigned)hi_q & 0x80000000u;
  // pe = estI*mq - estQ*mi with est = +-1.0: the products are exact sign flips (:82)
  const double a = __hiloint2double(hi_q ^ (int)sgnI, __double2loint(mq));
  const double b = __hiloint2double(hi_i ^ (int)sgnQ, __double2loint(mi));
  const double pe = a - b;
  S.freq += P.beta * pe;                                     // :85
  const double t = S.theta + (S.freq + P.alpha * pe);        // :86
  const double kPi = 3.14159265358979323846, kTwoPi = 2.0 * kPi;
  const double t_dn = t - kTwoPi, t_up = t + kTwoPi;
  S.theta = (t > kPi) ? t_dn : ((t < -kPi) ? t_up : t);      // :89-91
}
// costas_step_fast with the shortened sincos and the quadrant applied to the INPUT sample: theta = r + q*pi/2 and
// x * e^{-j theta} = (x * (-j)^q) * (cos r - j sin r); the factor (-j)^q is an exact swap / sign flip that runs while
// the polynomials are evaluated, and the mixer forms the same two products per component as :72-73 (signs are exact,
// a + b == b + a), so the select / XOR fix-up of the sin/cos pair leaves the dependency chain.
__device__ __forceinline__ void costas_step_fast2(const CostasParams& P, const SinCosK& K, double magic, CostasState& S, float inI,
                                                  float inQ, float& outI, float& outQ, unsigned& sgnI, unsigned& sgnQ,
                                                  bool& wild) {
  wild |= abs_ge_hi(S.theta, 0x40F86A00);                    // |theta| >= 1e5 or NaN
  double sr, cr;
  unsigned q;
  sincos_rq_f64_k(S.theta, K, magic, &sr, &cr, &q);
  const double dI = (double)inI, dQ = (double)inQ;
  // x' = x * (-j)^q:  q=0 (I, Q)   q=1 (Q, -I)   q=2 (-I, -Q)   q=3 (-Q, I)
  const bool odd = (q & 1u) != 0;
  const int fI = (int)((q & 2u) << 30);                      // sign of the first component: quadrants 2, 3
  const int fQ = (int)(((q + 1u) & 2u) << 30);               // sign of the second: quadrants 1, 2
  const double aI0 = odd ? dQ : dI, aQ0 = odd ? dI : dQ;
  const double aI = __hiloint2double(__double2hiint(aI0) ^ fI, __double2loint(aI0));
  const double aQ = __hiloint2double(__double2hiint(aQ0) ^ fQ, __double2loint(aQ0));
  const double mi = aI * cr + aQ * sr;                       // :72
  const double mq = aQ * cr - aI * sr;                       // :73
  outI = (float)mi;
  outQ = (float)mq;
  const int hi_i = __double2hiint(mi), hi_q = __double2hiint(mq);
  const unsigned ui = (unsigned)hi_i, uq = (unsigned)hi_q;
  wild |= (ui - 0x80000000u < 0x36A00000u) | ((ui & 0x7fffffffu) >= 0x7ff00000u) |      // -2^-149 < mi <= -0, Inf, NaN
          (uq - 0x80000000u < 0x36A00000u) | ((uq & 0x7fffffffu) >= 0x7ff00000u);
  sgnI = (unsigned)hi_i & 0x80000000u;
  sgnQ = (unsigned)hi_q & 0x80000000u;
  const double a = __hiloint2double(hi_q ^ (int)sgnI, __double2loint(mq));
  const double b = __hiloint2double(hi_i ^ (int)sgnQ, __double2loint(mi));
  const double pe = a - b;                                   // :82
  S.freq += P.beta * pe;                                     // :85
  const double t = S.theta + (S.freq + P.alpha * pe);        // :86
  const double kPi = 3.14159265358979323846, kTwoPi = 2.0 * kPi;
  const double t_dn = t - kTwoPi, t_up = t + kTwoPi;
  S.theta = (t > kPi) ? t_dn : ((t < -kPi) ? t_up : t);      // :89-91
}
// exact for every input: the reference's operation order with the library sincos
__device__ __forceinline__ void costas_step_exact(const CostasParams& P, CostasState& S, float inI, float inQ, float& outI,
                                                  float& outQ) {
  double s, c;
  sincos(S.theta, &s, &c);
  const double dI = (double)inI, dQ = (double)inQ;
  const double mi = dI * c + dQ * s;
  const double mq = dQ * c - dI * s;
  outI = (float)mi;
  outQ = (float)mq;
  const double estI = (outI >= 0.f) ? 1.0 : -1.0, estQ = (outQ >= 0.f) ? 1.0 : -1.0;
  const double pe = estI * mq - estQ * mi;
  S.freq += P.beta * pe;
  S.theta += S.freq + P.alpha * pe;
  const double kPi = 3.14159265358979323846, kTwoPi = 2.0 * kPi;
  if (S.theta > kPi) S.theta -= kTwoPi;
  else if (S.theta < -kPi) S.theta += kTwoPi;
}
__device__ __forceinline__ void costas_step(const CostasParams& P, const SinCosK& K, CostasState& S, float inI, float inQ,
                                            float& outI, float& outQ) {
  const CostasState S0 = S;
  unsigned nI, nQ;
  bool wild = false;
  costas_step_fast(P, K, S, inI, inQ, outI, outQ, nI, nQ, wild);
  if (wild) {
    S = S0;
    costas_step_exact(P, S, inI, inQ, outI, outQ);
  }
}

// ---------------------------------------------------------------------------------------------
// engines (host side)
// ---------------------------------------------------------------------------------------------
struct FllEngine : EngineBase {
  int channels = 1, n_taps = 0;
  FllParams P{};
  std::vector<float> lower, upper;
  DevBuf<float> d_taps;      // [2][N] reversed lower taps, planar
  DevBuf<float2> d_ring;     // [N][C] ring of past outputs
  DevBuf<int> d_head;        // [C]
  DevBuf<float2> d_pf;       // [C] (phase, freq)
  bool state_wild = false;   // a caller-set (phase, freq) outside the fast kernel's range is pending
  bool state_far = false;    // a caller-set |phase| >= 32 is pending (the pair kernel's short-range sin/cos)
  int init(float sps, float rolloff, int size, float bw, int channels_in);
  int process_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, cudaStream_t s);
};

// fll_duo.cu: two-warp (chain + side) FLL kernel for N = 8..55 taps
bool fll_duo_supported(int n_taps);
int fll_duo_launch(const FllParams& P, const float* taps, float2* ring, int* head, float2* pf, int C, const float2* x,
                   float2* y, long long L, long long ldx, long long ldy, cudaStream_t s);

// fll_pair.cu: two lanes per stream (16 streams per warp), for large batches (40 and 10 taps)
bool fll_pair_supported(int n_taps);
int fll_pair_launch(const FllParams& P, const std::vector<float>& lower, float2* ring, int* head, float2* pf, int C,
                    const float2* x, float2* y, long long L, long long ldx, long long ldy, cudaStream_t s);

struct MmEngine : EngineBase {
  int channels = 1;
  MmParams P{};
  DevBuf<MmState> d_state;
  DevBuf<float2> d_queue[2];  // [C][qcap], ping-pong
  int qcur = 0;
  int64_t qcap = 0;
  int64_t q_bound = 0;        // host-side upper bound of queued samples
  int init(double sps, double kp, double ki, int channels_in);
  int ensure_queue(int64_t need, cudaStream_t s);
  int process_dev(const float2* x, int64_t L, int64_t ldx, float2* y, int64_t cap_sym, int64_t ldy, int* d_nsym,
                  cudaStream_t s);
};

struct CostasEngine : EngineBase {
  int channels = 1;
  CostasParams P{};
  DevBuf<CostasState> d_state;
  int init(double fs, double bw, double damping, int channels_in);
  int process_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, const int* d_nsym, cudaStream_t s);
};

}  // namespace qpsk
