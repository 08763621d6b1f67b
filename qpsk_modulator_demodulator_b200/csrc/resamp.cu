// resamp.cu — batched rational resampler (spec: include/qpskcuda.h, "rational resampler"): rows of [channels][stride] cf32
// in, the same channels at L/M of the rate out, one real prototype h and one ratio per handle.
//
// Polyphase form: output m reads x[n_m - q], q = 0..P-1, with taps hT[phi_m][q] = h[phi_m + qL] (zero past N), where
// n_m = floor(mM / L) and phi_m = mM mod L come from exact integer arithmetic.  Every channel shares the schedule, so at a
// given output all channels read the same branch.
//
// Per channel z = history (the last P-1 input samples, zero before the stream) ++ this call's n samples.  Call output t has
// d_t = n_m - (inputs before the call) in [0, n), and tap q reads z[d_t + P-1 - q].
//
// resamp_kernel<CW, CPT, OPT, CJ>: 256 threads; thread (ci = tid % CW, oi = tid / CW) owns channels ci + a*CW (a < CPT)
// and outputs oi*OPT + b (b < OPT) of the CTA's tile of CB = CW*CPT channels x TB = (256/CW)*OPT outputs.
//   Prologue.  Each output's d_t and branch go to shared memory, then the tile's branch rows hT[phi_t][0..P-1] (taps of
//      outputs past the call's end are never read).
//   Staging.  The tile's z span [d_first, d_last + P-1] is walked from its high end down in chunks of CJ samples; a chunk
//      of all CB rows is copied to shared memory with consecutive threads on consecutive samples of a row (coalesced 8-byte
//      loads, so any 8-byte-aligned pointer and any even stride take the same path).
//   Micro-kernel.  Per sample j of the chunk (descending), a thread loads its CPT samples once and adds them to every one
//      of its OPT outputs whose window holds j: acc += (h, h) * (x.re, x.im), one FFMA2 each, q = d_t + P-1 - j.  As j
//      descends q ascends, so each output is the sum over q = 0 .. P-1 in increasing order, whatever the tile shape, the
//      chunk size, the channel count or the call boundaries: every shape and every chunking give the same bits.
//   Epilogue.  The CB x TB tile goes through shared memory and out as coalesced row segments.
// Two shapes: <32, 2, 4, 64> (64 channels x 32 outputs; lanes over channels, so the four outputs of a warp and their tap
// loads are warp-uniform) for K > 8, and <1, 1, 1, 2048> (one channel x 256 outputs, lanes over outputs) for K <= 8, where
// a 64-channel tile would be mostly padding.
// resamp_history_kernel writes the next call's history (z[n .. n+P-2]) into the other buffer of a ping-pong pair.
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

#include "handle.cuh"

namespace qpsk {

constexpr int kResampThreads = 256;
constexpr int kResampMaxTaps = 16384;
constexpr int kResampMaxFactor = 1024;        // L and M
constexpr int kResampMaxBranch = 64;          // P
constexpr int kResampMaxChannels = 16384;
constexpr int kResampSmallK = 8;              // K <= this: the one-channel shape

template <int CW, int CPT, int OPT, int CJ>
struct ResampShape {
  static constexpr int CB = CW * CPT;                     // channels per CTA
  static constexpr int TB = (kResampThreads / CW) * OPT;  // outputs per CTA
  static constexpr int XP = CJ + 1;                       // float2 per staged row: odd, so a warp's rows spread over banks
  static constexpr int YP = TB + 1;
  static constexpr size_t STAGE = (size_t)CB * (XP > YP ? XP : YP) * sizeof(float2);
  // staged samples / output tile, then d_t and phi_t (int) and the branch rows [TB][P | 1]
  static size_t smem(int P) { return STAGE + 2 * (size_t)TB * sizeof(int) + (size_t)TB * (P | 1) * sizeof(float); }
};

struct ResampArgs {
  const float* hT;        // [L][P] branch-major taps
  int P, L, M;
  const float2* hist;     // [C][P-1]
  const float2* x;
  long long ldx;
  int C;
  long long n_out;        // outputs per channel in this call
  long long d0;           // d of call output 0
  int phi0;               // branch of call output 0
  float2* y;
  long long ldy;
};

__device__ __forceinline__ float2 resamp_z(const ResampArgs& a, int c, long long j) {
  const int HL = a.P - 1;
  return j < HL ? a.hist[(long long)c * HL + j] : a.x[(long long)c * a.ldx + (j - HL)];
}

// call output t -> (d_t, phi_t): phi0 + t*M = (d_t - d0)*L + phi_t, exact in 64 bits
__device__ __forceinline__ long long resamp_d(const ResampArgs& a, long long t, int* phi) {
  const long long s = (long long)a.phi0 + t * (long long)a.M;
  *phi = (int)(s % a.L);
  return a.d0 + s / a.L;
}

template <int CW, int CPT, int OPT, int CJ>
__global__ void __launch_bounds__(kResampThreads) resamp_kernel(ResampArgs a) {
  using S = ResampShape<CW, CPT, OPT, CJ>;
  extern __shared__ __align__(16) unsigned char resamp_smem[];
  float2* sx = reinterpret_cast<float2*>(resamp_smem);                                  // [CB][XP], later [CB][YP]
  int* sd = reinterpret_cast<int*>(resamp_smem + S::STAGE);                    // [TB] d_t - d_first
  int* sphi = sd + S::TB;                                                               // [TB] phi_t
  const int PP = a.P | 1;
  float* sh = reinterpret_cast<float*>(sphi + S::TB);                                   // [TB][PP]
  const int tid = threadIdx.x, ci = tid % CW, oi = tid / CW;
  const long long t0 = (long long)blockIdx.x * S::TB;
  const int kc0 = blockIdx.y * S::CB;
  const int nt = (int)min((long long)S::TB, a.n_out - t0);                             // live outputs of the tile
  const int P = a.P;
  int phi_first;
  const long long d_first = resamp_d(a, t0, &phi_first);

  for (int tt = tid; tt < S::TB; tt += kResampThreads) {
    int phi = 0;
    const long long d = tt < nt ? resamp_d(a, t0 + tt, &phi) : d_first;
    sd[tt] = (int)(d - d_first);
    sphi[tt] = phi;
  }
  __syncthreads();
  for (int e = tid; e < nt * P; e += kResampThreads) {
    const int tt = e / P, q = e % P;
    sh[tt * PP + q] = a.hT[(long long)sphi[tt] * P + q];
  }

  // this thread's outputs: window of output b is z[d_b .. d_b + P-1] (relative to d_first); dead outputs get an empty one
  int db[OPT];
  int jlo = INT_MAX, jhi = INT_MIN;
#pragma unroll
  for (int b = 0; b < OPT; ++b) {
    const int tt = oi * OPT + b;
    db[b] = tt < nt ? sd[tt] : INT_MIN / 2;
    if (tt < nt) {
      jlo = min(jlo, db[b]);
      jhi = max(jhi, db[b] + P - 1);
    }
  }
  const int span = sd[nt - 1] + P;                                                       // tile's z span, relative

  float2 acc[CPT][OPT];
#pragma unroll
  for (int c = 0; c < CPT; ++c)
#pragma unroll
    for (int b = 0; b < OPT; ++b) acc[c][b] = make_float2(0.0f, 0.0f);

  for (int hi = span - 1; hi >= 0; hi -= CJ) {
    const int lo = max(0, hi - CJ + 1), len = hi - lo + 1;
    __syncthreads();
    for (int e = tid; e < S::CB * CJ; e += kResampThreads) {
      const int c = e / CJ, j = e % CJ;
      if (j >= len) continue;
      const int k = kc0 + c;
      sx[c * S::XP + j] = k < a.C ? resamp_z(a, k, d_first + lo + j) : make_float2(0.0f, 0.0f);
    }
    __syncthreads();
    const int jt = min(hi, jhi), jb = max(lo, jlo);
    for (int j = jt; j >= jb; --j) {
      float2 xv[CPT];
#pragma unroll
      for (int c = 0; c < CPT; ++c) xv[c] = sx[(ci + c * CW) * S::XP + (j - lo)];
#pragma unroll
      for (int b = 0; b < OPT; ++b) {
        const int q = db[b] + P - 1 - j;
        if ((unsigned)q < (unsigned)P) {
          const float h = sh[(oi * OPT + b) * PP + q];
          const float2 h2 = make_float2(h, h);
#pragma unroll
          for (int c = 0; c < CPT; ++c) acc[c][b] = ffma2(h2, xv[c], acc[c][b]);
        }
      }
    }
  }

  __syncthreads();
#pragma unroll
  for (int c = 0; c < CPT; ++c)
#pragma unroll
    for (int b = 0; b < OPT; ++b) sx[(ci + c * CW) * S::YP + oi * OPT + b] = acc[c][b];
  __syncthreads();
  for (int e = tid; e < S::CB * S::TB; e += kResampThreads) {
    const int c = e / S::TB, tt = e % S::TB;
    const int k = kc0 + c;
    if (k < a.C && tt < nt) a.y[(long long)k * a.ldy + t0 + tt] = sx[c * S::YP + tt];
  }
}

// hist_out[c][i] = z_c[n + i], i < P-1: the last P-1 samples of the stream so far
__global__ void resamp_history_kernel(ResampArgs a, long long n, float2* __restrict__ hist_out) {
  const int HL = a.P - 1;
  const long long tot = (long long)a.C * HL;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x)
    hist_out[e] = resamp_z(a, (int)(e / HL), n + e % HL);
}

// complete outputs after n inputs: n == 0 ? 0 : floor((nL - 1) / M) + 1, as (n / M) * L + that of n mod M (no overflow)
static unsigned long long resamp_count(unsigned long long n, int L, int M) {
  const unsigned long long r = n % (unsigned long long)M;
  return (n / (unsigned long long)M) * (unsigned long long)L + (r == 0 ? 0ULL : (r * (unsigned long long)L - 1) / (unsigned long long)M + 1);
}

struct ResampEngine : EngineBase {
  int C = 0, L = 0, M = 0, N = 0, P = 0;
  unsigned long long n_in = 0, n_outc = 0;   // inputs consumed and outputs produced since creation or the last reset
  int cur = 0;                               // which history buffer is live
  DevBuf<float> d_hT;                        // [L][P]
  DevBuf<float2> d_hist[2];                  // [C][P-1]
  int reset(cudaStream_t s) {
    n_in = n_outc = 0;
    cur = 0;
    QPSK_TRY(d_hist[0].zero(s));
    return QPSK_OK;
  }
  int init(const float* taps, int n_taps, int interp, int decim, int channels) {
    C = channels;
    L = interp;
    M = decim;
    N = n_taps;
    P = (N + L - 1) / L;
    QPSK_TRY(open());
    std::vector<float> hT((size_t)L * P, 0.0f);
    for (int i = 0; i < N; ++i) hT[(size_t)(i % L) * P + i / L] = taps[i];
    QPSK_TRY(d_hT.alloc(hT.size()));
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_hT.p, hT.data(), hT.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    if (P > 1)
      for (auto& hb : d_hist) QPSK_TRY(hb.alloc((size_t)C * (P - 1)));
    QPSK_TRY(reset(stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    return QPSK_OK;
  }
  long long outputs_for(long long n) const {
    return (long long)(resamp_count(n_in + (unsigned long long)n, L, M) - n_outc);
  }

  template <int CW, int CPT, int OPT, int CJ>
  int launch(const ResampArgs& a, cudaStream_t s) {
    using Sh = ResampShape<CW, CPT, OPT, CJ>;
    const auto k = resamp_kernel<CW, CPT, OPT, CJ>;
    QPSK_TRY(allow_max_dynamic_smem((const void*)k));
    const long long gx = (a.n_out + Sh::TB - 1) / Sh::TB;
    if (gx > 0x7fffffffLL) return QPSK_ERR_UNSUPPORTED;
    const dim3 grid((unsigned)gx, (unsigned)((C + Sh::CB - 1) / Sh::CB));
    k<<<grid, kResampThreads, Sh::smem(P), s>>>(a);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }

  // x: [C][ldx], n samples per row (device) -> y [C][ldy], outputs_for(n) per row; state advanced
  int process_dev(const float2* x, long long n, long long ldx, float2* y, long long ldy, cudaStream_t s) {
    if (n == 0) return QPSK_OK;
    if (!s) s = stream;
    ResampArgs a;
    a.hT = d_hT.p;
    a.P = P;
    a.L = L;
    a.M = M;
    a.hist = d_hist[cur].p;
    a.x = x;
    a.ldx = ldx;
    a.C = C;
    a.n_out = outputs_for(n);
    // first output m = n_outc: n_m = floor(mM / L), phi = mM mod L, from m = uL + v without forming mM
    const unsigned long long u = n_outc / (unsigned long long)L, v = n_outc % (unsigned long long)L;
    const unsigned long long n_m = u * (unsigned long long)M + v * (unsigned long long)M / (unsigned long long)L;
    a.phi0 = (int)(v * (unsigned long long)M % (unsigned long long)L);
    a.d0 = (long long)(n_m - n_in);
    a.y = y;
    a.ldy = ldy;
    if (a.n_out > 0) {
      if (C <= kResampSmallK)
        QPSK_TRY((launch<1, 1, 1, 2048>(a, s)));
      else
        QPSK_TRY((launch<32, 2, 4, 64>(a, s)));
    }
    if (P > 1) {
      const long long tot = (long long)C * (P - 1);
      const long long hb = std::min<long long>((tot + 255) / 256, 4096);
      resamp_history_kernel<<<(unsigned)hb, 256, 0, s>>>(a, n, d_hist[cur ^ 1].p);
      QPSK_LAUNCH_CHECK();
      cur ^= 1;
    }
    n_in += (unsigned long long)n;
    n_outc += (unsigned long long)a.n_out;
    return QPSK_OK;
  }
};

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_resamp {
  ResampEngine eng;
  DevBuf<float2> d_in, d_out;
};

extern "C" {

int qpsk_resamp_create(const float* taps, int n_taps, int interp, int decim, int channels, qpsk_resamp** out) {
  QPSK_TRY(clear_out(out));
  if (!taps) return QPSK_ERR_NULL;
  if (n_taps <= 0) return QPSK_ERR_ARG;
  if (n_taps > kResampMaxTaps || interp < 1 || interp > kResampMaxFactor || decim < 1 || decim > kResampMaxFactor ||
      channels < 1 || channels > kResampMaxChannels || (n_taps + interp - 1) / interp > kResampMaxBranch)
    return QPSK_ERR_UNSUPPORTED;
  for (int i = 0; i < n_taps; ++i)
    if (!isfinite(taps[i])) return QPSK_ERR_RANGE;
  return create_handle(out, taps, n_taps, interp, decim, channels);
}

int qpsk_resamp_destroy(qpsk_resamp* p) { return destroy_handle(p); }

int qpsk_resamp_reset(qpsk_resamp* p) { return reset_handle(p); }

int qpsk_resamp_process(qpsk_resamp* p, const float* iq_in, int64_t n_floats, float* iq_out, int64_t out_stride_floats,
                        int64_t* n_out_floats) {
  if (!p || !n_out_floats) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if (n_floats & 1) return QPSK_ERR_ARG;
  ResampEngine& g = p->eng;
  const long long n = n_floats >> 1, n_out = g.outputs_for(n);
  *n_out_floats = 2 * n_out;
  if (out_stride_floats < 2 * n_out) return QPSK_ERR_CAPACITY;
  if (n == 0) return QPSK_OK;
  if (!iq_in || (n_out > 0 && !iq_out)) return QPSK_ERR_NULL;
  return host_call(p, iq_in, g.C, (size_t)n * 8, iq_out, (size_t)out_stride_floats * 4, g.C, (size_t)n_out * 8,
                   [&](const float2* x, float2* y) { return g.process_dev(x, n, n, y, n_out, g.stream); });
}

int qpsk_resamp_process_dev(qpsk_resamp* p, const float* d_in, int64_t n_floats, int64_t in_stride_floats, float* d_out,
                            int64_t out_stride_floats, int64_t* n_out_floats, void* stream) {
  if (!p || !n_out_floats) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (in_stride_floats & 1) || (out_stride_floats & 1)) return QPSK_ERR_ARG;
  if (in_stride_floats < n_floats) return QPSK_ERR_ARG;
  ResampEngine& g = p->eng;
  const long long n = n_floats >> 1, n_out = g.outputs_for(n);
  *n_out_floats = 2 * n_out;
  if (out_stride_floats < 2 * n_out) return QPSK_ERR_CAPACITY;
  if (n == 0) return QPSK_OK;
  if (!d_in || (n_out > 0 && !d_out)) return QPSK_ERR_NULL;
  if (misaligned(d_in) || misaligned(d_out)) return QPSK_ERR_ARG;
  if (n_out > 0) {                                              // the rows read and the rows written must not overlap
    const uintptr_t i0 = reinterpret_cast<uintptr_t>(d_in), o0 = reinterpret_cast<uintptr_t>(d_out);
    const uintptr_t i1 = i0 + (uintptr_t)(((int64_t)(g.C - 1) * in_stride_floats + n_floats) * 4);
    const uintptr_t o1 = o0 + (uintptr_t)(((int64_t)(g.C - 1) * out_stride_floats + 2 * n_out) * 4);
    if (i0 < o1 && o0 < i1) return QPSK_ERR_ARG;
  }
  QPSK_TRY(ensure_device(g.device));
  return g.process_dev((const float2*)d_in, n, in_stride_floats >> 1, (float2*)d_out, out_stride_floats >> 1,
                       (cudaStream_t)stream);
}

}  // extern "C"
