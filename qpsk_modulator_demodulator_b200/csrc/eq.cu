// eq.cu — cma_eq_kernel: the blind CMA equalizer (symbol-spaced, or T/S-spaced with update stride S), batched over
// independent channels.  Compiled with --fmad=false: every product and sum of the spec (include/qpskcuda.h) rounds
// separately, as in the oracle.
//
// Layout: 8 lanes per channel, 4 channels per warp.  Lane l holds the taps w_k and window entries v_k with k = l + 8j
// (slot j < J = ceil(N/8)) in registers, so its running sum over its slots is the spec's lane partial s_l, and the
// xor-shuffle butterfly (1, 2, 4) forms ((s0+s1)+(s2+s3))+((s4+s5)+(s6+s7)) in every lane (a+b == b+a exactly, so all
// eight lanes hold the same bits of y and of the error).  The window shifts by one lane per symbol (lane 0 takes lane 7's
// previous slot), and input / output move in blocks of 8 symbols, one per lane, coalesced per channel row.
//
// Update stride S (the fractionally spaced form, include/qpskcuda.h): the taps update only on stream samples n with
// n % S == 0.  For S = 2, 4, 8 (divisors of the block of 8) a channel whose counter stands at phase o = n mod S when the
// call starts runs its block loop o slots early (its first o slots idle): the update samples are then the slots i = 0
// (mod S) of every block, known at compile time, and the S - 1 outputs between two updates use fixed taps, so their dot
// products are off the update chain and the scheduler overlaps them with it.  The phase differs between the channels of a
// warp; only the idle slots and the stores depend on it.  Other strides (3, 5, 6, 7: S = 0 below) keep a running phase per
// channel and test it at run time.  S = 1 is the symbol-spaced equalizer, and compiles to the code without the stride.
#include <math.h>

#include "eq.cuh"

namespace qpsk {

constexpr int kEqThreads = 64;   // 8 channels per CTA: 2048 channels fill 256 CTAs

int eq_check_params(int n_taps, float mu, float modulus, int sps) {
  if (!(isfinite(mu) && mu >= 0.0f) || !(isfinite(modulus) && modulus > 0.0f)) return QPSK_ERR_RANGE;
  if (n_taps < 1 || n_taps > kEqMaxTaps) return QPSK_ERR_UNSUPPORTED;
  if (sps < 1 || sps > kEqMaxSps) return QPSK_ERR_UNSUPPORTED;
  return QPSK_OK;
}

__global__ void eq_reset_kernel(float2* taps, float2* win, int* drop, int* phase, int N, int C) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)C * N) return;
  const int k = (int)(i % N);
  taps[i] = make_float2(k == (N - 1) / 2 ? 1.0f : 0.0f, 0.0f);
  win[i] = make_float2(0.0f, 0.0f);
  if (k == 0) drop[i / N] = (N - 1) / 2;
  if (k == 0 && phase) phase[i / N] = 0;
}

// S: the update stride, 1, 2, 4 or 8; 0 = the stride P.sps taken at run time.  phase[c] = the channel's stream counter
// mod the stride (unused, and may be null, for S = 1).  S != 1: at least 8 CTAs per SM (<= 128 registers) keeps ptxas
// from a 4-byte spill it otherwise picks at J = 6; S = 1 keeps the bounds it always had (0 = no minimum).
template <int J, int S>
__global__ void __launch_bounds__(kEqThreads, S == 1 ? 0 : 8)
    cma_eq_kernel(const EqParams P, float2* __restrict__ taps, float2* __restrict__ win, int* __restrict__ drop, int C,
                  const float2* __restrict__ x, long long ldx, float2* __restrict__ y, long long ldy, long long L,
                  const int* __restrict__ n_in, int* __restrict__ n_out, int* __restrict__ phase) {
  constexpr bool kShift = S == 2 || S == 4 || S == 8;   // idle leading slots put the updates on slots i = 0 (mod S)
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int c = t >> 3;
  const int l = t & 7;
  const int lane = threadIdx.x & 31;
  const int base = lane & ~7;                      // first lane of this channel's group
  const int left = base | ((l + 7) & 7);           // lane holding v_{k-1} of this lane's slots (lane 0: lane 7, slot j-1)
  const unsigned full = 0xffffffffu;
  const bool live = c < C;
  const int N = P.n_taps;
  const long long n = live ? (n_in ? (long long)n_in[c] : L) : 0;
  int ph = 0;                                      // kShift: idle leading slots; S = 0: phase of the next sample
  if (S != 1 && live) ph = phase[c];
  const int off = kShift ? ph : 0;
  const long long nv = n + off;                    // slots of this channel's loop
  float wr[J], wi[J], vr[J], vi[J];
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int k = l + 8 * j;
    float2 w0 = make_float2(0.f, 0.f), v0 = make_float2(0.f, 0.f);
    if (live && k < N) { w0 = taps[(long long)c * N + k]; v0 = win[(long long)c * N + k]; }
    wr[j] = w0.x; wi[j] = w0.y; vr[j] = v0.x; vi[j] = v0.y;
  }
  long long dc = 0;
  if (drop && live) {
    const long long d0 = drop[c];
    dc = d0 < n ? d0 : n;
  }
  // every lane of the warp runs the longest of its four channels' loops: the shuffles need the whole warp
  const int nmax = __reduce_max_sync(full, (int)nv);
  const float2* xc = x + (long long)(live ? c : 0) * ldx;
  float2* yc = y + (long long)(live ? c : 0) * ldy;
  float2 cur = make_float2(0.f, 0.f);
  if ((!kShift || l >= off) && l - off < n) cur = xc[l - off];
  for (long long b = 0; b < nmax; b += 8) {
    float2 nxt = make_float2(0.f, 0.f);
    const long long kn = b + 8 + l - off;
    if ((!kShift || kn >= 0) && kn < n) nxt = xc[kn];   // next block in flight while this one runs
    float2 keep = make_float2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float xr = __shfl_sync(full, cur.x, base | i);
      const float xi = __shfl_sync(full, cur.y, base | i);
      const bool active = kShift ? (b + i >= off && b + i < nv) : (b + i < n);
      // this sample updates the taps: every sample (S = 1), slot i = 0 (mod S), or the running phase at 0 (S = 0)
      const bool upd = active && (S == 1 || (kShift ? (i % (kShift ? S : 1)) == 0 : ph == 0));
      if (S == 0 && active) ph = (ph + 1 == P.sps) ? 0 : ph + 1;
      // window shift: v_k <- v_{k-1}, v_0 <- x_n
      float sr[J], si[J];
#pragma unroll
      for (int j = 0; j < J; ++j) {
        sr[j] = __shfl_sync(full, vr[j], left);
        si[j] = __shfl_sync(full, vi[j], left);
      }
      if (active) {
#pragma unroll
        for (int j = J - 1; j >= 0; --j) {
          if (l != 0) { vr[j] = sr[j]; vi[j] = si[j]; }
          else if (j > 0) { vr[j] = sr[j - 1]; vi[j] = si[j - 1]; }
          else { vr[0] = xr; vi[0] = xi; }
        }
      }
      // lane partial s_l = +0 + P_l + P_{l+8} + ...
      float pr = 0.0f, pi = 0.0f;
#pragma unroll
      for (int j = 0; j < J; ++j) {
        if (l + 8 * j < N) {
          const float a = wr[j] * vr[j], bb = wi[j] * vi[j], cc = wr[j] * vi[j], d = wi[j] * vr[j];
          pr = pr + (a - bb);
          pi = pi + (cc + d);
        }
      }
      pr = pr + __shfl_xor_sync(full, pr, 1);
      pi = pi + __shfl_xor_sync(full, pi, 1);
      pr = pr + __shfl_xor_sync(full, pr, 2);
      pi = pi + __shfl_xor_sync(full, pi, 2);
      pr = pr + __shfl_xor_sync(full, pr, 4);
      pi = pi + __shfl_xor_sync(full, pi, 4);
      const float dm = (pr * pr + pi * pi) - P.modulus;
      const float er = fminf(fmaxf(pr * dm, -1.0f), 1.0f);
      const float ei = fminf(fmaxf(pi * dm, -1.0f), 1.0f);
      if (upd) {
#pragma unroll
        for (int j = 0; j < J; ++j) {
          if (l + 8 * j < N) {
            const float gr = er * vr[j] + ei * vi[j];
            const float gi = ei * vr[j] - er * vi[j];
            wr[j] = wr[j] - P.mu * gr;
            wi[j] = wi[j] - P.mu * gi;
          }
        }
      }
      if (l == i) keep = make_float2(pr, pi);
    }
    const long long k = b + l - off;
    if (k < n && k >= dc) yc[k - dc] = keep;           // dc >= 0: the idle slots (k < 0) store nothing
    cur = nxt;
  }
  if (!live) return;
#pragma unroll
  for (int j = 0; j < J; ++j) {
    const int k = l + 8 * j;
    if (k < N) {
      taps[(long long)c * N + k] = make_float2(wr[j], wi[j]);
      win[(long long)c * N + k] = make_float2(vr[j], vi[j]);
    }
  }
  if (l == 0) {
    if (drop) drop[c] -= (int)dc;
    if (n_out) n_out[c] = (int)(n - dc);
    if (kShift) phase[c] = (int)((off + n) % (kShift ? S : 1));
    else if (S == 0) phase[c] = ph;
  }
}

EqEngine::~EqEngine() {
  if (stream) cudaStreamDestroy(stream);
}

int EqEngine::init(int n_taps, float mu, float modulus, int sps, int channels_in) {
  QPSK_TRY(eq_check_params(n_taps, mu, modulus, sps));
  if (channels_in <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device());
  device = current_device();
  channels = channels_in;
  P.n_taps = n_taps;
  P.mu = mu;
  P.modulus = modulus;
  P.sps = sps;
  QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  QPSK_TRY(d_taps.alloc((size_t)channels * n_taps));
  QPSK_TRY(d_win.alloc((size_t)channels * n_taps));
  QPSK_TRY(d_drop.alloc((size_t)channels));
  if (sps > 1) QPSK_TRY(d_phase.alloc((size_t)channels));
  QPSK_TRY(reset(stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  return QPSK_OK;
}

int EqEngine::reset(cudaStream_t s) {
  if (!s) s = stream;
  const long long tot = (long long)channels * P.n_taps;
  eq_reset_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, s>>>(d_taps.p, d_win.p, d_drop.p, d_phase.p, P.n_taps, channels);
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}

int EqEngine::process_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, const int* d_n_in, int* d_n_out,
                          bool drop, cudaStream_t s) {
  if (L == 0) return QPSK_OK;
  if (!x || !y) return QPSK_ERR_NULL;
  if (!s) s = stream;
  const long long threads = (long long)channels * 8;
  const unsigned grid = (unsigned)((threads + kEqThreads - 1) / kEqThreads);
  int* dr = drop ? d_drop.p : nullptr;
#define QPSK_EQ_LAUNCH(JJ, SS)                                                                                          \
  cma_eq_kernel<JJ, SS><<<grid, kEqThreads, 0, s>>>(P, d_taps.p, d_win.p, dr, channels, x, (long long)ldx, y,             \
                                                    (long long)ldy, (long long)L, d_n_in, d_n_out, d_phase.p)
#define QPSK_EQ_STRIDES(JJ)                  \
  switch (P.sps) {                           \
    case 1: QPSK_EQ_LAUNCH(JJ, 1); break;    \
    case 2: QPSK_EQ_LAUNCH(JJ, 2); break;    \
    case 4: QPSK_EQ_LAUNCH(JJ, 4); break;    \
    case 8: QPSK_EQ_LAUNCH(JJ, 8); break;    \
    default: QPSK_EQ_LAUNCH(JJ, 0); break;   \
  }
  switch ((P.n_taps + 7) / 8) {
    case 1: QPSK_EQ_STRIDES(1); break;
    case 2: QPSK_EQ_STRIDES(2); break;
    case 3: QPSK_EQ_STRIDES(3); break;
    case 4: QPSK_EQ_STRIDES(4); break;
    case 5: QPSK_EQ_STRIDES(5); break;
    case 6: QPSK_EQ_STRIDES(6); break;
    case 7: QPSK_EQ_STRIDES(7); break;
    default: QPSK_EQ_STRIDES(8); break;
  }
#undef QPSK_EQ_STRIDES
#undef QPSK_EQ_LAUNCH
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_eq {
  EqEngine eng;
  DevBuf<float2> d_in, d_out;
};

extern "C" {

int qpsk_eq_create_fractional(int n_taps, float mu, float modulus, int sps, int channels, qpsk_eq** out) {
  if (!out) return QPSK_ERR_NULL;
  *out = nullptr;
  QPSK_TRY(eq_check_params(n_taps, mu, modulus, sps));
  qpsk_eq* e = new (std::nothrow) qpsk_eq();
  if (!e) return QPSK_ERR_NOMEM;
  int st = e->eng.init(n_taps, mu, modulus, sps, channels);
  if (st != QPSK_OK) { delete e; return st; }
  *out = e;
  return QPSK_OK;
}
int qpsk_eq_create_batch(int n_taps, float mu, float modulus, int channels, qpsk_eq** out) {
  return qpsk_eq_create_fractional(n_taps, mu, modulus, 1, channels, out);
}
int qpsk_eq_create(int n_taps, float mu, float modulus, qpsk_eq** out) {
  return qpsk_eq_create_batch(n_taps, mu, modulus, 1, out);
}
int qpsk_eq_destroy(qpsk_eq* e) {
  if (e) {
    if (e->eng.stream) cudaStreamSynchronize(e->eng.stream);
    delete e;
  }
  return QPSK_OK;
}
int qpsk_eq_reset(qpsk_eq* e) {
  if (!e) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(e->eng.device));
  QPSK_TRY(e->eng.reset(e->eng.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e->eng.stream));
  return QPSK_OK;
}
int qpsk_eq_process(qpsk_eq* e, const float* in, float* out, int64_t n_floats, int64_t out_cap_floats) {
  if (!e) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;
  if (out_cap_floats < n_floats) return QPSK_ERR_CAPACITY;
  if (n_floats == 0) return QPSK_OK;
  if (!in || !out) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(e->eng.device));
  EqEngine& g = e->eng;
  const int64_t L = n_floats >> 1;
  const size_t tot = (size_t)L * g.channels;
  QPSK_TRY(e->d_in.ensure(tot));
  QPSK_TRY(e->d_out.ensure(tot));
  QPSK_CUDA_TRY(cudaMemcpyAsync(e->d_in.p, in, tot * 8, cudaMemcpyHostToDevice, g.stream));
  QPSK_TRY(g.process_dev(e->d_in.p, e->d_out.p, L, L, L, nullptr, nullptr, false, g.stream));
  QPSK_CUDA_TRY(cudaMemcpyAsync(out, e->d_out.p, tot * 8, cudaMemcpyDeviceToHost, g.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(g.stream));
  return QPSK_OK;
}
int qpsk_eq_process_dev(qpsk_eq* e, const float* d_in, float* d_out, int64_t n_floats, int64_t is, int64_t os, const int* d_n_sym,
                        void* stream) {
  if (!e) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (is & 1) || (os & 1)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(e->eng.device));
  return e->eng.process_dev((const float2*)d_in, (float2*)d_out, n_floats >> 1, is >> 1, os >> 1, d_n_sym, nullptr, false,
                            (cudaStream_t)stream);
}
int qpsk_eq_get_taps(qpsk_eq* e, float* taps_iq, int64_t cap_floats) {
  if (!e || !taps_iq) return QPSK_ERR_NULL;
  EqEngine& g = e->eng;
  const int64_t need = (int64_t)g.channels * 2 * g.P.n_taps;
  if (cap_floats < need) return QPSK_ERR_CAPACITY;
  QPSK_TRY(ensure_device(g.device));
  QPSK_CUDA_TRY(cudaStreamSynchronize(g.stream));
  QPSK_CUDA_TRY(cudaMemcpy(taps_iq, g.d_taps.p, (size_t)need * 4, cudaMemcpyDeviceToHost));
  return QPSK_OK;
}
int qpsk_eq_set_taps(qpsk_eq* e, const float* taps_iq, int64_t n_floats) {
  if (!e || !taps_iq) return QPSK_ERR_NULL;
  EqEngine& g = e->eng;
  const int64_t need = (int64_t)g.channels * 2 * g.P.n_taps;
  if (n_floats != need) return QPSK_ERR_ARG;
  for (int64_t i = 0; i < n_floats; ++i)
    if (!isfinite(taps_iq[i])) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device(g.device));
  QPSK_CUDA_TRY(cudaStreamSynchronize(g.stream));
  QPSK_CUDA_TRY(cudaMemcpy(g.d_taps.p, taps_iq, (size_t)need * 4, cudaMemcpyHostToDevice));
  return QPSK_OK;
}

}  // extern "C"
