// ddc.cu — frequency-translating decimating filter bank (spec: include/qpskcuda.h, "digital down-converter bank"): one
// wideband stream in, K channels tuned to their own frequencies f_k, each filtered by the real prototype h and decimated
// by D, out as [K][out_stride] rows.
//
// The kernel computes the rotated-tap form u_k[m] = sum_i g_k[i] x[n_m - i], g_k[i] = h[i] e^{+j 2 pi phi_k(i) / 2^64}
// (formed on the host in fp64, rounded to fp32), then y_k[m] = u_k[m] e^{-j 2 pi phi_k(n_m) / 2^64} in the epilogue.
// With r = N-1-i the sum is a complex matrix product per tile: U[k, t] = sum_r G[k, r] W[r, t], where
// W[r, t] = z[(m0+t)D + D-1 + r] and z = history ++ call input.
//
// ddc_kernel<CQW, WC, CC>: one CTA takes KB = 4*CQW*WC channels and TB consecutive outputs, and walks r in chunks of CC.
//   Staging.  Per chunk, the taps G[kc0 .., r0 + cc] go to shared memory as float4 (Re, Re, Im, Im), laid out [cc][kk][q]
//      (channel = 4q + kk) so the four channel quads a warp reads sit in 64 consecutive bytes; the input goes in
//      polyphase-transposed: row cc, column t holds z[(m0+t)D + D-1 + r0 + cc].  Consecutive outputs of one tap are then
//      consecutive in shared memory for every D, and a thread reads two outputs per LDS.128.  Every load is 8 bytes,
//      so no path depends on the caller's pointer alignment.
//   Micro-kernel.  A thread owns 4 channels x 4 outputs (outputs 2j, 2j+1, 2j+2*OQ, 2j+2*OQ+1 of its warp's span, so
//      each LDS.128 of a warp covers contiguous bytes).  Per tap: 4 LDS.128 of taps (broadcast within a channel quad),
//      2 LDS.128 of samples and 32 FFMA2: rr += (g.re, g.re) * (w.re, w.im) and ii += (g.im, g.im) * (w.re, w.im), so
//      u = (rr.x - ii.y, rr.y + ii.x) in the epilogue.
//   Epilogue.  phi = inc_k * n_m in exact 64-bit arithmetic; its top 32 bits give the angle (sincospif), applied once
//      per output.
// Two shapes: <4, 2, 32> (32 channels x 128 outputs per CTA) for K > 8, and <1, 1, 8> (4 channels x 1024 outputs) for
// K <= 8, where a 32-channel block would be mostly padding.  Every output is accumulated by the same instructions in the
// same order (r = 0 .. NP-1) wherever it falls in a tile, a call or the stream, so any chunking gives the same bits.
//
// History (like the FIR delay line): z starts with the N-1 samples before the open block and the pending samples of the
// open block, E = N-1 + pending, kept in a ping-pong buffer; ddc_history_kernel writes the next call's z head after the
// filter kernel.
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

#include "handle.cuh"

namespace qpsk {

constexpr int kDdcThreads = 256;
constexpr int kDdcMaxChannels = 2048;
constexpr int kDdcMaxDecim = 1024;
constexpr int kDdcMaxTaps = 4096;
constexpr int kDdcRowAlign = 32;        // tap rows padded to a multiple of every chunk size CC
constexpr int kDdcColAlign = 32;        // tap columns padded to a multiple of every channel block KB
constexpr int kDdcSmallK = 8;           // K <= this: the 4-channel shape

__device__ __forceinline__ float2 ddc_z(const float2* __restrict__ hist, long long E, const float2* __restrict__ x,
                                        long long j) {
  return j < E ? hist[j] : x[j - E];
}

template <int CQW, int WC, int CC>
struct DdcShape {
  static constexpr int OQ = 32 / CQW;             // output pairs-of-pairs per warp row
  static constexpr int OW = 4 * OQ;               // outputs per warp
  static constexpr int WO = (kDdcThreads / 32) / WC;
  static constexpr int TB = OW * WO;              // outputs per CTA
  static constexpr int KB = 4 * CQW * WC;         // channels per CTA
  static constexpr int PITCH = TB + 2;            // float2 per sample row: 16-byte rows, fewer store conflicts
  static constexpr size_t smem() { return (size_t)CC * PITCH * sizeof(float2) + (size_t)CC * KB * sizeof(float4); }
};

// g: [NP][ldg] rotated taps, row r = tap N-1-r (zero past N and past K); inc: [ldg] phase increments (zero past K).
// Output m of this call is stream output with n_m = n_base + m*D.
template <int CQW, int WC, int CC>
__global__ void __launch_bounds__(kDdcThreads, 2)
    ddc_kernel(const float2* __restrict__ g, int ldg, int NP, int N, const unsigned long long* __restrict__ inc, int K,
               int D, const float2* __restrict__ hist, long long E, const float2* __restrict__ x, long long n_out,
               unsigned long long n_base, float2* __restrict__ y, long long ldy) {
  using S = DdcShape<CQW, WC, CC>;
  extern __shared__ __align__(16) unsigned char ddc_smem[];
  float2* sx = reinterpret_cast<float2*>(ddc_smem);                                   // [CC][PITCH]
  float4* sg = reinterpret_cast<float4*>(ddc_smem + (size_t)CC * S::PITCH * sizeof(float2));  // [CC][4][KB/4]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cq = (warp / S::WO) * CQW + lane / S::OQ;       // channel quad in the CTA
  const int oq = lane % S::OQ;
  const int tA = (warp % S::WO) * S::OW + 2 * oq, tB = tA + 2 * S::OQ;
  const long long m0 = (long long)blockIdx.x * S::TB;
  const int kc0 = blockIdx.y * S::KB;
  const long long zb = m0 * D + (D - 1);

  float2 rr[4][4], ii[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) rr[a][b] = ii[a][b] = make_float2(0.0f, 0.0f);

  for (int r0 = 0; r0 < NP; r0 += CC) {
    __syncthreads();
    for (int e = tid; e < CC * S::KB; e += kDdcThreads) {
      const int cc = e / S::KB, c = e % S::KB;
      const float2 v = g[(long long)(r0 + cc) * ldg + kc0 + c];
      sg[(cc * 4 + (c & 3)) * (S::KB / 4) + (c >> 2)] = make_float4(v.x, v.x, v.y, v.y);
    }
    for (int e = tid; e < CC * S::TB; e += kDdcThreads) {
      const int cc = e % CC, t = e / CC;
      float2 v = make_float2(0.0f, 0.0f);
      if (r0 + cc < N && m0 + t < n_out) v = ddc_z(hist, E, x, zb + (long long)t * D + r0 + cc);
      sx[cc * S::PITCH + t] = v;
    }
    __syncthreads();
#pragma unroll 2
    for (int cc = 0; cc < CC; ++cc) {
      float4 tp[4];
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) tp[kk] = sg[(cc * 4 + kk) * (S::KB / 4) + cq];
      const float4 s0 = *reinterpret_cast<const float4*>(&sx[cc * S::PITCH + tA]);
      const float4 s1 = *reinterpret_cast<const float4*>(&sx[cc * S::PITCH + tB]);
      const float2 w[4] = {make_float2(s0.x, s0.y), make_float2(s0.z, s0.w), make_float2(s1.x, s1.y),
                           make_float2(s1.z, s1.w)};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float2 gr = make_float2(tp[kk].x, tp[kk].y), gi = make_float2(tp[kk].z, tp[kk].w);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          rr[kk][j] = ffma2(gr, w[j], rr[kk][j]);
          ii[kk][j] = ffma2(gi, w[j], ii[kk][j]);
        }
      }
    }
  }

#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    const int k = kc0 + cq * 4 + kk;
    if (k >= K) continue;
    const unsigned long long ik = inc[k];
    float2* yk = y + (long long)k * ldy;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long m = m0 + (j < 2 ? tA + j : tB + j - 2);
      if (m >= n_out) continue;
      const unsigned long long phi = ik * (n_base + (unsigned long long)m * (unsigned long long)D);
      // angle 2 pi phi / 2^64 = pi * (signed phi / 2^63); the top 32 bits carry it to 2^-31 of a half turn
      const float a = (float)(int)(unsigned)(phi >> 32) * 0x1p-31f;
      float sn, cs;
      sincospif(a, &sn, &cs);
      const float ur = rr[kk][j].x - ii[kk][j].y, ui = rr[kk][j].y + ii[kk][j].x;
      yk[m] = make_float2(fmaf(ur, cs, ui * sn), fmaf(ui, cs, -(ur * sn)));
    }
  }
}

// hist_out[i] = z[skip + i], i < n: the tail of z that becomes the next call's history
__global__ void ddc_history_kernel(const float2* __restrict__ hist, long long E, const float2* __restrict__ x, long long skip,
                                   float2* __restrict__ hist_out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    hist_out[i] = ddc_z(hist, E, x, skip + i);
}

// inc = nearbyint(ldexp(f, 64)) mod 2^64 for f in [-0.5, 0.5): the product fits int64 exactly
static unsigned long long ddc_phase_word(double f) { return (unsigned long long)(long long)nearbyint(ldexp(f, 64)); }

static bool ddc_freq_ok(double f) { return isfinite(f) && f >= -0.5 && f < 0.5; }

struct DdcEngine : EngineBase {
  int K = 0, D = 0, N = 0, NP = 0, ldg = 0;
  unsigned long long count = 0;          // samples since creation or the last reset
  int cur = 0;                           // which history buffer is live
  DevBuf<float2> d_g;                    // [NP][ldg]
  DevBuf<unsigned long long> d_inc;      // [ldg]
  DevBuf<float2> d_hist[2];              // [N-1 + D-1]
  long long pending() const { return (long long)(count % (unsigned long long)D); }
  long long hist_len() const { return (long long)N - 1 + pending(); }
  int reset(cudaStream_t s) {
    count = 0;
    cur = 0;
    QPSK_TRY(d_hist[0].zero(s));
    return QPSK_OK;
  }
  int init(const float* taps, int n_taps, const double* freqs, int channels, int decim) {
    K = channels;
    D = decim;
    N = n_taps;
    NP = (N + kDdcRowAlign - 1) / kDdcRowAlign * kDdcRowAlign;
    ldg = (K + kDdcColAlign - 1) / kDdcColAlign * kDdcColAlign;
    QPSK_TRY(open());
    std::vector<unsigned long long> inc((size_t)ldg, 0ULL);
    for (int k = 0; k < K; ++k) inc[k] = ddc_phase_word(freqs[k]);
    std::vector<float2> gt((size_t)NP * ldg, make_float2(0.0f, 0.0f));
    for (int i = 0; i < N; ++i) {
      const int r = N - 1 - i;
      for (int k = 0; k < K; ++k) {
        const long long ph = (long long)(inc[k] * (unsigned long long)i);       // phi_k(i), exact mod 2^64
        const double a = 2.0 * M_PI * ldexp((double)ph, -64);
        gt[(size_t)r * ldg + k] = make_float2((float)(taps[i] * cos(a)), (float)(taps[i] * sin(a)));
      }
    }
    QPSK_TRY(d_g.alloc(gt.size()));
    QPSK_TRY(d_inc.alloc(inc.size()));
    for (auto& hb : d_hist) QPSK_TRY(hb.alloc((size_t)N - 1 + D - 1 + 1));
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_g.p, gt.data(), gt.size() * sizeof(float2), cudaMemcpyHostToDevice, stream));
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_inc.p, inc.data(), inc.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, stream));
    QPSK_TRY(reset(stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    return QPSK_OK;
  }
  long long outputs_for(long long n) const { return (pending() + n) / D; }

  template <int CQW, int WC, int CC>
  int launch(const float2* h, long long E, const float2* x, long long n_out, unsigned long long n_base, float2* y,
             long long ldy, cudaStream_t s) {
    using Sh = DdcShape<CQW, WC, CC>;
    const auto k = ddc_kernel<CQW, WC, CC>;
    QPSK_TRY(allow_max_dynamic_smem((const void*)k));
    const dim3 grid((unsigned)((n_out + Sh::TB - 1) / Sh::TB), (unsigned)((K + Sh::KB - 1) / Sh::KB));
    k<<<grid, kDdcThreads, Sh::smem(), s>>>(d_g.p, ldg, NP, N, d_inc.p, K, D, h, E, x, n_out, n_base, y, ldy);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }

  // x: n samples (device) -> y [K][ldy], outputs_for(n) per row; state advanced
  int process_dev(const float2* x, long long n, float2* y, long long ldy, cudaStream_t s) {
    if (n == 0) return QPSK_OK;
    if (!s) s = stream;
    const long long n_out = outputs_for(n);
    const long long E = hist_len();
    const float2* h = d_hist[cur].p;
    if (n_out > 0) {
      const unsigned long long n_base = (count - (unsigned long long)pending()) + (unsigned long long)(D - 1);
      if (K <= kDdcSmallK)
        QPSK_TRY((launch<1, 1, 8>(h, E, x, n_out, n_base, y, ldy, s)));
      else
        QPSK_TRY((launch<4, 2, 32>(h, E, x, n_out, n_base, y, ldy, s)));
    }
    const long long keep = (long long)N - 1 + (pending() + n) % D;
    if (keep > 0) {
      const long long blocks = std::min<long long>((keep + 255) / 256, 4096);
      ddc_history_kernel<<<(unsigned)blocks, 256, 0, s>>>(h, E, x, n_out * D, d_hist[cur ^ 1].p, keep);
      QPSK_LAUNCH_CHECK();
    }
    cur ^= 1;
    count += (unsigned long long)n;
    return QPSK_OK;
  }
};

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_ddc {
  DdcEngine eng;
  DevBuf<float2> d_in, d_out;
};

extern "C" {

int qpsk_ddc_create(const float* taps, int n_taps, const double* freqs, int channels, int decim, qpsk_ddc** out) {
  QPSK_TRY(clear_out(out));
  if (!taps || !freqs) return QPSK_ERR_NULL;
  if (n_taps <= 0) return QPSK_ERR_ARG;
  if (n_taps > kDdcMaxTaps || channels < 1 || channels > kDdcMaxChannels || decim < 1 || decim > kDdcMaxDecim)
    return QPSK_ERR_UNSUPPORTED;
  for (int i = 0; i < n_taps; ++i)
    if (!isfinite(taps[i])) return QPSK_ERR_RANGE;
  for (int k = 0; k < channels; ++k)
    if (!ddc_freq_ok(freqs[k])) return QPSK_ERR_RANGE;
  return create_handle(out, taps, n_taps, freqs, channels, decim);
}

int qpsk_ddc_destroy(qpsk_ddc* p) { return destroy_handle(p); }

int qpsk_ddc_reset(qpsk_ddc* p) { return reset_handle(p); }

int qpsk_ddc_process(qpsk_ddc* p, const float* iq_in, int64_t n_floats, float* iq_out, int64_t out_stride_floats,
                     int64_t* n_out_floats) {
  if (!p || !n_out_floats) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if (n_floats & 1) return QPSK_ERR_ARG;
  DdcEngine& g = p->eng;
  const long long n = n_floats >> 1, n_out = g.outputs_for(n);
  *n_out_floats = 2 * n_out;
  if (out_stride_floats < 2 * n_out) return QPSK_ERR_CAPACITY;
  if (n == 0) return QPSK_OK;
  if (!iq_in || (n_out > 0 && !iq_out)) return QPSK_ERR_NULL;
  return host_call(p, iq_in, 1, (size_t)n * 8, iq_out, (size_t)out_stride_floats * 4, g.K, (size_t)n_out * 8,
                   [&](const float2* x, float2* y) { return g.process_dev(x, n, y, n_out, g.stream); });
}

int qpsk_ddc_process_dev(qpsk_ddc* p, const float* d_in, int64_t n_floats, float* d_out, int64_t out_stride_floats,
                         int64_t* n_out_floats, void* stream) {
  if (!p || !n_out_floats) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (out_stride_floats & 1)) return QPSK_ERR_ARG;
  DdcEngine& g = p->eng;
  const long long n = n_floats >> 1, n_out = g.outputs_for(n);
  *n_out_floats = 2 * n_out;
  if (out_stride_floats < 2 * n_out) return QPSK_ERR_CAPACITY;
  if (n == 0) return QPSK_OK;
  if (!d_in || (n_out > 0 && !d_out)) return QPSK_ERR_NULL;
  if (misaligned(d_in) || misaligned(d_out)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(g.device));
  return g.process_dev((const float2*)d_in, n, (float2*)d_out, out_stride_floats >> 1, (cudaStream_t)stream);
}

}  // extern "C"
