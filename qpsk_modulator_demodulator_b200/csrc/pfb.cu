// pfb.cu — critically sampled polyphase analysis channelizer (spec: include/qpskcuda.h, "polyphase analysis
// channelizer"): one wideband stream in, M channels of n/M samples out, channel-major.
//
// pfb_kernel<P>: one CTA takes T consecutive output blocks m0 .. m0+T-1.
//   1. Branch sums.  Thread (r, g) owns branch r and R consecutive blocks (g-th run of the tile).  Its P taps h[qM + r]
//      sit in registers and its window of P samples x[jM + M-1-r] is a circular register buffer (slot j mod P, resolved
//      at compile time by unrolling the block loop P-fold), so each block costs one 8-byte load and 2P FMAs.  The
//      warp's loads are 32 consecutive samples of the stream.  v_r[m] = sum_{q=0..P-1} h[qM + r] * x[(m-q)M + M-1-r],
//      accumulated from +0 in increasing q.  Each v_r[m] goes to shared memory, row m - m0, column r.
//   2. T inverse M-point DFTs in shared memory: decimation in frequency (natural-order input, bit-reversed output),
//      radix-2^2 passes (two radix-2 stages per pass, one sync each) after one radix-2 stage when log2 M is odd.  Twiddles
//      are e^{+j 2 pi t / M} from an fp64 table rounded to fp32.
//   3. Transposed store: output k of block m is read from row m - m0, column bitrev(k), and written to y[k][m]; a warp
//      writes 32 consecutive m of one k (256 B) where T >= 32.  Rows are M+1 entries long, so that read is free of bank
//      conflicts.
// Every output is computed by the same instructions in the same order wherever its block falls (in a tile, in a call,
// in the stream), so any chunking of a stream gives the same bits.  The input is read through z = history ++ call input
// (8-byte loads), so no path depends on the alignment of the caller's pointer.
//
// History (like the FIR delay line): z starts with the last (P-1) complete blocks and the pending samples of the open
// block, E = (P-1)M + pending samples kept in a ping-pong buffer; pfb_history_kernel writes the new tail of z into the
// other buffer after the channelizer kernel.
#include <math.h>

#include <algorithm>
#include <vector>

#include "handle.cuh"

namespace qpsk {

constexpr int kPfbThreads = 256;
constexpr int kPfbMaxChannels = 1024;
constexpr int kPfbMaxTapsPerBranch = 32;

// the sample at index j of z = hist[0..E) ++ x
__device__ __forceinline__ float2 pfb_z(const float2* __restrict__ hist, long long E, const float2* __restrict__ x,
                                        long long j) {
  return j < E ? hist[j] : x[j - E];
}

// Outputs m of this call are blocks n_out_done + m of the stream; z index (m + P-1)M + M-1-r is x[mM + M-1-r] of the
// spec relative to the call.  R: blocks per thread run; T = R * max(1, kPfbThreads / M).
template <int P>
__global__ void __launch_bounds__(kPfbThreads, 1)
    pfb_kernel(const float* __restrict__ taps, const float2* __restrict__ tw, int M, int log2m, int R,
               const float2* __restrict__ hist, long long E, const float2* __restrict__ x, long long n_out,
               float2* __restrict__ y, long long ldy) {
  extern __shared__ float2 sm[];
  const int tid = threadIdx.x;
  const int pitch = M + 1;
  const int G = M < kPfbThreads ? kPfbThreads / M : 1;
  const int T = R * G;                                      // M, R, G and T are powers of two: index math by shifts
  const int log2t = 31 - __clz(T);
  const long long m0 = (long long)blockIdx.x * T;
  const int tile = (int)(n_out - m0 < T ? n_out - m0 : T);

  // ---- 1. branch sums --------------------------------------------------------------------------------------------
  for (int rr = tid; rr < G * M; rr += kPfbThreads) {     // one pass when M <= kPfbThreads, M / kPfbThreads otherwise
    const int r = rr & (M - 1);
    const int g = rr >> log2m;
    const int b0 = g * R;                                   // first block of this run, relative to the tile
    const int b1 = min(b0 + R, tile);
    if (b0 >= b1) continue;
    float h[P];
#pragma unroll
    for (int q = 0; q < P; ++q) h[q] = taps[q * M + r];
    const long long zb = (m0 + b0) * M + (M - 1 - r);       // z index of the run's oldest sample (q = P-1 of block b0)
    float2 w[P];                                            // w[j mod P] = z[zb + j*M]
    long long zn = zb;                                      // z index of the next sample to load
#pragma unroll
    for (int j = 0; j < P - 1; ++j, zn += M) w[j] = pfb_z(hist, E, x, zn);
    for (int base = 0; base < b1 - b0; base += P) {
#pragma unroll
      for (int u = 0; u < P; ++u) {
        const int b = b0 + base + u;
        if (b < b1) {
          w[(u + P - 1) % P] = pfb_z(hist, E, x, zn);
          zn += M;
          float ar = 0.0f, ai = 0.0f;
#pragma unroll
          for (int q = 0; q < P; ++q) {
            const float2 s = w[(u + P - 1 - q) % P];
            ar = fmaf(h[q], s.x, ar);
            ai = fmaf(h[q], s.y, ai);
          }
          sm[b * pitch + r] = make_float2(ar, ai);
        }
      }
    }
  }
  __syncthreads();

  // ---- 2. inverse DFTs, decimation in frequency --------------------------------------------------------------------
  int h = M >> 1;                                           // butterfly span of the next radix-2 stage
  if (log2m & 1) {
    const int items = tile * (M >> 1);
    for (int it = tid; it < items; it += kPfbThreads) {
      const int b = it >> (log2m - 1), j = it & (h - 1);
      float2* row = sm + b * pitch;
      const float2 a = row[j], c = row[j + h];
      const float2 t = __ldg(&tw[j]);
      const float dr = a.x - c.x, di = a.y - c.y;
      row[j] = make_float2(a.x + c.x, a.y + c.y);
      row[j + h] = make_float2(fmaf(dr, t.x, -(di * t.y)), fmaf(dr, t.y, di * t.x));
    }
    h >>= 1;
    __syncthreads();
  }
  for (int log2h = 31 - __clz(max(h, 1)); h >= 2; h >>= 2, log2h -= 2) {   // stages h and h/2 in one pass over groups of 2h
    const int hh = h >> 1;
    const int items = tile << (log2m - 2);                  // M/4 groups of four per row
    const int s1 = M >> (log2h + 1), s2 = M >> log2h;       // twiddle strides of the two stages
    for (int it = tid; it < items; it += kPfbThreads) {
      const int b = it >> (log2m - 2), p = it & ((M >> 2) - 1);
      const int j = p & (hh - 1);
      const int i0 = ((p >> (log2h - 1)) << (log2h + 1)) + j;
      float2* row = sm + b * pitch;
      const float2 x0 = row[i0], x1 = row[i0 + hh], x2 = row[i0 + h], x3 = row[i0 + h + hh];
      const float2 ta = __ldg(&tw[j * s1]), tb = __ldg(&tw[(j + hh) * s1]), tc = __ldg(&tw[j * s2]);
      // stage h: (x0, x2) with ta, (x1, x3) with tb
      const float2 a0 = make_float2(x0.x + x2.x, x0.y + x2.y);
      const float2 a1 = make_float2(x1.x + x3.x, x1.y + x3.y);
      float dr = x0.x - x2.x, di = x0.y - x2.y;
      const float2 a2 = make_float2(fmaf(dr, ta.x, -(di * ta.y)), fmaf(dr, ta.y, di * ta.x));
      dr = x1.x - x3.x;
      di = x1.y - x3.y;
      const float2 a3 = make_float2(fmaf(dr, tb.x, -(di * tb.y)), fmaf(dr, tb.y, di * tb.x));
      // stage h/2: (a0, a1) and (a2, a3), both with tc
      row[i0] = make_float2(a0.x + a1.x, a0.y + a1.y);
      dr = a0.x - a1.x;
      di = a0.y - a1.y;
      row[i0 + hh] = make_float2(fmaf(dr, tc.x, -(di * tc.y)), fmaf(dr, tc.y, di * tc.x));
      row[i0 + h] = make_float2(a2.x + a3.x, a2.y + a3.y);
      dr = a2.x - a3.x;
      di = a2.y - a3.y;
      row[i0 + h + hh] = make_float2(fmaf(dr, tc.x, -(di * tc.y)), fmaf(dr, tc.y, di * tc.x));
    }
    __syncthreads();
  }

  // ---- 3. transposed store -------------------------------------------------------------------------------------------
  const int items = T * M;
  for (int it = tid; it < items; it += kPfbThreads) {
    const int k = it >> log2t, b = it & (T - 1);
    if (b < tile) {
      const int col = (int)(__brev((unsigned)k) >> (32 - log2m));
      y[(long long)k * ldy + m0 + b] = sm[b * pitch + col];
    }
  }
}

// hist_out[i] = z[skip + i], i < n: the tail of z that becomes the next call's history
__global__ void pfb_history_kernel(const float2* __restrict__ hist, long long E, const float2* __restrict__ x, long long skip,
                                   float2* __restrict__ hist_out, long long n) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    hist_out[i] = pfb_z(hist, E, x, skip + i);
}

using PfbKernel = void (*)(const float*, const float2*, int, int, int, const float2*, long long, const float2*, long long,
                           float2*, long long);

template <int... Ps>
struct PfbTable {
  static constexpr PfbKernel k[sizeof...(Ps)] = {&pfb_kernel<Ps>...};
};
using PfbKernels = PfbTable<1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22, 23, 24, 25, 26, 27,
                            28, 29, 30, 31, 32>;

// blocks per thread run: T = R * max(1, threads / M) blocks per tile, T * (M+1) * 8 bytes (about 64 KiB) of shared memory,
// three CTAs per SM.  Channel rows get 256 B per tile up to M = 256, 128 B at M = 512 and 64 B at M = 1024.
static int pfb_run_blocks(int M) { return M <= kPfbThreads ? 32 : 65536 / (M * 8); }

static bool pfb_pow2_channels(int M) { return M >= 2 && M <= kPfbMaxChannels && (M & (M - 1)) == 0; }

struct PfbEngine : EngineBase {
  int M = 0, log2m = 0, P = 0;
  long long pending = 0;                 // samples of the open block
  int cur = 0;                           // which history buffer is live
  DevBuf<float> d_taps;                  // [P][M], zero-padded
  DevBuf<float2> d_tw;                   // [M/2] e^{+j 2 pi t / M}
  DevBuf<float2> d_hist[2];              // [(P-1)M + M - 1]
  long long hist_len() const { return (long long)(P - 1) * M + pending; }
  int reset(cudaStream_t s) {
    pending = 0;
    cur = 0;
    QPSK_TRY(d_hist[0].zero(s));
    return QPSK_OK;
  }
  int init(const float* taps, int n_taps, int channels) {
    M = channels;
    P = (n_taps + M - 1) / M;
    while ((1 << log2m) < M) ++log2m;
    QPSK_TRY(open());
    std::vector<float> hp((size_t)P * M, 0.0f);
    for (int i = 0; i < n_taps; ++i) hp[i] = taps[i];
    std::vector<float2> tw((size_t)M / 2);
    for (int t = 0; t < M / 2; ++t) {
      const double a = 2.0 * M_PI * (double)t / (double)M;
      tw[t] = make_float2((float)cos(a), (float)sin(a));
    }
    QPSK_TRY(d_taps.alloc(hp.size()));
    QPSK_TRY(d_tw.alloc(tw.size()));
    for (auto& hb : d_hist) QPSK_TRY(hb.alloc((size_t)P * M));
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_taps.p, hp.data(), hp.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_tw.p, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice, stream));
    QPSK_TRY(reset(stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    return QPSK_OK;
  }
  long long outputs_for(long long n) const { return (pending + n) / M; }
  // x: n samples (device) -> y [M][ldy], outputs_for(n) per row; state advanced
  int process_dev(const float2* x, long long n, float2* y, long long ldy, cudaStream_t s) {
    if (n == 0) return QPSK_OK;
    if (!s) s = stream;
    const long long n_out = outputs_for(n);
    const long long E = hist_len();
    const float2* h = d_hist[cur].p;
    if (n_out > 0) {
      const int R = pfb_run_blocks(M);
      const int T = R * (M < kPfbThreads ? kPfbThreads / M : 1);
      const size_t smem = (size_t)T * (M + 1) * sizeof(float2);
      const PfbKernel k = PfbKernels::k[P - 1];
      QPSK_TRY(allow_max_dynamic_smem((const void*)k));
      const long long grid = (n_out + T - 1) / T;
      k<<<(unsigned)grid, kPfbThreads, smem, s>>>(d_taps.p, d_tw.p, M, log2m, R, h, E, x, n_out, y, ldy);
      QPSK_LAUNCH_CHECK();
    }
    const long long keep = (long long)(P - 1) * M + (pending + n) % M;
    if (keep > 0) {
      const long long blocks = std::min<long long>((keep + 255) / 256, 4096);
      pfb_history_kernel<<<(unsigned)blocks, 256, 0, s>>>(h, E, x, n_out * M, d_hist[cur ^ 1].p, keep);
      QPSK_LAUNCH_CHECK();
    }
    cur ^= 1;
    pending = (pending + n) % M;
    return QPSK_OK;
  }
};

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_pfb {
  PfbEngine eng;
  DevBuf<float2> d_in, d_out;
};

namespace {

double bessel_i0(double x) {
  const double q = 0.25 * x * x;
  double term = 1.0, sum = 1.0;
  for (int k = 1; k < 500; ++k) {
    term *= q / ((double)k * (double)k);
    sum += term;
    if (term < 1e-17 * sum) break;
  }
  return sum;
}

// scipy.signal.kaiser_beta
double kaiser_beta(double a) {
  if (a > 50.0) return 0.1102 * (a - 8.7);
  if (a > 21.0) return 0.5842 * pow(a - 21.0, 0.4) + 0.07886 * (a - 21.0);
  return 0.0;
}

}  // namespace

extern "C" {

int qpsk_pfb_taps(int channels, int taps_per_branch, double cutoff, double atten_db, double* out, int cap, int* n) {
  if (!n) return QPSK_ERR_NULL;
  if (!pfb_pow2_channels(channels) || taps_per_branch < 1 || taps_per_branch > kPfbMaxTapsPerBranch)
    return QPSK_ERR_UNSUPPORTED;
  if (!(cutoff > 0.0 && cutoff < 0.5) || !(isfinite(atten_db) && atten_db >= 0.0)) return QPSK_ERR_RANGE;
  const int L = channels * taps_per_branch;
  *n = L;
  if (!out) return QPSK_OK;
  if (cap < L) return QPSK_ERR_CAPACITY;
  const double beta = kaiser_beta(atten_db), i0b = bessel_i0(beta);
  const double alpha = 0.5 * (L - 1), fc = 2.0 * cutoff;
  double sum = 0.0;
  for (int i = 0; i < L; ++i) {
    const double m = i - alpha;
    const double arg = M_PI * fc * m;
    const double sinc = m == 0.0 ? 1.0 : sin(arg) / arg;
    const double rr = L > 1 ? m / alpha : 0.0;
    const double win = bessel_i0(beta * sqrt(fmax(0.0, 1.0 - rr * rr))) / i0b;
    out[i] = fc * sinc * win;
    sum += out[i];
  }
  for (int i = 0; i < L; ++i) out[i] /= sum;
  return QPSK_OK;
}

int qpsk_pfb_create(const float* taps, int n_taps, int channels, qpsk_pfb** out) {
  QPSK_TRY(clear_out(out));
  if (!taps) return QPSK_ERR_NULL;
  if (n_taps <= 0) return QPSK_ERR_ARG;
  for (int i = 0; i < n_taps; ++i)
    if (!isfinite(taps[i])) return QPSK_ERR_RANGE;
  if (!pfb_pow2_channels(channels)) return QPSK_ERR_UNSUPPORTED;
  if ((n_taps + channels - 1) / channels > kPfbMaxTapsPerBranch) return QPSK_ERR_UNSUPPORTED;
  return create_handle(out, taps, n_taps, channels);
}

int qpsk_pfb_destroy(qpsk_pfb* p) { return destroy_handle(p); }

int qpsk_pfb_reset(qpsk_pfb* p) { return reset_handle(p); }

int qpsk_pfb_process(qpsk_pfb* p, const float* iq_in, int64_t n_floats, float* iq_out, int64_t out_stride_floats,
                     int64_t* n_out_floats) {
  if (!p || !n_out_floats) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if (n_floats & 1) return QPSK_ERR_ARG;
  PfbEngine& g = p->eng;
  const long long n = n_floats >> 1, n_out = g.outputs_for(n);
  *n_out_floats = 2 * n_out;
  if (out_stride_floats < 2 * n_out) return QPSK_ERR_CAPACITY;
  if (n == 0) return QPSK_OK;
  if (!iq_in || (n_out > 0 && !iq_out)) return QPSK_ERR_NULL;
  return host_call(p, iq_in, 1, (size_t)n * 8, iq_out, (size_t)out_stride_floats * 4, g.M, (size_t)n_out * 8,
                   [&](const float2* x, float2* y) { return g.process_dev(x, n, y, n_out, g.stream); });
}

int qpsk_pfb_process_dev(qpsk_pfb* p, const float* d_in, int64_t n_floats, float* d_out, int64_t out_stride_floats,
                         int64_t* n_out_floats, void* stream) {
  if (!p || !n_out_floats) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (out_stride_floats & 1)) return QPSK_ERR_ARG;
  PfbEngine& g = p->eng;
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
