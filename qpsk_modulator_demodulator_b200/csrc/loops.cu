// loops.cu — K4/K5 building blocks: the generic FLL kernel, the Mueller-Muller and Costas kernels (one
// thread per independent stream) and the qpsk_fll_* / qpsk_mm_* / qpsk_costas_* entry points.
// Compiled with --fmad=false (see loops.cuh).
#include "loops.cuh"

namespace qpsk {

constexpr int kLoopThreads = 32;  // one warp per CTA: spreads few streams over many SMs

// ---------------------------------------------------------------------------------------------
// FLL kernels
// ---------------------------------------------------------------------------------------------
// fll_group_kernel: 8 lanes per stream — GPU lane g of a group IS lane g of the reference's
// Vector<float> dot product (FIRFilter.cs:165-180): it accumulates window elements i = g, g+8, ... of all
// four sums (lower I/Q, upper I/Q) in the reference's order, the eight partials are then added lane 0..7
// and the scalar tail follows (:176-192), every lane redundantly, so the loop state stays uniform in the
// group.  Four streams per warp, the recurrence itself strictly sequential per stream.
constexpr int kFllGroup = 8;
constexpr int kFllCtaThreads = 128;                       // 16 streams per CTA
constexpr int kFllCtaStreams = kFllCtaThreads / kFllGroup;
constexpr int kFllBlock = 32;                             // samples staged per round and stream
constexpr size_t kFllGroupMaxSmem = 200 * 1024;           // dynamic shared memory the generic kernel may ask for

// Dynamic shared memory of fll_group_kernel for an N-tap filter: taps (padded to even, + alignment), lane partials, input
// and output staging, and the ring of N past outputs per stream.  Every filter size must fit it: a caller-set phase sends
// any size to this kernel.
static size_t fll_group_smem(int n_taps) {
  const size_t n = (size_t)n_taps, np = n + (n & 1);
  return (2 * np + 4) * sizeof(float) + (size_t)kFllCtaStreams * kFllGroup * sizeof(float4) +
         (size_t)2 * kFllCtaStreams * kFllBlock * sizeof(float2) + (size_t)kFllCtaStreams * n * sizeof(float2);
}

__global__ void __launch_bounds__(kFllCtaThreads)
    fll_group_kernel(const FllParams P, const float* __restrict__ taps, float2* ring_g, int* head_g, float2* pf_g, int C,
                     const float2* __restrict__ x, float2* __restrict__ y, long long L, long long ldx, long long ldy) {
  extern __shared__ __align__(16) float sm[];
  const int N = P.n_taps;
  const int Np = N + (N & 1);
  float* tapI = sm;                                         // reversed lower taps
  float* tapQ = sm + Np;
  float4* part = reinterpret_cast<float4*>(sm + 2 * Np + ((2 * Np) & 3 ? 4 - ((2 * Np) & 3) : 0));   // [streams][8]
  float2* xin = reinterpret_cast<float2*>(part + kFllCtaStreams * kFllGroup);                       // [streams][block]
  float2* yout = xin + kFllCtaStreams * kFllBlock;
  float2* ring = yout + kFllCtaStreams * kFllBlock;                                                   // [streams][N]
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    tapI[i] = taps[i];
    tapQ[i] = taps[N + i];
  }
  const int sl = threadIdx.x / kFllGroup;                   // stream slot in the CTA
  const int g = threadIdx.x % kFllGroup;                    // reference SIMD lane
  const int c_raw = blockIdx.x * kFllCtaStreams + sl;
  const bool live = c_raw < C;
  const int c = live ? c_raw : C - 1;                       // idle groups shadow the last stream, no stores
  float4* mypart = part + sl * kFllGroup;
  float2* myx = xin + sl * kFllBlock;
  float2* myy = yout + sl * kFllBlock;
  float2* myring = ring + (size_t)sl * N;
  for (int i = g; i < N; i += kFllGroup) myring[i] = ring_g[(long long)i * C + c];
  int head = head_g[c];
  const float2 pf = pf_g[c];
  float phase = pf.x, freq = pf.y;
  const float2* xc = x + (long long)c * ldx;
  float2* yc = y + (long long)c * ldy;
  const int nVec = N - (N & 7);
  __syncthreads();
  for (long long n0 = 0; n0 < L; n0 += kFllBlock) {
    const int nb = (int)((L - n0) < kFllBlock ? (L - n0) : kFllBlock);
    for (int i = g; i < nb; i += kFllGroup) myx[i] = xc[n0 + i];
    __syncwarp();
    for (int n = 0; n < nb; ++n) {
      float s, co;
      sincos_f32_exact(phase, &s, &co);                    // MathF.Cos/Sin(phase) :108-109
      const float2 in = myx[n];
      const float oI = in.x * co - in.y * s;               // :111
      const float oQ = in.x * s + in.y * co;               // :112
      if (g == 0) {
        myring[head] = make_float2(oI, oQ);                // newest sample replaces the oldest
        myy[n] = make_float2(oI, oQ);
      }
      head = (head + 1 == N) ? 0 : head + 1;               // = window start (oldest element)
      __syncwarp();
      float loI = 0.f, loQ = 0.f, upI = 0.f, upQ = 0.f;
      int idx = head + g;
      if (idx >= N) idx -= N;
      for (int i = g; i < nVec; i += kFllGroup) {
        const float2 v = myring[idx];
        idx += kFllGroup;
        if (idx >= N) idx -= N;
        const float a = tapI[i], b = tapQ[i];
        const float p1 = a * v.x, p2 = b * v.y, p3 = a * v.y, p4 = b * v.x;
        loI = loI + (p1 - p2);
        loQ = loQ + (p3 + p4);
        upI = upI + (p1 + p2);
        upQ = upQ + (p3 - p4);
      }
      mypart[g] = make_float4(loI, loQ, upI, upQ);
      __syncwarp();
      float aLoI = 0.f, aLoQ = 0.f, aUpI = 0.f, aUpQ = 0.f;
#pragma unroll
      for (int l = 0; l < kFllGroup; ++l) {                // lanes summed 0..7 (:176-180)
        const float4 q = mypart[l];
        aLoI += q.x; aLoQ += q.y; aUpI += q.z; aUpQ += q.w;
      }
      int ti = head + nVec;
      if (ti >= N) ti -= N;
      for (int i = nVec; i < N; ++i) {                      // scalar tail (:183-192)
        const float2 v = myring[ti];
        ti = (ti + 1 == N) ? 0 : ti + 1;
        const float a = tapI[i], b = tapQ[i];
        const float p1 = a * v.x, p2 = b * v.y, p3 = a * v.y, p4 = b * v.x;
        aLoI += (p1 - p2); aLoQ += (p3 + p4); aUpI += (p1 + p2); aUpQ += (p3 - p4);
      }
      const float powUpper = aUpI * aUpI + aUpQ * aUpQ;    // :118
      const float powLower = aLoI * aLoI + aLoQ * aLoQ;    // :119
      const float error = powLower - powUpper;             // :121
      freq += P.beta * error;                              // :124
      phase += freq + P.alpha * error;                     // :125
      if (phase > kTwoPiF || phase < -kTwoPiF) phase = remainderf(phase, kTwoPiF);   // :185-189
      if (freq > P.max_freq) freq = P.max_freq;            // :191-195
      else if (freq < P.min_freq) freq = P.min_freq;
    }
    __syncwarp();
    if (live)
      for (int i = g; i < nb; i += kFllGroup) yc[n0 + i] = myy[i];
    __syncwarp();
  }
  if (live) {
    for (int i = g; i < N; i += kFllGroup) ring_g[(long long)i * C + c] = myring[i];
    if (g == 0) {
      head_g[c] = head;
      pf_g[c] = make_float2(phase, freq);
    }
  }
}

int FllEngine::init(float sps, float rolloff, int size, float bw, int channels_in) {
  if (!(sps > 0.0f)) return QPSK_ERR_RANGE;                  // Band-Edge Filter.cs:42
  if (rolloff < 0 || rolloff > 1.0f) return QPSK_ERR_RANGE;  // :43
  if (size <= 0) return QPSK_ERR_RANGE;                      // :44
  if (!(bw > 0.0f)) return QPSK_ERR_RANGE;                   // :45
  if (channels_in <= 0) return QPSK_ERR_RANGE;
  if (fll_group_smem(size) > kFllGroupMaxSmem) return QPSK_ERR_UNSUPPORTED;   // the ring lives in shared memory: N <= 1430
  QPSK_TRY(open());
  channels = channels_in;
  n_taps = size;
  P.alpha = 0.0f;                        // :55
  P.beta = 4.0f * bw / sps;              // :56
  P.max_freq = kTwoPiF * (2.0f / sps);   // :58
  P.min_freq = -P.max_freq;
  P.n_taps = size;
  design_band_edge(sps, rolloff, size, lower, upper);
  std::vector<float> rev((size_t)2 * size);
  for (int i = 0; i < size; ++i) {
    rev[(size_t)i] = lower[2 * (size_t)(size - 1 - i)];
    rev[(size_t)size + i] = lower[2 * (size_t)(size - 1 - i) + 1];
  }
  QPSK_TRY(d_taps.alloc(rev.size()));
  QPSK_TRY(d_ring.alloc((size_t)size * channels));
  QPSK_TRY(d_head.alloc((size_t)channels));
  QPSK_TRY(d_pf.alloc((size_t)channels));
  QPSK_CUDA_TRY(cudaMemcpyAsync(d_taps.p, rev.data(), rev.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
  QPSK_TRY(d_ring.zero(stream));
  QPSK_TRY(d_head.zero(stream));
  QPSK_TRY(d_pf.zero(stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  return QPSK_OK;
}

int FllEngine::process_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, cudaStream_t s) {
  if (L == 0) return QPSK_OK;
  if (!x || !y) return QPSK_ERR_NULL;
  if (!s) s = stream;
  // Kernel choice by stream count (40 taps, 4196 samples, ms; tools/fll_only.py):
  //   streams   1024   2048   4096   8192   16384
  //   duo       0.76   0.90   1.25   2.46   4.49    two warps per four streams: shortest recurrence (356 cycles / sample),
  //                                                   44 warp instructions per stream and sample -> issue-bound from ~4096
  //   pair      1.45   1.45   1.45   1.47   2.35    two lanes per stream, software-pipelined (680 cycles / sample, ~21 issue
  //                                                   slots per stream and sample)
  constexpr int kPairMinStreams = 5120;
  // The two-warp kernel evaluates sin/cos and the phase wrap with short-range formulas (|phase| < 1e5): the loop
  // keeps |phase| <= 2*pi + max|freq|, so only a caller-set state or an absurd frequency limit (sps < 1e-3) can
  // leave that range — those calls take the generic kernel, which uses the library routines.
  const bool wild = state_wild || !(P.max_freq < 1e4f);
  state_wild = false;                                          // any kernel leaves the state wrapped and clamped
  // the pair kernel's sin/cos is the |phase| < 64 form: a caller-set phase beyond that goes through the two-warp kernel once
  const bool far = state_far;
  state_far = false;
  if (!wild && !far && fll_pair_supported(n_taps) && channels >= kPairMinStreams)
    return fll_pair_launch(P, lower, d_ring.p, d_head.p, d_pf.p, channels, x, y, L, ldx, ldy, s);
  if (!wild && fll_duo_supported(n_taps))
    return fll_duo_launch(P, d_taps.p, d_ring.p, d_head.p, d_pf.p, channels, x, y, L, ldx, ldy, s);
  // 8 lanes per stream; ring, staging and partial sums in shared memory
  const size_t smem = fll_group_smem(n_taps);
  if (smem > kFllGroupMaxSmem) return QPSK_ERR_UNSUPPORTED;
  const int blocks = (channels + kFllCtaStreams - 1) / kFllCtaStreams;
  QPSK_TRY(allow_max_dynamic_smem((const void*)fll_group_kernel));
  fll_group_kernel<<<blocks, kFllCtaThreads, smem, s>>>(P, d_taps.p, d_ring.p, d_head.p, d_pf.p, channels, x, y, L, ldx, ldy);
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}

// ---------------------------------------------------------------------------------------------
// Mueller-Muller kernel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kLoopThreads)
    mm_kernel(const MmParams P, MmState* st_g, const float2* q_in, float2* q_out, long long qcap, int C,
              const float2* __restrict__ x, long long L, long long ldx, float2* __restrict__ y, long long cap_floats,
              long long ldy, int* n_sym_g) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  MmState S = st_g[c];
  MmView v;
  v.queue = q_in + (long long)c * qcap;
  v.in = x + (long long)c * ldx;
  v.queued = S.queued;
  const int buf_count = S.queued + (int)L;
  float2* yc = y + (long long)c * ldy;
  int out = 0;
  while (S.base_index + 2 < buf_count) {             // MuellerMuller.cs:62
    const long long o = (long long)out << 1;
    const bool room = !(o + 1 >= cap_floats);        // :101
    float ci, cq;
    bool stop_after = false;
    if (!mm_symbol(P, S, v, buf_count, room, ci, cq, stop_after)) break;
    yc[out] = make_float2(ci, cq);
    ++out;
    if (stop_after) break;
  }
  // drop consumed samples, keep at least the last three (:123-129)
  int consumed = min(max(0, S.base_index - 1), max(0, buf_count - 3));
  float2* qo = q_out + (long long)c * qcap;
  const int remain = buf_count - consumed;
  for (int i = 0; i < remain; ++i) qo[i] = v.at(consumed + i);
  S.queued = remain;
  S.base_index -= consumed;
  st_g[c] = S;
  n_sym_g[c] = out;
}

__global__ void mm_init_kernel(MmState* st, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  MmState S;
  S.mu = 0.0; S.integral = 0.0;                      // :45-46
  S.prevSI = S.prevSQ = S.prevDI = S.prevDQ = 0.f;
  S.base_index = 1;                                  // :44
  S.has_prev = 0; S.queued = 0; S.pad = 0;
  st[c] = S;
}

int MmEngine::init(double sps, double kp, double ki, int channels_in) {
  if (channels_in <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(open());
  channels = channels_in;
  P.sps = sps; P.kp = kp; P.ki = ki;
  QPSK_TRY(d_state.alloc((size_t)channels));
  mm_init_kernel<<<(channels + 127) / 128, 128, 0, stream>>>(d_state.p, channels);
  QPSK_LAUNCH_CHECK();
  qcap = 0; q_bound = 0; qcur = 0;
  QPSK_TRY(ensure_queue(8, stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  return QPSK_OK;
}

// grow both queue buffers to hold `need` complex samples per stream, keeping the current contents
int MmEngine::ensure_queue(int64_t need, cudaStream_t s) {
  if (need <= qcap) return QPSK_OK;
  int64_t ncap = qcap ? qcap : 8;
  while (ncap < need) ncap <<= 1;
  DevBuf<float2> nq0, nq1;
  QPSK_TRY(nq0.alloc((size_t)ncap * channels));
  QPSK_TRY(nq1.alloc((size_t)ncap * channels));
  if (qcap > 0) {
    QPSK_CUDA_TRY(cudaMemcpy2DAsync(nq0.p, (size_t)ncap * 8, d_queue[qcur].p, (size_t)qcap * 8, (size_t)qcap * 8,
                                    (size_t)channels, cudaMemcpyDeviceToDevice, s));
    QPSK_CUDA_TRY(cudaStreamSynchronize(s));
  }
  std::swap(d_queue[0].p, nq0.p); std::swap(d_queue[0].n, nq0.n);
  std::swap(d_queue[1].p, nq1.p); std::swap(d_queue[1].n, nq1.n);
  qcur = 0;
  qcap = ncap;
  return QPSK_OK;
}

int MmEngine::process_dev(const float2* x, int64_t L, int64_t ldx, float2* y, int64_t cap_floats, int64_t ldy,
                          int* d_nsym, cudaStream_t s) {
  if (!d_nsym) return QPSK_ERR_NULL;
  if (L > 0 && !x) return QPSK_ERR_NULL;
  if (cap_floats > 0 && !y) return QPSK_ERR_NULL;
  if (!s) s = stream;
  // queue bound: with room for every symbol the loop leaves <= 3 samples (+ tolerance); without,
  // the unconsumed tail stays queued like the reference's growing buffer (:200-241)
  const int64_t total = q_bound + L;
  // every emitted symbol advances time by >= sps - 0.1 (:87-89), so `total` samples yield at most this many
  const double min_adv = P.sps - 0.1;
  const int64_t max_sym = (min_adv > 1.0) ? (int64_t)((double)total / min_adv) + 2 : total;
  const bool roomy = (cap_floats >> 1) >= max_sym;
  const int64_t next_bound = roomy ? 4 : total;
  QPSK_TRY(ensure_queue(next_bound > 8 ? next_bound : 8, s));
  const int threads = kLoopThreads;
  mm_kernel<<<(channels + threads - 1) / threads, threads, 0, s>>>(P, d_state.p, d_queue[qcur].p, d_queue[qcur ^ 1].p,
                                                                  qcap, channels, x, L, ldx, y, cap_floats, ldy, d_nsym);
  QPSK_LAUNCH_CHECK();
  qcur ^= 1;
  q_bound = next_bound;
  return QPSK_OK;
}

// ---------------------------------------------------------------------------------------------
// Costas kernel
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kLoopThreads)
    costas_kernel(const CostasParams P, CostasState* st_g, int C, const float2* __restrict__ x, float2* __restrict__ y,
                  long long L, long long ldx, long long ldy, const int* __restrict__ n_sym) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const SinCosK K = sincos_load_consts();
  CostasState S = st_g[c];
  const long long n = n_sym ? (long long)n_sym[c] : L;
  const float2* xc = x + (long long)c * ldx;
  float2* yc = y + (long long)c * ldy;
  for (long long k = 0; k < n; ++k) {
    const float2 in = xc[k];
    float oI, oQ;
    costas_step(P, K, S, in.x, in.y, oI, oQ);
    yc[k] = make_float2(oI, oQ);
  }
  st_g[c] = S;
}

int CostasEngine::init(double fs, double bw, double damping, int channels_in) {
  if (channels_in <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(open());
  channels = channels_in;
  costas_gains(fs, bw, damping, &P.alpha, &P.beta);
  QPSK_TRY(d_state.alloc((size_t)channels));
  QPSK_TRY(d_state.zero(stream));   // theta = freq = 0 (:46-47)
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  return QPSK_OK;
}

int CostasEngine::process_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, const int* d_nsym,
                              cudaStream_t s) {
  if (L == 0) return QPSK_OK;
  if (!x || !y) return QPSK_ERR_NULL;
  if (!s) s = stream;
  const int threads = kLoopThreads;
  costas_kernel<<<(channels + threads - 1) / threads, threads, 0, s>>>(P, d_state.p, channels, x, y, L, ldx, ldy, d_nsym);
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_fll {
  FllEngine eng;
  DevBuf<float2> d_in, d_out;
};
struct qpsk_mm {
  MmEngine eng;
  DevBuf<float2> d_in, d_out;
  DevBuf<int> d_n;
};
struct qpsk_costas {
  CostasEngine eng;
  DevBuf<float2> d_in, d_out;
};

extern "C" {

// ---- FLL ----
int qpsk_fll_create_batch(float sps, float rolloff, int filter_size, float bandwidth, int channels, qpsk_fll** out) {
  QPSK_TRY(clear_out(out));
  return create_handle(out, sps, rolloff, filter_size, bandwidth, channels);
}
int qpsk_fll_create(float sps, float rolloff, int filter_size, float bandwidth, qpsk_fll** out) {
  return qpsk_fll_create_batch(sps, rolloff, filter_size, bandwidth, 1, out);
}
int qpsk_fll_destroy(qpsk_fll* f) { return destroy_handle(f); }
int qpsk_fll_process(qpsk_fll* f, const float* in, float* out, int64_t n_floats, int64_t out_cap_floats) {
  if (!f) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;          // Band-Edge Filter.cs:66-67
  if (out_cap_floats < n_floats) return QPSK_ERR_ARG;    // :68-69
  if (n_floats == 0) return QPSK_OK;
  if (!in || !out) return QPSK_ERR_NULL;
  FllEngine& e = f->eng;
  const int64_t L = n_floats >> 1;
  const size_t row = (size_t)L * 8;
  return host_call(f, in, e.channels, row, out, row, e.channels, row,
                   [&](const float2* x, float2* y) { return e.process_dev(x, y, L, L, L, e.stream); });
}
int qpsk_fll_process_dev(qpsk_fll* f, const float* d_in, float* d_out, int64_t n_floats, int64_t is, int64_t os, void* stream) {
  if (!f) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (is & 1) || (os & 1)) return QPSK_ERR_ARG;
  if (misaligned(d_in) || misaligned(d_out)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(f->eng.device));
  return f->eng.process_dev((const float2*)d_in, (float2*)d_out, n_floats >> 1, is >> 1, os >> 1, (cudaStream_t)stream);
}
int qpsk_fll_get_state(qpsk_fll* f, float* phase, float* freq) {
  if (!f || !phase || !freq) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  FllEngine& e = f->eng;
  std::vector<float2> h((size_t)e.channels);
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaMemcpy(h.data(), e.d_pf.p, h.size() * sizeof(float2), cudaMemcpyDeviceToHost));
  for (int c = 0; c < e.channels; ++c) { phase[c] = h[(size_t)c].x; freq[c] = h[(size_t)c].y; }
  return QPSK_OK;
}
int qpsk_fll_set_state(qpsk_fll* f, const float* phase, const float* freq) {
  if (!f || !phase || !freq) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  FllEngine& e = f->eng;
  std::vector<float2> h((size_t)e.channels);
  e.state_wild = false;
  e.state_far = false;
  for (int c = 0; c < e.channels; ++c) {
    h[(size_t)c] = make_float2(phase[c], freq[c]);
    if (!(fabsf(phase[c]) < 1e4f) || !(fabsf(freq[c]) < 1e4f)) e.state_wild = true;   // see FllEngine::process_dev
    if (!(fabsf(phase[c]) < 32.0f)) e.state_far = true;
  }
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaMemcpy(e.d_pf.p, h.data(), h.size() * sizeof(float2), cudaMemcpyHostToDevice));
  return QPSK_OK;
}

// ---- Mueller-Muller ----
int qpsk_mm_create_batch(double sps, double kp, double ki, int channels, qpsk_mm** out) {
  QPSK_TRY(clear_out(out));
  return create_handle(out, sps, kp, ki, channels);
}
int qpsk_mm_create(double sps, double kp, double ki, qpsk_mm** out) { return qpsk_mm_create_batch(sps, kp, ki, 1, out); }
int qpsk_mm_destroy(qpsk_mm* m) { return destroy_handle(m); }
int qpsk_mm_process(qpsk_mm* m, const float* in, int64_t n_floats, float* out, int64_t cap_floats, int* n_sym) {
  if (!m || !n_sym) return QPSK_ERR_NULL;
  if (n_floats < 0 || cap_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;          // MuellerMuller.cs:54-55
  if (n_floats > 0 && !in) return QPSK_ERR_NULL;
  if (cap_floats > 0 && !out) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(m->eng.device));
  MmEngine& e = m->eng;
  const int64_t L = n_floats >> 1;
  const int64_t cap_sym = cap_floats >> 1;
  QPSK_TRY(m->d_out.ensure((size_t)(cap_sym > 0 ? cap_sym : 1) * e.channels));
  QPSK_TRY(m->d_n.ensure((size_t)e.channels));
  QPSK_TRY(stage_in(m->d_in, in, (size_t)L * 8, (size_t)L * 8, e.channels, e.stream));
  QPSK_TRY(e.process_dev(m->d_in.p, L, L, m->d_out.p, cap_floats, cap_sym > 0 ? cap_sym : 1, m->d_n.p, e.stream));
  QPSK_CUDA_TRY(cudaMemcpyAsync(n_sym, m->d_n.p, sizeof(int) * e.channels, cudaMemcpyDeviceToHost, e.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  if (cap_sym > 0) {
    // out is [channels][cap_floats]; copy only the produced symbols
    for (int c = 0; c < e.channels; ++c)
      if (n_sym[c] > 0)
        QPSK_CUDA_TRY(cudaMemcpyAsync(out + (size_t)c * cap_floats, m->d_out.p + (size_t)c * cap_sym, (size_t)n_sym[c] * 8,
                                      cudaMemcpyDeviceToHost, e.stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  }
  return QPSK_OK;
}
int qpsk_mm_process_dev(qpsk_mm* m, const float* d_in, int64_t n_floats, int64_t is, float* d_out, int64_t cap_floats,
                        int64_t os, int* d_n_sym, void* stream) {
  if (!m) return QPSK_ERR_NULL;
  if (n_floats < 0 || cap_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (is & 1) || (os & 1)) return QPSK_ERR_ARG;
  if (misaligned(d_in) || misaligned(d_out)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(m->eng.device));
  return m->eng.process_dev((const float2*)d_in, n_floats >> 1, is >> 1, (float2*)d_out, cap_floats, os >> 1, d_n_sym,
                            (cudaStream_t)stream);
}
int qpsk_mm_get_state(qpsk_mm* m, int* base_index, double* mu, double* integral, int* queued) {
  if (!m) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(m->eng.device));
  MmEngine& e = m->eng;
  std::vector<MmState> h((size_t)e.channels);
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaMemcpy(h.data(), e.d_state.p, h.size() * sizeof(MmState), cudaMemcpyDeviceToHost));
  for (int c = 0; c < e.channels; ++c) {
    if (base_index) base_index[c] = h[(size_t)c].base_index;
    if (mu) mu[c] = h[(size_t)c].mu;
    if (integral) integral[c] = h[(size_t)c].integral;
    if (queued) queued[c] = h[(size_t)c].queued;
  }
  return QPSK_OK;
}

// ---- Costas ----
int qpsk_costas_create_batch(double fs, double bw, double damping, int channels, qpsk_costas** out) {
  QPSK_TRY(clear_out(out));
  return create_handle(out, fs, bw, damping, channels);
}
int qpsk_costas_create(double fs, double bw, double damping, qpsk_costas** out) {
  return qpsk_costas_create_batch(fs, bw, damping, 1, out);
}
int qpsk_costas_destroy(qpsk_costas* c) { return destroy_handle(c); }
int qpsk_costas_process(qpsk_costas* c, const float* in, float* out, int64_t n_floats, int64_t out_cap_floats) {
  if (!c) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;          // CostasLoopQpsk.cs:100-101
  if (out_cap_floats < n_floats) return QPSK_ERR_ARG;    // :102-103
  if (n_floats == 0) return QPSK_OK;
  if (!in || !out) return QPSK_ERR_NULL;
  CostasEngine& e = c->eng;
  const int64_t L = n_floats >> 1;
  const size_t row = (size_t)L * 8;
  return host_call(c, in, e.channels, row, out, row, e.channels, row,
                   [&](const float2* x, float2* y) { return e.process_dev(x, y, L, L, L, nullptr, e.stream); });
}
int qpsk_costas_process_dev(qpsk_costas* c, const float* d_in, float* d_out, int64_t n_floats, int64_t is, int64_t os,
                            const int* d_n_sym, void* stream) {
  if (!c) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (is & 1) || (os & 1)) return QPSK_ERR_ARG;
  if (misaligned(d_in) || misaligned(d_out)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(c->eng.device));
  return c->eng.process_dev((const float2*)d_in, (float2*)d_out, n_floats >> 1, is >> 1, os >> 1, d_n_sym, (cudaStream_t)stream);
}
int qpsk_costas_get_state(qpsk_costas* c, double* theta, double* freq) {
  if (!c || !theta || !freq) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(c->eng.device));
  CostasEngine& e = c->eng;
  std::vector<CostasState> h((size_t)e.channels);
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  QPSK_CUDA_TRY(cudaMemcpy(h.data(), e.d_state.p, h.size() * sizeof(CostasState), cudaMemcpyDeviceToHost));
  for (int i = 0; i < e.channels; ++i) { theta[i] = h[(size_t)i].theta; freq[i] = h[(size_t)i].freq; }
  return QPSK_OK;
}

}  // extern "C"
