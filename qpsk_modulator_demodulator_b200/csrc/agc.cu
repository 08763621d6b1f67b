// agc.cu — batched feed-forward AGC (spec: include/qpskcuda.h, "feed-forward AGC"): rows of [channels][stride] cf32 in
// and out, one gain per sample from the peak envelope of a W-sample window.
//
// Per channel z = history (the last W-1 samples, zero before the stream) ++ this call's n samples; output i takes the
// window z[i .. i+W-1] and scales its oldest sample z[i]:
//   m[i] = max(0, env(z[i]), ..., env(z[i+W-1])),  g[i] = fminf(ref / m[i], max_gain),  y[i] = z[i] * g[i].
// The sliding maximum is van Herk / Gil-Werman: cut z into blocks of W starting at the warp's first output i0; for output
// i = i0 + kW + r the window is the suffix of block k from r (S_k[r]) and the prefix of block k+1 up to r-1
// (P_{k+1}[r-1], nothing when r = 0), so m = fmaxf(S_k[r], P_{k+1}[r-1]) at O(1) per sample, whatever W is.  A maximum
// has no rounding and fmaxf ignores NaN in any order, so every tiling gives the same bits as the restatement.
//
// One warp owns a tile of T consecutive outputs of one row:
//   agc_small_kernel (W <= 32): groups of G = floor(32/W)*W lanes, a whole number of blocks per warp-wide round.  The
//      group's samples, S and P live in registers; segmented max-scans by shuffle (5 steps each way), and the prefix of
//      the next block comes from this group's P or the next group's (loaded one round ahead).
//   agc_block_kernel (W > 32): block by block.  A forward pass over block k+1 (rounds of 32, shuffle scan plus a carry)
//      stores P_{k+1} in shared memory (W floats per warp); a backward pass over block k forms S_k round by round from
//      the end, reads its samples and writes the outputs.  Each sample is read twice, the second time mostly from L2.
// Every load and store is 8 bytes, so one code path serves any 8-byte-aligned pointer and any even stride.
// agc_history_kernel writes the next call's history (z[n .. n+W-2]) into the other buffer of a ping-pong pair.
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "agc.cuh"

namespace qpsk {

constexpr int kAgcWarps = 4;              // warps per CTA
constexpr unsigned kFull = 0xffffffffu;

struct AgcArgs {
  const float2* hist;                     // [C][HL]
  int HL;                                 // W - 1
  const float2* x;
  long long ldx;
  float2* y;
  long long ldy;
  long long n;                            // samples (= outputs) per channel in this call
  int C, W;
  float ref, max_gain;
  long long T;                            // outputs per warp tile
  long long tiles;                        // tiles per row
  float* gain;                            // [C]
};

__device__ __forceinline__ float2 agc_z(const AgcArgs& a, int c, long long k) {
  return k < a.HL ? a.hist[(long long)c * a.HL + k] : a.x[(long long)c * a.ldx + (k - a.HL)];
}
__device__ __forceinline__ float agc_env(float2 v) { return fmaxf(fabsf(v.x), fabsf(v.y)); }

__device__ __forceinline__ void agc_out(const AgcArgs& a, int c, long long i, float2 v, float m) {
  const float g = fminf(a.ref / m, a.max_gain);                   // m = 0: ref / 0 = inf -> max_gain
  a.y[(long long)c * a.ldy + i] = make_float2(v.x * g, v.y * g);
  if (i == a.n - 1) a.gain[c] = g;
}

__global__ void __launch_bounds__(32 * kAgcWarps) agc_small_kernel(AgcArgs a) {
  const int lane = threadIdx.x & 31;
  const long long wid = (long long)blockIdx.x * kAgcWarps + (threadIdx.x >> 5);
  if (wid >= (long long)a.C * a.tiles) return;
  const int c = (int)(wid / a.tiles);
  const long long i0 = (wid % a.tiles) * a.T;
  const long long i_end = min(i0 + a.T, a.n);
  const long long zlen = a.HL + a.n;
  const int W = a.W, G = (32 / W) * W;
  const int r = lane % W;                                          // position in the lane's block
  const int src = lane + W - 1;                                    // last sample of the window, in (this group ++ next)
  auto load = [&](long long k) { return (lane < G && k < zlen) ? agc_z(a, c, k) : make_float2(0.0f, 0.0f); };
  auto fwd = [&](float v) {                                        // P: prefix max from the block start
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const float t = __shfl_up_sync(kFull, v, d);
      if (r >= d) v = fmaxf(v, t);
    }
    return v;
  };
  auto bwd = [&](float v) {                                        // S: suffix max to the block end
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const float t = __shfl_down_sync(kFull, v, d);
      if (W - 1 - r >= d) v = fmaxf(v, t);
    }
    return v;
  };
  float2 xq = load(i0 + lane);
  float eq = agc_env(xq);
  float pq = fwd(eq);
  for (long long g0 = i0; g0 < i_end; g0 += G) {
    const float2 xn = load(g0 + G + lane);
    const float en = agc_env(xn);
    const float pn = fwd(en);
    const float sq = bwd(eq);
    const float p_here = __shfl_sync(kFull, pq, src & 31);
    const float p_next = __shfl_sync(kFull, pn, (src - G) & 31);
    const float pe = r == 0 ? 0.0f : (src < G ? p_here : p_next);
    const long long i = g0 + lane;
    if (lane < G && i < i_end) agc_out(a, c, i, xq, fmaxf(sq, pe));
    xq = xn;
    eq = en;
    pq = pn;
  }
}

constexpr int kAgcBatch = 4;              // rounds whose loads are issued together

__global__ void __launch_bounds__(32 * kAgcWarps) agc_block_kernel(AgcArgs a) {
  extern __shared__ float agc_smem[];
  const int lane = threadIdx.x & 31;
  const long long wid = (long long)blockIdx.x * kAgcWarps + (threadIdx.x >> 5);
  if (wid >= (long long)a.C * a.tiles) return;
  float* P = agc_smem + (threadIdx.x >> 5) * a.W;                  // P_{k+1}[0 .. W-2]
  const int c = (int)(wid / a.tiles);
  const long long i0 = (wid % a.tiles) * a.T;
  const long long i_end = min(i0 + a.T, a.n);
  const long long zlen = a.HL + a.n;
  const int W = a.W;
  for (long long b0 = i0; b0 < i_end; b0 += W) {
    // forward over block k+1 = z[b0 + W ..]: P[r] = max env z[b0 + W .. b0 + W + r], r < W-1 (past zlen: never used)
    float carry = 0.0f;
    for (int rb = 0; rb < W - 1; rb += 32 * kAgcBatch) {
      float e[kAgcBatch];
#pragma unroll
      for (int u = 0; u < kAgcBatch; ++u) {
        const int r = rb + 32 * u + lane;
        const long long k = b0 + W + r;
        e[u] = (r < W - 1 && k < zlen) ? agc_env(agc_z(a, c, k)) : 0.0f;
      }
#pragma unroll
      for (int u = 0; u < kAgcBatch; ++u) {
        float v = e[u];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
          const float t = __shfl_up_sync(kFull, v, d);
          if (lane >= d) v = fmaxf(v, t);
        }
        v = fmaxf(v, carry);
        const int r = rb + 32 * u + lane;
        if (r < W - 1) P[r] = v;
        carry = __shfl_sync(kFull, v, 31);
      }
    }
    __syncwarp();
    // backward over block k = z[b0 .. b0 + W - 1] (inside z: b0 < n), outputs i = b0 + r
    carry = 0.0f;
    const int top = ((W - 1) >> 5) << 5;
    for (int rb = top; rb >= 0; rb -= 32 * kAgcBatch) {
      float2 v[kAgcBatch];
#pragma unroll
      for (int u = 0; u < kAgcBatch; ++u) {
        const int r = rb - 32 * u + lane;
        v[u] = (rb - 32 * u >= 0 && r < W) ? agc_z(a, c, b0 + r) : make_float2(0.0f, 0.0f);
      }
#pragma unroll
      for (int u = 0; u < kAgcBatch; ++u) {
        if (rb - 32 * u < 0) break;                                // warp-uniform
        const int r = rb - 32 * u + lane;
        float s = agc_env(v[u]);
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) s = fmaxf(s, __shfl_down_sync(kFull, s, d));   // past lane 31: own value
        s = fmaxf(s, carry);
        carry = __shfl_sync(kFull, s, 0);
        const long long i = b0 + r;
        if (r < W && i < i_end) agc_out(a, c, i, v[u], fmaxf(s, r == 0 ? 0.0f : P[r - 1]));
      }
    }
    __syncwarp();
  }
}

// hist_out[c][j] = z_c[n + j], j < HL: the last W-1 samples of the stream so far
__global__ void agc_history_kernel(AgcArgs a, float2* __restrict__ hist_out) {
  const long long tot = (long long)a.C * a.HL;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(e / a.HL);
    hist_out[e] = agc_z(a, c, a.n + e % a.HL);
  }
}

int agc_check_params(int window, float ref, float max_gain) {
  if (window < 1 || window > kAgcMaxWindow) return QPSK_ERR_UNSUPPORTED;
  if (!isfinite(ref) || !(ref > 0.0f) || !isfinite(max_gain) || !(max_gain > 0.0f)) return QPSK_ERR_RANGE;
  return QPSK_OK;
}

int AgcEngine::init(int window, float ref_in, float max_gain_in, int channels_in) {
  W = window;
  ref = ref_in;
  max_gain = max_gain_in;
  channels = channels_in;
  QPSK_TRY(open());
  for (auto& hb : d_hist) QPSK_TRY(hb.alloc((size_t)channels * (W - 1)));
  QPSK_TRY(d_gain.alloc((size_t)channels));
  QPSK_TRY(reset(stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  return QPSK_OK;
}

__global__ void agc_fill_kernel(float* p, int n, float v) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

int AgcEngine::reset(cudaStream_t s) {
  cur = 0;
  QPSK_TRY(d_hist[0].zero(s));
  agc_fill_kernel<<<(channels + 255) / 256, 256, 0, s>>>(d_gain.p, channels, max_gain);
  QPSK_LAUNCH_CHECK();
  return QPSK_OK;
}

int AgcEngine::process_dev(const float2* x, int64_t n, int64_t ldx, float2* y, int64_t ldy, cudaStream_t s) {
  if (n == 0) return QPSK_OK;
  if (!s) s = stream;
  AgcArgs a;
  a.hist = d_hist[cur].p;
  a.HL = W - 1;
  a.x = x;
  a.ldx = ldx;
  a.y = y;
  a.ldy = ldy;
  a.n = n;
  a.C = channels;
  a.W = W;
  a.ref = ref;
  a.max_gain = max_gain;
  a.gain = d_gain.p;
  if (W <= 32) {
    const int G = (32 / W) * W;
    a.T = (long long)G * 64;
  } else {
    a.T = (long long)W * std::max(8, (16384 + W - 1) / W);      // the tile re-reads W-1 samples past its end
  }
  a.tiles = (n + a.T - 1) / a.T;
  const long long warps = (long long)channels * a.tiles;
  const long long blocks = (warps + kAgcWarps - 1) / kAgcWarps;
  if (blocks > 0x7fffffffLL) return QPSK_ERR_UNSUPPORTED;
  if (W <= 32) {
    agc_small_kernel<<<(unsigned)blocks, 32 * kAgcWarps, 0, s>>>(a);
  } else {
    QPSK_TRY(allow_max_dynamic_smem((const void*)agc_block_kernel));
    agc_block_kernel<<<(unsigned)blocks, 32 * kAgcWarps, (size_t)kAgcWarps * W * sizeof(float), s>>>(a);
  }
  QPSK_LAUNCH_CHECK();
  if (W > 1) {
    const long long tot = (long long)channels * (W - 1);
    const long long hb = std::min<long long>((tot + 255) / 256, 4096);
    agc_history_kernel<<<(unsigned)hb, 256, 0, s>>>(a, d_hist[cur ^ 1].p);
    QPSK_LAUNCH_CHECK();
    cur ^= 1;
  }
  return QPSK_OK;
}

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_agc {
  AgcEngine eng;
  DevBuf<float2> d_in, d_out;
};

extern "C" {

int qpsk_agc_create_batch(int window, float ref, float max_gain, int channels, qpsk_agc** out) {
  QPSK_TRY(clear_out(out));
  if (channels < 1) return QPSK_ERR_RANGE;
  QPSK_TRY(agc_check_params(window, ref, max_gain));
  return create_handle(out, window, ref, max_gain, channels);
}

int qpsk_agc_destroy(qpsk_agc* p) { return destroy_handle(p); }

int qpsk_agc_reset(qpsk_agc* p) { return reset_handle(p); }

int qpsk_agc_process(qpsk_agc* p, const float* iq_in, float* iq_out, int64_t n_floats, int64_t out_cap_floats) {
  if (!p) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if (n_floats & 1) return QPSK_ERR_ARG;
  if (out_cap_floats < n_floats) return QPSK_ERR_CAPACITY;
  if (n_floats == 0) return QPSK_OK;
  if (!iq_in || !iq_out) return QPSK_ERR_NULL;
  AgcEngine& g = p->eng;
  const int64_t n = n_floats >> 1;
  const size_t row = (size_t)n * 8;
  return host_call(p, iq_in, g.channels, row, iq_out, row, g.channels, row,
                   [&](const float2* x, float2* y) { return g.process_dev(x, n, n, y, n, g.stream); });
}

int qpsk_agc_process_dev(qpsk_agc* p, const float* d_in, float* d_out, int64_t n_floats, int64_t in_stride_floats,
                         int64_t out_stride_floats, void* stream) {
  if (!p) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) || (in_stride_floats & 1) || (out_stride_floats & 1)) return QPSK_ERR_ARG;
  if (in_stride_floats < n_floats) return QPSK_ERR_ARG;
  if (out_stride_floats < n_floats) return QPSK_ERR_CAPACITY;
  if (n_floats == 0) return QPSK_OK;
  if (!d_in || !d_out) return QPSK_ERR_NULL;
  if (misaligned(d_in) || misaligned(d_out)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(p->eng.device));
  return p->eng.process_dev((const float2*)d_in, n_floats >> 1, in_stride_floats >> 1, (float2*)d_out,
                            out_stride_floats >> 1, (cudaStream_t)stream);
}

int qpsk_agc_gain(qpsk_agc* p, float* gain, int64_t cap) {
  if (!p || !gain) return QPSK_ERR_NULL;
  AgcEngine& g = p->eng;
  if (cap < g.channels) return QPSK_ERR_CAPACITY;
  QPSK_TRY(ensure_device(g.device));
  QPSK_CUDA_TRY(cudaStreamSynchronize(g.stream));
  QPSK_CUDA_TRY(cudaMemcpy(gain, g.d_gain.p, (size_t)g.channels * sizeof(float), cudaMemcpyDeviceToHost));
  return QPSK_OK;
}

int qpsk_agc_gain_dev(qpsk_agc* p, float* d_gain, void* stream) {
  if (!p || !d_gain) return QPSK_ERR_NULL;
  AgcEngine& g = p->eng;
  QPSK_TRY(ensure_device(g.device));
  cudaStream_t s = stream ? (cudaStream_t)stream : g.stream;
  QPSK_CUDA_TRY(cudaMemcpyAsync(d_gain, g.d_gain.p, (size_t)g.channels * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return QPSK_OK;
}

}  // extern "C"
