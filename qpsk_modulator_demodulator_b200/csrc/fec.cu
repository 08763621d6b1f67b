// fec.cu — rate-1/2 K = 7 convolutional code (generators 171, 133 octal) and a batched soft-decision Viterbi decoder
// (spec: include/qpskcuda.h, "convolutional code"; DESIGN.md §3 K13).  Both stream across calls, one state per channel.
//
// Trellis.  State S = the last six input bits, the newest at bit 5.  Input u from S forms the register s = (u << 6) | S,
// emits (parity(s & 0171), parity(s & 0133)) and moves to S' = s >> 1.  The predecessors of S' are 2j and 2j+1, j = S' & 31,
// and S' is j (u = 0) or j + 32 (u = 1): the butterfly (2j, 2j+1) -> (j, j+32).  Both generators have bits 0 and 6 set, so
// with m the branch metric of register 2j, the four branches of a butterfly cost m, -m, -m, m:
//   M'[j] = min(M[2j] + m, M[2j+1] - m),  M'[j+32] = min(M[2j] - m, M[2j+1] + m)   (ties: the lower predecessor, 2j)
//
// viterbi_kernel<DIFF>: one warp per channel, 8 channels per CTA; lane j owns the metrics of states j ("lo") and j+32
// ("hi") and computes butterfly j.  Per trellis step: one shuffle broadcasts the step's soft pair, two shuffles fetch
// M[2j] and M[2j+1] (lane parity picks which of its two metrics a lane offers, so each shuffle serves both halves of the
// warp), four adds and two compare-selects update the metrics, and two ballots give the step's 64 decisions, which lane 0
// stores in a ring of 128 steps in shared memory (persisted across calls in global memory).  Soft values of up to 32
// steps are computed at once, one symbol per lane, from coalesced loads of the symbol row; a batch of steps never crosses
// a multiple of B = 32 steps, so decisions are due only at a batch's end.  At step counts (k+3)*32 the best state is
// found by a warp reduction, every metric is renormalised by its value, and a traceback from it walks 64 steps back and
// reads the 32 bits of block k off the next 32; every lane runs the traceback on the same data, lane (t mod 32) keeps the
// bit of step t, and the block goes out as one 32-byte store.
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "handle.cuh"
#include "soft.cuh"

namespace qpsk {

constexpr int kFecMaxChannels = 16384;
constexpr int kVitB = 32;                    // bits per decision block
constexpr int kVitD = 64;                    // traceback depth past a block
constexpr int kVitRing = 128;                // decision ring (steps), > B + D
constexpr int kVitWarps = 8;                 // channels per CTA
constexpr int kVitStates = 64;
constexpr unsigned kFull = 0xffffffffu;

struct VitState {
  long long nstep;     // trellis steps processed since creation, reset or flush
  float2 prev;         // differential mode: the last symbol seen
  int have_prev;       // differential mode: prev is valid
  int pad;
};

struct VitArgs {
  const float2* sym;
  long long lds;          // complex symbols between rows
  const int* n_sym;
  int max_sym;            // row capacity, lds; a count past it is read as lds
  uint8_t* bits;
  long long ldb;
  long long* n_bits;
  int* metric;            // [C][64]
  uint2* ring;            // [C][128] decisions of step t at t % 128: .x states 0..31, .y states 32..63
  VitState* st;
  int C;
  float scale;
  int flush;
};

__device__ __forceinline__ int vit_pack(int s0, int s1) { return (s0 & 0xffff) | (s1 << 16); }

// Tracebacks index the ring with the low 32 bits of the step counter (it holds 128 steps; every span is < 128).
// From state S after step t, walk back through `count` steps (t, t-1, ...): the state after step t - count.
__device__ __forceinline__ int vit_walk(const uint2* ring, int S, unsigned t, int count) {
#pragma unroll 8
  for (int k = 0; k < count; ++k) {
    const uint2 d = ring[(t - (unsigned)k) & (kVitRing - 1)];
    const unsigned w = S >= 32 ? d.y : d.x;
    S = ((S & 31) << 1) | (int)((w >> (S & 31)) & 1u);
  }
  return S;
}

// From state S after step e1 - 1, the bits of steps [e0, e1) to out[0 .. e1 - e0): lane (t - e0) mod 32 keeps the bit of
// step t, and each group of 32 goes out in one store per lane
__device__ __forceinline__ void vit_emit(const uint2* ring, int S, unsigned e0, unsigned e1, uint8_t* out, int lane) {
  const unsigned n = e1 - e0;
  int mine = 0;
#pragma unroll 4
  for (unsigned k = n; k-- > 0;) {
    if (lane == (int)(k & 31)) mine = S >> 5;
    const uint2 d = ring[(e0 + k) & (kVitRing - 1)];
    const unsigned w = S >= 32 ? d.y : d.x;
    S = ((S & 31) << 1) | (int)((w >> (S & 31)) & 1u);
    if ((k & 31) == 0 && k + lane < n) out[k + lane] = (uint8_t)mine;
  }
}

// minimum metric, lowest state on ties; the result is the same in every lane
__device__ __forceinline__ void vit_best(int lo, int hi, int lane, int* bv, int* bs) {
  int v = lo, s = lane;
  if (hi < lo) {
    v = hi;
    s = lane + 32;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const int ov = __shfl_xor_sync(kFull, v, off), os = __shfl_xor_sync(kFull, s, off);
    if (ov < v || (ov == v && os < s)) {
      v = ov;
      s = os;
    }
  }
  *bv = v;
  *bs = s;
}

// steps emitted after N steps: block k goes out once step (k+1)B + D - 1 has been processed
__device__ __forceinline__ long long vit_emitted(long long N) { return N >= kVitD ? ((N - kVitD) / kVitB) * kVitB : 0; }

template <bool DIFF>
__global__ void __launch_bounds__(32 * kVitWarps) viterbi_kernel(const VitArgs a) {
  __shared__ uint2 sring[kVitWarps][kVitRing];
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int c = blockIdx.x * kVitWarps + wi;
  if (c >= a.C) return;                                                // warp-uniform
  uint2* ring = sring[wi];
  uint2* gring = a.ring + (long long)c * kVitRing;
  for (int e = lane; e < kVitRing; e += 32) ring[e] = gring[e];
  int* gm = a.metric + (long long)c * kVitStates;
  int lo = gm[lane], hi = gm[lane + 32];
  VitState st = a.st[c];
  long long nstep = st.nstep;
  float2 prev = st.prev;
  int have = st.have_prev;
  const int n = min(max(a.n_sym[c], 0), a.max_sym);
  const float2* x = a.sym + (long long)c * a.lds;
  uint8_t* out = a.bits + (long long)c * a.ldb;
  long long nout = 0;

  const int r = 2 * lane;                                               // register of predecessor 2j with u = 0
  const int a0 = (__popc(r & 0171) & 1) ? -1 : 1, a1 = (__popc(r & 0133) & 1) ? -1 : 1;
  const bool even = (lane & 1) == 0, low = lane < 16;
  const int srcA = (r & 31) | (low ? 0 : 1), srcB = (r & 31) | (low ? 1 : 0);
  __syncwarp();

  int i = 0;
  if (DIFF && !have && n > 0) {                                        // the first symbol ever seen yields no step
    prev = x[0];
    have = 1;
    i = 1;
  }
  while (i < n) {
    const int chunk = min(n - i, kVitB - (int)(nstep & (kVitB - 1)));
    int2 s;
    float2 y = make_float2(0.0f, 0.0f);
    if (lane < chunk) y = x[i + lane];
    if (DIFF) {
      float pr = __shfl_up_sync(kFull, y.x, 1), pi = __shfl_up_sync(kFull, y.y, 1);
      if (lane == 0) {
        pr = prev.x;
        pi = prev.y;
      }
      s = soft_differential(y, make_float2(pr, pi), a.scale);
      prev.x = __shfl_sync(kFull, y.x, chunk - 1);
      prev.y = __shfl_sync(kFull, y.y, chunk - 1);
    } else {
      s = soft_coherent(y, a.scale);
    }
    const int packed = vit_pack(s.x, s.y);
    for (int t = 0; t < chunk; ++t) {
      const int w = __shfl_sync(kFull, packed, t);
      const int s0 = (int)(short)(w & 0xffff), s1 = w >> 16;
      const int m = s0 * a0 + s1 * a1;
      const int A = even ? lo : hi, Bv = even ? hi : lo;
      const int v1 = __shfl_sync(kFull, A, srcA), v2 = __shfl_sync(kFull, Bv, srcB);
      const int Ma = low ? v1 : v2, Mb = low ? v2 : v1;                  // M[2j], M[2j+1]
      const int x0 = Ma + m, x1 = Mb - m, y0 = Ma - m, y1 = Mb + m;
      const bool dl = x1 < x0, dh = y1 < y0;
      lo = dl ? x1 : x0;
      hi = dh ? y1 : y0;
      const unsigned bl = __ballot_sync(kFull, dl), bh = __ballot_sync(kFull, dh);
      if (lane == 0) ring[(nstep + t) & (kVitRing - 1)] = make_uint2(bl, bh);
    }
    nstep += chunk;
    i += chunk;
    if ((nstep & (kVitB - 1)) == 0) {
      int bv, bs;
      vit_best(lo, hi, lane, &bv, &bs);
      lo -= bv;
      hi -= bv;
      if (nstep >= kVitB + kVitD) {
        __syncwarp();
        const unsigned n32 = (unsigned)nstep;
        const int S = vit_walk(ring, bs, n32 - 1, kVitD);
        vit_emit(ring, S, n32 - kVitD - kVitB, n32 - kVitD, out + nout, lane);
        nout += kVitB;
      }
    }
  }
  if (a.flush) {
    int bv, bs;
    vit_best(lo, hi, lane, &bv, &bs);
    __syncwarp();
    const long long e0 = vit_emitted(nstep);
    vit_emit(ring, bs, (unsigned)e0, (unsigned)nstep, out + nout, lane);
    nout += nstep - e0;
    lo = hi = 0;
    nstep = 0;
    have = 0;
    prev = make_float2(0.0f, 0.0f);
  }
  __syncwarp();
  for (int e = lane; e < kVitRing; e += 32) gring[e] = ring[e];
  gm[lane] = lo;
  gm[lane + 32] = hi;
  if (lane == 0) {
    st.nstep = nstep;
    st.prev = prev;
    st.have_prev = have;
    a.st[c] = st;
    a.n_bits[c] = nout;
  }
}

// one thread per channel: the code is cheap next to everything around it
__global__ void conv_encode_kernel(const uint8_t* __restrict__ in, long long n, long long ldi, uint8_t* __restrict__ out,
                                   long long ldo, int* reg, int C) {
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  int S = reg[c];
  const uint8_t* xi = in + (long long)c * ldi;
  uint8_t* yo = out + (long long)c * ldo;
  for (long long k = 0; k < n; ++k) {
    const int s = ((xi[k] != 0) << 6) | S;
    yo[2 * k] = (uint8_t)(__popc(s & 0171) & 1);
    yo[2 * k + 1] = (uint8_t)(__popc(s & 0133) & 1);
    S = s >> 1;
  }
  reg[c] = S;
}

struct ConvEngine : EngineBase {
  int C = 0;
  DevBuf<int> d_reg;
  int reset(cudaStream_t s) { return d_reg.zero(s); }
  int init(int channels) {
    C = channels;
    QPSK_TRY(open());
    QPSK_TRY(d_reg.alloc((size_t)C));
    QPSK_TRY(reset(stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    return QPSK_OK;
  }
  int encode_dev(const uint8_t* x, long long n, long long ldx, uint8_t* y, long long ldy, cudaStream_t s) {
    if (n == 0) return QPSK_OK;
    if (!s) s = stream;
    conv_encode_kernel<<<(C + 127) / 128, 128, 0, s>>>(x, n, ldx, y, ldy, d_reg.p, C);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }
};

struct VitEngine : EngineBase {
  int C = 0;
  bool diff = false;
  float scale = 1.0f;
  DevBuf<int> d_metric;
  DevBuf<uint2> d_ring;
  DevBuf<VitState> d_st;
  int reset(cudaStream_t s) {
    QPSK_TRY(d_metric.zero(s));
    QPSK_TRY(d_ring.zero(s));
    QPSK_TRY(d_st.zero(s));
    return QPSK_OK;
  }
  int init(int channels, int differential, float sc) {
    C = channels;
    diff = differential != 0;
    scale = sc;
    QPSK_TRY(open());
    QPSK_TRY(d_metric.alloc((size_t)C * kVitStates));
    QPSK_TRY(d_ring.alloc((size_t)C * kVitRing));
    QPSK_TRY(d_st.alloc((size_t)C));
    QPSK_TRY(reset(stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
    return QPSK_OK;
  }
  int run(const float2* sym, long long lds, const int* n_sym, uint8_t* bits, long long ldb, long long* n_bits, bool flush,
          cudaStream_t s) {
    if (!s) s = stream;
    VitArgs a;
    a.sym = sym;
    a.lds = lds;
    a.n_sym = n_sym;
    a.max_sym = (int)std::min<long long>(lds, INT_MAX);
    a.bits = bits;
    a.ldb = ldb;
    a.n_bits = n_bits;
    a.metric = d_metric.p;
    a.ring = d_ring.p;
    a.st = d_st.p;
    a.C = C;
    a.scale = scale;
    a.flush = flush ? 1 : 0;
    const int grid = (C + kVitWarps - 1) / kVitWarps;
    if (diff)
      viterbi_kernel<true><<<grid, 32 * kVitWarps, 0, s>>>(a);
    else
      viterbi_kernel<false><<<grid, 32 * kVitWarps, 0, s>>>(a);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }
};

// the most bits one call over at most max_sym symbols per channel emits: a decode call emits whole blocks, at most
// 32 * ceil(max_sym / 32) <= max_sym + 31 bits; a flush call also emits the up to B + D - 1 = 95 steps not yet emitted
static long long vit_bits_bound(long long max_sym) { return (max_sym + kVitB + kVitD) & ~1LL; }

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_conv {
  ConvEngine eng;
  DevBuf<uint8_t> d_in, d_out;
};

struct qpsk_viterbi {
  VitEngine eng;
  DevBuf<float2> d_sym;
  DevBuf<int> d_nsym;
  DevBuf<uint8_t> d_bits;
  DevBuf<long long> d_nbits;
};

extern "C" {

int qpsk_conv_create(int channels, qpsk_conv** out) {
  QPSK_TRY(clear_out(out));
  if (channels < 1 || channels > kFecMaxChannels) return QPSK_ERR_UNSUPPORTED;
  return create_handle(out, channels);
}

int qpsk_conv_destroy(qpsk_conv* p) { return destroy_handle(p); }

int qpsk_conv_reset(qpsk_conv* p) { return reset_handle(p); }

int qpsk_conv_encode(qpsk_conv* p, const uint8_t* bits, int64_t n_bits, uint8_t* out) {
  if (!p) return QPSK_ERR_NULL;
  if (n_bits < 0) return QPSK_ERR_RANGE;
  if (n_bits == 0) return QPSK_OK;
  if (!bits || !out) return QPSK_ERR_NULL;
  ConvEngine& g = p->eng;
  const size_t n = (size_t)n_bits;
  return host_call(p, bits, g.C, n, out, 2 * n, g.C, 2 * n,
                   [&](const uint8_t* x, uint8_t* y) { return g.encode_dev(x, n_bits, n_bits, y, 2 * n_bits, g.stream); });
}

int qpsk_conv_encode_dev(qpsk_conv* p, const uint8_t* d_bits, int64_t n_bits, int64_t bits_stride, uint8_t* d_out,
                         int64_t out_stride, void* stream) {
  if (!p) return QPSK_ERR_NULL;
  if (n_bits < 0) return QPSK_ERR_RANGE;
  if (bits_stride < n_bits) return QPSK_ERR_ARG;
  if (out_stride < 2 * n_bits) return QPSK_ERR_CAPACITY;
  if (n_bits == 0) return QPSK_OK;
  if (!d_bits || !d_out) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(p->eng.device));
  return p->eng.encode_dev(d_bits, n_bits, bits_stride, d_out, out_stride, (cudaStream_t)stream);
}

int qpsk_viterbi_create(int channels, int differential, float scale, qpsk_viterbi** out) {
  QPSK_TRY(clear_out(out));
  if (channels < 1 || channels > kFecMaxChannels) return QPSK_ERR_UNSUPPORTED;
  if (!(scale > 0.0f) || !isfinite(scale)) return QPSK_ERR_RANGE;
  return create_handle(out, channels, differential, scale);
}

int qpsk_viterbi_destroy(qpsk_viterbi* p) { return destroy_handle(p); }

int qpsk_viterbi_reset(qpsk_viterbi* p) { return reset_handle(p); }

int qpsk_viterbi_bits_bound(const qpsk_viterbi* p, int64_t max_sym, int64_t* cap) {
  if (!p || !cap) return QPSK_ERR_NULL;
  if (max_sym < 0 || max_sym > ((int64_t)1 << 40)) return QPSK_ERR_RANGE;
  *cap = vit_bits_bound(max_sym);
  return QPSK_OK;
}

static int viterbi_dev(qpsk_viterbi* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym, uint8_t* d_bits,
                       int64_t bits_cap, int64_t* d_n_bits, void* stream, bool flush) {
  if (!p) return QPSK_ERR_NULL;
  if (!d_sym || !d_n_sym || !d_bits || !d_n_bits) return QPSK_ERR_NULL;
  if (sym_stride_floats < 0 || bits_cap < 0) return QPSK_ERR_RANGE;
  if ((sym_stride_floats & 1) || (bits_cap & 1)) return QPSK_ERR_ARG;
  if (misaligned(d_sym) || misaligned(d_n_sym) || misaligned(d_bits) || misaligned(d_n_bits)) return QPSK_ERR_ARG;
  if (sym_stride_floats / 2 > INT_MAX) return QPSK_ERR_UNSUPPORTED;
  if (bits_cap < vit_bits_bound(sym_stride_floats / 2)) return QPSK_ERR_CAPACITY;
  QPSK_TRY(ensure_device(p->eng.device));
  return p->eng.run((const float2*)d_sym, sym_stride_floats / 2, d_n_sym, d_bits, bits_cap, (long long*)d_n_bits, flush,
                    (cudaStream_t)stream);
}

int qpsk_viterbi_decode_dev(qpsk_viterbi* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym,
                            uint8_t* d_bits, int64_t bits_cap, int64_t* d_n_bits, void* stream) {
  return viterbi_dev(p, d_sym, sym_stride_floats, d_n_sym, d_bits, bits_cap, d_n_bits, stream, false);
}

int qpsk_viterbi_flush_dev(qpsk_viterbi* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym,
                           uint8_t* d_bits, int64_t bits_cap, int64_t* d_n_bits, void* stream) {
  return viterbi_dev(p, d_sym, sym_stride_floats, d_n_sym, d_bits, bits_cap, d_n_bits, stream, true);
}

static int viterbi_host(qpsk_viterbi* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym, uint8_t* bits,
                        int64_t bits_cap, int64_t* n_bits, bool flush) {
  if (!p || !n_sym || !n_bits) return QPSK_ERR_NULL;
  if (sym_stride_floats < 0 || bits_cap < 0) return QPSK_ERR_RANGE;
  if (sym_stride_floats & 1) return QPSK_ERR_ARG;
  VitEngine& g = p->eng;
  const size_t C = (size_t)g.C;
  int64_t max_sym;
  QPSK_TRY(host_sym_counts(n_sym, C, sym_stride_floats, &max_sym));
  if (bits_cap < vit_bits_bound(max_sym)) {
    for (size_t c = 0; c < C; ++c) n_bits[c] = vit_bits_bound(max_sym);
    return QPSK_ERR_CAPACITY;
  }
  if (max_sym > 0 && !sym) return QPSK_ERR_NULL;
  if (!bits) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(g.device));
  cudaStream_t s = g.stream;
  const long long lds = std::max<long long>(max_sym, 1), ldb = vit_bits_bound(max_sym);
  QPSK_TRY(p->d_bits.ensure(C * (size_t)ldb));
  QPSK_TRY(p->d_nbits.ensure(C));
  QPSK_TRY(upload_syms(p->d_sym, p->d_nsym, sym, sym_stride_floats, n_sym, C, max_sym, s));
  QPSK_TRY(g.run(p->d_sym.p, lds, p->d_nsym.p, p->d_bits.p, ldb, p->d_nbits.p, flush, s));
  QPSK_CUDA_TRY(cudaMemcpyAsync(n_bits, p->d_nbits.p, C * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
  QPSK_CUDA_TRY(cudaStreamSynchronize(s));
  int64_t w = 0;
  for (size_t c = 0; c < C; ++c) w = std::max(w, n_bits[c]);
  if (w > 0)
    QPSK_CUDA_TRY(cudaMemcpy2D(bits, (size_t)bits_cap, p->d_bits.p, (size_t)ldb, (size_t)w, C, cudaMemcpyDeviceToHost));
  return QPSK_OK;
}

int qpsk_viterbi_decode(qpsk_viterbi* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym, uint8_t* bits,
                        int64_t bits_cap, int64_t* n_bits) {
  return viterbi_host(p, sym, sym_stride_floats, n_sym, bits, bits_cap, n_bits, false);
}

int qpsk_viterbi_flush(qpsk_viterbi* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym, uint8_t* bits,
                       int64_t bits_cap, int64_t* n_bits) {
  return viterbi_host(p, sym, sym_stride_floats, n_sym, bits, bits_cap, n_bits, true);
}

}  // extern "C"
