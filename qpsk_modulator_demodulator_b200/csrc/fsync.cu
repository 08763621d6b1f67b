// fsync.cu — soft-decision frame synchronizer for coded frames (spec: include/qpskcuda.h, "frame synchronizer";
// DESIGN.md §3 K15).  It correlates the known encoded start of a frame (the code bits of 32 zeros and START from state 0)
// against the soft values of the Costas output, picks the peak, and cuts one fixed-length window per frame.
//
// fsync_kernel<DIFF>: one warp per channel, 8 channels per CTA.  Soft pairs are computed once per symbol into a per-warp
// ring of packed int8 in shared memory (two symbols per 32-bit word, words past the ring end mirrored so a window never
// wraps), with a running sum of |s0| + |s1| beside it, so E(p) is one difference.  Lanes take 32 consecutive positions
// per pass.  With a = c_{2i} ? 1 : -1 and b = c_{2i+1} ? 1 : -1, X = sum a s0 + b s1 and Y = sum a s1 - b s0 give all four
// rotations (M_0 = X, M_1 = Y, M_2 = -X, M_3 = -Y); each is one __dp4a per two symbols against the pattern words
// (a, b, a', b') and (-b, a, -b', a') in shared memory.  A lane at an odd position reads from the even word below it
// against a copy of the pattern shifted by one symbol, so every lane reads whole words.  A ballot finds crossings; the
// peak pick over the next P positions and the frame copy (coalesced float2 stores, derotated) run warp-uniform.  No
// correlation is computed inside a frame: the search jumps to p* + F.
#include <limits.h>
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "handle.cuh"
#include "soft.cuh"

namespace qpsk {

constexpr int kFsMaxChannels = 16384;
constexpr int kFsWarps = 8;                       // channels per CTA
constexpr int kFsMaxStart = 24;                   // START bytes
constexpr int kFsMaxP = QPSK_CODED_LEAD_BITS + 8 * kFsMaxStart;   // 224 pattern symbols
constexpr int kFsPatWords = ((kFsMaxP / 2 + 1) + 3) & ~3;         // words per pattern copy, padded to a multiple of 4
constexpr int kFsRing = 512;                      // soft-pair ring (symbols), > 2P - 1 + 32
constexpr int kFsRingWords = kFsRing / 2 + kFsPatWords;           // + the mirrored words
constexpr int kFsMaxPayload = 65536;
constexpr int kFsMaxEnd = 32;
constexpr unsigned kFsFull = 0xffffffffu;

struct FsState {
  long long n;          // symbols received since create or reset
  long long next;       // next position to search; while collecting, the frame's p*
  long long fnb;        // collecting: window symbols already in the frame buffer
  int collecting;
  int rot, metric, energy;
  int hsel;             // which of the two history buffers holds the history
  int pad;
};

struct FsArgs {
  const float2* sym;
  long long lds;
  const int* n_sym;
  int max_sym;
  float2* frames;
  long long ldf;
  int* frame_n;
  long long* n_bytes;
  qpsk_fsync_frame* info;
  int slots;
  const int2* pattern;  // [2][kFsPatWords] {X word, Y word}: even-aligned, then shifted by one symbol
  FsState* st;
  float2* hist;         // [C][2][H]
  float2* fbuf;         // [C][F + 1]
  int C, P, F, H, payload, rho;
  float scale;
};

__device__ __forceinline__ float2 fs_derotate(float2 y, int r) {
  switch (r) {
    case 1: return make_float2(y.y, -y.x);
    case 2: return make_float2(-y.x, -y.y);
    case 3: return make_float2(-y.y, y.x);
    default: return y;
  }
}

template <bool DIFF>
__global__ void __launch_bounds__(32 * kFsWarps) fsync_kernel(const FsArgs a) {
  __shared__ int2 spat[2 * kFsPatWords];
  __shared__ int sring[kFsWarps][kFsRingWords];
  __shared__ unsigned ssum[kFsWarps][kFsRing];    // ssum[k % R]: running sum of |s0| + |s1| over the filled positions < k
  for (int i = threadIdx.x; i < 2 * kFsPatWords; i += blockDim.x) spat[i] = a.pattern[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  const int c = blockIdx.x * kFsWarps + wi;
  if (c >= a.C) return;                                                  // warp-uniform
  int* ring = sring[wi];
  unsigned short* ring16 = reinterpret_cast<unsigned short*>(ring);
  unsigned* sum = ssum[wi];
  const int P = a.P, F = a.F, H = a.H, delta = DIFF ? 1 : 0;
  const int PW = ((P / 2 + 1) + 3) & ~3;

  FsState st = a.st[c];
  const int n_in = min(max(a.n_sym[c], 0), a.max_sym);
  const long long n_old = st.n, n_new = n_old + n_in;
  const long long hbase = n_old - min(n_old, (long long)H);
  const float2* x = a.sym + (long long)c * a.lds;
  const float2* hold = a.hist + ((long long)c * 2 + st.hsel) * H;
  float2* hnew = a.hist + ((long long)c * 2 + (st.hsel ^ 1)) * H;
  float2* fb = a.fbuf + (long long)c * (F + 1);
  // symbol k of the stream: this call's row, or the history of the last H symbols before it (k >= hbase always)
  auto vload = [&](long long k) -> float2 { return k >= n_old ? x[k - n_old] : hold[k - hbase]; };

  int j = 0;                                                             // slots filled
  auto emit = [&](long long pstar, int rot, int metric, int energy, long long nb) {
    const long long w0 = pstar - delta;
    const int L = F + delta;
    if (j < a.slots) {
      const long long slot = (long long)c * a.slots + j;
      float2* out = a.frames + slot * a.ldf;
      for (int i = lane; i < L; i += 32) out[i] = fs_derotate(i < nb ? fb[i] : vload(w0 + i), rot);
      if (lane == 0) {
        a.frame_n[slot] = L;
        a.n_bytes[slot] = a.payload;
        qpsk_fsync_frame f;
        f.position = pstar;
        f.metric = metric;
        f.energy = energy;
        f.rotation = rot;
        f.channel = c;
        a.info[slot] = f;
      }
    }
    ++j;
  };
  // a frame whose window runs past this call: its symbols so far go to the frame buffer
  auto stash = [&](long long pstar, long long from) {
    const long long w0 = pstar - delta;
    for (long long k = from + lane; k < n_new; k += 32) fb[k - w0] = vload(k);
    st.fnb = n_new - w0;
  };

  long long p = st.next;
  if (st.collecting) {
    const long long end = p + F;
    if (end <= n_new) {
      emit(p, st.rot, st.metric, st.energy, st.fnb);
      st.collecting = 0;
      p = end;
    } else {
      stash(p, n_old);
    }
  }
  if (!st.collecting) {
    const long long lim = n_new - 2 * P + 2;                             // positions p < lim are decided in this call
    long long filled = p;                                                // soft values are in the ring for [.., filled)
    unsigned run = 0;
    if (lane == 0) sum[(int)p & (kFsRing - 1)] = 0;
    // soft values of positions [filled, T)
    auto ensure = [&](long long T) {
      while (filled < T) {
        const long long k = filled + lane;
        const bool v = k < T;
        int2 s = make_int2(0, 0);
        if (v) s = DIFF ? soft_differential(vload(k), vload(k - 1), a.scale) : soft_coherent(vload(k), a.scale);
        unsigned e = (unsigned)(abs(s.x) + abs(s.y));
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned t = __shfl_up_sync(kFsFull, e, o);
          if (lane >= o) e += t;
        }
        if (v) {
          const int idx = (int)k & (kFsRing - 1);
          const unsigned short h = (unsigned short)((s.x & 0xff) | ((s.y & 0xff) << 8));
          ring16[idx] = h;
          if (idx < 2 * kFsPatWords) ring16[idx + kFsRing] = h;
          sum[(idx + 1) & (kFsRing - 1)] = run + e;
        }
        run += __shfl_sync(kFsFull, e, 31);
        filled = min(filled + 32, T);
      }
      __syncwarp();
    };
    // M, rotation and E at position q
    auto corr = [&](long long q, int* M, int* r, int* E) {
      const int qi = (int)q;
      const int* w = ring + ((qi >> 1) & (kFsRing / 2 - 1));
      const int2* pt = spat + ((qi & 1) ? kFsPatWords : 0);
      int X = 0, Y = 0;
      for (int i = 0; i < PW; i += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int sw = w[i + u];
          const int2 pv = pt[i + u];
          X = __dp4a(sw, pv.x, X);
          if (!DIFF) Y = __dp4a(sw, pv.y, Y);
        }
      }
      int m = X, rr = 0;
      if (!DIFF) {
        if (Y > m) { m = Y; rr = 1; }
        if (-X > m) { m = -X; rr = 2; }
        if (-Y > m) { m = -Y; rr = 3; }
      }
      *M = m;
      *r = rr;
      *E = (int)(sum[(qi + P) & (kFsRing - 1)] - sum[qi & (kFsRing - 1)]);
    };
    while (p < lim) {
      ensure(min(p + 31 + P, n_new));
      int M, r, E;
      const bool v = p + lane < lim;
      bool hit = false;
      if (v) {
        corr(p + lane, &M, &r, &E);
        hit = E > 0 && 256 * M >= a.rho * E;
      }
      const unsigned b = __ballot_sync(kFsFull, hit);
      if (!b) {
        p = min(p + 32, lim);
        continue;
      }
      const long long p0 = p + __ffs(b) - 1;
      ensure(p0 + 2 * P - 1);
      int bm = INT_MIN, bo = 0, br = 0, be = 0;                          // the peak over [p0, p0 + P)
      for (int t = 0; t < P; t += 32) {
        if (t + lane < P) {
          corr(p0 + t + lane, &M, &r, &E);
          if (M > bm) { bm = M; bo = t + lane; br = r; be = E; }
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const int om = __shfl_xor_sync(kFsFull, bm, o), oo = __shfl_xor_sync(kFsFull, bo, o);
        const int orr = __shfl_xor_sync(kFsFull, br, o), oe = __shfl_xor_sync(kFsFull, be, o);
        if (om > bm || (om == bm && oo < bo)) { bm = om; bo = oo; br = orr; be = oe; }
      }
      const long long pstar = p0 + bo, end = pstar + F;
      if (end <= n_new) {
        emit(pstar, br, bm, be, 0);
      } else {
        st.collecting = 1;
        st.rot = br;
        st.metric = bm;
        st.energy = be;
        stash(pstar, pstar - delta);
        p = pstar;
        break;
      }
      p = end;
      if (p > filled) {                                                  // nothing of the ring is needed any more
        filled = p;
        if (lane == 0) sum[(int)p & (kFsRing - 1)] = run;
        __syncwarp();
      }
    }
  }
  // empty slots
  for (int s = j + lane; s < a.slots; s += 32) {
    const long long slot = (long long)c * a.slots + s;
    a.frame_n[slot] = 0;
    a.n_bytes[slot] = 0;
    qpsk_fsync_frame f;
    f.position = -1;
    f.metric = f.energy = f.rotation = 0;
    f.channel = c;
    a.info[slot] = f;
  }
  // the last H symbols, into the other history buffer
  const long long hb = n_new - min(n_new, (long long)H);
  for (long long k = hb + lane; k < n_new; k += 32) hnew[k - hb] = vload(k);
  if (lane == 0) {
    st.n = n_new;
    st.next = p;
    st.hsel ^= 1;
    a.st[c] = st;
  }
}

struct FsEngine : EngineBase {
  int C = 0, P = 0, F = 0, H = 0, payload = 0, rho = 0;
  bool diff = false;
  float scale = 1.0f;
  DevBuf<int2> d_pattern;
  DevBuf<FsState> d_st;
  DevBuf<float2> d_hist, d_fbuf;
  int delta() const { return diff ? 1 : 0; }
  int reset(cudaStream_t s) {
    std::vector<FsState> st((size_t)C);
    for (auto& v : st) {
      memset(&v, 0, sizeof(v));
      v.next = delta();
    }
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_st.p, st.data(), st.size() * sizeof(FsState), cudaMemcpyHostToDevice, s));
    QPSK_CUDA_TRY(cudaStreamSynchronize(s));
    return QPSK_OK;
  }
  int init(int channels, int differential, float sc, const uint8_t* start, int n_start, int payload_bytes, int n_end,
           int rho_in) {
    C = channels;
    diff = differential != 0;
    scale = sc;
    payload = payload_bytes;
    rho = rho_in ? rho_in : QPSK_FSYNC_RHO_DEFAULT;
    P = QPSK_CODED_LEAD_BITS + 8 * n_start;
    F = QPSK_CODED_LEAD_BITS + 8 * (n_start + payload_bytes + n_end) + QPSK_CODED_TAIL_BITS;
    H = 2 * P + 1;
    // the pattern: code bits of 32 zeros and START from state 0, as +-1 bytes
    std::vector<int> cb(2 * (size_t)P);
    int S = 0;
    for (int i = 0; i < P; ++i) {
      const int u = i < QPSK_CODED_LEAD_BITS ? 0 : (start[(i - QPSK_CODED_LEAD_BITS) / 8] >> (7 - (i - QPSK_CODED_LEAD_BITS) % 8)) & 1;
      const int s = (u << 6) | S;
      cb[2 * i] = __builtin_parity(s & 0171) ? 1 : -1;
      cb[2 * i + 1] = __builtin_parity(s & 0133) ? 1 : -1;
      S = s >> 1;
    }
    // symbol t of a word: pattern symbol t - shift (zero outside 0..P-1)
    auto sym = [&](int t, int* ab) {
      if (t < 0 || t >= P) {
        ab[0] = ab[1] = 0;
      } else {
        ab[0] = cb[2 * t];
        ab[1] = cb[2 * t + 1];
      }
    };
    std::vector<int2> pat(2 * kFsPatWords);
    for (int sh = 0; sh < 2; ++sh)
      for (int i = 0; i < kFsPatWords; ++i) {
        int A[2], B[2];
        sym(2 * i - sh, A);
        sym(2 * i + 1 - sh, B);
        auto byte = [](int v) { return (unsigned)(v & 0xff); };
        const unsigned wx = byte(A[0]) | byte(A[1]) << 8 | byte(B[0]) << 16 | byte(B[1]) << 24;
        const unsigned wy = byte(-A[1]) | byte(A[0]) << 8 | byte(-B[1]) << 16 | byte(B[0]) << 24;
        pat[sh * kFsPatWords + i] = make_int2((int)wx, (int)wy);
      }
    QPSK_TRY(open());
    QPSK_TRY(d_pattern.alloc(pat.size()));
    QPSK_TRY(d_st.alloc((size_t)C));
    QPSK_TRY(d_hist.alloc((size_t)C * 2 * H));
    QPSK_TRY(d_fbuf.alloc((size_t)C * (F + 1)));
    QPSK_CUDA_TRY(cudaMemcpyAsync(d_pattern.p, pat.data(), pat.size() * sizeof(int2), cudaMemcpyHostToDevice, stream));
    return reset(stream);
  }
  int run(const float2* sym, long long lds, const int* n_sym, int slots, float2* frames, long long ldf, int* frame_n,
          long long* n_bytes, qpsk_fsync_frame* info, cudaStream_t s) {
    if (!s) s = stream;
    FsArgs a;
    a.sym = sym;
    a.lds = lds;
    a.n_sym = n_sym;
    a.max_sym = (int)std::min<long long>(lds, INT_MAX);
    a.frames = frames;
    a.ldf = ldf;
    a.frame_n = frame_n;
    a.n_bytes = n_bytes;
    a.info = info;
    a.slots = slots;
    a.pattern = d_pattern.p;
    a.st = d_st.p;
    a.hist = d_hist.p;
    a.fbuf = d_fbuf.p;
    a.C = C;
    a.P = P;
    a.F = F;
    a.H = H;
    a.payload = payload;
    a.rho = rho;
    a.scale = scale;
    const int grid = (C + kFsWarps - 1) / kFsWarps;
    if (diff)
      fsync_kernel<true><<<grid, 32 * kFsWarps, 0, s>>>(a);
    else
      fsync_kernel<false><<<grid, 32 * kFsWarps, 0, s>>>(a);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }
  long long slots_bound(long long max_sym) const { return (max_sym + F - 1) / F; }
};

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_fsync {
  FsEngine eng;
  DevBuf<float2> d_sym, d_frames;
  DevBuf<int> d_nsym, d_fn;
  DevBuf<long long> d_nb;
  DevBuf<qpsk_fsync_frame> d_info;
};

extern "C" {

int qpsk_fsync_create(int channels, int differential, float scale, const uint8_t* start_marker, int n_start,
                      int payload_bytes, int n_end, int rho, qpsk_fsync** out) {
  QPSK_TRY(clear_out(out));
  if (!start_marker) return QPSK_ERR_NULL;
  if (channels < 1 || channels > kFsMaxChannels) return QPSK_ERR_UNSUPPORTED;
  if (!(scale > 0.0f) || !isfinite(scale)) return QPSK_ERR_RANGE;
  if (n_start < 1 || n_start > kFsMaxStart || payload_bytes < 1 || payload_bytes > kFsMaxPayload || n_end < 0 ||
      n_end > kFsMaxEnd || rho < 0 || rho > 256)
    return QPSK_ERR_RANGE;
  return create_handle(out, channels, differential, scale, start_marker, n_start, payload_bytes, n_end, rho);
}

int qpsk_fsync_destroy(qpsk_fsync* p) { return destroy_handle(p); }

int qpsk_fsync_reset(qpsk_fsync* p) { return reset_handle(p); }

int qpsk_fsync_shape(const qpsk_fsync* p, int* pattern_syms, int* frame_syms, int* window_syms, int* rho) {
  if (!p || !pattern_syms || !frame_syms || !window_syms || !rho) return QPSK_ERR_NULL;
  *pattern_syms = p->eng.P;
  *frame_syms = p->eng.F;
  *window_syms = p->eng.F + p->eng.delta();
  *rho = p->eng.rho;
  return QPSK_OK;
}

int qpsk_fsync_slots_bound(const qpsk_fsync* p, int64_t max_sym, int64_t* slots) {
  if (!p || !slots) return QPSK_ERR_NULL;
  if (max_sym < 0 || max_sym > ((int64_t)1 << 40)) return QPSK_ERR_RANGE;
  *slots = p->eng.slots_bound(max_sym);
  return QPSK_OK;
}

int qpsk_fsync_process_dev(qpsk_fsync* p, const float* d_sym, int64_t sym_stride_floats, const int* d_n_sym, int slots,
                           float* d_frames, int64_t frame_stride_floats, int* d_frame_n_sym, int64_t* d_n_bytes,
                           qpsk_fsync_frame* d_info, void* stream) {
  if (!p) return QPSK_ERR_NULL;
  if (!d_sym || !d_n_sym || !d_frames || !d_frame_n_sym || !d_n_bytes || !d_info) return QPSK_ERR_NULL;
  if (sym_stride_floats < 0 || frame_stride_floats < 0 || slots < 0) return QPSK_ERR_RANGE;
  if ((sym_stride_floats & 1) || (frame_stride_floats & 1)) return QPSK_ERR_ARG;
  if (misaligned(d_sym) || misaligned(d_n_sym) || misaligned(d_frames) || misaligned(d_frame_n_sym) ||
      misaligned(d_n_bytes) || misaligned(d_info))
    return QPSK_ERR_ARG;
  if (sym_stride_floats / 2 > INT_MAX) return QPSK_ERR_UNSUPPORTED;
  const FsEngine& g = p->eng;
  if (slots < g.slots_bound(sym_stride_floats / 2) || frame_stride_floats < 2LL * (g.F + g.delta()))
    return QPSK_ERR_CAPACITY;
  QPSK_TRY(ensure_device(g.device));
  return p->eng.run((const float2*)d_sym, sym_stride_floats / 2, d_n_sym, slots, (float2*)d_frames, frame_stride_floats / 2,
                    d_frame_n_sym, (long long*)d_n_bytes, d_info, (cudaStream_t)stream);
}

int qpsk_fsync_process(qpsk_fsync* p, const float* sym, int64_t sym_stride_floats, const int64_t* n_sym, int slots,
                       float* frames, int64_t frame_stride_floats, int* frame_n_sym, int64_t* n_bytes,
                       qpsk_fsync_frame* info, int64_t* need_slots) {
  if (!p || !n_sym || !need_slots) return QPSK_ERR_NULL;
  if (sym_stride_floats < 0 || frame_stride_floats < 0 || slots < 0) return QPSK_ERR_RANGE;
  if ((sym_stride_floats & 1) || (frame_stride_floats & 1)) return QPSK_ERR_ARG;
  FsEngine& g = p->eng;
  const size_t C = (size_t)g.C;
  int64_t max_sym;
  QPSK_TRY(host_sym_counts(n_sym, C, sym_stride_floats, &max_sym));
  *need_slots = g.slots_bound(max_sym);
  const long long L = g.F + g.delta();
  if (slots < *need_slots || frame_stride_floats < 2 * L) return QPSK_ERR_CAPACITY;
  if (max_sym > 0 && !sym) return QPSK_ERR_NULL;
  const size_t S = C * (size_t)slots;
  if (S > 0 && (!frames || !frame_n_sym || !n_bytes || !info)) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(g.device));
  cudaStream_t s = g.stream;
  const long long lds = std::max<long long>(max_sym, 1);
  QPSK_TRY(p->d_frames.ensure(std::max<size_t>(S, 1) * (size_t)L));
  QPSK_TRY(p->d_fn.ensure(std::max<size_t>(S, 1)));
  QPSK_TRY(p->d_nb.ensure(std::max<size_t>(S, 1)));
  QPSK_TRY(p->d_info.ensure(std::max<size_t>(S, 1)));
  QPSK_TRY(upload_syms(p->d_sym, p->d_nsym, sym, sym_stride_floats, n_sym, C, max_sym, s));
  QPSK_TRY(g.run(p->d_sym.p, lds, p->d_nsym.p, slots, p->d_frames.p, L, p->d_fn.p, p->d_nb.p, p->d_info.p, s));
  if (S > 0) {
    QPSK_CUDA_TRY(cudaMemcpyAsync(frame_n_sym, p->d_fn.p, S * sizeof(int), cudaMemcpyDeviceToHost, s));
    QPSK_CUDA_TRY(cudaMemcpyAsync(n_bytes, p->d_nb.p, S * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    QPSK_CUDA_TRY(cudaMemcpyAsync(info, p->d_info.p, S * sizeof(qpsk_fsync_frame), cudaMemcpyDeviceToHost, s));
  }
  QPSK_CUDA_TRY(cudaStreamSynchronize(s));
  for (size_t k = 0; k < S; ++k)
    if (frame_n_sym[k] > 0)
      QPSK_CUDA_TRY(cudaMemcpy(frames + k * (size_t)frame_stride_floats, p->d_frames.p + k * (size_t)L,
                               (size_t)frame_n_sym[k] * 8, cudaMemcpyDeviceToHost));
  return QPSK_OK;
}

}  // extern "C"
