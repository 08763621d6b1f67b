// rs.cu — batched Reed-Solomon outer code over GF(2^8), depth-I byte interleaving (spec: include/qpskcuda.h,
// "Reed-Solomon outer code"; DESIGN.md §3 K14).  Stateless: a handle holds the code's constants only.
//
// One warp per codeword, 8 per CTA; a CTA walks the codewords of the call with a grid stride, so the 32 KiB table it
// stages into shared memory is loaded once per CTA, not once per codeword.  Codeword bytes are loaded 32 at a time (one
// per lane, byte j of the codeword at block offset j*I + i) and broadcast by shuffle.
//
// rs_encode_kernel: lane j owns parity register j (the coefficient of x^(nroots-1-j) of the running remainder).  Per
//   message byte: fb = byte ^ p_0 (shuffle from lane 0), p_j <- p_{j+1} ^ fb * g_{nroots-1-j}; the product is one
//   conflict-free shared load from gen[fb][lane] (lanes >= nroots read 0 and stay 0).
// rs_decode_kernel: lane j owns S_j = r(alpha^j), by Horner: S <- S * alpha^j ^ r_i, one load of mul[S][lane].  All
//   syndromes zero: done (warp-uniform).  Otherwise Berlekamp-Massey in the warp, lane i holding Lambda_i and B_i; the
//   discrepancy sum_i Lambda_i S_{r-i} is an XOR reduction over the lanes.  Chien search with lanes over the n valid
//   positions, then Forney for the lanes that found a root; the checks of the header decide success.  Products in BM,
//   Chien and Forney use log/antilog tables in shared memory.
#include <stdint.h>

#include <algorithm>

#include "handle.cuh"

namespace qpsk {

constexpr int kRsWarps = 8;                 // codewords in flight per CTA
constexpr int kRsMaxN = 255;
constexpr int kRsChunks = 8;                // 32-byte chunks of a codeword
constexpr unsigned kRsFull = 0xffffffffu;

// constants of one code, built on the host at creation
struct RsTables {
  uint32_t mul_alpha[256][32];   // s * alpha^lane
  uint32_t mul_gen[256][32];     // fb * g_{nroots-1-lane} for lane < nroots, else 0
  uint8_t exp[512];              // alpha^(i mod 255)
  uint8_t log[256];              // log[0] unused
};

struct RsEncArgs {
  const uint8_t* msg;
  long long ldm;
  uint8_t* code;
  long long ldc;
  long long words;               // rows * blocks * depth
  long long per_row;             // blocks * depth
  const RsTables* tab;
  int n, k, nroots, depth;
};

struct RsDecArgs {
  const uint8_t* code;
  long long ldc;
  const long long* n_bytes;
  int rows;
  uint8_t* msg;
  long long ldm;
  long long* n_msg;
  int* status;
  long long lds;
  long long per_row;             // codewords a full row holds: (ldc / (depth n)) * depth
  const RsTables* tab;
  int n, k, nroots, depth;
};

__device__ __forceinline__ void rs_stage_table(uint32_t (*dst)[32], const uint32_t (*src)[32]) {
  const uint4* s = reinterpret_cast<const uint4*>(src);
  uint4* d = reinterpret_cast<uint4*>(dst);
  for (int e = threadIdx.x; e < 256 * 32 / 4; e += blockDim.x) d[e] = s[e];
}

__global__ void __launch_bounds__(32 * kRsWarps) rs_encode_kernel(const RsEncArgs a) {
  __shared__ __align__(16) uint32_t gen[256][32];
  rs_stage_table(gen, a.tab->mul_gen);
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int I = a.depth, k = a.k;
  for (long long w = (long long)blockIdx.x * kRsWarps + (threadIdx.x >> 5); w < a.words; w += (long long)gridDim.x * kRsWarps) {
    const long long row = w / a.per_row, q = w - row * a.per_row, b = q / I;
    const int i = (int)(q - b * I);
    const uint8_t* m = a.msg + row * a.ldm + b * I * k + i;
    uint8_t* c = a.code + row * a.ldc + b * I * a.n + i;
    uint32_t p = 0;
    for (int j0 = 0; j0 < k; j0 += 32) {
      const int j = j0 + lane, cnt = min(32, k - j0);
      uint32_t v = 0;
      if (j < k) {
        v = m[(long long)j * I];
        c[(long long)j * I] = (uint8_t)v;
      }
      for (int t = 0; t < cnt; ++t) {
        const uint32_t fb = __shfl_sync(kRsFull, v, t) ^ __shfl_sync(kRsFull, p, 0);
        const uint32_t up = __shfl_down_sync(kRsFull, p, 1);
        p = (lane == 31 ? 0u : up) ^ gen[fb][lane];
      }
    }
    if (lane < a.nroots) c[(long long)(k + lane) * I] = (uint8_t)p;
  }
}

// a * b for b = alpha^lb (lb = -1: b = 0)
__device__ __forceinline__ int rs_mul_log(const uint8_t* ex, const uint8_t* lg, int a, int lb) {
  return (a && lb >= 0) ? ex[lg[a] + lb] : 0;
}

__global__ void __launch_bounds__(32 * kRsWarps, 4) rs_decode_kernel(const RsDecArgs a) {
  __shared__ __align__(16) uint32_t mul[256][32];
  __shared__ uint8_t ex[512], lg[256];
  __shared__ __align__(8) uint8_t corr[kRsWarps][256];
  rs_stage_table(mul, a.tab->mul_alpha);
  for (int e = threadIdx.x; e < 512; e += blockDim.x) ex[e] = a.tab->exp[e];
  for (int e = threadIdx.x; e < 256; e += blockDim.x) lg[e] = a.tab->log[e];
  const int I = a.depth, n = a.n, k = a.k, nr = a.nroots, t = nr / 2;
  const long long bb = (long long)I * n;
  // message counts of every row, whatever the row holds
  for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < a.rows; r += (long long)gridDim.x * blockDim.x) {
    const long long cnt = min(max(a.n_bytes[r], 0LL), a.ldc);
    a.n_msg[r] = cnt / bb * I * k;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
  uint8_t* cw_corr = corr[wi];
  const long long words = (long long)a.rows * a.per_row;
  for (long long w = (long long)blockIdx.x * kRsWarps + wi; w < words; w += (long long)gridDim.x * kRsWarps) {
    const long long row = w / a.per_row, q = w - row * a.per_row, b = q / I;
    const int i = (int)(q - b * I);
    const long long cnt = min(max(a.n_bytes[row], 0LL), a.ldc);
    if (b >= cnt / bb) continue;                                       // warp-uniform
    const uint8_t* src = a.code + row * a.ldc + b * bb + i;
    // syndromes; the received bytes stay in registers, byte 32 q + lane in rx[q]
    uint32_t rx[kRsChunks];
    int s = 0;
#pragma unroll
    for (int qq = 0; qq < kRsChunks; ++qq) {
      rx[qq] = 0;
      const int j0 = qq * 32;
      if (j0 < n) {
        if (j0 + lane < n) rx[qq] = src[(long long)(j0 + lane) * I];
        const int c = min(32, n - j0);
        for (int u = 0; u < c; ++u) s = (int)mul[s][lane] ^ (int)__shfl_sync(kRsFull, rx[qq], u);
      }
    }
    if (lane >= nr) s = 0;
    int L = 0;
    bool ok = true;
    bool fixed = false;
    if (__ballot_sync(kRsFull, s != 0)) {
      fixed = true;
      // Berlekamp-Massey: lane i holds Lambda_i and B_i; b the discrepancy at the last length change (as a log)
      int lam = lane == 0, B = lane == 0, m = 1, lb = 0;
      for (int r = 0; r < nr; ++r) {
        const int sr = __shfl_sync(kRsFull, s, (r - lane) & 31);
        int d = lane <= r && lam && sr ? ex[lg[lam] + lg[sr]] : 0;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) d ^= __shfl_xor_sync(kRsFull, d, off);
        if (d == 0) {
          ++m;
          continue;
        }
        const int lcoef = (lg[d] + 255 - lb) % 255;                    // log(d / b)
        const int sh = __shfl_sync(kRsFull, B, (lane - m) & 31);
        const int upd = lam ^ rs_mul_log(ex, lg, lane >= m ? sh : 0, lcoef);
        if (2 * L <= r) {
          B = lam;
          L = r + 1 - L;
          lb = lg[d];
          m = 1;
        } else {
          ++m;
        }
        lam = upd;
        if (L > t) break;                                              // L never shrinks: no codeword within t
      }
      const unsigned nzl = __ballot_sync(kRsFull, lam != 0);
      ok = L <= t && 31 - __clz((int)nzl) == L;
      // Chien: Lambda(alpha^-e) over the valid exponents e = 32 qq + lane < n (byte n-1-e)
      const int llam = lam ? lg[lam] : -1;
      unsigned roots = 0;
      int nroot = 0;
      if (ok) {
#pragma unroll
        for (int qq = 0; qq < kRsChunks; ++qq) {
          if (qq * 32 >= n) break;
          const int e = qq * 32 + lane, step = e ? 255 - e : 0;
          int v = 0, acc = 0;
          for (int ii = 0; ii <= L; ++ii) {
            const int li = __shfl_sync(kRsFull, llam, ii);
            if (li >= 0) v ^= ex[li + acc];
            acc += step;
            if (acc >= 255) acc -= 255;
          }
          const bool root = e < n && v == 0;
          roots |= (unsigned)root << qq;
          nroot += __popc(__ballot_sync(kRsFull, root));
        }
        ok = nroot == L;
      }
      if (ok) {
        // Forney: Omega_i = sum_{j <= i} Lambda_j S_{i-j} for i < L; e = X Omega(X^-1) / Lambda'(X^-1), X = alpha^e
        int om = 0;
        for (int j = 0; j < L; ++j) {
          const int lj = __shfl_sync(kRsFull, llam, j), sj = __shfl_sync(kRsFull, s, (lane - j) & 31);
          if (j <= lane && lane < L) om ^= rs_mul_log(ex, lg, sj, lj);
        }
        const int lom = om ? lg[om] : -1;
        reinterpret_cast<uint2*>(cw_corr)[lane] = make_uint2(0u, 0u);
        __syncwarp();
        bool bad = false;
#pragma unroll
        for (int qq = 0; qq < kRsChunks; ++qq) {
          if (qq * 32 >= n) break;
          if (!__ballot_sync(kRsFull, (roots >> qq) & 1)) continue;
          const int e = qq * 32 + lane, step = e ? 255 - e : 0;
          int num = 0, den = 0, acc = 0;
          for (int ii = 0; ii <= L; ++ii) {                            // X^-i: acc = i * step mod 255
            const int lo = __shfl_sync(kRsFull, lom, ii), li = __shfl_sync(kRsFull, llam, ii);
            if (ii < L && lo >= 0) num ^= ex[lo + acc];
            if ((ii & 1) && li >= 0) den ^= ex[li + (acc + e) % 255];    // Lambda_i X^-(i-1)
            acc += step;
            if (acc >= 255) acc -= 255;
          }
          if ((roots >> qq) & 1) {
            if (num == 0 || den == 0) {
              bad = true;
            } else {
              cw_corr[n - 1 - e] = ex[(e + lg[num] + 255 - lg[den]) % 255];
            }
          }
        }
        ok = !__ballot_sync(kRsFull, bad);
        __syncwarp();
      }
    }
    uint8_t* dst = a.msg + row * a.ldm + b * I * k + i;
#pragma unroll
    for (int qq = 0; qq < kRsChunks; ++qq) {
      const int j = qq * 32 + lane;
      if (qq * 32 < k && j < k) dst[(long long)j * I] = (uint8_t)(rx[qq] ^ (fixed && ok ? cw_corr[j] : 0u));
    }
    if (lane == 0) a.status[row * a.lds + b * I + i] = ok ? L : -1;
    __syncwarp();
  }
}

static void rs_build_tables(int nroots, RsTables* T) {
  int x = 1;
  for (int e = 0; e < 255; ++e) {
    T->exp[e] = (uint8_t)x;
    T->log[x] = (uint8_t)e;
    x <<= 1;
    if (x & 0x100) x ^= 0x11d;
  }
  T->log[0] = 0;
  for (int e = 255; e < 512; ++e) T->exp[e] = T->exp[e - 255];
  auto mul = [T](int a, int b) { return (a && b) ? (int)T->exp[T->log[a] + T->log[b]] : 0; };
  int g[33] = {1};                                                      // g[i]: coefficient of x^i
  for (int j = 0; j < nroots; ++j) {
    const int r = T->exp[j];
    for (int i = j + 1; i >= 1; --i) g[i] = g[i - 1] ^ mul(g[i], r);
    g[0] = mul(g[0], r);
  }
  for (int s = 0; s < 256; ++s)
    for (int l = 0; l < 32; ++l) {
      T->mul_alpha[s][l] = (uint32_t)mul(s, T->exp[l]);
      T->mul_gen[s][l] = l < nroots ? (uint32_t)mul(s, g[nroots - 1 - l]) : 0u;
    }
}

struct RsEngine : EngineBase {
  int nroots = 0, k = 0, n = 0, depth = 0, grid_cap = 1;
  DevBuf<RsTables> d_tab;
  int init(int nr, int kk, int I) {
    nroots = nr;
    k = kk;
    n = kk + nr;
    depth = I;
    QPSK_TRY(open());
    RsTables* h = new (std::nothrow) RsTables();
    if (!h) return QPSK_ERR_NOMEM;
    rs_build_tables(nroots, h);
    int st = d_tab.alloc(1);
    if (st == QPSK_OK && cudaMemcpy(d_tab.p, h, sizeof(RsTables), cudaMemcpyHostToDevice) != cudaSuccess) st = QPSK_ERR_CUDA;
    delete h;
    QPSK_TRY(st);
    int per_sm = 0, per_sm_enc = 0;
    QPSK_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, rs_decode_kernel, 32 * kRsWarps, 0));
    QPSK_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm_enc, rs_encode_kernel, 32 * kRsWarps, 0));
    grid_cap = std::max(1, std::min(per_sm, per_sm_enc)) * device_sm_count();
    return QPSK_OK;
  }
  int grid(long long words) const { return (int)std::max(1LL, std::min<long long>(grid_cap, (words + kRsWarps - 1) / kRsWarps)); }
  int encode(const uint8_t* msg, long long ldm, int rows, long long blocks, uint8_t* code, long long ldc, cudaStream_t s) {
    RsEncArgs a;
    a.msg = msg;
    a.ldm = ldm;
    a.code = code;
    a.ldc = ldc;
    a.per_row = blocks * depth;
    a.words = a.per_row * rows;
    a.tab = d_tab.p;
    a.n = n;
    a.k = k;
    a.nroots = nroots;
    a.depth = depth;
    if (a.words == 0) return QPSK_OK;
    rs_encode_kernel<<<grid(a.words), 32 * kRsWarps, 0, s>>>(a);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }
  int decode(const uint8_t* code, long long ldc, const long long* n_bytes, int rows, uint8_t* msg, long long ldm,
             long long* n_msg, int* status, long long lds, cudaStream_t s) {
    RsDecArgs a;
    a.code = code;
    a.ldc = ldc;
    a.n_bytes = n_bytes;
    a.rows = rows;
    a.msg = msg;
    a.ldm = ldm;
    a.n_msg = n_msg;
    a.status = status;
    a.lds = lds;
    a.per_row = ldc / ((long long)depth * n) * depth;
    a.tab = d_tab.p;
    a.n = n;
    a.k = k;
    a.nroots = nroots;
    a.depth = depth;
    const long long words = std::max(a.per_row * rows, (long long)rows);   // every row gets its count
    rs_decode_kernel<<<grid(words), 32 * kRsWarps, 0, s>>>(a);
    QPSK_LAUNCH_CHECK();
    return QPSK_OK;
  }
};

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_rs {
  RsEngine eng;
};

extern "C" {

int qpsk_rs_create(int nroots, int k, int depth, qpsk_rs** out) {
  QPSK_TRY(clear_out(out));
  if (nroots < 2 || nroots > 32 || (nroots & 1) || depth < 1 || depth > 8) return QPSK_ERR_UNSUPPORTED;
  if (k < 1 || k > kRsMaxN - nroots) return QPSK_ERR_RANGE;
  return create_handle(out, nroots, k, depth);
}

int qpsk_rs_destroy(qpsk_rs* p) { return destroy_handle(p); }

int qpsk_rs_encode_dev(qpsk_rs* p, const uint8_t* d_msg, int64_t msg_stride, int rows, int64_t n_blocks, uint8_t* d_code,
                       int64_t code_stride, void* stream) {
  if (!p) return QPSK_ERR_NULL;
  if (rows < 0 || n_blocks < 0 || msg_stride < 0 || code_stride < 0) return QPSK_ERR_RANGE;
  const RsEngine& g = p->eng;
  if (n_blocks > ((int64_t)1 << 40) / (g.depth * g.n)) return QPSK_ERR_RANGE;
  if (msg_stride < n_blocks * g.depth * g.k) return QPSK_ERR_ARG;
  if (code_stride < n_blocks * g.depth * g.n) return QPSK_ERR_CAPACITY;
  if (rows == 0 || n_blocks == 0) return QPSK_OK;
  if (!d_msg || !d_code) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(g.device));
  return p->eng.encode(d_msg, msg_stride, rows, n_blocks, d_code, code_stride, stream ? (cudaStream_t)stream : g.stream);
}

int qpsk_rs_decode_dev(qpsk_rs* p, const uint8_t* d_code, int64_t code_stride, const int64_t* d_n_bytes, int rows,
                       uint8_t* d_msg, int64_t msg_stride, int64_t* d_n_msg, int* d_status, int64_t status_stride,
                       void* stream) {
  if (!p) return QPSK_ERR_NULL;
  if (rows < 0 || code_stride < 0 || msg_stride < 0 || status_stride < 0) return QPSK_ERR_RANGE;
  const RsEngine& g = p->eng;
  const int64_t blocks = code_stride / ((int64_t)g.depth * g.n);
  if (msg_stride < blocks * g.depth * g.k || status_stride < blocks * g.depth) return QPSK_ERR_CAPACITY;
  if (rows == 0) return QPSK_OK;
  if (!d_code || !d_n_bytes || !d_msg || !d_n_msg || !d_status) return QPSK_ERR_NULL;
  if (misaligned(d_n_bytes) || misaligned(d_n_msg) || misaligned(d_status, 4)) return QPSK_ERR_ARG;
  QPSK_TRY(ensure_device(g.device));
  return p->eng.decode(d_code, code_stride, (const long long*)d_n_bytes, rows, d_msg, msg_stride, (long long*)d_n_msg,
                       d_status, status_stride, stream ? (cudaStream_t)stream : g.stream);
}

int qpsk_rs_encode(qpsk_rs* p, const uint8_t* msg, int64_t n_blocks, uint8_t* code) {
  if (!p) return QPSK_ERR_NULL;
  if (n_blocks < 0) return QPSK_ERR_RANGE;
  RsEngine& g = p->eng;
  if (n_blocks > ((int64_t)1 << 40) / (g.depth * g.n)) return QPSK_ERR_RANGE;
  if (n_blocks == 0) return QPSK_OK;
  if (!msg || !code) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(g.device));
  const size_t nm = (size_t)n_blocks * g.depth * g.k, nc = (size_t)n_blocks * g.depth * g.n;
  cudaStream_t s = g.stream;
  uint8_t* d = nullptr;                    // per call: concurrent host calls share no buffer
  QPSK_CUDA_TRY(cudaMallocAsync((void**)&d, nm + nc, s));
  int st = QPSK_OK;
  if (cudaMemcpyAsync(d, msg, nm, cudaMemcpyHostToDevice, s) != cudaSuccess) st = QPSK_ERR_CUDA;
  if (st == QPSK_OK) st = g.encode(d, (long long)nm, 1, n_blocks, d + nm, (long long)nc, s);
  if (st == QPSK_OK && cudaMemcpyAsync(code, d + nm, nc, cudaMemcpyDeviceToHost, s) != cudaSuccess) st = QPSK_ERR_CUDA;
  cudaFreeAsync(d, s);
  if (cudaStreamSynchronize(s) != cudaSuccess && st == QPSK_OK) st = QPSK_ERR_CUDA;
  return st;
}

int qpsk_rs_decode(qpsk_rs* p, const uint8_t* code, int64_t n_blocks, uint8_t* msg, int* status) {
  if (!p) return QPSK_ERR_NULL;
  if (n_blocks < 0) return QPSK_ERR_RANGE;
  RsEngine& g = p->eng;
  if (n_blocks > ((int64_t)1 << 40) / (g.depth * g.n)) return QPSK_ERR_RANGE;
  if (n_blocks == 0) return QPSK_OK;
  if (!code || !msg || !status) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(g.device));
  const size_t nc = (size_t)n_blocks * g.depth * g.n, nm = (size_t)n_blocks * g.depth * g.k, ns = (size_t)n_blocks * g.depth;
  const size_t o_cnt = (nc + nm + 7) & ~(size_t)7, o_st = o_cnt + 16;
  cudaStream_t s = g.stream;
  uint8_t* d = nullptr;
  QPSK_CUDA_TRY(cudaMallocAsync((void**)&d, o_st + 4 * ns, s));
  const int64_t count = (int64_t)nc;
  int st = QPSK_OK;
  if (cudaMemcpyAsync(d, code, nc, cudaMemcpyHostToDevice, s) != cudaSuccess ||
      cudaMemcpyAsync(d + o_cnt, &count, 8, cudaMemcpyHostToDevice, s) != cudaSuccess)
    st = QPSK_ERR_CUDA;
  if (st == QPSK_OK)
    st = g.decode(d, (long long)nc, (const long long*)(d + o_cnt), 1, d + nc, (long long)nm, (long long*)(d + o_cnt + 8),
                  (int*)(d + o_st), (long long)ns, s);
  if (st == QPSK_OK && (cudaMemcpyAsync(msg, d + nc, nm, cudaMemcpyDeviceToHost, s) != cudaSuccess ||
                        cudaMemcpyAsync(status, d + o_st, 4 * ns, cudaMemcpyDeviceToHost, s) != cudaSuccess))
    st = QPSK_ERR_CUDA;
  cudaFreeAsync(d, s);
  if (cudaStreamSynchronize(s) != cudaSuccess && st == QPSK_OK) st = QPSK_ERR_CUDA;
  return st;
}

}  // extern "C"
