// fir.cu — K1/K2: complex-sample FIR kernels for sm_100a and the qpsk_fir_* entry points.
//
// Stands in for ComplexFIRFilter (MS/Models/FIRFilter.cs): streaming Filter(span,span) :80-91 with
// the (N-1)-sample delay line carried across calls, and the stateless fftFilter :96-141 alignment
// y[i] = conv(x,h)[i+N-1].  Both are the same correlation  y[n0+q] = sum_i g[i] * xs[q+i]  over a
// shared-memory tile xs (tile + halo), with g[i] = h[HL-i]; only the tile origin differs.
//
// The tile ring (TileRing, ring_produce): five kernels — fir_tma_kernel, fir_split2_kernel, fir_dec2_kernel,
// fir_exact_real_kernel, fir_decim_tma_kernel — share one pipeline and differ only in their consumer arithmetic:
//   * persistent CTAs, each walking tiles  blockIdx.x + k*gridDim.x  of a channel-major tile grid;
//   * one producer warp stages input tile + halo by TMA bulk copies (cp.async.bulk -> SASS UBLKCP) into a 2-4 deep
//     full/empty mbarrier ring, so loads for the next tiles are in flight while the current one is computed;
//   * the four that store per warp stage each consumer warp's outputs in shared memory and write them back with one
//     bulk store per warp and tile (warp_store).
// On the host, plan_ring sizes the ring from a shared-memory budget and launch_ring starts the persistent grid.
//
// fir_tma_kernel (the hot kernel): tiles of T = NT*R samples, 2 CTAs per SM;
//   * each thread owns R consecutive outputs and slides a register window over the tile: one
//     LDS.128 (two new samples) feeds 2*R packed FFMA2 (fma.rn.f32x2: I and Q of one sample in one
//     issue slot, the real tap broadcast from a uniform register);
//   * R = 10 -> thread stride 80 B = 5 x 16 B chunks, odd, so the LDS.128/STS.128 of a quarter-warp
//     hit 8 distinct 16-byte bank groups: conflict-free on a dense (TMA-compatible) layout.
//   Algorithmic traffic: 8 B read + 8 B written per complex sample; 4*N flop (real taps) or
//   8*N flop (complex taps) per sample.
//
// fir_generic_kernel: one thread per output straight from global memory.  Serves QPSK_FIR_EXACT
// (the reference's 8-lane summation order, no FMA: FIRFilter.cs:165-192), unaligned device
// pointers, and tap counts beyond the parameter-space table.
#include <algorithm>

#include "fir.cuh"

namespace qpsk {

// ---------------------------------------------------------------------------------------------
// PTX wrappers: mbarrier + bulk async copies (TMA, non-tensor form)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// global -> shared bulk copy, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// shared -> global bulk store (bulk-group completion)
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------------------------------------
// kernel arguments
// ---------------------------------------------------------------------------------------------
constexpr int kMaxG = 1040;  // correlation taps held in kernel-parameter (constant-bank) space

struct FirArgs {
  const float2* x;
  float2* y;
  long long ldx, ldy, L;
  const float2* hist_in;  // [C][HL] or null (stateless: zeros)
  float2* hist_out;       // [C][HL] or null
  long long total_tiles;
  int tiles_per_ch;
  int HL, G, advance;
  int E_load;       // samples staged per tile (even)
  int stage_elems;  // float2 slots per stage (even)
  int stages;
  long long n_out;  // outputs per channel (L for the full-rate kernels), counted in tiles by launch_ring
};
struct TapsReal {
  float g[kMaxG];
};
struct TapsCplx {
  float gi[kMaxG];
  float gq[kMaxG];
};

template <bool CPLX>
struct TapsOf {
  using type = TapsReal;
};
template <>
struct TapsOf<true> {
  using type = TapsCplx;
};

// ---------------------------------------------------------------------------------------------
// the hot kernel
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// NTAP (<= 2R, even) correlation taps starting at tap index i0, circular register window w[2R]:
// on entry w[0..R) holds xs[base+i0 .. base+i0+R); slot of element j is (j - i0) mod 2R.
template <int R, bool CPLX, int NTAP, typename Taps>
__device__ __forceinline__ void fir_block(const float2* __restrict__ xnext, const Taps& taps, int i0, float2 (&w)[2 * R],
                                          float2 (&acc)[R], float2 (&accq)[CPLX ? R : 1]) {
  constexpr int W = 2 * R;
  const float4* xn = reinterpret_cast<const float4*>(xnext);   // xs + base + i0 + R
#pragma unroll
  for (int ii = 0; ii < NTAP; ii += 2) {
    const float4 v = xn[ii >> 1];
    w[(R + ii) % W] = make_float2(v.x, v.y);
    w[(R + ii + 1) % W] = make_float2(v.z, v.w);
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if constexpr (!CPLX) {
        const float g = taps.g[i0 + ii + u];
        const float2 gg = make_float2(g, g);
#pragma unroll
        for (int r = 0; r < R; ++r) acc[r] = ffma2(w[(ii + u + r) % W], gg, acc[r]);
      } else {
        const float gi = taps.gi[i0 + ii + u];
        const float gq = taps.gq[i0 + ii + u];
        const float2 ggi = make_float2(gi, gi), ggq = make_float2(gq, gq);
#pragma unroll
        for (int r = 0; r < R; ++r) {
          acc[r] = ffma2(w[(ii + u + r) % W], ggi, acc[r]);
          accq[CPLX ? r : 0] = ffma2(w[(ii + u + r) % W], ggq, accq[CPLX ? r : 0]);
        }
      }
    }
  }
}

// Tile walk of a persistent CTA: tile = blockIdx.x + it*gridDim.x split into (channel, tile within the channel)
// incrementally — one division per kernel instead of one per tile (a 64-bit division costs ~70 instructions and a
// dependent I2F / MUFU.RCP / F2I chain in front of every tile's first LDS).
struct TileWalk {
  long long tile;
  int ch, k, tiles_per_ch, step_ch, step_k;
  __device__ __forceinline__ explicit TileWalk(int tpc) : tiles_per_ch(tpc) {
    tile = blockIdx.x;
    ch = (int)(blockIdx.x / (unsigned)tpc);
    k = (int)(blockIdx.x - (unsigned)ch * (unsigned)tpc);
    step_ch = (int)(gridDim.x / (unsigned)tpc);
    step_k = (int)(gridDim.x - (unsigned)step_ch * (unsigned)tpc);
  }
  __device__ __forceinline__ void next() {
    tile += gridDim.x;
    ch += step_ch;
    k += step_k;
    if (k >= tiles_per_ch) {
      k -= tiles_per_ch;
      ++ch;
    }
  }
};

// ---------------------------------------------------------------------------------------------
// The tile ring shared by the five TMA-pipelined kernels
// ---------------------------------------------------------------------------------------------
// A CTA is NW consumer warps and one producer warp.  The producer stages each tile's input (tile + halo) into the next of
// `stages` shared-memory slots by bulk copies and signals the slot's `full` mbarrier; each consumer warp waits on it, reads
// the slot and arrives on its `empty` mbarrier, which the producer waits on before it refills the slot.  No CTA-wide
// barrier in the steady state, so warps drift apart and one warp's prologue / epilogue overlaps the others' arithmetic.
// Dynamic shared memory: the slots, then the kernel's own region (output staging, ...), then 2 * stages mbarriers.

// A position in the ring: the slot and the phase parity its mbarriers are at
struct RingCursor {
  int stage = 0;
  uint32_t parity = 0;
  __device__ __forceinline__ void next(int stages) {
    if (++stage == stages) {
      stage = 0;
      parity ^= 1u;
    }
  }
};

struct TileRing {
  // stages and stage_elems are read from the kernel parameters where they are used: copies held in registers across the
  // consumer loop cost up to six registers in fir_tma_kernel
  const FirArgs* a;
  float2* slots;     // a->stages x a->stage_elems samples
  uint64_t* full;    // [stages] the slot's copies have landed (one producer arrival + the bytes)
  uint64_t* empty;   // [stages] every consumer warp is done with the slot

  __device__ __forceinline__ float2* slot(int stage) const { return slots + (size_t)stage * a->stage_elems; }
  // the kernel's own region, right after the slots
  __device__ __forceinline__ float2* region() const { return slot(a->stages); }

  // consumer warp: the samples of the cursor's slot, once they have landed
  __device__ __forceinline__ const float2* acquire(const RingCursor& c) const {
    mbar_wait(&full[c.stage], c.parity);
    return slot(c.stage);
  }
  // consumer warp: done reading the slot — hand it back to the producer, move the cursor on
  __device__ __forceinline__ void release(RingCursor& c, int lane) const {
    __syncwarp();
    if (lane == 0) mbar_arrive(&empty[c.stage]);
    c.next(a->stages);
  }
};

// Every thread of the CTA calls this: the ring over `smem` with a kernel region of `region_elems` float2, its mbarriers
// initialised (`empty` counts one arrival per consumer warp) and visible to the whole CTA.
__device__ __forceinline__ TileRing ring_init(unsigned char* smem, const FirArgs& a, int region_elems, int consumer_warps) {
  TileRing r;
  r.a = &a;
  r.slots = reinterpret_cast<float2*>(smem);
  r.full = reinterpret_cast<uint64_t*>(r.region() + region_elems);   // float2 granules: 8-byte aligned as mbarriers need
  r.empty = r.full + a.stages;
  if (threadIdx.x == 0) {
    for (int s = 0; s < a.stages; ++s) {
      mbar_init(&r.full[s], 1);
      mbar_init(&r.empty[s], consumer_warps);
    }
    fence_mbar_init();
  }
  __syncthreads();
  return r;
}

// The producer warp's loop.  Tile k of a channel covers stream indices s0 .. s0 + E_load, s0 = advance + k*T_IN - HL
// (even): T_IN input samples per tile, HL delay-line samples in front of the first.  The part before the stream start
// comes from hist_in by a bulk copy (zeros when hist_in is null: a stateless call), the in-range part by a bulk copy of an
// even count plus one plain load for an odd one, and plain zero stores fill what lies past the stream end.
template <int T_IN>
__device__ __forceinline__ void ring_produce(const FirArgs& a, const TileRing& ring) {
  const int lane = threadIdx.x & 31;
  RingCursor c;
  TileWalk w(a.tiles_per_ch);
  for (int it = 0; w.tile < a.total_tiles; ++it, w.next()) {
    if (it >= a.stages) mbar_wait(&ring.empty[c.stage], c.parity ^ 1u);   // consumers released this slot
    const int ch = w.ch;
    const long long s0 = (long long)a.advance + (long long)w.k * T_IN - a.HL;
    float2* dst = ring.slot(c.stage);
    const float2* xch = a.x + (long long)ch * a.ldx;
    uint64_t* bar = &ring.full[c.stage];
    const int E = a.E_load;
    uint32_t tx = 0;
    int nA = 0;
    if (s0 < 0) {
      nA = (int)((-s0) < (long long)E ? (-s0) : (long long)E);
      if (a.hist_in) {
        if (lane == 0) bulk_g2s(dst, a.hist_in + (long long)ch * a.HL + (a.HL + s0), (uint32_t)nA * 8u, bar);
        tx += (uint32_t)nA * 8u;
      } else {
        for (int i = lane; i < nA; i += 32) dst[i] = make_float2(0.f, 0.f);
      }
    }
    const long long m0 = s0 + nA;
    long long avail = a.L - m0;
    if (avail < 0) avail = 0;
    const int nB = (int)(avail < (long long)(E - nA) ? avail : (long long)(E - nA));
    const int nB2 = nB & ~1;
    if (nB2 > 0) {
      if (lane == 0) bulk_g2s(dst + nA, xch + m0, (uint32_t)nB2 * 8u, bar);
      tx += (uint32_t)nB2 * 8u;
    }
    if ((nB & 1) && lane == 0) dst[nA + nB2] = xch[m0 + nB2];
    for (int i = nA + nB + lane; i < E; i += 32) dst[i] = make_float2(0.f, 0.f);
    __syncwarp();
    if (lane == 0) mbar_arrive_expect_tx(bar, tx);
    c.next(a.stages);
  }
}

// Delay-line carry of a kernel that filters at the full rate: the last tile of a channel (first output n0) holds the
// stream's final HL samples, which the next call reads as hist_in.
template <int NT>
__device__ __forceinline__ void carry_history(const FirArgs& a, const float2* xs, int ch, int k, long long n0) {
  if (a.hist_out && k == a.tiles_per_ch - 1) {
    const int off = (int)(a.L - n0);
    float2* ho = a.hist_out + (long long)ch * a.HL;
    for (int i = threadIdx.x; i < a.HL; i += NT) ho[i] = xs[off + i];
  }
}

// A consumer warp's store of the WS outputs it staged at ys: the first `left` (clamped to 0..WS) go to yg by one bulk
// store, or by lane-strided stores when their count is odd (a bulk copy moves a multiple of 16 bytes).  Either way the
// warp commits one bulk group per tile, which the caller's bulk_wait_read<> before it next writes ys counts.
template <int WS>
__device__ __forceinline__ void warp_store(float2* yg, const float2* ys, int left, int lane) {
  fence_proxy_async_smem();
  __syncwarp();
  const int n = left < 0 ? 0 : (left > WS ? WS : left);
  if ((n & 1) == 0) {
    if (lane == 0) {
      if (n > 0) bulk_s2g(yg, ys, (uint32_t)n * 8u);
      bulk_commit();
    }
  } else {
    for (int i = lane; i < n; i += 32) yg[i] = ys[i];
    if (lane == 0) bulk_commit();
  }
}

// fir_tma_kernel: NT compute threads on the tile ring, R consecutive outputs each; every consumer warp stages its 32*R
// outputs in one of two shared-memory buffers and bulk-stores them.
template <int R, int NT, bool CPLX>
__global__ void __launch_bounds__(NT + 32, 2)
    fir_tma_kernel(const __grid_constant__ FirArgs a, const __grid_constant__ typename TapsOf<CPLX>::type taps) {
  static_assert(R % 2 == 0, "R must be even (LDS.128 moves two samples)");
  constexpr int T = R * NT;
  constexpr int W = 2 * R;   // circular register window
  constexpr int WS = 32 * R; // outputs per consumer warp and tile
  constexpr int NW = NT / 32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const TileRing ring = ring_init(smem_raw, a, 2 * T, NW);

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  if (warp == NW) {
    ring_produce<T>(a, ring);
    return;
  }

  // ---------------- consumer warps ----------------
  const int base = tid * R;
  float2* ys_warp = ring.region() + (size_t)warp * (2 * WS);   // two buffers of WS outputs
  RingCursor cur;
  TileWalk tw(a.tiles_per_ch);
  for (int it = 0; tw.tile < a.total_tiles; ++it, tw.next()) {
    const float2* xs = ring.acquire(cur);
    const int ch = tw.ch;
    const long long n0 = (long long)tw.k * T;
    carry_history<NT>(a, xs, ch, tw.k, n0);

    // ---- register-tiled correlation ----
    float2 w[W];
    float2 acc[R];
    float2 accq[CPLX ? R : 1];
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = make_float2(0.f, 0.f);
#pragma unroll
    for (int r = 0; r < (CPLX ? R : 1); ++r) accq[r] = make_float2(0.f, 0.f);
    const float4* xv = reinterpret_cast<const float4*>(xs + base);
#pragma unroll
    for (int r = 0; r < R; r += 2) {
      const float4 v = xv[r >> 1];
      w[r] = make_float2(v.x, v.y);
      w[r + 1] = make_float2(v.z, v.w);
    }
    int i0 = 0;
    for (; i0 + W <= a.G; i0 += W) fir_block<R, CPLX, W>(xs + base + i0 + R, taps, i0, w, acc, accq);
    // compile-time tail (G - i0 in {0, 2, ..., W-2}): same circular window, no register shuffling
    {
      const float2* xn = xs + base + i0 + R;
      switch ((a.G - i0) >> 1) {
#define QPSK_TAIL(K) case K: fir_block<R, CPLX, ((2 * K) < W ? (2 * K) : 0)>(xn, taps, i0, w, acc, accq); break;
        QPSK_TAIL(1) QPSK_TAIL(2) QPSK_TAIL(3) QPSK_TAIL(4) QPSK_TAIL(5) QPSK_TAIL(6) QPSK_TAIL(7) QPSK_TAIL(8) QPSK_TAIL(9)
        QPSK_TAIL(10) QPSK_TAIL(11) QPSK_TAIL(12) QPSK_TAIL(13) QPSK_TAIL(14) QPSK_TAIL(15)
#undef QPSK_TAIL
        default: break;
      }
    }
    ring.release(cur, lane);

    // ---- epilogue: registers -> this warp's smem slice -> TMA bulk store ----
    float2* ys = ys_warp + (size_t)(it & 1) * WS;
    if (lane == 0) bulk_wait_read<1>();   // the store issued two tiles ago has drained this buffer
    __syncwarp();
    float4* yv = reinterpret_cast<float4*>(ys + lane * R);
#pragma unroll
    for (int r = 0; r < R; r += 2) {
      float2 o0, o1;
      if constexpr (!CPLX) {
        o0 = acc[r];
        o1 = acc[r + 1];
      } else {
        // A = sum gI*(xI,xQ), B = sum gQ*(xI,xQ):  y = (A.x - B.y, A.y + B.x)
        o0 = make_float2(acc[r].x - accq[CPLX ? r : 0].y, acc[r].y + accq[CPLX ? r : 0].x);
        o1 = make_float2(acc[r + 1].x - accq[CPLX ? r + 1 : 0].y, acc[r + 1].y + accq[CPLX ? r + 1 : 0].x);
      }
      yv[r >> 1] = make_float4(o0.x, o0.y, o1.x, o1.y);
    }
    const long long left = a.L - n0;
    const int valid = (int)(left < (long long)T ? left : (long long)T);
    warp_store<WS>(a.y + (long long)ch * a.ldy + n0 + (long long)warp * WS, ys, valid - warp * WS, lane);
  }
  if (lane == 0) bulk_wait<0>();
}

// ---------------------------------------------------------------------------------------------
// fir_split2_kernel: QPSK_FIR_FAST for long real-tap filters — the 2-parallel fast-FIR split
// ---------------------------------------------------------------------------------------------
// The FMA kernel above is bound by the FP32 pipe from ~100 taps on (84 % of its cycles at 257 taps): the only way left to
// go faster is to issue fewer FFMA2.  Split samples and taps into even / odd phases, X0[k] = xs[b+2k], X1[k] = xs[b+2k+1],
// H0[j] = g[2j], H1[j] = g[2j+1] (correlation form, (H*X)[m] = sum_j H[j] X[m+j]):
//     y[b+2m]   = (H0*X0)[m] + (H1*X1)[m]
//     y[b+2m+1] = (H0*X1)[m] + (H1*X0)[m+1]
// and with S[k] = X1[k] + X0[k+1], H2 = H0 + H1:
//     (H2*S)[m] = y[b+2m+1] + (H0*X0)[m+1] + (H1*X1)[m]
// so A = H0*X0 (P+1 values), B = H1*X1 (P values), C = H2*S (P values) give 2P outputs with (3P+1) * G/2 multiply-adds
// instead of 2P * G: 0.8 of the FFMA2 for P = 5.  The summation order differs from both the FMA kernel's and the
// reference's (still inside north_star's 1e-5 of max|y|: tests/test_gpu_fir.py), so QPSK_FIR_EXACT never comes here.
// S is formed once per warp and tile in a warp-private plane of shared memory (one FADD2 per sample pair), not per thread.
// Register windows: three circular windows of P + 2 = 7 slots, 7 sub-taps (14 taps) per unrolled block, so every slot index
// is a compile-time constant; one LDS.128 (X0, X1) and one LDS.64 (S) per sub-tap feed 16 FFMA2.
__device__ __forceinline__ float2 fir_add2(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}
__device__ __forceinline__ float2 fir_sub2(float2 a, float2 b) {
  float2 d;
  asm("sub.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}

constexpr int kMaxGh = kMaxG / 2;
struct TapsSplit {
  float h0[kMaxGh];   // g[2j]
  float h1[kMaxGh];   // g[2j+1]
  float h2[kMaxGh];   // h0 + h1, rounded to fp32 on the host
};

// NJ (<= 7) sub-taps starting at sub-tap j0 (a multiple of 7).  On entry wa / wb hold X0 / X1[j0 .. j0+P] in slots 0..P and wc
// holds S[j0 .. j0+P-1] in slots 0..P-1; xn = float4 view at sample pair j0 + P + 1, sn = S plane at j0 + P.
template <int P, int NJ>
__device__ __forceinline__ void split2_block(const float4* __restrict__ xn, const float2* __restrict__ sn, const TapsSplit& taps, int j0,
                                             float2 (&wa)[P + 2], float2 (&wb)[P + 2], float2 (&wc)[P + 2], float2 (&A)[P + 1],
                                             float2 (&B)[P], float2 (&C)[P]) {
  constexpr int W = P + 2;
#pragma unroll
  for (int jj = 0; jj < NJ; ++jj) {
    const float4 v = xn[jj];                       // (X0, X1)[j + P + 1]: first used by the next sub-tap
    const float2 sv = sn[jj];                      // S[j + P]
    const float t0 = taps.h0[j0 + jj], t1 = taps.h1[j0 + jj], t2 = taps.h2[j0 + jj];
    const float2 g0 = make_float2(t0, t0), g1 = make_float2(t1, t1), g2 = make_float2(t2, t2);
#pragma unroll
    for (int m = 0; m <= P; ++m) A[m] = ffma2(wa[(jj + m) % W], g0, A[m]);
#pragma unroll
    for (int m = 0; m < P; ++m) B[m] = ffma2(wb[(jj + m) % W], g1, B[m]);
#pragma unroll
    for (int m = 0; m < P; ++m) C[m] = ffma2(wc[(jj + m) % W], g2, C[m]);
    wa[(jj + P + 1) % W] = make_float2(v.x, v.y);  // slot of X0[j - 1]: dead
    wb[(jj + P + 1) % W] = make_float2(v.z, v.w);  // slot of X1[j - 1]: dead
    wc[(jj + P) % W] = sv;                         // slot of S[j - 2]: dead
  }
}

template <int R, int NT>
__global__ void __launch_bounds__(NT + 32, 2)
    fir_split2_kernel(const __grid_constant__ FirArgs a, const __grid_constant__ TapsSplit taps) {
  static_assert(R % 4 == 2, "R/2 odd: the per-thread strides of 8R and 4R bytes stay odd multiples of 16 / 8 bytes");
  constexpr int P = R / 2;
  constexpr int T = R * NT;
  constexpr int W = P + 2;
  constexpr int WS = 32 * R;   // outputs per consumer warp and tile
  constexpr int NW = NT / 32;
  const int spw = (WS + a.G) / 2 + 1;                                 // S values per warp (odd or even: 8-byte accesses only)
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const TileRing ring = ring_init(smem_raw, a, T + NW * spw, NW);    // region: one buffer of WS outputs per warp, S planes

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  if (warp == NW) {
    ring_produce<T>(a, ring);
    return;
  }

  // ---------------- consumer warps ----------------
  const int base = tid * R;
  const int wbase = warp * WS;
  float2* ys = ring.region() + (size_t)warp * WS;
  float2* sp = ring.region() + T + (size_t)warp * spw;
  const int Gh = a.G >> 1;
  RingCursor cur;
  TileWalk tw(a.tiles_per_ch);
  for (; tw.tile < a.total_tiles; tw.next()) {
    const float2* xs = ring.acquire(cur);
    const int ch = tw.ch;
    const long long n0 = (long long)tw.k * T;
    carry_history<NT>(a, xs, ch, tw.k, n0);

    // ---- this warp's S plane: S[q] = xs[wbase + 2q + 1] + xs[wbase + 2q + 2] ----
    {
      const float2* xo = xs + wbase + 1;
      const int nq = (WS + a.G) / 2 - 1;            // the last pair a thread of this warp reads is q = WS/2 + Gh - 2
      for (int q0 = lane; q0 < nq; q0 += 96) {      // three pairs in flight per lane: loads first (xs and sp may alias for
        float2 u0[3], u1[3];                        // all the compiler knows, it would not hoist them over the stores)
#pragma unroll
        for (int u = 0; u < 3; ++u) {
          const int q = q0 + 32 * u;
          if (q < nq) {
            u0[u] = xo[2 * q];
            u1[u] = xo[2 * q + 1];
          }
        }
#pragma unroll
        for (int u = 0; u < 3; ++u) {
          const int q = q0 + 32 * u;
          if (q < nq) sp[q] = fir_add2(u0[u], u1[u]);
        }
      }
    }
    __syncwarp();

    // ---- register-tiled correlations A, B, C ----
    float2 wa[W], wb[W], wc[W];
    float2 A[P + 1], B[P], C[P];
#pragma unroll
    for (int m = 0; m <= P; ++m) A[m] = make_float2(0.f, 0.f);
#pragma unroll
    for (int m = 0; m < P; ++m) {
      B[m] = make_float2(0.f, 0.f);
      C[m] = make_float2(0.f, 0.f);
    }
    const float4* xv = reinterpret_cast<const float4*>(xs + base);
    const float2* sv = sp + lane * P;
#pragma unroll
    for (int m = 0; m <= P; ++m) {
      const float4 v = xv[m];
      wa[m] = make_float2(v.x, v.y);
      wb[m] = make_float2(v.z, v.w);
    }
#pragma unroll
    for (int m = 0; m < P; ++m) wc[m] = sv[m];
    int j0 = 0;
    for (; j0 + W <= Gh; j0 += W) split2_block<P, W>(xv + j0 + P + 1, sv + j0 + P, taps, j0, wa, wb, wc, A, B, C);
    switch (Gh - j0) {                              // compile-time tail, same circular windows
#define QPSK_TAIL2(K) case K: split2_block<P, (K < W ? K : 0)>(xv + j0 + P + 1, sv + j0 + P, taps, j0, wa, wb, wc, A, B, C); break;
      QPSK_TAIL2(1) QPSK_TAIL2(2) QPSK_TAIL2(3) QPSK_TAIL2(4) QPSK_TAIL2(5) QPSK_TAIL2(6) QPSK_TAIL2(7) QPSK_TAIL2(8)
#undef QPSK_TAIL2
      default: break;
    }
    // this warp is done reading the input slot and its S plane
    ring.release(cur, lane);

    // ---- epilogue: recombine, registers -> this warp's smem slice -> TMA bulk store ----
    if (lane == 0) bulk_wait_read<0>();   // the previous tile's store has drained the slice
    __syncwarp();
    float4* yv = reinterpret_cast<float4*>(ys + lane * R);
#pragma unroll
    for (int m = 0; m < P; ++m) {
      const float2 ye = fir_add2(A[m], B[m]);
      const float2 yo = fir_sub2(fir_sub2(C[m], A[m + 1]), B[m]);
      yv[m] = make_float4(ye.x, ye.y, yo.x, yo.y);
    }
    const long long left = a.L - n0;
    const int valid = (int)(left < (long long)T ? left : (long long)T);
    warp_store<WS>(a.y + (long long)ch * a.ldy + n0 + (long long)wbase, ys, valid - wbase, lane);
  }
  if (lane == 0) bulk_wait<0>();
}

// ---------------------------------------------------------------------------------------------
// fir_dec2_kernel: decimate-by-2 matched filter on the TMA pipeline (row N1, D = 2)
// ---------------------------------------------------------------------------------------------
// The even outputs of the split above need neither C nor S: y[b+2m] = (H0*X0)[m] + (H1*X1)[m] is the polyphase decimator
// itself, G/2 multiply-adds per input sample = the algorithmic count.  With D = 2 the thread stride on a DENSE tile is
// 8R bytes, an odd multiple of 16 for R = 10 / 14 — so, unlike D >= 4 (fir_decim_kernel's padded layout, filled through
// registers), the tile can arrive on the tile ring read in place, with the per-warp bulk store.  A kept-output phase of 1 (dec_skip) is a leading zero tap (host side), so the tile grid stays on even
// sample indices.  Windows: two circular windows of P + 1 slots (P = R/2 outputs per thread), P + 1 sub-taps per unrolled
// block; one LDS.128 (X0 and X1 of one position) per sub-tap feeds 2P FFMA2.  Measured, 2^28 samples, ms at 33 / 65 / 129 taps:
// (R, NT) = (14, 256) with two output buffers per warp (two ring stages) 0.492 0.773 1.368 | one output buffer (three stages)
// 0.539 0.768 1.359 | (10, 256), four stages 0.526 0.862 1.510.
template <int P, int NJ>
__device__ __forceinline__ void dec2_block(const float4* __restrict__ xn, const TapsReal& taps, int j0, float2 (&wa)[P + 1],
                                           float2 (&wb)[P + 1], float2 (&A)[P], float2 (&B)[P]) {
  constexpr int W = P + 1;
#pragma unroll
  for (int jj = 0; jj < NJ; ++jj) {
    const float4 v = xn[jj];                       // (X0, X1)[j + P]: first used by the next sub-tap
    const float t0 = taps.g[2 * (j0 + jj)], t1 = taps.g[2 * (j0 + jj) + 1];
    const float2 g0 = make_float2(t0, t0), g1 = make_float2(t1, t1);
#pragma unroll
    for (int m = 0; m < P; ++m) A[m] = ffma2(wa[(jj + m) % W], g0, A[m]);
#pragma unroll
    for (int m = 0; m < P; ++m) B[m] = ffma2(wb[(jj + m) % W], g1, B[m]);
    wa[(jj + P) % W] = make_float2(v.x, v.y);      // slot of X0[j - 1]: dead
    wb[(jj + P) % W] = make_float2(v.z, v.w);
  }
}

template <int R, int NT>
__global__ void __launch_bounds__(NT + 32, 2)
    fir_dec2_kernel(const __grid_constant__ FirArgs a, const __grid_constant__ TapsReal taps) {
  static_assert(R % 4 == 2, "R/2 odd: thread stride 8R bytes = an odd multiple of 16");
  constexpr int P = R / 2;
  constexpr int T = R * NT;       // input samples per tile
  constexpr int TO = T / 2;       // outputs per tile
  constexpr int W = P + 1;
  constexpr int WSO = 32 * P;     // outputs per consumer warp and tile
  constexpr int NW = NT / 32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const TileRing ring = ring_init(smem_raw, a, 2 * TO, NW);        // region: two buffers of WSO outputs per warp

  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  if (warp == NW) {
    ring_produce<T>(a, ring);
    return;
  }

  // ---------------- consumer warps ----------------
  const int base = tid * R;
  float2* ys_warp = ring.region() + (size_t)warp * (2 * WSO);
  const int Gh = a.G >> 1;
  RingCursor cur;
  TileWalk tw(a.tiles_per_ch);
  for (int it = 0; tw.tile < a.total_tiles; ++it, tw.next()) {
    const float2* xs = ring.acquire(cur);
    const int ch = tw.ch;
    const long long o0 = (long long)tw.k * TO;               // first output of the tile

    float2 wa[W], wb[W], A[P], B[P];
#pragma unroll
    for (int m = 0; m < P; ++m) {
      A[m] = make_float2(0.f, 0.f);
      B[m] = make_float2(0.f, 0.f);
    }
    const float4* xv = reinterpret_cast<const float4*>(xs + base);
#pragma unroll
    for (int m = 0; m < P; ++m) {
      const float4 v = xv[m];
      wa[m] = make_float2(v.x, v.y);
      wb[m] = make_float2(v.z, v.w);
    }
    int j0 = 0;
    for (; j0 + W <= Gh; j0 += W) dec2_block<P, W>(xv + j0 + P, taps, j0, wa, wb, A, B);
    switch (Gh - j0) {
#define QPSK_TAILD(K) case K: dec2_block<P, (K < W ? K : 0)>(xv + j0 + P, taps, j0, wa, wb, A, B); break;
      QPSK_TAILD(1) QPSK_TAILD(2) QPSK_TAILD(3) QPSK_TAILD(4) QPSK_TAILD(5) QPSK_TAILD(6) QPSK_TAILD(7)
#undef QPSK_TAILD
      default: break;
    }
    ring.release(cur, lane);

    // ---- epilogue: y = A + B -> this warp's smem slice -> TMA bulk store ----
    float2* ys = ys_warp + (size_t)(it & 1) * WSO;
    if (lane == 0) bulk_wait_read<1>();
    __syncwarp();
#pragma unroll
    for (int m = 0; m < P; ++m) ys[lane * P + m] = fir_add2(A[m], B[m]);
    const long long left = a.n_out - o0;
    const int valid = (int)(left < (long long)TO ? left : (long long)TO);
    warp_store<WSO>(a.y + (long long)ch * a.ldy + o0 + (long long)warp * WSO, ys, valid - warp * WSO, lane);
  }
  if (lane == 0) bulk_wait<0>();
}

// ---------------------------------------------------------------------------------------------
// fir_exact_real_kernel: QPSK_FIR_EXACT for real taps on the TMA pipeline
// ---------------------------------------------------------------------------------------------
// ComplexDotWindow's arithmetic (FIRFilter.cs:144-211, Vector<float>.Count == 8) bit for bit: window element i (oldest
// first) goes to lane partial i mod 8, each product and each sum rounded separately (no FMA), lanes added 0..7, then the
// N mod 8 tail elements one by one.  With real taps (imaginary parts +0, FIRFilter.cs users: QPSKDeModulator.cs:278-288)
// the reference's complex product tI = hi*xI - hq*xQ, tQ = hi*xQ + hq*xI reduces to (hi*xI, hi*xQ): the hq terms are +-0,
// and adding +-0 to an accumulator that starts at +0 never changes it (an accumulator is +0 or nonzero, never -0), so
// dropping them leaves every bit of every partial sum unchanged.  That makes it two packed instructions per tap and
// output (one mul.rn.f32x2 and two add.rn.f32) instead of eight scalar ones — about half the speed of the FMA kernel, against a
// fourteenth for the one-thread-per-output kernel below.
// Thread = 2 consecutive outputs (16-byte stride: conflict-free LDS/STS), 8 lane partials each, 8 taps per block with
// a 9-sample register window, on the tile ring with the per-warp bulk store.
__device__ __forceinline__ float2 fmul2(float2 a, float2 b) {
  float2 d;
  asm("mul.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}
// The sum that follows a product is formed with the scalar add.rn intrinsics: ptxas contracts mul.rn.f32x2 feeding
// add.rn.f32x2 into FFMA2 (even under --fmad=false), which rounds once where the reference rounds twice; scalar
// add.rn is never contracted.  Sums of sums (the lane reduction) may use the packed add.
__device__ __forceinline__ float2 fadd2_after_mul(float2 a, float2 prod) {
  return make_float2(__fadd_rn(a.x, prod.x), __fadd_rn(a.y, prod.y));
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 d;
  asm("add.rn.f32x2 %0, %1, %2;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return d;
}

// The product rounded on its own as ONE packed instruction: fma.rn.f32x2(x, g, -0) == round(x*g) exactly (the -0 addend changes
// neither value nor sign), and with the addend loaded at run time ptxas cannot contract it into the packed add that follows —
// so the sum can be add.rn.f32x2 as well: FFMA2 + FADD2 per tap and output instead of FMUL2 + two scalar FADD (the kernel
// was issue-bound on those: issue slots 76 % busy in ncu).
__device__ float2 g_fir_neg_zero2 = {-0.0f, -0.0f};
__device__ __forceinline__ float2 mul_then_add2(float2 acc, float2 x, float2 g, float2 nz) { return fadd2(acc, ffma2(x, g, nz)); }

template <int NT>
__global__ void __launch_bounds__(NT + 32, 3)
    fir_exact_real_kernel(const __grid_constant__ FirArgs a, const __grid_constant__ TapsReal taps, const int n_taps) {
  constexpr int R = 2;
  constexpr int T = R * NT;
  constexpr int WS = 32 * R;   // outputs per consumer warp and tile
  constexpr int NW = NT / 32;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const TileRing ring = ring_init(smem_raw, a, 2 * T, NW);         // region: two buffers of WS outputs per warp
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  if (warp == NW) {
    ring_produce<T>(a, ring);
    return;
  }

  // consumer warps
  float2 nz;
  asm volatile("ld.volatile.global.v2.f32 {%0, %1}, [%2];" : "=f"(nz.x), "=f"(nz.y) : "l"(&g_fir_neg_zero2));
  const int lead = a.HL - (n_taps - 1);      // 0 or 1: xs index of window element 0 relative to the output index
  const int n_vec = n_taps & ~7;
  const int base = tid * R;
  float2* ys_warp = ring.region() + (size_t)warp * (2 * WS);
  RingCursor cur;
  TileWalk tw(a.tiles_per_ch);
  for (int it = 0; tw.tile < a.total_tiles; ++it, tw.next()) {
    const float2* xs = ring.acquire(cur);
    const int ch = tw.ch;
    const long long n0 = (long long)tw.k * T;
    carry_history<NT>(a, xs, ch, tw.k, n0);
    float2 lp[R][8];
#pragma unroll
    for (int r = 0; r < R; ++r)
#pragma unroll
      for (int l = 0; l < 8; ++l) lp[r][l] = make_float2(0.f, 0.f);
    const float2* xw = xs + base + lead;         // window element i of output r is xw[i + r]
    float2 w0 = xw[0];
    for (int ib = 0; ib < n_vec; ib += 8) {
      float2 wv[9];
      wv[0] = w0;
#pragma unroll
      for (int j = 1; j < 9; ++j) wv[j] = xw[ib + j];
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        const float g = taps.g[ib + l + lead];
        const float2 gg = make_float2(g, g);
#pragma unroll
        for (int r = 0; r < R; ++r) lp[r][l] = mul_then_add2(lp[r][l], wv[l + r], gg, nz);
      }
      w0 = wv[8];
    }
    float2 acc[R];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      acc[r] = make_float2(0.f, 0.f);
#pragma unroll
      for (int l = 0; l < 8; ++l) acc[r] = fadd2(acc[r], lp[r][l]);   // lanes 0..7 (:176-180)
    }
    for (int i = n_vec; i < n_taps; ++i) {                             // scalar tail (:183-192)
      const float g = taps.g[i + lead];
      const float2 gg = make_float2(g, g);
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = mul_then_add2(acc[r], xw[i + r], gg, nz);
    }
    // Non-finite results: an infinite SAMPLE makes the reference's hq*x terms NaN (0 * Inf), which the reduction above
    // does not model — recompute such outputs with the full complex product (an overflow to Inf gives the same value
    // either way).
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if (!(fabsf(acc[r].x) <= 3.402823466e+38f) || !(fabsf(acc[r].y) <= 3.402823466e+38f)) {
        float lI[8], lQ[8];
        for (int l = 0; l < 8; ++l) lI[l] = lQ[l] = 0.f;
        for (int i = 0; i < n_vec; ++i) {
          const float2 xv = xw[i + r];
          const float hi = taps.g[i + lead], hq = 0.f;
          lI[i & 7] = __fadd_rn(lI[i & 7], __fsub_rn(__fmul_rn(hi, xv.x), __fmul_rn(hq, xv.y)));
          lQ[i & 7] = __fadd_rn(lQ[i & 7], __fadd_rn(__fmul_rn(hi, xv.y), __fmul_rn(hq, xv.x)));
        }
        float aI = 0.f, aQ = 0.f;
        for (int l = 0; l < 8; ++l) {
          aI = __fadd_rn(aI, lI[l]);
          aQ = __fadd_rn(aQ, lQ[l]);
        }
        for (int i = n_vec; i < n_taps; ++i) {
          const float2 xv = xw[i + r];
          const float hi = taps.g[i + lead], hq = 0.f;
          aI = __fadd_rn(aI, __fsub_rn(__fmul_rn(hi, xv.x), __fmul_rn(hq, xv.y)));
          aQ = __fadd_rn(aQ, __fadd_rn(__fmul_rn(hi, xv.y), __fmul_rn(hq, xv.x)));
        }
        acc[r] = make_float2(aI, aQ);
      }
    }
    ring.release(cur, lane);

    float2* ys = ys_warp + (size_t)(it & 1) * WS;
    if (lane == 0) bulk_wait_read<1>();
    __syncwarp();
    *reinterpret_cast<float4*>(ys + lane * R) = make_float4(acc[0].x, acc[0].y, acc[1].x, acc[1].y);
    const long long left = a.L - n0;
    const int valid = (int)(left < (long long)T ? left : (long long)T);
    warp_store<WS>(a.y + (long long)ch * a.ldy + n0 + (long long)warp * WS, ys, valid - warp * WS, lane);
  }
  if (lane == 0) bulk_wait<0>();
}

// ---------------------------------------------------------------------------------------------
// generic kernel: exact reference order / unaligned / very long filters
// ---------------------------------------------------------------------------------------------
struct GenArgs {
  const float2* x;
  float2* y;
  long long ldx, ldy, L;
  const float2* hist_in;
  const float* hI;  // h[j] real parts, j = 0..N-1
  const float* hQ;
  int C, N, HL, advance;
};

__device__ __forceinline__ float2 gen_in(const GenArgs& a, int ch, long long m) {
  if (m < 0) {
    if (!a.hist_in || m < -(long long)a.HL) return make_float2(0.f, 0.f);
    return a.hist_in[(long long)ch * a.HL + a.HL + m];
  }
  if (m >= a.L) return make_float2(0.f, 0.f);
  return a.x[(long long)ch * a.ldx + m];
}

template <bool EXACT>
__global__ void __launch_bounds__(256) fir_generic_kernel(const GenArgs a) {
  const long long total = (long long)a.C * a.L;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(idx / a.L);
    const long long n = idx - (long long)ch * a.L;
    float outI, outQ;
    if (EXACT) {
      // ComplexDotWindow (FIRFilter.cs:144-211) with Vector<float>.Count == 8: window element i
      // is x[n-(N-1)+i] against reversed tap h[N-1-i]; 8 lane partials, lanes summed 0..7, scalar
      // tail; every product and sum rounded separately (no FMA).
      const int N = a.N;
      const int nVec = N - (N & 7);
      float lI[8], lQ[8];
#pragma unroll
      for (int l = 0; l < 8; ++l) lI[l] = lQ[l] = 0.f;
      const long long first = n + a.advance - (N - 1);
      for (int i = 0; i < nVec; i += 8) {
#pragma unroll
        for (int l = 0; l < 8; ++l) {
          const float2 xv = gen_in(a, ch, first + i + l);
          const float hi = a.hI[N - 1 - (i + l)], hq = a.hQ[N - 1 - (i + l)];
          const float tI = __fsub_rn(__fmul_rn(hi, xv.x), __fmul_rn(hq, xv.y));
          const float tQ = __fadd_rn(__fmul_rn(hi, xv.y), __fmul_rn(hq, xv.x));
          lI[l] = __fadd_rn(lI[l], tI);
          lQ[l] = __fadd_rn(lQ[l], tQ);
        }
      }
      float accI = 0.f, accQ = 0.f;
#pragma unroll
      for (int l = 0; l < 8; ++l) {
        accI = __fadd_rn(accI, lI[l]);
        accQ = __fadd_rn(accQ, lQ[l]);
      }
      for (int i = nVec; i < N; ++i) {
        const float2 xv = gen_in(a, ch, first + i);
        const float hi = a.hI[N - 1 - i], hq = a.hQ[N - 1 - i];
        const float tI = __fsub_rn(__fmul_rn(hi, xv.x), __fmul_rn(hq, xv.y));
        const float tQ = __fadd_rn(__fmul_rn(hi, xv.y), __fmul_rn(hq, xv.x));
        accI = __fadd_rn(accI, tI);
        accQ = __fadd_rn(accQ, tQ);
      }
      outI = accI;
      outQ = accQ;
    } else {
      float aI = 0.f, aQ = 0.f;
      const long long top = n + a.advance;
      for (int j = 0; j < a.N; ++j) {
        const float2 xv = gen_in(a, ch, top - j);
        const float hi = a.hI[j], hq = a.hQ[j];
        aI = fmaf(hi, xv.x, aI);
        aI = fmaf(-hq, xv.y, aI);
        aQ = fmaf(hi, xv.y, aQ);
        aQ = fmaf(hq, xv.x, aQ);
      }
      outI = aI;
      outQ = aQ;
    }
    a.y[(long long)ch * a.ldy + n] = make_float2(outI, outQ);
  }
}

// hist_out[c][i] = element (L - HL + i) of the stream (hist_in ++ x)
__global__ void fir_hist_update_kernel(const float2* x, long long ldx, long long L, const float2* hist_in,
                                       float2* hist_out, int C, int HL) {
  const int total = C * HL;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
    const int ch = idx / HL, i = idx - ch * HL;
    const long long m = L - HL + i;
    hist_out[idx] = (m < 0) ? hist_in[(long long)ch * HL + HL + m] : x[(long long)ch * ldx + m];
  }
}


// ---------------------------------------------------------------------------------------------
// fir_decim_kernel: decimate-by-D streaming FIR, real taps (north_star (2), SURVEY §8d "decimate-by-D variant")
// ---------------------------------------------------------------------------------------------
// y_dec[m] = y[skip + m*D], y the full-rate streaming output of Filter() (FIRFilter.cs:80-91; the reference's matched
// filter is non-decimating, so the oracle is its output subsampled).  Only the kept outputs are computed: 4N/D flop and
// 8 + 8/D bytes per INPUT sample.  Polyphase form: with tap index i = k*D + p,
//     y_dec[m] = sum_p sum_k g[k*D + p] * x_p[m + k],     x_p[j] = xs[j*D + p]
// i.e. D non-decimating sub-filters of K = ceil(G/D) taps, each on one phase of the input.  A thread owns RO consecutive
// decimated outputs and, phase pair by phase pair (one LDS.128 = phases p, p+1 of one input position), slides a register
// window over k: 2*RO packed FFMA2 per LDS.128, the same ratio as fir_tma_kernel.
// Staging: the tile (+ halo) is read with coalesced 8-byte loads into a PADDED shared-memory layout — 16 bytes after every
// thread span of RO*D samples when D >= 4 — so that the thread stride in 16-byte chunks is odd (RO*D/2 + 1; RO*D/2 = 7
// itself for D = 2) and the LDS.128 of a quarter-warp fall in 8 different bank groups for every D.  A dense (TMA) layout
// cannot be conflict-free here: RO*D/2 is even for every D >= 4.  No mbarrier ring: 2-3 resident CTAs per SM overlap one
// CTA's loads with another's FFMA2 stream (the kernel is HBM-bound for all but D = 2 with long filters).
struct DecArgs {
  const float2* x;
  float2* y;
  long long ldx, ldy, L;       // input samples per channel
  const float2* hist_in;       // [C][HL]
  long long n_out;             // decimated outputs per channel
  long long total_tiles;
  int tiles_per_ch;
  int HL, K, skip;             // K polyphase taps per phase; first kept output at input index `skip`
};

template <int RO, int NSTEP, int DEC, bool DENSE = false>
__device__ __forceinline__ void dec_block(const float2* __restrict__ xk, const TapsReal& taps, int t0, float2 (&wA)[2 * RO],
                                          float2 (&wB)[2 * RO], float2 (&acc)[RO]) {
  // NSTEP (<= 2*RO) polyphase taps starting at k0 (t0 = k0*DEC + 2*pair); on entry slots 0..RO-1 of the circular windows
  // hold elements k0 .. k0+RO-1 of the two phases; xk = address of element k0 (first phase), pads not yet applied.
  // DENSE: the tile as a bulk copy left it (no pads).
  constexpr int W = 2 * RO;
  constexpr int PADS = (DEC == 2 || DENSE) ? 0 : 2;
#pragma unroll
  for (int kk = 0; kk < NSTEP; ++kk) {
    // element k0 + kk + RO: (kk + RO) / RO thread spans further on
    const float4 v = *reinterpret_cast<const float4*>(xk + (kk + RO) * DEC + PADS * ((kk + RO) / RO));
    wA[(kk + RO) % W] = make_float2(v.x, v.y);
    wB[(kk + RO) % W] = make_float2(v.z, v.w);
    const float ga = taps.g[t0 + kk * DEC], gb = taps.g[t0 + kk * DEC + 1];
    const float2 gga = make_float2(ga, ga), ggb = make_float2(gb, gb);
#pragma unroll
    for (int r = 0; r < RO; ++r) {
      acc[r] = ffma2(wA[(kk + r) % W], gga, acc[r]);
      acc[r] = ffma2(wB[(kk + r) % W], ggb, acc[r]);
    }
  }
}

// Threads = NTO output chunks x NG phase groups: group g of a chunk handles DEC/2/NG of the phase pairs and the groups'
// partial sums are added through shared memory, so that every decimation factor stages the same ~3600-sample tile with
// the same 256 threads (a wider D would otherwise leave a handful of threads to load a tile).
template <int RO, int NTO, int NG, int DEC>
__global__ void __launch_bounds__(NTO * NG, 4)
    fir_decim_kernel(const __grid_constant__ DecArgs a, const __grid_constant__ TapsReal taps) {
  static_assert(DEC % 2 == 0 && (DEC / 2) % NG == 0, "phase pairs split evenly over the groups");
  constexpr int NT = NTO * NG;
  constexpr int SPAN = RO * DEC;                 // input samples under one thread's outputs
  constexpr int PADS = (DEC == 2) ? 0 : 2;       // float2 slots of padding after every span
  constexpr int PITCH = SPAN + PADS;
  constexpr int T_OUT = RO * NTO;
  constexpr int W = 2 * RO;
  constexpr int PP = DEC / 2 / NG;               // phase pairs per group
  constexpr int LB = 8;                          // staged loads in flight per thread
  extern __shared__ __align__(16) unsigned char smem_dec[];
  float2* ys = reinterpret_cast<float2*>(smem_dec);          // [NG][T_OUT] partial sums
  float2* xs = ys + NG * T_OUT;
  const int tid = threadIdx.x;
  const int to = tid % NTO, grp = tid / NTO;
  const int K = a.K;
  const int E = (T_OUT + K) * DEC;               // staged samples: the tile, the halo and the window's one-step look-ahead
  for (long long tile = blockIdx.x; tile < a.total_tiles; tile += gridDim.x) {
    const int ch = (int)(tile / a.tiles_per_ch);
    const int kt = (int)(tile - (long long)ch * a.tiles_per_ch);
    const long long m0 = (long long)kt * T_OUT;
    const long long s0 = (long long)a.skip + m0 * DEC - a.HL;          // stream index of logical xs[0]
    const float2* xch = a.x + (long long)ch * a.ldx;
    const float2* hch = a.hist_in + (long long)ch * a.HL;
    // interior tiles whose first sample sits on a 16-byte boundary: two samples per load and store (a pair never straddles
    // a pad: spans are an even number of samples) — half the staging instructions of the general path below
    const bool wide = s0 >= 0 && s0 + E <= a.L && ((reinterpret_cast<uintptr_t>(xch + s0) & 15) == 0);
    if (wide) {
      const float4* src4 = reinterpret_cast<const float4*>(xch + s0);
      for (int p0 = tid; p0 < E / 2; p0 += NT * LB) {
        float4 v4[LB];
#pragma unroll
        for (int b = 0; b < LB; ++b) {
          const int p = p0 + b * NT;
          v4[b] = (p < E / 2) ? src4[p] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int b = 0; b < LB; ++b) {
          const int p = p0 + b * NT;
          const int e = 2 * p;
          if (p < E / 2) *reinterpret_cast<float4*>(xs + e + PADS * (e / SPAN)) = v4[b];
        }
      }
    }
    for (int e0 = wide ? E : tid; e0 < E; e0 += NT * LB) {
      float2 v[LB];
#pragma unroll
      for (int b = 0; b < LB; ++b) {             // LB independent loads, then LB stores: the loads overlap
        const int e = e0 + b * NT;
        const long long sidx = s0 + e;
        v[b] = make_float2(0.f, 0.f);
        if (e < E) {
          if (sidx < 0) {
            if (sidx >= -(long long)a.HL) v[b] = hch[a.HL + sidx];
          } else if (sidx < a.L) {
            v[b] = xch[sidx];
          }
        }
      }
#pragma unroll
      for (int b = 0; b < LB; ++b) {
        const int e = e0 + b * NT;
        if (e < E) xs[e + PADS * (e / SPAN)] = v[b];
      }
    }
    __syncthreads();
    float2 acc[RO];
#pragma unroll
    for (int r = 0; r < RO; ++r) acc[r] = make_float2(0.f, 0.f);
    const float2* xb = xs + to * PITCH;
    for (int pp = 0; pp < PP; ++pp) {
      const int pair = grp * PP + pp;
      float2 wA[W], wB[W];
      const float2* xp = xb + 2 * pair;
#pragma unroll
      for (int j = 0; j < RO; ++j) {
        const float4 v = *reinterpret_cast<const float4*>(xp + j * DEC);
        wA[j] = make_float2(v.x, v.y);
        wB[j] = make_float2(v.z, v.w);
      }
      int k0 = 0;
      for (; k0 + W <= K; k0 += W)               // k0 is a multiple of 2*RO: element k0 lies k0/RO spans further on
        dec_block<RO, W, DEC>(xp + k0 * DEC + PADS * (k0 / RO), taps, k0 * DEC + 2 * pair, wA, wB, acc);
      const float2* xk = xp + k0 * DEC + PADS * (k0 / RO);
      const int t0 = k0 * DEC + 2 * pair;
      switch (K - k0) {
#define QPSK_DTAIL(S) case S: dec_block<RO, (S < W ? S : 0), DEC>(xk, taps, t0, wA, wB, acc); break;
        QPSK_DTAIL(1) QPSK_DTAIL(2) QPSK_DTAIL(3) QPSK_DTAIL(4) QPSK_DTAIL(5) QPSK_DTAIL(6) QPSK_DTAIL(7) QPSK_DTAIL(8)
        QPSK_DTAIL(9) QPSK_DTAIL(10) QPSK_DTAIL(11) QPSK_DTAIL(12) QPSK_DTAIL(13)
#undef QPSK_DTAIL
        default: break;
      }
    }
    // partial sums -> shared memory -> one coalesced store per output (the groups' partials added on the way out)
    float2* yp = ys + grp * T_OUT + to * RO;
#pragma unroll
    for (int r = 0; r < RO; ++r) yp[r] = acc[r];
    __syncthreads();
    float2* yc = a.y + (long long)ch * a.ldy + m0;
    const long long left = a.n_out - m0;
    for (int o = tid; o < T_OUT && o < left; o += NT) {
      float2 sum = ys[o];
#pragma unroll
      for (int g2 = 1; g2 < NG; ++g2) {
        const float2 p = ys[g2 * T_OUT + o];
        sum.x += p.x;
        sum.y += p.y;
      }
      yc[o] = sum;
    }
    __syncthreads();                             // tile and partial sums are dead: the next tile may overwrite them
  }
}

// fir_decim_kernel's arithmetic on the tile ring, D = 4, 8, 16: the DENSE tile (+ halo) arrives by bulk copies, so the
// loads of tile t+1 are in flight under the arithmetic of tile t (the register-staged kernel alternates the two inside a
// CTA and leans on four resident CTAs).  The groups' partial sums leave through its own epilogue, not warp_store.  Read in place, a dense tile costs
// 2- / 4- / 8-way bank conflicts on every LDS.128 for D = 4 / 8 / 16 (thread span 56*D bytes = 14 / 28 / 56 sixteen-byte chunks;
// measured: 0.56 / 0.87 / 1.64 ms against 0.68 / 0.65 / 0.62 for the padded register-staged kernel) — so the compute threads
// first move the tile into the PADDED layout of fir_decim_kernel (one LDS.128 + STS.128 per sample pair, both conflict-free),
// hand the ring slot back at once, and run the same phase-pair loops on the padded copy.  An odd kept-output phase is a
// leading zero tap (host side): the ring stays on even sample indices.
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}

template <int RO, int NTO, int NG, int DEC, bool REPACK>
__global__ void __launch_bounds__(NTO * NG + 32, 2)
    fir_decim_tma_kernel(const __grid_constant__ FirArgs a, const __grid_constant__ TapsReal taps) {
  static_assert(DEC % 2 == 0 && (DEC / 2) % NG == 0, "phase pairs split evenly over the groups");
  constexpr int NT = NTO * NG;
  constexpr int NW = NT / 32;
  constexpr int SPAN = RO * DEC;
  constexpr int T_OUT = RO * NTO;
  constexpr int T_IN = T_OUT * DEC;
  constexpr int W = 2 * RO;
  constexpr int PP = DEC / 2 / NG;
  constexpr int PADS = 2;
  constexpr int PITCH = SPAN + PADS;
  const int pad_elems = REPACK ? ((a.E_load + PADS * (a.E_load / SPAN + 1) + 1) & ~1) : 0;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const TileRing ring = ring_init(smem_raw, a, NG * T_OUT + pad_elems, NW);
  float2* ys = ring.region();                                         // [NG][T_OUT] partial sums
  float2* xpad = ys + NG * T_OUT;                                     // REPACK: the tile in the padded layout
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int warp = tid >> 5;
  const int K = a.G;                                                  // polyphase taps per phase
  if (warp == NW) {
    ring_produce<T_IN>(a, ring);                                      // advance = the even part of the kept-output phase
    return;
  }

  const int to = tid % NTO, grp = tid / NTO;
  RingCursor cur;
  TileWalk tw(a.tiles_per_ch);
  for (; tw.tile < a.total_tiles; tw.next()) {
    const float2* xs = ring.acquire(cur);
    const int ch = tw.ch;
    const long long m0 = (long long)tw.k * T_OUT;
    // dense ring slot -> padded layout (a pair never straddles a pad: spans are an even number of samples)
    if constexpr (REPACK) {
      const float4* src4 = reinterpret_cast<const float4*>(xs);
      const int np = a.E_load >> 1;
      for (int p0 = tid; p0 < np; p0 += 4 * NT) {
        float4 v4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int p = p0 + u * NT;
          if (p < np) v4[u] = src4[p];
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int p = p0 + u * NT;
          if (p < np) *reinterpret_cast<float4*>(xpad + 2 * p + PADS * ((2 * p) / SPAN)) = v4[u];
        }
      }
      ring.release(cur, lane);                                        // the ring slot goes back before the arithmetic starts
      named_bar_sync(1, NT);
    }
    constexpr int PD = REPACK ? PADS : 0;                             // pad slots per span in the layout the loops read
    float2 acc[RO];
#pragma unroll
    for (int r = 0; r < RO; ++r) acc[r] = make_float2(0.f, 0.f);
    const float2* xb = REPACK ? xpad + to * PITCH : xs + to * SPAN;
    for (int pp = 0; pp < PP; ++pp) {
      const int pair = grp * PP + pp;
      float2 wA[W], wB[W];
      const float2* xp = xb + 2 * pair;
#pragma unroll
      for (int j = 0; j < RO; ++j) {
        const float4 v = *reinterpret_cast<const float4*>(xp + j * DEC);
        wA[j] = make_float2(v.x, v.y);
        wB[j] = make_float2(v.z, v.w);
      }
      int k0 = 0;
      for (; k0 + W <= K; k0 += W)
        dec_block<RO, W, DEC, !REPACK>(xp + k0 * DEC + PD * (k0 / RO), taps, k0 * DEC + 2 * pair, wA, wB, acc);
      const float2* xk = xp + k0 * DEC + PD * (k0 / RO);
      const int t0 = k0 * DEC + 2 * pair;
      switch (K - k0) {
#define QPSK_DTAIL(S) case S: dec_block<RO, (S < W ? S : 0), DEC, !REPACK>(xk, taps, t0, wA, wB, acc); break;
        QPSK_DTAIL(1) QPSK_DTAIL(2) QPSK_DTAIL(3) QPSK_DTAIL(4) QPSK_DTAIL(5) QPSK_DTAIL(6) QPSK_DTAIL(7) QPSK_DTAIL(8)
        QPSK_DTAIL(9) QPSK_DTAIL(10) QPSK_DTAIL(11) QPSK_DTAIL(12) QPSK_DTAIL(13)
#undef QPSK_DTAIL
        default: break;
      }
    }
    if constexpr (!REPACK) ring.release(cur, lane);                   // this warp is done with the ring slot
    float2* yp = ys + grp * T_OUT + to * RO;
#pragma unroll
    for (int r = 0; r < RO; ++r) yp[r] = acc[r];
    named_bar_sync(1, NT);
    float2* yc = a.y + (long long)ch * a.ldy + m0;
    const long long left = a.n_out - m0;
    for (int o = tid; o < T_OUT && o < left; o += NT) {
      float2 sum = ys[o];
#pragma unroll
      for (int g2 = 1; g2 < NG; ++g2) {
        const float2 p = ys[g2 * T_OUT + o];
        sum.x += p.x;
        sum.y += p.y;
      }
      yc[o] = sum;
    }
    named_bar_sync(1, NT);                                            // the partial sums and the padded tile are dead
  }
}

__global__ void fir_subsample_kernel(const float2* __restrict__ y, long long ldy, long long skip, int dec, long long n_out,
                                     float2* __restrict__ out, long long ldo, int C) {
  const long long total = (long long)C * n_out;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int ch = (int)(idx / n_out);
    const long long m = idx - (long long)ch * n_out;
    out[(long long)ch * ldo + m] = y[(long long)ch * ldy + skip + m * dec];
  }
}

// ---------------------------------------------------------------------------------------------
// FirEngine
// ---------------------------------------------------------------------------------------------
FirEngine::~FirEngine() {
  if (stream) cudaStreamDestroy(stream);
}

int FirEngine::init(const float* taps_in, int n_floats, int channels_in) {
  if (!taps_in) return QPSK_ERR_NULL;
  if ((n_floats & 1) != 0 || n_floats == 0) return QPSK_ERR_ARG;  // FIRFilter.cs:32-33
  if (channels_in <= 0) return QPSK_ERR_RANGE;
  QPSK_TRY(ensure_device());
  device = current_device();
  n_taps = n_floats >> 1;
  channels = channels_in;
  taps_iq.assign(taps_in, taps_in + n_floats);
  real_taps = true;
  for (int j = 0; j < n_taps; ++j)
    if (taps_iq[2 * j + 1] != 0.0f) real_taps = false;
  HL = (n_taps - 1) + ((n_taps - 1) & 1);
  if (HL == 0) HL = 2;  // keep a non-empty, 16-byte sized history even for a 1-tap filter
  QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
  QPSK_TRY(hist[0].alloc((size_t)channels * HL));
  QPSK_TRY(hist[1].alloc((size_t)channels * HL));
  QPSK_TRY(d_taps.alloc((size_t)2 * n_taps));
  std::vector<float> planar((size_t)2 * n_taps);
  for (int j = 0; j < n_taps; ++j) {
    planar[j] = taps_iq[2 * j];
    planar[n_taps + j] = taps_iq[2 * j + 1];
  }
  QPSK_CUDA_TRY(cudaMemcpyAsync(d_taps.p, planar.data(), planar.size() * sizeof(float), cudaMemcpyHostToDevice, stream));
  QPSK_TRY(reset(stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  return QPSK_OK;
}

int FirEngine::reset(cudaStream_t s) {
  QPSK_TRY(hist[0].zero(s));
  QPSK_TRY(hist[1].zero(s));
  cur = 0;
  dec_skip = 0;
  return QPSK_OK;
}

int FirEngine::get_state(float* out, int64_t cap_floats) {
  if (!out) return QPSK_ERR_NULL;
  const int keep = n_taps - 1;
  if (cap_floats < (int64_t)channels * keep * 2) return QPSK_ERR_CAPACITY;
  if (keep == 0) return QPSK_OK;
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  // the newest N-1 of the HL kept samples
  QPSK_CUDA_TRY(cudaMemcpy2D(out, (size_t)keep * 8, hist[cur].p + (HL - keep), (size_t)HL * 8, (size_t)keep * 8,
                             (size_t)channels, cudaMemcpyDeviceToHost));
  return QPSK_OK;
}

int FirEngine::set_state(const float* in, int64_t n_floats) {
  if (!in) return QPSK_ERR_NULL;
  const int keep = n_taps - 1;
  if (n_floats != (int64_t)channels * keep * 2) return QPSK_ERR_ARG;
  QPSK_CUDA_TRY(cudaStreamSynchronize(stream));
  QPSK_CUDA_TRY(cudaMemset(hist[cur].p, 0, hist[cur].n * sizeof(float2)));
  if (keep == 0) return QPSK_OK;
  QPSK_CUDA_TRY(cudaMemcpy2D(hist[cur].p + (HL - keep), (size_t)HL * 8, in, (size_t)keep * 8, (size_t)keep * 8,
                             (size_t)channels, cudaMemcpyHostToDevice));
  return QPSK_OK;
}

namespace {

constexpr int kR = 10;
constexpr int kNT = 256;
constexpr int kNTWide = 320;
constexpr int kSmemBudget = 112 * 1024;  // per CTA, two CTAs per SM

// tile geometry of the TMA kernel: R outputs per thread, NT compute threads, two CTAs per SM.  Measured on a B200, 2^28
// samples, ms for 33 / 65 / 129 / 257 taps (R, NT, CTAs per SM):  (10,256,2) 0.79 1.32 2.37 4.46 | (10,320,2) 0.79 1.29
// 2.43 4.72 | (14,224,2) 0.83 1.40 2.56 4.97 | (6,256,3) 0.92 1.52 2.73 5.15 | (10,192,3) 0.88 1.52 2.78 5.35 |
// (14,192,2) 0.96 1.64 3.01 5.80 | (10,288,2) 0.91 1.59 3.01 5.85: eight consumer warps per CTA (four per scheduler with
// two CTAs) beat both fewer, fatter threads and warp counts that do not divide over the four schedulers.  Ten consumer
// warps (kNTWide) are ahead for real-tap filters of ~48-96 taps (65 taps: 1.29 against 1.32 ms), eight everywhere else.
inline bool fir_wide(int G, bool cplx) { return !cplx && G >= 48 && G <= 96; }

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// fir_split2_kernel geometry and the tap count from which QPSK_FIR_FAST uses it for real taps
// Measured on a B200, 2^28 samples, ms for 33 / 65 / 129 / 257 taps: FMA kernel 0.797 1.296 2.367 4.456 | split (10, 256)
// 0.825 1.187 2.020 3.656 | split (10, 320), two ring stages only: - 1.301 2.243 4.199.  Ahead from ~48 taps on, where the
// FMA pipe rather than HBM sets the time.
constexpr int kS2R = 10, kS2NT = 256;
constexpr int kS2MinForced = 14;        // QPSK_FIR_SPLIT: at least one full block of seven sub-taps
constexpr int kS2MinFast = 48;
inline bool fir_mode_is_fast(int mode) { return mode != QPSK_FIR_EXACT; }

// fir_exact_real_kernel geometry: two outputs per thread, three CTAs per SM in 72 KiB each
constexpr int kENT = 256, kET = 2 * kENT;
constexpr int kExactSmemBudget = 72 * 1024;

// The correlation taps of a delay line of hl samples: g[i + shift] = h[hl - i] for 0 <= i <= hl (zero where hl - i >= N),
// zero elsewhere; im = 0 / 1 takes the real / imaginary parts of h.  shift = 1 is one leading zero tap: a decimator's odd
// kept-output phase, so that its tiles stay on even sample indices.
void corr_taps(float (&g)[kMaxG], const std::vector<float>& taps_iq, int hl, int shift = 0, int im = 0) {
  std::fill(g, g + kMaxG, 0.0f);
  const int N = (int)(taps_iq.size() / 2);
  for (int i = 0; i <= hl; ++i)
    if (hl - i < N) g[i + shift] = taps_iq[2 * (hl - i) + im];
}

// The ring of a kernel whose tiles stage `span` input samples plus a `halo`, next to the kernel's own `fixed` bytes of
// shared memory (ring_init's region): as many stages as `budget` holds, at most four.  Fewer than two (no tile's loads
// in flight under another's arithmetic) does not fit.  Fills a's ring fields; returns the dynamic shared-memory size, or 0
// when the ring does not fit.
size_t plan_ring(FirArgs& a, int span, int halo, size_t fixed, size_t budget) {
  a.E_load = span + halo;
  a.stage_elems = a.E_load + 2;
  const size_t stage_bytes = (size_t)a.stage_elems * 8;
  if (fixed + 128 + 2 * stage_bytes > budget) return 0;
  a.stages = (int)std::min<size_t>(4, (budget - fixed - 128) / stage_bytes);
  return (size_t)a.stages * stage_bytes + fixed + (size_t)a.stages * 16;
}

// Launches a ring kernel over tiles of `tile_out` of the a.n_out outputs per channel: a persistent grid of `per_sm` CTAs
// per SM, never more CTAs than tiles.  On success `last_kernel` names it.
template <typename Kern, typename... Taps>
int launch_ring(Kern kern, const char* name, int threads, int per_sm, int tile_out, size_t smem, FirArgs a, int channels,
                cudaStream_t s, const char*& last_kernel, const Taps&... taps) {
  a.tiles_per_ch = (int)((a.n_out + tile_out - 1) / tile_out);
  a.total_tiles = (long long)a.tiles_per_ch * channels;
  long long grid = (long long)per_sm * device_sm_count();
  if (grid > a.total_tiles) grid = a.total_tiles;
  QPSK_TRY(allow_max_dynamic_smem((const void*)kern));
  kern<<<(int)grid, threads, smem, s>>>(a, taps...);
  QPSK_LAUNCH_CHECK();
  last_kernel = name;
  return QPSK_OK;
}

}  // namespace

int FirEngine::run(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, bool stateless, cudaStream_t s) {
  if (L == 0) return QPSK_OK;
  if (!x || !y) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(device));
  if (!s) s = stream;
  const int N = n_taps;
  // geometry: y[n0+q] = sum_i g[i]*xs[q+i], xs[0] = stream index n0 + advance - hl, g[i] = h[hl-i]
  const int advance = stateless ? (N - 1) : 0;
  const int hl = stateless ? (N - 1) : HL;
  const int G = (hl + 1 + 1) & ~1;
  // the kernels read hist[cur] and leave the updated delay line in hist[cur^1]
  const float2* hin = stateless ? nullptr : hist[cur].p;
  float2* hout = stateless ? nullptr : hist[cur ^ 1].p;
  // bulk copies need 16-byte aligned rows
  const bool rows_ok = aligned16(x) && aligned16(y) && !(channels > 1 && ((ldx & 1) || (ldy & 1)));
  FirArgs a = {};
  a.x = x; a.y = y; a.ldx = ldx; a.ldy = ldy; a.L = L; a.n_out = L;
  a.hist_in = hin; a.hist_out = hout;
  a.HL = hl; a.G = G; a.advance = advance;

  const bool wide = fir_wide(G, !real_taps);
  const int T = kR * (wide ? kNTWide : kNT);
  const bool use_tma = (fir_mode_is_fast(mode) || stateless) && G <= kMaxG && hl <= T && rows_ok;
  const bool want_split = (mode == QPSK_FIR_SPLIT && G >= kS2MinForced) ||
                          (mode == QPSK_FIR_FAST && G >= kS2MinFast);
  int st = QPSK_ERR_UNSUPPORTED;   // UNSUPPORTED: no kernel launched yet, the next one in line takes the call
  constexpr int T2 = kS2R * kS2NT;
  if (use_tma && real_taps && want_split && hl <= T2) {
    const size_t fixed = (size_t)T2 * 8 + (size_t)(kS2NT / 32) * ((32 * kS2R + G) / 2 + 1) * 8;   // outputs, S planes
    if (const size_t smem = plan_ring(a, T2, G, fixed, kSmemBudget)) {
      TapsReal g;
      corr_taps(g.g, taps_iq, hl);
      TapsSplit t;
      for (int j = 0; j < kMaxGh; ++j) {
        t.h0[j] = g.g[2 * j];
        t.h1[j] = g.g[2 * j + 1];
        t.h2[j] = t.h0[j] + t.h1[j];
      }
      st = launch_ring(fir_split2_kernel<kS2R, kS2NT>, "fir_split2_kernel<R=10,NT=256,real taps>", kS2NT + 32, 2, T2, smem,
                       a, channels, s, last_kernel, t);
    }
  }
  if (st == QPSK_ERR_UNSUPPORTED && use_tma) {
    if (const size_t smem = plan_ring(a, T, G, (size_t)2 * T * 8, kSmemBudget)) {
      if (!real_taps) {
        TapsCplx t;
        corr_taps(t.gi, taps_iq, hl, 0, 0);
        corr_taps(t.gq, taps_iq, hl, 0, 1);
        st = launch_ring(fir_tma_kernel<kR, kNT, true>, "fir_tma_kernel<R=10,NT=256,complex taps>", kNT + 32, 2, T, smem, a,
                         channels, s, last_kernel, t);
      } else {
        TapsReal t;
        corr_taps(t.g, taps_iq, hl);
        st = wide ? launch_ring(fir_tma_kernel<kR, kNTWide, false>, "fir_tma_kernel<R=10,NT=320,real taps>", kNTWide + 32, 2,
                                T, smem, a, channels, s, last_kernel, t)
                  : launch_ring(fir_tma_kernel<kR, kNT, false>, "fir_tma_kernel<R=10,NT=256,real taps>", kNT + 32, 2, T, smem,
                                a, channels, s, last_kernel, t);
      }
    }
  }
  // QPSK_FIR_EXACT with real taps: the reference's summation order on the tile ring (streaming: hl = HL, advance = 0)
  if (st == QPSK_ERR_UNSUPPORTED && mode == QPSK_FIR_EXACT && !stateless && real_taps && N >= 8 && rows_ok && G <= kMaxG &&
      HL <= kET) {
    if (const size_t smem = plan_ring(a, kET, G, (size_t)2 * kET * 8, kExactSmemBudget)) {
      TapsReal t;
      corr_taps(t.g, taps_iq, HL);
      st = launch_ring(fir_exact_real_kernel<kENT>, "fir_exact_real_kernel<NT=256>", kENT + 32, 3, kET, smem, a, channels, s,
                       last_kernel, t, N);
    }
  }
  if (st == QPSK_ERR_UNSUPPORTED) {
    GenArgs g;
    g.x = x; g.y = y; g.ldx = ldx; g.ldy = ldy; g.L = L;
    g.hist_in = hin; g.hI = d_taps.p; g.hQ = d_taps.p + N;
    g.C = channels; g.N = N; g.HL = HL; g.advance = advance;
    const long long total = (long long)channels * L;
    long long blocks = (total + 255) / 256;
    const long long cap = 32LL * device_sm_count();
    if (blocks > cap) blocks = cap;
    if (mode == QPSK_FIR_EXACT && !stateless)
      fir_generic_kernel<true><<<(int)blocks, 256, 0, s>>>(g);
    else
      fir_generic_kernel<false><<<(int)blocks, 256, 0, s>>>(g);
    QPSK_LAUNCH_CHECK();
    last_kernel = (mode == QPSK_FIR_EXACT && !stateless) ? "fir_generic_kernel<EXACT>" : "fir_generic_kernel";
    if (!stateless) {
      const int tot = channels * HL;
      fir_hist_update_kernel<<<(tot + 255) / 256, 256, 0, s>>>(x, ldx, L, hin, hout, channels, HL);
      QPSK_LAUNCH_CHECK();
    }
  } else {
    QPSK_TRY(st);
  }
  if (!stateless) cur ^= 1;
  return QPSK_OK;
}


int FirEngine::decimate_dev(const float2* x, int64_t L, int64_t ldx, int dec, float2* y, int64_t cap, int64_t ldy, int64_t* n_out,
                            cudaStream_t s) {
  if (!n_out) return QPSK_ERR_NULL;
  *n_out = 0;
  if (dec < 1) return QPSK_ERR_RANGE;
  if (dec != dec_last) {          // a new decimation factor restarts the phase at the next input sample
    dec_skip = 0;
    dec_last = dec;
  }
  const int64_t nout = (L > dec_skip) ? (L - dec_skip + dec - 1) / dec : 0;
  if (cap < nout) return QPSK_ERR_CAPACITY;          // before anything advances
  if (L == 0) return QPSK_OK;
  if (!x || (nout > 0 && !y)) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(device));
  if (!s) s = stream;
  const int64_t skip = dec_skip;
  int K = (HL + 1 + dec - 1) / dec;
  const bool fast = fir_mode_is_fast(mode) && real_taps && (dec == 2 || dec == 4 || dec == 8 || dec == 16) &&
                    (long long)K * dec <= kMaxG && nout > 0;
  int st = QPSK_ERR_UNSUPPORTED;   // UNSUPPORTED: no kernel launched yet, the next one in line takes the call
  if (fast) {
    const bool x_ok = aligned16(x) && !(channels > 1 && (ldx & 1));
    const bool y_ok = aligned16(y) && !(channels > 1 && (ldy & 1));
    // the ring kernels: an odd kept-output phase is a leading zero tap (sk), the even part of it the ring's advance, so
    // that the tiles stay on even sample indices
    const int sk = (int)(skip & 1);
    FirArgs fa = {};
    fa.x = x; fa.y = y; fa.ldx = ldx; fa.ldy = ldy; fa.L = L; fa.n_out = nout;
    fa.hist_in = hist[cur].p; fa.hist_out = nullptr;
    fa.HL = HL; fa.advance = (int)(skip & ~1LL);
    if (dec == 2 && x_ok && y_ok) {
      // D = 2: fir_dec2_kernel
      constexpr int R2 = 14, NT2 = 256, T2 = R2 * NT2, TO2 = T2 / 2;
      fa.G = (HL + 1 + sk + 1) & ~1;
      if (fa.G <= kMaxG && HL <= T2) {
        if (const size_t smem = plan_ring(fa, T2, fa.G, (size_t)2 * TO2 * 8, kSmemBudget)) {
          TapsReal t;
          corr_taps(t.g, taps_iq, HL, sk);
          st = launch_ring(fir_dec2_kernel<R2, NT2>, "fir_dec2_kernel<R=14,NT=256,D=2>", NT2 + 32, 2, TO2, smem, fa, channels,
                           s, last_kernel, t);
        }
      }
    } else if (dec > 2 && x_ok) {
      // D = 4, 8, 16: fir_decim_tma_kernel on dense tiles
      fa.G = (HL + 1 + sk + dec - 1) / dec;          // polyphase taps per phase
      auto go_tma = [&](auto kern, int NTO, int NG, bool repack, const char* name) -> int {
        const int T_OUT = 7 * NTO, T_IN = T_OUT * dec, halo = fa.G * dec;
        if (halo > kMaxG) return QPSK_ERR_UNSUPPORTED;
        const int E = T_IN + halo;
        const size_t pad_elems = repack ? (size_t)((E + 2 * (E / (7 * dec) + 1) + 1) & ~1) : 0;
        const size_t smem = plan_ring(fa, T_IN, halo, (size_t)NG * T_OUT * 8 + pad_elems * 8, kSmemBudget);
        if (!smem) return QPSK_ERR_UNSUPPORTED;
        TapsReal t;
        corr_taps(t.g, taps_iq, HL, sk);
        return launch_ring(kern, name, NTO * NG + 32, 2, T_OUT, smem, fa, channels, s, last_kernel, t);
      };
      switch (dec) {
        // D = 4 reads the dense tile in place (2-way conflicts cost less than the repack and its barrier: 0.558 against
        // 0.638 ms at 65 taps); D = 8 / 16 repack (0.614 / 0.590 against 0.874 / 1.636 in place)
        case 4: st = go_tma(fir_decim_tma_kernel<7, 128, 2, 4, false>, 128, 2, false, "fir_decim_tma_kernel<RO=7,NTO=128,NG=2,D=4,dense>"); break;
        case 8: st = go_tma(fir_decim_tma_kernel<7, 64, 4, 8, true>, 64, 4, true, "fir_decim_tma_kernel<RO=7,NTO=64,NG=4,D=8,repack>"); break;
        case 16: st = go_tma(fir_decim_tma_kernel<7, 32, 8, 16, true>, 32, 8, true, "fir_decim_tma_kernel<RO=7,NTO=32,NG=8,D=16,repack>"); break;
      }
    }
    if (st == QPSK_ERR_UNSUPPORTED) {
      // the register-staged kernel (fir_decim_kernel): any alignment
      DecArgs a;
      a.x = x; a.y = y; a.ldx = ldx; a.ldy = ldy; a.L = L;
      a.hist_in = hist[cur].p; a.n_out = nout; a.HL = HL; a.skip = (int)skip; a.K = K; a.tiles_per_ch = 0; a.total_tiles = 0;
      TapsReal t;
      corr_taps(t.g, taps_iq, HL);
      auto go = [&](auto kern, int NTO, int NG, int PADS, const char* name) -> int {
        const int T_OUT = 7 * NTO, SPAN = 7 * dec;
        a.tiles_per_ch = (int)((nout + T_OUT - 1) / T_OUT);
        a.total_tiles = (long long)a.tiles_per_ch * channels;
        const int E = (T_OUT + K) * dec;
        const size_t smem = (size_t)(NG * T_OUT + E + PADS * (E / SPAN + 1)) * sizeof(float2);
        if (smem > 200 * 1024) return QPSK_ERR_UNSUPPORTED;
        QPSK_TRY(allow_max_dynamic_smem((const void*)kern));
        long long per_sm = (long long)(224 * 1024) / (long long)(smem + 1024);
        if (per_sm > 4) per_sm = 4;
        if (per_sm < 1) per_sm = 1;
        long long grid = per_sm * device_sm_count();
        if (grid > a.total_tiles) grid = a.total_tiles;
        kern<<<(int)grid, NTO * NG, smem, s>>>(a, t);
        QPSK_LAUNCH_CHECK();
        last_kernel = name;
        return QPSK_OK;
      };
      switch (dec) {
        case 2: st = go(fir_decim_kernel<7, 256, 1, 2>, 256, 1, 0, "fir_decim_kernel<RO=7,NTO=256,NG=1,D=2>"); break;
        case 4: st = go(fir_decim_kernel<7, 128, 2, 4>, 128, 2, 2, "fir_decim_kernel<RO=7,NTO=128,NG=2,D=4>"); break;
        case 8: st = go(fir_decim_kernel<7, 64, 4, 8>, 64, 4, 2, "fir_decim_kernel<RO=7,NTO=64,NG=4,D=8>"); break;
        case 16: st = go(fir_decim_kernel<7, 32, 8, 16>, 32, 8, 2, "fir_decim_kernel<RO=7,NTO=32,NG=8,D=16>"); break;
      }
    }
    if (st != QPSK_OK && st != QPSK_ERR_UNSUPPORTED) return st;
  }
  if (st == QPSK_OK) {
    // the delay line advances exactly as Filter() would advance it
    const int tot = channels * HL;
    fir_hist_update_kernel<<<(tot + 255) / 256, 256, 0, s>>>(x, ldx, L, hist[cur].p, hist[cur ^ 1].p, channels, HL);
    QPSK_LAUNCH_CHECK();
    cur ^= 1;
  } else {
    // any other case (complex taps, QPSK_FIR_EXACT, odd or large D, very long filters): the full-rate filter into
    // scratch, then the kept samples — same values by construction
    const int64_t ld = L + (L & 1);
    QPSK_TRY(dec_tmp.ensure((size_t)ld * channels));
    QPSK_TRY(run(x, dec_tmp.p, L, ldx, ld, false, s));
    if (nout > 0) {
      const long long total = (long long)channels * nout;
      long long blocks = (total + 255) / 256;
      const long long capb = 32LL * device_sm_count();
      if (blocks > capb) blocks = capb;
      fir_subsample_kernel<<<(int)blocks, 256, 0, s>>>(dec_tmp.p, ld, skip, dec, nout, y, ldy, channels);
      QPSK_LAUNCH_CHECK();
    }
  }
  dec_skip = (L > skip) ? (skip + nout * dec - L) : (skip - L);
  *n_out = nout;
  return QPSK_OK;
}

int FirEngine::filter_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, cudaStream_t s) {
  return run(x, y, L, ldx, ldy, false, s);
}
int FirEngine::fft_filter_dev(const float2* x, float2* y, int64_t L, int64_t ldx, int64_t ldy, cudaStream_t s) {
  return run(x, y, L, ldx, ldy, true, s);
}

}  // namespace qpsk

// =============================================================================================
// C ABI
// =============================================================================================
using namespace qpsk;

struct qpsk_fir {
  FirEngine eng;
  // host-pointer pipeline: H2D / kernel / D2H on three streams over kSlots device slots
  static constexpr int kSlots = 3;
  cudaStream_t s_in = nullptr, s_out = nullptr;
  cudaEvent_t ev_h2d[kSlots] = {}, ev_k[kSlots] = {}, ev_d2h[kSlots] = {};
  DevBuf<float2> d_in[kSlots], d_out[kSlots];
  // page-locked staging slots of the pageable-memory path (allocated on first use, one chunk each)
  float2* h_in[kSlots] = {};
  float2* h_out[kSlots] = {};
  size_t h_elems = 0;
  int staging(size_t elems) {
    if (elems <= h_elems) return QPSK_OK;
    for (int i = 0; i < kSlots; ++i) {
      if (h_in[i]) cudaFreeHost(h_in[i]);
      if (h_out[i]) cudaFreeHost(h_out[i]);
      h_in[i] = h_out[i] = nullptr;
    }
    h_elems = 0;
    for (int i = 0; i < kSlots; ++i) {
      QPSK_CUDA_TRY(cudaHostAlloc((void**)&h_in[i], elems * sizeof(float2), cudaHostAllocPortable));
      QPSK_CUDA_TRY(cudaHostAlloc((void**)&h_out[i], elems * sizeof(float2), cudaHostAllocPortable));
    }
    h_elems = elems;
    return QPSK_OK;
  }
  ~qpsk_fir() {
    for (int i = 0; i < kSlots; ++i) {
      if (ev_h2d[i]) cudaEventDestroy(ev_h2d[i]);
      if (ev_k[i]) cudaEventDestroy(ev_k[i]);
      if (ev_d2h[i]) cudaEventDestroy(ev_d2h[i]);
      if (h_in[i]) cudaFreeHost(h_in[i]);
      if (h_out[i]) cudaFreeHost(h_out[i]);
    }
    if (s_in) cudaStreamDestroy(s_in);
    if (s_out) cudaStreamDestroy(s_out);
  }
};

namespace {

// complex samples per pipelined chunk (16 MiB each way): PCIe is the bound of the host-pointer path (8 B in + 8 B
// out per sample, full duplex), so the only losses are the pipeline fill (one chunk H2D) and drain (one chunk D2H)
constexpr int64_t kChunk = 2LL << 20;
constexpr int kSlots = qpsk_fir::kSlots;

int fir_pipeline_init(qpsk_fir* f) {
  if (f->s_in) return QPSK_OK;
  QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&f->s_in, cudaStreamNonBlocking));
  QPSK_CUDA_TRY(cudaStreamCreateWithFlags(&f->s_out, cudaStreamNonBlocking));
  for (int i = 0; i < kSlots; ++i) {
    QPSK_CUDA_TRY(cudaEventCreateWithFlags(&f->ev_h2d[i], cudaEventDisableTiming));
    QPSK_CUDA_TRY(cudaEventCreateWithFlags(&f->ev_k[i], cudaEventDisableTiming));
    QPSK_CUDA_TRY(cudaEventCreateWithFlags(&f->ev_d2h[i], cudaEventDisableTiming));
  }
  return QPSK_OK;
}

// one stream of L complex samples, host to host, chunked so copies overlap the kernels.  The streaming form
// carries the delay line from chunk to chunk; the stateless form (fftFilter alignment, output i needs inputs
// i .. i+N-1) stages N-1 look-ahead samples with every chunk and keeps the first `len` outputs.
int fir_host_stream(qpsk_fir* f, const float* in, float* out, int64_t L, bool stateless) {
  FirEngine& e = f->eng;
  QPSK_TRY(fir_pipeline_init(f));
  const int64_t look = stateless ? (e.n_taps - 1) : 0;
  if (L <= kChunk) {
    QPSK_TRY(f->d_in[0].ensure((size_t)L));
    QPSK_TRY(f->d_out[0].ensure((size_t)L));
    QPSK_CUDA_TRY(cudaMemcpyAsync(f->d_in[0].p, in, (size_t)L * 8, cudaMemcpyHostToDevice, e.stream));
    QPSK_TRY(stateless ? e.fft_filter_dev(f->d_in[0].p, f->d_out[0].p, L, L, L, e.stream)
                       : e.filter_dev(f->d_in[0].p, f->d_out[0].p, L, L, L, e.stream));
    QPSK_CUDA_TRY(cudaMemcpyAsync(out, f->d_out[0].p, (size_t)L * 8, cudaMemcpyDeviceToHost, e.stream));
    QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
    return QPSK_OK;
  }
  for (int b = 0; b < kSlots; ++b) {
    QPSK_TRY(f->d_in[b].ensure((size_t)(kChunk + look)));
    QPSK_TRY(f->d_out[b].ensure((size_t)(kChunk + look)));
  }
  const int64_t chunks = (L + kChunk - 1) / kChunk;
  // pageable caller memory: an asynchronous copy on it blocks the calling thread and the three stages run one after the
  // other; the chunks go through page-locked staging slots instead, filled / drained by the host copy pool (common.cuh)
  const bool bounce_in = host_ptr_is_pageable(in), bounce_out = host_ptr_is_pageable(out);
  if (bounce_in || bounce_out) QPSK_TRY(f->staging((size_t)(kChunk + look)));
  auto drain = [&](int64_t c) -> int {                    // chunk c of the output: staging slot -> caller memory
    const int b = (int)(c % kSlots);
    const int64_t off = c * kChunk;
    const int64_t len = (L - off < kChunk) ? (L - off) : kChunk;
    QPSK_CUDA_TRY(cudaEventSynchronize(f->ev_d2h[b]));
    host_parallel_copy(out + 2 * off, f->h_out[b], (size_t)len * 8);
    return QPSK_OK;
  };
  for (int64_t c = 0; c < chunks; ++c) {
    const int b = (int)(c % kSlots);
    const int64_t off = c * kChunk;
    const int64_t len = (L - off < kChunk) ? (L - off) : kChunk;
    const int64_t in_len = (L - off < len + look) ? (L - off) : (len + look);
    const float* src = in + 2 * off;
    if (bounce_in) {
      if (c >= kSlots) QPSK_CUDA_TRY(cudaEventSynchronize(f->ev_h2d[b]));        // the slot's previous DMA has read it
      host_parallel_copy(f->h_in[b], src, (size_t)in_len * 8);
      src = reinterpret_cast<const float*>(f->h_in[b]);
    }
    if (c >= kSlots) QPSK_CUDA_TRY(cudaStreamWaitEvent(f->s_in, f->ev_k[b], 0));  // slot's previous kernel done
    QPSK_CUDA_TRY(cudaMemcpyAsync(f->d_in[b].p, src, (size_t)in_len * 8, cudaMemcpyHostToDevice, f->s_in));
    QPSK_CUDA_TRY(cudaEventRecord(f->ev_h2d[b], f->s_in));
    QPSK_CUDA_TRY(cudaStreamWaitEvent(e.stream, f->ev_h2d[b], 0));
    if (c >= kSlots) QPSK_CUDA_TRY(cudaStreamWaitEvent(e.stream, f->ev_d2h[b], 0));  // slot's previous D2H done
    QPSK_TRY(stateless ? e.fft_filter_dev(f->d_in[b].p, f->d_out[b].p, in_len, in_len, in_len, e.stream)
                       : e.filter_dev(f->d_in[b].p, f->d_out[b].p, len, len, len, e.stream));
    QPSK_CUDA_TRY(cudaEventRecord(f->ev_k[b], e.stream));
    QPSK_CUDA_TRY(cudaStreamWaitEvent(f->s_out, f->ev_k[b], 0));
    float* dst = bounce_out ? reinterpret_cast<float*>(f->h_out[b]) : out + 2 * off;
    QPSK_CUDA_TRY(cudaMemcpyAsync(dst, f->d_out[b].p, (size_t)len * 8, cudaMemcpyDeviceToHost, f->s_out));
    QPSK_CUDA_TRY(cudaEventRecord(f->ev_d2h[b], f->s_out));
    // the slot of chunk c is written again by chunk c + kSlots: chunk c - 1 leaves its slot now, two iterations early
    if (bounce_out && c >= 1) QPSK_TRY(drain(c - 1));
  }
  if (bounce_out) QPSK_TRY(drain(chunks - 1));
  QPSK_CUDA_TRY(cudaStreamSynchronize(f->s_out));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  return QPSK_OK;
}

int fir_host_batch(qpsk_fir* f, const float* in, float* out, int64_t L, bool stateless) {
  FirEngine& e = f->eng;
  const size_t tot = (size_t)L * e.channels;
  QPSK_TRY(f->d_in[0].ensure(tot));
  QPSK_TRY(f->d_out[0].ensure(tot));
  QPSK_CUDA_TRY(cudaMemcpyAsync(f->d_in[0].p, in, tot * 8, cudaMemcpyHostToDevice, e.stream));
  QPSK_TRY(stateless ? e.fft_filter_dev(f->d_in[0].p, f->d_out[0].p, L, L, L, e.stream)
                     : e.filter_dev(f->d_in[0].p, f->d_out[0].p, L, L, L, e.stream));
  QPSK_CUDA_TRY(cudaMemcpyAsync(out, f->d_out[0].p, tot * 8, cudaMemcpyDeviceToHost, e.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  return QPSK_OK;
}

}  // namespace

extern "C" {

int qpsk_fir_create_batch(const float* taps_iq, int n_floats, int channels, qpsk_fir** out) {
  if (!taps_iq || !out) return QPSK_ERR_NULL;
  *out = nullptr;
  if ((n_floats & 1) != 0 || n_floats <= 0) return QPSK_ERR_ARG;
  qpsk_fir* f = new (std::nothrow) qpsk_fir();
  if (!f) return QPSK_ERR_NOMEM;
  int st = f->eng.init(taps_iq, n_floats, channels);
  if (st != QPSK_OK) {
    delete f;
    return st;
  }
  *out = f;
  return QPSK_OK;
}
int qpsk_fir_create(const float* taps_iq, int n_floats, qpsk_fir** out) {
  return qpsk_fir_create_batch(taps_iq, n_floats, 1, out);
}
int qpsk_fir_destroy(qpsk_fir* f) {
  if (f) {
    cudaSetDevice(f->eng.device);
    if (f->eng.stream) cudaStreamSynchronize(f->eng.stream);
    delete f;
  }
  return QPSK_OK;
}
int qpsk_fir_reset(qpsk_fir* f) {
  if (!f) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  QPSK_TRY(f->eng.reset(f->eng.stream));
  QPSK_CUDA_TRY(cudaStreamSynchronize(f->eng.stream));
  return QPSK_OK;
}
int qpsk_fir_last_kernel(const qpsk_fir* f, char* name, int cap) {
  if (!f || !name) return QPSK_ERR_NULL;
  if (cap < 1) return QPSK_ERR_RANGE;
  snprintf(name, (size_t)cap, "%s", f->eng.last_kernel);
  return QPSK_OK;
}
int qpsk_fir_set_mode(qpsk_fir* f, int mode) {
  if (!f) return QPSK_ERR_NULL;
  if (mode != QPSK_FIR_FAST && mode != QPSK_FIR_EXACT && mode != QPSK_FIR_FMA && mode != QPSK_FIR_SPLIT) return QPSK_ERR_RANGE;
  f->eng.mode = mode;
  return QPSK_OK;
}
int qpsk_fir_num_taps(const qpsk_fir* f, int* n) {
  if (!f || !n) return QPSK_ERR_NULL;
  *n = f->eng.n_taps;
  return QPSK_OK;
}

int qpsk_fir_filter(qpsk_fir* f, const float* in, float* out, int64_t n_floats, int64_t out_cap_floats) {
  if (!f) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;            // FIRFilter.cs:82
  if (out_cap_floats < n_floats) return QPSK_ERR_ARG;      // FIRFilter.cs:83
  if (n_floats == 0) return QPSK_OK;
  if (!in || !out) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  const int64_t L = n_floats >> 1;
  return (f->eng.channels == 1) ? fir_host_stream(f, in, out, L, false) : fir_host_batch(f, in, out, L, false);
}


// decimating matched filter (north_star (2)): host pointers, [channels][n_floats] in, [channels][out_cap_floats] out
int qpsk_fir_decimate(qpsk_fir* f, const float* in, int64_t n_floats, int decim, float* out, int64_t out_cap_floats,
                      int64_t* n_out_floats) {
  if (!f || !n_out_floats) return QPSK_ERR_NULL;
  *n_out_floats = 0;
  if (n_floats < 0 || decim < 1 || out_cap_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;            // FIRFilter.cs:82
  if (n_floats == 0) return QPSK_OK;
  if (!in) return QPSK_ERR_NULL;
  FirEngine& e = f->eng;
  QPSK_TRY(ensure_device(e.device));
  const int64_t L = n_floats >> 1, ld = L + (L & 1);
  const int64_t cap = out_cap_floats >> 1;
  const int64_t ldo = (L + decim - 1) / decim + 2;
  QPSK_TRY(f->d_in[0].ensure((size_t)ld * e.channels));
  QPSK_TRY(f->d_out[0].ensure((size_t)ldo * e.channels));
  int64_t nout = 0;
  // capacity is judged inside decimate_dev before any state moves; the staging copy does not touch the handle's state
  QPSK_CUDA_TRY(cudaMemcpy2DAsync(f->d_in[0].p, (size_t)ld * 8, in, (size_t)L * 8, (size_t)L * 8, (size_t)e.channels,
                                  cudaMemcpyHostToDevice, e.stream));
  QPSK_TRY(e.decimate_dev(f->d_in[0].p, L, ld, decim, f->d_out[0].p, cap < ldo ? cap : ldo, ldo, &nout, e.stream));
  if (nout > 0) {
    if (!out) return QPSK_ERR_NULL;
    QPSK_CUDA_TRY(cudaMemcpy2DAsync(out, (size_t)out_cap_floats * 4, f->d_out[0].p, (size_t)ldo * 8, (size_t)nout * 8,
                                    (size_t)e.channels, cudaMemcpyDeviceToHost, e.stream));
  }
  QPSK_CUDA_TRY(cudaStreamSynchronize(e.stream));
  *n_out_floats = 2 * nout;
  return QPSK_OK;
}

int qpsk_fir_decimate_dev(qpsk_fir* f, const float* d_in, int64_t n_floats, int64_t in_stride_floats, int decim, float* d_out,
                          int64_t out_cap_floats, int64_t out_stride_floats, int64_t* n_out_floats, void* stream) {
  if (!f || !n_out_floats) return QPSK_ERR_NULL;
  *n_out_floats = 0;
  if (n_floats < 0 || decim < 1 || out_cap_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;
  if (n_floats == 0) return QPSK_OK;
  if (!d_in) return QPSK_ERR_NULL;
  if ((in_stride_floats & 1) || (out_stride_floats & 1)) return QPSK_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(d_in) & 7) || (reinterpret_cast<uintptr_t>(d_out) & 7)) return QPSK_ERR_ARG;
  if (f->eng.channels > 1 && (in_stride_floats < n_floats || out_stride_floats < out_cap_floats)) return QPSK_ERR_ARG;
  int64_t nout = 0;
  QPSK_TRY(f->eng.decimate_dev((const float2*)d_in, n_floats >> 1, in_stride_floats >> 1, decim, (float2*)d_out, out_cap_floats >> 1,
                               out_stride_floats >> 1, &nout, (cudaStream_t)stream));
  *n_out_floats = 2 * nout;
  return QPSK_OK;
}

int qpsk_fir_fft_filter(qpsk_fir* f, const float* in, float* out, int64_t n_floats) {
  if (!f || !in) return QPSK_ERR_NULL;                     // FIRFilter.cs:98
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;            // :99
  if (n_floats == 0) return QPSK_OK;                       // :100
  if (!out) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  const int64_t L = n_floats >> 1;
  return (f->eng.channels == 1) ? fir_host_stream(f, in, out, L, true) : fir_host_batch(f, in, out, L, true);
}

static int fir_dev_common(qpsk_fir* f, const float* d_in, float* d_out, int64_t n_floats, int64_t is, int64_t os,
                          void* stream, bool stateless) {
  if (!f) return QPSK_ERR_NULL;
  if (n_floats < 0) return QPSK_ERR_RANGE;
  if ((n_floats & 1) != 0) return QPSK_ERR_ARG;
  if (n_floats == 0) return QPSK_OK;
  if (!d_in || !d_out) return QPSK_ERR_NULL;
  if ((is & 1) || (os & 1)) return QPSK_ERR_ARG;
  if (f->eng.channels > 1 && (is < n_floats || os < n_floats)) return QPSK_ERR_ARG;
  {  // in-place or overlapping buffers would let one tile overwrite another tile's halo
    const char* a0 = (const char*)d_in;
    const char* a1 = a0 + ((size_t)(f->eng.channels - 1) * is + n_floats) * 4;
    const char* b0 = (const char*)d_out;
    const char* b1 = b0 + ((size_t)(f->eng.channels - 1) * os + n_floats) * 4;
    if (a0 < b1 && b0 < a1) return QPSK_ERR_ARG;
  }
  const int64_t L = n_floats >> 1;
  cudaStream_t s = (cudaStream_t)stream;
  return stateless ? f->eng.fft_filter_dev((const float2*)d_in, (float2*)d_out, L, is >> 1, os >> 1, s)
                   : f->eng.filter_dev((const float2*)d_in, (float2*)d_out, L, is >> 1, os >> 1, s);
}
int qpsk_fir_filter_dev(qpsk_fir* f, const float* d_in, float* d_out, int64_t n_floats, int64_t is, int64_t os, void* stream) {
  return fir_dev_common(f, d_in, d_out, n_floats, is, os, stream, false);
}
int qpsk_fir_fft_filter_dev(qpsk_fir* f, const float* d_in, float* d_out, int64_t n_floats, int64_t is, int64_t os, void* stream) {
  return fir_dev_common(f, d_in, d_out, n_floats, is, os, stream, true);
}

int qpsk_fir_get_state(qpsk_fir* f, float* hist_iq, int64_t cap_floats) {
  if (!f) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  return f->eng.get_state(hist_iq, cap_floats);
}
int qpsk_fir_set_state(qpsk_fir* f, const float* hist_iq, int64_t n_floats) {
  if (!f) return QPSK_ERR_NULL;
  QPSK_TRY(ensure_device(f->eng.device));
  return f->eng.set_state(hist_iq, n_floats);
}

}  // extern "C"
