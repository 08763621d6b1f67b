// common.cuh — shared host/device helpers for libqpskcuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <new>
#include <string>
#include <vector>

#include "../../include/qpskcuda.h"

namespace qpsk {

// ---- error plumbing ------------------------------------------------------------------------
void set_cuda_error(cudaError_t e, const char* what, const char* file, int line);
void count_launch(int n = 1);

#define QPSK_CUDA_TRY(expr)                                          \
  do {                                                               \
    cudaError_t _e = (expr);                                         \
    if (_e != cudaSuccess) {                                         \
      ::qpsk::set_cuda_error(_e, #expr, __FILE__, __LINE__);         \
      return (_e == cudaErrorMemoryAllocation) ? QPSK_ERR_NOMEM : QPSK_ERR_CUDA; \
    }                                                                \
  } while (0)

#define QPSK_TRY(expr)                 \
  do {                                 \
    int _s = (expr);                   \
    if (_s != QPSK_OK) return _s;      \
  } while (0)

// after a kernel launch
#define QPSK_LAUNCH_CHECK()                      \
  do {                                           \
    ::qpsk::count_launch();                      \
    QPSK_CUDA_TRY(cudaGetLastError());           \
  } while (0)

int current_device();          // ordinal handles created by THIS thread get: the thread's qpsk_set_device choice, else the
                               // process-wide one (last qpsk_set_device of any thread), else 0
int ensure_device(int dev = -1);  // cudaSetDevice(dev, or current_device()) + arch check; status code
// Raise a kernel's dynamic shared-memory limit to the device's opt-in maximum, once per (kernel, device).  The limit is a
// per-function, per-context setting: setting it to each launch's own size from several host threads races (thread A
// lowers it between thread B's set and launch -> cudaErrorInvalidValue on B's launch).
int allow_max_dynamic_smem(const void* kernel);
int device_sm_count();         // of the device the calling thread has current (call after ensure_device)

// Host side of the pageable-memory path.  cudaMemcpyAsync on memory the driver has not page-locked is a blocking, staged copy on
// the calling thread: the H2D / kernel / D2H pipelines of the host entry points degenerate into a sequence (FIR end to end:
// 0.85 Gsample/s against 5.6 on page-locked buffers).  Such calls go through page-locked staging slots instead, filled and
// drained by a pool of six host threads (fewer on smaller hosts) while the DMA engines work on the other slots.
bool host_ptr_is_pageable(const void* p);            // true when the driver does not know the address as page-locked memory
void host_parallel_copy(void* dst, const void* src, size_t bytes);   // blocking; split over the pool and the caller
// `rows` pieces of `width` bytes, `spitch` / `dpitch` bytes apart (a time chunk of a [channels][samples] block)
void host_parallel_copy_rows(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows);

// RAII device buffer
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t n = 0;
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  ~DevBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    n = 0;
  }
  int alloc(size_t count) {
    release();
    if (count == 0) return QPSK_OK;
    QPSK_CUDA_TRY(cudaMalloc((void**)&p, count * sizeof(T)));
    n = count;
    return QPSK_OK;
  }
  int ensure(size_t count) { return (count <= n) ? QPSK_OK : alloc(count); }
  int zero(cudaStream_t s) {
    if (p) QPSK_CUDA_TRY(cudaMemsetAsync(p, 0, n * sizeof(T), s));
    return QPSK_OK;
  }
};

// ---- counter RNG (spec: DESIGN.md "counter RNG"; the oracle restates the same function) -----
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t rng_u64(uint64_t seed, uint64_t stream, uint64_t counter) {
  uint64_t a = mix64(seed + 0x9E3779B97F4A7C15ULL * (stream + 1));
  return mix64(a + 0xD1B54A32D192ED03ULL * (counter + 1));
}
__host__ __device__ __forceinline__ double rng_double(uint64_t seed, uint64_t stream, uint64_t counter) {
  return (double)(rng_u64(seed, stream, counter) >> 11) * (1.0 / 9007199254740992.0);
}

// ---- device math helpers -------------------------------------------------------------------
#ifdef __CUDACC__
// packed fp32x2 FMA (Blackwell FFMA2): d = a*b + c on both halves, one issue slot.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;"
      : "=l"(reinterpret_cast<unsigned long long&>(d))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)),
        "l"(reinterpret_cast<unsigned long long&>(c)));
  return d;
}
// MathF.Sin/Cos model: the correctly rounded fp32 value, i.e. fp64 evaluation rounded once.  The
// oracle uses the same definition (cr_sinf/cr_cosf), so results agree except where the fp64 value
// lies within an fp64 ulp of an fp32 rounding boundary (probability ~2^-28 per call).
__device__ __forceinline__ void sincos_f32_exact(float x, float* s, float* c) {
  double sd, cd;
  sincos((double)x, &sd, &cd);
  *s = (float)sd;
  *c = (float)cd;
}
// Branch-free fp64 sincos for |x| < 1e5: 3-term Cody-Waite reduction to [-pi/4, pi/4] and Taylor
// polynomials (Estrin form) with DFMA.  Within 1 ulp of glibc's sin/cos (checked on 4e8 arguments on
// the host with fma(): identical after the cast to fp32), like CUDA's own sincos() — but straight-line
// code, so the scheduler can interleave it with the independent filter arithmetic of the loop kernels.
__device__ __forceinline__ void sincos_fast_f64(double x, double* sn, double* cs) {
  const double k = rint(x * 0.63661977236758134308);
  double r = fma(-k, 1.5707963267948966e+00, x);
  r = fma(-k, 6.123233995736766e-17, r);
  r = fma(-k, -1.4973849048591698e-33, r);
  const double z = r * r, z2 = z * z, z4 = z2 * z2, z8 = z4 * z4;
  // Estrin's scheme: dependent depth 4 instead of 10.  (Immediate constants on purpose: fetching them
  // from the constant bank measured slower in the loop kernels.)
  // sin(r) = r + r*z*S(z),  S = sum_{i<10} (-1)^(i+1) z^i / (2i+3)!
  const double a01 = fma(1.0 / 120.0, z, -1.0 / 6.0);
  const double a23 = fma(1.0 / 362880.0, z, -1.0 / 5040.0);
  const double a45 = fma(1.0 / 6227020800.0, z, -1.0 / 39916800.0);
  const double a67 = fma(1.0 / 355687428096000.0, z, -1.0 / 1307674368000.0);
  const double a89 = fma(1.0 / 51090942171709440000.0, z, -1.0 / 121645100408832000.0);
  const double S = fma(a89, z8, fma(fma(a67, z2, a45), z4, fma(a23, z2, a01)));
  const double sr = fma(r * z, S, r);
  // cos(r) = 1 - z/2 + z^2*C(z),  C = sum_{i<10} (-1)^i z^i / (2i+4)!
  const double d01 = fma(-1.0 / 720.0, z, 1.0 / 24.0);
  const double d23 = fma(-1.0 / 3628800.0, z, 1.0 / 40320.0);
  const double d45 = fma(-1.0 / 87178291200.0, z, 1.0 / 479001600.0);
  const double d67 = fma(-1.0 / 6402373705728000.0, z, 1.0 / 20922789888000.0);
  const double d89 = fma(-1.0 / 1124000727777607680000.0, z, 1.0 / 2432902008176640000.0);
  const double Cc = fma(d89, z8, fma(fma(d67, z2, d45), z4, fma(d23, z2, d01)));
  const double hz = 0.5 * z;
  const double w = 1.0 - hz;
  const double cr = w + (((1.0 - w) - hz) + z2 * Cc);     // compensated 1 - z/2 + z^2*C
  const int q = (int)k;
  const double s0 = (q & 1) ? cr : sr;
  const double c0 = (q & 1) ? sr : cr;
  *sn = (q & 2) ? -s0 : s0;
  *cs = ((q + 1) & 2) ? -c0 : c0;
}
// The same function for the serial loop kernels, where it sits on the loop-carried dependency chain (one warp per
// scheduler, nothing to hide latency behind): the 26 fp64 constants are loaded ONCE into registers through an opaque
// asm (otherwise ptxas rematerialises each as two 32-bit immediates per use: ~50 extra issue slots per call), and the
// quadrant fix-up is four FSELs plus a sign-bit XOR instead of fp64 negations.  Same operations in the same order as
// sincos_fast_f64 on the value path, so the results are bit-identical to it.
struct SinCosK {
  double two_over_pi, p1, p2, p3;
  double s[10], c[10];
  double half, one;
};
// constant table: [0..3] 2/pi and the three Cody-Waite pieces of pi/2, [4..13] sin coefficients, [14..23] cos
// coefficients, [24] 0.5, [25] 1.0
static __constant__ double kSinCosTab[26] = {
    0.63661977236758134308, 1.5707963267948966e+00, 6.123233995736766e-17, -1.4973849048591698e-33,
    -1.0 / 6.0, 1.0 / 120.0, -1.0 / 5040.0, 1.0 / 362880.0, -1.0 / 39916800.0, 1.0 / 6227020800.0,
    -1.0 / 1307674368000.0, 1.0 / 355687428096000.0, -1.0 / 121645100408832000.0, 1.0 / 51090942171709440000.0,
    1.0 / 24.0, -1.0 / 720.0, 1.0 / 40320.0, -1.0 / 3628800.0, 1.0 / 479001600.0, -1.0 / 87178291200.0,
    1.0 / 20922789888000.0, -1.0 / 6402373705728000.0, 1.0 / 2432902008176640000.0, -1.0 / 1124000727777607680000.0,
    0.5, 1.0};
static __constant__ double kSinCosMagic = 6755399441055744.0;   // 1.5 * 2^52: x + magic rounds x to an integer
// a volatile load ptxas can neither fold nor re-execute: the value has to stay in a register pair
__device__ __forceinline__ double ld_const_pinned(const double* p) {
  double v;
  asm volatile("ld.const.f64 %0, [%1];" : "=d"(v) : "l"(__cvta_generic_to_constant(p)));
  return v;
}
__device__ __forceinline__ SinCosK sincos_load_consts() {
  SinCosK K;
  K.two_over_pi = ld_const_pinned(&kSinCosTab[0]);
  K.p1 = ld_const_pinned(&kSinCosTab[1]);
  K.p2 = ld_const_pinned(&kSinCosTab[2]);
  K.p3 = ld_const_pinned(&kSinCosTab[3]);
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    K.s[i] = ld_const_pinned(&kSinCosTab[4 + i]);
    K.c[i] = ld_const_pinned(&kSinCosTab[14 + i]);
  }
  K.half = ld_const_pinned(&kSinCosTab[24]);
  K.one = ld_const_pinned(&kSinCosTab[25]);
  return K;
}
__device__ __forceinline__ void sincos_fast_f64_k(double x, const SinCosK& K, double* sn, double* cs) {
  const double k = rint(x * K.two_over_pi);
  const int q = (int)k;                                   // off the value path: only the final selects use it
  double r = fma(-k, K.p1, x);
  r = fma(-k, K.p2, r);
  r = fma(-k, K.p3, r);
  const double z = r * r, z2 = z * z, z4 = z2 * z2, z8 = z4 * z4;
  const double a01 = fma(K.s[1], z, K.s[0]);
  const double a23 = fma(K.s[3], z, K.s[2]);
  const double a45 = fma(K.s[5], z, K.s[4]);
  const double a67 = fma(K.s[7], z, K.s[6]);
  const double a89 = fma(K.s[9], z, K.s[8]);
  const double S = fma(a89, z8, fma(fma(a67, z2, a45), z4, fma(a23, z2, a01)));
  const double sr = fma(r * z, S, r);
  const double d01 = fma(K.c[1], z, K.c[0]);
  const double d23 = fma(K.c[3], z, K.c[2]);
  const double d45 = fma(K.c[5], z, K.c[4]);
  const double d67 = fma(K.c[7], z, K.c[6]);
  const double d89 = fma(K.c[9], z, K.c[8]);
  const double Cc = fma(d89, z8, fma(fma(d67, z2, d45), z4, fma(d23, z2, d01)));
  const double hz = K.half * z;
  const double w = K.one - hz;
  const double cr = w + (((K.one - w) - hz) + z2 * Cc);
  const bool swap = (q & 1) != 0;
  const unsigned s_flip = ((unsigned)q & 2u) << 30;        // sign bit when quadrant 2 or 3
  const unsigned c_flip = ((unsigned)(q + 1) & 2u) << 30;  // sign bit when quadrant 1 or 2
  const int sr_hi = __double2hiint(sr), sr_lo = __double2loint(sr);
  const int cr_hi = __double2hiint(cr), cr_lo = __double2loint(cr);
  const int s_hi = (swap ? cr_hi : sr_hi) ^ (int)s_flip, s_lo = swap ? cr_lo : sr_lo;
  const int c_hi = (swap ? sr_hi : cr_hi) ^ (int)c_flip, c_lo = swap ? sr_lo : cr_lo;
  *sn = __hiloint2double(s_hi, s_lo);
  *cs = __hiloint2double(c_hi, c_lo);
}
// fp64 sin/cos of an fp32 ARGUMENT (the FLL's MathF.Sin/Cos(phase)), shortened on the dependency chain:
//   * k = round(x*2/pi) by the 1.5*2^52 magic-number add (one DFMA + one DADD instead of DMUL + FRND.F64), the
//     quadrant read from the low word of the same sum (no F2I);
//   * two Cody-Waite pieces (the third, k*1.5e-33, is below half an ulp of r for every fp32 x != 0: r cannot come
//     closer than ~1e-9 to a multiple of pi/2);
//   * eight Taylor coefficients per polynomial (the z^8, z^9 terms are below 2^-56 of the sum for |r| <= pi/4):
//     Estrin depth 3 instead of 4;  cos tail folded into one DFMA (exact: the compensation term is a multiple of
//     the product's ulp).
// Checked on the host (fma(), -ffp-contract=off) against sincos_fast_f64 for EVERY fp32 argument with |x| < 64:
// bit-identical fp64 results (tools/sincos_check.cpp), so it is a drop-in on the FLL value path.
struct SinCosF {
  double two_over_pi, magic, p1, p2;
  double s[8], c[8];
  double half, one;
};
static __device__ double kSinCosTabF[22] = {
    0.63661977236758134308, 6755399441055744.0, 1.5707963267948966e+00, 6.123233995736766e-17,
    -1.0 / 6.0, 1.0 / 120.0, -1.0 / 5040.0, 1.0 / 362880.0, -1.0 / 39916800.0, 1.0 / 6227020800.0,
    -1.0 / 1307674368000.0, 1.0 / 355687428096000.0,
    1.0 / 24.0, -1.0 / 720.0, 1.0 / 40320.0, -1.0 / 3628800.0, 1.0 / 479001600.0, -1.0 / 87178291200.0,
    1.0 / 20922789888000.0, -1.0 / 6402373705728000.0,
    0.5, 1.0};
// global-memory load ptxas cannot rematerialise (constant-bank loads it re-issues on every use): the value stays in
// a register pair for the life of the kernel
__device__ __forceinline__ double ld_global_pinned(const double* p) {
  double v;
  asm volatile("ld.volatile.global.f64 %0, [%1];" : "=d"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ SinCosF sincos_f_load_consts() {
  SinCosF K;
  K.two_over_pi = ld_global_pinned(&kSinCosTabF[0]);
  K.magic = ld_global_pinned(&kSinCosTabF[1]);
  K.p1 = ld_global_pinned(&kSinCosTabF[2]);
  K.p2 = ld_global_pinned(&kSinCosTabF[3]);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    K.s[i] = ld_global_pinned(&kSinCosTabF[4 + i]);
    K.c[i] = ld_global_pinned(&kSinCosTabF[12 + i]);
  }
  K.half = ld_global_pinned(&kSinCosTabF[20]);
  K.one = ld_global_pinned(&kSinCosTabF[21]);
  return K;
}
__device__ __forceinline__ void sincos_f32arg_k(float xf, const SinCosF& K, float* sn, float* cs) {
  const double x = (double)xf;
  const double t = fma(x, K.two_over_pi, K.magic);
  const double k = t - K.magic;
  const unsigned q = (unsigned)__double2loint(t);          // k mod 2^32 (two's complement)
  double r = fma(-k, K.p1, x);
  r = fma(-k, K.p2, r);
  const double z = r * r, z2 = z * z, z4 = z2 * z2;
  const double a01 = fma(K.s[1], z, K.s[0]);
  const double a23 = fma(K.s[3], z, K.s[2]);
  const double a45 = fma(K.s[5], z, K.s[4]);
  const double a67 = fma(K.s[7], z, K.s[6]);
  const double S = fma(fma(a67, z2, a45), z4, fma(a23, z2, a01));
  const double sr = fma(r * z, S, r);
  const double d01 = fma(K.c[1], z, K.c[0]);
  const double d23 = fma(K.c[3], z, K.c[2]);
  const double d45 = fma(K.c[5], z, K.c[4]);
  const double d67 = fma(K.c[7], z, K.c[6]);
  const double Cc = fma(fma(d67, z2, d45), z4, fma(d23, z2, d01));
  const double hz = K.half * z;
  const double w = K.one - hz;
  const double cr = w + fma(z2, Cc, (K.one - w) - hz);
  const bool swap = (q & 1u) != 0;
  const unsigned s_flip = (q & 2u) << 30;                   // sign bit when quadrant 2 or 3
  const unsigned c_flip = ((q + 1u) & 2u) << 30;            // sign bit when quadrant 1 or 2
  const int sr_hi = __double2hiint(sr), sr_lo = __double2loint(sr);
  const int cr_hi = __double2hiint(cr), cr_lo = __double2loint(cr);
  const int s_hi = (swap ? cr_hi : sr_hi) ^ (int)s_flip, s_lo = swap ? cr_lo : sr_lo;
  const int c_hi = (swap ? sr_hi : cr_hi) ^ (int)c_flip, c_lo = swap ? sr_lo : cr_lo;
  *sn = (float)__hiloint2double(s_hi, s_lo);
  *cs = (float)__hiloint2double(c_hi, c_lo);
}
// The same value path with the quadrant fix-up left to the caller: phi = r + q*pi/2, returns (float)sin(r),
// (float)cos(r) and q mod 2^32.  e^{j phi} = e^{j r} * j^q, and multiplying the INPUT sample by j^q is an exact
// swap / sign flip that does not wait for the polynomials (see fll_duo.cu), so the selects and sign XORs of
// sincos_f32arg_k leave the dependency chain.  x is (double)phase, converted by the caller.
__device__ __forceinline__ void sincos_f32arg_rq(double x, const SinCosF& K, float* sr_out, float* cr_out, unsigned* q_out) {
  const double t = fma(x, K.two_over_pi, K.magic);
  const double k = t - K.magic;
  *q_out = (unsigned)__double2loint(t);
  double r = fma(-k, K.p1, x);
  r = fma(-k, K.p2, r);
  const double z = r * r, z2 = z * z, z4 = z2 * z2;
  const double a01 = fma(K.s[1], z, K.s[0]);
  const double a23 = fma(K.s[3], z, K.s[2]);
  const double a45 = fma(K.s[5], z, K.s[4]);
  const double a67 = fma(K.s[7], z, K.s[6]);
  const double S = fma(fma(a67, z2, a45), z4, fma(a23, z2, a01));
  const double sr = fma(r * z, S, r);
  const double d01 = fma(K.c[1], z, K.c[0]);
  const double d23 = fma(K.c[3], z, K.c[2]);
  const double d45 = fma(K.c[5], z, K.c[4]);
  const double d67 = fma(K.c[7], z, K.c[6]);
  const double Cc = fma(fma(d67, z2, d45), z4, fma(d23, z2, d01));
  const double hz = K.half * z;
  const double w = K.one - hz;
  const double cr = w + fma(z2, Cc, (K.one - w) - hz);
  *sr_out = (float)sr;
  *cr_out = (float)cr;
}
// fp64 argument, reduced pair + quadrant, for the Costas step (|theta| <= pi + |step|): the chain-shortening of
// sincos_f32arg_rq (magic-number quadrant, two Cody-Waite pieces, 8 coefficients — the first dropped terms are
// r z^9/19! and z^9/18!, below 1e-19 of the result for |r| <= pi/4 — and the cos tail in one DFMA) on the constants
// of SinCosK.  Against sincos_fast_f64_k the value can differ in the last bit only where x*2/pi lies within an ulp
// of a half-integer (the quadrant may then be the neighbour's: an equally valid reduction) — the Costas tests pin
// bits exactly and loop state to 1e-5.
__device__ __forceinline__ void sincos_rq_f64_k(double x, const SinCosK& K, double magic, double* sr_out, double* cr_out,
                                                unsigned* q_out) {
  const double t = fma(x, K.two_over_pi, magic);
  const double k = t - magic;
  *q_out = (unsigned)__double2loint(t);
  double r = fma(-k, K.p1, x);
  r = fma(-k, K.p2, r);
  const double z = r * r, z2 = z * z, z4 = z2 * z2;
  const double a01 = fma(K.s[1], z, K.s[0]);
  const double a23 = fma(K.s[3], z, K.s[2]);
  const double a45 = fma(K.s[5], z, K.s[4]);
  const double a67 = fma(K.s[7], z, K.s[6]);
  const double S = fma(fma(a67, z2, a45), z4, fma(a23, z2, a01));
  *sr_out = fma(r * z, S, r);
  const double d01 = fma(K.c[1], z, K.c[0]);
  const double d23 = fma(K.c[3], z, K.c[2]);
  const double d45 = fma(K.c[5], z, K.c[4]);
  const double d67 = fma(K.c[7], z, K.c[6]);
  const double Cc = fma(fma(d67, z2, d45), z4, fma(d23, z2, d01));
  const double hz = K.half * z;
  const double w = K.one - hz;
  *cr_out = w + fma(z2, Cc, (K.one - w) - hz);
}
#endif

}  // namespace qpsk
