// soft.cuh — the int8 soft values of one QPSK symbol, rule 1 of the convolutional-code section of include/qpskcuda.h.
// The Viterbi decoder (fec.cu) and the frame synchronizer (fsync.cu) read the same values from the same code.
#pragma once
#include <cuda_runtime.h>

namespace qpsk {

// q(v) = clamp(rint_half_even(v), -127, 127); NaN -> 0 (cvt.rni.s32.f32 saturates and maps NaN to 0)
__device__ __forceinline__ int vit_q(float v) { return max(-127, min(127, __float2int_rn(v))); }

// coherent: (s0, s1) = (q(scale I), q(scale Q))
__device__ __forceinline__ int2 soft_coherent(float2 y, float scale) {
  return make_int2(vit_q(__fmul_rn(scale, y.x)), vit_q(__fmul_rn(scale, y.y)));
}

// differential, y against the previous symbol p: z = y conj(p), s0 = q(-(scale (re + im))), s1 = q(scale (im - re))
__device__ __forceinline__ int2 soft_differential(float2 y, float2 p, float scale) {
  const float re = __fadd_rn(__fmul_rn(y.x, p.x), __fmul_rn(y.y, p.y));
  const float im = __fsub_rn(__fmul_rn(y.y, p.x), __fmul_rn(y.x, p.y));
  return make_int2(vit_q(-__fmul_rn(scale, __fadd_rn(re, im))), vit_q(__fmul_rn(scale, __fsub_rn(im, re))));
}

}  // namespace qpsk
