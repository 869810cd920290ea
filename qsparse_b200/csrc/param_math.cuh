// Scalar parameter updates of the quantize / prune callbacks, shared by the tiny
// parameter kernels (params.cu) and the row-resident fused kernel (rowquant.cu).
#pragma once
#include <math.h>

#include "qsb_common.cuh"

namespace qsb {

// new = absmax / 2^(bits-1); EMA with a host step counter.
// ref qsparse/quantize.py:340,344-348
__device__ __forceinline__ float scale_ema_step(float w, float absmax,
                                                float limit, int64_t t) {
  const float nw = __fdiv_rn(absmax, limit);
  if (t == 0) return nw;
  return __fdiv_rn(__fadd_rn(__fmul_rn((float)t, w), nw), (float)(t + 1));
}

// d = round(log2(nan_to_num(1 / s, posinf=1, neginf=1)))
// ref qsparse/quantize.py:316.  log2 is evaluated in fp64 and rounded to fp32,
// i.e. the correctly rounded fp32 log2, then rint (half to even).
__device__ __forceinline__ float scale_to_decimal(float s) {
  float r = __fdiv_rn(1.0f, s);
  if (r != r) r = 0.0f;
  else if (isinf(r)) r = 1.0f;
  const float l = (float)log2((double)r);
  return rintf(l);
}

// What a PRUNED channel with max|x| bits `b` adds to the abs-max of `x * mask` (ref sparse.py:66,
// quantize.py:329-340): |x * 0| is 0 for finite x, but inf * 0 and NaN * 0 are NaN, which the max keeps.
__device__ __forceinline__ uint32_t pruned_max_bits(uint32_t b) {
  return b >= 0x7f800000u ? 0x7fffffffu : 0u;
}

// mag = (t * mag + m) / (t + 1)      ref qsparse/sparse.py:89
__device__ __forceinline__ float magnitude_ema_step(float mag, float m,
                                                    int64_t t) {
  return __fdiv_rn(__fadd_rn(__fmul_rn((float)t, mag), m), (float)(t + 1));
}

// full-size magnitude EMA  mag = (t * mag + |x|) / (t + 1)   ref qsparse/sparse.py:85-89
// (t_f = float(t), tp1 = float(t + 1), rcp = RN(1 / tp1) computed on the host)
__device__ __forceinline__ float ema_full_step(float mag, float x, float t_f, float tp1, float rcp) {
  return div_rn_by(__fadd_rn(__fmul_rn(t_f, mag), fabsf(x)), tp1, rcp, true);
}

// lines = (w * (t - 1) + new) / t     ref qsparse/quantize.py:428-430
__device__ __forceinline__ float lines_ema_step(float w, float nw, float tm1, float t) {
  return __fdiv_rn(__fadd_rn(__fmul_rn(w, tm1), nw), t);
}

}  // namespace qsb
