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

// What channel c of `x * mask` adds to the (min, max) of the line quantizer's statistics (ref sparse.py:66,
// quantize.py:396-418), from the channel's own min / max of x (both NaN when it holds a NaN).  A kept channel adds
// them unchanged.  A pruned one adds min / max over x * 0: NaN when it holds an inf or a NaN (inf * 0, NaN * 0),
// otherwise only zeros, each carrying the sign of its x.  min / max (fminf / fmaxf, the FMNMX instruction) order
// -0 below +0, so the reduction over those zeros gives -0 for the min iff some x has its sign bit set — iff the
// channel's own min does — and +0 for the max iff some x has it clear — iff the channel's own max does.  The
// signs are then exactly what reduce_stats(minmax) computes on the fp32 output of mask_apply, whatever its order.
__device__ __forceinline__ void masked_line(bool keep, float mn, float mx, float &lo, float &hi) {
  if (keep) {
    lo = mn, hi = mx;
  } else if (mn != mn || isinf(mn) || isinf(mx)) {
    lo = hi = __uint_as_float(0x7fc00000u);
  } else {
    lo = signbit(mn) ? -0.0f : 0.0f;
    hi = signbit(mx) ? -0.0f : 0.0f;
  }
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
