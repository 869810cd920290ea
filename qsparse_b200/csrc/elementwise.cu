// K1 / K2 / K6 / K7 and the full-size EMA: every elementwise op of the
// quantize/prune hot path, as Op functors over the streaming map kernel.
//
// Arithmetic is written with explicit round-to-nearest intrinsics so that no
// FMA contraction can happen (the reference rounds after every ATen op).
#include <math.h>

#include <vector>

#include "fq_ops.cuh"
#include "map_kernel.cuh"
#include "reduce_internal.cuh"
namespace qsb {
void set_select_fast(int v);
}

namespace qsb {

template <class Op, class IO>
int launch_map_big_out(const Op &op, const IO &io, const Layout &L, cudaStream_t stream) {
  if (L.numel() * 4 >= kStreamStoreBytes) return launch_map<Op, Hint::STREAM, Hint::STREAM>(op, io, L, stream);
  return launch_map<Op, Hint::STREAM, Hint::KEEP>(op, io, L, stream);
}

int &map_reverse_tiles() {
  static int v = 1;
  return v;
}

// ---------------------------------------------------------------------------
// K2  STE backward (+ fused prune backward)   ref qsparse/quantize.py:65-77
// ---------------------------------------------------------------------------
template <int MASK, bool WRITE_GC, bool WRITE_GX>
struct SteOp {
  static constexpr bool kIn1 = false, kInB = (MASK == QSB_MASK_ELEMENT),
                        kOut0 = WRITE_GC, kOut1 = WRITE_GX, kOutB = false,
                        kCanSkip = false,
                        kHasFast = false;  // v * 0 keeps the sign of v
  const float *scale;
  int scale_stride;
  float scale_host;  // already 2^-d when the host decimal is used
  bool is_decimal;   // device values are decimals: s = 2^-d
  float n_lo, n_hi;  // (-L + notch), (L - 1 + notch) as fp32
  const uint8_t *cmask;
  struct P {
    float lo, hi, m;
    bool zero_bound;  // a bound is +-0 (1-bit layers, a zero scale): the sign of a zero result matters
  };
  __device__ __forceinline__ P params(int32_t c) const {
    float s = scale_host;
    if (scale) {
      s = __ldg(scale + (int64_t)c * scale_stride);
      if (is_decimal) s = pow2f_exact(-s);
    }
    P p;
    p.lo = __fmul_rn(n_lo, s);
    p.hi = __fmul_rn(n_hi, s);
    p.zero_bound = p.lo == 0.0f || p.hi == 0.0f;
    p.m = 1.0f;
    if constexpr (MASK == QSB_MASK_CHANNEL) p.m = __ldg(cmask + c) ? 1.0f : 0.0f;
    return p;
  }
  __device__ __forceinline__ bool skip(const P &) const { return false; }
  __device__ __forceinline__ void apply(float g, float, uint8_t mb, const P &p,
                                        float &o0, float &o1, uint8_t &) const {
    // (:72-75) clamp with tensor bounds: NaN in g or in a bound gives NaN — exactly what the
    // NaN-propagating FMNMX pair computes, in 2 instructions instead of 7.  FMNMX orders -0 < +0
    // while torch's clamp keeps g when g == bound, so a zero bound takes the compare/select form.
    float v = p.zero_bound ? clamp_torch_tensor(g, p.lo, p.hi) : clamp_fmnmx_nan(g, p.lo, p.hi);
    if (v != v) v = 0.0f;                         // (:76) fires only for NaN
    o0 = v;
    if constexpr (MASK == QSB_MASK_CHANNEL)
      o1 = __fmul_rn(v, p.m);
    else if constexpr (MASK == QSB_MASK_ELEMENT)
      o1 = mask_mul(v, mb != 0);
    else
      o1 = v;
  }
};

// ---------------------------------------------------------------------------
// K6  mask apply   ref qsparse/sparse.py:66,116,122,263
// ---------------------------------------------------------------------------
template <int MASK>
struct MaskApplyOp {
  static constexpr bool kIn1 = false, kInB = (MASK == QSB_MASK_ELEMENT),
                        kOut0 = true, kOut1 = false, kOutB = false,
                        kCanSkip = false,
                        kHasFast = false;  // x * 0 keeps the sign of x
  const uint8_t *cmask;
  struct P {
    float m;
  };
  __device__ __forceinline__ P params(int32_t c) const {
    P p;
    p.m = 1.0f;
    if constexpr (MASK == QSB_MASK_CHANNEL) p.m = __ldg(cmask + c) ? 1.0f : 0.0f;
    return p;
  }
  __device__ __forceinline__ bool skip(const P &) const { return false; }
  __device__ __forceinline__ void apply(float a, float, uint8_t mb, const P &p,
                                        float &o0, float &, uint8_t &) const {
    if constexpr (MASK == QSB_MASK_ELEMENT)
      o0 = mask_mul(a, mb != 0);
    else
      o0 = __fmul_rn(a, p.m);
  }
};

// mask = importance >= threshold (+ optional y = x * mask)
// ref qsparse/util.py:117, qsparse/sparse.py:65-66
template <bool APPLY>
struct MaskBuildOp {
  static constexpr bool kIn1 = APPLY, kInB = false, kOut0 = APPLY,
                        kOut1 = false, kOutB = true, kCanSkip = false,
                        kHasFast = false;
  const float *thr;
  bool take_abs;
  __device__ __forceinline__ void bind(const float *aux) { thr = aux; }  // multi-tensor: per layer
  struct P {
    float thr;
  };
  __device__ __forceinline__ P params(int32_t) const {
    P p;
    p.thr = __ldg(thr);
    return p;
  }
  __device__ __forceinline__ bool skip(const P &) const { return false; }
  __device__ __forceinline__ void apply(float imp, float x, uint8_t, const P &p,
                                        float &o0, float &, uint8_t &ob) const {
    if (take_abs) imp = fabsf(imp);
    const bool keep = imp >= p.thr;  // false for NaN on either side
    ob = keep ? 1 : 0;
    if constexpr (APPLY) o0 = mask_mul(x, keep);
  }
};

// full-size magnitude EMA   ref qsparse/sparse.py:85-89
//   mag = (t * mag + |x|) / (t + 1)
struct EmaFullOp {
  static constexpr bool kIn1 = true, kInB = false, kOut0 = true, kOut1 = false,
                        kOutB = false, kCanSkip = false,
                        kHasFast = false;
  const float *tensor_min;  // device scalar, only read when use_l0
  bool use_l0;
  float t_f, t_plus_1_f, r_t_plus_1;  // r = RN(1 / (t + 1)), host computed
  __device__ __forceinline__ void bind(const float *) {}
  struct P {
    bool indicator;
  };
  __device__ __forceinline__ P params(int32_t) const {
    P p;
    p.indicator = use_l0 && (__ldg(tensor_min) == 0.0f);
    return p;
  }
  __device__ __forceinline__ bool skip(const P &) const { return false; }
  __device__ __forceinline__ void apply(float x, float mag, uint8_t, const P &p,
                                        float &o0, float &, uint8_t &) const {
    const float ax = p.indicator ? (x != 0.0f ? 1.0f : 0.0f) : fabsf(x);
    o0 = div_rn_by(__fadd_rn(__fmul_rn(t_f, mag), ax), t_plus_1_f, r_t_plus_1, true);
  }
};

// ---------------------------------------------------------------------------
// integer export (SURVEY 8f-3): the integer CODE of the fake-quantizers, one byte per
// element instead of a float — 5 B/elem instead of 8.  Inside the representable range
// dequantising the code (q * 2^-d, q * s, q * step + lo) reproduces the fake-quant output
// bit for bit (the property tests/test_quantize.py:73-101 of the reference relies on).
// The parameter derivation is the fake-quant ops' own (Op::params).
// ---------------------------------------------------------------------------
struct ExportPow2Op : Pow2Op<QSB_MASK_NONE> {
  static constexpr bool kOut0 = false, kOutB = true, kCanSkip = false;
  int q_min, q_max;
  __device__ __forceinline__ void apply(float a, float, uint8_t, const P &p, float &, float &,
                                        uint8_t &ob) const {
    int q = __float2int_rz(__fmul_rn(a, p.toi));
    q = q < q_min ? q_min : (q > q_max ? q_max : q);
    ob = (uint8_t)(int8_t)q;
  }
};

struct ExportScalerOp : ScalerOp<QSB_MASK_NONE> {
  static constexpr bool kOut0 = false, kOutB = true, kCanSkip = false, kHasFast = false;
  int q_min, q_max;
  __device__ __forceinline__ void apply(float a, float, uint8_t, const P &p, float &, float &,
                                        uint8_t &ob) const {
    int q = __float2int_rn(div_rn_by_q(a, p.s, p.r, p.ok));
    q = q < q_min ? q_min : (q > q_max ? q_max : q);
    ob = (uint8_t)(int8_t)q;
  }
};

struct ExportLineOp : LineOp<QSB_MASK_NONE, true> {
  static constexpr bool kOut0 = false, kOutB = true, kCanSkip = false, kHasFast = false;
  __device__ __forceinline__ void apply(float a, float, uint8_t, const P &p, float &, float &,
                                        uint8_t &ob) const {
    const float xc = clamp_torch_tensor(a, p.lo, p.hi);
    const float d = __fsub_rn(xc, p.lo);
    float q = p.fast ? div_rn_by_unchecked(d, p.step, p.rstep) : __fdiv_rn(d, p.step);
    q = clamp_torch(rintf(q), 0.0f, q_max);
    ob = (uint8_t)__float2int_rn(q);  // NaN -> 0
  }
};

// The same codes packed two per byte on the streaming-map skeleton (window parameter tables, one CTA per
// tile, 256-bit loads, one 32-bit store per 8 codes): what qsb_quant_export_int4 launches for 32-byte
// aligned tensors whose size is a multiple of 8.
struct ExportPow2Op4 : ExportPow2Op {
  static constexpr bool kPack4 = true;
};
struct ExportScalerOp4 : ExportScalerOp {
  static constexpr bool kPack4 = true;
};
struct ExportLineOp4 : ExportLineOp {
  static constexpr bool kPack4 = true;
};

// Packed 4-bit export: two codes per byte (even element in the low nibble), 4.5 B/elem.  A
// thread owns 8 consecutive elements = one 32-bit store; it walks the channel of its elements
// itself (one 64-bit division per thread), so every [outer, C, inner] layout takes this one
// kernel.  The per-element arithmetic is the int8 export ops' own apply().
template <class Op>
__global__ void __launch_bounds__(QSB_THREADS)
    export_pack4_kernel(Op op, const float *__restrict__ x, uint8_t *__restrict__ out, int64_t n,
                        int64_t inner, int64_t channels, int vec_ok) {
  pdl_wait();
  pdl_trigger();
  constexpr int U = 2;  // vectors per thread, QSB_THREADS * 8 elements apart: both loads in flight
  const int64_t t0 = (int64_t)blockIdx.x * (QSB_THREADS * 8 * U) + threadIdx.x * 8;
  float v[U][8];
  int cnt[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t e0 = t0 + (int64_t)u * (QSB_THREADS * 8);
    cnt[u] = e0 >= n ? 0 : ((n - e0 < 8) ? (int)(n - e0) : 8);
    if (cnt[u] == 8 && vec_ok) {
      const VecF<8> a = ld_vec<8, Hint::STREAM>(x + e0);
#pragma unroll
      for (int j = 0; j < 8; ++j) v[u][j] = a.v[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[u][j] = j < cnt[u] ? x[e0 + j] : 0.f;
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (cnt[u] == 0) continue;
    const int64_t e0 = t0 + (int64_t)u * (QSB_THREADS * 8);
    int64_t col, c;
    if (n <= 0xffffffffLL) {  // 32-bit divisions when they are enough
      const uint32_t row = (uint32_t)e0 / (uint32_t)inner;
      col = (uint32_t)e0 - row * (uint32_t)inner;
      c = row % (uint32_t)channels;
    } else {
      const int64_t row = e0 / inner;
      col = e0 - row * inner;
      c = row % channels;
    }
    typename Op::P p = op.params((int32_t)c);
    uint32_t word = 0;
    if (inner - col >= 8) {  // the whole vector in one row: one set of parameters
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float o0, o1;
        uint8_t ob = 0;
        if (j < cnt[u]) op.apply(v[u][j], 0.f, (uint8_t)1, p, o0, o1, ob);
        word |= (uint32_t)(ob & 0xF) << (4 * j);
      }
    } else {  // walk the rows (kept rolled: the parameter derivation must not be replicated 8 times)
#pragma unroll 1
      for (int j = 0; j < cnt[u]; ++j) {
        float o0, o1;
        uint8_t ob = 0;
        float vj = v[u][0];
#pragma unroll
        for (int k = 1; k < 8; ++k) vj = (j == k) ? v[u][k] : vj;
        op.apply(vj, 0.f, (uint8_t)1, p, o0, o1, ob);
        word |= (uint32_t)(ob & 0xF) << (4 * j);
        if (++col == inner) {
          col = 0;
          c = (c + 1 == channels) ? 0 : c + 1;
          p = op.params((int32_t)c);
        }
      }
    }
    uint8_t *o = out + (e0 >> 1);
    if (cnt[u] == 8 && (reinterpret_cast<uintptr_t>(o) & 3) == 0) {
      *reinterpret_cast<uint32_t *>(o) = word;
    } else {
      for (int b2 = 0; b2 < (cnt[u] + 1) / 2; ++b2) o[b2] = (uint8_t)(word >> (8 * b2));
    }
  }
}

}  // namespace qsb

// ===========================================================================
// C-ABI
// ===========================================================================
using namespace qsb;

namespace {

int check_layout(int64_t outer, int64_t channels, int64_t inner) {
  if (outer < 0 || channels < 0 || inner < 0) return QSB_E_BADARG;
  return 0;
}

// n: elements of the tensor — an empty tensor (and its empty mask) has no storage, a null pointer is fine
int check_mask(const uint8_t *mask, int kind, int64_t n) {
  if (kind != QSB_MASK_NONE && kind != QSB_MASK_CHANNEL &&
      kind != QSB_MASK_ELEMENT)
    return QSB_E_BADARG;
  if (kind != QSB_MASK_NONE && !mask && n != 0) return QSB_E_BADARG;
  return 0;
}

// An element mask addresses the tensor flat, so the op itself only needs the
// channel structure when its own parameters are per channel.
template <class F>
int dispatch_mask(int kind, F &&f) {
  switch (kind) {
    case QSB_MASK_NONE:
      return f(std::integral_constant<int, QSB_MASK_NONE>{});
    case QSB_MASK_CHANNEL:
      return f(std::integral_constant<int, QSB_MASK_CHANNEL>{});
    default:
      return f(std::integral_constant<int, QSB_MASK_ELEMENT>{});
  }
}

// n_param must be 1 or `channels`; returns the stride (0 / 1) or -1.
int param_stride(int64_t n_param, int64_t channels) {
  if (n_param == 1) return 0;
  if (n_param == channels) return 1;
  return -1;
}

// When neither the parameters nor the mask are per channel the tensor is
// processed flat (no channel arithmetic in the kernel).
Layout effective_layout(int64_t outer, int64_t channels, int64_t inner,
                        bool per_channel) {
  if (per_channel) return Layout{outer, channels, inner};
  return Layout{1, 1, outer * channels * inner};
}

}  // namespace

extern "C" int qsb_fq_pow2_fwd_dt(const void *x_, int x_dtype, float *y,
                                  const float *decimal_dev, int64_t n_decimal,
                                  double decimal_host, const uint8_t *mask_dev,
                                  int mask_kind, int64_t outer, int64_t channels,
                                  int64_t inner, void *stream) {
  if (!dtype_ok(x_dtype)) return QSB_E_BADARG;
  if (int e = check_layout(outer, channels, inner)) return e;
  if (int e = check_mask(mask_dev, mask_kind, outer * channels * inner)) return e;
  if (outer * channels * inner == 0) return 0;
  if (!x_ || !y) return QSB_E_BADARG;
  int stride = 0;
  if (decimal_dev) {
    stride = param_stride(n_decimal, channels);
    if (stride < 0) return QSB_E_BADARG;
  }
  const bool per_channel = stride == 1 || mask_kind == QSB_MASK_CHANNEL;
  const Layout L = effective_layout(outer, channels, inner, per_channel);
  // Python: toi = 2.0**decimal (double) then cast to the tensor dtype.
  const float toi = (float)pow(2.0, decimal_host);
  const float tof = (float)pow(2.0, -decimal_host);
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    MapIOT<T> io{static_cast<const T *>(x_), nullptr, mask_kind == QSB_MASK_ELEMENT ? mask_dev : nullptr,
                 y, nullptr, nullptr};
    return dispatch_mask(mask_kind, [&](auto mk) {
      Pow2Op<decltype(mk)::value> op{decimal_dev, stride, toi, tof, mask_dev};
      return launch_map_big_out(op, io, L, (cudaStream_t)stream);
    });
  });
}

extern "C" int qsb_fq_pow2_fwd(const float *x, float *y, const float *decimal_dev, int64_t n_decimal,
                               double decimal_host, const uint8_t *mask_dev, int mask_kind, int64_t outer,
                               int64_t channels, int64_t inner, void *stream) {
  return qsb_fq_pow2_fwd_dt(x, QSB_DTYPE_F32, y, decimal_dev, n_decimal, decimal_host, mask_dev, mask_kind, outer,
                            channels, inner, stream);
}

extern "C" int qsb_fq_scaler_fwd_dt(const void *x_, int x_dtype, float *y,
                                    const float *scaler_dev, int64_t n_scaler,
                                    float scaler_host, const uint8_t *mask_dev,
                                    int mask_kind, int64_t outer, int64_t channels,
                                    int64_t inner, void *stream) {
  if (!dtype_ok(x_dtype)) return QSB_E_BADARG;
  if (int e = check_layout(outer, channels, inner)) return e;
  if (int e = check_mask(mask_dev, mask_kind, outer * channels * inner)) return e;
  if (outer * channels * inner == 0) return 0;
  if (!x_ || !y) return QSB_E_BADARG;
  int stride = 0;
  if (scaler_dev) {
    stride = param_stride(n_scaler, channels);
    if (stride < 0) return QSB_E_BADARG;
  }
  const bool per_channel = stride == 1 || mask_kind == QSB_MASK_CHANNEL;
  const Layout L = effective_layout(outer, channels, inner, per_channel);
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    MapIOT<T> io{static_cast<const T *>(x_), nullptr, mask_kind == QSB_MASK_ELEMENT ? mask_dev : nullptr,
                 y, nullptr, nullptr};
    return dispatch_mask(mask_kind, [&](auto mk) {
      ScalerOp<decltype(mk)::value> op{scaler_dev, stride, scaler_host, mask_dev};
      return launch_map_big_out(op, io, L, (cudaStream_t)stream);
    });
  });
}

extern "C" int qsb_fq_scaler_fwd(const float *x, float *y, const float *scaler_dev, int64_t n_scaler,
                                 float scaler_host, const uint8_t *mask_dev, int mask_kind, int64_t outer,
                                 int64_t channels, int64_t inner, void *stream) {
  return qsb_fq_scaler_fwd_dt(x, QSB_DTYPE_F32, y, scaler_dev, n_scaler, scaler_host, mask_dev, mask_kind, outer,
                              channels, inner, stream);
}

extern "C" int qsb_fq_line_fwd_dt(const void *x_, int x_dtype, float *y, const float *lines_dev,
                                  int64_t n_lines, float lo_host, float hi_host,
                                  int bits, int float_zero_point,
                                  const uint8_t *mask_dev, int mask_kind,
                                  int64_t outer, int64_t channels, int64_t inner,
                                  void *stream) {
  if (!dtype_ok(x_dtype)) return QSB_E_BADARG;
  if (int e = check_layout(outer, channels, inner)) return e;
  if (int e = check_mask(mask_dev, mask_kind, outer * channels * inner)) return e;
  if (bits < 0 || bits > 62) return QSB_E_BADARG;
  if (outer * channels * inner == 0) return 0;
  if (!x_ || !y) return QSB_E_BADARG;
  int stride = 0;
  if (lines_dev) {
    stride = param_stride(n_lines, channels);
    if (stride < 0) return QSB_E_BADARG;
    if (!aligned_to(lines_dev, 8)) return QSB_E_ALIGN;
  }
  const bool per_channel = stride == 1 || mask_kind == QSB_MASK_CHANNEL;
  const Layout L = effective_layout(outer, channels, inner, per_channel);
  const double N = ldexp(1.0, bits);
  const float n_levels = (float)N;
  const float q_max = (float)(N - 1.0);
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    MapIOT<T> io{static_cast<const T *>(x_), nullptr, mask_kind == QSB_MASK_ELEMENT ? mask_dev : nullptr,
                 y, nullptr, nullptr};
    return dispatch_mask(mask_kind, [&](auto mk) {
      constexpr int MK = decltype(mk)::value;
      if (float_zero_point) {
        LineOp<MK, true> op{lines_dev, stride, lo_host, hi_host,
                            n_levels,  q_max,  mask_dev};
        return launch_map<decltype(op), Hint::STREAM, Hint::KEEP>(
            op, io, L, (cudaStream_t)stream);
      } else {
        LineOp<MK, false> op{lines_dev, stride, lo_host, hi_host,
                             n_levels,  q_max,  mask_dev};
        return launch_map<decltype(op), Hint::STREAM, Hint::KEEP>(
            op, io, L, (cudaStream_t)stream);
      }
    });
  });
}

extern "C" int qsb_fq_line_fwd(const float *x, float *y, const float *lines_dev, int64_t n_lines, float lo_host,
                               float hi_host, int bits, int float_zero_point, const uint8_t *mask_dev,
                               int mask_kind, int64_t outer, int64_t channels, int64_t inner, void *stream) {
  return qsb_fq_line_fwd_dt(x, QSB_DTYPE_F32, y, lines_dev, n_lines, lo_host, hi_host, bits, float_zero_point,
                            mask_dev, mask_kind, outer, channels, inner, stream);
}

/* integer codes of the three fake-quantizers */
extern "C" int qsb_quant_export_int8(const float *x, uint8_t *q_out, int kind,
                                     const float *param_dev, int64_t n_param,
                                     double param_host, double param_host2, int bits,
                                     int64_t outer, int64_t channels, int64_t inner,
                                     void *stream) {
  if (int e = check_layout(outer, channels, inner)) return e;
  if (kind < 0 || kind > 2 || bits < 1 || bits > 8) return QSB_E_BADARG;
  if (outer * channels * inner == 0) return 0;
  if (!x || !q_out) return QSB_E_BADARG;
  int stride = 0;
  if (param_dev) {
    stride = param_stride(n_param, channels);
    if (stride < 0) return QSB_E_BADARG;
    if (kind == 2 && !aligned_to(param_dev, 8)) return QSB_E_ALIGN;
  }
  const Layout L = effective_layout(outer, channels, inner, stride == 1);
  MapIO io{x, nullptr, nullptr, nullptr, nullptr, q_out};
  const int q_min = -(1 << (bits - 1)), q_max = (1 << (bits - 1)) - 1;
  if (kind == 0) {
    ExportPow2Op op;
    op.dec = param_dev, op.dec_stride = stride;
    op.toi_host = (float)pow(2.0, param_host), op.tof_host = (float)pow(2.0, -param_host);
    op.cmask = nullptr, op.q_min = q_min, op.q_max = q_max;
    return launch_map<ExportPow2Op, Hint::STREAM, Hint::KEEP>(op, io, L, (cudaStream_t)stream);
  }
  if (kind == 1) {
    ExportScalerOp op;
    op.scale = param_dev, op.scale_stride = stride, op.scale_host = (float)param_host;
    op.cmask = nullptr, op.q_min = q_min, op.q_max = q_max;
    return launch_map<ExportScalerOp, Hint::STREAM, Hint::KEEP>(op, io, L, (cudaStream_t)stream);
  }
  ExportLineOp op;
  op.lines = param_dev, op.lines_stride = stride;
  op.lo_host = (float)param_host, op.hi_host = (float)param_host2;
  const double N = ldexp(1.0, bits);
  op.n_levels = (float)N, op.q_max = (float)(N - 1.0), op.cmask = nullptr;
  return launch_map<ExportLineOp, Hint::STREAM, Hint::KEEP>(op, io, L, (cudaStream_t)stream);
}

/* the same codes, two per byte */
extern "C" int qsb_quant_export_int4(const float *x, uint8_t *q_out, int kind,
                                     const float *param_dev, int64_t n_param,
                                     double param_host, double param_host2, int bits,
                                     int64_t outer, int64_t channels, int64_t inner,
                                     void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (int e = check_layout(outer, channels, inner)) return e;
  if (kind < 0 || kind > 2 || bits < 1 || bits > 4) return QSB_E_BADARG;
  const int64_t n = outer * channels * inner;
  if (n == 0) return 0;
  if (!x || !q_out) return QSB_E_BADARG;
  if (!aligned_to(x, 4)) return QSB_E_ALIGN;
  int stride = 0;
  if (param_dev) {
    stride = param_stride(n_param, channels);
    if (stride < 0) return QSB_E_BADARG;
    if (kind == 2 && !aligned_to(param_dev, 8)) return QSB_E_ALIGN;
  }
  const int q_min = -(1 << (bits - 1)), q_max = (1 << (bits - 1)) - 1;
  if (n % 8 == 0 && aligned_to(x, 32) && aligned_to(q_out, 4)) {
    // the streaming-map skeleton (0.67 -> see profiles/ of the copy peak with the generic kernel below)
    const Layout L = effective_layout(outer, channels, inner, stride == 1);
    MapIO io{x, nullptr, nullptr, nullptr, nullptr, q_out};
    if (kind == 0) {
      ExportPow2Op4 op;
      op.dec = param_dev, op.dec_stride = stride;
      op.toi_host = (float)pow(2.0, param_host), op.tof_host = (float)pow(2.0, -param_host);
      op.cmask = nullptr, op.q_min = q_min, op.q_max = q_max;
      return launch_map<ExportPow2Op4, Hint::STREAM, Hint::KEEP>(op, io, L, stream);
    }
    if (kind == 1) {
      ExportScalerOp4 op;
      op.scale = param_dev, op.scale_stride = stride, op.scale_host = (float)param_host;
      op.cmask = nullptr, op.q_min = q_min, op.q_max = q_max;
      return launch_map<ExportScalerOp4, Hint::STREAM, Hint::KEEP>(op, io, L, stream);
    }
    ExportLineOp4 op;
    op.lines = param_dev, op.lines_stride = stride;
    op.lo_host = (float)param_host, op.hi_host = (float)param_host2;
    const double N = ldexp(1.0, bits);
    op.n_levels = (float)N, op.q_max = (float)(N - 1.0), op.cmask = nullptr;
    return launch_map<ExportLineOp4, Hint::STREAM, Hint::KEEP>(op, io, L, stream);
  }
  const int64_t per_cta = (int64_t)QSB_THREADS * 8 * 2;  // two vectors per thread
  const dim3 grid((unsigned)((n + per_cta - 1) / per_cta));
  const int vec_ok = aligned_to(x, 32) ? 1 : 0;
  // per-tensor parameters: one channel of n elements, so the walk never reloads them
  const int64_t k_inner = stride ? inner : n, k_ch = stride ? channels : 1;
  if (kind == 0) {
    ExportPow2Op op;
    op.dec = param_dev, op.dec_stride = stride;
    op.toi_host = (float)pow(2.0, param_host), op.tof_host = (float)pow(2.0, -param_host);
    op.cmask = nullptr, op.q_min = q_min, op.q_max = q_max;
    QSB_CUDA_TRY(launch_k(export_pack4_kernel<ExportPow2Op>, grid, dim3(QSB_THREADS), 0, stream, op, x, q_out, n,
                          k_inner, k_ch, vec_ok));
  } else if (kind == 1) {
    ExportScalerOp op;
    op.scale = param_dev, op.scale_stride = stride, op.scale_host = (float)param_host;
    op.cmask = nullptr, op.q_min = q_min, op.q_max = q_max;
    QSB_CUDA_TRY(launch_k(export_pack4_kernel<ExportScalerOp>, grid, dim3(QSB_THREADS), 0, stream, op, x, q_out, n,
                          k_inner, k_ch, vec_ok));
  } else {
    ExportLineOp op;
    op.lines = param_dev, op.lines_stride = stride;
    op.lo_host = (float)param_host, op.hi_host = (float)param_host2;
    const double N = ldexp(1.0, bits);
    op.n_levels = (float)N, op.q_max = (float)(N - 1.0), op.cmask = nullptr;
    QSB_CUDA_TRY(launch_k(export_pack4_kernel<ExportLineOp>, grid, dim3(QSB_THREADS), 0, stream, op, x, q_out, n,
                          k_inner, k_ch, vec_ok));
  }
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_ste_bwd_dt(const float *g, float *g_clamped_out, void *gx_out, int gx_dtype,
                              const float *scale_dev, int64_t n_scale,
                              double scale_host, int scale_is_decimal, int bits,
                              int notch, const uint8_t *mask_dev, int mask_kind,
                              int64_t outer, int64_t channels, int64_t inner,
                              void *stream) {
  if (!dtype_ok(gx_dtype)) return QSB_E_BADARG;
  if (int e = check_layout(outer, channels, inner)) return e;
  if (int e = check_mask(mask_dev, mask_kind, outer * channels * inner)) return e;
  if (outer * channels * inner == 0) return 0;
  if (!g) return QSB_E_BADARG;
  if (!g_clamped_out && !gx_out) return QSB_E_BADARG;
  int stride = 0;
  if (scale_dev) {
    stride = param_stride(n_scale, channels);
    if (stride < 0) return QSB_E_BADARG;
  }
  const bool per_channel = stride == 1 || mask_kind == QSB_MASK_CHANNEL;
  const Layout L = effective_layout(outer, channels, inner, per_channel);
  // limit = torch.tensor(2.0 ** (bits - 1)) (fp32); the bounds are fp32 ops.
  const float limit = (float)pow(2.0, (double)bits - 1.0);
  const float n_lo = -limit + (float)notch;
  volatile float lm1 = limit - 1.0f;
  const float n_hi = lm1 + (float)notch;
  float s_host = (float)scale_host;
  if (scale_is_decimal) s_host = (float)pow(2.0, -scale_host);
  const bool gc = g_clamped_out != nullptr, gx = gx_out != nullptr;
  // without gx the output type does not matter: one instantiation
  return dispatch_dtype(gx ? gx_dtype : QSB_DTYPE_F32, [&](auto *tg) {
    using TG = std::remove_pointer_t<decltype(tg)>;
    MapIOT<float, float, TG> io{g, nullptr, mask_kind == QSB_MASK_ELEMENT ? mask_dev : nullptr,
                                g_clamped_out, static_cast<TG *>(gx_out), nullptr};
    return dispatch_mask(mask_kind, [&](auto mk) {
      constexpr int MK = decltype(mk)::value;
      auto run = [&](auto op) {
        return launch_map_big_out(op, io, L, (cudaStream_t)stream);
      };
      if (gc && gx)
        return run(SteOp<MK, true, true>{scale_dev, stride, s_host,
                                         scale_is_decimal != 0, n_lo, n_hi,
                                         mask_dev});
      if constexpr (std::is_same<TG, float>::value) {
        if (gc)
          return run(SteOp<MK, true, false>{scale_dev, stride, s_host,
                                            scale_is_decimal != 0, n_lo, n_hi,
                                            mask_dev});
      }
      return run(SteOp<MK, false, true>{scale_dev, stride, s_host,
                                        scale_is_decimal != 0, n_lo, n_hi,
                                        mask_dev});
    });
  });
}

extern "C" int qsb_ste_bwd(const float *g, float *g_clamped_out, float *gx_out, const float *scale_dev,
                           int64_t n_scale, double scale_host, int scale_is_decimal, int bits, int notch,
                           const uint8_t *mask_dev, int mask_kind, int64_t outer, int64_t channels,
                           int64_t inner, void *stream) {
  return qsb_ste_bwd_dt(g, g_clamped_out, gx_out, QSB_DTYPE_F32, scale_dev, n_scale, scale_host, scale_is_decimal,
                        bits, notch, mask_dev, mask_kind, outer, channels, inner, stream);
}

extern "C" int qsb_mask_apply_dt(const void *x, int x_dtype, void *y, int y_dtype, const uint8_t *mask_dev,
                                 int mask_kind, int64_t outer, int64_t channels,
                                 int64_t inner, void *stream) {
  if (!dtype_ok(x_dtype) || !dtype_ok(y_dtype)) return QSB_E_BADARG;
  if (int e = check_layout(outer, channels, inner)) return e;
  if (int e = check_mask(mask_dev, mask_kind, outer * channels * inner)) return e;
  if (mask_kind == QSB_MASK_NONE) return QSB_E_BADARG;
  if (outer * channels * inner == 0) return 0;
  if (!x || !y) return QSB_E_BADARG;
  const Layout L = effective_layout(outer, channels, inner,
                                    mask_kind == QSB_MASK_CHANNEL);
  // (16-bit in, fp32 out): the forward of `x * mask`; (fp32 in, 16-bit out): its backward; (T, T): plain
  if (x_dtype != QSB_DTYPE_F32 && y_dtype != QSB_DTYPE_F32 && x_dtype != y_dtype) return QSB_E_UNSUPPORTED;
  const int dt16 = x_dtype != QSB_DTYPE_F32 ? x_dtype : y_dtype;
  return dispatch_dtype(dt16, [&](auto *t16) {
    using T = std::remove_pointer_t<decltype(t16)>;
    auto run = [&](auto io) {
      if (mask_kind == QSB_MASK_CHANNEL) {
        MaskApplyOp<QSB_MASK_CHANNEL> op{mask_dev};
        return launch_map<decltype(op), Hint::STREAM, Hint::KEEP>(op, io, L, (cudaStream_t)stream);
      }
      MaskApplyOp<QSB_MASK_ELEMENT> op{mask_dev};
      return launch_map<decltype(op), Hint::STREAM, Hint::KEEP>(op, io, L, (cudaStream_t)stream);
    };
    const uint8_t *inb = mask_kind == QSB_MASK_ELEMENT ? mask_dev : nullptr;
    if constexpr (std::is_same<T, float>::value) {
      return run(MapIO{static_cast<const float *>(x), nullptr, inb, static_cast<float *>(y), nullptr, nullptr});
    } else {
      if (x_dtype == y_dtype)
        return run(MapIOT<T, T>{static_cast<const T *>(x), nullptr, inb, static_cast<T *>(y), nullptr, nullptr});
      if (y_dtype == QSB_DTYPE_F32)
        return run(MapIOT<T, float>{static_cast<const T *>(x), nullptr, inb, static_cast<float *>(y), nullptr,
                                    nullptr});
      return run(MapIOT<float, T>{static_cast<const float *>(x), nullptr, inb, static_cast<T *>(y), nullptr,
                                  nullptr});
    }
  });
}

extern "C" int qsb_mask_apply(const float *x, float *y, const uint8_t *mask_dev, int mask_kind, int64_t outer,
                              int64_t channels, int64_t inner, void *stream) {
  return qsb_mask_apply_dt(x, QSB_DTYPE_F32, y, QSB_DTYPE_F32, mask_dev, mask_kind, outer, channels, inner, stream);
}

#ifdef QSB_KERNEL_TIMING
namespace qsb {
int ktime_reduce_op(unsigned long long *out, cudaStream_t stream);
}
#endif
// development only: reset (out == NULL) or read (3 x 2 x 256 uint64: [kernel][start / end][SM]) the kernel stamps
// of a -DQSB_KERNEL_TIMING build; QSB_E_UNSUPPORTED in a normal build
extern "C" int qsb_debug_kernel_times(unsigned long long *out_host, void *stream) {
#ifdef QSB_KERNEL_TIMING
  if (!out_host) {
    int rc = qsb::ktime_reduce_op(nullptr, (cudaStream_t)stream);
    if (rc) return rc;
    return qsb::ktime_host_op(nullptr, (cudaStream_t)stream);
  }
  static unsigned long long a[3][2][256], b[3][2][256];
  int rc = qsb::ktime_reduce_op(&a[0][0][0], nullptr);
  if (rc) return rc;
  if ((rc = qsb::ktime_host_op(&b[0][0][0], nullptr))) return rc;
  for (int s = 0; s < 2 * 256; ++s) {
    out_host[s] = (&a[0][0][0])[s];                          // slot 0: the statistics kernel (reduce.cu)
    out_host[2 * 256 + s] = (&b[1][0][0])[s];                // slots 1, 2: the map kernels (this file)
    out_host[4 * 256 + s] = (&b[2][0][0])[s];
  }
  return 0;
#else
  (void)out_host;
  (void)stream;
  return QSB_E_UNSUPPORTED;
#endif
}

extern "C" int qsb_set_tuning(int key, int value) {
  if (key == 2) {
    map_reverse_tiles() = value;
    return 0;
  }
  if (key == 4) {
    set_select_fast(value);
    return 0;
  }
  if (key == 12) {
    set_pdl_enabled(value);
    return 0;
  }
  if (key == 17) {
    set_reduce_row_variant(value);
    return 0;
  }
  if (key == 18) {
    set_reduce_keep_hint(value);
    return 0;
  }
  if (key == 21) {
    // L2 set-aside for persisting accesses, in MB (device-wide, like cudaDeviceSetLimit): the keep hint of the
    // fused training step reads the kept channels with L2::evict_last, which only has capacity of its own when a
    // set-aside exists.  0 removes the set-aside; the value is clamped to the device maximum.
    int dev = 0, max_bytes = 0;
    QSB_CUDA_TRY(cudaGetDevice(&dev));
    QSB_CUDA_TRY(cudaDeviceGetAttribute(&max_bytes, cudaDevAttrMaxPersistingL2CacheSize, dev));
    size_t want = (size_t)(value < 0 ? 0 : value) << 20;
    if (want > (size_t)max_bytes) want = (size_t)max_bytes;
    QSB_CUDA_TRY(cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, want));
    return 0;
  }
  return QSB_E_BADARG;
}

// ---- self test: div_rn_by == __fdiv_rn on pseudo-random operand pairs ----------
namespace qsb {
__device__ __forceinline__ uint32_t mix32(uint64_t z) {
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return (uint32_t)((z ^ (z >> 31)) >> 16);
}
__global__ void selftest_fastdiv_kernel(uint64_t pairs_per_thread, uint64_t seed,
                                        unsigned long long *mismatches) {
  const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  // one divisor per thread (as in the kernels: shared by many elements)
  uint32_t sb = mix32(seed * 0x9e3779b97f4a7c15ull + tid * 2 + 1);
  const uint32_t mode = tid & 3;
  uint32_t sexp = 87 + (mix32(seed + tid * 7919) % 80);        // inside the fast range
  if (mode == 3) sexp = mix32(seed ^ (tid * 104729)) & 0xff;    // anywhere (slow path too)
  const float s = __uint_as_float((sb & 0x807fffffu) | (sexp << 23));
  const float r = __frcp_rn(s);
  const bool ok = fastdiv_divisor_ok(s);
  unsigned long long bad = 0;
  for (uint64_t i = 0; i < pairs_per_thread; ++i) {
    uint32_t xb = mix32((seed + 0x1234567ull) * (tid + 1) + i * 0x9e3779b97f4a7c15ull);
    float x;
    if ((i & 7) == 0) {
      // near rounding boundaries of rint(x / s): x ~ (k + 0.5) * s
      const float k = (float)((int)(xb & 0xffff) - 32768) + 0.5f;
      x = __fmul_rn(k, s);
      x = __uint_as_float(__float_as_uint(x) + ((xb >> 16) & 3) - 1);
    } else if ((i & 7) == 1) {
      x = __uint_as_float(xb);  // anything, incl. NaN / inf / subnormal
    } else {
      const uint32_t xexp = 100 + (mix32(xb) % 56);
      x = __uint_as_float((xb & 0x807fffffu) | (xexp << 23));
    }
    const float a = div_rn_by(x, s, r, ok);
    const float b = __fdiv_rn(x, s);
    const bool same = (__float_as_uint(a) == __float_as_uint(b)) || (a != a && b != b);
    bad += same ? 0 : 1;
  }
  if (bad) atomicAdd(mismatches, bad);
}
}  // namespace qsb

extern "C" int qsb_selftest_fastdiv(int64_t n_threads, int64_t pairs_per_thread,
                                    uint64_t seed,
                                    unsigned long long *mismatches_dev,
                                    void *stream) {
  if (n_threads <= 0 || pairs_per_thread <= 0 || !mismatches_dev) return QSB_E_BADARG;
  const unsigned blocks = (unsigned)((n_threads + 255) / 256);
  selftest_fastdiv_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(
      (uint64_t)pairs_per_thread, seed, mismatches_dev);
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_mask_from_threshold(const float *importance, int take_abs,
                                       const float *thr_dev, uint8_t *mask_out,
                                       int64_t n, void *stream) {
  if (n < 0) return QSB_E_BADARG;
  if (n == 0) return 0;
  if (!importance || !thr_dev || !mask_out) return QSB_E_BADARG;
  MapIO io{importance, nullptr, nullptr, nullptr, nullptr, mask_out};
  MaskBuildOp<false> op{thr_dev, take_abs != 0};
  return launch_map<decltype(op), Hint::KEEP, Hint::KEEP>(
      op, io, Layout{1, 1, n}, (cudaStream_t)stream);
}

extern "C" int qsb_mask_build_apply(const float *importance, int take_abs,
                                    const float *thr_dev, const float *x,
                                    float *y, uint8_t *mask_out, int64_t n,
                                    void *stream) {
  if (n < 0) return QSB_E_BADARG;
  if (n == 0) return 0;
  if (!importance || !thr_dev || !x || !y || !mask_out) return QSB_E_BADARG;
  MapIO io{importance, x, nullptr, y, nullptr, mask_out};
  MaskBuildOp<true> op{thr_dev, take_abs != 0};
  return launch_map<decltype(op), Hint::STREAM, Hint::KEEP>(
      op, io, Layout{1, 1, n}, (cudaStream_t)stream);
}

// ---- multi-tensor forms (the layers of a weight set in one launch) ----------------------
static bool all_aligned32(const void *const *p, int count) {
  for (int i = 0; i < count; ++i)
    if (!aligned_to(p[i], 32)) return false;
  return true;
}

extern "C" int qsb_mask_build_apply_multi(const float *const *importance, int take_abs,
                                          const float *thr_dev, const float *const *x,
                                          float *const *y, uint8_t *const *mask_out,
                                          const int64_t *n, int count, void *stream) {
  if (count < 0) return QSB_E_BADARG;
  if (count == 0) return 0;
  if (!importance || !thr_dev || !x || !y || !mask_out || !n) return QSB_E_BADARG;
  if (!all_aligned32((const void *const *)importance, count) ||
      !all_aligned32((const void *const *)x, count) || !all_aligned32((const void *const *)y, count))
    return QSB_E_UNSUPPORTED;
  std::vector<MultiEntry> ent((size_t)count);
  for (int i = 0; i < count; ++i) {
    if (n[i] < 0 || !importance[i] || !x[i] || !y[i] || !mask_out[i]) return QSB_E_BADARG;
    if (!aligned_to(mask_out[i], 8)) return QSB_E_UNSUPPORTED;
    ent[i] = MultiEntry{importance[i], x[i], y[i], mask_out[i], thr_dev + i, n[i], 0};
  }
  MaskBuildOp<true> op{thr_dev, take_abs != 0};
  return launch_map_multi<decltype(op), Hint::STREAM, Hint::KEEP>(op, ent.data(), count,
                                                                   (cudaStream_t)stream);
}

extern "C" int qsb_magnitude_ema_full_multi(float *const *magnitude, const float *const *x,
                                            const int64_t *n, int count, int64_t t,
                                            void *stream) {
  if (count < 0 || t < 0) return QSB_E_BADARG;
  if (count == 0) return 0;
  if (!magnitude || !x || !n) return QSB_E_BADARG;
  if (!all_aligned32((const void *const *)magnitude, count) ||
      !all_aligned32((const void *const *)x, count))
    return QSB_E_UNSUPPORTED;
  std::vector<MultiEntry> ent((size_t)count);
  for (int i = 0; i < count; ++i) {
    if (n[i] < 0 || !magnitude[i] || !x[i]) return QSB_E_BADARG;
    ent[i] = MultiEntry{x[i], magnitude[i], magnitude[i], nullptr, nullptr, n[i], 0};
  }
  const float tp1 = (float)(t + 1);
  volatile float rcp = 1.0f / tp1;  // IEEE round-to-nearest on the host
  EmaFullOp op{nullptr, false, (float)t, tp1, rcp};
  return launch_map_multi<decltype(op), Hint::STREAM, Hint::KEEP>(op, ent.data(), count,
                                                                   (cudaStream_t)stream);
}

extern "C" int qsb_magnitude_ema_full(float *magnitude, const float *x,
                                      const float *tensor_min, int use_l0,
                                      int64_t n, int64_t t, void *stream) {
  if (n < 0 || t < 0) return QSB_E_BADARG;
  if (n == 0) return 0;
  if (!magnitude || !x) return QSB_E_BADARG;
  if (use_l0 && !tensor_min) return QSB_E_BADARG;
  MapIO io{x, magnitude, nullptr, magnitude, nullptr, nullptr};
  const float tp1 = (float)(t + 1);
  volatile float rcp = 1.0f / tp1;  // IEEE round-to-nearest on the host
  EmaFullOp op{tensor_min, use_l0 != 0, (float)t, tp1, rcp};
  return launch_map<decltype(op), Hint::STREAM, Hint::KEEP>(
      op, io, Layout{1, 1, n}, (cudaStream_t)stream);
}
