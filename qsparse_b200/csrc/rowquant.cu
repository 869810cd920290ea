// K8  row-resident fused scale estimation + fake-quantization for tensors whose
// quantization channel is the leading axis (the `channelwise=0` weight case:
// `quantize(nn.Linear(4096, 4096), bits=4, channelwise=0, callback=AdaptiveQuantizer())`,
// BASELINE config 3).
//
// The reference runs, per training access of the weight,
//     optimize: min / max (or abs-max) per row  -> EMA into the layer's parameter
//               qsparse/quantize.py:327-349 (Decimal/Scaler), :393-430 (Adaptive)
//     forward : fake-quantize every row with its updated parameter
//               qsparse/quantize.py:44-63, :100-117, :148-181
// i.e. read (reduce) + tiny kernel + read + write = 12 B/elem in three launches with a
// grid-wide dependency in the middle.  A channel here is ONE contiguous row, so nothing
// crosses CTAs: a CTA (rows of 1 Ki .. 16 Ki elements) or a warp (shorter rows) loads its
// row ONCE into registers, reduces it, updates the row's parameter, and quantizes the row
// from the registers: 8 B/elem, one launch, no dependency between CTAs.
//
// row_quant_kernel: the row lives in registers: a CTA per row (1 Ki .. 16 Ki elements, one
// barrier: every thread merges the warps' partials and derives the new parameter itself) or a
// warp per row (shorter rows).  Measured on [4096, 4096] (134 MB of traffic): 25.6 us scaler /
// 28.7 us line — the same as the plain fake-quant kernel alone on that tensor (28.6 us), against
// 50.2 us for reduce -> EMA -> quantize.
//
// A TMA-pipelined persistent variant (ONE thread streamed a CTA's rows into a ring of
// shared-memory stages with cp.async.bulk, 2-4 rows ahead) was measured at 30.7 us for every
// (CTAs per SM, stages) in {2..8} x {2..4} and removed: the row's dependent chain (wait -> LDS ->
// reduce -> barrier -> quantize -> store) bounds a persistent CTA, and one CTA per row with
// 5 CTAs per SM overlaps those chains better.
//
// Arithmetic is the same device code as the unfused kernels (fq_ops.cuh, param_math.cuh),
// so the results are bit-identical to reduce_stats -> *_ema -> fq_*_fwd.
#include <math.h>

#include "fq_ops.cuh"
#include "map_kernel.cuh"
#include "param_math.cuh"

namespace qsb {

constexpr int kRowDecimal = 0, kRowScaler = 1, kRowLine = 2;

struct RowConsts {
  float limit;     // 2^(bits-1)                      (decimal / scaler)
  float n_levels;  // 2^bits                          (line)
  float q_max;     // 2^bits - 1                      (line)
  int64_t t;       // scale EMA: calls so far (0-based); lines EMA: this call's number (1-based)
  const long long *t_dev;  // optional device step counter (CUDA graphs): the index is *t_dev + t
};

struct RowStat {
  uint32_t amax;  // bits of max |x|; NaN patterns order above inf (as in reduce.cu)
  float mn, mx;
  int nan;
};

template <int KIND>
__device__ __forceinline__ void stat_add(RowStat &s, float v) {
  if constexpr (KIND == kRowLine) {
    s.mn = fminf(s.mn, v);
    s.mx = fmaxf(s.mx, v);
    s.nan |= (v != v);
  } else {
    const uint32_t b = __float_as_uint(v) & 0x7fffffffu;
    s.amax = b > s.amax ? b : s.amax;
  }
}

template <int KIND>
__device__ __forceinline__ void stat_merge(RowStat &s, const RowStat &o) {
  if constexpr (KIND == kRowLine) {
    s.mn = fminf(s.mn, o.mn);
    s.mx = fmaxf(s.mx, o.mx);
    s.nan |= o.nan;
  } else {
    s.amax = o.amax > s.amax ? o.amax : s.amax;
  }
}

template <int KIND>
__device__ __forceinline__ RowStat stat_warp(RowStat s) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    RowStat t;
    if constexpr (KIND == kRowLine) {
      t.mn = __shfl_xor_sync(0xffffffffu, s.mn, o);
      t.mx = __shfl_xor_sync(0xffffffffu, s.mx, o);
      t.nan = __shfl_xor_sync(0xffffffffu, s.nan, o);
    } else {
      t.amax = __shfl_xor_sync(0xffffffffu, s.amax, o);
    }
    stat_merge<KIND>(s, t);
  }
  return s;
}

// statistics + the row's old parameter -> its updated parameter (x = scale or lo, y = hi)
template <int KIND>
__device__ __forceinline__ float2 ema_param(const RowStat &s, float2 w, const RowConsts &k) {
  float2 r;
  if constexpr (KIND == kRowLine) {
    const float mn = s.nan ? __uint_as_float(0x7fc00000u) : s.mn;
    const float mx = s.nan ? __uint_as_float(0x7fc00000u) : s.mx;
    const int64_t t = k.t_dev ? (int64_t)__ldg(k.t_dev) + k.t : k.t;
    const float tm1 = (float)(t - 1), tf = (float)t;
    r.x = lines_ema_step(w.x, mn, tm1, tf);
    r.y = lines_ema_step(w.y, mx, tm1, tf);
  } else {
    const int64_t t = k.t_dev ? (int64_t)__ldg(k.t_dev) + k.t : k.t;
    r.x = scale_ema_step(w.x, __uint_as_float(s.amax), k.limit, t);
    r.y = 0.f;
  }
  return r;
}

template <int KIND>
__device__ __forceinline__ float2 load_param(const float *prm) {
  if constexpr (KIND == kRowLine) return *reinterpret_cast<const float2 *>(prm);
  return make_float2(prm[0], 0.f);
}

template <int KIND>
__device__ __forceinline__ void store_param(float *prm, float2 v) {
  if constexpr (KIND == kRowLine) *reinterpret_cast<float2 *>(prm) = v;
  else prm[0] = v.x;
}

template <int KIND, bool FZP>
struct RowOp;
template <bool FZP>
struct RowOp<kRowDecimal, FZP> {
  using Op = Pow2Op<QSB_MASK_NONE>;
  __device__ static Op make(const RowConsts &) { return Op{nullptr, 0, 1.f, 1.f, nullptr}; }
  __device__ static typename Op::P derive(const Op &, float2 v) { return Op::derive(v.y); }
};
template <bool FZP>
struct RowOp<kRowScaler, FZP> {
  using Op = ScalerOp<QSB_MASK_NONE>;
  __device__ static Op make(const RowConsts &) { return Op{nullptr, 0, 1.f, nullptr}; }
  __device__ static typename Op::P derive(const Op &, float2 v) { return Op::derive(v.x); }
};
template <bool FZP>
struct RowOp<kRowLine, FZP> {
  using Op = LineOp<QSB_MASK_NONE, FZP>;
  __device__ static Op make(const RowConsts &k) {
    return Op{nullptr, 0, 0.f, 0.f, k.n_levels, k.q_max, nullptr};
  }
  __device__ static typename Op::P derive(const Op &op, float2 v) { return op.derive(v.x, v.y); }
};

// G threads own one row: G = QSB_THREADS (a CTA per row) or 32 (a warp per row, 8 rows per CTA).
// MASKED: an element prune mask is applied first (the weight chain quantize(prune(layer)),
// ref qsparse/imitation.py:61-71): statistics and quantization both see x * mask — a real multiply by
// 0.0 / 1.0 like the reference's — in the same single read of the row (+1 B/elem for the mask).
// 6 CTAs / SM (<= 42 registers) for the unmasked kernels with <= 2 vectors per thread: the line quantizer otherwise
// takes 54 registers = 4 CTAs / SM, whose load / reduce / quantize phases then overlap too little.  A/B on one box
// (benchmarks/time_c3.py, 20 launches per graph on [4096,4096]): line 26.8 -> 21.9 us, scaler 21.0 -> 20.1 us,
// decimal 22.4 -> 21.0 us; ncu, cold and isolated: line 24.5 -> 21.8 us.  (Single event-bracketed launches vary by
// +-1.5 us from box to box, which hid this in bench.py --config 3.)
#ifndef QSB_K8_MIN_CTAS
#define QSB_K8_MIN_CTAS 6
#endif
template <int KIND, bool FZP, int U, int G, bool MASKED>
__global__ void __launch_bounds__(QSB_THREADS, (U <= 2 && !MASKED) ? QSB_K8_MIN_CTAS : 1)
    row_quant_kernel(const float *__restrict__ x, float *__restrict__ y, float *__restrict__ param,
                     float *__restrict__ decimal_out, const uint8_t *__restrict__ mask, int64_t rows, int inner,
                     RowConsts k) {
  constexpr int V = 8;
  constexpr int kRowsPerCta = QSB_THREADS / G;
  constexpr int kWsz = (KIND == kRowLine) ? 2 : 1;
  const int tid = threadIdx.x, g = tid % G, lane = tid & 31;
  const int64_t row = (int64_t)blockIdx.x * kRowsPerCta + tid / G;
  const bool live = row < rows;  // uniform per warp (G is a multiple of 32)
  const float *xr = x + row * inner;
  float *yr = y + row * inner;
  const int nvec = inner / V;

  VecF<V> a[U];
  float2 w_old = make_float2(0.f, 0.f);
  if (live) {
    VecB<V> mb[U];
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (u * G + g < nvec) {
        a[u] = ld_vec<V, Hint::KEEP>(xr + (int64_t)(u * G + g) * V);
        if constexpr (MASKED) mb[u] = ld_bytes<V>(mask + row * inner + (int64_t)(u * G + g) * V);
      }
    w_old = load_param<KIND>(param + row * kWsz);  // in flight together with the row
    if constexpr (MASKED) {
#pragma unroll
      for (int u = 0; u < U; ++u)
        if (u * G + g < nvec) {
#pragma unroll
          for (int j = 0; j < V; ++j) a[u].v[j] = __fmul_rn(a[u].v[j], mb[u].b[j] ? 1.0f : 0.0f);
        }
    }
  }
  RowStat s{0u, INFINITY, -INFINITY, 0};
  if (live) {
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (u * G + g < nvec) {
#pragma unroll
        for (int j = 0; j < V; ++j) stat_add<KIND>(s, a[u].v[j]);
      }
  }
  s = stat_warp<KIND>(s);
  if constexpr (G != 32) {  // one barrier: every thread merges the warps' partials itself
    __shared__ RowStat s_part[QSB_THREADS / 32];
    if (lane == 0) s_part[tid >> 5] = s;
    __syncthreads();
    s = s_part[0];
#pragma unroll
    for (int w = 1; w < QSB_THREADS / 32; ++w) stat_merge<KIND>(s, s_part[w]);
  }
  // every thread derives the new parameter (a few flops, no second barrier); one writes it
  float2 pv = ema_param<KIND>(s, w_old, k);
  if (live && g == 0) store_param<KIND>(param + row * kWsz, pv);
  if constexpr (KIND == kRowDecimal) {
    // the fp64 log2 of scale -> decimal is worth computing once per row
    if constexpr (G == 32) {
      if (lane == 0) pv.y = scale_to_decimal(pv.x);
      pv.y = __shfl_sync(0xffffffffu, pv.y, 0);
    } else {
      __shared__ float s_dec;
      if (tid == 0) s_dec = scale_to_decimal(pv.x);
      __syncthreads();
      pv.y = s_dec;
    }
    if (live && g == 0 && decimal_out) decimal_out[row] = pv.y;
  }
  if (!live) return;

  using RO = RowOp<KIND, FZP>;
  const typename RO::Op op = RO::make(k);
  const typename RO::Op::P p = RO::derive(op, pv);
#pragma unroll
  for (int u = 0; u < U; ++u)
    if (u * G + g < nvec) {
      VecF<V> o0, o1;
      VecB<V> mb, ob;
      apply_vec<typename RO::Op, V>(op, a[u], a[u], mb, false, p, o0, o1, ob);
      st_vec<V, Hint::KEEP>(yr + (int64_t)(u * G + g) * V, o0);
    }
}

template <int KIND, bool FZP, int U, int G>
static int launch_rows(const float *x, float *y, float *param, float *decimal_out, const uint8_t *mask,
                       int64_t rows, int64_t inner, const RowConsts &k, cudaStream_t stream) {
  constexpr int kRowsPerCta = QSB_THREADS / G;
  const int64_t grid = (rows + kRowsPerCta - 1) / kRowsPerCta;
  if (grid > 0x7fffffffll) return QSB_E_UNSUPPORTED;
  if (mask)
    row_quant_kernel<KIND, FZP, U, G, true>
        <<<(unsigned)grid, QSB_THREADS, 0, stream>>>(x, y, param, decimal_out, mask, rows, (int)inner, k);
  else
    row_quant_kernel<KIND, FZP, U, G, false>
        <<<(unsigned)grid, QSB_THREADS, 0, stream>>>(x, y, param, decimal_out, nullptr, rows, (int)inner, k);
  QSB_LAUNCH_CHECK();
  return 0;
}

template <int KIND, bool FZP>
static int dispatch_rows(const float *x, float *y, float *param, float *decimal_out, const uint8_t *mask,
                         int64_t rows, int64_t inner, const RowConsts &k, cudaStream_t stream) {
  // a warp per row up to 1 Ki elements, a CTA per row up to 16 Ki
  if (inner <= 256) return launch_rows<KIND, FZP, 1, 32>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  if (inner <= 512) return launch_rows<KIND, FZP, 2, 32>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  if (inner <= 1024) return launch_rows<KIND, FZP, 4, 32>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  if (inner <= 2048) return launch_rows<KIND, FZP, 1, QSB_THREADS>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  if (inner <= 4096) return launch_rows<KIND, FZP, 2, QSB_THREADS>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  if (inner <= 8192) return launch_rows<KIND, FZP, 4, QSB_THREADS>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  if (inner <= 16384) return launch_rows<KIND, FZP, 8, QSB_THREADS>(x, y, param, decimal_out, mask, rows, inner, k, stream);
  return QSB_E_UNSUPPORTED;
}

}  // namespace qsb

using namespace qsb;

static int row_quant_fused_impl(const float *x, float *y, float *param, float *decimal_out,
                                const uint8_t *mask, int kind, int bits, int float_zero_point,
                                int64_t rows, int64_t inner, int64_t t, void *stream_,
                                const int64_t *t_dev = nullptr) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (rows < 0 || inner < 0 || bits < 0 || bits > 62) return QSB_E_BADARG;
  if (kind < kRowDecimal || kind > kRowLine) return QSB_E_BADARG;
  if (!t_dev && (kind == kRowLine ? t < 1 : t < 0)) return QSB_E_BADARG;
  if (rows == 0 || inner == 0) return 0;
  if (!x || !y || !param) return QSB_E_BADARG;
  if (kind == kRowLine && !aligned_to(param, 8)) return QSB_E_ALIGN;
  // rows must be whole 256-bit vectors: anything else takes the two-kernel path
  if (inner % 8 != 0 || inner > 16384 || !aligned_to(x, 32) || !aligned_to(y, 32))
    return QSB_E_UNSUPPORTED;
  RowConsts k;
  k.limit = (float)pow(2.0, (double)bits - 1.0);
  const double N = ldexp(1.0, bits);
  k.n_levels = (float)N;
  k.q_max = (float)(N - 1.0);
  k.t = t;
  k.t_dev = reinterpret_cast<const long long *>(t_dev);
  switch (kind) {
    case kRowDecimal:
      return dispatch_rows<kRowDecimal, true>(x, y, param, decimal_out, mask, rows, inner, k, stream);
    case kRowScaler:
      return dispatch_rows<kRowScaler, true>(x, y, param, nullptr, mask, rows, inner, k, stream);
    default:
      return float_zero_point
                 ? dispatch_rows<kRowLine, true>(x, y, param, nullptr, mask, rows, inner, k, stream)
                 : dispatch_rows<kRowLine, false>(x, y, param, nullptr, mask, rows, inner, k, stream);
  }
}

extern "C" int qsb_row_quant_fused(const float *x, float *y, float *param, float *decimal_out,
                                   int kind, int bits, int float_zero_point, int64_t rows,
                                   int64_t inner, int64_t t, void *stream) {
  return row_quant_fused_impl(x, y, param, decimal_out, nullptr, kind, bits, float_zero_point, rows, inner, t,
                              stream);
}

// the weight chain quantize(prune(layer)) with a frozen mask: y = Q(x * mask), parameters estimated
// on x * mask, one read of x (4) + mask (1) + one write (4) = 9 B/elem instead of mask-apply (9) +
// estimate/quantize (8).  mask_dev: uint8 [rows * inner], 8-byte aligned.
extern "C" int qsb_row_quant_fused_masked(const float *x, float *y, float *param, float *decimal_out,
                                          const uint8_t *mask_dev, int kind, int bits,
                                          int float_zero_point, int64_t rows, int64_t inner,
                                          int64_t t, void *stream) {
  if (!mask_dev) return QSB_E_BADARG;
  if (!aligned_to(mask_dev, 8)) return QSB_E_UNSUPPORTED;
  return row_quant_fused_impl(x, y, param, decimal_out, mask_dev, kind, bits, float_zero_point, rows, inner,
                              t, stream);
}

// CUDA-graph form of the two entry points above: the EMA index is *t_dev + t_offset, read by the kernel
// (launch arguments of a captured graph are frozen); mask_dev may be NULL.  The caller advances the counter.
extern "C" int qsb_row_quant_fused_at(const float *x, float *y, float *param, float *decimal_out,
                                      const uint8_t *mask_dev, int kind, int bits, int float_zero_point,
                                      int64_t rows, int64_t inner, const int64_t *t_dev, int64_t t_offset,
                                      void *stream) {
  if (!t_dev) return QSB_E_BADARG;
  if (mask_dev && !aligned_to(mask_dev, 8)) return QSB_E_UNSUPPORTED;
  return row_quant_fused_impl(x, y, param, decimal_out, mask_dev, kind, bits, float_zero_point, rows, inner,
                              t_offset, stream, t_dev);
}
