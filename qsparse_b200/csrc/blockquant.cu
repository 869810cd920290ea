// Block-scaled FP8 / FP4 fake quantization and its packed export: MXFP8, MXFP4 (OCP Microscaling v1.0:
// blocks of 32 elements, E8M0 power-of-two scale) and NVFP4 (blocks of 16, E4M3 scale times one fp32 tensor
// scale).  The numerics are DESIGN §2 "Block-scaled formats"; oracle/block_scaled.py restates them in numpy.
//
// x is walked as [rows, L] in its physical order; each row splits into blocks of B consecutive elements, the last
// one possibly shorter.  The streaming skeleton of map_kernel.cuh: one CTA per tile, U vectors of 8 elements per
// thread with all loads issued before the arithmetic, int64 element indices, programmatic dependent launch.  The
// B / 8 consecutive lanes of a "block group" hold the consecutive 8-element vectors of one block, so a block's
// abs-max is an xor-shuffle over 4 (B = 32) or 2 (B = 16) lanes; the lanes of a short last block that fall past
// the row end hold nothing.  Two routes, picked on the host:
//   VEC  L % 8 == 0 and every pointer aligned for whole-vector accesses: one 256-bit (fp32) or 128-bit (16-bit)
//        load per vector, one 256-bit y store / one 64-bit E4M3 or 32-bit E2M1 code store;
//   any  other row lengths and views (a 16-bit view may start at any even address): element accesses.
// All conversions are the sm_100a cvt instructions: cvt.rn.satfinite.{e4m3x2,e2m1x2}.f32 (F2FP.SATFINITE.E4M3 /
// .E2M1), cvt.rp.satfinite.ue8m0x2.f32 (F2FP.SATFINITE.E8) and the f16x2 unpacks (F2FP.F16.E4M3 / .E2M1.UNPACK_B).
#include "map_kernel.cuh"

namespace qsb {
namespace {

enum : int { kMXFP8 = 0, kMXFP4 = 1, kNVFP4 = 2 };

template <int FMT>
struct BlockFmt {
  static constexpr int B = FMT == kNVFP4 ? 16 : 32;  // elements per block
  static constexpr int G = B / 8;                    // lanes per block
  static constexpr bool kFp8 = FMT == kMXFP8;        // E4M3 elements, else E2M1
};

// ---- conversions (first PTX source operand -> upper half of the packed result) ------------------------------
__device__ __forceinline__ uint32_t e4m3x2(float lo, float hi) {
  unsigned short d;
  asm("cvt.rn.satfinite.e4m3x2.f32 %0, %1, %2;" : "=h"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ float2 e4m3x2_decode(uint32_t v) {
  uint32_t h;
  asm("cvt.rn.f16x2.e4m3x2 %0, %1;" : "=r"(h) : "h"((unsigned short)v));
  return __half22float2(*reinterpret_cast<const __half2 *>(&h));
}
// 8 values -> 8 E2M1 nibbles, element j in nibble j
__device__ __forceinline__ uint32_t e2m1x8(const float (&q)[8]) {
  uint32_t w;
  asm("{\n\t.reg .b8 b0, b1, b2, b3;\n\t"
      "cvt.rn.satfinite.e2m1x2.f32 b0, %2, %1;\n\t"
      "cvt.rn.satfinite.e2m1x2.f32 b1, %4, %3;\n\t"
      "cvt.rn.satfinite.e2m1x2.f32 b2, %6, %5;\n\t"
      "cvt.rn.satfinite.e2m1x2.f32 b3, %8, %7;\n\t"
      "mov.b32 %0, {b0, b1, b2, b3};\n\t}"
      : "=r"(w)
      : "f"(q[0]), "f"(q[1]), "f"(q[2]), "f"(q[3]), "f"(q[4]), "f"(q[5]), "f"(q[6]), "f"(q[7]));
  return w;
}
__device__ __forceinline__ void e2m1x8_decode(uint32_t w, float (&v)[8]) {
  uint32_t h[4];
  asm("{\n\t.reg .b8 b0, b1, b2, b3;\n\t"
      "mov.b32 {b0, b1, b2, b3}, %4;\n\t"
      "cvt.rn.f16x2.e2m1x2 %0, b0;\n\t"
      "cvt.rn.f16x2.e2m1x2 %1, b1;\n\t"
      "cvt.rn.f16x2.e2m1x2 %2, b2;\n\t"
      "cvt.rn.f16x2.e2m1x2 %3, b3;\n\t}"
      : "=r"(h[0]), "=r"(h[1]), "=r"(h[2]), "=r"(h[3])
      : "r"(w));
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const float2 f = __half22float2(*reinterpret_cast<const __half2 *>(&h[k]));
    v[2 * k] = f.x;
    v[2 * k + 1] = f.y;
  }
}
// the E8M0 byte of a power of two 2^k, k in [-127, 127]: k + 127
__device__ __forceinline__ uint32_t ue8m0(float p2) {
  unsigned short d;
  asm("cvt.rp.satfinite.ue8m0x2.f32 %0, %1, %1;" : "=h"(d) : "f"(p2));
  return d & 0xffu;
}

// 2^k for k in [-127, 127] (2^-127 is subnormal)
__device__ __forceinline__ float pow2_bits(int k) {
  return __uint_as_float(k >= -126 ? (uint32_t)(k + 127) << 23 : 0x00400000u);
}

// floor(log2(a)) of a finite a > 0 from its bits (subnormals included); a == 0 gives -150, below every clamp
__device__ __forceinline__ int exponent_of(uint32_t abits) {
  if (abits >= 0x00800000u) return (int)(abits >> 23) - 127;
  if (abits == 0u) return -150;
  return (31 - __clz(abits)) - 149;
}

// one thread: U vectors; EXPORT writes codes + scales, otherwise y
template <int FMT, bool VEC, bool EXPORT, Hint SH, class T>
__global__ void __launch_bounds__(QSB_THREADS)
    block_quant_kernel(const T *__restrict__ x, float *__restrict__ y, uint8_t *__restrict__ codes,
                       uint8_t *__restrict__ scales, int64_t L, int64_t blocks_per_row, int64_t n_slots,
                       const float *__restrict__ tensor_amax) {
  using F = BlockFmt<FMT>;
  constexpr int U = 2;
  pdl_wait();
  pdl_trigger();
  const bool full_rows = L % F::B == 0;  // no short blocks: block b starts at element b * B
  const int64_t half_row = (L + 1) >> 1;  // bytes per row of E2M1 codes
  float s_t = 0.f;
  bool st_zero = false, st_nan = false;
  if constexpr (FMT == kNVFP4) {
    s_t = __fdiv_rn(__ldg(tensor_amax), 2688.0f);  // 6 * 448
    st_zero = s_t == 0.0f;
    st_nan = s_t != s_t;
  }

  float v[U][8];
  int64_t e0[U], b_of[U], cidx[U];  // first element, block, first code byte (E2M1)
  int cnt[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t slot = (int64_t)blockIdx.x * (QSB_THREADS * U) + u * QSB_THREADS + threadIdx.x;
    cnt[u] = 0;
    e0[u] = b_of[u] = cidx[u] = 0;
    if (slot < n_slots) {
      const int64_t b = slot / F::G;  // G is a power of two
      const int s = (int)(slot & (F::G - 1));
      if (full_rows) {
        e0[u] = b * F::B + 8 * s;
        cnt[u] = 8;
        cidx[u] = e0[u] >> 1;
      } else {
        const int64_t r = b / blocks_per_row;
        const int64_t off = (b - r * blocks_per_row) * F::B + 8 * s;
        e0[u] = r * L + off;
        const int64_t left = L - off;
        cnt[u] = left <= 0 ? 0 : (left < 8 ? (int)left : 8);
        cidx[u] = r * half_row + (off >> 1);
      }
      b_of[u] = b;
    }
    if constexpr (VEC) {
      if (cnt[u] == 8) {
        VecF<8> a;
        if constexpr (is_half16<T>) a = unpack8<T>(ld_raw16(x + e0[u]));
        else a = ld_vec<8, Hint::STREAM>(x + e0[u]);
#pragma unroll
        for (int j = 0; j < 8; ++j) v[u][j] = a.v[j];
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) v[u][j] = 0.f;
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[u][j] = j < cnt[u] ? to_f(x[e0[u] + j]) : 0.f;
    }
  }

#pragma unroll
  for (int u = 0; u < U; ++u) {
    // block abs-max as integer bits: NaN > inf > every finite value, so one max also finds the NaN / inf blocks
    uint32_t amax = 0;
#pragma unroll
    for (int j = 0; j < 8; ++j) amax = max(amax, __float_as_uint(v[u][j]) & 0x7fffffffu);
#pragma unroll
    for (int o = 1; o < F::G; o <<= 1) amax = max(amax, __shfl_xor_sync(0xffffffffu, amax, o));
    if (cnt[u] == 0) continue;
    const bool block_nan = amax >= 0x7f800000u;

    float q[8], scale;
    bool nan_out = block_nan, zero_out = false;
    uint32_t scale_byte;
    if constexpr (FMT == kNVFP4) {
      const float t2 = __fdiv_rn(__fdiv_rn(__uint_as_float(amax), 6.0f), s_t);
      const uint32_t sb_bits = e4m3x2(t2, 0.f) & 0xffu;
      const float s_b = e4m3x2_decode(sb_bits).x;
      scale = __fmul_rn(s_b, s_t);
      nan_out = block_nan || st_nan || (!st_zero && scale != scale);
      zero_out = !nan_out && (st_zero || scale == 0.0f);
      scale_byte = (block_nan || st_nan) ? 0x7fu : (st_zero ? 0u : sb_bits);
      const float r = __frcp_rn(scale);
      const bool ok = fastdiv_divisor_ok(scale);
#pragma unroll
      for (int j = 0; j < 8; ++j) q[j] = div_rn_by(v[u][j], scale, r, ok);
    } else {
      int k = exponent_of(amax) - (F::kFp8 ? 8 : 2);  // e(max element): 448 = 1.75 * 2^8, 6 = 1.5 * 2^2
      k = k < -127 ? -127 : (k > 127 ? 127 : k);
      scale = pow2_bits(k);
      const float inv = pow2_bits(-k);  // x * 2^-k == RN(x / 2^k): one rounding of the same real number
#pragma unroll
      for (int j = 0; j < 8; ++j) q[j] = __fmul_rn(v[u][j], inv);
      scale_byte = block_nan ? 0xffu : ue8m0(scale);
    }

    // codes: element j in byte j (E4M3) or nibble j (E2M1); zero for a NaN or zero-scale block
    uint32_t c_lo, c_hi = 0;  // E4M3: bytes 0-3 / 4-7; E2M1: the 8 nibbles in c_lo
    if constexpr (F::kFp8) {
      c_lo = e4m3x2(q[0], q[1]) | (e4m3x2(q[2], q[3]) << 16);
      c_hi = e4m3x2(q[4], q[5]) | (e4m3x2(q[6], q[7]) << 16);
    } else {
      c_lo = e2m1x8(q);
    }
    if (nan_out || zero_out) c_lo = c_hi = 0;

    if constexpr (EXPORT) {
      if ((threadIdx.x & (F::G - 1)) == 0) scales[b_of[u]] = (uint8_t)scale_byte;
      if constexpr (F::kFp8) {
        if (VEC && cnt[u] == 8) {
          *reinterpret_cast<uint2 *>(codes + e0[u]) = make_uint2(c_lo, c_hi);
        } else {
          for (int j = 0; j < cnt[u]; ++j) codes[e0[u] + j] = (uint8_t)((j < 4 ? c_lo : c_hi) >> (8 * (j & 3)));
        }
      } else {
        if (cnt[u] < 8) c_lo &= (1u << (4 * cnt[u])) - 1u;  // the pad nibble of an odd row is 0
        if (VEC && cnt[u] == 8) {
          *reinterpret_cast<uint32_t *>(codes + cidx[u]) = c_lo;
        } else {
          for (int b2 = 0; b2 < (cnt[u] + 1) / 2; ++b2) codes[cidx[u] + b2] = (uint8_t)(c_lo >> (8 * b2));
        }
      }
    } else {
      float dv[8];
      if constexpr (F::kFp8) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const float2 f = e4m3x2_decode(((k < 2 ? c_lo : c_hi) >> (16 * (k & 1))) & 0xffffu);
          dv[2 * k] = f.x;
          dv[2 * k + 1] = f.y;
        }
      } else {
        e2m1x8_decode(c_lo, dv);
      }
      VecF<8> o;
#pragma unroll
      for (int j = 0; j < 8; ++j) o.v[j] = nan_out ? __uint_as_float(0x7fc00000u) : (zero_out ? 0.0f : __fmul_rn(dv[j], scale));
      if (VEC && cnt[u] == 8) {
        st_vec<8, SH>(y + e0[u], o);
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (j < cnt[u]) y[e0[u] + j] = o.v[j];
      }
    }
  }
}

template <int FMT, bool EXPORT, Hint SH, class T>
int launch_block(const T *x, float *y, uint8_t *codes, uint8_t *scales, int64_t rows, int64_t L,
                 const float *tensor_amax, cudaStream_t stream) {
  using F = BlockFmt<FMT>;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * 2;  // slots per CTA (U = 2)
  const int64_t blocks_per_row = (L + F::B - 1) / F::B;
  const int64_t n_slots = rows * blocks_per_row * F::G;
  const int64_t tiles = (n_slots + kTile - 1) / kTile;
  if (tiles > 0x7fffffffLL) return QSB_E_UNSUPPORTED;
  bool vec = L % 8 == 0 && aligned_to(x, 8 * sizeof(T));
  if (EXPORT) vec = vec && aligned_to(codes, F::kFp8 ? 8 : 4);
  else vec = vec && aligned_to(y, 32);
  auto kern = vec ? block_quant_kernel<FMT, true, EXPORT, SH, T> : block_quant_kernel<FMT, false, EXPORT, SH, T>;
  QSB_CUDA_TRY(launch_k(kern, dim3((unsigned)tiles), dim3(QSB_THREADS), 0, stream, x, y, codes, scales, L,
                        blocks_per_row, n_slots, tensor_amax));
  return 0;
}

template <bool EXPORT>
int block_entry(const void *x, int x_dtype, float *y, uint8_t *codes, uint8_t *scales, int64_t rows, int64_t L,
                int fmt, const float *tensor_amax, void *stream) {
  if (!dtype_ok(x_dtype) || fmt < kMXFP8 || fmt > kNVFP4) return QSB_E_BADARG;
  if (rows < 0 || L < 0) return QSB_E_BADARG;
  if (rows == 0 || L == 0) return 0;
  if (rows > INT64_MAX / 64 / L) return QSB_E_BADARG;
  if (!x || (EXPORT ? (!codes || !scales) : !y)) return QSB_E_BADARG;
  if (fmt == kNVFP4 && !tensor_amax) return QSB_E_BADARG;
  const int esize = x_dtype == QSB_DTYPE_F32 ? 4 : 2;
  if (!aligned_to(x, esize) || (!EXPORT && !aligned_to(y, 4))) return QSB_E_ALIGN;
  cudaStream_t s = (cudaStream_t)stream;
  // y stores bypass the L2 (evict_first) when the output cannot stay there anyway, as the other forwards do
  const bool big = !EXPORT && rows * L * 4 >= kStreamStoreBytes;
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    const T *xt = static_cast<const T *>(x);
    auto go = [&](auto fc) {
      constexpr int F = decltype(fc)::value;
      if (big) return launch_block<F, EXPORT, Hint::STREAM>(xt, y, codes, scales, rows, L, tensor_amax, s);
      return launch_block<F, EXPORT, Hint::KEEP>(xt, y, codes, scales, rows, L, tensor_amax, s);
    };
    switch (fmt) {
      case kMXFP8: return go(std::integral_constant<int, kMXFP8>{});
      case kMXFP4: return go(std::integral_constant<int, kMXFP4>{});
      default: return go(std::integral_constant<int, kNVFP4>{});
    }
  });
}

}  // namespace
}  // namespace qsb

using namespace qsb;

extern "C" int qsb_fq_block_fwd_dt(const void *x, int x_dtype, float *y, int64_t rows, int64_t L, int fmt,
                                   const float *tensor_amax_dev, void *stream) {
  return block_entry<false>(x, x_dtype, y, nullptr, nullptr, rows, L, fmt, tensor_amax_dev, stream);
}

extern "C" int qsb_block_export_dt(const void *x, int x_dtype, uint8_t *codes, uint8_t *scales, int64_t rows,
                                   int64_t L, int fmt, const float *tensor_amax_dev, void *stream) {
  return block_entry<true>(x, x_dtype, nullptr, codes, scales, rows, L, fmt, tensor_amax_dev, stream);
}
