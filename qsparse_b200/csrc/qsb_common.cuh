// Shared device/host helpers for the qsparse_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "../../include/qsparse_b200.h"

#ifndef QSB_THREADS
#define QSB_THREADS 256
#endif

namespace qsb {

// ---------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------
#define QSB_CUDA_TRY(expr)                      \
  do {                                          \
    cudaError_t _e = (expr);                    \
    if (_e != cudaSuccess) return (int)_e;      \
  } while (0)

#define QSB_LAUNCH_CHECK()                      \
  do {                                          \
    cudaError_t _e = cudaPeekAtLastError();     \
    if (_e != cudaSuccess) return (int)_e;      \
  } while (0)

struct DeviceProps {
  int sm_count;
  int64_t l2_bytes;
};
// Cached per device (queried once; never synchronises).
const DeviceProps &device_props();

__host__ __device__ inline bool aligned_to(const void *p, uintptr_t a) {
  return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0;
}

// ---------------------------------------------------------------------------
// programmatic dependent launch (PDL): a kernel launched with launch_pdl() may become
// resident while its predecessor in the stream is still running; it must execute
// pdl_wait() before it touches anything the predecessor writes (the wait returns when the
// predecessor grid has completed and its writes are visible).  A predecessor calls
// pdl_trigger() once it no longer minds the successor's CTAs occupying free SM resources.
// Both are no-ops in a kernel launched the ordinary way.
// ---------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

template <class... KArgs, class... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Launch policy of the streaming / reduction / parameter kernels (tuning key 12): with PDL
// every such kernel starts with pdl_wait(), so it is ordered after ANY predecessor in the
// stream exactly like an ordinary launch, but its launch latency and CTA ramp-up overlap
// the predecessor's tail.
bool pdl_enabled();
void set_pdl_enabled(int v);

template <class... KArgs, class... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                            cudaStream_t stream, Args... args) {
  if (pdl_enabled()) return launch_pdl(kernel, grid, block, smem, stream, args...);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// ---------------------------------------------------------------------------
// development only (-DQSB_KERNEL_TIMING): first-CTA-start / last-CTA-end %globaltimer stamps of the streaming
// kernels, per SM (one atomic per CTA and SM slot), so that the in-situ duration of every kernel of a
// graph-replayed step — and the gaps between them — can be read without event records (which undo the
// programmatic-dependent-launch overlap).  Slots: 0 = statistics kernel, 1 = forward map, 2 = backward map.
// ---------------------------------------------------------------------------
#ifdef QSB_KERNEL_TIMING
// (no relocatable device code: every translation unit has its own copy; qsb_debug_kernel_times collects them)
static __device__ unsigned long long g_ktime[3][2][256];
// reset (out == nullptr) or read this translation unit's copy
static inline int ktime_host_op(unsigned long long *out, cudaStream_t stream) {
  static unsigned long long init[3][2][256];
  if (!out) {
    for (int k = 0; k < 3; ++k)
      for (int s = 0; s < 256; ++s) init[k][0][s] = ~0ull, init[k][1][s] = 0ull;
    return (int)cudaMemcpyToSymbolAsync(g_ktime, init, sizeof(init), 0, cudaMemcpyHostToDevice, stream);
  }
  return (int)cudaMemcpyFromSymbol(out, g_ktime, sizeof(init));
}
__device__ __forceinline__ unsigned long long ktime_now() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void ktime_begin(int id) {
  if (threadIdx.x == 0) {
    unsigned smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    atomicMin(&g_ktime[id][0][smid & 255], ktime_now());
  }
}
__device__ __forceinline__ void ktime_end(int id) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    atomicMax(&g_ktime[id][1][smid & 255], ktime_now());
  }
}
#else
__device__ __forceinline__ void ktime_begin(int) {}
__device__ __forceinline__ void ktime_end(int) {}
#endif

// ---------------------------------------------------------------------------
// vector global-memory access.  V floats per access: 8 -> one 256-bit
// LDG/STG (new on sm_100), 4 -> 128-bit, 1 -> scalar.
// Loads: L1::no_allocate (every element is touched once per kernel); not .nc,
// because several ops run in place (STE backward, EMA) and the read-only path
// must not be used on memory the same kernel writes.
//   KEEP  : default L2 policy  (a following pass may hit L2)
//   STREAM: L2::evict_first    (nothing re-reads it; PTX allows the L2 level
//           qualifier on the 256-bit forms only, 128-bit accesses ignore it)
// Stores: L1::no_allocate; STREAM adds L2::evict_first so a write-once output
// does not push re-usable input lines out of the 126 MB L2.
// ---------------------------------------------------------------------------
enum class Hint { KEEP, STREAM };

template <int V>
struct VecF {
  float v[V];
};

template <int V, Hint H>
__device__ __forceinline__ VecF<V> ld_vec(const float *p) {
  VecF<V> r;
  if constexpr (V == 8) {
    if constexpr (H == Hint::STREAM) {
      asm volatile(
          "ld.global.L1::no_allocate.L2::evict_first.v8.f32 "
          "{%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
          : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]),
            "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
          : "l"(p));
    } else {
      asm volatile(
          "ld.global.L1::no_allocate.v8.f32 "
          "{%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
          : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]),
            "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]), "=f"(r.v[7])
          : "l"(p));
    }
  } else if constexpr (V == 4) {
    if constexpr (H == Hint::STREAM) {
      asm volatile(
          "ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
          : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3])
          : "l"(p));
    } else {
      asm volatile(
          "ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
          : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3])
          : "l"(p));
    }
  } else {
    static_assert(V == 1, "V must be 1, 4 or 8");
    r.v[0] = __ldg(p);
  }
  return r;
}

template <int V, Hint H>
__device__ __forceinline__ void st_vec(float *p, const VecF<V> &r) {
  if constexpr (V == 8) {
    if constexpr (H == Hint::STREAM) {
      asm volatile(
          "st.global.L1::no_allocate.L2::evict_first.v8.f32 [%0], "
          "{%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p),
          "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]), "f"(r.v[3]), "f"(r.v[4]),
          "f"(r.v[5]), "f"(r.v[6]), "f"(r.v[7])
          : "memory");
    } else {
      asm volatile(
          "st.global.L1::no_allocate.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p),
          "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]), "f"(r.v[3]), "f"(r.v[4]),
          "f"(r.v[5]), "f"(r.v[6]), "f"(r.v[7])
          : "memory");
    }
  } else if constexpr (V == 4) {
    if constexpr (H == Hint::STREAM) {
      asm volatile(
          "st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p),
          "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]), "f"(r.v[3])
          : "memory");
    } else {
      asm volatile(
          "st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p),
          "f"(r.v[0]), "f"(r.v[1]), "f"(r.v[2]), "f"(r.v[3])
          : "memory");
    }
  } else {
    p[0] = r.v[0];
  }
}

// ---------------------------------------------------------------------------
// 16-bit activations (bf16 / fp16): V elements per access — 8 -> one 128-bit
// access — upcast into the same VecF<V>, so every op computes in fp32 exactly as
// on an fp32 input (bf16 -> fp32 and fp16 -> fp32 are exact).  Stores round
// to nearest even like torch's CUDA cast (__float2bfloat16_rn / __float2half_rn).
// The L2 level qualifier is only legal on 256-bit accesses: STREAM loads and
// stores of 16-bit data use the default L2 policy, like the 128-bit fp32 forms.
// ---------------------------------------------------------------------------
__device__ __forceinline__ float to_f(float v) { return v; }
__device__ __forceinline__ float to_f(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f(__half v) { return __half2float(v); }
__device__ __forceinline__ void st1(float *p, float v) { *p = v; }
__device__ __forceinline__ void st1(__nv_bfloat16 *p, float v) { *p = __float2bfloat16_rn(v); }
__device__ __forceinline__ void st1(__half *p, float v) { *p = __float2half_rn(v); }

// two packed 16-bit values (element 0 in the low half) -> two floats
__device__ __forceinline__ void unpack2(uint32_t w, const __nv_bfloat16 *, float &a, float &b) {
  a = __uint_as_float(w << 16);
  b = __uint_as_float(w & 0xffff0000u);
}
__device__ __forceinline__ void unpack2(uint32_t w, const __half *, float &a, float &b) {
  a = __half2float(__ushort_as_half((unsigned short)(w & 0xffffu)));
  b = __half2float(__ushort_as_half((unsigned short)(w >> 16)));
}
__device__ __forceinline__ uint32_t pack2(float a, float b, const __nv_bfloat16 *) {
  return (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(a)) |
         ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(b)) << 16);
}
__device__ __forceinline__ uint32_t pack2(float a, float b, const __half *) {
  return (uint32_t)__half_as_ushort(__float2half_rn(a)) | ((uint32_t)__half_as_ushort(__float2half_rn(b)) << 16);
}

template <class T>
inline constexpr bool is_half16 = std::is_same<T, __nv_bfloat16>::value || std::is_same<T, __half>::value;

// 8 packed 16-bit values as one 128-bit load; kept packed (4 registers instead of 8) until unpack8()
__device__ __forceinline__ uint4 ld_raw16(const void *p) {
  uint4 w;
  asm volatile("ld.global.L1::no_allocate.v4.b32 {%0,%1,%2,%3}, [%4];"
               : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w)
               : "l"(p));
  return w;
}
template <class T>
__device__ __forceinline__ VecF<8> unpack8(const uint4 &w) {
  VecF<8> r;
  unpack2(w.x, (const T *)nullptr, r.v[0], r.v[1]);
  unpack2(w.y, (const T *)nullptr, r.v[2], r.v[3]);
  unpack2(w.z, (const T *)nullptr, r.v[4], r.v[5]);
  unpack2(w.w, (const T *)nullptr, r.v[6], r.v[7]);
  return r;
}

template <int V, Hint H, class T, std::enable_if_t<is_half16<T>, int> = 0>
__device__ __forceinline__ VecF<V> ld_vec(const T *p) {
  VecF<V> r;
  if constexpr (V == 8) {
    r = unpack8<T>(ld_raw16(p));
  } else if constexpr (V == 4) {
    uint32_t w[2];
    asm volatile("ld.global.L1::no_allocate.v2.b32 {%0,%1}, [%2];" : "=r"(w[0]), "=r"(w[1]) : "l"(p));
    unpack2(w[0], p, r.v[0], r.v[1]);
    unpack2(w[1], p, r.v[2], r.v[3]);
  } else {
    static_assert(V == 1, "V must be 1, 4 or 8");
    r.v[0] = to_f(p[0]);
  }
  return r;
}

template <int V, Hint H, class T, std::enable_if_t<is_half16<T>, int> = 0>
__device__ __forceinline__ void st_vec(T *p, const VecF<V> &r) {
  if constexpr (V == 8) {
    uint32_t w[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) w[k] = pack2(r.v[2 * k], r.v[2 * k + 1], (const T *)nullptr);
    asm volatile("st.global.L1::no_allocate.v4.b32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(w[0]), "r"(w[1]),
                 "r"(w[2]), "r"(w[3])
                 : "memory");
  } else if constexpr (V == 4) {
    const uint32_t w0 = pack2(r.v[0], r.v[1], (const T *)nullptr), w1 = pack2(r.v[2], r.v[3], (const T *)nullptr);
    asm volatile("st.global.L1::no_allocate.v2.b32 [%0], {%1,%2};" ::"l"(p), "r"(w0), "r"(w1) : "memory");
  } else {
    st1(p, r.v[0]);
  }
}

// 8 elements of a vector whose 16-byte alignment is only known at run time (a 16-bit view may start at
// any even byte address): one 128-bit load when it is aligned, else element by element.
template <Hint H, class T>
__device__ __forceinline__ VecF<8> ld_vec8_any(const T *p, bool vec_ok) {
  if constexpr (!is_half16<T>) {
    return ld_vec<8, H>(p);
  } else {
    if (vec_ok) return ld_vec<8, H>(p);
    VecF<8> r;
#pragma unroll
    for (int j = 0; j < 8; ++j) r.v[j] = to_f(p[j]);
    return r;
  }
}

// dtype codes of the C-ABI (QSB_DTYPE_*) -> element type; any other code is QSB_E_BADARG
inline bool dtype_ok(int dt) { return dt == QSB_DTYPE_F32 || dt == QSB_DTYPE_BF16 || dt == QSB_DTYPE_F16; }
template <class F>
inline int dispatch_dtype(int dt, F &&f) {
  switch (dt) {
    case QSB_DTYPE_F32: return f((float *)nullptr);
    case QSB_DTYPE_BF16: return f((__nv_bfloat16 *)nullptr);
    case QSB_DTYPE_F16: return f((__half *)nullptr);
    default: return QSB_E_BADARG;
  }
}

// V mask bytes (uint8 0/1) for V consecutive elements.
template <int V>
struct VecB {
  uint8_t b[V];
};

template <int V>
__device__ __forceinline__ VecB<V> ld_bytes(const uint8_t *p) {
  VecB<V> r;
  if constexpr (V == 8) {
    uint2 w = __ldg(reinterpret_cast<const uint2 *>(p));
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      r.b[j] = (w.x >> (8 * j)) & 0xff;
      r.b[4 + j] = (w.y >> (8 * j)) & 0xff;
    }
  } else if constexpr (V == 4) {
    uint32_t w = __ldg(reinterpret_cast<const uint32_t *>(p));
#pragma unroll
    for (int j = 0; j < 4; ++j) r.b[j] = (w >> (8 * j)) & 0xff;
  } else {
    r.b[0] = __ldg(p);
  }
  return r;
}

template <int V>
__device__ __forceinline__ void st_bytes(uint8_t *p, const VecB<V> &r) {
  if constexpr (V == 8) {
    uint2 w;
    w.x = r.b[0] | (r.b[1] << 8) | (r.b[2] << 16) | ((uint32_t)r.b[3] << 24);
    w.y = r.b[4] | (r.b[5] << 8) | (r.b[6] << 16) | ((uint32_t)r.b[7] << 24);
    *reinterpret_cast<uint2 *>(p) = w;
  } else if constexpr (V == 4) {
    uint32_t w =
        r.b[0] | (r.b[1] << 8) | (r.b[2] << 16) | ((uint32_t)r.b[3] << 24);
    *reinterpret_cast<uint32_t *>(p) = w;
  } else {
    p[0] = r.b[0];
  }
}

// ---------------------------------------------------------------------------
// exact arithmetic helpers (every ATen op in the reference rounds separately:
// no FMA contraction, IEEE division, SURVEY Q7)
// ---------------------------------------------------------------------------

// 2^d for a float d the way torch.pow(2.0, d) gives it for integral d: exact,
// including subnormal results and overflow to inf.  Non-integral d -> exp2f.
__device__ __forceinline__ float pow2f_exact(float d) {
  if (d == rintf(d) && fabsf(d) < 400.f) return ldexpf(1.0f, (int)d);
  return exp2f(d);  // also +-inf and NaN
}

// torch.clamp(v, lo, hi) with scalar/tensor bounds: NaN in v propagates,
// lo > hi gives hi (min(max(v, lo), hi)).
__device__ __forceinline__ float clamp_torch(float v, float lo, float hi) {
  float t = (v < lo) ? lo : v;
  return (t > hi) ? hi : t;
}

// x / s, correctly rounded (== __fdiv_rn), for a divisor that is shared by many
// elements: r = RN(1/s) is computed once per channel (__frcp_rn) and the quotient
// is refined with two exact-residual FMA steps (Markstein: with a correctly
// rounded reciprocal and a faithful quotient estimate, q + (x - s*q)*r rounds to
// RN(x/s)).  No MUFU / FCHK per element.  The fast path is taken when no
// intermediate can overflow or lose bits to underflow: s_ok <=> |s| in
// [2^-40, 2^40] (checked once per channel), |x| in [2^-64, 2^64) or x == 0;
// everything else goes through __fdiv_rn.  tests: qsb_selftest_fastdiv.
__device__ __forceinline__ bool fastdiv_divisor_ok(float s) {
  const uint32_t as = __float_as_uint(s) & 0x7fffffffu;
  return (as - 0x2b800000u) < 0x28000000u;  // exponent field in [87, 167)
}
__device__ __forceinline__ float div_rn_by(float x, float s, float r, bool s_ok) {
  const uint32_t ax = __float_as_uint(x) & 0x7fffffffu;
  if (s_ok && (((ax - 0x1f800000u) < 0x40000000u) || ax == 0u)) {
    const float q0 = __fmul_rn(x, r);
    float e = __fmaf_rn(-s, q0, x);
    float q = __fmaf_rn(e, r, q0);
    e = __fmaf_rn(-s, q, x);
    q = __fmaf_rn(e, r, q);
    return ax == 0u ? q0 : q;  // keeps the sign of a zero quotient
  }
  return __fdiv_rn(x, s);
}

// The same refinement without any range check: the caller guarantees s_ok and
// |x| < 2^64.  Tiny x needs no guard when the quotient only feeds a rounding to
// integer: a residual that underflows leaves q ~ q0, |q| << 0.5, which rounds to 0
// exactly like the true quotient.
__device__ __forceinline__ float div_rn_by_unchecked(float x, float s, float r) {
  const float q0 = __fmul_rn(x, r);
  float e = __fmaf_rn(-s, q0, x);
  float q = __fmaf_rn(e, r, q0);
  e = __fmaf_rn(-s, q, x);
  q = __fmaf_rn(e, r, q);
  return (x == 0.0f) ? q0 : q;
}
// For quotients that are rounded to an integer next: one upper-bound compare.
__device__ __forceinline__ float div_rn_by_q(float x, float s, float r, bool s_ok) {
  if (s_ok && fabsf(x) < 1.8446744e19f)  // 2^64; false for NaN / inf
    return div_rn_by_unchecked(x, s, r);
  return __fdiv_rn(x, s);
}

// order-preserving float -> uint32 key; every NaN maps to the largest key so
// NaNs order last like torch.sort.
__device__ __forceinline__ uint32_t float_to_key(float f) {
  uint32_t b = __float_as_uint(f);
  if ((b & 0x7fffffffu) > 0x7f800000u) return 0xffffffffu;
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float key_to_float(uint32_t k) {
  if (k == 0xffffffffu) return __uint_as_float(0x7fc00000u);
  uint32_t b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
  return __uint_as_float(b);
}

// ---------------------------------------------------------------------------
// flat element index -> (column in row, channel) without divisions in the loop
// ---------------------------------------------------------------------------
struct Layout {
  int64_t outer, channels, inner;
  __host__ __device__ int64_t numel() const { return outer * channels * inner; }
};

struct ChanPos {
  int64_t col;  // position inside the current row, [0, inner)
  int32_t c;    // channel, [0, channels)
};

__device__ __forceinline__ ChanPos chan_pos_of(int64_t e, const Layout &L) {
  ChanPos p;
  int64_t row = e / L.inner;
  p.col = e - row * L.inner;
  p.c = (int32_t)(row % L.channels);
  return p;
}

// Constant advance of a ChanPos by `step` elements (step_rows = step / inner
// reduced mod channels, step_cols = step % inner; both precomputed on the host).
struct ChanStep {
  int64_t cols;
  int32_t chans;
};
inline ChanStep make_chan_step(int64_t step, const Layout &L) {
  ChanStep s;
  s.cols = step % L.inner;
  s.chans = (int32_t)((step / L.inner) % L.channels);
  return s;
}
__device__ __forceinline__ void advance(ChanPos &p, const ChanStep &s,
                                        const Layout &L) {
  p.col += s.cols;
  p.c += s.chans;
  if (p.col >= L.inner) {
    p.col -= L.inner;
    p.c += 1;
  }
  if (p.c >= (int32_t)L.channels) p.c -= (int32_t)L.channels;
  if (p.c >= (int32_t)L.channels) p.c -= (int32_t)L.channels;
}

// ---------------------------------------------------------------------------
// warp reductions
// ---------------------------------------------------------------------------
template <class T, class F>
__device__ __forceinline__ T warp_reduce(T v, F f) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = f(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace qsb
