// Streaming elementwise "map" kernels shared by every fake-quant / STE / mask op.
//
// HBM-bound: 4 B read + 4 B written per element and per stream; nothing is staged
// in shared memory because no element is touched twice.  Each thread moves U
// vectors of V floats per step: all loads are issued first (U x 32 B in flight
// per thread), then the arithmetic, then the stores.
//
//   map_kernel       per-tensor parameters.  One CTA per tile (measured on B200:
//                    6.18 TB/s vs 5.65 TB/s for a persistent grid, profiles/).
//   map_chan_win_kernel  per-channel parameters ([outer, C, inner]), inner >= V.
//                    One CTA per tile, like the per-tensor kernel (persistent
//                    grids run their warps in lock-step load/compute phases and
//                    measured 4-9 % slower, profiles/).  The CTA derives the
//                    per-channel constants (2^d, reciprocals, clamp bounds, mask)
//                    only for the rows its tile touches — a "window" table of
//                    tile/inner + 2 entries in shared memory, independent of C —
//                    then every vector needs one 32-bit division to find its row.
//                    MODE 0: inner % V == 0, a vector never straddles two rows;
//                    MODE 1: a vector touches at most two channels.
//   map_chan_kernel  rows shorter than a vector (inner < V, MODE 2: walk the
//                    channels element by element) and unaligned pointers.
//                    Persistent grid, full per-channel table in shared memory
//                    when it fits, 32-bit (column, channel) bookkeeping advanced
//                    by constants — no division in the loop.
#pragma once
#include <type_traits>

#include "qsb_common.cuh"

namespace qsb {

// TI: element type of in0, TO0 / TO1: of out0 / out1 (float, or __nv_bfloat16 / __half for 16-bit
// activations and their gradients); the ops always compute in fp32.
template <class TI = float, class TO0 = float, class TO1 = float>
struct MapIOT {
  const TI *in0;
  const float *in1;
  const uint8_t *inb;
  TO0 *out0;
  TO1 *out1;
  uint8_t *outb;
};
using MapIO = MapIOT<>;

// Op requirements:
//   struct P;                                  per-channel derived constants
//   static constexpr bool kIn1, kInB, kOut0, kOut1, kOutB, kCanSkip, kHasFast;
//   __device__ P params(int32_t c) const;
//   __device__ bool skip(const P&) const;      (kCanSkip) output independent of in0
//   __device__ void apply(float a, float b, uint8_t mb, const P&,
//                         float &o0, float &o1, uint8_t &ob) const;

// One vector of V elements that all use the same per-channel constants.  Ops with
// a cheaper arithmetic path that is only valid on part of the input domain expose
// it as apply_fast() and decide ONCE per vector (fast()), so the generic IEEE path
// is not inlined behind a branch for every element.
template <class Op, int V>
__device__ __forceinline__ void apply_vec(const Op &op, const VecF<V> &a,
                                          const VecF<V> &b, const VecB<V> &mb,
                                          bool skip, const typename Op::P &p,
                                          VecF<V> &o0, VecF<V> &o1, VecB<V> &ob) {
  if constexpr (Op::kHasFast) {
    if (op.template fast<V>(p, a.v)) {
#pragma unroll
      for (int j = 0; j < V; ++j)
        op.apply_fast(skip ? 0.f : a.v[j], Op::kIn1 ? b.v[j] : 0.f,
                      Op::kInB ? mb.b[j] : (uint8_t)1, p, o0.v[j], o1.v[j], ob.b[j]);
      return;
    }
  }
#pragma unroll
  for (int j = 0; j < V; ++j)
    op.apply(skip ? 0.f : a.v[j], Op::kIn1 ? b.v[j] : 0.f,
             Op::kInB ? mb.b[j] : (uint8_t)1, p, o0.v[j], o1.v[j], ob.b[j]);
}

// Byte outputs are one byte per element (masks, int8 codes) or, for ops that declare
// `static constexpr bool kPack4 = true`, one NIBBLE per element (packed 4-bit codes, element 2i in the
// low nibble of byte i): a vector of 8 codes is then ONE 32-bit store.
template <class Op, class = void>
struct is_pack4 : std::false_type {};
template <class Op>
struct is_pack4<Op, std::void_t<decltype(Op::kPack4)>> : std::bool_constant<Op::kPack4> {};

template <class Op, int V>
__device__ __forceinline__ void store_outb(uint8_t *outb, int64_t e, const VecB<V> &ob) {
  if constexpr (is_pack4<Op>::value) {
    if constexpr (V == 8) {
      uint32_t w = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) w |= (uint32_t)(ob.b[j] & 0xF) << (4 * j);
      *reinterpret_cast<uint32_t *>(outb + (e >> 1)) = w;
    } else if constexpr (V == 4) {
      uint16_t w = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) w |= (uint16_t)((ob.b[j] & 0xF) << (4 * j));
      *reinterpret_cast<uint16_t *>(outb + (e >> 1)) = w;
    }
    // V == 1 would make two threads share a byte: the launcher never picks it for a packed output
  } else {
    st_bytes<V>(outb + e, ob);
  }
}

struct MapTuning {
  int ctas_per_sm;   // per-tensor kernel: 0 = one CTA per tile (default); >0 persistent
  int chan_ctas_per_sm;  // channel kernel: 0 = occupancy-derived persistent grid
  // Tile order of the one-CTA-per-tile kernels.  1 (default): last tile first.  The
  // tensor a streaming kernel reads was normally just produced / reduced front to
  // back, so its TAIL is what still sits in the 126 MB L2; walking backwards turns
  // up to ~100 MB of the second pass into L2 hits instead of HBM reads.
  int reverse_tiles;
  int lastdim;  // 1 (default): channel-last layouts use the group-resident kernel; 0: the MODE 2 walk
};
MapTuning &map_tuning();

// reverse_tiles: 0 never, 1 (default) every map kernel EXCEPT the channel-masked ones, 2 always.  The masked
// forward / backward follow the fused statistics kernel, which has already tagged the kept channels
// L2::evict_last: there the natural order measured 3 us faster on the bench step (20.7 vs 25.5 MB of DRAM reads
// in the forward, profiles/r02_tile_order.json), while the untagged pair {statistics -> quantize} gains 4 us
// from walking backwards at every size above ~90 MB.
template <class Op>
inline int reverse_for() {
  const int v = map_tuning().reverse_tiles;
  return (v == 2 || (v == 1 && !Op::kCanSkip)) ? 1 : 0;
}

// ---------------------------------------------------------------------------
// per-tensor
// ---------------------------------------------------------------------------
template <class Op, int V, int U, Hint LH, Hint SH, class IO>
__global__ void __launch_bounds__(QSB_THREADS)
    map_kernel(Op op, IO io, int64_t n, int reverse) {
  pdl_wait();
  pdl_trigger();
  using P = typename Op::P;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  constexpr int64_t kStrideU = (int64_t)QSB_THREADS * V;
  const int64_t n_main = (n / V) * V;
  const P p = op.params(0);
  // reverse is only set for one-CTA-per-tile launches (the loop then runs once)
  const int64_t first_tile = reverse ? (int64_t)(gridDim.x - 1 - blockIdx.x) : (int64_t)blockIdx.x;

  for (int64_t e_base = first_tile * kTile + (int64_t)threadIdx.x * V;
       e_base < n_main; e_base += (int64_t)gridDim.x * kTile) {
    VecF<V> a[U], b[U];
    VecB<V> mb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = e_base + u * kStrideU;
      if (e < n_main) {
        a[u] = ld_vec<V, LH>(io.in0 + e);
        if constexpr (Op::kIn1) b[u] = ld_vec<V, LH>(io.in1 + e);
        if constexpr (Op::kInB) mb[u] = ld_bytes<V>(io.inb + e);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = e_base + u * kStrideU;
      if (e < n_main) {
        VecF<V> o0, o1;
        VecB<V> ob;
        apply_vec<Op, V>(op, a[u], b[u], mb[u], false, p, o0, o1, ob);
        if constexpr (Op::kOut0) st_vec<V, SH>(io.out0 + e, o0);
        if constexpr (Op::kOut1) st_vec<V, SH>(io.out1 + e, o1);
        if constexpr (Op::kOutB) store_outb<Op, V>(io.outb, e, ob);
      }
    }
  }
  // tail: the last n % V elements, scalar, by block 0
  if (blockIdx.x == 0) {
    const int64_t e = n_main + threadIdx.x;
    if (e < n) {
      float o0, o1;
      uint8_t ob;
      op.apply(to_f(io.in0[e]), Op::kIn1 ? io.in1[e] : 0.f,
               Op::kInB ? io.inb[e] : (uint8_t)1, p, o0, o1, ob);
      if constexpr (Op::kOut0) st1(io.out0 + e, o0);
      if constexpr (Op::kOut1) st1(io.out1 + e, o1);
      if constexpr (Op::kOutB) io.outb[e] = ob;
    }
  }
}

template <class Op, int V, int U, Hint LH, Hint SH, class IO>
int launch_map_tensor(const Op &op, const IO &io, int64_t n,
                      cudaStream_t stream) {
  auto kern = map_kernel<Op, V, U, LH, SH, IO>;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  const int64_t tiles = (n + kTile - 1) / kTile;
  int64_t grid = tiles;
  const int per_sm = map_tuning().ctas_per_sm;
  if (per_sm > 0) {
    grid = (int64_t)device_props().sm_count * per_sm;
    if (grid > tiles) grid = tiles;
  }
  if (grid > 0x7fffffffLL) grid = 0x7fffffffLL;  // the kernel loops
  const int reverse = (grid == tiles && reverse_for<Op>()) ? 1 : 0;
  QSB_CUDA_TRY(launch_k(kern, dim3((unsigned)grid), dim3(QSB_THREADS), 0, stream, op, io, n, reverse));
  return 0;
}

// ---------------------------------------------------------------------------
// multi-tensor: one launch applies a per-tensor op to many separate tensors (the layers of
// a weight set).  The tensors' pointers, sizes and first tile live in a table in the kernel
// parameters; a CTA owns one tile and finds its tensor by binary search (<= 6 steps,
// uniform over the CTA).  A [512,512,3,3] layer alone is a 10 us launch of which half is
// ramp-up and tail; 29 of them in one grid stream like one 268 MB tensor.
// ---------------------------------------------------------------------------
constexpr int kMultiMax = 48;
struct MultiEntry {
  const float *in0, *in1;
  float *out0;
  uint8_t *outb;
  const float *aux;  // per-tensor op argument (Op::bind), e.g. the layer's threshold
  int64_t n;
  int64_t tile0;     // index of the tensor's first tile in the grid
};
struct MultiTable {
  MultiEntry e[kMultiMax];
  int count;
};

template <class Op, int U, Hint LH, Hint SH>
__global__ void __launch_bounds__(QSB_THREADS)
    map_multi_kernel(const __grid_constant__ MultiTable tab, Op op) {
  pdl_wait();
  pdl_trigger();
  constexpr int V = 8;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  constexpr int64_t kStrideU = (int64_t)QSB_THREADS * V;
  int lo = 0, hi = tab.count - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (tab.e[mid].tile0 <= (int64_t)blockIdx.x) lo = mid;
    else hi = mid - 1;
  }
  const MultiEntry &t = tab.e[lo];
  op.bind(t.aux);
  const typename Op::P p = op.params(0);
  const int64_t n = t.n, n_main = (n / V) * V;
  const int64_t tile = (int64_t)blockIdx.x - t.tile0;
  const int64_t e_base = tile * kTile + (int64_t)threadIdx.x * V;
  VecF<V> a[U], b[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t e = e_base + u * kStrideU;
    if (e < n_main) {
      a[u] = ld_vec<V, LH>(t.in0 + e);
      if constexpr (Op::kIn1) b[u] = ld_vec<V, LH>(t.in1 + e);
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t e = e_base + u * kStrideU;
    if (e < n_main) {
      VecF<V> o0, o1;
      VecB<V> mb, ob;
      apply_vec<Op, V>(op, a[u], b[u], mb, false, p, o0, o1, ob);
      if constexpr (Op::kOut0) st_vec<V, SH>(t.out0 + e, o0);
      if constexpr (Op::kOutB) store_outb<Op, V>(t.outb, e, ob);
    }
  }
  // the last n % V elements of the tensor, scalar, by the CTA that owns that position
  if (n_main < n && tile == n_main / kTile) {
    const int64_t e = n_main + threadIdx.x;
    if (e < n) {
      float o0, o1;
      uint8_t ob;
      op.apply(t.in0[e], Op::kIn1 ? t.in1[e] : 0.f, (uint8_t)1, p, o0, o1, ob);
      if constexpr (Op::kOut0) t.out0[e] = o0;
      if constexpr (Op::kOutB) t.outb[e] = ob;
    }
  }
}

// entries[0..count): launches ceil(count / kMultiMax) grids.  Every pointer must be 32-byte
// aligned (the caller checks and otherwise falls back to one launch per tensor).
template <class Op, Hint LH, Hint SH>
int launch_map_multi(const Op &op, const MultiEntry *entries, int count, cudaStream_t stream) {
  static_assert(!Op::kInB && !Op::kOut1, "multi-tensor map: in0 [, in1] -> out0 [, outb]");
  constexpr int U = 2;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * 8 * U;
  for (int first = 0; first < count; first += kMultiMax) {
    MultiTable tab;
    tab.count = count - first < kMultiMax ? count - first : kMultiMax;
    int64_t tiles = 0;
    for (int i = 0; i < tab.count; ++i) {
      tab.e[i] = entries[first + i];
      tab.e[i].tile0 = tiles;
      // a tensor whose size is a multiple of the tile still needs no extra CTA for a tail
      tiles += (tab.e[i].n + kTile - 1) / kTile;
    }
    if (tiles == 0) continue;
    if (tiles > 0x7fffffffLL) return QSB_E_UNSUPPORTED;
    auto kern = map_multi_kernel<Op, U, LH, SH>;
    QSB_CUDA_TRY(launch_k(kern, dim3((unsigned)tiles), dim3(QSB_THREADS), 0, stream, tab, op));
  }
  return 0;
}

// ---------------------------------------------------------------------------
// per-channel
// ---------------------------------------------------------------------------
struct ChanGeom {
  uint32_t inner, channels;
  uint32_t su_cols, su_ch;  // advance by one vector stride (QSB_THREADS * V)
  uint32_t si_cols, si_ch;  // advance by one grid stride
  int use_table;
};

__device__ __forceinline__ void advance32(uint32_t &col, uint32_t &c,
                                          uint32_t dcol, uint32_t dch,
                                          const ChanGeom &G) {
  col += dcol;
  c += dch;
  if (col >= G.inner) {
    col -= G.inner;
    c += 1;
  }
  if (c >= G.channels) c -= G.channels;
}

template <class Op, int V, int U, int MODE, Hint LH, Hint SH, class IO>
__global__ void __launch_bounds__(QSB_THREADS)
    map_chan_kernel(Op op, IO io, int64_t n, ChanGeom G) {
  pdl_wait();
  pdl_trigger();
  using P = typename Op::P;
  extern __shared__ __align__(16) unsigned char qsb_smem_raw[];
  P *tab = reinterpret_cast<P *>(qsb_smem_raw);
  if (G.use_table) {
    for (uint32_t c = threadIdx.x; c < G.channels; c += QSB_THREADS)
      tab[c] = op.params((int32_t)c);
    __syncthreads();
  }
  auto param_of = [&](uint32_t c) -> P {
    return G.use_table ? tab[c] : op.params((int32_t)c);
  };

  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  constexpr int64_t kStrideU = (int64_t)QSB_THREADS * V;
  const int64_t n_main = (n / V) * V;

  int64_t e_base = (int64_t)blockIdx.x * kTile + (int64_t)threadIdx.x * V;
  uint32_t col0, c0;
  {
    const int64_t eb = e_base < n ? e_base : 0;
    const int64_t row = eb / G.inner;  // the only division: once per thread
    col0 = (uint32_t)(eb - row * G.inner);
    c0 = (uint32_t)(row % G.channels);
  }

  for (; e_base < n_main; e_base += (int64_t)gridDim.x * kTile) {
    VecF<V> a[U], b[U];
    VecB<V> mb[U];
    uint32_t cu[U], colu[U];
    bool skipv[U];
    uint32_t col = col0, c = c0;
    // ---- phase 1: positions, skip decision, loads ------------------------
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = e_base + u * kStrideU;
      cu[u] = c;
      colu[u] = col;
      skipv[u] = false;
      if (e < n_main) {
        if constexpr (Op::kCanSkip && MODE != 2) {
          bool s = op.skip(param_of(c));
          if (MODE == 1 && s && col + V > G.inner) {
            const uint32_t c1 = (c + 1 >= G.channels) ? 0 : c + 1;
            s = op.skip(param_of(c1));
          }
          skipv[u] = s;
        }
        if (!skipv[u]) a[u] = ld_vec<V, LH>(io.in0 + e);
        if constexpr (Op::kIn1) b[u] = ld_vec<V, LH>(io.in1 + e);
        if constexpr (Op::kInB) mb[u] = ld_bytes<V>(io.inb + e);
      }
      advance32(col, c, G.su_cols, G.su_ch, G);
    }
    // ---- phase 2: arithmetic + stores ------------------------------------
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = e_base + u * kStrideU;
      if (e < n_main) {
        VecF<V> o0, o1;
        VecB<V> ob;
        if constexpr (MODE == 2) {
          uint32_t qc = cu[u], qcol = colu[u];
#pragma unroll
          for (int j = 0; j < V; ++j) {
            const P pj = param_of(qc);
            op.apply(a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                     Op::kInB ? mb[u].b[j] : (uint8_t)1, pj, o0.v[j], o1.v[j],
                     ob.b[j]);
            if (++qcol >= G.inner) {
              qcol = 0;
              if (++qc >= G.channels) qc = 0;
            }
          }
        } else {
          const P p0 = param_of(cu[u]);
          const uint32_t left = G.inner - colu[u];  // elements left in this row
          if (MODE == 0 || left >= (uint32_t)V) {
            apply_vec<Op, V>(op, a[u], b[u], mb[u], skipv[u], p0, o0, o1, ob);
          } else {
            const uint32_t c1 = (cu[u] + 1 >= G.channels) ? 0 : cu[u] + 1;
            const P p1 = param_of(c1);
            // a vector across two rows: still the cheap arithmetic when both rows allow it (with
            // 7x7 feature maps one vector in six straddles; the generic IEEE path on those alone
            // made the line quantizer 2.4x slower than the pow2 one)
            bool fast2 = Op::kHasFast;
            if constexpr (Op::kHasFast)
              fast2 = op.template fast<V>(p0, a[u].v) && op.template fast<V>(p1, a[u].v);
            if (fast2) {
              if constexpr (Op::kHasFast) {
#pragma unroll
                for (int j = 0; j < V; ++j)
                  op.apply_fast(skipv[u] ? 0.f : a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                                Op::kInB ? mb[u].b[j] : (uint8_t)1,
                                ((uint32_t)j < left) ? p0 : p1, o0.v[j], o1.v[j], ob.b[j]);
              }
            } else {
#pragma unroll
              for (int j = 0; j < V; ++j)
                op.apply(skipv[u] ? 0.f : a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                         Op::kInB ? mb[u].b[j] : (uint8_t)1,
                         ((uint32_t)j < left) ? p0 : p1, o0.v[j], o1.v[j], ob.b[j]);
            }
          }
        }
        if constexpr (Op::kOut0) st_vec<V, SH>(io.out0 + e, o0);
        if constexpr (Op::kOut1) st_vec<V, SH>(io.out1 + e, o1);
        if constexpr (Op::kOutB) store_outb<Op, V>(io.outb, e, ob);
      }
    }
    advance32(col0, c0, G.si_cols, G.si_ch, G);
  }

  // tail: the last n % V elements, scalar, by block 0
  if (blockIdx.x == 0) {
    const int64_t e = n_main + threadIdx.x;
    if (e < n) {
      const int64_t row = e / G.inner;
      const P pj = param_of((uint32_t)(row % G.channels));
      float o0, o1;
      uint8_t ob;
      op.apply(to_f(io.in0[e]), Op::kIn1 ? io.in1[e] : 0.f,
               Op::kInB ? io.inb[e] : (uint8_t)1, pj, o0, o1, ob);
      if constexpr (Op::kOut0) st1(io.out0 + e, o0);
      if constexpr (Op::kOut1) st1(io.out1 + e, o1);
      if constexpr (Op::kOutB) io.outb[e] = ob;
    }
  }
}

// ---------------------------------------------------------------------------
// per-channel, one CTA per tile, window table (inner >= V)
// ---------------------------------------------------------------------------
constexpr uint32_t kUnifyInner = 512;  // P(a warp holds a straddling vector) > ~0.35 below this row length
template <class Op, int V, int U, int MODE, Hint LH, Hint SH, class IO>
__global__ void __launch_bounds__(QSB_THREADS)
    map_chan_win_kernel(Op op, IO io, int64_t n, uint32_t inner,
                        uint32_t channels, int reverse) {
  pdl_wait();
  pdl_trigger();
  ktime_begin(Op::kOut1 ? 2 : 1);
  using P = typename Op::P;
  static_assert(MODE == 0 || MODE == 1, "window kernel needs inner >= V");
  extern __shared__ __align__(16) unsigned char qsb_smem_raw[];
  P *tab = reinterpret_cast<P *>(qsb_smem_raw);
  constexpr uint32_t kTile = QSB_THREADS * V * U;
  constexpr uint32_t kStrideU = QSB_THREADS * V;
  const int64_t n_main = (n / V) * V;
  const int64_t t0 =
      (int64_t)(reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x) * kTile;
  // first row / column / channel of the tile (uniform across the CTA); 32-bit divisions whenever the
  // tile starts below 2^32 (a 64-bit one is ~100 instructions, executed by every thread of every CTA:
  // with the prune mask folded in, three quarters of the bench tensor's CTAs only store zeros and
  // their ~300 instructions per warp made the kernel issue-bound, 61 % SM throughput in ncu)
  uint32_t col0, c0;
  if (t0 <= 0xffffffffLL) {
    const uint32_t row0 = (uint32_t)t0 / inner;
    col0 = (uint32_t)t0 - row0 * inner;
    c0 = row0 % channels;
  } else {
    const int64_t row0 = t0 / inner;
    col0 = (uint32_t)(t0 - row0 * inner);
    c0 = (uint32_t)(row0 % channels);
  }
  const uint32_t rows = (col0 + kTile - 1) / inner + 1;
  for (uint32_t k = threadIdx.x; k < rows; k += QSB_THREADS)
    tab[k] = op.params((int32_t)((c0 + k) % channels));
  __syncthreads();

  VecF<V> a[U], b[U];
  VecB<V> mb[U];
  uint32_t ru[U], leftu[U];
  bool skipv[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const uint32_t o = threadIdx.x * V + u * kStrideU;
    const int64_t e = t0 + o;
    const uint32_t pos = col0 + o;
    ru[u] = pos / inner;
    leftu[u] = inner - (pos - ru[u] * inner);  // elements left in this row
    skipv[u] = false;
    if (e < n_main) {
      if constexpr (Op::kCanSkip) {
        bool s = op.skip(tab[ru[u]]);
        if (MODE == 1 && s && leftu[u] < (uint32_t)V) s = op.skip(tab[ru[u] + 1]);
        skipv[u] = s;
      }
      if (!skipv[u]) a[u] = ld_vec<V, LH>(io.in0 + e);
      if constexpr (Op::kIn1) b[u] = ld_vec<V, LH>(io.in1 + e);
      if constexpr (Op::kInB) mb[u] = ld_bytes<V>(io.inb + e);
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t e = t0 + threadIdx.x * V + u * kStrideU;
    if (e < n_main) {
      VecF<V> o0, o1;
      VecB<V> ob;
      const P p0 = tab[ru[u]];
      if constexpr (Op::kCanSkip) {
        // a vector of a skipped (pruned) channel: its output is the op's value at 0 — the same for all 8
        // elements — so evaluate it once instead of eight times (and never touch the unread registers)
        if (skipv[u] && (MODE == 0 || leftu[u] >= (uint32_t)V)) {
          float z0 = 0.f, z1 = 0.f;
          uint8_t zb = 0;
          op.apply(0.f, 0.f, (uint8_t)1, p0, z0, z1, zb);
#pragma unroll
          for (int j = 0; j < V; ++j) o0.v[j] = z0, o1.v[j] = z1, ob.b[j] = zb;
          if constexpr (Op::kOut0) st_vec<V, SH>(io.out0 + e, o0);
          if constexpr (Op::kOut1) st_vec<V, SH>(io.out1 + e, o1);
          if constexpr (Op::kOutB) store_outb<Op, V>(io.outb, e, ob);
          continue;
        }
      }
      // Short rows: almost every warp holds a lane whose vector straddles two rows (one vector in six with 7x7
      // maps), so the two branches below would BOTH be issued for nearly every warp.  Below kUnifyInner the
      // per-element parameter select is therefore the only path (a few SELs per element, no divergence).
      const bool unify = MODE == 1 && inner < kUnifyInner;  // uniform across the grid
      if (MODE == 0 || (!unify && leftu[u] >= (uint32_t)V)) {
        apply_vec<Op, V>(op, a[u], b[u], mb[u], skipv[u], p0, o0, o1, ob);
      } else {
        const P p1 = tab[ru[u] + (leftu[u] < (uint32_t)V ? 1 : 0)];
        bool fast2 = Op::kHasFast;  // see map_chan_win_kernel: straddling vectors stay on the cheap path
        if constexpr (Op::kHasFast)
          fast2 = op.template fast<V>(p0, a[u].v) && op.template fast<V>(p1, a[u].v);
        if (fast2) {
          if constexpr (Op::kHasFast) {
#pragma unroll
            for (int j = 0; j < V; ++j)
              op.apply_fast(skipv[u] ? 0.f : a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                            Op::kInB ? mb[u].b[j] : (uint8_t)1,
                            ((uint32_t)j < leftu[u]) ? p0 : p1, o0.v[j], o1.v[j], ob.b[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < V; ++j)
            op.apply(skipv[u] ? 0.f : a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                     Op::kInB ? mb[u].b[j] : (uint8_t)1,
                     ((uint32_t)j < leftu[u]) ? p0 : p1, o0.v[j], o1.v[j], ob.b[j]);
        }
      }
      if constexpr (Op::kOut0) st_vec<V, SH>(io.out0 + e, o0);
      if constexpr (Op::kOut1) st_vec<V, SH>(io.out1 + e, o1);
      if constexpr (Op::kOutB) store_outb<Op, V>(io.outb, e, ob);
    }
  }
  // tail: the last n % V elements, scalar, by the CTA that owns them
  if (t0 <= n_main && n_main < t0 + kTile) {
    const int64_t e = n_main + threadIdx.x;
    if (e < n) {
      const P pj = tab[(uint32_t)((col0 + (uint32_t)(e - t0)) / inner)];
      float o0, o1;
      uint8_t ob;
      op.apply(to_f(io.in0[e]), Op::kIn1 ? io.in1[e] : 0.f,
               Op::kInB ? io.inb[e] : (uint8_t)1, pj, o0, o1, ob);
      if constexpr (Op::kOut0) st1(io.out0 + e, o0);
      if constexpr (Op::kOut1) st1(io.out1 + e, o1);
      if constexpr (Op::kOutB) io.outb[e] = ob;
    }
  }
#ifdef QSB_KERNEL_TIMING
  ktime_end(Op::kOut1 ? 2 : 1);
#endif
}

template <class Op, int V, int U, int MODE, Hint LH, Hint SH, class IO>
int launch_map_chan_win(const Op &op, const IO &io, int64_t n,
                        const Layout &L, cudaStream_t stream) {
  using P = typename Op::P;
  auto kern = map_chan_win_kernel<Op, V, U, MODE, LH, SH, IO>;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  const int64_t tiles = (n + kTile - 1) / kTile;
  const size_t rows_max = (size_t)((L.inner - 1 + kTile - 1) / L.inner + 2);
  const size_t smem = rows_max * sizeof(P);
  if (tiles > 0x7fffffffLL) return QSB_E_UNSUPPORTED;
  QSB_CUDA_TRY(launch_k(kern, dim3((unsigned)tiles), dim3(QSB_THREADS), smem, stream, op, io, n,
                        (uint32_t)L.inner, (uint32_t)L.channels, reverse_for<Op>()));
  return 0;
}

template <class Op, int V, int U, int MODE, Hint LH, Hint SH, class IO>
int launch_map_chan_variant(const Op &op, const IO &io, int64_t n,
                            const Layout &L, cudaStream_t stream) {
  using P = typename Op::P;
  auto kern = map_chan_kernel<Op, V, U, MODE, LH, SH, IO>;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  ChanGeom G;
  G.inner = (uint32_t)L.inner;
  G.channels = (uint32_t)L.channels;
  const size_t tab_bytes = (size_t)L.channels * sizeof(P);
  G.use_table = tab_bytes <= 48 * 1024;
  const size_t smem = G.use_table ? tab_bytes : 0;
  int occ = 0;
  QSB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern,
                                                             QSB_THREADS, smem));
  if (occ < 1) occ = 1;
  const int per_sm = map_tuning().chan_ctas_per_sm;
  const int64_t tiles = (n + kTile - 1) / kTile;
  int64_t grid = (int64_t)device_props().sm_count * (per_sm > 0 ? per_sm : occ);
  if (per_sm < 0) grid = tiles;  // one CTA per tile
  if (grid > tiles) grid = tiles;
  if (grid < 1) grid = 1;
  if (grid > 0x7fffffffLL) grid = 0x7fffffffLL;
  const int64_t su = (int64_t)QSB_THREADS * V, si = grid * kTile;
  G.su_cols = (uint32_t)(su % L.inner);
  G.su_ch = (uint32_t)((su / L.inner) % L.channels);
  G.si_cols = (uint32_t)(si % L.inner);
  G.si_ch = (uint32_t)((si / L.inner) % L.channels);
  QSB_CUDA_TRY(launch_k(kern, dim3((unsigned)grid), dim3(QSB_THREADS), smem, stream, op, io, n, G));
  return 0;
}

// ---------------------------------------------------------------------------
// per-channel, the channel is the FASTEST axis (inner == 1, channels % 8 == 0): the
// [tokens, hidden] activations of linear layers and NHWC tensors.  A 256-bit vector holds 8
// different channels, so per-vector parameter lookups (the MODE 2 walk: three shared-memory
// reads and a wrap test per ELEMENT, or a re-derivation when the table does not fit) cost more
// than the data.  Here a thread keeps ONE group of 8 consecutive channels for its whole life:
// it derives their constants once into registers and then strides over the rows in steps
// that are multiples of the row length, so consecutive threads still read consecutive
// memory.  Measured on [32768, 4096]: pow2 290 -> see profiles (was 0.57 of the copy peak),
// line 486 us (0.34).
// ---------------------------------------------------------------------------
template <class Op, int U, Hint LH, Hint SH, class IO>
__global__ void __launch_bounds__(QSB_THREADS)
    map_lastdim_kernel(Op op, IO io, int64_t n_vec, uint32_t groups, int64_t span) {
  pdl_wait();
  pdl_trigger();
  using P = typename Op::P;
  constexpr int V = 8;
  const int64_t i0 = (int64_t)blockIdx.x * QSB_THREADS + threadIdx.x;
  if (i0 >= span) return;  // span = the largest multiple of `groups` the grid covers
  const uint32_t c0 = (uint32_t)(i0 % groups) * V;
  P p[V];
  bool all_skip = Op::kCanSkip;
#pragma unroll
  for (int j = 0; j < V; ++j) {
    p[j] = op.params((int32_t)(c0 + j));
    if constexpr (Op::kCanSkip) all_skip = all_skip && op.skip(p[j]);
  }
  for (int64_t i = i0; i < n_vec; i += (int64_t)U * span) {
    VecF<V> a[U], b[U];
    VecB<V> mb[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = (i + (int64_t)u * span) * V;
      if (i + (int64_t)u * span < n_vec) {
        if (!all_skip) a[u] = ld_vec<V, LH>(io.in0 + e);
        if constexpr (Op::kIn1) b[u] = ld_vec<V, LH>(io.in1 + e);
        if constexpr (Op::kInB) mb[u] = ld_bytes<V>(io.inb + e);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = (i + (int64_t)u * span) * V;
      if (i + (int64_t)u * span < n_vec) {
        VecF<V> o0, o1;
        VecB<V> ob;
        bool fast = Op::kHasFast;
        if constexpr (Op::kHasFast) {
#pragma unroll
          for (int j = 0; j < V; ++j) fast = fast && op.template fast<1>(p[j], &a[u].v[j]);
        }
        if (fast) {
          if constexpr (Op::kHasFast) {
#pragma unroll
            for (int j = 0; j < V; ++j)
              op.apply_fast(all_skip ? 0.f : a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                            Op::kInB ? mb[u].b[j] : (uint8_t)1, p[j], o0.v[j], o1.v[j], ob.b[j]);
          }
        } else {
#pragma unroll
          for (int j = 0; j < V; ++j)
            op.apply(all_skip ? 0.f : a[u].v[j], Op::kIn1 ? b[u].v[j] : 0.f,
                     Op::kInB ? mb[u].b[j] : (uint8_t)1, p[j], o0.v[j], o1.v[j], ob.b[j]);
        }
        if constexpr (Op::kOut0) st_vec<V, SH>(io.out0 + e, o0);
        if constexpr (Op::kOut1) st_vec<V, SH>(io.out1 + e, o1);
        if constexpr (Op::kOutB) store_outb<Op, V>(io.outb, e, ob);
      }
    }
  }
}

template <class Op, Hint LH, Hint SH, class IO>
int launch_map_lastdim(const Op &op, const IO &io, int64_t n, const Layout &L, cudaStream_t stream) {
  constexpr int U = 2;
  auto kern = map_lastdim_kernel<Op, U, LH, SH, IO>;
  static int occ = 0;
  if (occ == 0) {
    int o = 0;
    QSB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&o, kern, QSB_THREADS, 0));
    occ = o > 0 ? o : 1;
  }
  const int64_t n_vec = n / 8, groups = L.channels / 8;
  int64_t grid = (int64_t)device_props().sm_count * occ;
  const int64_t need = (n_vec + QSB_THREADS - 1) / QSB_THREADS;
  if (grid > need) grid = need;
  const int64_t min_grid = (groups + QSB_THREADS - 1) / QSB_THREADS;  // one row must fit the grid
  if (grid < min_grid) grid = min_grid;
  const int64_t span = grid * QSB_THREADS / groups * groups;
  QSB_CUDA_TRY(launch_k(kern, dim3((unsigned)grid), dim3(QSB_THREADS), 0, stream, op, io, n_vec,
                        (uint32_t)groups, span));
  return 0;
}

// Picks per-tensor vs per-channel addressing and the widest vector the pointers
// allow (32 B -> V = 8; otherwise scalar for the channel kernel, 16 B -> V = 4
// for the per-tensor kernel).
template <class Op, Hint LH = Hint::STREAM, Hint SH = Hint::KEEP, class IO = MapIO>
int launch_map(const Op &op, const IO &io, const Layout &L,
               cudaStream_t stream) {
  const int64_t n = L.numel();
  if (n <= 0) return 0;
  uintptr_t bits = 0;
  auto acc = [&](const void *p, int scale) {
    // byte streams advance 1 B per element: a V-element vector needs V-byte
    // alignment, i.e. the same element alignment as 4V bytes of floats.
    if (p) bits |= reinterpret_cast<uintptr_t>(p) * scale;
  };
  // 16-bit streams: a V-element vector needs 2V-byte alignment, i.e. the same as 4V bytes of floats
  acc(io.in0, 4 / (int)sizeof(*io.in0));
  if (Op::kIn1) acc(io.in1, 1);
  if (Op::kOut0) acc(io.out0, 4 / (int)sizeof(*io.out0));
  if (Op::kOut1) acc(io.out1, 4 / (int)sizeof(*io.out1));
  if (Op::kInB) acc(io.inb, 4);
  if (Op::kOutB) acc(io.outb, is_pack4<Op>::value ? 8 : 4);  // packed nibbles: V / 2 bytes per vector
  if (bits & 3) return QSB_E_ALIGN;
  if (L.channels <= 1) {
    if ((bits & 31) == 0) return launch_map_tensor<Op, 8, 2, LH, SH, IO>(op, io, n, stream);
    if ((bits & 15) == 0) return launch_map_tensor<Op, 4, 4, LH, SH, IO>(op, io, n, stream);
    return launch_map_tensor<Op, 1, 4, LH, SH, IO>(op, io, n, stream);
  }
  if (L.inner >= (1LL << 31) || L.channels >= (1LL << 31)) return QSB_E_UNSUPPORTED;
  if ((bits & 31) == 0) {
    if (map_tuning().chan_ctas_per_sm == 0) {
      if (L.inner % 8 == 0) return launch_map_chan_win<Op, 8, 2, 0, LH, SH, IO>(op, io, n, L, stream);
      if (L.inner >= 8) return launch_map_chan_win<Op, 8, 2, 1, LH, SH, IO>(op, io, n, L, stream);
    } else {  // benchmark knob: the persistent full-table kernel for every shape
      if (L.inner % 8 == 0) return launch_map_chan_variant<Op, 8, 2, 0, LH, SH, IO>(op, io, n, L, stream);
      if (L.inner >= 8) return launch_map_chan_variant<Op, 8, 2, 1, LH, SH, IO>(op, io, n, L, stream);
    }
    if (L.inner == 1 && L.channels % 8 == 0 && map_tuning().lastdim)
      return launch_map_lastdim<Op, LH, SH, IO>(op, io, n, L, stream);
    return launch_map_chan_variant<Op, 8, 2, 2, LH, SH, IO>(op, io, n, L, stream);
  }
  return launch_map_chan_variant<Op, 1, 4, 0, LH, SH, IO>(op, io, n, L, stream);
}

}  // namespace qsb
