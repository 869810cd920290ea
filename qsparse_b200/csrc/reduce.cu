// K3  statistic reductions: abs-max, min/max, sum|x| (fp64) and count(x != 0),
// per tensor or per channel of an [outer, channels, inner] tensor, in ONE read
// of x (4 B/elem), deterministic (two stages, fixed combination order, no
// floating-point atomics).
//
// Stage 1 has two shapes:
//   row mode    (inner > 256): work items are (row, segment) pieces; a "virtual
//                warp" v owns items v, v + W, v + 2W, ... where W is a multiple of
//                channels * segments_per_row, so all its items belong to ONE
//                channel: it accumulates them in registers and writes a single
//                partial at the end (W partials in total instead of one per item).
//                256-bit loads, 4 in flight per lane, scalar head/tail peel for
//                pieces that do not start on a 32-byte boundary;
//   column mode (inner <= 256): the tensor is [outer, channels*inner]; one
//                thread per column (or 4 columns) walks a chunk of rows, so a
//                warp still reads contiguous 128/512-byte lines.
// Stage 2 (finalize) combines the partials of each channel in a fixed order (a transposed
// variant when the entries of one channel are `channels` apart).
//
// sum|x|: the 8 values of one 256-bit vector are first added pairwise in fp32
// (3 levels, |x| >= 0 so there is no cancellation), the vector sum is then
// accumulated in fp64.  That keeps the fp32->fp64 conversions (XU pipe, quarter
// rate) at one per 8 elements; accumulating every element in fp64 left the kernel
// XU-bound at 47 % pipe utilisation (profiles/).  The result is within ~1e-7
// relative of the exact sum — an order of magnitude closer than the reference's
// own fp32 cascade sums (SURVEY Q14).
#include <math.h>

#include "qsb_common.cuh"
#include "reduce_internal.cuh"
#include "step_epilogue.cuh"

#include <type_traits>

namespace qsb {

constexpr int kRowCtasPerSm = 4;  // column mode / default row variant
// row-kernel variant (tuning key 17): 0 = 4 x 256-bit loads per lane in flight, 4 CTAs / SM;
// 2 = 8 loads, 2 CTAs / SM (default: half as many partials for the finalize / the fused tail).
// The plan's warp count follows.
static int g_row_variant = -1;  // -1 = by row length (default), 0 / 2 = forced
void set_reduce_row_variant(int v) { g_row_variant = (v == 0 || v == 2) ? v : -1; }
// Long rows (>= 2048 elements: 8 full vectors per lane and round) keep 8 loads in flight per lane at 2 CTAs / SM
// — measured on the bench step 158.7 -> 156.8 us, and half as many partials for the tail; on shorter rows a
// round has fewer than 8 vectors per lane, so the extra registers only cost warps ([256,128,28,28]: 0.62 -> 0.54
// of the copy peak with the 8-load variant): those keep 4 loads at 4 CTAs / SM.
static inline int row_variant_for(int64_t inner) {
  if (g_row_variant >= 0) return g_row_variant;
  return inner >= 2048 ? 2 : 0;
}
static inline int row_ctas_per_sm(int variant) { return variant == 0 ? 4 : 2; }
// Rows up to this many elements use the COLUMN kernel (the tensor seen as [outer, C * inner]: vertical
// accumulation, perfectly coalesced, ~4 instructions per element).  Against the tile kernel that used to take rows
// of 64..256 elements (profiles/r02_colmode_probe_r2t.jsonl, sum|x| + max|x|, us): [256,256,14,14] 23.6 -> 17.4,
// [512,512,10,10] 35.8 -> 25.6, [256,512,16,16] 46.1 -> 29.7, [4096,64,14,14] 60.4 -> 39.9 (0.53 -> 0.80 of the copy
// peak), [256,2048,8,8] 42.0 -> 27.6, so the tile kernel was removed; rows of 784 elements and more are better off in
// the row kernel (23.6 vs 27.6).
constexpr int64_t kColMaxInner = 256;
// tuning key 18: the fused step reads the previous mask's kept channels with L2::evict_last
static int g_keep_hint = 1;
void set_reduce_keep_hint(int v) { g_keep_hint = v != 0; }

template <int WHAT>
struct Acc {
  uint32_t amax = 0;
  float mn = INFINITY, mx = -INFINITY;
  bool nan = false;
  double asum = 0.0;
  uint32_t nnz = 0;
  __device__ __forceinline__ void add(float v) {
    if constexpr (WHAT & QSB_STAT_ABSMAX) {
      uint32_t b = __float_as_uint(v) & 0x7fffffffu;
      amax = b > amax ? b : amax;
    }
    if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
      mn = fminf(mn, v);
      nan |= (v != v);
    }
    if constexpr (WHAT & QSB_STAT_MINMAX) mx = fmaxf(mx, v);
    if constexpr (WHAT & QSB_STAT_ABSSUM) asum += (double)fabsf(v);
    if constexpr (WHAT & QSB_STAT_NNZ) nnz += (v != 0.0f) ? 1u : 0u;
  }
  // N values at once (N = 8: one vector; N = 4: four rows of one column)
  template <int N>
  __device__ __forceinline__ void add_n(const float *v) {
    if constexpr (WHAT & QSB_STAT_ABSSUM) {
      float t[N];
#pragma unroll
      for (int k = 0; k < N; ++k) t[k] = fabsf(v[k]);
#pragma unroll
      for (int w = N / 2; w >= 1; w >>= 1)
#pragma unroll
        for (int k = 0; k < w; ++k) t[k] = __fadd_rn(t[k], t[k + w]);
      asum += (double)t[0];
    }
#pragma unroll
    for (int k = 0; k < N; ++k) {
      const float x = v[k];
      if constexpr (WHAT & QSB_STAT_ABSMAX) {
        uint32_t b = __float_as_uint(x) & 0x7fffffffu;
        amax = b > amax ? b : amax;
      }
      if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
        mn = fminf(mn, x);
        nan |= (x != x);
      }
      if constexpr (WHAT & QSB_STAT_MINMAX) mx = fmaxf(mx, x);
      if constexpr (WHAT & QSB_STAT_NNZ) nnz += (x != 0.0f) ? 1u : 0u;
    }
  }
};

__device__ __forceinline__ float nan_f() { return __uint_as_float(0x7fc00000u); }

template <int WHAT>
__device__ __forceinline__ void warp_store(const Acc<WHAT> &a_in, int lane,
                                           const Partials &P, int64_t item) {
  Acc<WHAT> a = a_in;
  if constexpr (WHAT & QSB_STAT_ABSMAX) {
    a.amax = warp_reduce(a.amax, [](uint32_t x, uint32_t y) { return x > y ? x : y; });
    if (lane == 0) P.amax[item] = a.amax;
  }
  if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
    int nan = __any_sync(0xffffffffu, a.nan);
    a.mn = warp_reduce(a.mn, [](float x, float y) { return fminf(x, y); });
    if (lane == 0) P.mn[item] = nan ? nan_f() : a.mn;
    if constexpr (WHAT & QSB_STAT_MINMAX) {
      a.mx = warp_reduce(a.mx, [](float x, float y) { return fmaxf(x, y); });
      if (lane == 0) P.mx[item] = nan ? nan_f() : a.mx;
    }
  }
  if constexpr (WHAT & QSB_STAT_ABSSUM) {
    a.asum = warp_reduce(a.asum, [](double x, double y) { return x + y; });
    if (lane == 0) P.asum[item] = a.asum;
  }
  if constexpr (WHAT & QSB_STAT_NNZ) {
    a.nnz = warp_reduce(a.nnz, [](uint32_t x, uint32_t y) { return x + y; });
    if (lane == 0) P.nnz[item] = (double)a.nnz;
  }
}

// ---------------------------------------------------------------------------
// Fused tail: a stage-1 kernel instantiated with StepTail ends with the parameter step of the
// structured prune -> quantize training step (step_epilogue.cuh), run by whichever CTA arrives
// LAST at a device-wide counter — no separate finalize / parameter launch, and across GPUs
// the peer exchange starts the moment this GPU's statistics are complete.  NoTail: plain stage 1.
// ---------------------------------------------------------------------------
struct NoTail {};
struct StepTail {
  StepArgs a;
  unsigned int *arrival;     // zero before the first launch; the last CTA resets it
  const uint8_t *keep_hint;  // optional channel mask of the previous step (L2 residency hint)
};

// the statistics a stage-1 kernel gathers decide the form of its parameter step: sum|x| + max|x| the pow2 form,
// sum|x| + min / max x the line form (AdaptiveQuantizer)
template <int WHAT>
constexpr bool kLineStep = (WHAT & QSB_STAT_MINMAX) != 0;

template <bool LINES>
__device__ __forceinline__ void fused_step_tail(const StepTail &t, unsigned char *smem, const StepPrefetch &pre) {
  __shared__ int s_last;
  // The CTA barrier orders every thread's partial stores before thread 0's fence + atomic (the grid-sync
  // pattern of cooperative groups): ONE device-scope fence per CTA instead of one per thread — each is a
  // MEMBAR.SC.GPU + CCTL.IVALL on the last CTA's critical path.
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned total = gridDim.x * gridDim.y;
    __threadfence();
    const int last = atomicAdd(t.arrival, 1u) == total - 1;
    if (last) {
      __threadfence();   // the other CTAs' partials are visible to the loads below (they go to L2: __ldcg)
      *t.arrival = 0;    // ready for the next launch
    }
    s_last = last;
  }
  __syncthreads();
  if (!s_last) return;
  step_epilogue<LINES>(t.a, carve_step_smem(smem, t.a.channels), pre);
}

// kernel start: the old state into registers (StepPrefetch) and, for the bench's evidence, the earliest
// start time of any CTA
template <int WHAT, class Tail>
__device__ __forceinline__ StepPrefetch fused_step_begin(const Tail &tail) {
  if constexpr (std::is_same<Tail, StepTail>::value) {
    if (tail.a.timing && threadIdx.x == 0) atomicMin(tail.a.timing, global_ns());
    return step_prefetch<kLineStep<WHAT>>(tail.a);
  } else {
    return StepPrefetch{false, 0.f, 0.f, 0};
  }
}

// where stage 2 writes the finalized statistics (NULL: not wanted).  Stand-alone reductions always finalize in a
// second launch: letting stage 1's last-arriving CTA do it was measured slower (DESIGN §8, row 8).
struct FinalOut {
  float *absmax, *mn, *mx;
  double *abssum, *nnz;
};

// 256-bit load with a run-time L2 eviction policy (createpolicy): kept channels of the previous
// mask are read evict_last — the forward pass re-reads exactly those a few microseconds later,
// 51 MB of the bench tensor — everything else evict_first.
__device__ __forceinline__ uint64_t l2_policy(bool keep) {
  uint64_t pol;
  if (keep) asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  else asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ VecF<8> ld_vec8_policy(const float *p, uint64_t pol) {
  VecF<8> r;
  asm volatile(
      "ld.global.L1::no_allocate.L2::cache_hint.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8], %9;"
      : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3]), "=f"(r.v[4]), "=f"(r.v[5]), "=f"(r.v[6]),
        "=f"(r.v[7])
      : "l"(p), "l"(pol));
  return r;
}
// 8 16-bit values, 16-byte aligned: one 128-bit load with the policy, still packed
__device__ __forceinline__ uint4 ld_raw16_policy(const void *p, uint64_t pol) {
  uint4 w;
  asm volatile("ld.global.L1::no_allocate.L2::cache_hint.v4.b32 {%0,%1,%2,%3}, [%4], %5;"
               : "=r"(w.x), "=r"(w.y), "=r"(w.z), "=r"(w.w)
               : "l"(p), "l"(pol));
  return w;
}

// ---------------------------------------------------------------------------
// stage 1, row mode.  U = 256-bit loads in flight per lane and round, MINB = resident CTAs
// per SM the register budget is set for (the plan's warp count follows, row_ctas_per_sm()).
// ---------------------------------------------------------------------------
// T: element type of x; VEC (16-bit x only): x is 16-byte aligned, so every vector is one 128-bit load —
// false for a view that starts at any other even address (element loads, same vectors, same order)
template <int WHAT, int U, int MINB, class Tail, class T, bool VEC = true>
__global__ void __launch_bounds__(QSB_THREADS, MINB)
    reduce_rows_kernel(const T *__restrict__ x, int64_t rows, int64_t inner,
                       int64_t seg, int64_t segs_per_row, int64_t vwarps,
                       Partials P, int cta_combine, int channels, const __grid_constant__ Tail tail) {
  pdl_wait();
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char qsb_dyn_smem[];
  const StepPrefetch pre = fused_step_begin<WHAT>(tail);
  if constexpr (std::is_same<Tail, StepTail>::value) ktime_begin(0);
  const int lane = threadIdx.x & 31;
  const int64_t warps_phys = (int64_t)gridDim.x * (QSB_THREADS / 32);
  const int64_t items = rows * segs_per_row;
  // 16-bit x: vectors start at multiples of 8 elements from x[0] (what an fp32 copy of x starting on a 32-byte
  // boundary gets)
  static_assert(VEC || is_half16<T>, "an fp32 x is always read with 256-bit loads");
  auto run_vw = [&](Acc<WHAT> &acc, int64_t vw) {
    // every item of a virtual warp belongs to ONE channel
    uint64_t pol = 0;
    bool use_pol = false;
    if constexpr (std::is_same<Tail, StepTail>::value) {
      if (tail.keep_hint) {
        use_pol = true;
        pol = l2_policy(tail.keep_hint[(vw / segs_per_row) % channels] != 0);
      }
    }
    for (int64_t item = vw; item < items; item += vwarps) {
      const int64_t row = item / segs_per_row;
      const int64_t s = item - row * segs_per_row;
      const int64_t c0 = s * seg;
      const int64_t c1 = (c0 + seg < inner) ? c0 + seg : inner;
      const T *p = x + row * inner + c0;
      const int64_t len = c1 - c0;
      // head: scalars up to the first 32-byte boundary (16-bit x: up to the next multiple of 8 elements)
      int64_t head;
      if constexpr (is_half16<T>) head = (8 - ((row * inner + c0) & 7)) & 7;
      else head = ((32 - (reinterpret_cast<uintptr_t>(p) & 31)) & 31) >> 2;
      if (head > len) head = len;
      if (lane < head) acc.add(to_f(p[lane]));
      const T *pv = p + head;
      const int64_t nv = (len - head) >> 3;
      // body: 256-bit loads, up to U in flight per lane (predicated, so short pieces do not
      // fall back to one load per round trip); vector order per lane is the same for every U
      for (int64_t j = lane; j < nv; j += 32 * U) {
        if constexpr (!VEC) {  // element loads, one vector at a time
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (j + 32 * u < nv) {
              const VecF<8> w = ld_vec8_any<Hint::KEEP>(pv + ((j + 32 * u) << 3), false);
              acc.template add_n<8>(w.v);
            }
        } else if constexpr (is_half16<T>) {
          // the U loads in flight stay packed (4 registers each, half of fp32's) until they are accumulated:
          // unpacked up front, the 4-load variant at 64 registers spilled
          uint4 w[U];
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (j + 32 * u < nv) {
              if (std::is_same<Tail, StepTail>::value && use_pol) w[u] = ld_raw16_policy(pv + ((j + 32 * u) << 3), pol);
              else w[u] = ld_raw16(pv + ((j + 32 * u) << 3));
            }
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (j + 32 * u < nv) {
              const VecF<8> v = unpack8<T>(w[u]);
              acc.template add_n<8>(v.v);
            }
        } else {
          VecF<8> v[U];
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (j + 32 * u < nv) {
              if (std::is_same<Tail, StepTail>::value && use_pol) v[u] = ld_vec8_policy(pv + ((j + 32 * u) << 3), pol);
              else v[u] = ld_vec<8, Hint::KEEP>(pv + ((j + 32 * u) << 3));
            }
#pragma unroll
          for (int u = 0; u < U; ++u)
            if (j + 32 * u < nv) acc.template add_n<8>(v[u].v);
        }
      }
      // tail
      const int64_t done = head + (nv << 3);
      if (done + lane < len) acc.add(to_f(p[done + lane]));
    }
  };
  if (cta_combine) {
    // one channel (per-tensor statistics): every warp of the CTA — one virtual warp each — feeds the same
    // result, so the CTA combines its 8 warps in warp order and writes ONE partial; the finalize (or the
    // fused parameter step) then reads gridDim.x entries instead of 8x as many
    constexpr int kW = QSB_THREADS / 32;
    __shared__ uint32_t s_amax[kW];
    __shared__ float s_mn[kW], s_mx[kW];
    __shared__ double s_asum[kW], s_nnz[kW];
    const Partials Ps{s_amax, s_mn, s_mx, s_asum, s_nnz};
    const int w = threadIdx.x >> 5;
    const int64_t vw = (int64_t)blockIdx.x * kW + w;
    Acc<WHAT> acc;
    if (vw < vwarps) run_vw(acc, vw);
    warp_store<WHAT>(acc, lane, Ps, w);
    __syncthreads();
    if (threadIdx.x == 0) {
      uint32_t amax = 0;
      float mn = INFINITY, mx = -INFINITY;
      bool nan = false;
      double asum = 0.0, nnz = 0.0;
      for (int k = 0; k < kW; ++k) {
        if constexpr (WHAT & QSB_STAT_ABSMAX) amax = s_amax[k] > amax ? s_amax[k] : amax;
        if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
          nan |= (s_mn[k] != s_mn[k]);
          mn = fminf(mn, s_mn[k]);
        }
        if constexpr (WHAT & QSB_STAT_MINMAX) {
          nan |= (s_mx[k] != s_mx[k]);
          mx = fmaxf(mx, s_mx[k]);
        }
        if constexpr (WHAT & QSB_STAT_ABSSUM) asum += s_asum[k];
        if constexpr (WHAT & QSB_STAT_NNZ) nnz += s_nnz[k];
      }
      const int64_t o = blockIdx.x;
      if constexpr (WHAT & QSB_STAT_ABSMAX) P.amax[o] = amax;
      if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) P.mn[o] = nan ? nan_f() : mn;
      if constexpr (WHAT & QSB_STAT_MINMAX) P.mx[o] = nan ? nan_f() : mx;
      if constexpr (WHAT & QSB_STAT_ABSSUM) P.asum[o] = asum;
      if constexpr (WHAT & QSB_STAT_NNZ) P.nnz[o] = nnz;
    }
  } else {
    for (int64_t vw = (int64_t)blockIdx.x * (QSB_THREADS / 32) + (threadIdx.x >> 5);
         vw < vwarps; vw += warps_phys) {
      Acc<WHAT> acc;
      run_vw(acc, vw);
      warp_store<WHAT>(acc, lane, P, vw);
    }
  }
  if constexpr (std::is_same<Tail, StepTail>::value) fused_step_tail<kLineStep<WHAT>>(tail, qsb_dyn_smem, pre);
#ifdef QSB_KERNEL_TIMING
  if constexpr (std::is_same<Tail, StepTail>::value) ktime_end(0);
#endif
}

// ---------------------------------------------------------------------------
// stage 1, column mode.  partial index = chunk * ncols + col.
// A CTA owns a band of rows (blockIdx.y) and `tpr` column-vectors of it (blockIdx.x); when
// the tensor has fewer than 256 column-vectors ([N, 64] activations: 16 of them) the CTA's
// 256 / tpr "row lanes" walk interleaved rows of the band, so every thread is busy and a
// warp still reads consecutive memory; the row lanes are then combined through shared
// memory in lane order (deterministic) and row lane 0 writes the partial.
// ---------------------------------------------------------------------------
template <int WHAT, int V, class T>
__device__ __forceinline__ void reduce_cols_body(const T *__restrict__ x, int64_t nrows, int64_t ncols,
                                                 int64_t rows_per_chunk, int tpr, Partials P) {
  pdl_wait();
  pdl_trigger();
  const int64_t vcols = ncols / V;  // V == 4 requires ncols % 4 == 0
  const int rpb = QSB_THREADS / tpr;  // row lanes
  const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr;
  const int64_t vc = (int64_t)blockIdx.x * tpr + cl;
  const bool live = vc < vcols;
  const int64_t chunk = blockIdx.y;
  const int64_t r0 = chunk * rows_per_chunk;
  const int64_t r1 = (r0 + rows_per_chunk < nrows) ? r0 + rows_per_chunk : nrows;
  Acc<WHAT> acc[V];
  if (live) {
    const T *p = x + vc * V;
    int64_t r = r0 + rl;
    for (; r + 3 * (int64_t)rpb < r1; r += 4 * (int64_t)rpb) {
      VecF<V> v[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = ld_vec<V, Hint::KEEP>(p + (r + (int64_t)k * rpb) * ncols);
#pragma unroll
      for (int q = 0; q < V; ++q) {
        const float col4[4] = {v[0].v[q], v[1].v[q], v[2].v[q], v[3].v[q]};
        acc[q].template add_n<4>(col4);
      }
    }
    for (; r < r1; r += rpb) {
      VecF<V> v = ld_vec<V, Hint::KEEP>(p + r * ncols);
#pragma unroll
      for (int q = 0; q < V; ++q) acc[q].add(v.v[q]);
    }
  }
  // staging for the two in-kernel combines: [field][q][thread]
  __shared__ uint32_t s_amax[V][QSB_THREADS];
  __shared__ float s_mn[V][QSB_THREADS], s_mx[V][QSB_THREADS];
  __shared__ double s_asum[V][QSB_THREADS];
  __shared__ uint32_t s_nnz[V][QSB_THREADS];
  __shared__ uint8_t s_nan[V][QSB_THREADS];
  auto stage = [&](int t) {
#pragma unroll
    for (int q = 0; q < V; ++q) {
      if constexpr (WHAT & QSB_STAT_ABSMAX) s_amax[q][t] = acc[q].amax;
      if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
        s_mn[q][t] = acc[q].mn;
        s_nan[q][t] = acc[q].nan ? 1 : 0;
      }
      if constexpr (WHAT & QSB_STAT_MINMAX) s_mx[q][t] = acc[q].mx;
      if constexpr (WHAT & QSB_STAT_ABSSUM) s_asum[q][t] = acc[q].asum;
      if constexpr (WHAT & QSB_STAT_NNZ) s_nnz[q][t] = acc[q].nnz;
    }
  };
  if (rpb > 1) {
    // combine the row lanes in shared memory, summed by row lane 0 in lane order (deterministic)
    stage(threadIdx.x);
    __syncthreads();
    if (rl == 0) {
      for (int l = 1; l < rpb; ++l) {
        const int t = l * tpr + cl;
#pragma unroll
        for (int q = 0; q < V; ++q) {
          if constexpr (WHAT & QSB_STAT_ABSMAX) acc[q].amax = s_amax[q][t] > acc[q].amax ? s_amax[q][t] : acc[q].amax;
          if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
            acc[q].mn = fminf(acc[q].mn, s_mn[q][t]);
            acc[q].nan |= s_nan[q][t] != 0;
          }
          if constexpr (WHAT & QSB_STAT_MINMAX) acc[q].mx = fmaxf(acc[q].mx, s_mx[q][t]);
          if constexpr (WHAT & QSB_STAT_ABSSUM) acc[q].asum += s_asum[q][t];
          if constexpr (WHAT & QSB_STAT_NNZ) acc[q].nnz += s_nnz[q][t];
        }
      }
    }
  }
  // (Combining the row bands of 8 CTAs through a thread-block cluster's distributed shared memory before
  // writing — 8x fewer partials — was measured and dropped: the finalize went 10 -> 5 us but this kernel
  // 16 -> 28 us on [16384, 1000], with every cluster resident.)
  if (!live || rl != 0) return;
#pragma unroll
  for (int q = 0; q < V; ++q) {
    const int64_t idx = chunk * ncols + vc * V + q;
    if constexpr (WHAT & QSB_STAT_ABSMAX) P.amax[idx] = acc[q].amax;
    if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ))
      P.mn[idx] = acc[q].nan ? nan_f() : acc[q].mn;
    if constexpr (WHAT & QSB_STAT_MINMAX)
      P.mx[idx] = acc[q].nan ? nan_f() : acc[q].mx;
    if constexpr (WHAT & QSB_STAT_ABSSUM) P.asum[idx] = acc[q].asum;
    if constexpr (WHAT & QSB_STAT_NNZ) P.nnz[idx] = (double)acc[q].nnz;
  }
}

template <int WHAT, int V, class Tail, class T>
__global__ void __launch_bounds__(QSB_THREADS)
    reduce_cols_kernel(const T *__restrict__ x, int64_t nrows, int64_t ncols,
                       int64_t rows_per_chunk, int tpr, Partials P, const __grid_constant__ Tail tail) {
  extern __shared__ __align__(16) unsigned char qsb_dyn_smem[];
  if constexpr (std::is_same<Tail, StepTail>::value) pdl_wait();  // the old state may have been written by the kernel just before
  const StepPrefetch pre = fused_step_begin<WHAT>(tail);
  reduce_cols_body<WHAT, V, T>(x, nrows, ncols, rows_per_chunk, tpr, P);
  if constexpr (std::is_same<Tail, StepTail>::value) fused_step_tail<kLineStep<WHAT>>(tail, qsb_dyn_smem, pre);
}

// ---------------------------------------------------------------------------
// stage 2: channel c combines entries j = 0..count-1 at
//   idx(j) = (j / q) * (channels * q) + c * q + (j % q)
// (q = segments per row in row mode, `inner` in column mode).
// G threads per channel (32: a warp; 256: a CTA), fixed order.
// ---------------------------------------------------------------------------
template <int WHAT, int G>
__global__ void __launch_bounds__(QSB_THREADS)
    reduce_finalize_kernel(Partials P, FinalOut out, int64_t channels,
                           int64_t count, int64_t q) {
  pdl_wait();
  pdl_trigger();
  constexpr int kGroupsPerBlock = QSB_THREADS / G;
  const int g = threadIdx.x / G;
  const int tg = threadIdx.x % G;
  const int64_t c = (int64_t)blockIdx.x * kGroupsPerBlock + g;
  const bool active = c < channels;

  uint32_t amax = 0;
  float mn = INFINITY, mx = -INFINITY;
  bool nan = false;
  double asum = 0.0, nnz = 0.0;
  if (active) {
    // 32-bit division whenever the entry index fits (a 64-bit one is ~100 instructions per entry)
    const bool small = count < 0x7fffffffLL && q < 0x7fffffffLL;
    auto index_of = [&](int64_t j) {
      const int64_t hi = small ? (int64_t)((uint32_t)j / (uint32_t)q) : j / q;
      return hi * (channels * q) + c * q + (j - hi * q);
    };
    for (int64_t j0 = tg; j0 < count; j0 += 4 * G) {
      int64_t idx[4];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        ok[u] = j0 + (int64_t)u * G < count;
        idx[u] = ok[u] ? index_of(j0 + (int64_t)u * G) : 0;
      }
      if constexpr (WHAT & QSB_STAT_ABSMAX) {
        uint32_t b[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) b[u] = ok[u] ? P.amax[idx[u]] : 0u;
#pragma unroll
        for (int u = 0; u < 4; ++u) amax = b[u] > amax ? b[u] : amax;
      }
      if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ok[u] ? P.mn[idx[u]] : INFINITY;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          nan |= (v[u] != v[u]);
          mn = fminf(mn, v[u]);
        }
      }
      if constexpr (WHAT & QSB_STAT_MINMAX) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ok[u] ? P.mx[idx[u]] : -INFINITY;
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          nan |= (v[u] != v[u]);
          mx = fmaxf(mx, v[u]);
        }
      }
      if constexpr (WHAT & QSB_STAT_ABSSUM) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ok[u] ? P.asum[idx[u]] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) asum += v[u];
      }
      if constexpr (WHAT & QSB_STAT_NNZ) {
        double v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = ok[u] ? P.nnz[idx[u]] : 0.0;
#pragma unroll
        for (int u = 0; u < 4; ++u) nnz += v[u];
      }
    }
  }
  // warp level
  amax = warp_reduce(amax, [](uint32_t a, uint32_t b) { return a > b ? a : b; });
  mn = warp_reduce(mn, [](float a, float b) { return fminf(a, b); });
  mx = warp_reduce(mx, [](float a, float b) { return fmaxf(a, b); });
  nan = __any_sync(0xffffffffu, nan);
  asum = warp_reduce(asum, [](double a, double b) { return a + b; });
  nnz = warp_reduce(nnz, [](double a, double b) { return a + b; });
  if constexpr (G > 32) {
    __shared__ uint32_t s_amax[QSB_THREADS / 32];
    __shared__ float s_mn[QSB_THREADS / 32], s_mx[QSB_THREADS / 32];
    __shared__ int s_nan[QSB_THREADS / 32];
    __shared__ double s_asum[QSB_THREADS / 32], s_nnz[QSB_THREADS / 32];
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
      s_amax[w] = amax; s_mn[w] = mn; s_mx[w] = mx; s_nan[w] = nan;
      s_asum[w] = asum; s_nnz[w] = nnz;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 1; k < QSB_THREADS / 32; ++k) {
        amax = s_amax[k] > amax ? s_amax[k] : amax;
        mn = fminf(mn, s_mn[k]);
        mx = fmaxf(mx, s_mx[k]);
        nan = nan || s_nan[k];
        asum += s_asum[k];
        nnz += s_nnz[k];
      }
    }
  }
  if (active && tg == 0) {
    if constexpr (WHAT & QSB_STAT_ABSMAX)
      if (out.absmax) out.absmax[c] = __uint_as_float(amax);
    if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ))
      if (out.mn) out.mn[c] = nan ? nan_f() : mn;
    if constexpr (WHAT & QSB_STAT_MINMAX)
      if (out.mx) out.mx[c] = nan ? nan_f() : mx;
    if constexpr (WHAT & QSB_STAT_ABSSUM)
      if (out.abssum) out.abssum[c] = asum;
    if constexpr (WHAT & QSB_STAT_NNZ)
      if (out.nnz) out.nnz[c] = nnz;
  }
}

// stage 2 when fin_q == 1 (channel-last column mode): entry j of channel c sits
// at j * channels + c, so a warp that walks j touches 32 sectors for 32 values (the finalize took
// 12 us behind a 16 us stage 1 on [16384, 1000]).  Here a CTA owns 8 ADJACENT channels: thread t
// reads channel (t & 7) of entries (t >> 3), (t >> 3) + 32, ... — each 8-lane group reads whole
// sectors — and the 32 entry lanes are combined by shuffles, then across warps in warp order.
template <int WHAT>
__global__ void __launch_bounds__(QSB_THREADS)
    reduce_finalize_t_kernel(Partials P, FinalOut out, int64_t channels, int64_t count) {
  pdl_wait();
  pdl_trigger();
  constexpr int kU = 8;  // independent loads in flight per statistic
  const int cl = threadIdx.x & 7, jl = threadIdx.x >> 3;
  const int64_t c = (int64_t)blockIdx.x * 8 + cl;
  const bool active = c < channels;
  uint32_t amax = 0;
  float mn = INFINITY, mx = -INFINITY;
  bool nan = false;
  double asum = 0.0, nnz = 0.0;
  if (active) {
    for (int64_t j0 = jl; j0 < count; j0 += kU * 32) {
      int64_t idx[kU];
      bool ok[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        ok[u] = j0 + 32 * u < count;
        idx[u] = ok[u] ? (j0 + 32 * u) * channels + c : 0;
      }
      if constexpr (WHAT & QSB_STAT_ABSMAX) {
        uint32_t b[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) b[u] = ok[u] ? P.amax[idx[u]] : 0u;
#pragma unroll
        for (int u = 0; u < kU; ++u) amax = b[u] > amax ? b[u] : amax;
      }
      if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ)) {
        float v[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) v[u] = ok[u] ? P.mn[idx[u]] : INFINITY;
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          nan |= (v[u] != v[u]);
          mn = fminf(mn, v[u]);
        }
      }
      if constexpr (WHAT & QSB_STAT_MINMAX) {
        float v[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) v[u] = ok[u] ? P.mx[idx[u]] : -INFINITY;
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          nan |= (v[u] != v[u]);
          mx = fmaxf(mx, v[u]);
        }
      }
      if constexpr (WHAT & QSB_STAT_ABSSUM) {
        double v[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) v[u] = ok[u] ? P.asum[idx[u]] : 0.0;
#pragma unroll
        for (int u = 0; u < kU; ++u) asum += v[u];
      }
      if constexpr (WHAT & QSB_STAT_NNZ) {
        double v[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) v[u] = ok[u] ? P.nnz[idx[u]] : 0.0;
#pragma unroll
        for (int u = 0; u < kU; ++u) nnz += v[u];
      }
    }
  }
  // the 4 entry lanes of a warp that share a channel
#pragma unroll
  for (int o = 8; o <= 16; o <<= 1) {
    const uint32_t a2 = __shfl_xor_sync(0xffffffffu, amax, o);
    amax = a2 > amax ? a2 : amax;
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nan = (__shfl_xor_sync(0xffffffffu, (int)nan, o) != 0) || nan;
    asum += __shfl_xor_sync(0xffffffffu, asum, o);
    nnz += __shfl_xor_sync(0xffffffffu, nnz, o);
  }
  __shared__ uint32_t s_amax[QSB_THREADS / 32][8];
  __shared__ float s_mn[QSB_THREADS / 32][8], s_mx[QSB_THREADS / 32][8];
  __shared__ int s_nan[QSB_THREADS / 32][8];
  __shared__ double s_asum[QSB_THREADS / 32][8], s_nnz[QSB_THREADS / 32][8];
  const int w = threadIdx.x >> 5;
  if ((threadIdx.x & 31) < 8) {
    s_amax[w][cl] = amax; s_mn[w][cl] = mn; s_mx[w][cl] = mx; s_nan[w][cl] = nan;
    s_asum[w][cl] = asum; s_nnz[w][cl] = nnz;
  }
  __syncthreads();
  if (threadIdx.x < 8 && active) {
    for (int k = 1; k < QSB_THREADS / 32; ++k) {
      amax = s_amax[k][cl] > amax ? s_amax[k][cl] : amax;
      mn = fminf(mn, s_mn[k][cl]);
      mx = fmaxf(mx, s_mx[k][cl]);
      nan = nan || s_nan[k][cl];
      asum += s_asum[k][cl];
      nnz += s_nnz[k][cl];
    }
    if constexpr (WHAT & QSB_STAT_ABSMAX)
      if (out.absmax) out.absmax[c] = __uint_as_float(amax);
    if constexpr (WHAT & (QSB_STAT_MINMAX | QSB_STAT_NNZ))
      if (out.mn) out.mn[c] = nan ? nan_f() : mn;
    if constexpr (WHAT & QSB_STAT_MINMAX)
      if (out.mx) out.mx[c] = nan ? nan_f() : mx;
    if constexpr (WHAT & QSB_STAT_ABSSUM)
      if (out.abssum) out.abssum[c] = asum;
    if constexpr (WHAT & QSB_STAT_NNZ)
      if (out.nnz) out.nnz[c] = nnz;
  }
}

// min over the per-channel minima (l0 gate, qsparse/sparse.py:85)
__global__ void tensor_min_kernel(const float *mn, int64_t channels, float *out) {
  float m = INFINITY;
  bool nan = false;
  for (int64_t j = threadIdx.x; j < channels; j += 32) {
    float v = mn[j];
    nan |= (v != v);
    m = fminf(m, v);
  }
  m = warp_reduce(m, [](float a, float b) { return fminf(a, b); });
  nan = __any_sync(0xffffffffu, nan);
  if (threadIdx.x == 0) *out = nan ? nan_f() : m;
}

// ---------------------------------------------------------------------------
// host-side planning
// ---------------------------------------------------------------------------
// Physical warps of the row kernel: SMs x resident CTAs x 8.  The CTA count per
// SM is fixed (not queried per instantiation) so that the plan — and with it the
// summation order — only depends on the device, never on which statistics run.
constexpr int64_t kSegMin = 1024;
// column mode on wide tensors (more column vectors than this): threads of a CTA along a row; the other
// 256 / tpr threads are row lanes whose results are combined in shared memory before the partial
// is written, so the partial array (and the finalize's read) shrinks by that factor
constexpr int64_t kColTprWide = 64;  // measured: [16384,1000] 14.7 + 6.3 -> 14.2 + 3.7 us, [512,512,7,7] 15.4 + 7.5 -> 11.4 + 6.4 us vs 256

ReducePlan make_plan(int64_t outer, int64_t channels, int64_t inner,
                            const void *x, int x_bytes) {
  ReducePlan p{};
  p.row_variant = row_variant_for(inner);
  const int64_t warps_phys =
      (int64_t)device_props().sm_count * row_ctas_per_sm(p.row_variant) * (QSB_THREADS / 32);
  if (inner > kColMaxInner) {
    p.row_mode = true;
    p.rows = outer * channels;
    // balanced segments: aim for >= 6 work items per physical warp, but keep every
    // segment >= kSegMin elements (two rounds of 4 x 256-bit loads per lane) unless the
    // machine could not be filled otherwise
    int64_t spr_max = inner / kSegMin > 0 ? inner / kSegMin : 1;
    int64_t spr = (6 * warps_phys + p.rows - 1) / p.rows;
    if (spr > spr_max) spr = spr_max;
    if (spr < 1) spr = 1;
    if (p.rows * spr < warps_phys) {
      spr_max = inner / 512 > 0 ? inner / 512 : 1;
      spr = (warps_phys + p.rows - 1) / p.rows;
      if (spr > spr_max) spr = spr_max;
    }
    int64_t seg = (inner + spr - 1) / spr;
    seg = (seg + 7) / 8 * 8;
    spr = (inner + seg - 1) / seg;
    p.seg = seg;
    p.segs_per_row = spr;
    const int64_t items = p.rows * spr;
    const int64_t period = channels * spr;  // items with the same (channel, segment)
    int64_t m;                              // virtual warps = m * period
    if (channels == 1) {
      // one channel: any assignment works; one virtual warp per physical warp, one partial per CTA
      p.vwarps = items < warps_phys ? items : warps_phys;
      p.cta_combine = 1;
      p.fin_count = (p.vwarps + QSB_THREADS / 32 - 1) / (QSB_THREADS / 32);
      p.fin_q = 1;
    } else {
      const int64_t m_max = outer;
      if (period * 4 <= warps_phys)
        m = warps_phys / period;
      else
        m = (4 * warps_phys + period - 1) / period;
      if (m > m_max) m = m_max;
      if (m < 1) m = 1;
      p.vwarps = m * period;
      p.fin_count = m * spr;
      p.fin_q = spr;
    }
    p.n_partials = p.vwarps;
  } else {
    const int64_t target = (int64_t)device_props().sm_count * kRowCtasPerSm * QSB_THREADS;
    p.row_mode = false;
    p.nrows = outer;
    p.ncols = channels * inner;
    p.vcol = (p.ncols % 4 == 0 && (x == nullptr || aligned_to(x, 4 * x_bytes))) ? 4 : 1;
    // The grid is planned for the vector width the SHAPE allows, whatever the alignment of x: the row
    // bands (and with them the partial layout that qsb_prune_quant_step_params re-derives without x)
    // must not depend on the pointer; an unaligned x only gets 4x more CTAs along the row.
    const int64_t threads = p.ncols / (p.ncols % 4 == 0 ? 4 : 1);
    // threads of one row that a CTA covers: a power of two <= 256; the other 256 / tpr "row lanes"
    // of the CTA walk interleaved rows of the chunk
    int64_t tpr_max = 1;
    while (tpr_max < threads && tpr_max < QSB_THREADS) tpr_max <<= 1;
    // at least 8 rows per chunk so the partial array stays small
    const int64_t max_chunks = (outer + 7) / 8;
    const int64_t want = target / QSB_THREADS;  // resident CTAs
    auto chunks_for = [&](int64_t tpr_) {
      const int64_t ctas_x_ = (threads + tpr_ - 1) / tpr_;
      int64_t c = (want + ctas_x_ / 2) / ctas_x_;  // nearest: do not spill into a second wave
      if (c > max_chunks) c = max_chunks;
      if (c < 1) c = 1;
      if (c > 65535) c = 65535;
      return c;
    };
    // wide tensors: from kColTprWide threads along the row upwards, the first width whose grid fills
    // one wave best ([1024, 2048, 7, 7] at 64: 392 x 2 CTAs = 1.3 waves, 83 us instead of 71)
    int64_t tpr = tpr_max;
    if (tpr_max > kColTprWide) {
      double best = -1.0;
      for (int64_t t = kColTprWide; t <= tpr_max; t <<= 1) {
        const int64_t total = (threads + t - 1) / t * chunks_for(t);
        const int64_t waves = (total + want - 1) / want;
        const double eff = (double)total / (double)(waves * want);
        if (eff > best + 0.02) best = eff, tpr = t;
      }
    }
    p.tpr = (int)tpr;
    const int64_t chunks = chunks_for(tpr);
    p.rows_per_chunk = (outer + chunks - 1) / chunks;
    p.chunks = (outer + p.rows_per_chunk - 1) / p.rows_per_chunk;
    if (p.chunks < 1) p.chunks = 1;
    p.n_partials = p.chunks * p.ncols;
    p.fin_count = p.chunks * inner;
    p.fin_q = inner;
  }
  return p;
}

// a finalized statistics row in a workspace: fp64 sums, fp32 maxima and fp32 minima (line form), each 256-byte
// aligned
static inline int64_t stat_row_bytes(int64_t channels) {
  return (channels * 8 + 255) / 256 * 256 + 2 * ((channels * 4 + 255) / 256 * 256);
}

int64_t partial_bytes(int64_t n) {
  // amax(4) + mn(4) + mx(4) + pad(4) + asum(8) + nnz(8), each array 256-aligned
  auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
  return up(n * 4) * 3 + up(n * 8) * 2;
}

Partials partials_from_workspace(void *workspace, int64_t n_partials) {
  auto up = [](int64_t b) { return (b + 255) / 256 * 256; };
  uintptr_t base = (reinterpret_cast<uintptr_t>(workspace) + 255) / 256 * 256;
  Partials P;
  P.amax = reinterpret_cast<uint32_t *>(base); base += up(n_partials * 4);
  P.mn = reinterpret_cast<float *>(base);      base += up(n_partials * 4);
  P.mx = reinterpret_cast<float *>(base);      base += up(n_partials * 4);
  P.asum = reinterpret_cast<double *>(base);   base += up(n_partials * 8);
  P.nnz = reinterpret_cast<double *>(base);
  return P;
}

template <int WHAT, class Tail = NoTail, class T = float>
static int run_reduce(const T *x, const ReducePlan &pl, int64_t channels,
                      int64_t inner, const Partials &P, const FinalOut &out,
                      cudaStream_t stream, bool finalize = true, const Tail &tail = Tail{}) {
  // dynamic shared memory of the fused parameter step
  const size_t dyn = std::is_same<Tail, StepTail>::value ? step_smem_bytes((int)channels, kLineStep<WHAT>) : 0;
  if (pl.row_mode) {
    constexpr int kWarps = QSB_THREADS / 32;
    int64_t grid = (int64_t)device_props().sm_count * row_ctas_per_sm(pl.row_variant);
    const int64_t need = (pl.vwarps + kWarps - 1) / kWarps;
    if (grid > need) grid = need;
    auto go = [&](auto kernel) {
      return launch_k(kernel, dim3((unsigned)grid), dim3(QSB_THREADS), dyn, stream, x, pl.rows, inner, pl.seg,
                      pl.segs_per_row, pl.vwarps, P, pl.cta_combine, (int)channels, tail);
    };
    if (!is_half16<T> || aligned_to(x, 16)) {
      if (pl.row_variant == 2) QSB_CUDA_TRY(go(reduce_rows_kernel<WHAT, 8, 2, Tail, T>));
      else QSB_CUDA_TRY(go(reduce_rows_kernel<WHAT, 4, 4, Tail, T>));
    } else if constexpr (is_half16<T>) {
      if (pl.row_variant == 2) QSB_CUDA_TRY(go(reduce_rows_kernel<WHAT, 8, 2, Tail, T, false>));
      else QSB_CUDA_TRY(go(reduce_rows_kernel<WHAT, 4, 4, Tail, T, false>));
    }
  } else {
    const int64_t threads = pl.ncols / pl.vcol;
    dim3 grid((unsigned)((threads + pl.tpr - 1) / pl.tpr), (unsigned)pl.chunks);
    if (pl.vcol == 4)
      QSB_CUDA_TRY(launch_k(reduce_cols_kernel<WHAT, 4, Tail, T>, grid, dim3(QSB_THREADS), dyn, stream, x, pl.nrows,
                            pl.ncols, pl.rows_per_chunk, pl.tpr, P, tail));
    else
      QSB_CUDA_TRY(launch_k(reduce_cols_kernel<WHAT, 1, Tail, T>, grid, dim3(QSB_THREADS), dyn, stream, x, pl.nrows,
                            pl.ncols, pl.rows_per_chunk, pl.tpr, P, tail));
  }
  QSB_LAUNCH_CHECK();
  if (!finalize) return 0;
  // few channels: a whole CTA per channel; many: a warp per channel
  if (pl.fin_q == 1 && channels >= 8 && pl.fin_count >= 16 && pl.fin_count <= 1024) {
    QSB_CUDA_TRY(launch_k(reduce_finalize_t_kernel<WHAT>, dim3((unsigned)((channels + 7) / 8)), dim3(QSB_THREADS),
                          0, stream, P, out, channels, pl.fin_count));
  } else if (pl.fin_count > 1024 || (pl.fin_count >= 128 && channels <= 4 * device_props().sm_count)) {
    // a CTA per channel: many entries, or few channels (a warp per channel would leave the GPU empty)
    QSB_CUDA_TRY(launch_k(reduce_finalize_kernel<WHAT, QSB_THREADS>, dim3((unsigned)channels),
                          dim3(QSB_THREADS), 0, stream, P, out, channels, pl.fin_count, pl.fin_q));
  } else {
    constexpr int kPer = QSB_THREADS / 32;
    QSB_CUDA_TRY(launch_k(reduce_finalize_kernel<WHAT, 32>, dim3((unsigned)((channels + kPer - 1) / kPer)),
                          dim3(QSB_THREADS), 0, stream, P, out, channels, pl.fin_count, pl.fin_q));
  }
  QSB_LAUNCH_CHECK();
  return 0;
}

}  // namespace qsb

using namespace qsb;

#ifdef QSB_KERNEL_TIMING
namespace qsb {
int ktime_reduce_op(unsigned long long *out, cudaStream_t stream) { return ktime_host_op(out, stream); }
}
#endif

extern "C" int64_t qsb_reduce_workspace_bytes(int64_t outer, int64_t channels,
                                              int64_t inner) {
  if (outer <= 0 || channels <= 0 || inner <= 0) return 256;
  const ReducePlan pl = make_plan(outer, channels, inner, nullptr);
  // column mode falls back to scalar columns for an unaligned x: same row bands, same size.
  // + one finalized statistics row (fp64 sums | fp32 maxima) for the multi-launch form of the training step
  return partial_bytes(pl.n_partials) + 256 + stat_row_bytes(channels);
}

template <class T>
static int reduce_stats_impl(const T *x, int what, int64_t outer, int64_t channels, int64_t inner,
                             float *absmax, float *mn, float *mx, double *abssum, double *nnz,
                             float *tensor_min, void *workspace, int64_t workspace_bytes, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (outer <= 0 || channels <= 0 || inner <= 0) return QSB_E_BADARG;
  if (!x || !workspace) return QSB_E_BADARG;
  if (!aligned_to(x, sizeof(T))) return QSB_E_ALIGN;
  if ((what & ~(QSB_STAT_ABSMAX | QSB_STAT_MINMAX | QSB_STAT_ABSSUM |
                QSB_STAT_NNZ)) || what == 0)
    return QSB_E_BADARG;
  if ((what & QSB_STAT_NNZ) && !(what & QSB_STAT_ABSSUM)) return QSB_E_BADARG;
  const ReducePlan pl = make_plan(outer, channels, inner, x, (int)sizeof(T));
  if (workspace_bytes < partial_bytes(pl.n_partials) + 256) return QSB_E_WORKSPACE;
  const Partials P = partials_from_workspace(workspace, pl.n_partials);
  FinalOut out{absmax, mn, mx, abssum, nnz};
  int rc;
  auto go = [&](auto w) { return run_reduce<decltype(w)::value, NoTail, T>(x, pl, channels, inner, P, out, stream); };
  switch (what) {
#define QSB_CASE(W)                                  \
  case W:                                            \
    rc = go(std::integral_constant<int, W>{});       \
    break;
    QSB_CASE(QSB_STAT_ABSMAX)
    QSB_CASE(QSB_STAT_MINMAX)
    QSB_CASE(QSB_STAT_ABSSUM)
    QSB_CASE(QSB_STAT_ABSSUM | QSB_STAT_ABSMAX)
    QSB_CASE(QSB_STAT_ABSSUM | QSB_STAT_NNZ)
    QSB_CASE(QSB_STAT_ABSSUM | QSB_STAT_NNZ | QSB_STAT_ABSMAX)
    QSB_CASE(QSB_STAT_ABSMAX | QSB_STAT_MINMAX)
#undef QSB_CASE
    default:
      // any other combination: everything in one pass
      rc = go(std::integral_constant<int, QSB_STAT_ABSMAX | QSB_STAT_MINMAX | QSB_STAT_ABSSUM | QSB_STAT_NNZ>{});
  }
  if (rc) return rc;
  if ((what & QSB_STAT_NNZ) && tensor_min) {
    // the finalize wrote per-channel minima to `mn` if given, else we need a
    // scratch: reuse the (now consumed) first partial array.
    float *chan_min = mn;
    if (!chan_min) return QSB_E_BADARG;
    tensor_min_kernel<<<1, 32, 0, stream>>>(chan_min, channels, tensor_min);
    QSB_LAUNCH_CHECK();
  }
  return 0;
}

extern "C" int qsb_reduce_stats(const float *x, int what, int64_t outer, int64_t channels, int64_t inner,
                                float *absmax, float *mn, float *mx, double *abssum, double *nnz,
                                float *tensor_min, void *workspace, int64_t workspace_bytes, void *stream) {
  return reduce_stats_impl(x, what, outer, channels, inner, absmax, mn, mx, abssum, nnz, tensor_min, workspace,
                           workspace_bytes, stream);
}

extern "C" int qsb_reduce_stats_dt(const void *x, int x_dtype, int what, int64_t outer, int64_t channels,
                                   int64_t inner, float *absmax, float *mn, float *mx, double *abssum, double *nnz,
                                   float *tensor_min, void *workspace, int64_t workspace_bytes, void *stream) {
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    return reduce_stats_impl(static_cast<const T *>(x), what, outer, channels, inner, absmax, mn, mx, abssum, nnz,
                             tensor_min, workspace, workspace_bytes, stream);
  });
}

// Stage 1 only: leaves the per-virtual-warp partials of sum|x| and max|x| (WHAT: sum|x| and min / max x) in the
// workspace for qsb_prune_quant_step_params (qsb_prune_line_step_params), which finalizes them itself.
template <int WHAT>
static int reduce_partials_impl(const void *x_, int x_dtype, int64_t outer, int64_t channels, int64_t inner,
                                void *workspace, int64_t workspace_bytes, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!dtype_ok(x_dtype)) return QSB_E_BADARG;
  if (outer <= 0 || channels <= 0 || inner <= 0) return QSB_E_BADARG;
  if (!x_ || !workspace) return QSB_E_BADARG;
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    const T *x = static_cast<const T *>(x_);
    if (!aligned_to(x, sizeof(T))) return QSB_E_ALIGN;
    const ReducePlan pl = make_plan(outer, channels, inner, x, (int)sizeof(T));
    if (workspace_bytes < partial_bytes(pl.n_partials) + 256) return QSB_E_WORKSPACE;
    const Partials P = partials_from_workspace(workspace, pl.n_partials);
    FinalOut out{nullptr, nullptr, nullptr, nullptr, nullptr};
    return run_reduce<WHAT, NoTail, T>(x, pl, channels, inner, P, out, stream, /*finalize=*/false);
  });
}

extern "C" int qsb_reduce_partials_dt(const void *x, int x_dtype, int64_t outer, int64_t channels, int64_t inner,
                                      void *workspace, int64_t workspace_bytes, void *stream) {
  return reduce_partials_impl<QSB_STAT_ABSSUM | QSB_STAT_ABSMAX>(x, x_dtype, outer, channels, inner, workspace,
                                                                 workspace_bytes, stream);
}

extern "C" int qsb_reduce_line_partials_dt(const void *x, int x_dtype, int64_t outer, int64_t channels,
                                           int64_t inner, void *workspace, int64_t workspace_bytes, void *stream) {
  return reduce_partials_impl<QSB_STAT_ABSSUM | QSB_STAT_MINMAX>(x, x_dtype, outer, channels, inner, workspace,
                                                                 workspace_bytes, stream);
}

extern "C" int qsb_reduce_partials(const float *x, int64_t outer, int64_t channels, int64_t inner, void *workspace,
                                   int64_t workspace_bytes, void *stream) {
  return qsb_reduce_partials_dt(x, QSB_DTYPE_F32, outer, channels, inner, workspace, workspace_bytes, stream);
}

// the last-arriving CTA finalizes channels x fin_count partials; beyond this many a second, parallel
// finalize launch is cheaper than the serial tail (12 loads per thread and batch, 256 threads, <= 4 batches)
constexpr int64_t kStepTailMaxEntries = 12288;

// Stage 1 of the fused training step with its parameter step (step_epilogue.cuh): ONE launch whose
// last-arriving CTA finalizes the partials and runs the step.  With too many partials per channel (column mode
// on wide tensors) it is three launches instead: stage 1, a parallel finalize into a statistics row in the
// workspace, then the step kernel on that row.  `a` is filled by fill_step_args / fill_line_step_args;
// `keep_hint`: the previous step's mask (pow2 form) or NULL.
template <int WHAT, class T>
static int run_step(const T *x, int64_t outer, int64_t channels, int64_t inner, void *workspace,
                    int64_t workspace_bytes, unsigned int *arrival_counter_dev, StepArgs a, const uint8_t *keep_hint,
                    cudaStream_t stream) {
  const ReducePlan pl = make_plan(outer, channels, inner, x, (int)sizeof(T));
  if (workspace_bytes < partial_bytes(pl.n_partials) + 256) return QSB_E_WORKSPACE;
  if (pl.fin_count > 0x7fffffffLL || pl.fin_q > 0x7fffffffLL) return QSB_E_UNSUPPORTED;
  const Partials P = partials_from_workspace(workspace, pl.n_partials);
  if (channels * pl.fin_count > kStepTailMaxEntries) {
    if (workspace_bytes < partial_bytes(pl.n_partials) + 256 + stat_row_bytes(channels)) return QSB_E_WORKSPACE;
    unsigned char *row = reinterpret_cast<unsigned char *>(
        (reinterpret_cast<uintptr_t>(workspace) + 255) / 256 * 256 + (uintptr_t)partial_bytes(pl.n_partials));
    double *row_sum = reinterpret_cast<double *>(row);
    float *row_max = reinterpret_cast<float *>(row + (channels * 8 + 255) / 256 * 256);
    float *row_min = reinterpret_cast<float *>(reinterpret_cast<unsigned char *>(row_max) +
                                               (channels * 4 + 255) / 256 * 256);
    // the pow2 form finalizes max|x| into row_max, the line form min / max x into row_min / row_max
    const FinalOut out = kLineStep<WHAT> ? FinalOut{nullptr, row_min, row_max, row_sum, nullptr}
                                         : FinalOut{row_max, nullptr, nullptr, row_sum, nullptr};
    const int rc = run_reduce<WHAT, NoTail, T>(x, pl, channels, inner, P, out, stream);
    if (rc) return rc;
    if constexpr (kLineStep<WHAT>) a.row_min = row_min;
    a.timing = nullptr;  // the phase stamps are those of the one-launch kernel
    return launch_step_kernel_on_rows(a, row_sum, row_max, 1, 0, stream);
  }
  StepTail tail;
  tail.a = a;
  tail.a.P = P;
  tail.a.fin_count = (int)pl.fin_count;
  tail.a.fin_q = (int)pl.fin_q;
  tail.arrival = arrival_counter_dev;
  // channels the previous mask keeps are about to be re-read by the forward pass (only meaningful for a
  // per-channel mask in row mode)
  tail.keep_hint = (g_keep_hint && pl.row_mode && channels > 1) ? keep_hint : nullptr;
  FinalOut out{nullptr, nullptr, nullptr, nullptr, nullptr};
  return run_reduce<WHAT, StepTail, T>(x, pl, channels, inner, P, out, stream, /*finalize=*/false, tail);
}

// The fused structured prune -> pow2 quantize training step: the stage-1 reduction of sum|x| / max|x| whose
// last-arriving CTA finalizes, exchanges the statistics row with the peer GPUs and derives
// magnitude EMA / threshold / mask / scale / decimal (step_epilogue.cuh).
template <class T>
static int reduce_prune_quant_step_impl(
    const T *x, int64_t outer, int64_t channels, int64_t inner, void *workspace,
    int64_t workspace_bytes, unsigned int *arrival_counter_dev, float *magnitude, uint8_t *mask,
    float *scale, float *decimal_out, qsb_p2p_group *group, int64_t step_stamp, double count,
    int64_t t_prune, int update_magnitude, int refresh_mask, int64_t k, int bits, int64_t t_quant,
    int update_scale, double *abssum_out, float *absmax_out, int stats_local,
    int64_t *step_counter_dev, uint64_t *timing_out_dev, void *stream) {
  if (outer <= 0 || channels <= 0 || inner <= 0) return QSB_E_BADARG;
  if (channels > kStepFusedMaxChannels) return QSB_E_UNSUPPORTED;
  if (!x || !workspace || !arrival_counter_dev) return QSB_E_BADARG;
  if (!aligned_to(x, sizeof(T)) || !aligned_to(arrival_counter_dev, 4)) return QSB_E_ALIGN;
  StepArgs a;
  const int rc = fill_step_args(a, magnitude, mask, scale, decimal_out, channels, group, step_stamp, count,
                                t_prune, update_magnitude, refresh_mask, k, bits, t_quant, update_scale,
                                abssum_out, absmax_out, stats_local, step_counter_dev, QSB_THREADS);
  if (rc) return rc;
  a.timing = reinterpret_cast<unsigned long long *>(timing_out_dev);
  return run_step<QSB_STAT_ABSSUM | QSB_STAT_ABSMAX>(x, outer, channels, inner, workspace, workspace_bytes,
                                                     arrival_counter_dev, a, mask, (cudaStream_t)stream);
}

extern "C" int qsb_reduce_prune_quant_step_dt(
    const void *x, int x_dtype, int64_t outer, int64_t channels, int64_t inner, void *workspace,
    int64_t workspace_bytes, unsigned int *arrival_counter_dev, float *magnitude, uint8_t *mask,
    float *scale, float *decimal_out, qsb_p2p_group *group, int64_t step_stamp, double count,
    int64_t t_prune, int update_magnitude, int refresh_mask, int64_t k, int bits, int64_t t_quant,
    int update_scale, double *abssum_out, float *absmax_out, int stats_local,
    int64_t *step_counter_dev, uint64_t *timing_out_dev, void *stream) {
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    return reduce_prune_quant_step_impl(static_cast<const T *>(x), outer, channels, inner, workspace,
                                        workspace_bytes, arrival_counter_dev, magnitude, mask, scale, decimal_out,
                                        group, step_stamp, count, t_prune, update_magnitude, refresh_mask, k, bits,
                                        t_quant, update_scale, abssum_out, absmax_out, stats_local,
                                        step_counter_dev, timing_out_dev, stream);
  });
}

extern "C" int qsb_reduce_prune_quant_step(
    const float *x, int64_t outer, int64_t channels, int64_t inner, void *workspace,
    int64_t workspace_bytes, unsigned int *arrival_counter_dev, float *magnitude, uint8_t *mask,
    float *scale, float *decimal_out, qsb_p2p_group *group, int64_t step_stamp, double count,
    int64_t t_prune, int update_magnitude, int refresh_mask, int64_t k, int bits, int64_t t_quant,
    int update_scale, double *abssum_out, float *absmax_out, int stats_local,
    int64_t *step_counter_dev, uint64_t *timing_out_dev, void *stream) {
  return reduce_prune_quant_step_impl(x, outer, channels, inner, workspace, workspace_bytes, arrival_counter_dev,
                                      magnitude, mask, scale, decimal_out, group, step_stamp, count, t_prune,
                                      update_magnitude, refresh_mask, k, bits, t_quant, update_scale, abssum_out,
                                      absmax_out, stats_local, step_counter_dev, timing_out_dev, stream);
}

// The line form of the same step (AdaptiveQuantizer): the stage-1 reduction gathers sum|x| and min / max x, the
// last-arriving CTA runs finalize -> magnitude EMA -> threshold -> mask -> (min, max) of x * mask -> lines EMA.
// Same reduction plan, same summation order of sum|x| (the magnitudes equal those of the pow2 step bit for bit).
// No L2 keep hint: the line forward reads the pruned channels too.
extern "C" int qsb_reduce_prune_line_step_dt(
    const void *x, int x_dtype, int64_t outer, int64_t channels, int64_t inner, void *workspace,
    int64_t workspace_bytes, unsigned int *arrival_counter_dev, float *magnitude, uint8_t *mask, float *lines,
    int64_t n_lines, qsb_p2p_group *group, double count, int64_t t_prune, int update_magnitude, int refresh_mask,
    int64_t k, int64_t t_line, double *abssum_out, float *min_out, float *max_out, int64_t *step_counter_dev,
    void *stream) {
  if (!dtype_ok(x_dtype)) return QSB_E_BADARG;
  if (outer <= 0 || channels <= 0 || inner <= 0) return QSB_E_BADARG;
  if (!x || !workspace || !arrival_counter_dev) return QSB_E_BADARG;
  if (channels > kStepFusedMaxChannels) return QSB_E_UNSUPPORTED;
  StepArgs a;
  const int rc = fill_line_step_args(a, magnitude, mask, lines, n_lines, channels, group, count, t_prune,
                                     update_magnitude, refresh_mask, k, t_line, abssum_out, min_out, max_out,
                                     step_counter_dev);
  if (rc) return rc;
  return dispatch_dtype(x_dtype, [&](auto *tx) {
    using T = std::remove_pointer_t<decltype(tx)>;
    const T *xt = static_cast<const T *>(x);
    if (!aligned_to(xt, sizeof(T)) || !aligned_to(arrival_counter_dev, 4)) return QSB_E_ALIGN;
    return run_step<QSB_STAT_ABSSUM | QSB_STAT_MINMAX>(xt, outer, channels, inner, workspace, workspace_bytes,
                                                       arrival_counter_dev, a, nullptr, (cudaStream_t)stream);
  });
}
