// K5  exact k-th smallest value (0-based rank k) of n floats.  Replaces the reference's
// full sort (qsparse/util.py:113-116: values = sort(flat); thr = values[idx + 1]) —
// O(n) reads instead of O(n log n); the result equals sort()[k] (as a float; the sign
// of a zero result and the payload of a NaN result are not defined by sort either).
//
// Core: MSB-first radix select on the order-preserving uint32 key, digits 8 / 12 / 12:
//   pass 0: the top 8 bits (sign + 7 exponent bits) of real data land in a handful of
//           bins, so the shared-memory histogram is laid out [256 bins][32 lanes]:
//           lane l only ever touches bank l — no bank conflicts, no same-address
//           serialisation inside a warp.
//   pass 1/2: only elements whose higher bits equal the selected prefix are counted;
//           the tests run on the raw IEEE bits (inside one 8-bit key bucket every value
//           has the same sign, so "top bits of the key == prefix" is a compare of the raw
//           word against a per-launch constant).
// Each pass re-derives the prefix from the global histograms of the earlier passes in
// its prologue; the last CTA of pass 2 (atomic ticket) turns the histograms into the
// answer, so a select is memset + 3 launches.  Counters are 64-bit (n may exceed 2^32).
//
// Large inputs (n >= 2^22) first try a ~1-pass route:
//   sample    ONE CTA gathers 8192 evenly spaced values into shared memory and radix-
//             selects (top 22 key bits, in shared memory) the two order statistics
//             +-4.5 sigma (binomial rank error) around rank k * 8192 / n -> pivots
//             lo <= hi (floor / ceiling of the 22-bit prefixes).  The same CTA zeroes
//             the workspace header while its gathers are in flight (no memset node).
//   partition ONE streaming pass over v: every CTA counts its values < lo and appends
//             its values in [lo, hi] (~5 %) to a dense candidate array (one cursor
//             atomic per CTA; totals by fire-and-forget RED).
//   passes    radix select over the candidates on the RANGE-RELATIVE key
//             rel = key - key(lo) < 2^W, W = bits of key(hi) - key(lo) (~20): digits of
//             11 bits from bit W down, so two passes over the (L2-resident) candidates
//             finish W <= 22 and a third finishes any W.  Exact for any data: ties,
//             +-0 (canonicalised to +0), infinities.
// If rank k is not inside [lo, hi] (adversarial order) or the candidates do not fit
// (n/8 slots), the 3 generic passes run over v itself.  Fast and generic passes share
// the same three launches: the route is chosen ON THE DEVICE in the prologue of each
// pass from the counters — no host synchronisation, no extra launches.
#include <cooperative_groups.h>
#include <math.h>
#include <stddef.h>

#include "param_math.cuh"
#include "qsb_common.cuh"

namespace cg = cooperative_groups;

namespace qsb {

constexpr int kBits0 = 8, kBits1 = 12, kBits2 = 12;
constexpr int kBins0 = 1 << kBits0, kBins1 = 1 << kBits1, kBins2 = 1 << kBits2;
static_assert(kBins0 == QSB_THREADS, "pass-0 merge maps one thread to one bin");

// fast route
constexpr int kSampleThreads = 1024;
constexpr int kSampleCtas = 8;  // one thread-block cluster
// samples per sampler thread: four neighbours per location (one 128-bit load), 32 Ki samples for the lines
// 8 Ki single samples would touch — what matters for the layers of a weight set, where the sample is a
// visible fraction of the tensor
constexpr int kSamplePer = 4;
constexpr int kPartitionU = 4;  // 256-bit loads in flight per thread of the select's partition pass
constexpr int kFastBits = 11, kFastBins = 1 << kFastBits;
constexpr int kCandShift = 3;      // candidate slots = n >> 3 (12.5 %)
constexpr int kSegs = 32;          // independent candidate segments (one packed counter each)
constexpr int kCtasPerSeg = 18;
constexpr int kFastCtas = kSegs * kCtasPerSeg;  // CTAs of a pass that work on the candidates
constexpr int kSegStride = 16;     // counters are 128 B apart: same-line atomics serialise in L2
constexpr int64_t kFastMinN = 1 << 22;
constexpr uint32_t kKeyNegInf = 0x007fffffu, kKeyPosInf = 0xff800000u;
constexpr uint32_t kKeyNegZero = 0x7fffffffu, kKeyPosZero = 0x80000000u;

struct SelectWs {
  unsigned long long *hist0;  // [256]
  unsigned long long *hist1;  // [4096]
  unsigned long long *hist2;  // [4096]
};

// device-side state of one select call (zeroed at its start)
struct SelState {
  float lo, hi;                 // pivots
  uint32_t lo_key;              // key(lo); candidates have key - lo_key < 2^width
  uint32_t shift_a;             // digit A = rel >> shift_a
  uint32_t shift_b;             // digit B = (rel >> shift_b) & ..
  uint32_t width;               // W
  uint32_t tie_lo;              // values == lo are counted, not stored (heavy ties at lo, or lo == hi)
  uint32_t route;               // first pass's verdict: 1 = radix passes over the candidates,
                                // 2 = generic passes over v, 3 = the answer is lo (written)
  unsigned long long count_below;  // values < lo plus (ties) values == lo   (written by the first pass)
  uint32_t done;                // generic pass 2 ticket
  uint32_t done_b, done_c;      // fast pass tickets
  float mid;                    // fused prune step: provisional threshold (key midpoint of [lo, hi])
  uint32_t need_full;           // fused prune step: the provisional masks cannot be patched, redo them all
  uint32_t from_hint;           // the pivots came from the caller's hint, not from a sample
};

// Fused unstructured prune step (EMA -> threshold -> mask -> apply in ONE streaming pass, see
// qsb_prune_unstructured_step_batched): extra per-call constants of the magnitude EMA.
struct EmaC {
  float t_f, tp1, rcp;
  const long long *t_dev;  // optional device step counter (CUDA graphs): t = *t_dev + t_off, resolved by the kernel
  long long t_off;
};
// rcp: the host computes RN(1 / (t + 1)) with an IEEE division; __frcp_rn is the same correctly rounded value
__device__ __forceinline__ EmaC ema_resolve(EmaC ec) {
  if (ec.t_dev) {
    const long long t = __ldg(ec.t_dev) + ec.t_off;
    ec.t_f = (float)t;
    ec.tp1 = (float)(t + 1);
    ec.rcp = __frcp_rn(ec.tp1);
  }
  return ec;
}
static_assert(offsetof(SelState, lo) == 0 && offsetof(SelState, hi) == 4, "the partition kernel loads both pivots at once");

// ---------------------------------------------------------------------------
// Pivot hints (warm start).  A training loop asks for the SAME order statistic of a slowly drifting
// tensor every step (the running-average magnitudes of a layer: mag_t = (t mag_{t-1} + |w|) / (t + 1)),
// so the previous answer brackets the next one far better than 32 Ki fresh samples do.  The caller may
// keep 8 words of state per tensor ("hint", zero-initialised) across calls:
//   [0] state: 0 nothing, 1 one answer seen (the next call still samples), 2 pivots available
//   [1] key of the last answer      [2] delta: half-width of the next pivot bracket, in key steps (ulps)
// With state 2 the sampler kernel does not sample at all — it only zeroes the header and publishes
// lo / hi = last answer -/+ delta — and the bracket is so tight (a few thousand candidates instead of
// 2.5 % of n) that the candidate passes and the fix-up of the fused prune step become trivial.  The
// answer is exact whatever the hint says: if rank k is not inside [lo, hi] the device takes the generic
// route exactly as for a missed sample bracket, and the hint widens (delta x 8) or falls back to state 1.
// After every call: delta = max(8 x |key drift|, delta / 2, 64).
// ---------------------------------------------------------------------------
constexpr uint32_t kHintMinDelta = 64, kHintMaxDelta = 1u << 24;
__device__ __forceinline__ void hint_update(uint32_t *hint, float thr, bool missed) {
  if (!hint) return;
  if (thr != thr) {  // a NaN threshold cannot bracket anything
    hint[0] = 0;
    return;
  }
  const uint32_t key = float_to_key(thr + 0.0f), state = hint[0], old = hint[1], delta = hint[2];
  if (state == 0) {
    hint[0] = 1, hint[1] = key, hint[2] = 0;
    return;
  }
  const unsigned long long drift = key > old ? key - old : old - key;
  unsigned long long nd = 8ull * drift;
  if (state == 2) {
    if (missed) nd += 8ull * delta;
    else if (nd < delta / 2) nd = delta / 2;
  }
  if (nd < kHintMinDelta) nd = kHintMinDelta;
  hint[1] = key;
  if (nd > kHintMaxDelta) {  // too wide to be worth it: the next call samples again
    hint[0] = 1, hint[2] = 0;
    return;
  }
  hint[0] = 2, hint[2] = (uint32_t)nd;
}

#ifdef QSB_SELECT_TIMING
#define QSB_TICK(st, slot)                                                      \
  do {                                                                          \
    if (threadIdx.x == 0 && blockIdx.x == 0)                                    \
      reinterpret_cast<long long *>(st)[16 + (slot)] = clock64();               \
  } while (0)
#else
#define QSB_TICK(st, slot) do {} while (0)
#endif

// Candidates live in kSegs dense segments.  Segment s has ONE packed 64-bit counter
// (segctr[s * kSegStride]): low 32 bits = candidates appended (also the append cursor),
// high 32 bits = values < lo seen by the CTAs that use the segment — a partition CTA
// issues a single atomic, and the kSegs counters sit in different 128-byte lines.  The
// next word of the line counts the values == lo when those are not stored (tie_lo).
struct FastBufs {
  const SelState *st;              // nullptr: there is no fast route (small n)
  const float *cand;               // [kSegs][seg_cap], 32-byte aligned, |.| already applied
  const unsigned long long *segctr;
  uint32_t *fh;                    // [3][kFastBins] histograms of the range-relative digits
  uint32_t seg_cap;                // slots per segment (multiple of 8)
  uint32_t *hint;                  // caller's pivot hint (may be null)
};

// Totals of the packed counters -> where is rank k?  Pass 0: every CTA derives the route
// from the counters (CTA 0 also records it, and writes the answer when it is lo itself);
// later passes read the record.  Returns the route; *k_in_cand = rank among the candidates.
__device__ uint32_t fast_route(const FastBufs &fb, SelState *st_rw, int pass,
                               unsigned long long k, unsigned long long *k_in_cand,
                               float *thr_out) {
  __shared__ unsigned long long s_below;
  __shared__ uint32_t s_route;
  if (pass > 0) {
    *k_in_cand = k - fb.st->count_below;
    return fb.st->route;
  }
  if (threadIdx.x < 32) {
    static_assert(kSegs == 32, "one lane per segment");
    const ulonglong2 c2 =
        __ldcg(reinterpret_cast<const ulonglong2 *>(fb.segctr + threadIdx.x * kSegStride));
    const uint32_t cand = (uint32_t)c2.x;
    unsigned long long lt = c2.x >> 32, eq = c2.y, nc = cand;
    int over = cand > fb.seg_cap;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      lt += __shfl_xor_sync(0xffffffffu, lt, o);
      eq += __shfl_xor_sync(0xffffffffu, eq, o);
      nc += __shfl_xor_sync(0xffffffffu, nc, o);
      over |= __shfl_xor_sync(0xffffffffu, over, o);
    }
    if (threadIdx.x == 0) {
      uint32_t route = 2;
      if (k >= lt) {
        if (k - lt < eq) route = 3;
        else if (!over && k - lt - eq < nc) route = 1;
      }
      s_below = lt + eq;
      s_route = route;
      if (blockIdx.x == 0) {
        st_rw->count_below = lt + eq;
        st_rw->route = route;
        // (fused prune step) ties at lo were provisionally pruned and are not in the candidate list
        st_rw->need_full = (route == 2) || (route == 3 && fb.st->width > 0);
        if (route == 3) {
          *thr_out = fb.st->lo;
          hint_update(fb.hint, fb.st->lo, false);
        }
      }
    }
  }
  __syncthreads();
  *k_in_cand = k - s_below;
  return s_route;
}

// Find the bin where the running count first exceeds k; result broadcast to the CTA.
// REPS > 1: the histogram is the sum of REPS replicas, BINS apart.
template <int BINS, int REPS = 1, class T>
__device__ void find_bin(const T *hist, unsigned long long k, uint32_t *bin_out,
                         unsigned long long *k_out) {
  constexpr int PER = (BINS + QSB_THREADS - 1) / QSB_THREADS;
  __shared__ unsigned long long s_warp[QSB_THREADS / 32];
  __shared__ uint32_t s_bin;
  __shared__ unsigned long long s_k;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  unsigned long long local[PER];
  unsigned long long sum = 0;
  // L2 loads (__ldcg): the counters were written by other CTAs' atomics.  Every CTA of a
  // pass reads the same few lines, so use the widest loads (fewest requests per line).
  if constexpr (sizeof(T) == 4 && PER % 4 == 0) {
#pragma unroll
    for (int i = 0; i < PER; i += 4) {
      local[i] = local[i + 1] = local[i + 2] = local[i + 3] = 0;
#pragma unroll
      for (int r = 0; r < REPS; ++r) {
        const uint4 q = __ldcg(reinterpret_cast<const uint4 *>(hist + r * BINS + tid * PER + i));
        local[i] += q.x, local[i + 1] += q.y, local[i + 2] += q.z, local[i + 3] += q.w;
      }
    }
  } else if constexpr (sizeof(T) == 8 && PER % 2 == 0) {
#pragma unroll
    for (int i = 0; i < PER; i += 2) {
      const ulonglong2 q = __ldcg(reinterpret_cast<const ulonglong2 *>(hist + tid * PER + i));
      local[i] = q.x, local[i + 1] = q.y;
    }
  } else {
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int b = tid * PER + i;
      local[i] = (b < BINS) ? (unsigned long long)__ldcg(hist + b) : 0ull;
    }
  }
#pragma unroll
  for (int i = 0; i < PER; ++i) sum += local[i];
  unsigned long long incl = sum;  // block-wide exclusive scan: shuffles + one smem hop
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) s_warp[warp] = incl;
  if (tid == 0) {
    s_bin = BINS - 1;
    s_k = 0;
  }
  __syncthreads();
  unsigned long long before = incl - sum;
  for (int w = 0; w < warp; ++w) before += s_warp[w];
  if (k >= before && k < before + sum) {
    unsigned long long run = before;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      if (k < run + local[i]) {
        s_bin = tid * PER + i;
        s_k = k - run;
        break;
      }
      run += local[i];
    }
  }
  __syncthreads();
  *bin_out = s_bin;
  *k_out = s_k;
  __syncthreads();
}

struct PassConst {
  uint32_t raw_prefix;  // PASS 1: wanted raw bits >> 24; PASS 2: wanted raw bits >> 12
  uint32_t flip;        // 0xfff for a negative bucket (key = ~bits), else 0
};

__device__ __forceinline__ PassConst make_pass_const(int pass, uint32_t key_prefix) {
  PassConst pc;
  if (pass == 1) {
    const bool neg = (key_prefix & 0x80u) == 0;  // key top bit clear <=> negative
    pc.raw_prefix = neg ? (key_prefix ^ 0xffu) : (key_prefix ^ 0x80u);
    pc.flip = neg ? 0xfffu : 0u;
  } else {
    const bool neg = (key_prefix & 0x80000u) == 0;
    pc.raw_prefix = neg ? (~key_prefix & 0xfffffu) : (key_prefix ^ 0x80000u);
    pc.flip = neg ? 0xfffu : 0u;
  }
  return pc;
}

// Only negative NaNs need a fix up front (every NaN must order last): remapped to 0x7fffffff.
template <int PASS, bool ABS>
__device__ __forceinline__ void count_value(float f, const PassConst &pc,
                                            uint32_t *s_hist, int lane) {
  uint32_t b = __float_as_uint(f);
  if constexpr (ABS) b &= 0x7fffffffu;
  else b = (b > 0xff800000u) ? 0x7fffffffu : b;
  if constexpr (PASS == 0) {
    const uint32_t t = b >> 24;
    const uint32_t digit = ((int32_t)b < 0) ? (t ^ 0xffu) : (t | 0x80u);
    atomicAdd(&s_hist[digit * 32 + lane], 1u);
  } else if constexpr (PASS == 1) {
    if ((b >> 24) == pc.raw_prefix)
      atomicAdd(&s_hist[((b >> 12) & 0xfffu) ^ pc.flip], 1u);
  } else {
    if ((b >> 12) == pc.raw_prefix) atomicAdd(&s_hist[(b & 0xfffu) ^ pc.flip], 1u);
  }
}

// ---------------------------------------------------------------------------
// fast route: passes over the candidate segments
// ---------------------------------------------------------------------------
// key of a candidate; -0.0 was never stored as such but be safe: x + 0 canonicalises it
__device__ __forceinline__ uint32_t cand_rel(float f, uint32_t lo_key) {
  const uint32_t b = __float_as_uint(f + 0.0f);
  const uint32_t key = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return key - lo_key;
}

// STAGE 0: digit A of every candidate.  STAGE 1: digit B of those whose digit A is the
// selected one.  STAGE 2: the low bits of those whose digits A and B are selected.
// (Counting digit A inside the partition kernel was tried twice and lost: atomic
// transactions to one 128-byte line serialise at ~2.6 ns in L2, so one RED per candidate
// (2.4 M on 64 lines) cost +100 us, and a per-CTA shared-memory histogram flushed with
// line-coalesced REDs (8192 CTAs x 32 lines) cost +15 us against the 10 us pass it saves.)
template <int STAGE>
__device__ __forceinline__ void fast_count(float f, uint32_t lo_key, uint32_t shift,
                                           uint32_t want_shift, uint32_t want,
                                           uint32_t mask, uint32_t *s_hist) {
  const uint32_t rel = cand_rel(f, lo_key);
  if constexpr (STAGE == 0) {
    atomicAdd(&s_hist[rel >> shift], 1u);
  } else {
    if ((rel >> want_shift) == want) atomicAdd(&s_hist[(rel >> shift) & mask], 1u);
  }
}

template <int STAGE>
__device__ void fast_pass(const FastBufs &fb, unsigned long long kc, SelState *st_rw,
                          float *thr_out, uint32_t *s_hist, int *s_last) {
  const SelState *st = fb.st;
  const int tid = threadIdx.x;
  QSB_TICK(st_rw, 8 + STAGE * 8 + 1);
  const uint32_t lo_key = st->lo_key, shift_a = st->shift_a, shift_b = st->shift_b;
  if (STAGE == 2 && shift_b == 0) return;  // stage 1 already wrote the answer
  // a multiple of kSegs CTAs works on the candidates (the grid has >= kSegs CTAs: n >= 2^22)
  const unsigned nctas = gridDim.x < (unsigned)kFastCtas ? gridDim.x / kSegs * kSegs : (unsigned)kFastCtas;
  if (blockIdx.x >= nctas) return;
  uint32_t b0 = 0, b1 = 0;
  unsigned long long k1 = kc, k2 = 0;
  if constexpr (STAGE >= 1) {
    find_bin<kFastBins>(fb.fh, kc, &b0, &k1);
    if (shift_a == 0) {  // the whole range fitted digit A
      if (STAGE == 1 && blockIdx.x == 0 && tid == 0) {
        *thr_out = key_to_float(lo_key + b0);
        hint_update(fb.hint, *thr_out, false);
      }
      return;
    }
  }
  if constexpr (STAGE == 2) find_bin<kFastBins>(fb.fh + kFastBins, k1, &b1, &k2);
  const uint32_t bits_b = shift_a - shift_b;
  uint32_t shift, want_shift = 0, want = 0, mask = 0;
  if constexpr (STAGE == 0) {
    shift = shift_a;
  } else if constexpr (STAGE == 1) {
    shift = shift_b, want_shift = shift_a, want = b0, mask = (1u << bits_b) - 1u;
  } else {
    shift = 0, want_shift = shift_b, want = (b0 << bits_b) | b1, mask = (1u << shift_b) - 1u;
  }
  QSB_TICK(st_rw, 8 + STAGE * 8 + 2);
  for (int i = tid; i < kFastBins; i += QSB_THREADS) s_hist[i] = 0;
  __syncthreads();
  // kCtasPerSeg CTAs share one segment
  const int seg = blockIdx.x % kSegs, part = blockIdx.x / kSegs, parts = nctas / kSegs;
  const uint32_t nc = (uint32_t)__ldcg(fb.segctr + seg * kSegStride), n4 = nc >> 2;
  const float *cseg = fb.cand + (size_t)seg * fb.seg_cap;
  const float4 *c4 = reinterpret_cast<const float4 *>(cseg);
  const uint32_t step = (uint32_t)parts * QSB_THREADS;
  uint32_t i = (uint32_t)part * QSB_THREADS + tid;
  for (; i < n4; i += 4 * step) {  // four 128-bit loads in flight
    float4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i + u * step < n4) q[u] = c4[i + u * step];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i + u * step < n4) {
        fast_count<STAGE>(q[u].x, lo_key, shift, want_shift, want, mask, s_hist);
        fast_count<STAGE>(q[u].y, lo_key, shift, want_shift, want, mask, s_hist);
        fast_count<STAGE>(q[u].z, lo_key, shift, want_shift, want, mask, s_hist);
        fast_count<STAGE>(q[u].w, lo_key, shift, want_shift, want, mask, s_hist);
      }
  }
  if (part == 0 && tid < (int)(nc & 3))
    fast_count<STAGE>(cseg[(n4 << 2) + tid], lo_key, shift, want_shift, want, mask, s_hist);
  __syncthreads();
  QSB_TICK(st_rw, 8 + STAGE * 8 + 3);
  uint32_t *g = fb.fh + STAGE * kFastBins;
  for (int b = tid; b < kFastBins; b += QSB_THREADS) {
    const uint32_t c = s_hist[b];
    if (c) atomicAdd(&g[b], c);  // result unused: RED
  }
  QSB_TICK(st_rw, 8 + STAGE * 8 + 4);
  const bool finishes = (STAGE == 1 && shift_b == 0) || STAGE == 2;
  if (!finishes) return;
  __threadfence();
  __syncthreads();
  if (tid == 0)
    *s_last = (atomicAdd(STAGE == 1 ? &st_rw->done_b : &st_rw->done_c, 1u) == nctas - 1);
  __syncthreads();
  if (!*s_last) return;
  if constexpr (STAGE == 1) {
    find_bin<kFastBins>(fb.fh + kFastBins, k1, &b1, &k2);
    if (tid == 0) {
      *thr_out = key_to_float(lo_key + (b0 << shift_a) + b1);
      hint_update(fb.hint, *thr_out, false);
    }
  } else if constexpr (STAGE == 2) {
    uint32_t b2;
    unsigned long long k3;
    find_bin<kFastBins>(fb.fh + 2 * kFastBins, k2, &b2, &k3);
    if (tid == 0) {
      *thr_out = key_to_float(lo_key + (b0 << shift_a) + (b1 << shift_b) + b2);
      hint_update(fb.hint, *thr_out, false);
    }
  }
}

// ---------------------------------------------------------------------------
// one radix pass; route chosen on the device
// ---------------------------------------------------------------------------
template <int PASS, int V, bool ABS>
__device__ __forceinline__ void select_pass_body(const float *__restrict__ v, int64_t n, int64_t k,
                                                 SelectWs ws, FastBufs fb, SelState *st_rw,
                                                 float *thr_out, uint32_t *hint) {
  constexpr int kSmemWords = (PASS == 0) ? kBins0 * 32 : kBins1;
  static_assert(kSmemWords >= kFastBins, "the fast passes reuse the histogram");
  __shared__ uint32_t s_hist[kSmemWords];
  __shared__ int s_last;
  const int tid = threadIdx.x, lane = tid & 31;
  const unsigned long long kk = (unsigned long long)k;
  pdl_wait();     // everything below reads what the previous launch of the chain wrote
  pdl_trigger();  // the next launch may take the SM resources this grid leaves free
  if (fb.st) QSB_TICK(st_rw, 8 + PASS * 8 + 0);
  if (fb.st) {
    unsigned long long kc;
    const uint32_t route = fast_route(fb, st_rw, PASS, kk, &kc, thr_out);
    if (route == 3) return;  // the answer was lo
    if (route == 1) {
      fast_pass<PASS>(fb, kc, st_rw, thr_out, s_hist, &s_last);
      return;
    }
  }
  for (int i = tid; i < kSmemWords; i += QSB_THREADS) s_hist[i] = 0;
  PassConst pc{0, 0};
  if constexpr (PASS >= 1) {
    unsigned long long k1;
    uint32_t b0;
    find_bin<kBins0>(ws.hist0, kk, &b0, &k1);
    uint32_t prefix = b0;
    if constexpr (PASS == 2) {
      uint32_t b1;
      find_bin<kBins1>(ws.hist1, k1, &b1, &k1);
      prefix = (b0 << 12) | b1;
    }
    pc = make_pass_const(PASS, prefix);
  }
  __syncthreads();

  {
    constexpr int U = (V == 8) ? 2 : 4;
    constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
    const int64_t n_main = (n / V) * V;
    for (int64_t base = (int64_t)blockIdx.x * kTile + (int64_t)tid * V; base < n_main;
         base += (int64_t)gridDim.x * kTile) {
      VecF<V> x[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t e = base + (int64_t)u * QSB_THREADS * V;
        if (e < n_main) x[u] = ld_vec<V, Hint::KEEP>(v + e);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int64_t e = base + (int64_t)u * QSB_THREADS * V;
        if (e < n_main) {
#pragma unroll
          for (int j = 0; j < V; ++j) count_value<PASS, ABS>(x[u].v[j], pc, s_hist, lane);
        }
      }
    }
    if (blockIdx.x == 0) {
      const int64_t e = n_main + tid;
      if (e < n) count_value<PASS, ABS>(v[e], pc, s_hist, lane);
    }
  }
  __syncthreads();

  if constexpr (PASS == 0) {
    // bin = tid; rotate the lane index so the 32 reads of a warp hit 32 banks
    unsigned long long sum = 0;
#pragma unroll 8
    for (int l = 0; l < 32; ++l) sum += s_hist[tid * 32 + ((l + tid) & 31)];
    if (sum) atomicAdd(&ws.hist0[tid], sum);
  } else {
    unsigned long long *g = (PASS == 1) ? ws.hist1 : ws.hist2;
    for (int b = tid; b < kBins1; b += QSB_THREADS) {
      const uint32_t c = s_hist[b];
      if (c) atomicAdd(&g[b], (unsigned long long)c);
    }
  }

  if constexpr (PASS == 2) {
    // the last CTA to finish turns the three histograms into the answer
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = (atomicAdd(&st_rw->done, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
      unsigned long long k1;
      uint32_t b0, b1, b2;
      find_bin<kBins0>(ws.hist0, kk, &b0, &k1);
      find_bin<kBins1>(ws.hist1, k1, &b1, &k1);
      find_bin<kBins2>(ws.hist2, k1, &b2, &k1);
      if (tid == 0 && thr_out) {
        *thr_out = key_to_float((b0 << 24) | (b1 << 12) | b2);
        // the generic route after hinted pivots = the bracket missed rank k
        hint_update(hint, *thr_out, fb.st != nullptr && fb.st->from_hint != 0);
      }
    }
  }
}

// the answer from three (globally complete) histograms: the last step of a select whose
// histograms were summed over several GPUs between the passes
__global__ void __launch_bounds__(QSB_THREADS)
    select_final_kernel(SelectWs ws, int64_t k, float *thr_out) {
  unsigned long long k1;
  uint32_t b0, b1, b2;
  find_bin<kBins0>(ws.hist0, (unsigned long long)k, &b0, &k1);
  find_bin<kBins1>(ws.hist1, k1, &b1, &k1);
  find_bin<kBins2>(ws.hist2, k1, &b2, &k1);
  if (threadIdx.x == 0) *thr_out = key_to_float((b0 << 24) | (b1 << 12) | b2);
}

// ---------------------------------------------------------------------------
// fast route, step 1: pivots.  ONE cluster of 8 CTAs x 1024 threads, one sample per
// thread (a single SM cannot issue 8192 scattered sector requests in less than ~8 us;
// eight SMs can).  The CTAs zero the workspace header while the gathers fly, histogram
// their keys' top 11 bits in their own shared memory, and CTA 0 adds the eight
// histograms through distributed shared memory and finds the bins of the sample ranks
// r_lo and r_hi; a second round does the same for the next 11 bits under those two
// prefixes.  lo = floor, hi = ceiling of the selected 22-bit prefixes.
// ---------------------------------------------------------------------------
// bins where the running count first exceeds rank r_a in hist_a and r_b in hist_b (the
// two may be the same array): ONE block scan for both (1024 threads, 2 bins each).
// out[0..2] = bin, rank inside the bin, count of the bin for a; out[3..5] for b.
__device__ void sample_find2(const uint32_t *hist_a, int r_a, const uint32_t *hist_b, int r_b,
                             uint32_t *s_scan, uint32_t *out) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint2 ca = reinterpret_cast<const uint2 *>(hist_a)[tid];
  const uint2 cb = reinterpret_cast<const uint2 *>(hist_b)[tid];
  const uint32_t sum_a = ca.x + ca.y, sum_b = cb.x + cb.y;
  uint32_t ia = sum_a, ib = sum_b;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t ta = __shfl_up_sync(0xffffffffu, ia, o);
    const uint32_t tb = __shfl_up_sync(0xffffffffu, ib, o);
    if (lane >= o) ia += ta, ib += tb;
  }
  if (lane == 31) s_scan[warp] = ia, s_scan[32 + warp] = ib;
  __syncthreads();
  if (warp < 2) {
    const uint32_t w = s_scan[warp * 32 + lane];
    uint32_t wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    s_scan[64 + warp * 32 + lane] = wi - w;  // exclusive warp offsets
  }
  __syncthreads();
  const uint32_t before_a = s_scan[64 + warp] + ia - sum_a, before_b = s_scan[96 + warp] + ib - sum_b;
  const uint32_t ua = (uint32_t)r_a, ub = (uint32_t)r_b;
  if (ua >= before_a && ua < before_a + sum_a) {
    const bool first = ua < before_a + ca.x;
    out[0] = 2 * tid + (first ? 0 : 1);
    out[1] = ua - before_a - (first ? 0 : ca.x);
    out[2] = first ? ca.x : ca.y;
  }
  if (ub >= before_b && ub < before_b + sum_b) {
    const bool first = ub < before_b + cb.x;
    out[3] = 2 * tid + (first ? 0 : 1);
    out[4] = ub - before_b - (first ? 0 : cb.x);
    out[5] = first ? cb.x : cb.y;
  }
  __syncthreads();
}

// CTA 0 of the cluster: h[b] += the same bin of the other CTAs' histograms
__device__ __forceinline__ void cluster_sum_hist(cg::cluster_group &cluster, uint32_t *h) {
  uint2 acc = reinterpret_cast<uint2 *>(h)[threadIdx.x];
#pragma unroll
  for (int r = 1; r < kSampleCtas; ++r) {
    const uint2 q = reinterpret_cast<const uint2 *>(cluster.map_shared_rank(h, r))[threadIdx.x];
    acc.x += q.x;
    acc.y += q.y;
  }
  reinterpret_cast<uint2 *>(h)[threadIdx.x] = acc;
}

template <int PER, bool STEP>
__device__ __forceinline__ void select_sample_body(const float *__restrict__ v, int64_t n,
                                                   int take_abs, int r_lo, int r_hi, SelState *st,
                                                   uint4 *zero_base, int zero_vecs,
                                                   const float *__restrict__ w, EmaC ec,
                                                   const uint32_t *hint) {
  static_assert(kFastBins == 2 * kSampleThreads, "two bins per thread");
  static_assert(PER == 4, "four neighbours per sampler thread: one 128-bit load");
  constexpr int kSampleSize = kSampleThreads * kSampleCtas * PER;
  constexpr int kTieMinCount = kSampleSize / 50;  // >= 2 % of the sample in lo's bucket: ties at lo
  cg::cluster_group cluster = cg::this_cluster();
  __shared__ __align__(16) uint32_t h0[kFastBins];  // top 11 bits
  __shared__ __align__(16) uint32_t ha[kFastBins];  // next 11 bits under r_lo's prefix
  __shared__ __align__(16) uint32_t hb[kFastBins];  // next 11 bits under r_hi's prefix
  __shared__ uint32_t s_scan[128];
  __shared__ uint32_t s_res[12];  // [0..5] first digit (bin, rank, count) x (lo, hi); [6..11] second
  const int tid = threadIdx.x;
  const unsigned rank = cluster.block_rank();
  const int i = (int)rank * kSampleThreads + tid;
#ifdef QSB_SELECT_TIMING
  const long long t_start = clock64();
#endif
  pdl_wait();     // v may come from the kernel launched just before (e.g. the magnitude EMA)
  pdl_trigger();  // the partition kernel may start loading v on the other SMs right away
  if (hint && hint[0] == 2) {
    // warm start: no sample at all — zero the header, then publish last answer -/+ delta as the pivots
    const uint32_t thr_key = hint[1], delta = hint[2];
    for (int j = i; j < zero_vecs; j += kSampleThreads * kSampleCtas) zero_base[j] = make_uint4(0, 0, 0, 0);
    cluster.sync();  // the header (SelState included) is zero before it is written
    if (rank == 0 && tid == 0) {
      uint32_t lo_key = thr_key > kKeyNegInf + delta ? thr_key - delta : kKeyNegInf;
      uint32_t hi_key = thr_key < kKeyPosInf - delta ? thr_key + delta : kKeyPosInf;
      if (lo_key < kKeyNegInf) lo_key = kKeyNegInf;
      if (hi_key > kKeyPosInf) hi_key = kKeyPosInf;
      if (lo_key == kKeyNegZero) lo_key = kKeyPosZero;  // stored candidates are canonical (+0)
      if (hi_key == kKeyNegZero) hi_key = kKeyPosZero;
      if (hi_key < lo_key) hi_key = lo_key;
      const uint32_t span = hi_key - lo_key;
      const uint32_t width = span ? 32u - (uint32_t)__clz(span) : 0u;
      st->lo = key_to_float(lo_key);
      st->hi = key_to_float(hi_key);
      st->lo_key = lo_key;
      st->width = width;
      st->shift_a = width > (uint32_t)kFastBits ? width - kFastBits : 0u;
      st->shift_b = width > 2u * kFastBits ? width - 2u * kFastBits : 0u;
      st->tie_lo = (span == 0u);
      st->mid = key_to_float(lo_key + (span >> 1) + (span & 1u));
      st->from_hint = 1;
    }
    return;
  }
  float f[PER];
  // four neighbours per location: one 128-bit load
  const int64_t stride4 = n / (kSampleThreads * kSampleCtas);
  const int64_t at = ((int64_t)i * stride4 + (stride4 >> 1)) & ~(int64_t)3;
  const float4 q4 = *reinterpret_cast<const float4 *>(v + at);
  f[0] = q4.x, f[1] = q4.y, f[2] = q4.z, f[3] = q4.w;
  if constexpr (STEP) {  // fused prune step: sample the magnitudes the EMA is ABOUT to produce
    const float4 w4 = *reinterpret_cast<const float4 *>(w + at);
    f[0] = ema_full_step(f[0], w4.x, ec.t_f, ec.tp1, ec.rcp);
    f[1] = ema_full_step(f[1], w4.y, ec.t_f, ec.tp1, ec.rcp);
    f[2] = ema_full_step(f[2], w4.z, ec.t_f, ec.tp1, ec.rcp);
    f[3] = ema_full_step(f[3], w4.w, ec.t_f, ec.tp1, ec.rcp);
  }
  for (int j = i; j < zero_vecs; j += kSampleThreads * kSampleCtas) zero_base[j] = make_uint4(0, 0, 0, 0);
  reinterpret_cast<uint2 *>(h0)[tid] = make_uint2(0, 0);
  reinterpret_cast<uint2 *>(ha)[tid] = make_uint2(0, 0);
  reinterpret_cast<uint2 *>(hb)[tid] = make_uint2(0, 0);
  if (tid < 12) s_res[tid] = 0;
  __syncthreads();
  uint32_t key[PER];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    key[q] = float_to_key((take_abs ? fabsf(f[q]) : f[q]) + 0.0f);  // -0 -> +0
    atomicAdd(&h0[key[q] >> 21], 1u);
  }
  cluster.sync();
  QSB_TICK(st, 1);
  if (rank == 0) {
    cluster_sum_hist(cluster, h0);
    __syncthreads();
    // r_hi >= kSampleSize: hi = +inf.  r_lo < 0: lo = -inf, unless the smallest sample's
    // bucket is a heavy tie (the zeros of a ReLU output) — then that value is lo.
    sample_find2(h0, r_lo >= 0 ? r_lo : 0, h0, r_hi < kSampleSize ? r_hi : kSampleSize - 1, s_scan, s_res);
  }
  cluster.sync();
  QSB_TICK(st, 2);
  const uint32_t *res0 = cluster.map_shared_rank(s_res, 0);
  const uint32_t p_lo = res0[0], p_hi = res0[3];
#pragma unroll
  for (int q = 0; q < PER; ++q) {
    const uint32_t top = key[q] >> 21, mid = (key[q] >> 10) & (kFastBins - 1);
    if (top == p_lo) atomicAdd(&ha[mid], 1u);
    if (top == p_hi) atomicAdd(&hb[mid], 1u);
  }
  cluster.sync();
  QSB_TICK(st, 3);
  if (rank == 0) {
    cluster_sum_hist(cluster, ha);
    cluster_sum_hist(cluster, hb);
    __syncthreads();
    sample_find2(ha, (int)s_res[1], hb, (int)s_res[4], s_scan, s_res + 6);
    QSB_TICK(st, 4);
    if (tid == 0) {
      const bool lo_tie = s_res[8] >= (uint32_t)kTieMinCount;
      uint32_t lo_key = (r_lo >= 0 || lo_tie) ? ((p_lo << 21) | (s_res[6] << 10)) : kKeyNegInf;
      uint32_t hi_key = (r_hi < kSampleSize) ? ((p_hi << 21) | (s_res[9] << 10) | 0x3ffu) : kKeyPosInf;
      // keep both pivots ordinary floats whose compare order equals the (canonical) key order
      if (lo_key < kKeyNegInf) lo_key = kKeyNegInf;
      if (hi_key > kKeyPosInf) hi_key = kKeyPosInf;
      if (hi_key == kKeyNegZero) hi_key = kKeyPosZero;  // a <= -0.0 also admits +0.0
      if (hi_key < lo_key) hi_key = lo_key;
      const uint32_t span = hi_key - lo_key;
      const uint32_t width = span ? 32u - (uint32_t)__clz(span) : 0u;
      st->lo = key_to_float(lo_key);
      st->hi = key_to_float(hi_key);
      st->lo_key = lo_key;
      st->width = width;
      st->shift_a = width > (uint32_t)kFastBits ? width - kFastBits : 0u;
      st->shift_b = width > 2u * kFastBits ? width - 2u * kFastBits : 0u;
      // many samples in lo's 22-bit bucket (zeros of a ReLU output, a value of a quantisation
      // grid): count the values == lo instead of storing them.  Also when lo == hi.
      st->tie_lo = (span == 0u) || lo_tie;
      st->mid = key_to_float(lo_key + (span >> 1) + (span & 1u));  // > lo whenever lo < hi
    }
  }
  cluster.sync();  // the other CTAs' shared memory must outlive CTA 0's reads
  QSB_TICK(st, 5);
#ifdef QSB_SELECT_TIMING
  if (tid == 0 && rank == 0) reinterpret_cast<long long *>(st)[16] = t_start;
#endif
}

// ---------------------------------------------------------------------------
// fast route, step 2: ONE streaming pass.  Plain float compares against the pivots
// (NaNs compare false and so count as "above hi"); every CTA owns a tile of
// 256 * 8 * U elements, appends its candidates to the dense array behind one cursor
// atomic, and adds its totals by fire-and-forget RED.
// ---------------------------------------------------------------------------
// 1.0f / 0.0f compare results (one FSET.BF each, no predicate round trip); NaN -> 0
__device__ __forceinline__ float setf_lt(float a, float b) {
  float m;
  asm("set.lt.f32.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
  return m;
}
__device__ __forceinline__ float setf_le(float a, float b) {
  float m;
  asm("set.le.f32.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
  return m;
}
__device__ __forceinline__ float setf_eq(float a, float b) {
  float m;
  asm("set.eq.f32.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
  return m;
}

// Classify the 8 elements of one vector against the pivots: a base-4 digit per element,
// 3 = below lo, 2 = equal to lo (TIE only), 1 = candidate (lo <= a <= hi), 0 = above hi or
// NaN, accumulated EXACTLY in one float (16 bits) by FSET.BF + FFMA — 4 instructions per
// element instead of 6 through predicates.  Returns the digits as an integer.
template <bool ABS, bool TIE>
__device__ __forceinline__ uint32_t classify8(const VecF<8> &x, float lo, float hi) {
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float a = ABS ? fabsf(x.v[j]) : x.v[j];
    const float w = (float)(1u << (2 * j));
    acc = __fmaf_rn(setf_lt(a, lo), 2.0f * w, acc);
    acc = __fmaf_rn(setf_le(a, hi), w, acc);
    if constexpr (TIE) acc = __fmaf_rn(setf_eq(a, lo), w, acc);
  }
  return (uint32_t)__float2int_rz(acc);
}

struct StepPtrs {  // fused prune step only
  const float *w;       // the tensor behind the magnitudes; the mask is applied to it
  float *mag;           // == v, writable
  float *y;
  uint8_t *mask;
  uint32_t *cand_idx;   // element index of every stored candidate (parallel to cand)
};

template <int U, bool ABS, bool STEP>
__device__ __forceinline__ void select_partition_body(const float *__restrict__ v, int64_t n,
                                                      const SelState *st, unsigned long long *segctr,
                                                      float *__restrict__ cand, uint32_t seg_cap,
                                                      StepPtrs sp, EmaC ec) {
  static_assert(!STEP || !ABS, "magnitudes are non-negative");
  constexpr int V = 8;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  // every thread parks its own elements here so that the (rare) candidates can be picked
  // by index: [u][half][tid] float4 — conflict-free 128-bit stores, read back by the owner only
  __shared__ float4 s_x[U * 2 * QSB_THREADS];
  __shared__ uint32_t s_nc, s_lt, s_eq;
  __shared__ long long s_gbase;
  const int tid = threadIdx.x, lane = tid & 31;
  const int64_t n_main = (n / V) * V;
  const int64_t t0 = (int64_t)blockIdx.x * kTile;
  const int64_t base = t0 + (int64_t)tid * V;
  VecF<V> x[U];
  VecF<V> wv[STEP ? U : 1];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t e = base + (int64_t)u * QSB_THREADS * V;
    if (e < n_main) {
      x[u] = ld_vec<V, Hint::KEEP>(v + e);
      if constexpr (STEP) wv[u] = ld_vec<V, Hint::KEEP>(sp.w + e);
    }
  }
  const bool tail_owner = (t0 <= n_main && n_main < t0 + kTile);
  float tail_val = 0.f, tail_w = 0.f;
  const bool has_tail = tail_owner && (n_main + tid < n);
  if (has_tail) {
    tail_val = v[n_main + tid];
    if constexpr (STEP) tail_w = sp.w[n_main + tid];
  }
  pdl_wait();     // the loads above are in flight; the pivots come from the sampler
  pdl_trigger();
  if constexpr (STEP) {
    // the magnitude EMA itself: x becomes the NEW magnitude, written back in place
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = base + (int64_t)u * QSB_THREADS * V;
      if (e < n_main) {
#pragma unroll
        for (int j = 0; j < V; ++j) x[u].v[j] = ema_full_step(x[u].v[j], wv[u].v[j], ec.t_f, ec.tp1, ec.rcp);
        st_vec<V, Hint::KEEP>(sp.mag + e, x[u]);
      }
    }
    if (has_tail) {
      tail_val = ema_full_step(tail_val, tail_w, ec.t_f, ec.tp1, ec.rcp);
      sp.mag[n_main + tid] = tail_val;
    }
  }
  const float2 piv = *reinterpret_cast<const float2 *>(st);
  const float lo = piv.x, hi = piv.y;
  const bool tie = st->tie_lo != 0;
  if (tid == 0) {
    s_nc = 0;
    s_lt = 0;
    s_eq = 0;
  }
  __syncthreads();
  // digits of vectors (2w, 2w + 1) in word w: bit0 of a digit = candidate-or-below, bit1 = ..
  constexpr int W = (U + 1) / 2;
  uint32_t dig[W];
#pragma unroll
  for (int w = 0; w < W; ++w) dig[w] = 0;
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const int64_t e = base + (int64_t)u * QSB_THREADS * V;
    if (e < n_main) {
      const uint32_t d = tie ? classify8<ABS, true>(x[u], lo, hi) : classify8<ABS, false>(x[u], lo, hi);
      dig[u >> 1] |= d << (16 * (u & 1));
    }
  }
  uint32_t lt = 0, eq = 0, nc = 0;
  uint32_t cbits[W];  // bit 2j (+16 for the odd vector) set: element j is a candidate
#pragma unroll
  for (int w = 0; w < W; ++w) {
    const uint32_t b0 = dig[w] & 0x55555555u, b1 = (dig[w] >> 1) & 0x55555555u;
    cbits[w] = b0 & ~b1;
    lt += __popc(b0 & b1);
    eq += __popc(b1 & ~b0);
    nc += __popc(cbits[w]);
  }
  bool tail_c = false;
  if (has_tail) {
    tail_val = ABS ? fabsf(tail_val) : tail_val;
    if (tail_val < lo) ++lt;
    else if (tie && tail_val == lo) ++eq;
    else if (tail_val <= hi) tail_c = true, ++nc;
  }
  if constexpr (STEP) {
    // provisional mask and output: keep what is >= mid.  Everything outside [lo, hi] is final;
    // the candidates on the wrong side of the true threshold are patched by the fix-up kernel.
    const float mid = st->mid;
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int64_t e = base + (int64_t)u * QSB_THREADS * V;
      if (e < n_main) {
        VecF<V> yv;
        VecB<V> mb;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const bool keep = x[u].v[j] >= mid;  // false for NaN, like importance >= threshold
          mb.b[j] = keep ? 1 : 0;
          yv.v[j] = __fmul_rn(wv[u].v[j], keep ? 1.0f : 0.0f);
        }
        st_vec<V, Hint::KEEP>(sp.y + e, yv);
        st_bytes<V>(sp.mask + e, mb);
      }
    }
    if (has_tail) {
      const bool keep = tail_val >= mid;
      sp.mask[n_main + tid] = keep ? 1 : 0;
      sp.y[n_main + tid] = __fmul_rn(tail_w, keep ? 1.0f : 0.0f);
    }
  }
  if (nc) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      s_x[(u * 2 + 0) * QSB_THREADS + tid] = make_float4(x[u].v[0], x[u].v[1], x[u].v[2], x[u].v[3]);
      s_x[(u * 2 + 1) * QSB_THREADS + tid] = make_float4(x[u].v[4], x[u].v[5], x[u].v[6], x[u].v[7]);
    }
  }
  uint32_t incl = nc;  // warp scan, then one shared-memory atomic per warp
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const uint32_t wlt = __reduce_add_sync(0xffffffffu, lt);
  const uint32_t weq = tie ? __reduce_add_sync(0xffffffffu, eq) : 0u;
  uint32_t wbase = 0;
  if (lane == 31) {
    if (incl) wbase = atomicAdd(&s_nc, incl);
    if (wlt) atomicAdd(&s_lt, wlt);
    if (weq) atomicAdd(&s_eq, weq);
  }
  wbase = __shfl_sync(0xffffffffu, wbase, 31);
  __syncthreads();
  const int seg = blockIdx.x % kSegs;
  if (tid == 0) {
    const uint32_t total = s_nc, tlt = s_lt, teq = s_eq;
    long long g = -1;
    if (teq) atomicAdd(segctr + seg * kSegStride + 1, (unsigned long long)teq);  // unused result: RED
    if (total | tlt) {
      // ONE atomic per CTA: candidates in the low word (the append cursor), "< lo" in the high
      const unsigned long long old = atomicAdd(
          segctr + seg * kSegStride, ((unsigned long long)tlt << 32) | (unsigned long long)total);
      const uint32_t at = (uint32_t)old;
      if (total && at <= seg_cap && total <= seg_cap - at) g = at;  // else: overflow, seen in
    }                                                               // the counter by the passes
    s_gbase = g;
  }
  __syncthreads();
  const long long g = s_gbase;
  if (nc == 0 || g < 0) return;  // nothing to store, or the segment is full
  float *out = cand + (size_t)seg * seg_cap + (uint32_t)g;
  uint32_t *out_idx = STEP ? sp.cand_idx + (size_t)seg * seg_cap + (uint32_t)g : nullptr;
  uint32_t pos = wbase + (incl - nc);
  const float *sx = reinterpret_cast<const float *>(s_x);
#pragma unroll
  for (int w = 0; w < W; ++w) {
    uint32_t m = cbits[w];
    while (m) {
      const int b = __ffs(m) - 1;  // vector u = 2w + b / 16, element j = (b % 16) / 2
      m &= m - 1;
      const int q = 4 * w + (b >> 3);  // float4 row of s_x: u * 2 + j / 4
      const float a = sx[((q * QSB_THREADS) + tid) * 4 + ((b >> 1) & 3)];
      if constexpr (STEP)  // where the candidate lives, for the fix-up of its mask / output
        out_idx[pos] = (uint32_t)(base + (int64_t)(2 * w + (b >> 4)) * QSB_THREADS * V + ((b & 15) >> 1));
      out[pos++] = (ABS ? fabsf(a) : a) + 0.0f;  // -0 -> +0
    }
  }
  if (tail_c) {
    if constexpr (STEP) out_idx[pos] = (uint32_t)(n_main + tid);
    out[pos] = tail_val + 0.0f;
  }
}

// fused prune step, after the threshold is known: patch the candidates whose provisional
// decision (>= mid) differs from the final one (>= thr) — a few 0.1 % of the elements.
__device__ __forceinline__ void step_fixup_body(const SelState *st, const unsigned long long *segctr,
                                                const float *__restrict__ cand,
                                                const uint32_t *__restrict__ cand_idx, uint32_t seg_cap,
                                                const float *__restrict__ thr_dev, StepPtrs sp) {
  pdl_wait();
  pdl_trigger();
  if (st->need_full) return;  // the gated full pass rebuilds everything instead
  const unsigned nctas = gridDim.x / kSegs * kSegs;
  if (blockIdx.x >= nctas) return;
  const float thr = *thr_dev, mid = st->mid;
  const int seg = blockIdx.x % kSegs, part = blockIdx.x / kSegs, parts = nctas / kSegs;
  const uint32_t nc = (uint32_t)__ldcg(segctr + seg * kSegStride);
  const float *cv = cand + (size_t)seg * seg_cap;
  const uint32_t *ci = cand_idx + (size_t)seg * seg_cap;
  auto patch = [&](float val, uint32_t i) {
    const bool prov = val >= mid, fin = val >= thr;
    if (prov != fin) {
      const uint32_t e = ci[i];
      sp.mask[e] = fin ? 1 : 0;
      sp.y[e] = __fmul_rn(sp.w[e], fin ? 1.0f : 0.0f);
    }
  };
  // four 128-bit loads of candidate values in flight per thread; positions are only read for a patch
  const uint32_t n4 = nc >> 2, step = (uint32_t)parts * QSB_THREADS;
  const float4 *c4 = reinterpret_cast<const float4 *>(cv);
  for (uint32_t i = (uint32_t)part * QSB_THREADS + threadIdx.x; i < n4; i += 4 * step) {
    float4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i + u * step < n4) q[u] = c4[i + u * step];
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (i + u * step < n4) {
        const uint32_t b = (i + u * step) << 2;
        patch(q[u].x, b);
        patch(q[u].y, b + 1);
        patch(q[u].z, b + 2);
        patch(q[u].w, b + 3);
      }
  }
  if (part == 0 && threadIdx.x < (nc & 3u)) patch(cv[(n4 << 2) + threadIdx.x], (n4 << 2) + threadIdx.x);
}

// fused prune step, the rare complete redo (generic route, or rank k inside a block of ties at
// lo): mask = magnitude >= thr, y = w * mask over the whole segment.  Always launched, gated
// on the device; `force`: the segment never had provisional outputs (too small for the fast route).
__device__ __forceinline__ void step_full_mask_body(const SelState *st, bool force, int64_t n,
                                                    const float *__restrict__ thr_dev, StepPtrs sp) {
  pdl_wait();
  pdl_trigger();
  if (!force && !st->need_full) return;
  const float thr = *thr_dev;
  constexpr int V = 8;
  const int64_t n_main = (n / V) * V;
  for (int64_t e = ((int64_t)blockIdx.x * QSB_THREADS + threadIdx.x) * V; e < n_main;
       e += (int64_t)gridDim.x * QSB_THREADS * V) {
    const VecF<V> m = ld_vec<V, Hint::KEEP>(sp.mag + e), wv = ld_vec<V, Hint::KEEP>(sp.w + e);
    VecF<V> yv;
    VecB<V> mb;
#pragma unroll
    for (int j = 0; j < V; ++j) {
      const bool keep = m.v[j] >= thr;
      mb.b[j] = keep ? 1 : 0;
      yv.v[j] = __fmul_rn(wv.v[j], keep ? 1.0f : 0.0f);
    }
    st_vec<V, Hint::KEEP>(sp.y + e, yv);
    st_bytes<V>(sp.mask + e, mb);
  }
  if (blockIdx.x == 0 && n_main + threadIdx.x < n) {
    const int64_t e = n_main + threadIdx.x;
    const bool keep = sp.mag[e] >= thr;
    sp.mask[e] = keep ? 1 : 0;
    sp.y[e] = __fmul_rn(sp.w[e], keep ? 1.0f : 0.0f);
  }
}

// ---------------------------------------------------------------------------
// several independent selects ("segments": the layers of a weight set) in the same launches:
// blockIdx.y picks the segment, every kernel reads its segment's arguments from a table in
// the kernel parameters.  One select is the table with one entry.
// ---------------------------------------------------------------------------
constexpr int64_t kHistBytes = (int64_t)(kBins0 + kBins1 + kBins2) * sizeof(unsigned long long);
constexpr int64_t kFastHistBytes = 3 * (int64_t)kFastBins * sizeof(uint32_t);
constexpr int64_t kSegCtrBytes = (int64_t)kSegs * kSegStride * sizeof(unsigned long long);
// per segment: [hist x3 | fast hist x3 | segment counters | SelState | pad] | candidate segments
constexpr int64_t kSelectHeaderBytes = kHistBytes + kFastHistBytes + kSegCtrBytes + 1024;
static_assert(kSelectHeaderBytes % 256 == 0, "headers of consecutive segments stay 256-byte aligned");
static_assert(sizeof(SelState) <= 128, "SelState must fit the header pad (timing slots follow it)");

struct SegDesc {
  const float *v;
  int64_t n, k;
  float *thr_out;
  unsigned char *hdr;  // kSelectHeaderBytes, 256-byte aligned
  float *cand;         // [kSegs][seg_cap]
  uint32_t seg_cap;
  int r_lo, r_hi;      // sample ranks of the pivots
  int fast;            // 0: generic passes only (small or unaligned input)
  // fused prune step only (v is then the magnitude tensor, updated in place)
  const float *w;
  float *y;
  uint8_t *mask;
  uint32_t *cand_idx;
  uint32_t *hint;      // caller's pivot hint of this segment (8 words, may be null)
};
constexpr int kMaxSegs = 32;  // 32 x 104 B of kernel parameters
struct SegTable {
  SegDesc d[kMaxSegs];
};

__host__ __device__ inline SelectWs ws_of(unsigned char *hdr) {
  SelectWs ws;
  ws.hist0 = reinterpret_cast<unsigned long long *>(hdr);
  ws.hist1 = ws.hist0 + kBins0;
  ws.hist2 = ws.hist1 + kBins1;
  return ws;
}
__host__ __device__ inline uint32_t *fh_of(unsigned char *hdr) {
  return reinterpret_cast<uint32_t *>(hdr + kHistBytes);
}
__host__ __device__ inline unsigned long long *segctr_of(unsigned char *hdr) {
  return reinterpret_cast<unsigned long long *>(hdr + kHistBytes + kFastHistBytes);
}
__host__ __device__ inline SelState *st_of(unsigned char *hdr) {
  return reinterpret_cast<SelState *>(hdr + kHistBytes + kFastHistBytes + kSegCtrBytes);
}

__device__ __forceinline__ StepPtrs step_ptrs(const SegDesc &d) {
  return StepPtrs{d.w, const_cast<float *>(d.v), d.y, d.mask, d.cand_idx};
}

template <int PER, bool STEP>
__global__ void __cluster_dims__(kSampleCtas, 1, 1) __launch_bounds__(kSampleThreads)
    select_sample_kernel(const __grid_constant__ SegTable tab, int take_abs, EmaC ec) {
  if constexpr (STEP) ec = ema_resolve(ec);
  const SegDesc &d = tab.d[blockIdx.y];
  uint4 *zb = reinterpret_cast<uint4 *>(d.hdr);
  constexpr int zv = (int)(kSelectHeaderBytes / 16);
  if (!d.fast) {  // generic passes only: this launch just zeroes the segment's header
    pdl_wait();   // ... which the previous select on this workspace may still be reading
    for (int j = blockIdx.x * kSampleThreads + threadIdx.x; j < zv; j += kSampleThreads * kSampleCtas)
      zb[j] = make_uint4(0, 0, 0, 0);
    return;
  }
  select_sample_body<PER, STEP>(d.v, d.n, take_abs, d.r_lo, d.r_hi, st_of(d.hdr), zb, zv, d.w, ec, d.hint);
}

template <int U, bool ABS>
__global__ void __launch_bounds__(QSB_THREADS, 5)
    select_partition_kernel(const __grid_constant__ SegTable tab) {
  const SegDesc &d = tab.d[blockIdx.y];
  if (!d.fast || (int64_t)blockIdx.x * (QSB_THREADS * 8 * U) >= d.n) return;
  select_partition_body<U, ABS, false>(d.v, d.n, st_of(d.hdr), segctr_of(d.hdr), d.cand, d.seg_cap,
                                       StepPtrs{}, EmaC{});
}

// fused prune step: EMA + partition + provisional mask / output in one streaming pass
__global__ void __launch_bounds__(QSB_THREADS, 4)
    step_partition_kernel(const __grid_constant__ SegTable tab, EmaC ec) {
  ec = ema_resolve(ec);
  constexpr int U = 2;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * 8 * U;
  const SegDesc &d = tab.d[blockIdx.y];
  const int64_t t0 = (int64_t)blockIdx.x * kTile;
  if (t0 >= d.n) return;
  if (d.fast) {
    select_partition_body<U, false, true>(d.v, d.n, st_of(d.hdr), segctr_of(d.hdr), d.cand, d.seg_cap,
                                          step_ptrs(d), ec);
    return;
  }
  // a segment too small for the sampled route: just the EMA (its mask comes from the full pass)
  pdl_wait();
  pdl_trigger();
  float *mag = const_cast<float *>(d.v);
  const int64_t end = t0 + kTile < d.n ? t0 + kTile : d.n;
  for (int64_t e = t0 + threadIdx.x; e < end; e += QSB_THREADS)
    mag[e] = ema_full_step(mag[e], d.w[e], ec.t_f, ec.tp1, ec.rcp);
}

__global__ void __launch_bounds__(QSB_THREADS)
    step_fixup_kernel(const __grid_constant__ SegTable tab) {
  const SegDesc &d = tab.d[blockIdx.y];
  if (!d.fast) return;
  step_fixup_body(st_of(d.hdr), segctr_of(d.hdr), d.cand, d.cand_idx, d.seg_cap, d.thr_out, step_ptrs(d));
}

__global__ void __launch_bounds__(QSB_THREADS)
    step_full_mask_kernel(const __grid_constant__ SegTable tab) {
  const SegDesc &d = tab.d[blockIdx.y];
  step_full_mask_body(st_of(d.hdr), !d.fast, d.n, d.thr_out, step_ptrs(d));
}

template <int PASS, int V, bool ABS>
__global__ void __launch_bounds__(QSB_THREADS)
    select_pass_kernel(const __grid_constant__ SegTable tab) {
  const SegDesc &d = tab.d[blockIdx.y];
  FastBufs fb{nullptr, nullptr, nullptr, nullptr, 0, nullptr};
  if (d.fast) fb = FastBufs{st_of(d.hdr), d.cand, segctr_of(d.hdr), fh_of(d.hdr), d.seg_cap, d.hint};
  select_pass_body<PASS, V, ABS>(d.v, d.n, d.k, ws_of(d.hdr), fb, st_of(d.hdr), d.thr_out, d.fast ? d.hint : nullptr);
}

static int g_select_fast = 1;  // tuning key 4 (test hook): 0 forces the three generic passes
constexpr int64_t kFastMinNBatched = 1 << 17;  // segments of a batch share the launches' fixed costs

void set_select_fast(int v) { g_select_fast = v; }

// slots per candidate segment: n/8 in total, a multiple of 8 per segment, < 2^32
static int64_t seg_slots(int64_t n) {
  int64_t c = ((n >> kCandShift) / kSegs) & ~(int64_t)7;
  return c > 0xfffffff8ll ? 0xfffffff8ll : c;
}
// workspace of one segment: header + candidates (reserved whenever the fast route could be taken)
static int64_t seg_workspace_bytes(int64_t n) {
  const int64_t cand = n >= kFastMinNBatched ? kSegs * seg_slots(n) * (int64_t)sizeof(float) : 0;
  return kSelectHeaderBytes + (cand + 255) / 256 * 256;
}

template <class K, class... A>
static int launch_seg(K kernel, dim3 grid, dim3 block, cudaStream_t stream, bool pdl, const SegTable &tab,
                      A... extra) {
  if (pdl) {  // the previous kernel of this select is the dependency
    QSB_CUDA_TRY(launch_pdl(kernel, grid, block, 0, stream, tab, extra...));
    return 0;
  }
  kernel<<<grid, block, 0, stream>>>(tab, extra...);
  QSB_LAUNCH_CHECK();
  return 0;
}

template <int PASS, int V, bool ABS>
static int launch_pass(const SegTable &tab, int L, int64_t max_n, bool any_fast, cudaStream_t stream,
                       bool pdl) {
  static int occ = 0;
  if (occ == 0) {
    int o = 0;
    QSB_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(
        &o, select_pass_kernel<PASS, V, ABS>, QSB_THREADS, 0));
    occ = o > 0 ? o : 1;
  }
  constexpr int U = (V == 8) ? 2 : 4;
  constexpr int64_t kTile = (int64_t)QSB_THREADS * V * U;
  int64_t grid = (int64_t)device_props().sm_count * occ / L;  // the chip is shared by the L segments
  const int64_t tiles = (max_n + kTile - 1) / kTile;
  if (grid > tiles) grid = tiles;
  if (any_fast && grid < kSegs) grid = kSegs;  // the candidate passes work in multiples of kSegs CTAs
  if (grid < 1) grid = 1;
  return launch_seg(select_pass_kernel<PASS, V, ABS>, dim3((unsigned)grid, (unsigned)L), dim3(QSB_THREADS),
                    stream, pdl, tab);
}

// descs[0..L): one launch sequence.  v8: every segment is 32-byte aligned (256-bit loads).
template <bool ABS, bool STEP = false>
static int run_group(SegDesc *descs, int L, bool v8, bool first_after_kernel, cudaStream_t stream, EmaC ec = EmaC{}) {
  SegTable tab;
  int64_t max_n = 0, max_fast_n = 0;
  for (int i = 0; i < L; ++i) {
    tab.d[i] = descs[i];
    if (descs[i].n > max_n) max_n = descs[i].n;
    if (descs[i].fast && descs[i].n > max_fast_n) max_fast_n = descs[i].n;
  }
  const bool any_fast = max_fast_n > 0;
  int rc;
  if (first_after_kernel) {
    // pivots for the fast segments; zeroes every segment's header (no memset node)
    const dim3 sg(kSampleCtas, (unsigned)L);
    // (PDL: the sampler starts with griddepcontrol.wait, so it is ordered after whatever precedes it
    // in the stream, but its launch latency overlaps that kernel's tail)
    const int abs_i = ABS ? 1 : 0;
    rc = launch_seg(select_sample_kernel<kSamplePer, STEP>, sg, dim3(kSampleThreads), stream, true, tab, abs_i, ec);
    if (rc) return rc;
  }
  if constexpr (STEP) {
    // EMA for every segment, partition + provisional outputs for the fast ones: one streaming pass
    const int64_t tile = (int64_t)QSB_THREADS * 8 * 2;
    const dim3 pg((unsigned)((max_n + tile - 1) / tile), (unsigned)L);
    if ((rc = launch_seg(step_partition_kernel, pg, dim3(QSB_THREADS), stream, true, tab, ec))) return rc;
  } else if (any_fast) {
    const int64_t tile = (int64_t)QSB_THREADS * 8 * kPartitionU;
    const dim3 pg((unsigned)((max_fast_n + tile - 1) / tile), (unsigned)L);
    if ((rc = launch_seg(select_partition_kernel<kPartitionU, ABS>, pg, dim3(QSB_THREADS), stream, true, tab)))
      return rc;
  }
  if (v8) {
    if ((rc = launch_pass<0, 8, ABS>(tab, L, max_n, any_fast, stream, first_after_kernel))) return rc;
    if ((rc = launch_pass<1, 8, ABS>(tab, L, max_n, any_fast, stream, true))) return rc;
    if ((rc = launch_pass<2, 8, ABS>(tab, L, max_n, any_fast, stream, true))) return rc;
    if constexpr (STEP) {
      // patch the few candidates on the wrong side of the threshold; redo whole segments only where
      // the sampled route was not taken (both decide on the device and mostly exit at once)
      if (any_fast) {
        int parts = 16 * device_props().sm_count / (kSegs * L);  // ~16 CTAs per SM over all segments
        if (parts < 1) parts = 1;
        if (parts > 16) parts = 16;
        if ((rc = launch_seg(step_fixup_kernel, dim3((unsigned)(kSegs * parts), (unsigned)L),
                             dim3(QSB_THREADS), stream, true, tab)))
          return rc;
      }
      int64_t fg = 4 * (int64_t)device_props().sm_count / L;
      const int64_t vt = (max_n + QSB_THREADS * 8 - 1) / (QSB_THREADS * 8);
      if (fg > vt) fg = vt;
      if (fg < 1) fg = 1;
      return launch_seg(step_full_mask_kernel, dim3((unsigned)fg, (unsigned)L), dim3(QSB_THREADS), stream,
                        true, tab);
    }
    return 0;
  }
  if ((rc = launch_pass<0, 1, ABS>(tab, L, max_n, any_fast, stream, first_after_kernel))) return rc;
  if ((rc = launch_pass<1, 1, ABS>(tab, L, max_n, any_fast, stream, true))) return rc;
  return launch_pass<2, 1, ABS>(tab, L, max_n, any_fast, stream, true);
}

// fill one descriptor; returns the bytes of workspace it uses
static int64_t make_desc(SegDesc &d, const float *v, int64_t n, int64_t k, float *thr_out,
                         unsigned char *hdr, bool batched, bool step = false) {
  d.v = v;
  d.n = n;
  d.k = k;
  d.thr_out = thr_out;
  d.hdr = hdr;
  d.cand = reinterpret_cast<float *>(hdr + kSelectHeaderBytes);
  d.seg_cap = (uint32_t)seg_slots(n);
  d.w = nullptr;
  d.y = nullptr;
  d.mask = nullptr;
  d.cand_idx = nullptr;
  d.hint = nullptr;
  d.fast = g_select_fast && aligned_to(v, 32) && n >= (batched ? kFastMinNBatched : kFastMinN);
  // sample ranks bracketing k: +-4.5 sigma of the binomial rank error, +3
  const double m = (double)(kSampleThreads * kSampleCtas * kSamplePer), p = (double)k / (double)n;
  // a miss of the pivots costs one full redo of the step's masks (~the price of the step), so the fused
  // step brackets tighter than a select whose miss costs three full passes
  const double sigmas = step ? 3.5 : 4.5;
  const double delta = sigmas * sqrt(m * p * (1.0 - p)) + 3.0;
  d.r_lo = (int)floor(p * m - delta);
  d.r_hi = (int)ceil(p * m + delta);
  return seg_workspace_bytes(n);
}

}  // namespace qsb

using namespace qsb;

extern "C" int64_t qsb_kth_workspace_bytes(int64_t n) { return 256 + seg_workspace_bytes(n); }

extern "C" int64_t qsb_kth_batched_workspace_bytes(const int64_t *n, int count) {
  int64_t total = 256;
  for (int i = 0; i < count; ++i) total += seg_workspace_bytes(n[i]);
  return total;
}

static int kth_value_batched_impl(const float *const *v, const int64_t *n, const int64_t *k, int count,
                                  int take_abs, float *thr_out_dev, uint32_t *hints_dev, void *workspace,
                                  int64_t workspace_bytes, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (count < 0 || !v || !n || !k || !thr_out_dev || !workspace) return QSB_E_BADARG;
  if (count == 0) return 0;
  for (int i = 0; i < count; ++i) {
    if (n[i] <= 0 || k[i] < 0 || k[i] >= n[i] || !v[i]) return QSB_E_BADARG;
    if (!aligned_to(v[i], 4)) return QSB_E_ALIGN;
  }
  if (workspace_bytes < qsb_kth_batched_workspace_bytes(n, count)) return QSB_E_WORKSPACE;
  unsigned char *hdr =
      reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(workspace) + 255) / 256 * 256);
  const bool batched = count > 1;
  SegDesc group[kMaxSegs];
  int L = 0;
  auto flush = [&](bool v8) -> int {
    if (L == 0) return 0;
    const int rc = take_abs ? run_group<true>(group, L, v8, true, stream)
                            : run_group<false>(group, L, v8, true, stream);
    L = 0;
    return rc;
  };
  int rc;
  // 32-byte aligned segments share launches (up to kMaxSegs per sequence) ...
  for (int i = 0; i < count; ++i) {
    SegDesc d;
    const int64_t used = make_desc(d, v[i], n[i], k[i], thr_out_dev + i, hdr, batched);
    hdr += used;
    if (!aligned_to(v[i], 32)) continue;
    d.hint = hints_dev ? hints_dev + 8 * (int64_t)i : nullptr;
    group[L++] = d;
    if (L == kMaxSegs && (rc = flush(true))) return rc;
  }
  if ((rc = flush(true))) return rc;
  // ... the others go one by one through the scalar-load kernels
  hdr = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(workspace) + 255) / 256 * 256);
  for (int i = 0; i < count; ++i) {
    SegDesc d;
    const int64_t used = make_desc(d, v[i], n[i], k[i], thr_out_dev + i, hdr, batched);
    hdr += used;
    if (aligned_to(v[i], 32)) continue;
    group[L++] = d;
    if ((rc = flush(false))) return rc;
  }
  return 0;
}

// ---------------------------------------------------------------------------
// fused unstructured prune step over a set of tensors
// ---------------------------------------------------------------------------
static int64_t step_seg_workspace_bytes(int64_t n) {
  const int64_t cand = n >= kFastMinNBatched ? kSegs * seg_slots(n) * (int64_t)sizeof(float) : 0;
  return kSelectHeaderBytes + 2 * ((cand + 255) / 256 * 256);  // values + element indices
}

extern "C" int64_t qsb_prune_step_workspace_bytes(const int64_t *n, int count) {
  int64_t total = 256;
  for (int i = 0; i < count; ++i) total += step_seg_workspace_bytes(n[i]);
  return total;
}

static int prune_step_batched_impl(float *const *magnitude, const float *const *x, float *const *y,
                                   uint8_t *const *mask_out, const int64_t *n, const int64_t *k, int count,
                                   int64_t t, float *thr_out_dev, uint32_t *hints_dev, void *workspace,
                                   int64_t workspace_bytes, void *stream_, const int64_t *t_dev = nullptr) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (count < 0 || (!t_dev && t < 0) || !magnitude || !x || !y || !mask_out || !n || !k || !thr_out_dev || !workspace)
    return QSB_E_BADARG;
  if (count == 0) return 0;
  for (int i = 0; i < count; ++i) {
    if (n[i] <= 0 || k[i] < 0 || k[i] >= n[i] || !magnitude[i] || !x[i] || !y[i] || !mask_out[i])
      return QSB_E_BADARG;
    // whole 256-bit vectors everywhere: anything else takes the separate kernels
    if (!aligned_to(magnitude[i], 32) || !aligned_to(x[i], 32) || !aligned_to(y[i], 32) ||
        !aligned_to(mask_out[i], 8))
      return QSB_E_UNSUPPORTED;
  }
  if (workspace_bytes < qsb_prune_step_workspace_bytes(n, count)) return QSB_E_WORKSPACE;
  const float tp1 = (float)(t + 1);
  volatile float rcp = 1.0f / tp1;  // IEEE round-to-nearest on the host, as in qsb_magnitude_ema_full
  const EmaC ec{(float)t, tp1, rcp, reinterpret_cast<const long long *>(t_dev), (long long)t};
  unsigned char *hdr =
      reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(workspace) + 255) / 256 * 256);
  SegDesc group[kMaxSegs];
  int L = 0, rc;
  for (int i = 0; i < count; ++i) {
    SegDesc d;
    make_desc(d, magnitude[i], n[i], k[i], thr_out_dev + i, hdr, true, true);
    const int64_t cand_bytes = (step_seg_workspace_bytes(n[i]) - kSelectHeaderBytes) / 2;
    d.cand_idx = reinterpret_cast<uint32_t *>(hdr + kSelectHeaderBytes + cand_bytes);
    d.w = x[i];
    d.y = y[i];
    d.mask = mask_out[i];
    d.hint = hints_dev ? hints_dev + 8 * (int64_t)i : nullptr;
    if (n[i] >= (1ll << 32)) d.fast = 0;  // candidate positions are 32-bit
    hdr += step_seg_workspace_bytes(n[i]);
    group[L++] = d;
    if (L == kMaxSegs || i == count - 1) {
      if ((rc = run_group<false, true>(group, L, true, true, stream, ec))) return rc;
      L = 0;
    }
  }
  return 0;
}

extern "C" int qsb_kth_value_batched(const float *const *v, const int64_t *n, const int64_t *k,
                                     int count, int take_abs, float *thr_out_dev, void *workspace,
                                     int64_t workspace_bytes, void *stream) {
  return kth_value_batched_impl(v, n, k, count, take_abs, thr_out_dev, nullptr, workspace, workspace_bytes,
                                stream);
}

// the same with pivot hints: hints_dev = count x 8 uint32 words owned by the caller, zero before the
// first call and then left alone between calls on the same tensors (see "Pivot hints" at the top)
extern "C" int qsb_kth_value_batched_hinted(const float *const *v, const int64_t *n, const int64_t *k,
                                            int count, int take_abs, float *thr_out_dev,
                                            uint32_t *hints_dev, void *workspace,
                                            int64_t workspace_bytes, void *stream) {
  if (hints_dev && !aligned_to(hints_dev, 4)) return QSB_E_ALIGN;
  return kth_value_batched_impl(v, n, k, count, take_abs, thr_out_dev, hints_dev, workspace, workspace_bytes,
                                stream);
}

extern "C" int qsb_kth_value(const float *v, int64_t n, int64_t k, int take_abs,
                             float *thr_out_dev, void *workspace,
                             int64_t workspace_bytes, void *stream) {
  if (n <= 0 || k < 0 || k >= n) return QSB_E_BADARG;
  if (!v || !thr_out_dev || !workspace) return QSB_E_BADARG;
  return qsb_kth_value_batched(&v, &n, &k, 1, take_abs, thr_out_dev, workspace, workspace_bytes, stream);
}

extern "C" int qsb_prune_unstructured_step_batched(float *const *magnitude, const float *const *x,
                                                   float *const *y, uint8_t *const *mask_out,
                                                   const int64_t *n, const int64_t *k, int count,
                                                   int64_t t, float *thr_out_dev, void *workspace,
                                                   int64_t workspace_bytes, void *stream) {
  return prune_step_batched_impl(magnitude, x, y, mask_out, n, k, count, t, thr_out_dev, nullptr, workspace,
                                 workspace_bytes, stream);
}

// the same with pivot hints (count x 8 uint32 words, zero before the first step of these layers): from the
// third step on the sampler is skipped and the candidate set shrinks from ~2 % of a layer to a few thousand
extern "C" int qsb_prune_unstructured_step_batched_hinted(
    float *const *magnitude, const float *const *x, float *const *y, uint8_t *const *mask_out,
    const int64_t *n, const int64_t *k, int count, int64_t t, float *thr_out_dev, uint32_t *hints_dev,
    void *workspace, int64_t workspace_bytes, void *stream) {
  if (hints_dev && !aligned_to(hints_dev, 4)) return QSB_E_ALIGN;
  return prune_step_batched_impl(magnitude, x, y, mask_out, n, k, count, t, thr_out_dev, hints_dev, workspace,
                                 workspace_bytes, stream);
}

// CUDA-graph form: the EMA index is *t_dev + t_offset, read by the kernels (hints_dev may be NULL)
extern "C" int qsb_prune_unstructured_step_batched_at(
    float *const *magnitude, const float *const *x, float *const *y, uint8_t *const *mask_out,
    const int64_t *n, const int64_t *k, int count, const int64_t *t_dev, int64_t t_offset, float *thr_out_dev,
    uint32_t *hints_dev, void *workspace, int64_t workspace_bytes, void *stream) {
  if (!t_dev) return QSB_E_BADARG;
  if (hints_dev && !aligned_to(hints_dev, 4)) return QSB_E_ALIGN;
  return prune_step_batched_impl(magnitude, x, y, mask_out, n, k, count, t_offset, thr_out_dev, hints_dev,
                                 workspace, workspace_bytes, stream, t_dev);
}

// ---------------------------------------------------------------------------
// sharded select: the values live on several GPUs (each holds n_local of them); the rank k is
// global.  Per pass every GPU histograms its shard with the prefix derived from the
// (already summed) earlier histograms, the caller sums the new histogram over the GPUs
// (an all-reduce of <= 32 KB of 64-bit counters: exact), and after the third pass
// qsb_kth_dist_final reads the answer — identical on every GPU.  SURVEY 8(e), weights.
// ---------------------------------------------------------------------------
static unsigned char *dist_hdr(void *workspace) {
  return reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(workspace) + 255) / 256 * 256);
}
static SelectWs dist_ws(void *workspace) { return ws_of(dist_hdr(workspace)); }

extern "C" int qsb_kth_dist_begin(void *workspace, int64_t workspace_bytes, void *stream) {
  if (!workspace || workspace_bytes < qsb_kth_workspace_bytes(0)) return QSB_E_WORKSPACE;
  QSB_CUDA_TRY(cudaMemsetAsync(dist_ws(workspace).hist0, 0, kSelectHeaderBytes, (cudaStream_t)stream));
  return 0;
}

extern "C" int qsb_kth_dist_pass(const float *v, int64_t n_local, int64_t k_global, int pass,
                                 int take_abs, void *workspace, int64_t workspace_bytes,
                                 void **hist_out, int64_t *hist_counters_out, void *stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (n_local < 0 || k_global < 0 || pass < 0 || pass > 2) return QSB_E_BADARG;
  if (!workspace || workspace_bytes < qsb_kth_workspace_bytes(0)) return QSB_E_WORKSPACE;
  if (n_local > 0 && (!v || !aligned_to(v, 4))) return QSB_E_ALIGN;
  const SelectWs ws = dist_ws(workspace);
  unsigned long long *h = pass == 0 ? ws.hist0 : pass == 1 ? ws.hist1 : ws.hist2;
  if (hist_out) *hist_out = h;
  if (hist_counters_out) *hist_counters_out = pass == 0 ? kBins0 : kBins1;
  if (n_local == 0) return 0;  // an empty shard still takes part in the all-reduce
  SegDesc d;
  make_desc(d, v, n_local, k_global, nullptr, dist_hdr(workspace), false);
  d.fast = 0;  // histograms only; the answer is read by qsb_kth_dist_final after the last all-reduce
  SegTable tab;
  tab.d[0] = d;
  const bool v8 = aligned_to(v, 32);
#define QSB_DIST_PASS(P)                                                                        \
  (v8 ? (take_abs ? launch_pass<P, 8, true>(tab, 1, n_local, false, stream, false)               \
                  : launch_pass<P, 8, false>(tab, 1, n_local, false, stream, false))             \
      : (take_abs ? launch_pass<P, 1, true>(tab, 1, n_local, false, stream, false)               \
                  : launch_pass<P, 1, false>(tab, 1, n_local, false, stream, false)))
  if (pass == 0) return QSB_DIST_PASS(0);
  if (pass == 1) return QSB_DIST_PASS(1);
  return QSB_DIST_PASS(2);
#undef QSB_DIST_PASS
}

extern "C" int qsb_kth_dist_final(int64_t k_global, void *workspace, float *thr_out_dev,
                                  void *stream) {
  if (!workspace || !thr_out_dev || k_global < 0) return QSB_E_BADARG;
  select_final_kernel<<<1, QSB_THREADS, 0, (cudaStream_t)stream>>>(dist_ws(workspace), k_global,
                                                                   thr_out_dev);
  QSB_LAUNCH_CHECK();
  return 0;
}
