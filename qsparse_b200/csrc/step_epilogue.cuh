// The parameter step of the fused structured prune -> pow2 quantize training step, as a
// device function that ONE CTA runs:
//
//   local statistics  (finalize the stage-1 partials of this GPU, or sum finalized rows)
//   -> exchange with the peer GPUs over NVLink (low-latency packets, no fence, no NCCL launch)
//   -> combine in rank order (SUM of fp64 sums, MAX of maxima: bit-identical on every rank)
//   -> magnitude EMA (sparse.py:89) -> threshold = sorted(mag)[k] (util.py:113-116)
//   -> mask (util.py:117) -> abs-max of the kept channels (quantize.py:329-340)
//   -> scale EMA (quantize.py:344-348) -> decimal (quantize.py:316)
//
// Two callers:
//   * reduce.cu: the LAST-ARRIVING CTA of the stage-1 reduction runs it as the kernel's tail
//     (qsb_reduce_prune_quant_step: the step has no single-CTA launch and the peer latency
//     overlaps the tail of the reduction),
//   * params.cu: prune_quant_step_kernel, a stand-alone one-CTA launch (partials or rows).
//
// Peer exchange ("LL" packets).  A rank's statistics row is 3 * C 32-bit words (low / high
// half of the fp64 sum, bits of max|x|).  Every word travels as ONE 8-byte packet
// {data, flag} written with a single 64-bit store straight into the peer's buffer
// (slot [parity][sender rank]); flag = the step stamp with bit 31 set.  An 8-byte aligned
// store is delivered as a unit, so the receiver just polls each packet until its flag is
// the current stamp — data and "ready" arrive together: no fence, no separate flag, one
// one-way NVLink latency.  Slots alternate with the parity of the stamp; a rank cannot run
// two steps ahead of a peer (it needs the peer's packets of the step in between), so two
// slots are enough.
#pragma once
#include <math.h>

#include "p2p_internal.cuh"
#include "param_math.cuh"
#include "qsb_common.cuh"
#include "reduce_internal.cuh"

namespace qsb {

// Both forms carve step_smem_bytes(channels) of dynamic shared memory (20 B / channel; the line form 28).
constexpr int kStepMaxChannels = 4096;      // stand-alone kernel: ~82 KB, opted in above the 48 KB default
constexpr int kStepFusedMaxChannels = 1024; // fused tail: shares the CTA with the reduction
constexpr int kLineStepMaxChannels = 2048;  // line form, stand-alone kernel (partials route)

struct StepArgs {
  float *magnitude;
  uint8_t *mask;
  float *scale;
  float *decimal_out;
  // local statistics, one of:
  Partials P;  // stage-1 partials, entry j of channel c at (j / fin_q) * (channels * fin_q) + c * fin_q + j % fin_q
  int fin_count, fin_q;
  const double *row_sum;  // or n_rows > 0 finalized rows (chunks of a host tensor), row_stride bytes apart;
  const float *row_max;   // either may be NULL when the step does not use it (no magnitude / scale update)
  int n_rows;
  int64_t row_stride;
  int channels;
  int group;  // threads per channel in the finalize / rank count (power of two)
  P2PDev px;
  unsigned long long stamp;
  double count;
  int64_t t_prune;
  int update_magnitude;
  int refresh_mask;
  int64_t k;
  float limit;
  int64_t t_quant;
  int update_scale;
  double *abssum_out;  // optional: the statistics (combined over ranks, or this rank's own
  float *absmax_out;   // row when stats_local != 0)
  int stats_local;
  long long *step_counter;  // optional device step index (CUDA graphs)
  unsigned long long *timing;  // optional: %globaltimer stamps of the phases (development / bench evidence)
  // line form (step_epilogue<true>, AdaptiveQuantizer): in place of abs-max -> scale -> decimal, the (min, max)
  // of x * mask -> lines EMA.  The statistics are sum|x| and min / max x (row_max then holds max x, not max|x|).
  float *lines;           // [n_lines, 2], n_lines == 1 (per tensor) or channels
  int n_lines;
  int64_t t_line;         // the quantizer's 1-based call index (an offset to *step_counter when that is given)
  const float *row_min;
  float *min_out, *max_out;  // optional, like abssum_out: this step's min / max x per channel
};

struct StepSmem {
  double *sum;    // [channels]
  uint32_t *max;  // [channels]
  float *imp;     // [channels]
  uint32_t *key;  // [channels]
  double *psum;   // [32]
  uint32_t *pmax; // [32]
  uint32_t *amax; // [32]
  float *thr;     // [1]
  int *flag;      // [1]
  float *mn, *mx; // [channels] each, line form only (min / max x, NaN when the channel holds a NaN)
};

__host__ __device__ inline size_t step_smem_bytes(int channels, bool lines = false) {
  return (size_t)channels * 20 + 32 * 8 + 32 * 4 + 32 * 4 + 16 + (lines ? (size_t)channels * 8 : 0);
}
__device__ __forceinline__ StepSmem carve_step_smem(unsigned char *base, int channels) {
  StepSmem s;
  s.sum = reinterpret_cast<double *>(base);
  s.psum = s.sum + channels;
  s.max = reinterpret_cast<uint32_t *>(s.psum + 32);
  s.imp = reinterpret_cast<float *>(s.max + channels);
  s.key = reinterpret_cast<uint32_t *>(s.imp + channels);
  s.pmax = s.key + channels;
  s.amax = s.pmax + 32;
  s.thr = reinterpret_cast<float *>(s.amax + 32);
  s.flag = reinterpret_cast<int *>(s.thr + 1);
  s.mn = reinterpret_cast<float *>(base + step_smem_bytes(channels));
  s.mx = s.mn + channels;
  return s;
}

__device__ __forceinline__ unsigned long long global_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void st_packet(void *p, uint32_t data, uint32_t flag) {
  asm volatile("st.volatile.global.v2.u32 [%0], {%1,%2};" ::"l"(p), "r"(data), "r"(flag) : "memory");
}
__device__ __forceinline__ uint2 ld_packet(const void *p) {
  uint2 v;
  asm volatile("ld.volatile.global.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float nan_poison() { return __uint_as_float(0x7fc00000u); }

// What a CTA may already hold when it enters the parameter step: the fused kernels load the layer's
// old state at KERNEL START (a few hundred bytes that the streaming traffic of the previous step has
// long evicted from L2, i.e. DRAM-latency loads), so that the tail does not wait for them.
struct StepPrefetch {
  bool valid;
  float mag_old;        // magnitude[tid / group] for the threads with tid % group == 0
  float scale_old;      // scale[0] (thread 0)
  long long t;          // *step_counter (every thread)
};

template <bool LINES = false>
__device__ __forceinline__ StepPrefetch step_prefetch(const StepArgs &a) {
  StepPrefetch p;
  const int tid = threadIdx.x, nthr = blockDim.x;
  p.valid = a.channels * a.group <= nthr;   // one finalize pass: thread (c * group) owns channel c
  p.mag_old = 0.0f;
  p.scale_old = 0.0f;
  p.t = 0;
  if (!p.valid) return p;
  const int c = tid / a.group;
  if (tid % a.group == 0 && c < a.channels && a.update_magnitude != 2) p.mag_old = a.magnitude[c];
  if (!LINES && tid == 0) p.scale_old = a.scale[0];
  if (a.step_counter) p.t = *a.step_counter;
  return p;
}

__device__ __forceinline__ void step_stamp_time(const StepArgs &a, int slot) {
  if (a.timing && threadIdx.x == 0) a.timing[slot] = global_ns();
}

// Runs on every thread of ONE CTA (blockDim.x a multiple of 32).  sm: shared memory of that CTA.
// LINES: the line form (StepArgs::lines); it takes no peer group.
template <bool LINES = false>
__device__ __forceinline__ void step_epilogue(const StepArgs &a, const StepSmem &sm,
                                              const StepPrefetch pre = StepPrefetch{false, 0.f, 0.f, 0}) {
  int64_t t_prune = a.t_prune, t_quant = a.t_quant;
  unsigned long long stamp = a.stamp;
  int refresh_mask = a.refresh_mask;
  long long t_counter = 0;
  if (a.step_counter) {
    // graph mode: the step index lives on the device (the launch arguments of a captured
    // CUDA graph are frozen).  `t_prune` / `t_quant` are then OFFSETS added to the counter (a prune
    // callback and a quantizer started at different steps keep a constant distance) and
    // `refresh_mask` carries the refresh interval.
    t_counter = pre.valid ? pre.t : *a.step_counter;
    t_prune = t_counter + a.t_prune;
    t_quant = t_counter + a.t_quant;
    stamp = (unsigned long long)(t_counter + 1);
    const int interval = refresh_mask > 0 ? refresh_mask : 1;
    refresh_mask = (t_prune % interval == 0) && (t_prune > 0 || a.update_magnitude == 2);
  }
  const int channels = a.channels, group = a.group;
  const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
  const int gl = tid % group, gc = tid / group, cpp = nthr / group;
  const float scale_old = LINES ? 0.0f : pre.valid ? pre.scale_old : ((tid == 0) ? a.scale[0] : 0.0f);  // prefetch
  if (tid == 0) *sm.flag = 0;
  step_stamp_time(a, 1);

  // ---- 1. this GPU's statistics, fixed order ------------------------------------------
  if (a.n_rows) {
    for (int c = tid; c < channels; c += nthr) {
      double sum = 0.0;
      uint32_t mx = 0;
      float cmin = INFINITY, cmax = -INFINITY;  // line form: min / max x
      bool nan = false;
      for (int r = 0; r < a.n_rows; ++r) {
        if (a.row_sum)
          sum += *reinterpret_cast<const double *>(reinterpret_cast<const char *>(a.row_sum + c) +
                                                   (int64_t)r * a.row_stride);
        if constexpr (LINES) {
          const int64_t off = (int64_t)r * a.row_stride;
          const float l = *reinterpret_cast<const float *>(reinterpret_cast<const char *>(a.row_min + c) + off);
          const float h = *reinterpret_cast<const float *>(reinterpret_cast<const char *>(a.row_max + c) + off);
          nan = nan || l != l || h != h;
          cmin = fminf(cmin, l);
          cmax = fmaxf(cmax, h);
        } else if (a.row_max) {
          const float v = *reinterpret_cast<const float *>(reinterpret_cast<const char *>(a.row_max + c) +
                                                           (int64_t)r * a.row_stride);
          const uint32_t b = __float_as_uint(v) & 0x7fffffffu;
          mx = b > mx ? b : mx;
        }
      }
      sm.sum[c] = sum;
      if constexpr (LINES) {
        sm.mn[c] = nan ? nan_poison() : cmin;
        sm.mx[c] = nan ? nan_poison() : cmax;
      } else {
        sm.max[c] = mx;
      }
      sm.imp[c] = (a.update_magnitude != 2) ? a.magnitude[c] : 0.0f;
    }
  } else {
    // `group` threads share a channel, so the few thousand partials are fetched with
    // independent loads by the whole CTA (strided per thread, xor tree across the group).
    // __ldcg: in the fused kernel the partials were written by other SMs of this grid.
    for (int base = 0; base < channels; base += cpp) {
      const int c = base + gc;
      const bool act = c < channels;
      float mag_old = pre.mag_old;
      if (!pre.valid && act && gl == 0 && a.update_magnitude != 2) mag_old = a.magnitude[c];  // prefetch
      double sum = 0.0;
      uint32_t mx = 0;
      float cmin = INFINITY, cmax = -INFINITY;  // line form: min / max x, NaN-propagating through `nan`
      bool nan = false;
      if (act) {
        // kFinBatch independent loads per thread in flight (L2 hits): the C2 plan has 9 entries per
        // thread, i.e. ONE round trip; the additions run in ascending j whatever the batch size
        constexpr int kFinBatch = 12;
        for (int j0 = gl; j0 < a.fin_count; j0 += kFinBatch * group) {
          double v[kFinBatch];
          uint32_t b[kFinBatch];
          float l[kFinBatch], h[kFinBatch];
#pragma unroll
          for (int u = 0; u < kFinBatch; ++u) {
            const int j = j0 + u * group;
            const bool ok = j < a.fin_count;
            const int hi = ok ? j / a.fin_q : 0;
            const int64_t idx =
                (int64_t)hi * ((int64_t)channels * a.fin_q) + (int64_t)c * a.fin_q + (ok ? j - hi * a.fin_q : 0);
            v[u] = ok ? __ldcg(a.P.asum + idx) : 0.0;
            if constexpr (LINES) {
              l[u] = ok ? __ldcg(a.P.mn + idx) : INFINITY;
              h[u] = ok ? __ldcg(a.P.mx + idx) : -INFINITY;
            } else {
              b[u] = ok ? __ldcg(a.P.amax + idx) : 0u;
            }
          }
#pragma unroll
          for (int u = 0; u < kFinBatch; ++u) {
            sum += v[u];
            if constexpr (LINES) {
              nan = nan || l[u] != l[u] || h[u] != h[u];
              cmin = fminf(cmin, l[u]);
              cmax = fmaxf(cmax, h[u]);
            } else {
              mx = b[u] > mx ? b[u] : mx;
            }
          }
        }
      }
      for (int o = (group < 32 ? group : 32) >> 1; o > 0; o >>= 1) {
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        if constexpr (LINES) {
          nan = __shfl_xor_sync(0xffffffffu, (int)nan, o) || nan;
          cmin = fminf(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
          cmax = fmaxf(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
        } else {
          const uint32_t other = __shfl_xor_sync(0xffffffffu, mx, o);
          mx = other > mx ? other : mx;
        }
      }
      if constexpr (LINES) {
        if (nan) cmin = cmax = nan_poison();
      }
      if (group > 32) {
        // one channel, the whole CTA (per-tensor statistics): combine the warps of the group
        // through shared memory, in warp order (line form: min / max bits in pmax / amax)
        if (lane == 0) {
          sm.psum[warp] = sum;
          if constexpr (LINES) {
            sm.pmax[warp] = __float_as_uint(cmin);
            sm.amax[warp] = __float_as_uint(cmax);
          } else {
            sm.pmax[warp] = mx;
          }
        }
        __syncthreads();
        if (gl == 0)
          for (int w = 1; w < group / 32; ++w) {
            sum += sm.psum[warp + w];
            if constexpr (LINES) {
              const float l = __uint_as_float(sm.pmax[warp + w]), h = __uint_as_float(sm.amax[warp + w]);
              nan = nan || l != l || h != h;
              cmin = fminf(cmin, l);
              cmax = fmaxf(cmax, h);
            } else {
              mx = sm.pmax[warp + w] > mx ? sm.pmax[warp + w] : mx;
            }
          }
        if constexpr (LINES) {
          if (nan) cmin = cmax = nan_poison();
        }
        __syncthreads();
      }
      if (act && gl == 0) {
        sm.sum[c] = sum;
        if constexpr (LINES) {
          sm.mn[c] = cmin;
          sm.mx[c] = cmax;
        } else {
          sm.max[c] = mx;
        }
        sm.imp[c] = mag_old;
      }
    }
  }
  __syncthreads();
  step_stamp_time(a, 2);
  if constexpr (LINES) {
    for (int c = tid; c < channels; c += nthr) {
      if (a.abssum_out) a.abssum_out[c] = sm.sum[c];
      if (a.min_out) a.min_out[c] = sm.mn[c];
      if (a.max_out) a.max_out[c] = sm.mx[c];
    }
  } else if (a.abssum_out && a.stats_local) {
    for (int c = tid; c < channels; c += nthr) {
      a.abssum_out[c] = sm.sum[c];
      a.absmax_out[c] = __uint_as_float(sm.max[c]);
    }
  }

  // ---- 2. exchange with the peers (weak scaling over the batch) -------------------------
  if (!LINES && a.px.world > 1) {
    const P2PDev &px = a.px;
    const int parity = (int)(stamp & 1ull);
    const uint32_t flag = (uint32_t)(stamp & 0x7fffffffull) | 0x80000000u;
    const int npk = 3 * channels;
    // push my row into slot [parity][rank] of every PEER's buffer
    for (int i = tid; i < npk * px.world; i += nthr) {
      const int r = i / npk, j = i - r * npk;
      if (r == px.rank) continue;
      uint32_t data;
      if (j < channels) data = (uint32_t)__double2loint(sm.sum[j]);
      else if (j < 2 * channels) data = (uint32_t)__double2hiint(sm.sum[j - channels]);
      else data = sm.max[j - 2 * channels];
      st_packet(px.bufs[r] + p2p_slot_offset(px, parity, px.rank) + (int64_t)j * 8, data, flag);
    }
    // Receive + combine, one thread per channel.  A thread polls the three packets of its channel from up
    // to kRankBatch peers AT ONCE (all loads in flight: one L2 round trip per poll, where a packet-by-packet
    // loop paid one per packet — 3.2 us at 8 GPUs even with everything already there), and adds the rows in
    // rank order (SUM of sums, MAX of maxima: identical on every rank) as the batches complete.
    // Bounded: a peer that never shows up must not hang the GPU — the step is then poisoned, see below.
    constexpr int kRankBatch = 8;
    bool late = false;
    const unsigned long long t0 = global_ns();
    const unsigned char *mine = px.bufs[px.rank];
    for (int c = tid; c < channels && !late; c += nthr) {
      double sum = 0.0;
      uint32_t mx = 0;
      for (int r0 = 0; r0 < px.world && !late; r0 += kRankBatch) {
        uint2 pk[kRankBatch][3];
        unsigned spins = 0;
        while (true) {
          bool ok = true;
#pragma unroll
          for (int u = 0; u < kRankBatch; ++u) {
            const int r = r0 + u;
            if (r < px.world && r != px.rank) {
              const unsigned char *slot = mine + p2p_slot_offset(px, parity, r);
              pk[u][0] = ld_packet(slot + (int64_t)c * 8);
              pk[u][1] = ld_packet(slot + (int64_t)(channels + c) * 8);
              pk[u][2] = ld_packet(slot + (int64_t)(2 * channels + c) * 8);
            }
          }
#pragma unroll
          for (int u = 0; u < kRankBatch; ++u) {
            const int r = r0 + u;
            if (r < px.world && r != px.rank)
              ok = ok && pk[u][0].y == flag && pk[u][1].y == flag && pk[u][2].y == flag;
          }
          if (ok) break;
          if ((++spins & 63u) == 0) {
            if (global_ns() - t0 > px.timeout_ns) {
              late = true;
              break;
            }
            __nanosleep(64);
          }
        }
        if (late) break;
#pragma unroll
        for (int u = 0; u < kRankBatch; ++u) {
          const int r = r0 + u;
          if (r < px.world) {
            double s_;
            uint32_t b_;
            if (r == px.rank) {
              s_ = sm.sum[c];
              b_ = sm.max[c];
            } else {
              s_ = __hiloint2double((int)pk[u][1].x, (int)pk[u][0].x);
              b_ = pk[u][2].x;
            }
            sum += s_;
            mx = b_ > mx ? b_ : mx;
          }
        }
      }
      if (!late) {  // each thread only rewrites the channels it read: no barrier needed in between
        sm.sum[c] = sum;
        sm.max[c] = mx;
      }
    }
    if (late) *sm.flag = 1;
    __syncthreads();
    if (*sm.flag) {
      // Do NOT continue with whatever is in the slots (a peer's row from two steps ago):
      // poison the parameters so every later output is NaN, and raise the group's error flag.
      for (int c = tid; c < channels; c += nthr)
        if (a.update_magnitude == 1) a.magnitude[c] = nan_poison();
      if (tid == 0) {
        *px.error = 1;
        a.scale[0] = nan_poison();
        if (a.decimal_out) a.decimal_out[0] = nan_poison();
        if (a.step_counter) *a.step_counter = t_counter + 1;
      }
      return;
    }
  }

  // ---- 3. importance (magnitude EMA) -----------------------------------------------------
  step_stamp_time(a, 3);
  for (int c = tid; c < channels; c += nthr) {
    if (!LINES && a.abssum_out && !a.stats_local) {
      a.abssum_out[c] = sm.sum[c];
      a.absmax_out[c] = __uint_as_float(sm.max[c]);
    }
    const float m = (float)(sm.sum[c] / a.count);
    float imp;
    if (a.update_magnitude == 2) {
      imp = m;
    } else {
      imp = sm.imp[c];  // the prefetched old magnitude
      if (a.update_magnitude == 1) {
        imp = magnitude_ema_step(imp, m, t_prune);
        a.magnitude[c] = imp;
      }
    }
    sm.imp[c] = imp;
    sm.key[c] = float_to_key(imp);
  }
  __syncthreads();

  // ---- 4. threshold = sorted(importance)[k] by rank counting, `group` threads per channel ----
  step_stamp_time(a, 4);
  if (refresh_mask) {
    for (int base = 0; base < channels; base += cpp) {
      const int c = base + gc;
      const bool act = c < channels;
      const uint32_t kc = act ? sm.key[c] : 0u;
      int cnt = 0;
      if (act)
        for (int j = gl; j < channels; j += group) {
          const uint32_t kj = sm.key[j];
          cnt += (kj < kc) || (kj == kc && j < c);
        }
      for (int o = (group < 32 ? group : 32) >> 1; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
      if (group > 32) {  // channels == 1: rank 0 by definition
        cnt = 0;
      }
      if (act && gl == 0 && cnt == a.k) *sm.thr = sm.imp[c];
    }
    __syncthreads();
  }

  // ---- 5. mask, abs-max of the kept channels, scale EMA, decimal ---------------------------
  step_stamp_time(a, 5);
  const float thr = refresh_mask ? *sm.thr : 0.0f;
  if constexpr (LINES) {
    // line form: (min, max) of x * mask per channel or over the tensor (quantize.py:396-418) -> lines EMA
    // (quantize.py:428-430) at the quantizer's call index
    const int64_t tl = a.step_counter ? t_counter + a.t_line : a.t_line;
    const float tm1 = (float)(tl - 1), tf = (float)tl;
    float lo = INFINITY, hi = -INFINITY;
    bool nan = false;
    for (int c = tid; c < channels; c += nthr) {
      bool keep;
      if (refresh_mask) {
        keep = sm.imp[c] >= thr;
        a.mask[c] = keep ? 1 : 0;
      } else {
        keep = a.mask[c] != 0;
      }
      float l, h;
      masked_line(keep, sm.mn[c], sm.mx[c], l, h);
      if (a.n_lines == 1) {
        nan = nan || l != l;
        lo = fminf(lo, l);
        hi = fmaxf(hi, h);
      } else {
        a.lines[2 * c] = lines_ema_step(a.lines[2 * c], l, tm1, tf);
        a.lines[2 * c + 1] = lines_ema_step(a.lines[2 * c + 1], h, tm1, tf);
      }
    }
    if (a.n_lines == 1) {
      lo = warp_reduce(lo, [](float x, float y) { return fminf(x, y); });
      hi = warp_reduce(hi, [](float x, float y) { return fmaxf(x, y); });
      if (lane == 0) {
        sm.pmax[warp] = __float_as_uint(lo);
        sm.amax[warp] = __float_as_uint(hi);
      }
      if (nan) *sm.flag = 1;
      __syncthreads();
      if (tid == 0) {
        for (int w = 1; w < (nthr >> 5); ++w) {
          lo = fminf(lo, __uint_as_float(sm.pmax[w]));
          hi = fmaxf(hi, __uint_as_float(sm.amax[w]));
        }
        if (*sm.flag) lo = hi = nan_poison();
        a.lines[0] = lines_ema_step(a.lines[0], lo, tm1, tf);
        a.lines[1] = lines_ema_step(a.lines[1], hi, tm1, tf);
      }
    }
    if (tid == 0) {
      if (a.step_counter) *a.step_counter = t_counter + 1;
      if (a.timing) a.timing[6] = global_ns();
    }
    return;
  }
  uint32_t am = 0;
  for (int c = tid; c < channels; c += nthr) {
    bool keep;
    if (refresh_mask) {
      keep = sm.imp[c] >= thr;
      a.mask[c] = keep ? 1 : 0;
    } else {
      keep = a.mask[c] != 0;
    }
    if (a.update_scale) {
      const uint32_t b = keep ? sm.max[c] : pruned_max_bits(sm.max[c]);
      am = b > am ? b : am;
    }
  }
  am = warp_reduce(am, [](uint32_t x, uint32_t y) { return x > y ? x : y; });
  if (lane == 0) sm.amax[warp] = am;
  __syncthreads();
  if (tid == 0) {
    float s = scale_old;
    if (a.update_scale) {
      for (int w = 1; w < (nthr >> 5); ++w) am = sm.amax[w] > am ? sm.amax[w] : am;
      s = scale_ema_step(s, __uint_as_float(am), a.limit, t_quant);
      a.scale[0] = s;
    }
    if (a.decimal_out) a.decimal_out[0] = scale_to_decimal(s);
    if (a.step_counter) *a.step_counter = t_counter + 1;
    if (a.timing) a.timing[6] = global_ns();
  }
}

// shared argument checks + StepArgs assembly of the parameter-step entry points (params.cu)
int fill_step_args(StepArgs &a, float *magnitude, uint8_t *mask, float *scale, float *decimal_out,
                   int64_t channels, qsb_p2p_group *group, int64_t step_stamp, double count, int64_t t_prune,
                   int update_magnitude, int refresh_mask, int64_t k, int bits, int64_t t_quant,
                   int update_scale, double *abssum_out, float *absmax_out, int stats_local,
                   int64_t *step_counter_dev, int threads);
// the same for the line form (no scale, no group): lines [n_lines, 2], n_lines 1 or channels
int fill_line_step_args(StepArgs &a, float *magnitude, uint8_t *mask, float *lines, int64_t n_lines,
                        int64_t channels, qsb_p2p_group *group, double count, int64_t t_prune, int update_magnitude,
                        int refresh_mask, int64_t k, int64_t t_line, double *abssum_out, float *min_out,
                        float *max_out, int64_t *step_counter_dev);

// the stand-alone one-CTA launch of the parameter step on n_rows >= 1 finalized statistics rows (params.cu)
int launch_step_kernel_on_rows(StepArgs a, const double *row_sum, const float *row_max, int64_t n_rows,
                               int64_t row_stride, cudaStream_t stream);

// threads per channel for a CTA of `threads` threads: the largest power of two
// <= min(32, threads / channels); one channel: the whole CTA
inline int step_group_for(int64_t channels, int threads) {
  if (channels == 1) return threads;
  int tpc = 32;
  while (tpc > 1 && (int64_t)tpc * channels > threads) tpc >>= 1;
  return tpc;
}

}  // namespace qsb
