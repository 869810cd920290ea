// K4  tiny on-device parameter updates (scale / lines / magnitude EMAs, the
// scale -> decimal derivation, the fused structured prune->quantize parameter
// step) plus library plumbing (device properties, error strings).
//
// These kernels touch a few hundred bytes; what matters is that they run on
// the device, in stream order, so the training step never synchronises with
// the host (the reference does 6-8 `.item()` round trips per layer-step,
// SURVEY Q17).
#include <math.h>

#include <mutex>

#include "p2p_internal.cuh"
#include "param_math.cuh"
#include "qsb_common.cuh"
#include "reduce_internal.cuh"
#include "step_epilogue.cuh"

namespace qsb {

static int g_pdl_enabled = 1;  // tuning key 12 (default on: eager step 168.6 -> 165.1 us, = the CUDA-graph time)
bool pdl_enabled() { return g_pdl_enabled != 0; }
void set_pdl_enabled(int v) { g_pdl_enabled = v != 0; }

const DeviceProps &device_props() {
  static DeviceProps props[64];
  static bool init[64] = {false};
  static std::mutex mu;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  if (!init[dev]) {
    std::lock_guard<std::mutex> lock(mu);
    if (!init[dev]) {
      int sm = 148, l2 = 0;
      cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, dev);
      cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev);
      props[dev].sm_count = sm > 0 ? sm : 148;
      props[dev].l2_bytes = l2;
      init[dev] = true;
    }
  }
  return props[dev];
}

__global__ void scale_ema_kernel(float *w, const float *absmax, int64_t n,
                                 float limit, int64_t t, const long long *t_dev) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t_dev) t += (int64_t)__ldg(t_dev);
  if (i < n) w[i] = scale_ema_step(w[i], absmax[i], limit, t);
}

__global__ void scale_to_decimal_kernel(const float *s, float *d, int64_t n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) d[i] = scale_to_decimal(s[i]);
}

// lines = (w * (t - 1) + new) / t     ref qsparse/quantize.py:428-430
__global__ void lines_ema_kernel(float *lines, const float *mn, const float *mx,
                                 int64_t channels, float tm1, float t, const long long *t_dev,
                                 int64_t t_offset) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t_dev) {
    const int64_t ti = (int64_t)__ldg(t_dev) + t_offset;
    tm1 = (float)(ti - 1);
    t = (float)ti;
  }
  if (i < channels) {
    lines[2 * i] = lines_ema_step(lines[2 * i], mn[i], tm1, t);
    lines[2 * i + 1] = lines_ema_step(lines[2 * i + 1], mx[i], tm1, t);
  }
}

__global__ void magnitude_ema_reduced_kernel(float *mag, const double *abssum,
                                             const double *nnz,
                                             const float *tensor_min,
                                             int use_l0, int64_t channels,
                                             double count, int64_t t) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= channels) return;
  const bool indicator = use_l0 && (*tensor_min == 0.0f);
  const float m = (float)((indicator ? nnz[i] : abssum[i]) / count);
  mag[i] = magnitude_ema_step(mag[i], m, t);
}

// group-wise scale sharing (ref qsparse/quantize.py:361-366): every channel's parameter row is replaced
// by the mean of its group's rows.  One CTA; thread (g, col) sums the group's members in ascending
// channel order in fp64 and rounds once (the correctly rounded mean: within 1 ulp of torch's fp32 mean
// whatever its summation order), then every channel picks up its group's mean.  Replaces a Python loop
// of `group_num` boolean-index + mean + scatter launches (each with a host sync for the index count).
__global__ void __launch_bounds__(1024)
    group_mean_kernel(const float *values, const long long *labels, float *out, int channels, int wsz,
                      int groups) {
  extern __shared__ float s_mean[];  // [groups * wsz]
  for (int i = threadIdx.x; i < groups * wsz; i += blockDim.x) {
    const int g = i / wsz, col = i - g * wsz;
    double acc = 0.0;
    int cnt = 0;
    for (int c = 0; c < channels; ++c)
      if (labels[c] == g) {
        acc += (double)values[(int64_t)c * wsz + col];
        ++cnt;
      }
    s_mean[i] = cnt ? (float)(acc / (double)cnt) : 0.0f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < channels * wsz; i += blockDim.x) {
    const int c = i / wsz, col = i - c * wsz;
    const long long g = labels[c];
    out[i] = (g >= 0 && g < groups) ? s_mean[(int)g * wsz + col] : values[i];
  }
}

// ---------------------------------------------------------------------------
// The fused structured prune -> pow2 quantize parameter step as a stand-alone one-CTA launch
// (step_epilogue.cuh): used when the statistics come as finalized rows (reduce_stats output,
// chunks of a host tensor, all-gathered ranks), for > 1024 channels, or when the caller ran
// qsb_reduce_partials itself.  The training step proper uses the fused form,
// qsb_reduce_prune_quant_step (reduce.cu), where the last CTA of the reduction does this.
// ---------------------------------------------------------------------------
constexpr int kStepKernelThreads = 512;  // 128 registers per thread: the batched peer poll keeps 24 packets in flight
// LINES: the line form (a.lines != NULL)
template <bool LINES>
__global__ void __launch_bounds__(kStepKernelThreads)
    prune_quant_step_kernel(const __grid_constant__ StepArgs a) {
  pdl_wait();     // the partials come from the reduction launched just before
  pdl_trigger();  // the forward kernel's CTAs may queue up behind this single CTA
  extern __shared__ __align__(16) unsigned char qsb_dyn_smem[];  // step_smem_bytes(a.channels, LINES)
  step_epilogue<LINES>(a, carve_step_smem(qsb_dyn_smem, a.channels));
}

// Above the 48 KB of dynamic shared memory any kernel may take (from ~2400 channels) the kernel needs
// the opt-in, once per device.  cudaFuncSetAttribute is not a stream operation: it is legal while the
// caller's stream is being captured.
template <bool LINES>
static cudaError_t step_kernel_smem_opt_in() {
  static std::once_flag once[64];
  static cudaError_t err[64];
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) dev = 0;
  std::call_once(once[dev], [dev] {
    err[dev] = cudaFuncSetAttribute(prune_quant_step_kernel<LINES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)step_smem_bytes(LINES ? kLineStepMaxChannels : kStepMaxChannels, LINES));
  });
  return err[dev];
}

template <bool LINES>
static int launch_step_kernel_form(const StepArgs &a, cudaStream_t stream) {
  const size_t smem = step_smem_bytes(a.channels, LINES);
  if (smem > 48 * 1024) QSB_CUDA_TRY(step_kernel_smem_opt_in<LINES>());
  QSB_CUDA_TRY(launch_k(prune_quant_step_kernel<LINES>, dim3(1), dim3(kStepKernelThreads), smem, stream, a));
  return 0;
}

static int launch_step_kernel(const StepArgs &a, cudaStream_t stream) {
  return a.lines ? launch_step_kernel_form<true>(a, stream) : launch_step_kernel_form<false>(a, stream);
}

}  // namespace qsb

using namespace qsb;

extern "C" int qsb_abi_version(void) { return QSB_ABI_VERSION; }

extern "C" const char *qsb_error_string(int code) {
  switch (code) {
    case 0: return "success";
    case QSB_E_BADARG: return "qsparse_b200: bad argument";
    case QSB_E_WORKSPACE: return "qsparse_b200: workspace too small";
    case QSB_E_ALIGN: return "qsparse_b200: pointer not sufficiently aligned";
    case QSB_E_UNSUPPORTED: return "qsparse_b200: unsupported configuration";
    default:
      if (code > 0) return cudaGetErrorString((cudaError_t)code);
      return "qsparse_b200: unknown error";
  }
}

extern "C" int qsb_device_info(int *sm_count, int64_t *l2_bytes) {
  int dev = 0;
  QSB_CUDA_TRY(cudaGetDevice(&dev));
  const DeviceProps &p = device_props();
  if (sm_count) *sm_count = p.sm_count;
  if (l2_bytes) *l2_bytes = p.l2_bytes;
  return 0;
}

static inline unsigned blocks_for(int64_t n, int threads) {
  return (unsigned)((n + threads - 1) / threads);
}

extern "C" int qsb_scale_ema(float *weight, const float *absmax, int64_t n,
                             int bits, int64_t t, void *stream) {
  if (n < 0 || t < 0) return QSB_E_BADARG;
  if (n == 0) return 0;
  if (!weight || !absmax) return QSB_E_BADARG;
  const float limit = (float)pow(2.0, (double)bits - 1.0);
  scale_ema_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      weight, absmax, n, limit, t, nullptr);
  QSB_LAUNCH_CHECK();
  return 0;
}

// CUDA-graph forms: the step index is *t_dev + t_offset, read by the kernel; the caller advances the counter.
extern "C" int qsb_scale_ema_at(float *weight, const float *absmax, int64_t n, int bits,
                                const int64_t *t_dev, int64_t t_offset, void *stream) {
  if (n < 0 || !t_dev) return QSB_E_BADARG;
  if (n == 0) return 0;
  if (!weight || !absmax) return QSB_E_BADARG;
  const float limit = (float)pow(2.0, (double)bits - 1.0);
  scale_ema_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      weight, absmax, n, limit, t_offset, reinterpret_cast<const long long *>(t_dev));
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_lines_ema_at(float *lines, const float *mn, const float *mx, int64_t channels,
                                const int64_t *t_dev, int64_t t_offset, void *stream) {
  if (channels < 0 || !t_dev) return QSB_E_BADARG;
  if (channels == 0) return 0;
  if (!lines || !mn || !mx) return QSB_E_BADARG;
  lines_ema_kernel<<<blocks_for(channels, 256), 256, 0, (cudaStream_t)stream>>>(
      lines, mn, mx, channels, 0.f, 1.f, reinterpret_cast<const long long *>(t_dev), t_offset);
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_scale_to_decimal(const float *scale, float *decimal,
                                    int64_t n, void *stream) {
  if (n < 0) return QSB_E_BADARG;
  if (n == 0) return 0;
  if (!scale || !decimal) return QSB_E_BADARG;
  scale_to_decimal_kernel<<<blocks_for(n, 256), 256, 0, (cudaStream_t)stream>>>(
      scale, decimal, n);
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_lines_ema(float *lines, const float *mn, const float *mx,
                             int64_t channels, int64_t t, void *stream) {
  if (channels < 0 || t < 1) return QSB_E_BADARG;
  if (channels == 0) return 0;
  if (!lines || !mn || !mx) return QSB_E_BADARG;
  lines_ema_kernel<<<blocks_for(channels, 256), 256, 0, (cudaStream_t)stream>>>(
      lines, mn, mx, channels, (float)(t - 1), (float)t, nullptr, 0);
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_magnitude_ema_reduced(float *magnitude, const double *abssum,
                                         const double *nnz,
                                         const float *tensor_min, int use_l0,
                                         int64_t channels, double count,
                                         int64_t t, void *stream) {
  if (channels < 0 || t < 0 || !(count > 0)) return QSB_E_BADARG;
  if (channels == 0) return 0;
  if (!magnitude || !abssum) return QSB_E_BADARG;
  if (use_l0 && (!nnz || !tensor_min)) return QSB_E_BADARG;
  magnitude_ema_reduced_kernel<<<blocks_for(channels, 256), 256, 0,
                                 (cudaStream_t)stream>>>(
      magnitude, abssum, nnz, tensor_min, use_l0, channels, count, t);
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_group_mean(const float *values, const int64_t *labels, float *out, int64_t channels,
                              int64_t weight_size, int64_t groups, void *stream) {
  if (channels < 0 || weight_size < 1 || groups < 1) return QSB_E_BADARG;
  if (channels == 0) return 0;
  if (!values || !labels || !out) return QSB_E_BADARG;
  if (groups * weight_size > 8192 || channels > (1 << 24)) return QSB_E_UNSUPPORTED;
  group_mean_kernel<<<1, 1024, (size_t)(groups * weight_size) * sizeof(float), (cudaStream_t)stream>>>(
      values, reinterpret_cast<const long long *>(labels), out, (int)channels, (int)weight_size, (int)groups);
  QSB_LAUNCH_CHECK();
  return 0;
}

extern "C" int qsb_prune_quant_params(float *magnitude, uint8_t *mask,
                                      float *scale, float *decimal_out,
                                      const double *abssum, const float *absmax,
                                      int64_t n_stat_rows,
                                      int64_t stat_row_stride_bytes,
                                      int64_t channels, double count,
                                      int64_t t_prune, int update_magnitude,
                                      int refresh_mask, int64_t k, int bits,
                                      int64_t t_quant, int update_scale,
                                      void *stream) {
  if (channels <= 0 || channels > kStepMaxChannels) return QSB_E_UNSUPPORTED;
  // a statistic the step does not use may be NULL here (qsb_prune_quant_rows_step_params requires both)
  if (update_magnitude && (!abssum || !(count > 0))) return QSB_E_BADARG;
  if (update_scale && !absmax) return QSB_E_BADARG;
  if (n_stat_rows < 1 || n_stat_rows > 4096) return QSB_E_BADARG;
  StepArgs a;
  // `count` only divides the sums of an updated magnitude: any value is accepted otherwise
  const int rc = fill_step_args(a, magnitude, mask, scale, decimal_out, channels, nullptr, 0,
                                update_magnitude ? count : 1.0, t_prune, update_magnitude, refresh_mask, k, bits,
                                t_quant, update_scale, nullptr, nullptr, 0, nullptr, 1024);
  if (rc) return rc;
  return launch_step_kernel_on_rows(a, abssum, absmax, n_stat_rows, stat_row_stride_bytes, (cudaStream_t)stream);
}

// shared argument checks + StepArgs assembly of the parameter-step entry points
namespace qsb {
int launch_step_kernel_on_rows(StepArgs a, const double *row_sum, const float *row_max, int64_t n_rows,
                               int64_t row_stride, cudaStream_t stream) {
  a.row_sum = row_sum;
  a.row_max = row_max;
  a.n_rows = (int)n_rows;
  a.row_stride = row_stride;
  return launch_step_kernel(a, stream);
}

int fill_step_args(qsb::StepArgs &a, float *magnitude, uint8_t *mask, float *scale, float *decimal_out,
                   int64_t channels, qsb_p2p_group *group, int64_t step_stamp, double count, int64_t t_prune,
                   int update_magnitude, int refresh_mask, int64_t k, int bits, int64_t t_quant,
                   int update_scale, double *abssum_out, float *absmax_out, int stats_local,
                   int64_t *step_counter_dev, int threads) {
  if (!mask || !scale) return QSB_E_BADARG;
  if (update_magnitude < 0 || update_magnitude > 2) return QSB_E_BADARG;
  if (update_magnitude != 2 && !magnitude) return QSB_E_BADARG;
  if (!(count > 0)) return QSB_E_BADARG;
  if (refresh_mask && (k < 0 || k >= channels)) return QSB_E_BADARG;
  if ((abssum_out == nullptr) != (absmax_out == nullptr)) return QSB_E_BADARG;
  if (group && (group->channels != channels || (!step_counter_dev && step_stamp <= 0)))
    return QSB_E_BADARG;
  a = qsb::StepArgs{};
  a.magnitude = magnitude;
  a.mask = mask;
  a.scale = scale;
  a.decimal_out = decimal_out;
  a.channels = (int)channels;
  // the summation order of a channel depends on `group` only: derive it for the 256-thread CTA of the
  // fused reduction whatever the launch, so every route produces the same bits
  (void)threads;
  a.group = qsb::step_group_for(channels, 256);
  a.px.world = 1;
  if (group) a.px = group->dev;
  a.stamp = (unsigned long long)step_stamp;
  a.count = count;
  a.t_prune = t_prune;
  a.update_magnitude = update_magnitude;
  a.refresh_mask = refresh_mask;
  a.k = k;
  a.limit = (float)pow(2.0, (double)bits - 1.0);
  a.t_quant = t_quant;
  a.update_scale = update_scale;
  a.abssum_out = abssum_out;
  a.absmax_out = absmax_out;
  a.stats_local = stats_local;
  a.step_counter = reinterpret_cast<long long *>(step_counter_dev);
  return 0;
}

int fill_line_step_args(StepArgs &a, float *magnitude, uint8_t *mask, float *lines, int64_t n_lines,
                        int64_t channels, qsb_p2p_group *group, double count, int64_t t_prune, int update_magnitude,
                        int refresh_mask, int64_t k, int64_t t_line, double *abssum_out, float *min_out,
                        float *max_out, int64_t *step_counter_dev) {
  if (!lines || group) return QSB_E_BADARG;  // the line form runs on one GPU
  if (n_lines != 1 && n_lines != channels) return QSB_E_BADARG;
  if (!step_counter_dev && t_line < 1) return QSB_E_BADARG;
  // the pow2 checks and fields; `lines` stands in for the scale, which the line form never touches
  const int rc = fill_step_args(a, magnitude, mask, lines, nullptr, channels, nullptr, 0, count, t_prune,
                                update_magnitude, refresh_mask, k, 8, 0, 0, nullptr, nullptr, 0, step_counter_dev,
                                256);
  if (rc) return rc;
  a.scale = nullptr;
  a.lines = lines;
  a.n_lines = (int)n_lines;
  a.t_line = t_line;
  a.abssum_out = abssum_out;
  a.min_out = min_out;
  a.max_out = max_out;
  return 0;
}
}  // namespace qsb

extern "C" int qsb_prune_quant_step_params(
    float *magnitude, uint8_t *mask, float *scale, float *decimal_out,
    void *reduce_workspace, int64_t workspace_bytes, int64_t outer,
    int64_t channels, int64_t inner, qsb_p2p_group *group, int64_t step_stamp,
    double count, int64_t t_prune, int update_magnitude, int refresh_mask,
    int64_t k, int bits, int64_t t_quant, int update_scale, double *abssum_out,
    float *absmax_out, int64_t *step_counter_dev, void *stream) {
  if (channels <= 0 || channels > kStepMaxChannels) return QSB_E_UNSUPPORTED;
  if (outer <= 0 || inner <= 0 || !reduce_workspace) return QSB_E_BADARG;
  StepArgs a;
  const int rc = fill_step_args(a, magnitude, mask, scale, decimal_out, channels, group, step_stamp, count,
                                t_prune, update_magnitude, refresh_mask, k, bits, t_quant, update_scale,
                                abssum_out, absmax_out, 0, step_counter_dev, 1024);
  if (rc) return rc;
  const ReducePlan pl = make_plan(outer, channels, inner, nullptr);
  if (workspace_bytes < partial_bytes(pl.n_partials) + 256) return QSB_E_WORKSPACE;
  if (pl.fin_count > 0x7fffffffLL || pl.fin_q > 0x7fffffffLL) return QSB_E_UNSUPPORTED;
  a.P = partials_from_workspace(reduce_workspace, pl.n_partials);
  a.fin_count = (int)pl.fin_count;
  a.fin_q = (int)pl.fin_q;
  return launch_step_kernel(a, (cudaStream_t)stream);
}

// The same parameter step on FINALIZED statistics rows (one per staged chunk of a host
// tensor), with the peer exchange: what the host-buffer pipeline uses at N > 1 GPUs.
extern "C" int qsb_prune_quant_rows_step_params(
    float *magnitude, uint8_t *mask, float *scale, float *decimal_out, const double *abssum,
    const float *absmax, int64_t n_stat_rows, int64_t stat_row_stride_bytes, int64_t channels,
    qsb_p2p_group *group, int64_t step_stamp, double count, int64_t t_prune, int update_magnitude,
    int refresh_mask, int64_t k, int bits, int64_t t_quant, int update_scale, void *stream) {
  if (channels <= 0 || channels > kStepMaxChannels) return QSB_E_UNSUPPORTED;
  if (!abssum || !absmax || n_stat_rows < 1 || n_stat_rows > 4096) return QSB_E_BADARG;
  StepArgs a;
  const int rc = fill_step_args(a, magnitude, mask, scale, decimal_out, channels, group, step_stamp, count,
                                t_prune, update_magnitude, refresh_mask, k, bits, t_quant, update_scale,
                                nullptr, nullptr, 0, nullptr, 1024);
  if (rc) return rc;
  return launch_step_kernel_on_rows(a, abssum, absmax, n_stat_rows, stat_row_stride_bytes, (cudaStream_t)stream);
}

// The line form on the partials of qsb_reduce_line_partials_dt (1025 - 2048 channels).
extern "C" int qsb_prune_line_step_params(
    float *magnitude, uint8_t *mask, float *lines, int64_t n_lines, void *reduce_workspace, int64_t workspace_bytes,
    int64_t outer, int64_t channels, int64_t inner, qsb_p2p_group *group, double count, int64_t t_prune,
    int update_magnitude, int refresh_mask, int64_t k, int64_t t_line, double *abssum_out, float *min_out,
    float *max_out, int64_t *step_counter_dev, void *stream) {
  if (outer <= 0 || channels <= 0 || inner <= 0 || !reduce_workspace) return QSB_E_BADARG;
  if (channels > kLineStepMaxChannels) return QSB_E_UNSUPPORTED;
  StepArgs a;
  const int rc = fill_line_step_args(a, magnitude, mask, lines, n_lines, channels, group, count, t_prune,
                                     update_magnitude, refresh_mask, k, t_line, abssum_out, min_out, max_out,
                                     step_counter_dev);
  if (rc) return rc;
  const ReducePlan pl = make_plan(outer, channels, inner, nullptr);
  if (workspace_bytes < partial_bytes(pl.n_partials) + 256) return QSB_E_WORKSPACE;
  if (pl.fin_count > 0x7fffffffLL || pl.fin_q > 0x7fffffffLL) return QSB_E_UNSUPPORTED;
  a.P = partials_from_workspace(reduce_workspace, pl.n_partials);
  a.fin_count = (int)pl.fin_count;
  a.fin_q = (int)pl.fin_q;
  return launch_step_kernel(a, (cudaStream_t)stream);
}
