// Host-buffer entry points: what a caller that keeps its tensors in CPU memory
// binds to.  One fused training step of prune(channel) -> pow2 quantize on HOST
// tensors (x, g in; y, gx out), pipelined over batch chunks on three streams:
//
//   h2d stream : x chunk 0..n-1, then g chunk 0..n-1              (PCIe up)
//   compute    : reduce(x_i) as each x chunk lands -> params (all chunks' stats,
//                combined in chunk order) -> y_i = Q(x_i * mask) -> gx_i
//   d2h stream : y chunk i as soon as it is computed, then gx chunks (PCIe down)
//
// The step's statistics need every x chunk before anything can be applied, so the
// critical path is  upload(x) -> [download(y) || upload(g)] -> download(gx).
// The context owns the device buffers, streams and events; host buffers should be
// pinned (cudaHostAlloc / torch pin_memory) for the copies to be asynchronous.
//
// The PCIe link is full duplex, and a single step only uses one direction at a time for
// most of its life.  qsb_host_prune_quant_step_submit() / qsb_host_ctx_wait() run TWO steps
// in flight on two sets of staging buffers ("slots"): step t+1's x and g go up while step
// t's y and gx come down, so the steady state is max(up, down) = 2 tensors per step per
// direction instead of the 3 serial transfers of one step.
#include <stdlib.h>

#include <vector>

#include "p2p_internal.cuh"
#include "qsb_common.cuh"

constexpr int kHostSlots = 2;  // steps in flight: step t+1 uploads while step t downloads

struct qsb_host_slot {
  float *d_x, *d_g, *d_y, *d_gx;
  std::vector<cudaEvent_t> ev_x, ev_g, ev_y, ev_gx;
  cudaEvent_t ev_comp_done;  // compute stream: the slot's device inputs are no longer read
  cudaEvent_t ev_down_done;  // download stream: the slot's results are in the host buffers
  bool busy;
};

struct qsb_host_ctx {
  int64_t max_elems;
  int n_chunks;
  qsb_host_slot slot[kHostSlots];
  unsigned char *d_ws;       // n_chunks reduce workspaces
  int64_t ws_bytes_per_chunk;
  unsigned char *d_stats;    // n_chunks rows of [C doubles | C floats], padded
  int64_t stats_row_bytes;
  int64_t max_channels;
  cudaStream_t s_h2d, s_comp, s_d2h;
  cudaEvent_t ev_begin;
};

extern "C" int qsb_host_ctx_create(qsb_host_ctx **out, int64_t max_elems,
                                   int64_t max_channels, int n_chunks) {
  if (!out || max_elems <= 0 || max_channels <= 0 || n_chunks < 1 || n_chunks > 256)
    return QSB_E_BADARG;
  qsb_host_ctx *c = new qsb_host_ctx();
  c->max_elems = max_elems;
  c->n_chunks = n_chunks;
  c->max_channels = max_channels;
  const size_t bytes = (size_t)max_elems * sizeof(float);
  auto make = [&](std::vector<cudaEvent_t> &v) {
    v.resize(n_chunks);
    for (auto &e : v)
      if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return false;
    return true;
  };
  for (auto &sl : c->slot) {
    QSB_CUDA_TRY(cudaMalloc(&sl.d_x, bytes));
    QSB_CUDA_TRY(cudaMalloc(&sl.d_g, bytes));
    QSB_CUDA_TRY(cudaMalloc(&sl.d_y, bytes));
    QSB_CUDA_TRY(cudaMalloc(&sl.d_gx, bytes));
    if (!make(sl.ev_x) || !make(sl.ev_g) || !make(sl.ev_y) || !make(sl.ev_gx))
      return (int)cudaGetLastError();
    QSB_CUDA_TRY(cudaEventCreateWithFlags(&sl.ev_comp_done, cudaEventDisableTiming));
    QSB_CUDA_TRY(cudaEventCreateWithFlags(&sl.ev_down_done, cudaEventDisableTiming));
    sl.busy = false;
  }
  // the reduce workspace is sized at the first step
  c->ws_bytes_per_chunk = 0;
  c->d_ws = nullptr;
  c->stats_row_bytes = ((max_channels * 12 + 255) / 256) * 256;
  QSB_CUDA_TRY(cudaMalloc(&c->d_stats, (size_t)c->stats_row_bytes * n_chunks));
  QSB_CUDA_TRY(cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking));
  QSB_CUDA_TRY(cudaStreamCreateWithFlags(&c->s_comp, cudaStreamNonBlocking));
  QSB_CUDA_TRY(cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking));
  QSB_CUDA_TRY(cudaEventCreateWithFlags(&c->ev_begin, cudaEventDisableTiming));
  *out = c;
  return 0;
}

extern "C" int qsb_host_ctx_destroy(qsb_host_ctx *c) {
  if (!c) return 0;
  cudaStreamSynchronize(c->s_h2d);
  cudaStreamSynchronize(c->s_comp);
  cudaStreamSynchronize(c->s_d2h);
  for (auto &sl : c->slot) {
    cudaFree(sl.d_x);
    cudaFree(sl.d_g);
    cudaFree(sl.d_y);
    cudaFree(sl.d_gx);
    for (auto *v : {&sl.ev_x, &sl.ev_g, &sl.ev_y, &sl.ev_gx})
      for (auto e : *v) cudaEventDestroy(e);
    cudaEventDestroy(sl.ev_comp_done);
    cudaEventDestroy(sl.ev_down_done);
  }
  if (c->d_ws) cudaFree(c->d_ws);
  cudaFree(c->d_stats);
  cudaEventDestroy(c->ev_begin);
  cudaStreamDestroy(c->s_h2d);
  cudaStreamDestroy(c->s_comp);
  cudaStreamDestroy(c->s_d2h);
  delete c;
  return 0;
}

extern "C" int qsb_host_ctx_wait(qsb_host_ctx *c, int slot) {
  if (!c || slot < 0 || slot >= kHostSlots) return QSB_E_BADARG;
  qsb_host_slot &sl = c->slot[slot];
  if (!sl.busy) return 0;
  // the download stream runs behind the compute stream, so this covers both
  QSB_CUDA_TRY(cudaEventSynchronize(sl.ev_down_done));
  QSB_CUDA_TRY(cudaEventSynchronize(sl.ev_comp_done));
  sl.busy = false;
  return 0;
}

extern "C" int qsb_host_prune_quant_step_submit(
    qsb_host_ctx *c, int slot, const float *x_host, const float *g_host, float *y_host,
    float *gx_host, float *magnitude_dev, uint8_t *mask_dev, float *scale_dev,
    float *decimal_dev, int64_t outer, int64_t channels, int64_t inner,
    int64_t t_prune, int64_t k, int bits, int64_t t_quant, qsb_p2p_group *group,
    int64_t step_stamp, void *caller_stream) {
  if (!c || slot < 0 || slot >= kHostSlots) return QSB_E_BADARG;
  if (!x_host || !g_host || !y_host || !gx_host) return QSB_E_BADARG;
  if (outer <= 0 || channels <= 0 || inner <= 0) return QSB_E_BADARG;
  if (channels > c->max_channels || outer * channels * inner > c->max_elems)
    return QSB_E_BADARG;
  qsb_host_slot &sl = c->slot[slot];
  if (sl.busy) {  // the slot's previous step must have been waited for: its host buffers
    int rc = qsb_host_ctx_wait(c, slot);  // and device staging are about to be reused
    if (rc) return rc;
  }
  int n_chunks = c->n_chunks;
  if (n_chunks > outer) n_chunks = (int)outer;
  const int64_t rows_per_chunk = (outer + n_chunks - 1) / n_chunks;
  n_chunks = (int)((outer + rows_per_chunk - 1) / rows_per_chunk);
  const int64_t row_elems = channels * inner;

  // reduce workspace (sized once for the largest chunk seen so far)
  const int64_t last_rows = outer - (int64_t)(n_chunks - 1) * rows_per_chunk;
  int64_t need_ws = qsb_reduce_workspace_bytes(rows_per_chunk, channels, inner);
  const int64_t need_last = qsb_reduce_workspace_bytes(last_rows, channels, inner);
  if (need_last > need_ws) need_ws = need_last;
  if (need_ws > c->ws_bytes_per_chunk) {
    QSB_CUDA_TRY(cudaDeviceSynchronize());
    if (c->d_ws) cudaFree(c->d_ws);
    c->ws_bytes_per_chunk = (need_ws + 255) / 256 * 256;
    QSB_CUDA_TRY(cudaMalloc(&c->d_ws, (size_t)c->ws_bytes_per_chunk * c->n_chunks));
  }

  // order the pipeline after whatever the caller queued on its stream (the state tensors).
  // The three streams are in-order, so consecutive steps line up behind each other:
  //   upload   : x_t, g_t, x_t+1, g_t+1, ...
  //   compute  : reduce_t, params_t, fwd_t, bwd_t, reduce_t+1, ...   (the layer state is
  //              only touched here: params_t+1 runs after bwd_t has used mask_t / decimal_t)
  //   download : y_t, gx_t, y_t+1, ...
  cudaStream_t cs = (cudaStream_t)caller_stream;
  QSB_CUDA_TRY(cudaEventRecord(c->ev_begin, cs));
  QSB_CUDA_TRY(cudaStreamWaitEvent(c->s_comp, c->ev_begin, 0));
  QSB_CUDA_TRY(cudaStreamWaitEvent(c->s_h2d, c->ev_begin, 0));

  auto chunk_range = [&](int i, int64_t &r0, int64_t &nr) {
    r0 = (int64_t)i * rows_per_chunk;
    nr = (r0 + rows_per_chunk <= outer) ? rows_per_chunk : outer - r0;
  };
  int rc;
  // ---- upload x chunk by chunk; reduce each as it lands -------------------
  for (int i = 0; i < n_chunks; ++i) {
    int64_t r0, nr;
    chunk_range(i, r0, nr);
    const int64_t off = r0 * row_elems, cnt = nr * row_elems;
    QSB_CUDA_TRY(cudaMemcpyAsync(sl.d_x + off, x_host + off, cnt * sizeof(float),
                                 cudaMemcpyHostToDevice, c->s_h2d));
    QSB_CUDA_TRY(cudaEventRecord(sl.ev_x[i], c->s_h2d));
    QSB_CUDA_TRY(cudaStreamWaitEvent(c->s_comp, sl.ev_x[i], 0));
    unsigned char *row = c->d_stats + (int64_t)i * c->stats_row_bytes;
    double *abssum = reinterpret_cast<double *>(row);
    float *absmax = reinterpret_cast<float *>(row + channels * sizeof(double));
    rc = qsb_reduce_stats(sl.d_x + off, QSB_STAT_ABSSUM | QSB_STAT_ABSMAX, nr,
                          channels, inner, absmax, nullptr, nullptr, abssum,
                          nullptr, nullptr, c->d_ws + (int64_t)i * c->ws_bytes_per_chunk,
                          c->ws_bytes_per_chunk, c->s_comp);
    if (rc) return rc;
  }
  // ---- upload g behind x on the same copy stream ---------------------------
  for (int i = 0; i < n_chunks; ++i) {
    int64_t r0, nr;
    chunk_range(i, r0, nr);
    const int64_t off = r0 * row_elems, cnt = nr * row_elems;
    QSB_CUDA_TRY(cudaMemcpyAsync(sl.d_g + off, g_host + off, cnt * sizeof(float),
                                 cudaMemcpyHostToDevice, c->s_h2d));
    QSB_CUDA_TRY(cudaEventRecord(sl.ev_g[i], c->s_h2d));
  }
  // ---- parameters from all chunks' statistics -------------------------------
  // The chunk rows are summed in chunk order and, with N > 1 GPUs, exchanged with the peers over
  // NVLink inside the same kernel and combined in rank order — the same computation as the
  // resident path's fused step.
  {
    const double *abssum0 = reinterpret_cast<const double *>(c->d_stats);
    const float *absmax0 =
        reinterpret_cast<const float *>(c->d_stats + channels * sizeof(double));
    const double world = group ? (double)group->dev.world : 1.0;
    rc = qsb_prune_quant_rows_step_params(
        magnitude_dev, mask_dev, scale_dev, decimal_dev, abssum0, absmax0, n_chunks,
        c->stats_row_bytes, channels, group, step_stamp, (double)outer * (double)inner * world, t_prune, 1,
        t_prune > 0, k, bits, t_quant, 1, c->s_comp);
    if (rc) return rc;
  }
  // ---- forward apply per chunk, download y ---------------------------------
  for (int i = 0; i < n_chunks; ++i) {
    int64_t r0, nr;
    chunk_range(i, r0, nr);
    const int64_t off = r0 * row_elems, cnt = nr * row_elems;
    rc = qsb_fq_pow2_fwd(sl.d_x + off, sl.d_y + off, decimal_dev, 1, 0.0, mask_dev,
                         QSB_MASK_CHANNEL, nr, channels, inner, c->s_comp);
    if (rc) return rc;
    QSB_CUDA_TRY(cudaEventRecord(sl.ev_y[i], c->s_comp));
    QSB_CUDA_TRY(cudaStreamWaitEvent(c->s_d2h, sl.ev_y[i], 0));
    QSB_CUDA_TRY(cudaMemcpyAsync(y_host + off, sl.d_y + off, cnt * sizeof(float),
                                 cudaMemcpyDeviceToHost, c->s_d2h));
  }
  // ---- backward per chunk, download gx --------------------------------------
  for (int i = 0; i < n_chunks; ++i) {
    int64_t r0, nr;
    chunk_range(i, r0, nr);
    const int64_t off = r0 * row_elems, cnt = nr * row_elems;
    QSB_CUDA_TRY(cudaStreamWaitEvent(c->s_comp, sl.ev_g[i], 0));
    rc = qsb_ste_bwd(sl.d_g + off, nullptr, sl.d_gx + off, decimal_dev, 1, 0.0, 1,
                     bits, 0, mask_dev, QSB_MASK_CHANNEL, nr, channels, inner,
                     c->s_comp);
    if (rc) return rc;
    QSB_CUDA_TRY(cudaEventRecord(sl.ev_gx[i], c->s_comp));
    QSB_CUDA_TRY(cudaStreamWaitEvent(c->s_d2h, sl.ev_gx[i], 0));
    QSB_CUDA_TRY(cudaMemcpyAsync(gx_host + off, sl.d_gx + off, cnt * sizeof(float),
                                 cudaMemcpyDeviceToHost, c->s_d2h));
  }
  QSB_CUDA_TRY(cudaEventRecord(sl.ev_comp_done, c->s_comp));
  QSB_CUDA_TRY(cudaEventRecord(sl.ev_down_done, c->s_d2h));
  sl.busy = true;
  return 0;
}

extern "C" int qsb_host_prune_quant_step(
    qsb_host_ctx *c, const float *x_host, const float *g_host, float *y_host,
    float *gx_host, float *magnitude_dev, uint8_t *mask_dev, float *scale_dev,
    float *decimal_dev, int64_t outer, int64_t channels, int64_t inner,
    int64_t t_prune, int64_t k, int bits, int64_t t_quant, qsb_p2p_group *group,
    int64_t step_stamp, void *caller_stream) {
  // results are in the host buffers when this returns
  int rc = qsb_host_prune_quant_step_submit(c, 0, x_host, g_host, y_host, gx_host, magnitude_dev,
                                            mask_dev, scale_dev, decimal_dev, outer, channels,
                                            inner, t_prune, k, bits, t_quant, group, step_stamp,
                                            caller_stream);
  if (rc) return rc;
  return qsb_host_ctx_wait(c, 0);
}
