/*
 * qsparse_b200 — C-ABI of the B200-native quantize/prune hot path.
 *
 * This header is the drop-in boundary (SURVEY.md §8b).  Every entry point is a
 * stateless launcher: plain device pointers + sizes + a cudaStream_t (passed as
 * void*), no torch types, no allocation, no host synchronisation.  The caller
 * owns every buffer (inputs, outputs, workspace).  Scalars that the reference
 * derives on the device (learned decimal / scale / lines / threshold) stay on
 * the device and are passed as pointers.
 *
 * Tensor layout convention: a contiguous fp32 tensor is described as
 * [outer, channels, inner] (row-major).  Per-tensor parameters use
 * channels == 1 (outer == 1, inner == numel).  The channel of flat element e
 * is (e / inner) % channels.
 *
 * Return value: 0 on success, a positive cudaError_t on a CUDA failure, a
 * negative QSB_E_* code on an argument error.  qsb_error_string() names both.
 *
 * "ref:" comments cite the file:line of mlzxy/qsparse v2.0.1 that the entry
 * point replaces.
 */
#ifndef QSPARSE_B200_H_
#define QSPARSE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QSB_ABI_VERSION 4

/* argument errors */
#define QSB_E_BADARG (-1)     /* null pointer / negative size / bad enum        */
#define QSB_E_WORKSPACE (-2)  /* workspace too small (see *_workspace_bytes)    */
#define QSB_E_ALIGN (-3)      /* pointer not 4-byte aligned                     */
#define QSB_E_UNSUPPORTED (-4)

/* element type of a tensor argument of the *_dt entry points.  16-bit inputs are
 * upcast on load (exact) and computed in fp32, so a bf16 / fp16 x gives bit for
 * bit what the fp32 entry point gives on x converted to fp32; 16-bit outputs are
 * rounded to nearest even (what a cast of the fp32 result rounds to).  16-bit
 * pointers need only 2-byte alignment.  Any other code is QSB_E_BADARG. */
#define QSB_DTYPE_F32 0
#define QSB_DTYPE_BF16 1
#define QSB_DTYPE_F16 2

/* mask_kind */
#define QSB_MASK_NONE 0
#define QSB_MASK_CHANNEL 1 /* uint8 mask[channels]  (structured prune)          */
#define QSB_MASK_ELEMENT 2 /* uint8 mask[numel]     (unstructured prune)        */

/* `what` bits of qsb_reduce_stats */
#define QSB_STAT_ABSMAX 1 /* max |x|            -> float  absmax[channels]      */
#define QSB_STAT_MINMAX 2 /* min x, max x       -> float  mn[channels], mx[..]  */
#define QSB_STAT_ABSSUM 4 /* sum |x| (fp64)     -> double abssum[channels]      */
#define QSB_STAT_NNZ 8    /* count(x != 0), min x (whole tensor, for l0 mode)   */

int qsb_abi_version(void);
const char *qsb_error_string(int code);
/* SM count and L2 size of the current device. */
int qsb_device_info(int *sm_count, int64_t *l2_bytes);
/* Development only (library built with -DQSB_KERNEL_TIMING, else QSB_E_UNSUPPORTED): out_host == NULL resets,
 * otherwise reads 3 x 2 x 256 uint64 %globaltimer stamps [statistics / forward / backward kernel][first CTA
 * start, last CTA end][SM] — the in-situ durations of a graph-replayed step without event records. */
int qsb_debug_kernel_times(unsigned long long *out_host, void *stream);
/* Benchmark knobs and one test hook; defaults are what the product uses.
 *   key 2: tile order of the one-CTA-per-tile kernels: 1 (default) = last tile first
 *          (re-reads the L2-resident tail of a just-touched tensor) except in the
 *          channel-masked kernels, which follow the fused statistics kernel and its
 *          L2 keep tags and measured faster first tile first; 2 = always last tile
 *          first; 0 = always first tile first;
 *   key 4: test hook: 1 = sampled-pivot ~1-pass route of qsb_kth_value for n >= 2^22
 *          (default), 0 = always the 3-pass radix select;
 *   key 12: 1 = the streaming, reduction and fused-parameter kernels are launched with
 *          programmatic stream serialization (each begins with griddepcontrol.wait, so
 *          stream order is unchanged; launch latency overlaps the predecessor's tail);
 *   key 17: row-mode statistics kernels: 2 = 8 x 256-bit loads in flight per lane, 2 CTAs / SM,
 *          0 = 4 loads, 4 CTAs / SM, any other value = by row length (default: 2 for rows of
 *          >= 2048 elements, else 0); the reduction plan — and with it the summation order — follows;
 *   key 18: 1 = qsb_reduce_prune_quant_step reads the channels the previous mask keeps with
 *          L2::evict_last (the forward pass re-reads exactly those next) and the rest with
 *          L2::evict_first (default), 0 = default policy for everything;
 *   key 21: L2 set-aside for persisting accesses in MB (cudaLimitPersistingL2CacheSize, device-wide;
 *          untouched by default).  A development probe only: every set-aside >= 32 MB HALVED the
 *          speed of the streaming kernels on B200 (profiles/r02_l2_set_aside.jsonl).
 * Any other key returns QSB_E_BADARG. */
int qsb_set_tuning(int key, int value);
/* Test hook: compares the kernels' reciprocal-based exact division with
 * __fdiv_rn on n_threads * pairs_per_thread pseudo-random operand pairs and
 * adds the number of bit mismatches to *mismatches_dev (must be zeroed). */
int qsb_selftest_fastdiv(int64_t n_threads, int64_t pairs_per_thread,
                         uint64_t seed, unsigned long long *mismatches_dev,
                         void *stream);

/* ------------------------------------------------------------------------
 * K1  fake-quant forward.  y may alias x.  An optional prune mask is applied
 * first (y = Q(x * mask)): that is the fused prune->quantize of K7.
 * ---------------------------------------------------------------------- */

/* ref: DecimalQuantization.forward  qsparse/quantize.py:30-63
 *   y = float(int32_rz(x * 2^d)) * 2^-d          (the clamp at :56-62 is dead)
 * decimal_dev: device float[n_decimal] (n_decimal == 1 or == channels), or NULL
 * to use the host scalar decimal_host. */
int qsb_fq_pow2_fwd(const float *x, float *y, const float *decimal_dev,
                    int64_t n_decimal, double decimal_host,
                    const uint8_t *mask_dev, int mask_kind, int64_t outer,
                    int64_t channels, int64_t inner, void *stream);

/* ref: ScalerQuantization.forward  qsparse/quantize.py:86-117
 *   y = float(int32_rz(rint(x / s))) * s          (IEEE division) */
int qsb_fq_scaler_fwd(const float *x, float *y, const float *scaler_dev,
                      int64_t n_scaler, float scaler_host,
                      const uint8_t *mask_dev, int mask_kind, int64_t outer,
                      int64_t channels, int64_t inner, void *stream);

/* ref: LineQuantization.forward  qsparse/quantize.py:140-181
 * lines_dev: device float[n_lines][2] = (lo, hi) rows (n_lines == 1 or
 * channels), or NULL to use (lo_host, hi_host).
 * float_zero_point != 0: training form (:168-181); == 0: eval form (:161-166). */
int qsb_fq_line_fwd(const float *x, float *y, const float *lines_dev,
                    int64_t n_lines, float lo_host, float hi_host, int bits,
                    int float_zero_point, const uint8_t *mask_dev,
                    int mask_kind, int64_t outer, int64_t channels,
                    int64_t inner, void *stream);

/* The three forwards on an x of element type x_dtype (QSB_DTYPE_*); y stays fp32.
 * The fp32 entry points above are the QSB_DTYPE_F32 case. */
int qsb_fq_pow2_fwd_dt(const void *x, int x_dtype, float *y, const float *decimal_dev,
                       int64_t n_decimal, double decimal_host,
                       const uint8_t *mask_dev, int mask_kind, int64_t outer,
                       int64_t channels, int64_t inner, void *stream);
int qsb_fq_scaler_fwd_dt(const void *x, int x_dtype, float *y, const float *scaler_dev,
                         int64_t n_scaler, float scaler_host,
                         const uint8_t *mask_dev, int mask_kind, int64_t outer,
                         int64_t channels, int64_t inner, void *stream);
int qsb_fq_line_fwd_dt(const void *x, int x_dtype, float *y, const float *lines_dev,
                       int64_t n_lines, float lo_host, float hi_host, int bits,
                       int float_zero_point, const uint8_t *mask_dev,
                       int mask_kind, int64_t outer, int64_t channels,
                       int64_t inner, void *stream);

/* Integer export (SURVEY 8f-3): the integer CODE of a fake-quantizer, one byte per
 * element (5 B/elem instead of 8), for deployment after quantization-aware training.
 *   kind 0 (decimal): q = clamp(int32_rz(x * 2^d), -2^(b-1), 2^(b-1)-1)   as int8
 *                     param = decimal; dequantised value  q * 2^-d
 *   kind 1 (scaler) : q = clamp(int32(rint(x / s)), -2^(b-1), 2^(b-1)-1)  as int8
 *                     param = scale;   dequantised value  q * s
 *   kind 2 (line)   : q = clamp(rint((clamp(x, lo, hi) - lo) / step), 0, 2^b - 1) as uint8
 *                     param = (lo, hi) rows; step = (hi - lo) / 2^b; value q * step + lo
 * param_dev: per tensor (n_param == 1) or per channel (n_param == channels), or NULL to
 * use param_host (and param_host2 = hi for kind 2).  bits <= 8.  Inside the clamp range
 * the dequantised value equals qsb_fq_*_fwd's output bit for bit.
 * ref: the integer-arithmetic property qsparse proves in tests/test_quantize.py:73-101;
 *      qsparse/quantize.py:55-63, :107-117, :168-181 for the codes. */
int qsb_quant_export_int8(const float *x, uint8_t *q_out, int kind,
                          const float *param_dev, int64_t n_param,
                          double param_host, double param_host2, int bits,
                          int64_t outer, int64_t channels, int64_t inner,
                          void *stream);

/* The same codes for bits <= 4, packed two per byte in flat element order: byte i holds
 * element 2i in its low nibble and element 2i+1 in its high nibble (kinds 0/1: 4-bit two's
 * complement; kind 2: unsigned); q_out has (n + 1) / 2 bytes, an odd n leaves the last high
 * nibble 0.  4.5 B/elem.  ref: as qsb_quant_export_int8 (SURVEY 8f-3 "int4-packed"). */
int qsb_quant_export_int4(const float *x, uint8_t *q_out, int kind,
                          const float *param_dev, int64_t n_param,
                          double param_host, double param_host2, int bits,
                          int64_t outer, int64_t channels, int64_t inner,
                          void *stream);

/* Block-scaled FP8 / FP4 fake quantization (EXTENSION; DESIGN §2 "Block-scaled formats").
 * x (element type x_dtype, QSB_DTYPE_*) is [rows, L] in memory order; each row splits into
 * blocks of B consecutive elements (the last one may be shorter), a = the block's max |x|:
 *   fmt 0 MXFP8: B 32, E4M3 elements, X = 2^clamp(e(a) - 8, -127, 127), y = cvt_e4m3(x / X) * X
 *   fmt 1 MXFP4: B 32, E2M1 elements, X = 2^clamp(e(a) - 2, -127, 127), y = cvt_e2m1(x / X) * X
 *   fmt 2 NVFP4: B 16, E2M1 elements, s_t = w / 2688, s_b = cvt_e4m3(a / 6 / s_t),
 *                d = s_b * s_t, y = cvt_e2m1(x / d) * d  (+0 for the block when d == 0)
 * e(a) = floor(log2 a) from the bits of a; cvt_* round to nearest even and saturate.  A block
 * holding a NaN or +-inf gives NaN; for NVFP4 a NaN s_t gives NaN and a zero s_t +0 everywhere.
 * w = *tensor_amax_dev (NVFP4 only; ignored otherwise).  y is fp32 [rows, L].  8 B/elem (fp32
 * x), 6 B/elem (16-bit x).  NULL pointers, a bad fmt / dtype or negative sizes: QSB_E_BADARG. */
#define QSB_BLOCK_MXFP8 0
#define QSB_BLOCK_MXFP4 1
#define QSB_BLOCK_NVFP4 2
int qsb_fq_block_fwd_dt(const void *x, int x_dtype, float *y, int64_t rows, int64_t L, int fmt,
                        const float *tensor_amax_dev, void *stream);

/* The packed form of the same quantizer, in one pass:
 *   codes  E4M3 (MXFP8): uint8 [rows, L];  E2M1: uint8 [rows, (L + 1) / 2], element 2i in the
 *          low nibble, a zero pad nibble when L is odd (codes are 0 in a NaN or zero-scale block)
 *   scales uint8 [rows, ceil(L / B)]: E8M0 (0xFF for a NaN block) or, for NVFP4, E4M3 s_b
 *          (0x7F for a NaN block or a NaN s_t, 0 for a zero s_t).
 * Decoding code * 2^(scale - 127), or code * RN(s_b * s_t), gives qsb_fq_block_fwd_dt's y. */
int qsb_block_export_dt(const void *x, int x_dtype, uint8_t *codes, uint8_t *scales, int64_t rows,
                        int64_t L, int fmt, const float *tensor_amax_dev, void *stream);

/* ------------------------------------------------------------------------
 * K2  straight-through-estimator backward (and the fused prune backward).
 * ref: DecimalQuantization.backward qsparse/quantize.py:65-77,
 *      ScalerQuantization.backward  qsparse/quantize.py:119-131
 *   v = clamp(g, (-L+notch)*s, (L-1+notch)*s), NaN -> 0,  L = 2^(bits-1)
 *   s = 2^-d when scale_is_decimal, else the scaler itself.
 * g_clamped_out: where v is written; pass g itself for the reference's in-place
 *   side effect (quantize.py:72), or NULL to skip it.
 * gx_out: where v * mask is written (the autograd of `x * mask`,
 *   sparse.py:66,116), or v itself when mask_kind == QSB_MASK_NONE; may be NULL.
 * ---------------------------------------------------------------------- */
int qsb_ste_bwd(const float *g, float *g_clamped_out, float *gx_out,
                const float *scale_dev, int64_t n_scale, double scale_host,
                int scale_is_decimal, int bits, int notch,
                const uint8_t *mask_dev, int mask_kind, int64_t outer,
                int64_t channels, int64_t inner, void *stream);
/* The same with gx_out of element type gx_dtype (QSB_DTYPE_*): the input gradient
 * of a 16-bit x written in x's dtype in the same pass that clamps g in place
 * (g and g_clamped_out stay fp32). */
int qsb_ste_bwd_dt(const float *g, float *g_clamped_out, void *gx_out, int gx_dtype,
                   const float *scale_dev, int64_t n_scale, double scale_host,
                   int scale_is_decimal, int bits, int notch,
                   const uint8_t *mask_dev, int mask_kind, int64_t outer,
                   int64_t channels, int64_t inner, void *stream);

/* ------------------------------------------------------------------------
 * K6  prune mask apply, forward and backward (same arithmetic).
 * ref: `x * mask`  qsparse/sparse.py:66,116,122,263  (fp32 multiply by 0.0/1.0,
 * so the sign of zero and inf*0 = NaN are preserved). y may alias x.
 * ---------------------------------------------------------------------- */
int qsb_mask_apply(const float *x, float *y, const uint8_t *mask_dev,
                   int mask_kind, int64_t outer, int64_t channels,
                   int64_t inner, void *stream);
/* x of element type x_dtype, y of element type y_dtype (QSB_DTYPE_*): a 16-bit
 * activation masked into an fp32 y (forward), an fp32 gradient masked into a
 * 16-bit gx (backward).  y may alias x only when the dtypes are equal. */
int qsb_mask_apply_dt(const void *x, int x_dtype, void *y, int y_dtype,
                      const uint8_t *mask_dev, int mask_kind, int64_t outer,
                      int64_t channels, int64_t inner, void *stream);

/* ------------------------------------------------------------------------
 * K3  statistic reductions, one read of x for any combination of `what`.
 * ref: DecimalQuantizer.optimize  qsparse/quantize.py:329-340 (abs-max)
 *      AdaptiveQuantizer.optimize qsparse/quantize.py:396-418 (min / max)
 *      squeeze_tensor_to_shape    qsparse/util.py:79-99       (mean |x|)
 *      MagnitudePruningCallback.update_magnitude sparse.py:85-87 (l0: x != 0)
 * Outputs are per channel; unused outputs may be NULL.
 *   absmax/mn/mx : float[channels]
 *   abssum       : double[channels]   (fp64 accumulation, fixed order)
 *   nnz          : double[channels]   count of x != 0
 *   tensor_min   : float[1]           min over the whole tensor (l0 gate)
 * Deterministic: two-stage with a fixed combination order, no float atomics.
 * ---------------------------------------------------------------------- */
int64_t qsb_reduce_workspace_bytes(int64_t outer, int64_t channels,
                                   int64_t inner);
int qsb_reduce_stats(const float *x, int what, int64_t outer, int64_t channels,
                     int64_t inner, float *absmax, float *mn, float *mx,
                     double *abssum, double *nnz, float *tensor_min,
                     void *workspace, int64_t workspace_bytes, void *stream);
/* qsb_reduce_stats on an x of element type x_dtype (QSB_DTYPE_*).  The reduction plan —
 * segments, row bands, vectors of 8, fp32 pre-sums and with them the summation order — is
 * the same function of the shape for every dtype (vectors are counted from x[0], i.e. as
 * for an fp32 x that starts on a 32-byte boundary), so a 16-bit x gives the statistics of
 * its fp32 copy bit for bit. */
int qsb_reduce_stats_dt(const void *x, int x_dtype, int what, int64_t outer, int64_t channels,
                        int64_t inner, float *absmax, float *mn, float *mx,
                        double *abssum, double *nnz, float *tensor_min,
                        void *workspace, int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * K4  tiny on-device parameter updates (no host sync).
 * ---------------------------------------------------------------------- */

/* ref: DecimalQuantizer.optimize qsparse/quantize.py:340,344-348
 *   new = absmax / 2^(bits-1);  t == 0: w = new;  else w = (t*w + new)/(t+1) */
int qsb_scale_ema(float *weight, const float *absmax, int64_t n, int bits,
                  int64_t t, void *stream);

/* ref: DecimalQuantizer.quantize qsparse/quantize.py:316
 *   d = round(log2(nan_to_num(1/s, posinf=1, neginf=1))) */
int qsb_scale_to_decimal(const float *scale, float *decimal, int64_t n,
                         void *stream);

/* ref: AdaptiveQuantizer.optimize qsparse/quantize.py:412-430
 *   lines[c] = (w[c]*(t-1) + (mn[c], mx[c])) / t       (t >= 1, after increment)
 * The min-of-mins / max-of-maxes over the batch (:415-418) is already folded
 * into qsb_reduce_stats by passing outer = batch. */
int qsb_lines_ema(float *lines, const float *mn, const float *mx,
                  int64_t channels, int64_t t, void *stream);

/* CUDA-graph forms of the two running means above (no reference counterpart: the
 * reference's step indices are Python ints, qsparse/quantize.py:340-348,426-430):
 * the index is *t_dev + t_offset, read by the kernel, because the launch arguments
 * of a captured graph are frozen.  The caller advances the counter (stream-ordered). */
int qsb_scale_ema_at(float *weight, const float *absmax, int64_t n, int bits,
                     const int64_t *t_dev, int64_t t_offset, void *stream);
int qsb_lines_ema_at(float *lines, const float *mn, const float *mx, int64_t channels,
                     const int64_t *t_dev, int64_t t_offset, void *stream);

/* ------------------------------------------------------------------------
 * K8  row-resident fused estimate + quantize for tensors quantized along their
 * LEADING axis (x is [rows][inner] contiguous, one parameter row per x row —
 * the `channelwise=0` weight case).  One launch, 8 B/elem, replaces
 *   QuantizeLayer.forward -> callback.optimize + callback.forward
 *   (qsparse/quantize.py:501-508) =
 *     kind 0 (Decimal): abs-max (:329-340) -> scale EMA (:344-348) ->
 *            decimal = round(log2(1/s)) (:316) -> pow2 fake-quant (:44-63)
 *     kind 1 (Scaler) : abs-max -> scale EMA -> scaler fake-quant (:100-117)
 *     kind 2 (Adaptive): min / max (:396-411) -> lines EMA (:428-430) ->
 *            line fake-quant (:148-181; float_zero_point as in qsb_fq_line_fwd)
 * param: float[rows][1] (scale) or float[rows][2] (lo, hi), updated IN PLACE
 * exactly like qsb_scale_ema / qsb_lines_ema would (t has the same meaning as
 * in those calls: 0-based for kinds 0/1, 1-based for kind 2).
 * decimal_out: float[rows] or NULL, kind 0 only (what the STE backward needs).
 * Results are bit-identical to qsb_reduce_stats + qsb_*_ema + qsb_fq_*_fwd.
 * Returns QSB_E_UNSUPPORTED when a row is not a whole number of 32-byte
 * vectors (inner % 8, pointer alignment) or longer than 16384 elements; the
 * caller then uses the three-kernel sequence above. */
int qsb_row_quant_fused(const float *x, float *y, float *param,
                        float *decimal_out, int kind, int bits,
                        int float_zero_point, int64_t rows, int64_t inner,
                        int64_t t, void *stream);

/* ref: MagnitudePruningCallback.update_magnitude qsparse/sparse.py:82-89 with a
 * reduced (structured) magnitude:  m = abssum / count  (or nnz / count when
 * use_l0 and *tensor_min == 0);  mag = (t*mag + m) / (t+1) */
/* The same with an element prune mask applied first — the weight chain quantize(prune(layer))
 * (ref qsparse/imitation.py:61-71) with a frozen mask: y = Q(x * mask), the row's parameter is
 * estimated on x * mask.  9 B/elem in one launch.  mask_dev: uint8 [rows * inner], 8-byte aligned. */
int qsb_row_quant_fused_masked(const float *x, float *y, float *param,
                               float *decimal_out, const uint8_t *mask_dev,
                               int kind, int bits, int float_zero_point,
                               int64_t rows, int64_t inner, int64_t t,
                               void *stream);
/* CUDA-graph form of qsb_row_quant_fused[_masked]: the EMA index is *t_dev + t_offset, read by
 * the kernel (mask_dev may be NULL); the caller advances the counter. */
int qsb_row_quant_fused_at(const float *x, float *y, float *param,
                           float *decimal_out, const uint8_t *mask_dev,
                           int kind, int bits, int float_zero_point,
                           int64_t rows, int64_t inner, const int64_t *t_dev,
                           int64_t t_offset, void *stream);

int qsb_magnitude_ema_reduced(float *magnitude, const double *abssum,
                              const double *nnz, const float *tensor_min,
                              int use_l0, int64_t channels, double count,
                              int64_t t, void *stream);

/* Same, full-size (unstructured) magnitude, fused with |x|:
 *   mag[i] = (t*mag[i] + |x[i]|) / (t+1)            12 B/elem.
 * use_l0 and *tensor_min == 0: |x| is replaced by (x != 0). */
int qsb_magnitude_ema_full(float *magnitude, const float *x,
                           const float *tensor_min, int use_l0, int64_t n,
                           int64_t t, void *stream);

/* Multi-tensor forms for a weight SET (BASELINE config 4): the same arithmetic as
 * qsb_magnitude_ema_full (without l0) / qsb_mask_build_apply on `count` separate
 * tensors in ONE launch; tensor i has n[i] elements, thr_dev[i] is its threshold.
 * The pointer / size arrays are HOST arrays.  Returns QSB_E_UNSUPPORTED when a
 * tensor is not 32-byte aligned (use the single-tensor calls then). */
int qsb_magnitude_ema_full_multi(float *const *magnitude, const float *const *x,
                                 const int64_t *n, int count, int64_t t,
                                 void *stream);
int qsb_mask_build_apply_multi(const float *const *importance, int take_abs,
                               const float *thr_dev, const float *const *x,
                               float *const *y, uint8_t *const *mask_out,
                               const int64_t *n, int count, void *stream);

/* One unstructured, running-average prune step of `count` tensors in ONE streaming pass
 * (17 B/elem instead of 12 + 4 + 13 = 29 for the three calls above), per tensor i:
 *   magnitude[i] = (t*magnitude[i] + |x[i]|) / (t+1)        ref qsparse/sparse.py:82-89
 *   thr[i]       = sort(magnitude[i])[k[i]]                 ref qsparse/util.py:113-116
 *   mask_out[i]  = magnitude[i] >= thr[i];  y[i] = x[i] * mask_out[i]   ref sparse.py:65-66
 * How: the sampler estimates, from 8 Ki of the magnitudes the EMA is about to produce, two
 * pivots that bracket the threshold and their midpoint; the streaming pass computes the
 * EMA, writes mask / y provisionally (>= midpoint), and records the ~4 % of elements
 * between the pivots with their positions; the select runs on those; a fix-up kernel
 * patches the few records whose provisional decision differs from the final one.  When
 * the pivots miss (decided on the device) the masks are rebuilt by a gated full pass.
 * Results are bit-identical to the three separate calls.  Host arrays of pointers /
 * sizes; QSB_E_UNSUPPORTED when a tensor is not 32-byte aligned. */
int64_t qsb_prune_step_workspace_bytes(const int64_t *n, int count);
int qsb_prune_unstructured_step_batched(float *const *magnitude,
                                        const float *const *x, float *const *y,
                                        uint8_t *const *mask_out, const int64_t *n,
                                        const int64_t *k, int count, int64_t t,
                                        float *thr_out_dev, void *workspace,
                                        int64_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------
 * K5  exact k-th value (ascending, 0-based rank k) by radix select on the
 * order-preserving uint32 key; NaNs order last (like torch.sort).
 * ref: calculate_mask_given_importance qsparse/util.py:113-116
 *      (values = sort(flat); threshold = values[idx + 1])
 * ---------------------------------------------------------------------- */
int64_t qsb_kth_workspace_bytes(int64_t n);
/* The same select over values SHARDED across GPUs (SURVEY 8(e), one monolithic
 * weight tensor split by element range): rank k_global is global, every GPU passes
 * its n_local values.  Protocol, identical on every rank, same workspace throughout:
 *   qsb_kth_dist_begin(ws)
 *   for pass in 0, 1, 2:
 *     qsb_kth_dist_pass(v, n_local, k_global, pass, ..., &hist, &count)
 *     all-reduce(SUM) the `count` 64-bit counters at `hist` over the ranks
 *     (e.g. ncclAllReduce ncclUint64 / torch.distributed on an int64 view)
 *   qsb_kth_dist_final(k_global, ws, thr_out)   -> the same threshold everywhere
 * Exact (integer histograms); 3 all-reduces of <= 32 KB.  The workspace is
 * qsb_kth_workspace_bytes(n_local) bytes.  replaces: the reference has no multi-GPU
 * path; equals calculate_mask_given_importance (qsparse/util.py:103-117) on the
 * concatenated tensor. */
int qsb_kth_dist_begin(void *workspace, int64_t workspace_bytes, void *stream);
int qsb_kth_dist_pass(const float *v, int64_t n_local, int64_t k_global,
                      int pass, int take_abs, void *workspace,
                      int64_t workspace_bytes, void **hist_out,
                      int64_t *hist_counters_out, void *stream);
int qsb_kth_dist_final(int64_t k_global, void *workspace, float *thr_out_dev,
                       void *stream);

/* take_abs != 0 selects on |v| (importance = x.abs() without materialising it,
 * running_average=False, qsparse/sparse.py:63-64). */
int qsb_kth_value(const float *v, int64_t n, int64_t k, int take_abs,
                  float *thr_out_dev, void *workspace, int64_t workspace_bytes,
                  void *stream);

/* `count` independent selects (the layers of a weight set, SURVEY 8d config 4) in one
 * launch sequence: v[i] has n[i] values, thr_out_dev[i] = its k[i]-th smallest.  The
 * pointer / size arrays are HOST arrays (read during the call).  Segments of >= 2^17
 * values take the sampled-pivot route together (blockIdx.y = segment), so 29 layers of
 * 2.4 M values cost about as much as one select over their total. */
int64_t qsb_kth_batched_workspace_bytes(const int64_t *n, int count);
int qsb_kth_value_batched(const float *const *v, const int64_t *n,
                          const int64_t *k, int count, int take_abs,
                          float *thr_out_dev, void *workspace,
                          int64_t workspace_bytes, void *stream);

/* ref: calculate_mask_given_importance qsparse/util.py:117  mask = imp >= thr */
/* Warm-started forms for training loops, which ask for the same order statistic of a slowly drifting
 * tensor every step.  hints_dev: count x 8 uint32 words owned by the caller, ZERO before the first
 * call and left alone between calls on the same tensors (reset them when a tensor or its rank k
 * changes abruptly, e.g. at a sparsity ramp point).  From the third call on the pivots are the previous
 * answer -/+ an adaptive delta instead of a 32 Ki-element sample: no sampler pass, a few thousand
 * candidates instead of ~2 % of n.  Results are exact whatever the hints contain (a bracket that misses
 * rank k takes the generic route on the device and widens). */
int qsb_kth_value_batched_hinted(const float *const *v, const int64_t *n,
                                 const int64_t *k, int count, int take_abs,
                                 float *thr_out_dev, uint32_t *hints_dev,
                                 void *workspace, int64_t workspace_bytes,
                                 void *stream);
int qsb_prune_unstructured_step_batched_hinted(
    float *const *magnitude, const float *const *x, float *const *y,
    uint8_t *const *mask_out, const int64_t *n, const int64_t *k, int count,
    int64_t t, float *thr_out_dev, uint32_t *hints_dev, void *workspace,
    int64_t workspace_bytes, void *stream);
/* CUDA-graph form: the EMA index is *t_dev + t_offset, read by the kernels (the launch
 * arguments of a captured graph are frozen); hints_dev may be NULL.  The caller advances
 * the counter. */
int qsb_prune_unstructured_step_batched_at(
    float *const *magnitude, const float *const *x, float *const *y,
    uint8_t *const *mask_out, const int64_t *n, const int64_t *k, int count,
    const int64_t *t_dev, int64_t t_offset, float *thr_out_dev,
    uint32_t *hints_dev, void *workspace, int64_t workspace_bytes, void *stream);

int qsb_mask_from_threshold(const float *importance, int take_abs,
                            const float *thr_dev, uint8_t *mask_out, int64_t n,
                            void *stream);

/* Fused unstructured mask build + apply (13 B/elem; 9 when importance aliases
 * x with take_abs, i.e. running_average=False):
 *   mask = imp >= thr;  y = x * mask           ref: qsparse/sparse.py:65-66 */
int qsb_mask_build_apply(const float *importance, int take_abs,
                         const float *thr_dev, const float *x, float *y,
                         uint8_t *mask_out, int64_t n, void *stream);

/* ref: DecimalQuantizer.forward group-wise sharing  qsparse/quantize.py:361-366
 *   out[c, :] = mean over {c' : labels[c'] == labels[c]} of values[c', :]
 * values / out: float [channels, weight_size] (may alias), labels: int64 [channels] in [0, groups).
 * One launch instead of a host loop over the groups; the mean is the correctly rounded one. */
int qsb_group_mean(const float *values, const int64_t *labels, float *out,
                   int64_t channels, int64_t weight_size, int64_t groups,
                   void *stream);

/* ------------------------------------------------------------------------
 * Fused structured prune -> pow2 quantize parameter step: everything the
 * reference does between "statistics are reduced" and "apply" for
 *   Sequential(PruneLayer(dimensions={channel}), QuantizeLayer(channelwise=-1))
 * in one tiny kernel, on device:
 *   magnitude EMA (sparse.py:89) -> threshold = sorted(mag)[k] (util.py:113-116)
 *   -> mask = mag >= thr (util.py:117) -> absmax of kept channels
 *   (= max |x*mask|, quantize.py:329-340) -> scale EMA (quantize.py:344-348)
 *   -> decimal (quantize.py:316).
 * refresh_mask == 0 keeps the existing mask (sparse.py:115-116).
 * update_scale == 0 skips the quantizer's optimize (eval / before timeout).
 * update_magnitude: 0 keep, 1 running average, 2 importance = this step's
 * mean |x| (running_average=False, sparse.py:63-64).
 * The statistics may come as n_stat_rows rows (one per rank after an
 * all-gather, or one per staged chunk of a host tensor), stat_row_stride_bytes
 * apart; they are combined in row order: SUM for abssum, MAX for absmax.
 * `count` is the number of elements per channel over ALL rows.
 * Requires 1 <= channels <= 4096 and 1 <= n_stat_rows <= 4096.  abssum may be
 * NULL, and `count` is not checked, when update_magnitude == 0; absmax may be
 * NULL when update_scale == 0.  Runs the one-CTA kernel of
 * qsb_prune_quant_rows_step_params with group == NULL.
 * ---------------------------------------------------------------------- */
int qsb_prune_quant_params(float *magnitude, uint8_t *mask, float *scale,
                           float *decimal_out, const double *abssum,
                           const float *absmax, int64_t n_stat_rows,
                           int64_t stat_row_stride_bytes, int64_t channels,
                           double count,
                           int64_t t_prune, int update_magnitude,
                           int refresh_mask, int64_t k, int bits,
                           int64_t t_quant, int update_scale, void *stream);

/* ------------------------------------------------------------------------
 * The same parameter step as ONE kernel that also finalizes the reduction and,
 * across GPUs, exchanges the statistics row over peer memory (NVLink) — the
 * fused compute + collective form of the training step:
 *   qsb_reduce_partials(x)           stage 1 only, partials stay in the workspace
 *   qsb_prune_quant_step_params(...) finalize -> push my [C x fp64 sum | C x max]
 *       row into every peer's exchange buffer + stamp -> wait for all stamps ->
 *       combine in rank order -> EMA / threshold / mask / scale / decimal
 *   qsb_fq_pow2_fwd(mask), qsb_ste_bwd(mask)
 * group == NULL: single GPU.  step_stamp must be > 0, equal on all ranks and
 * increase by one per step (two slots are used alternately).  `count` is the
 * number of elements per channel over ALL ranks.  abssum_out / absmax_out
 * (optional, both or neither) receive the combined statistics.
 * Requires channels <= 4096 and the same (outer, channels, inner) that was
 * passed to qsb_reduce_partials.
 * step_counter_dev (optional): a device int64 step index for CUDA-graph capture
 * (launch arguments of a captured graph are frozen).  When given, with t =
 * *step_counter_dev the kernel uses t_prune = t + <the t_prune argument> and
 * t_quant = t + <the t_quant argument> (the arguments become OFFSETS: a prune
 * callback and a quantizer that started at different steps keep a constant
 * distance; pass 0 for both to index everything by the counter itself),
 * step_stamp = t + 1, treats refresh_mask as the refresh INTERVAL (refresh when
 * t_prune % interval == 0 and (t_prune > 0 or update_magnitude == 2)) and stores
 * t + 1 into the counter at the end.
 * ---------------------------------------------------------------------- */
int qsb_reduce_partials(const float *x, int64_t outer, int64_t channels,
                        int64_t inner, void *workspace, int64_t workspace_bytes,
                        void *stream);
/* x of element type x_dtype (QSB_DTYPE_*); plan and summation order as qsb_reduce_stats_dt. */
int qsb_reduce_partials_dt(const void *x, int x_dtype, int64_t outer, int64_t channels,
                           int64_t inner, void *workspace, int64_t workspace_bytes,
                           void *stream);

typedef struct qsb_p2p_group qsb_p2p_group;
/* exchange-buffer size for `world` ranks (<= 16) and `channels` channels */
int64_t qsb_p2p_group_bytes(int world, int64_t channels);
/* cudaMalloc'ed, zeroed buffer + its 64-byte CUDA IPC handle (send it to the peers) */
int qsb_p2p_alloc(int64_t bytes, void **dev_ptr, unsigned char *handle64);
int qsb_p2p_open(const unsigned char *handle64, void **peer_ptr);
int qsb_p2p_close(void *peer_ptr);
int qsb_p2p_free(void *dev_ptr);
/* bufs[r] = rank r's exchange buffer as mapped in THIS process (bufs[rank] local) */
int qsb_p2p_group_create(qsb_p2p_group **out, int rank, int world,
                         int64_t channels, void *const *bufs);
/* *error_out != 0 if a peer's statistics did not arrive within the timeout (synchronises).
 * A step that timed out does NOT continue on stale data: it writes NaN into scale / decimal /
 * magnitude (every later output of the layer is NaN) and raises this flag. */
int qsb_p2p_group_error(qsb_p2p_group *group, int *error_out);
/* the same without synchronising: the copy into *error_out_pinned (pinned host memory) is
 * ordered after the work already queued on `stream`. */
int qsb_p2p_group_error_async(qsb_p2p_group *group, int *error_out_pinned, void *stream);
/* how long a step waits for its peers before it poisons itself (default 30 000 ms) */
int qsb_p2p_group_set_timeout_ms(qsb_p2p_group *group, int64_t timeout_ms);
int qsb_p2p_group_destroy(qsb_p2p_group *group);

int qsb_prune_quant_step_params(float *magnitude, uint8_t *mask, float *scale,
                                float *decimal_out, void *reduce_workspace,
                                int64_t workspace_bytes, int64_t outer,
                                int64_t channels, int64_t inner,
                                qsb_p2p_group *group, int64_t step_stamp,
                                double count, int64_t t_prune,
                                int update_magnitude, int refresh_mask,
                                int64_t k, int bits, int64_t t_quant,
                                int update_scale, double *abssum_out,
                                float *absmax_out, int64_t *step_counter_dev,
                                void *stream);

/* The same parameter step on FINALIZED statistics rows (as qsb_prune_quant_params takes
 * them: one row per staged chunk, combined in row order) with the peer exchange of
 * qsb_prune_quant_step_params — what the host-buffer pipeline runs.  Requires
 * channels <= 4096, 1 <= n_stat_rows <= 4096 and both statistics pointers.
 * `count` is the number of elements per channel over ALL ranks. */
int qsb_prune_quant_rows_step_params(float *magnitude, uint8_t *mask, float *scale,
                                     float *decimal_out, const double *abssum,
                                     const float *absmax, int64_t n_stat_rows,
                                     int64_t stat_row_stride_bytes, int64_t channels,
                                     qsb_p2p_group *group, int64_t step_stamp,
                                     double count, int64_t t_prune,
                                     int update_magnitude, int refresh_mask,
                                     int64_t k, int bits, int64_t t_quant,
                                     int update_scale, void *stream);

/* ------------------------------------------------------------------------
 * The training step's "everything before apply" as ONE launch (the default route):
 * the stage-1 reduction of sum|x| / max|x| over x [outer, channels, inner] whose
 * LAST-ARRIVING CTA runs the parameter step of qsb_prune_quant_step_params as the
 * kernel's tail (finalize -> peer exchange -> magnitude EMA -> threshold -> mask ->
 * scale EMA -> decimal).  No single-CTA launch, no host sync; across GPUs the peer
 * exchange starts the moment this GPU's statistics are complete.
 * ref: sparse.py:58-66,82-89 + util.py:79-117 + quantize.py:316,329-348 in one launch.
 * workspace: qsb_reduce_workspace_bytes(outer, channels, inner).
 * arrival_counter_dev: one device uint32 owned by the caller, ZERO before the first use;
 * the kernel leaves it zero (one counter per stream that may run this concurrently).
 * stats_local != 0: abssum_out / absmax_out receive THIS rank's statistics row (before
 * the exchange) instead of the combined one.  Other arguments as in
 * qsb_prune_quant_step_params.  Requires channels <= 1024.
 * timing_out_dev (optional, 8 x uint64): %globaltimer stamps in ns — [0] earliest CTA start
 * (atomicMin: set it to UINT64_MAX before the launch), [1] the last-arriving CTA enters the
 * parameter step, [2] statistics finalized, [3] peer exchange done, [4] magnitude EMA done,
 * [5] threshold found, [6] scale / decimal written.  bench.py reports the phases from it. */
int qsb_reduce_prune_quant_step(const float *x, int64_t outer, int64_t channels,
                                int64_t inner, void *workspace,
                                int64_t workspace_bytes,
                                unsigned int *arrival_counter_dev,
                                float *magnitude, uint8_t *mask, float *scale,
                                float *decimal_out, qsb_p2p_group *group,
                                int64_t step_stamp, double count, int64_t t_prune,
                                int update_magnitude, int refresh_mask, int64_t k,
                                int bits, int64_t t_quant, int update_scale,
                                double *abssum_out, float *absmax_out,
                                int stats_local, int64_t *step_counter_dev,
                                uint64_t *timing_out_dev, void *stream);
/* x of element type x_dtype (QSB_DTYPE_*); plan and summation order as qsb_reduce_stats_dt. */
int qsb_reduce_prune_quant_step_dt(const void *x, int x_dtype, int64_t outer, int64_t channels,
                                   int64_t inner, void *workspace,
                                   int64_t workspace_bytes,
                                   unsigned int *arrival_counter_dev,
                                   float *magnitude, uint8_t *mask, float *scale,
                                   float *decimal_out, qsb_p2p_group *group,
                                   int64_t step_stamp, double count, int64_t t_prune,
                                   int update_magnitude, int refresh_mask, int64_t k,
                                   int bits, int64_t t_quant, int update_scale,
                                   double *abssum_out, float *absmax_out,
                                   int stats_local, int64_t *step_counter_dev,
                                   uint64_t *timing_out_dev, void *stream);

/* ------------------------------------------------------------------------
 * The line form of the structured prune -> quantize step, for an AdaptiveQuantizer
 * (ref sparse.py:58-66,82-89 + util.py:79-117 + quantize.py:396-430): the same
 * statistics reduction, finalize, magnitude EMA, threshold and mask as
 * qsb_reduce_prune_quant_step (same plan, same summation order of sum|x|), then
 * in place of abs-max -> scale -> decimal the (min, max) of x * mask and the
 * lines EMA  lines = (lines * (t - 1) + new) / t  at the quantizer's 1-based call
 * index t = t_line (t = 1 writes `new`, as qsb_lines_ema does).  A pruned channel
 * adds min / max of x * 0: +-0 (the sign that min / max of the fp32 output of
 * qsb_mask_apply_dt has), or NaN when it holds an inf or a NaN.
 *   lines [n_lines, 2] (lo, hi): n_lines == 1 takes the NaN-propagating min / max
 *   over all channels (per tensor), n_lines == channels each channel's own pair.
 * Then qsb_fq_line_fwd_dt(mask, float_zero_point = 1) and qsb_mask_apply_dt(g).
 * abssum_out / min_out / max_out (optional, each may be NULL) receive this step's
 * sum|x|, min x and max x per channel (of x, not of x * mask).
 * step_counter_dev (optional) as in qsb_prune_quant_step_params; the call index is
 * then *step_counter_dev + t_line (t_line an offset) and the kernel advances the
 * counter.  Without it t_line must be >= 1.
 * Returns QSB_E_BADARG before any CUDA call for NULL x / workspace / arrival
 * counter / mask / lines, n_lines not 1 or channels, t_line < 1 without a counter,
 * k outside [0, channels) on a refresh, a bad update_magnitude or count, or any
 * group (the line form runs on one GPU: group must be NULL).
 *
 * qsb_reduce_prune_line_step_dt: ONE launch (as qsb_reduce_prune_quant_step_dt,
 * also its three-launch form for wide column-mode tensors).  Requires channels <=
 * 1024 (QSB_E_UNSUPPORTED above).  No L2 residency hint: the line forward reads
 * the pruned channels too.
 * ---------------------------------------------------------------------- */
int qsb_reduce_prune_line_step_dt(const void *x, int x_dtype, int64_t outer, int64_t channels,
                                  int64_t inner, void *workspace, int64_t workspace_bytes,
                                  unsigned int *arrival_counter_dev, float *magnitude,
                                  uint8_t *mask, float *lines, int64_t n_lines,
                                  qsb_p2p_group *group, double count, int64_t t_prune,
                                  int update_magnitude, int refresh_mask, int64_t k,
                                  int64_t t_line, double *abssum_out, float *min_out,
                                  float *max_out, int64_t *step_counter_dev, void *stream);
/* Stage 1 of sum|x| and min / max x only (plan and summation order as qsb_reduce_partials_dt);
 * the partials stay in the workspace for qsb_prune_line_step_params. */
int qsb_reduce_line_partials_dt(const void *x, int x_dtype, int64_t outer, int64_t channels,
                                int64_t inner, void *workspace, int64_t workspace_bytes,
                                void *stream);
/* The line step as a one-CTA launch on the partials of qsb_reduce_line_partials_dt (same
 * outer, channels, inner).  Requires channels <= 2048 (QSB_E_UNSUPPORTED above). */
int qsb_prune_line_step_params(float *magnitude, uint8_t *mask, float *lines, int64_t n_lines,
                               void *reduce_workspace, int64_t workspace_bytes, int64_t outer,
                               int64_t channels, int64_t inner, qsb_p2p_group *group,
                               double count, int64_t t_prune, int update_magnitude,
                               int refresh_mask, int64_t k, int64_t t_line,
                               double *abssum_out, float *min_out, float *max_out,
                               int64_t *step_counter_dev, void *stream);

/* ------------------------------------------------------------------------
 * Host-buffer entry points (what a host-side caller that keeps its tensors in
 * CPU memory binds to).  They stage through pinned memory owned by a context,
 * pipeline H2D / kernels / D2H over chunks on several streams, and return after
 * the results are in the host buffers.
 * ---------------------------------------------------------------------- */
typedef struct qsb_host_ctx qsb_host_ctx;
/* The context owns two slots of device staging buffers (4 tensors of max_elems
 * floats each), three streams (upload / compute / download) and per-chunk events. */
int qsb_host_ctx_create(qsb_host_ctx **out, int64_t max_elems,
                        int64_t max_channels, int n_chunks);
int qsb_host_ctx_destroy(qsb_host_ctx *ctx);

/* One fused training step of prune(dimensions={channel}) -> pow2 quantize on
 * HOST tensors (config 2 of BASELINE.json): forward y = Q(x*mask) with this
 * step's statistics (magnitude EMA at step t_prune, mask refresh when
 * t_prune > 0 with threshold rank k, scale EMA at step t_quant), backward
 * gx = clamp(g)*mask.  The layer state (magnitude[C], mask[C], scale[1],
 * decimal[1]) lives on the device in caller-provided buffers.  Host buffers
 * should be pinned.  Work is ordered after caller_stream; the call returns when
 * y_host and gx_host are complete.
 * group (optional, NULL = one GPU): the batch is sharded over the ranks of the group; the
 * chunk statistics are exchanged with the peers (step_stamp as in
 * qsb_prune_quant_step_params) so every rank derives the parameters of the concatenated batch.
 * ref: PruneLayer.forward sparse.py:215-273 -> QuantizeLayer.forward
 * quantize.py:473-518 and their backward passes. */
int qsb_host_prune_quant_step(qsb_host_ctx *ctx, const float *x_host,
                              const float *g_host, float *y_host,
                              float *gx_host, float *magnitude_dev,
                              uint8_t *mask_dev, float *scale_dev,
                              float *decimal_dev, int64_t outer,
                              int64_t channels, int64_t inner, int64_t t_prune,
                              int64_t k, int bits, int64_t t_quant,
                              qsb_p2p_group *group, int64_t step_stamp,
                              void *caller_stream);

/* The same step, asynchronous: enqueue everything for `slot` (0 or 1) and return.
 * Two steps may be in flight, one per slot — the upload of step t+1 then overlaps
 * the download of step t (PCIe is full duplex), and the steady state costs 2
 * transfers per direction per step instead of 3 serial ones.  Steps are applied to
 * the layer state in submission order.  Each slot needs its own four host buffers;
 * qsb_host_ctx_wait(ctx, slot) returns when that slot's y_host / gx_host are
 * complete (submitting to a busy slot waits for it first).
 * Returns its code before any CUDA call (no wait, no copy, no launch) for a NULL
 * ctx / host buffer / magnitude / mask / scale / decimal, a slot other than 0 or 1,
 * a zero or negative dimension, more channels or elements than the context was
 * created for, k outside [0, channels) when t_prune > 0, or a group whose channel
 * count differs (QSB_E_BADARG), and for channels > 4096 (QSB_E_UNSUPPORTED). */
int qsb_host_prune_quant_step_submit(qsb_host_ctx *ctx, int slot,
                                     const float *x_host, const float *g_host,
                                     float *y_host, float *gx_host,
                                     float *magnitude_dev, uint8_t *mask_dev,
                                     float *scale_dev, float *decimal_dev,
                                     int64_t outer, int64_t channels,
                                     int64_t inner, int64_t t_prune, int64_t k,
                                     int bits, int64_t t_quant,
                                     qsb_p2p_group *group, int64_t step_stamp,
                                     void *caller_stream);
int qsb_host_ctx_wait(qsb_host_ctx *ctx, int slot);

#ifdef __cplusplus
}
#endif
#endif /* QSPARSE_B200_H_ */
