// Internals of the two-stage reductions shared between reduce.cu (stage 1 + the
// stand-alone finalize) and params.cu (the fused finalize + exchange + parameter kernel).
#pragma once
#include "qsb_common.cuh"

namespace qsb {

struct Partials {
  uint32_t *amax;  // bits of max |x|  (NaN bit patterns order above inf)
  float *mn;
  float *mx;
  double *asum;
  double *nnz;
};

struct ReducePlan {
  bool row_mode;
  int64_t rows, seg, segs_per_row, vwarps;       // row mode
  int tile_spans, tile_span_stride;  // tile kernel: pieces per CTA visit, floats between them in shared memory
  int row_variant;  // row mode: 0 = 4 loads in flight per lane, 4 CTAs / SM; 2 = 8 loads, 2 CTAs / SM
  int cta_combine;  // row mode, one channel: a CTA writes one partial for its 8 warps
  int tile_rows;  // > 0: short rows, the tile kernel (tile_rows consecutive rows per CTA visit)
  int64_t nrows, ncols, chunks, rows_per_chunk;  // column mode
  int vcol;
  int tpr;  // column mode: threads of a CTA along a row (the CTA's other 256 / tpr row lanes interleave rows)
  // channel c combines entries j = 0..fin_count-1 at
  //   idx(j) = (j / fin_q) * (channels * fin_q) + c * fin_q + (j % fin_q)
  int64_t n_partials, fin_count, fin_q;
};

int64_t reduce_seg_min();
void set_reduce_seg_min(int v);
void set_reduce_col_tpr_wide(int v);
void set_reduce_row_variant(int v);
void set_reduce_keep_hint(int v);
void set_reduce_col_max_inner(int v);
// x (element size x_bytes) only decides the column kernel's vector width; the plan's partial layout and
// summation order depend on the shape alone
ReducePlan make_plan(int64_t outer, int64_t channels, int64_t inner, const void *x, int x_bytes = 4);
int64_t partial_bytes(int64_t n);
// carve the five partial arrays out of a caller workspace (256-byte aligned)
Partials partials_from_workspace(void *workspace, int64_t n_partials);

}  // namespace qsb
