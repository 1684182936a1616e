// Row-wise fused kernels shared by the GraphDiT and GIN paths (HBM-bound; one warp per row).  Each launcher issues at most one
// kernel (none for rows <= 0) and counts it on ctr, which may be null.
#pragma once
#include "llb_common.cuh"

namespace llb {

// out = resid + gate[g] * act( LN(in) * gamma + beta  ->  * (1 + scale[g]) + shift[g] ) + addvec[g]
// every stage optional; g = row_group[row] (or row).  Writes fp32 and/or bf16, optionally a second copy
// `dup_rows` rows further down (the unconditional half of the CFG batch shares the token embedding).
struct RowLnArgs {
  const void* in = nullptr;
  int in_ld = 0;
  bool in_bf16 = false;
  int in_parts = 1;          // the input row is the sum of in_parts pieces, in_part_stride elements apart (split-K partials),
  int in_part_stride = 0;    // added in index order
  int rows = 0, width = 0;
  int valid = 0;             // columns that carry data (0 = width): the statistics cover [0, valid), columns [valid, width) are
                             // written as 0 (zero-padded operands of a wider internal width)
  bool normalize = true;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  const int32_t* row_group = nullptr;
  const float* shift = nullptr;
  const float* scale = nullptr;
  const float* gate = nullptr;
  int mod_ld = 0;
  int act = LLB_ACT_NONE;
  const float* resid = nullptr;
  int resid_ld = 0;
  const float* addvec = nullptr;  // (groups, width) fp32, added last
  int addvec_ld = 0;
  float* out_f32 = nullptr;
  int out_f32_ld = 0;
  __nv_bfloat16* out_bf16 = nullptr;
  int out_bf16_ld = 0;
  int dup_rows = 0;
  bool l2_normalize = false;  // out = v / ||v|| instead of LN (GraphCLIP head)
  int prof_slot = LLB_PROF_LN_MOD_RES;
};
int launch_row_ln(const RowLnArgs& a, cudaStream_t stream, LaunchCounter* ctr);

// Backward of the row LayerNorm above without residual / addvec (they pass the gradient through unchanged): with
//   xh = LN(x) over the first `valid` columns,  t = xh * gamma + beta  or  xh * (1 + scale[g]) + shift[g],  out = gate[g] * act(t),
// and dy = dL/d(out), writes dx = dL/dx (bf16 and/or fp32, 0 in the padded columns; the fp32 copy may overwrite dy in place)
// and, when `prod` is set, the per-row products whose per-group sums are the gradients of [shift | scale | gate] (or, summed
// over all rows, of [beta | gamma]): [dt | dt * xh | dy * act(t)] at columns 0, width, 2 width (the first prod_sets of them).
// act is GELU (exact derivative of the erf form) or none.  One warp per row, sums in a fixed order: run-to-run deterministic.
struct RowLnBwdArgs {
  const void* x = nullptr;   // the forward's LayerNorm input
  int x_ld = 0;
  bool x_bf16 = false;
  const float* dy = nullptr;
  int dy_ld = 0;
  int dy_parts = 1;          // dy is the sum of dy_parts pieces, dy_part_stride elements apart (split-K partials), added in index order
  int dy_part_stride = 0;
  int rows = 0, width = 0, valid = 0;
  const float* gamma = nullptr;
  const float* beta = nullptr;
  const int32_t* row_group = nullptr;
  const float* shift = nullptr;
  const float* scale = nullptr;
  const float* gate = nullptr;
  int mod_ld = 0;
  bool gelu = false;
  float* prod = nullptr;
  int prod_ld = 0;
  int prod_sets = 3;
  __nv_bfloat16* out_bf16 = nullptr;
  int out_ld = 0;
  float* out_f32 = nullptr;   // row stride out_ld as well
  int prof_slot = LLB_PROF_GIN_ROWLN;
};
int launch_row_ln_bwd(const RowLnBwdArgs& a, cudaStream_t stream, LaunchCounter* ctr);

// fp32 (rows, cols) -> bf16 (rows, dst_ld) with zero padding up to pad_cols.
int launch_f32_to_bf16(const float* src, int src_ld, __nv_bfloat16* dst, int dst_ld, int rows, int cols, int pad_cols,
                       cudaStream_t stream, LaunchCounter* ctr);
// out[r, o] = act(sum_k in[r,k] W[o,k] + b[o]) in fp32 on CUDA cores (tiny set-up linears only).
int launch_linear_f32(const float* in, int in_ld, const float* W, int w_ld, const float* b, float* out, int out_ld,
                      int rows, int out_f, int in_f, int act, cudaStream_t stream, LaunchCounter* ctr);

}  // namespace llb
