// Kernels shared by the backward passes (llb_gin_grad.cu, llb_dit_grad.cu).
#pragma once
#include "llb_common.cuh"

namespace llb {
namespace {

__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
__device__ __forceinline__ float to_f32(__half v) { return __half2float(v); }
__device__ __forceinline__ float to_f32(float v) { return v; }

// dst (cols, rows_out) bf16 with row stride ld_d  <-  src (rows, cols) with row stride ld_s, zero in dst columns [rows, rows_out)
// (the K padding of a split-K product); 32 x 32 tiles through shared memory, grid (ceil(cols/32), ceil(rows_out/32))
template <class T>
__global__ void __launch_bounds__(256) grad_transpose_kernel(const T* __restrict__ src, int ld_s, int rows, int cols,
                                                             __nv_bfloat16* __restrict__ dst, int ld_d, int rows_out) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32, tx = threadIdx.x, ty = threadIdx.y;
  for (int k = ty; k < 32; k += 8) {
    const int r = r0 + k, c = c0 + tx;
    tile[k][tx] = (r < rows && c < cols) ? to_f32(src[(size_t)r * ld_s + c]) : 0.f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int c = c0 + k, r = r0 + tx;
    if (c < cols && r < rows_out) dst[(size_t)c * ld_d + r] = __float2bfloat16(tile[tx][k]);
  }
}

// Per-segment sums over contiguous row ranges (graphs, molecules), in row order: out[g] = add[g] + sum_{i in g} in[i] (fp32
// and/or bf16 out; add may alias out_f32).  grid (B, ceil(W/256)).
__global__ void __launch_bounds__(256) grad_segsum_kernel(const float* __restrict__ in, int in_ld, const int32_t* __restrict__ graph_ptr,
                                                          int W, const float* add, float* out_f32, __nv_bfloat16* __restrict__ out_bf16,
                                                          int out_ld) {
  const int g = blockIdx.x;
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= W) return;
  float acc = 0.f;
  for (int i = graph_ptr[g], end = graph_ptr[g + 1]; i < end; ++i) acc += in[(size_t)i * in_ld + c];
  if (add) acc += add[(size_t)g * out_ld + c];
  if (out_f32) out_f32[(size_t)g * out_ld + c] = acc;
  if (out_bf16) out_bf16[(size_t)g * out_ld + c] = __float2bfloat16(acc);
}

}  // namespace
}  // namespace llb
