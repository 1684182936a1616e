// GIN message passing: GraphCLIP encoder and GNNRetrosynthsizer predictor.
// Reference: graph_encoder/model.py:37-41,124-205; graph_predictor/model.py:306-353,387-423.
//
// Data layout in HBM: nodes are rows of (n,H) matrices -- h (fp32 master: residual, self term, pooling) and hb
// (bf16 copy: the gather source of the aggregation and nothing else).  Edges are a destination-sorted CSR
// (rowptr/col/etype), graphs are contiguous node ranges (graph_ptr), so every reduction (neighbour sum,
// per-graph max / sum pooling) is a segmented loop with no atomics.
#include <math.h>
#include <stdlib.h>

#include "llb_gemm_ln.cuh"
#include "llb_gin.cuh"
#include "llb_rowops.cuh"

namespace llb {
namespace {

constexpr int ATOM_VOCAB = 118;
constexpr int BOND_VOCAB = 5;
constexpr int HEAD_FUSED_MIN_WIDTH = 16384;   // fused head + softmax + top-k from this many templates on ...
constexpr int HEAD_FUSED_MIN_ROWS = 512;      // ... and this many graphs (below: materialise the few logit rows, no host sync)
constexpr int HEAD_PILOT_COLS = 4096;         // strided sample of the templates that fixes each row's threshold
constexpr int HEAD_CAND_CAP = 2048;           // candidates above the threshold kept per row
constexpr int HEAD_ROW_CHUNK = 8192;          // rows per fused pass: 50 MB of head inputs stay L2-resident while the weight streams once

}  // namespace

int make_layout(const llb_gin_config& c, GinLayout& G) {
  LLB_CHECK_ARG(c.hidden > 0, "gin: hidden=%d must be positive", c.hidden);
  LLB_CHECK_ARG(c.layers >= 2, "gin: layers=%d must be >= 2 (reference raises ValueError too)", c.layers);
  LLB_CHECK_ARG(!c.predictor || (c.out_dim >= 1 && c.text_dim > 0 && c.text_dim % 8 == 0), "gin: bad predictor out_dim/text_dim");
  G.H = c.hidden, G.L = c.layers, G.predictor = c.predictor ? 1 : 0, G.out_dim = c.out_dim, G.tdim = c.text_dim;
  G.Hp = (int)align_up(G.H, 64), G.I = (int)align_up(4 * (size_t)G.H, 64);
  G.HH = G.predictor ? G.I : G.Hp;
  G.HHt = G.predictor ? 4 * G.H : G.H;
  G.HO = G.predictor ? G.out_dim : G.Hp;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    off = align_up(off, 256);
    size_t o = off;
    off += bytes;
    return o;
  };
  const size_t H = G.Hp, I = G.I;
  for (int l = 0; l < G.L; ++l) {
    G.mlp0_w.push_back(take(I * H * 2));
    G.mlp4_w.push_back(take(I * H * 2));
    G.mlp_chol.push_back(take(H * H * 2));
    if (l < G.L - 1) {
      G.vn0_w.push_back(take(I * H * 2));
      G.vn4_w.push_back(take(I * H * 2));
    }
    if (G.predictor) G.adapter_w.push_back(take(3 * H * (size_t)G.tdim * 2));
  }
  G.head0_w = take((size_t)G.HH * H * 2);
  G.head4_w = take((size_t)G.HO * G.HH * 2);
  G.atom_emb = take(ATOM_VOCAB * H * 4);
  G.vn_emb = take(H * 4);
  G.text_drop = take((size_t)(G.predictor ? G.tdim : 1) * 4);
  for (int l = 0; l < G.L; ++l) {
    G.eps.push_back(take(4));
    G.mlp0_b.push_back(take(I * 4)), G.mlp_ln_w.push_back(take(I * 4)), G.mlp_ln_b.push_back(take(I * 4));
    G.mlp4_b.push_back(take(H * 4));
    G.mlp_stat.push_back(take((H + 4) * 4));
    G.mlp_bg.push_back(take(I * 4));
    G.bond_emb.push_back(take(BOND_VOCAB * H * 4));
    G.norm_w.push_back(take(H * 4)), G.norm_b.push_back(take(H * 4));
    if (l < G.L - 1) {
      G.vn0_b.push_back(take(I * 4)), G.vn_ln_w.push_back(take(I * 4)), G.vn_ln_b.push_back(take(I * 4));
      G.vn4_b.push_back(take(H * 4));
    }
    if (G.predictor) G.adapter_b.push_back(take(3 * H * 4));
  }
  G.head0_b = take((size_t)G.HH * 4), G.head_ln_w = take((size_t)G.HH * 4), G.head_ln_b = take((size_t)G.HH * 4);
  G.head4_b = take((size_t)G.HO * 4);
  // fused head + top-k (wide predictor heads only): a strided sample of the templates gives every row its threshold
  G.pilot_cols = (G.predictor && G.out_dim >= HEAD_FUSED_MIN_WIDTH) ? HEAD_PILOT_COLS : 0;
  G.pilot_stride = G.pilot_cols ? G.out_dim / G.pilot_cols : 0;
  G.pilot_w = take((size_t)G.pilot_cols * G.HH * 2), G.pilot_b = take((size_t)G.pilot_cols * 4);
  G.chol_scratch = take(((size_t)G.H + 1) * (G.H + 1) * 8);
  G.total = align_up(off, 256);
  return LLB_OK;
}

namespace {

// ---------------------------------------------------------------------------------------------
// Graph preparation
// ---------------------------------------------------------------------------------------------
// Input defects are recorded in a flag word (llb_gin_input_flags) and made harmless here: ids are clamped, a graph id outside
// [0, B) or a descending `batch` never indexes outside graph_ptr[0..B].  The reference raises an index error for the same inputs
// (nn.Embedding / scatter); the Python classes turn a non-zero flag word into that error.
__global__ void gin_prep_nodes_kernel(const int64_t* __restrict__ x, const int64_t* __restrict__ batch, int32_t* __restrict__ x32,
                                      int32_t* __restrict__ batch32, int32_t* __restrict__ graph_ptr, int32_t* __restrict__ flags, int n,
                                      int B) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const long long xv = x[i];
  if (xv < 0 || xv >= ATOM_VOCAB) atomicOr(flags, LLB_GIN_BAD_ATOM_ID);
  x32[i] = xv < 0 ? 0 : (xv >= ATOM_VOCAB ? ATOM_VOCAB - 1 : (int)xv);
  const long long gl = batch[i];
  const long long pl = i == 0 ? -1 : batch[i - 1];
  if (gl < 0 || gl >= B || gl < pl) atomicOr(flags, LLB_GIN_BAD_BATCH);
  const int g = gl < 0 ? 0 : (gl >= B ? B - 1 : (int)gl);
  const int prev = pl < -1 ? -1 : (pl >= B ? B - 1 : (int)pl);
  batch32[i] = g;
  for (int k = prev + 1; k <= g; ++k) graph_ptr[k] = i;   // first node of graph k (empty graphs collapse onto i); k <= g < B
  if (i == n - 1)
    for (int k = g + 1; k <= B; ++k) graph_ptr[k] = n;
}

__global__ void gin_degree_kernel(const int64_t* __restrict__ edge_index, const int64_t* __restrict__ edge_attr, int32_t* __restrict__ deg,
                                  int32_t* __restrict__ flags, int e, int n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= e) return;
  const long long src = edge_index[k], dst = edge_index[(size_t)e + k], a = edge_attr[k];
  if (src < 0 || src >= n || dst < 0 || dst >= n) atomicOr(flags, LLB_GIN_BAD_EDGE);
  if (a < 0 || a >= BOND_VOCAB) atomicOr(flags, LLB_GIN_BAD_BOND_ID);
  if (dst >= 0 && dst < n) atomicAdd(&deg[(int)dst], 1);
}

// Exclusive scan in three phases (block sums of 1024 elements).
__global__ void __launch_bounds__(1024) scan_block_kernel(const int32_t* __restrict__ in, int32_t* __restrict__ out,
                                                          int32_t* __restrict__ block_sums, int n) {
  __shared__ int32_t wsum[32];
  const int i = blockIdx.x * 1024 + threadIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int v = i < n ? in[i] : 0;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = wsum[lane];
    int wi = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, wi, o);
      if (lane >= o) wi += t;
    }
    wsum[lane] = wi - w;
    if (lane == 31 && block_sums) block_sums[blockIdx.x] = wi;
  }
  __syncthreads();
  if (i < n) out[i] = incl - v + wsum[warp];
}
__global__ void scan_add_kernel(int32_t* __restrict__ out, const int32_t* __restrict__ block_offs, int n) {
  const int i = blockIdx.x * 1024 + threadIdx.x;
  if (i < n) out[i] += block_offs[blockIdx.x];
}

__global__ void gin_fill_kernel(const int64_t* __restrict__ edge_index, const int64_t* __restrict__ edge_attr,
                                const int32_t* __restrict__ rowptr, int32_t* __restrict__ cursor, int32_t* __restrict__ col,
                                int32_t* __restrict__ eid, int e, int n) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= e) return;
  const long long srcl = edge_index[k], dstl = edge_index[(size_t)e + k];
  if (dstl < 0 || dstl >= n) return;
  const int dst = (int)dstl;
  const int pos = rowptr[dst] + atomicAdd(&cursor[dst], 1);
  const long long al = edge_attr[k];
  const int a = al < 0 ? 0 : (al >= BOND_VOCAB ? BOND_VOCAB - 1 : (int)al);
  col[pos] = (srcl < 0 || srcl >= n) ? dst : (int)srcl;
  eid[pos] = (k << 3) | a;   // edge id (deterministic order key) with the bond type in the low bits
}
// Sort every row by original edge id so that the floating-point summation order is run-to-run deterministic.
__global__ void gin_sort_rows_kernel(const int32_t* __restrict__ rowptr, int32_t* __restrict__ col, int32_t* __restrict__ eid, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int beg = rowptr[i], end = rowptr[i + 1];
  for (int a = beg + 1; a < end; ++a) {
    const int ke = eid[a], kc = col[a];
    int b = a - 1;
    while (b >= beg && eid[b] > ke) {
      eid[b + 1] = eid[b];
      col[b + 1] = col[b];
      --b;
    }
    eid[b + 1] = ke;
    col[b + 1] = kc;
  }
}

// Source-sorted CSR for the predictor's backward (the transpose of the aggregation scatters along out-edges), built from the
// destination-sorted one so that it holds exactly the edges the forward aggregated (input defects already resolved by
// gin_fill_kernel).  One thread per destination row: FILL = 0 counts out-degrees, FILL = 1 places (destination, edge id) at
// the source's rows; gin_sort_rows_kernel then orders every row by edge id.
template <int FILL>
__global__ void gin_csr_transpose_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, const int32_t* __restrict__ eid,
                                         const int32_t* __restrict__ srowptr, int32_t* __restrict__ cnt, int32_t* __restrict__ sdst,
                                         int32_t* __restrict__ seid, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  for (int p = rowptr[i]; p < rowptr[i + 1]; ++p) {
    const int j = col[p];
    if (FILL) {
      const int pos = srowptr[j] + atomicAdd(&cnt[j], 1);
      sdst[pos] = i;
      seid[pos] = eid[p];
    } else {
      atomicAdd(&cnt[j], 1);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Node kernels
// ---------------------------------------------------------------------------------------------
// h0 = atom_emb[x] + vn_emb (virtual node of layer 0 is the learned row for every graph).
__global__ void gin_embed_kernel(const int32_t* __restrict__ x32, const float* __restrict__ atom_emb, const float* __restrict__ vn_emb,
                                 float* __restrict__ h, __nv_bfloat16* __restrict__ hb, int n, int H) {
  const size_t total = (size_t)n * (H / 4);
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int i = (int)(idx / (H / 4)), c = (int)(idx % (H / 4)) * 4;
    const float4 a = *reinterpret_cast<const float4*>(atom_emb + (size_t)x32[i] * H + c);
    const float4 v = *reinterpret_cast<const float4*>(vn_emb + c);
    const float4 o = make_float4(a.x + v.x, a.y + v.y, a.z + v.z, a.w + v.w);
    *reinterpret_cast<float4*>(h + (size_t)i * H + c) = o;
    *reinterpret_cast<uint2*>(hb + (size_t)i * H + c) = make_uint2(pack_bf16x2(o.x, o.y), pack_bf16x2(o.z, o.w));
  }
}
__global__ void gin_broadcast_rows_kernel(const float* __restrict__ row, float* __restrict__ out, int rows, int W) {
  const size_t total = (size_t)rows * W;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x)
    out[idx] = row[idx % W];
}

// GIN aggregation (graph_encoder/model.py:167-173): out_i = (1+eps) h_i + sum_{j->i} gelu(h_j + bond_emb[e_ji]) -> bf16.
// One warp per destination node, 8 columns (16 B of bf16) per lane per sweep; CSR rows are short (degree <= ~4).  The self term is
// read from the bf16 copy (the row the node's neighbours gather anyway; the sum is rounded to bf16 on the way out).  This is the
// any-width fallback (H a multiple of 8); H = 256, 512, 768, 1024 go to gin_aggregate_wide_kernel.
// Width-specialised variant (H = 256 NSW): the neighbour loop is the OUTER one, so a neighbour's index / bond type are read once
// and its NSW 16-byte gathers are in flight together (three loads per lane instead of one when H = 768); 8 NSW fp32 accumulators.
template <int NSW>
__global__ void __launch_bounds__(256) gin_aggregate_wide_kernel(const __nv_bfloat16* __restrict__ hb, const int32_t* __restrict__ rowptr,
                                                                 const int32_t* __restrict__ col, const int32_t* __restrict__ eid,
                                                                 const float* __restrict__ bond_emb, const float* __restrict__ eps_ptr,
                                                                 __nv_bfloat16* __restrict__ out, int n) {
  constexpr int H = 256 * NSW;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const float one_eps = 1.0f + __ldg(eps_ptr);
  const int beg = rowptr[i], end = rowptr[i + 1];
  float acc[NSW][8];
#pragma unroll
  for (int w = 0; w < NSW; ++w) {
    const uint4 a = *reinterpret_cast<const uint4*>(hb + (size_t)i * H + w * 256 + lane * 8);
    acc[w][0] = one_eps * bf16_lo(a.x), acc[w][1] = one_eps * bf16_hi(a.x), acc[w][2] = one_eps * bf16_lo(a.y), acc[w][3] = one_eps * bf16_hi(a.y);
    acc[w][4] = one_eps * bf16_lo(a.z), acc[w][5] = one_eps * bf16_hi(a.z), acc[w][6] = one_eps * bf16_lo(a.w), acc[w][7] = one_eps * bf16_hi(a.w);
  }
  for (int k = beg; k < end; ++k) {
    const int j = __ldg(col + k);
    const int et = __ldg(eid + k) & 7;
    const __nv_bfloat16* src = hb + (size_t)j * H + lane * 8;
    const float* emb = bond_emb + (size_t)et * H + lane * 8;
    uint4 u[NSW];
#pragma unroll
    for (int w = 0; w < NSW; ++w) u[w] = *reinterpret_cast<const uint4*>(src + w * 256);
#pragma unroll
    for (int w = 0; w < NSW; ++w) {
      const float4 e0 = __ldg(reinterpret_cast<const float4*>(emb + w * 256));
      const float4 e1 = __ldg(reinterpret_cast<const float4*>(emb + w * 256 + 4));
      acc[w][0] += gelu_bf16(bf16_lo(u[w].x) + e0.x), acc[w][1] += gelu_bf16(bf16_hi(u[w].x) + e0.y);
      acc[w][2] += gelu_bf16(bf16_lo(u[w].y) + e0.z), acc[w][3] += gelu_bf16(bf16_hi(u[w].y) + e0.w);
      acc[w][4] += gelu_bf16(bf16_lo(u[w].z) + e1.x), acc[w][5] += gelu_bf16(bf16_hi(u[w].z) + e1.y);
      acc[w][6] += gelu_bf16(bf16_lo(u[w].w) + e1.z), acc[w][7] += gelu_bf16(bf16_hi(u[w].w) + e1.w);
    }
  }
#pragma unroll
  for (int w = 0; w < NSW; ++w)
    *reinterpret_cast<uint4*>(out + (size_t)i * H + w * 256 + lane * 8) = make_uint4(
        pack_bf16x2(acc[w][0], acc[w][1]), pack_bf16x2(acc[w][2], acc[w][3]), pack_bf16x2(acc[w][4], acc[w][5]), pack_bf16x2(acc[w][6], acc[w][7]));
}

__global__ void __launch_bounds__(256) gin_aggregate_kernel(const __nv_bfloat16* __restrict__ hb,
                                                            const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                                            const int32_t* __restrict__ eid, const float* __restrict__ bond_emb,
                                                            const float* __restrict__ eps_ptr, __nv_bfloat16* __restrict__ out,
                                                            int n, int H) {
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const float one_eps = 1.0f + __ldg(eps_ptr);
  const int beg = rowptr[i], end = rowptr[i + 1];
  for (int c = lane * 8; c < H; c += 256) {
    float acc[8];
    {
      // the self term comes from the bf16 copy as well: the sum is rounded to bf16 on the way out anyway (same error scale), the
      // row is the one this node's neighbours gather (L2-resident), and the fp32 row it replaces was a quarter of the kernel's
      // DRAM reads
      const uint4 a = *reinterpret_cast<const uint4*>(hb + (size_t)i * H + c);
      acc[0] = one_eps * bf16_lo(a.x), acc[1] = one_eps * bf16_hi(a.x), acc[2] = one_eps * bf16_lo(a.y), acc[3] = one_eps * bf16_hi(a.y);
      acc[4] = one_eps * bf16_lo(a.z), acc[5] = one_eps * bf16_hi(a.z), acc[6] = one_eps * bf16_lo(a.w), acc[7] = one_eps * bf16_hi(a.w);
    }
    for (int k = beg; k < end; ++k) {
      const int j = __ldg(col + k);
      const int et = __ldg(eid + k) & 7;
      const uint4 u = *reinterpret_cast<const uint4*>(hb + (size_t)j * H + c);
      const float4 e0 = *reinterpret_cast<const float4*>(bond_emb + (size_t)et * H + c);
      const float4 e1 = *reinterpret_cast<const float4*>(bond_emb + (size_t)et * H + c + 4);
      acc[0] += gelu_bf16(bf16_lo(u.x) + e0.x), acc[1] += gelu_bf16(bf16_hi(u.x) + e0.y);
      acc[2] += gelu_bf16(bf16_lo(u.y) + e0.z), acc[3] += gelu_bf16(bf16_hi(u.y) + e0.w);
      acc[4] += gelu_bf16(bf16_lo(u.z) + e1.x), acc[5] += gelu_bf16(bf16_hi(u.z) + e1.y);
      acc[6] += gelu_bf16(bf16_lo(u.w) + e1.z), acc[7] += gelu_bf16(bf16_hi(u.w) + e1.w);
    }
    *reinterpret_cast<uint4*>(out + (size_t)i * H + c) =
        make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]), pack_bf16x2(acc[4], acc[5]), pack_bf16x2(acc[6], acc[7]));
  }
}

// ---------------------------------------------------------------------------------------------
// Analytic LayerNorm statistics for the node MLP (Linear(H,4H) -> LayerNorm(4H) -> GELU -> Linear(4H,H), model.py:156-165).
// The LayerNorm needs the mean and variance of a 4H-wide row z = W a + b that no single CTA holds (3072 fp32 accumulator
// columns against 512 of tensor memory), which is why the unfused path writes z (757 MB per layer for 123 k nodes), re-reads
// and rewrites it in a row kernel and reads it again in the second GEMM.  Both moments are functions of the H-wide INPUT row a:
//   * mean.  LayerNorm is invariant to a shift of its input, so the weight is CENTRED over its 4H outputs at pack time,
//     Wc = W - 1 wbar^T, bc = b - bbar: zc = Wc a + bc has zero mean by construction and LN(zc) = LN(z).  (The bf16 rounding of
//     Wc leaves a residual mean of ~1e-4 sigma, which is ignored.)
//   * variance.  |zc|^2 = |Wt at|^2 with the augmented Wt = [Wc | bc] (4H x (H+1)) and at = [a; 1].  With the Cholesky factor
//     Wt^T Wt = Rt^T Rt (upper triangular, fp64 on the host at pack time, from the bf16-rounded Wc the tensor core multiplies by)
//     |zc|^2 = |Rt at|^2 = sum_{k<H} (R[k,:] . a + r[k])^2 + c0,   R = Rt[:H,:H], r = Rt[:H,H], c0 = Rt[H,H]^2,
//     i.e. ONE extra (n,H) x (H,H) GEMM per layer (a quarter of the first linear) whose epilogue only squares and adds its
//     accumulators (EpiRowSq: no output matrix, no operand re-reads) into (n, 6) partial sums.
// The first linear's epilogue (EpiLnGelu) then turns a row's partial sums into rstd and applies LayerNorm + affine + GELU
// directly, so z never exists un-normalised and the row kernel over the 4H-wide matrix disappears.
// Numerics (tests/test_analytic_ln_numerics.py): against the fp64-weight result the error of GELU(LN(z)) is the same as that of
// the two-pass LayerNorm on bf16 weights (rms 1.2e-3 = the bf16 rounding of the weights); rstd itself is within 4e-4.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) gin_colmean_kernel(const float* __restrict__ W, int rows, int H, float* __restrict__ wbar) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= H) return;
  double s = 0.0;
  for (int o = 0; o < rows; ++o) s += (double)W[(size_t)o * H + k];
  wbar[k] = (float)(s / rows);
}
// W (rows, H) contiguous -> out (rows, H) with row stride out_ld
__global__ void gin_center_weight_kernel(const float* __restrict__ W, const float* __restrict__ wbar, int rows, int H,
                                         __nv_bfloat16* __restrict__ out, int out_ld) {
  const size_t total = (size_t)rows * H;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x)
    out[(idx / H) * out_ld + idx % H] = __float2bfloat16(W[idx] - wbar[idx % H]);
}
// bc = b - mean(b), bg = bc * gamma (one block)
__global__ void __launch_bounds__(1024) gin_center_bias_kernel(const float* __restrict__ b, const float* __restrict__ gamma, int rows,
                                                               float* __restrict__ bc, float* __restrict__ bg) {
  __shared__ double red[32];
  __shared__ double s_mean;
  double s = 0.0;
  for (int o = threadIdx.x; o < rows; o += blockDim.x) s += (double)b[o];
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += red[w];
    s_mean = t / rows;
  }
  __syncthreads();
  const float m = (float)s_mean;
  for (int o = threadIdx.x; o < rows; o += blockDim.x) {
    const float c = b[o] - m;
    bc[o] = c;
    bg[o] = c * gamma[o];
  }
}
// Gram matrix of the augmented weight Wt = [Wc (bf16, row stride ld) | bc] in fp64: Gm (H+1, H+1), one thread per entry, pack
// time only.  H is the true width: the padded columns of Wc would make the matrix singular.
__global__ void __launch_bounds__(256) gin_gram64_kernel(const __nv_bfloat16* __restrict__ Wc, int ld, const float* __restrict__ bc, int rows,
                                                         int H, double* __restrict__ Gm) {
  const int j = blockIdx.x * 16 + (threadIdx.x & 15), i = blockIdx.y * 16 + (threadIdx.x >> 4);
  if (i > H || j > H || j < i) return;   // upper triangle; the host mirrors it
  double acc = 0.0;
  for (int o = 0; o < rows; ++o) {
    const double wi = i < H ? (double)__bfloat162float(Wc[(size_t)o * ld + i]) : (double)bc[o];
    const double wj = j < H ? (double)__bfloat162float(Wc[(size_t)o * ld + j]) : (double)bc[o];
    acc = fma(wi, wj, acc);
  }
  Gm[(size_t)i * (H + 1) + j] = acc;
}

// Host: lower Cholesky factor L of the symmetric positive (semi-)definite matrix whose UPPER triangle is in Gm (n x n), in place
// in Lm (row-major, L[i][j] for j <= i).  Row-oriented (Cholesky-Crout): both operands of every dot product are contiguous.
static void cholesky_lower_host(const std::vector<double>& Gm, int n, std::vector<double>& Lm) {
  Lm.assign((size_t)n * n, 0.0);
  double trace = 0.0;
  for (int i = 0; i < n; ++i) trace += Gm[(size_t)i * n + i];
  const double floor_d = 1e-14 * (trace / n) + 1e-300;
  for (int i = 0; i < n; ++i) {
    double* Li = &Lm[(size_t)i * n];
    for (int j = 0; j <= i; ++j) {
      const double* Lj = &Lm[(size_t)j * n];
      double s = Gm[(size_t)j * n + i];   // G[j][i], j <= i: upper triangle
      for (int k = 0; k < j; ++k) s -= Li[k] * Lj[k];
      if (j < i) Li[j] = s / Lj[j];
      else Li[i] = sqrt(s > floor_d ? s : floor_d);   // a rank-deficient weight gets a harmless tiny pivot
    }
  }
}

// Epilogue of the statistics GEMM Y = a R^T: no matrix output, per row the sum of (Y + r)^2 over the warp's columns.
struct EpiRowSq {
  static constexpr int CHUNK = 32;
  static constexpr bool OUT_F32 = true;
  static constexpr bool NO_STORE = true;
  void* C;     // unused
  int ldc;     // unused
  const float* r;   // (N) bias column of the factor
  float* part;      // (M, slots) partial sums, slot = (N tile, column group)
  int slots;
  struct RowState {
    float q;
  };
  __device__ __forceinline__ RowState row_begin(int, int) const { return RowState{0.f}; }
  __device__ __forceinline__ void transform(int, int col0, float* v, int, int, RowState& st) const {
    float q0 = 0.f, q1 = 0.f;   // two chains: the 32 dependent FMAs would otherwise serialise on the 4-cycle FMA latency
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(r + col0 + i)), b = __ldg(reinterpret_cast<const float4*>(r + col0 + i + 4));
      const float t0 = v[i] + a.x, t1 = v[i + 1] + a.y, t2 = v[i + 2] + a.z, t3 = v[i + 3] + a.w;
      const float t4 = v[i + 4] + b.x, t5 = v[i + 5] + b.y, t6 = v[i + 6] + b.z, t7 = v[i + 7] + b.w;
      q0 = fmaf(t0, t0, q0), q1 = fmaf(t4, t4, q1);
      q0 = fmaf(t1, t1, q0), q1 = fmaf(t5, t5, q1);
      q0 = fmaf(t2, t2, q0), q1 = fmaf(t6, t6, q1);
      q0 = fmaf(t3, t3, q0), q1 = fmaf(t7, t7, q1);
    }
    st.q += q0 + q1;
  }
  __device__ __forceinline__ void row_end(int row, int slot, RowState& st, int M) const {
    if (row < M) part[(size_t)row * slots + slot] = st.q;
  }
};

// Epilogue of the first linear (centred weight) with the row's |zc|^2 known: GELU(zc * rstd * gamma + beta) -> fp16.
// The affine part runs in fp32 on the accumulators; the GELU runs on PAIRS in fp16 (gelu_h2) and its result is stored as is:
// the intermediate of the node MLP is an fp16 matrix (values of order one: three more mantissa bits than bf16), consumed by the
// second linear with fp16 operands.  With K = H the epilogue of this GEMM, not its MMAs, sets the pace (ncu: tensor pipe 72 %
// active with the fp32 GELU + bf16 pack); the row's partial sums are fetched before the thread waits for the accumulators.
struct EpiLnGelu {
  static constexpr int CHUNK = 32;
  static constexpr bool OUT_F32 = false;
  static constexpr bool PACKS_OUTPUT = true;
  static constexpr int WARP_VECS = 3;   // gamma, bgamma, beta: each warp stages its 128 columns once per tile
  void* C;
  int ldc;
  const float *gamma, *bgamma, *beta;   // (N): LayerNorm weight, centred bias x weight, LayerNorm bias
  __device__ __forceinline__ const float* warp_vec(int i) const { return i == 0 ? gamma : (i == 1 ? bgamma : beta); }
  const float* part;                    // (M, slots) from EpiRowSq
  int slots;                            // even
  // constant of the factor, 1 / 4H with the TRUE 4H: at a padded width the GEMM runs N = I columns, but the padded ones have
  // zc = 0 and gamma = bgamma = beta = 0, so they come out as GELU(0) = 0 and add nothing to the statistics
  float c0, inv_rows;
  struct RowState {
    float rstd;
  };
  __device__ __forceinline__ RowState row_begin(int row, int M) const {
    float q = c0;
    if (row < M) {
      const float2* p = reinterpret_cast<const float2*>(part + (size_t)row * slots);
      float2 v[4];
#pragma unroll
      for (int s = 0; s < 4; ++s) v[s] = 2 * s < slots ? __ldg(p + s) : make_float2(0.f, 0.f);   // independent loads, fixed order
#pragma unroll
      for (int s = 0; s < 4; ++s) q += v[s].x, q += v[s].y;
      for (int s = 8; s < slots; ++s) q += __ldg(part + (size_t)row * slots + s);
    }
    return RowState{rsqrtf(q * inv_rows + 1e-5f)};
  }
  // sv: shared-space address of this warp's staged [gamma | bgamma | beta] x 128 columns, at the chunk's first column
  __device__ __forceinline__ void transform_pack(int, int, const float* v, uint32_t* out, int, int, RowState& st, uint32_t sv) const {
    const float rs = st.rstd;
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 g = lds128(sv + i * 4);
      const float4 b = lds128(sv + (128 + i) * 4);
      const float4 t = lds128(sv + (256 + i) * 4);
      const __half2 h0 = gelu_h2(__floats2half2_rn(fmaf(rs, fmaf(v[i], g.x, b.x), t.x), fmaf(rs, fmaf(v[i + 1], g.y, b.y), t.y)));
      const __half2 h1 = gelu_h2(__floats2half2_rn(fmaf(rs, fmaf(v[i + 2], g.z, b.z), t.z), fmaf(rs, fmaf(v[i + 3], g.w, b.w), t.w)));
      out[i / 2] = *reinterpret_cast<const uint32_t*>(&h0);
      out[i / 2 + 1] = *reinterpret_cast<const uint32_t*>(&h1);
    }
  }
  __device__ __forceinline__ void row_end(int, int, RowState&, int) const {}
};

// fp32 (rows, cols) -> fp16 (rows, cols) with row strides src_ld / dst_ld (second linear of the node MLP: its A operand is the
// fp16 intermediate above)
__global__ void gin_f32_to_f16_kernel(const float* __restrict__ src, int src_ld, __half* __restrict__ dst, int dst_ld, int rows, int cols) {
  const size_t total = (size_t)rows * cols;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x)
    dst[(idx / cols) * dst_ld + idx % cols] = __float2half_rn(src[(idx / cols) * src_ld + idx % cols]);
}

// Per-graph pooling over the contiguous node range (graph_encoder/model.py:148,152): max -> bf16 operand of the
// virtual-node MLP, sum -> fp32 (+bf16) read-out.  grid (B, ceil(H/256)).
// hb != null: read the bf16 copy of the rows instead (max-pooling into a bf16 result only: rounding is monotone, so the maximum of
// the rounded values IS the rounded maximum -- same bits, half the bytes).
__global__ void __launch_bounds__(256) gin_pool_kernel(const float* __restrict__ h, const __nv_bfloat16* __restrict__ hb,
                                                       const int32_t* __restrict__ graph_ptr, int H, int is_max, float* __restrict__ out_f32,
                                                       __nv_bfloat16* __restrict__ out_bf16) {
  const int g = blockIdx.x;
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= H) return;
  const int beg = graph_ptr[g], end = graph_ptr[g + 1];
  float acc = is_max ? -INFINITY : 0.f;
  for (int i = beg; i < end; ++i) {
    const float v = hb ? __bfloat162float(hb[(size_t)i * H + c]) : h[(size_t)i * H + c];
    acc = is_max ? fmaxf(acc, v) : acc + v;
  }
  if (beg == end) acc = 0.f;
  if (out_f32) out_f32[(size_t)g * H + c] = acc;
  if (out_bf16) out_bf16[(size_t)g * H + c] = __float2bfloat16(acc);
}

// Max-pool of the bf16 copy, two columns per thread (H even): rounding is monotone, so the maximum of the rounded values IS the
// rounded maximum of the fp32 rows -- same bits as gin_pool_kernel on h, half the bytes.  grid (B, ceil(H/512)).
__global__ void __launch_bounds__(256) gin_pool_max_bf16_kernel(const __nv_bfloat16* __restrict__ hb, const int32_t* __restrict__ graph_ptr,
                                                                int H, __nv_bfloat16* __restrict__ out) {
  const int g = blockIdx.x;
  const int c = (blockIdx.y * 256 + threadIdx.x) * 2;
  if (c >= H) return;
  const int beg = graph_ptr[g], end = graph_ptr[g + 1];
  float a0 = -INFINITY, a1 = -INFINITY;
#pragma unroll 4
  for (int i = beg; i < end; ++i) {
    const uint32_t u = *reinterpret_cast<const uint32_t*>(hb + (size_t)i * H + c);
    a0 = fmaxf(a0, bf16_lo(u)), a1 = fmaxf(a1, bf16_hi(u));
  }
  if (beg == end) a0 = a1 = 0.f;
  *reinterpret_cast<uint32_t*>(out + (size_t)g * H + c) = pack_bf16x2(a0, a1);
}

// Per-graph maxima accumulated by the fused layer tail (order-preserving uint encoding, 0 = no node seen) -> bf16 operand of
// the virtual-node MLP.
__global__ void gin_pool_decode_kernel(const uint32_t* __restrict__ enc, __nv_bfloat16* __restrict__ out, size_t total) {
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const uint32_t e = enc[idx];
    out[idx] = __float2bfloat16(e == 0u ? 0.f : __uint_as_float(float_order_dec(e)));
  }
}

// SiLU(c) -> bf16 (adapter operand, graph_predictor/model.py:247-252); c == null broadcasts text_dropping (:315-316).
__global__ void gin_text_operand_kernel(const float* __restrict__ c, const float* __restrict__ text_drop, __nv_bfloat16* __restrict__ out,
                                        int B, int W) {
  const size_t total = (size_t)B * W;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const float v = c ? c[idx] : text_drop[idx % W];
    out[idx] = __float2bfloat16(silu(v));
  }
}

// softmax + top-k of one logits row per CTA (graph_predictor/model.py:177-179).  k selection passes over the
// L2-resident row; ties resolve to the lowest index like torch.topk's stable behaviour on CPU.
__global__ void __launch_bounds__(1024) gin_topk_kernel(const float* __restrict__ logits, int ld, int W, int k, float* __restrict__ topv,
                                                        int32_t* __restrict__ topi, const int32_t* __restrict__ only_flagged) {
  if (only_flagged != nullptr && only_flagged[blockIdx.x] == 0) return;   // the single-pass kernel already produced this row
  __shared__ float red_v[32];
  __shared__ int red_i[32];
  __shared__ float s_max, s_sum, s_lastv;
  __shared__ int s_lasti;
  const float* row = logits + (size_t)blockIdx.x * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float m = -INFINITY;
  for (int c = tid; c < W; c += 1024) m = fmaxf(m, row[c]);
  m = warp_max(m);
  if (lane == 0) red_v[warp] = m;
  __syncthreads();
  if (warp == 0) {
    float x = warp_max(red_v[lane]);
    if (lane == 0) s_max = x;
  }
  __syncthreads();
  m = s_max;
  float s = 0.f;
  for (int c = tid; c < W; c += 1024) s += __expf(row[c] - m);
  s = warp_sum(s);
  __syncthreads();
  if (lane == 0) red_v[warp] = s;
  __syncthreads();
  if (warp == 0) {
    float x = warp_sum(red_v[lane]);
    if (lane == 0) s_sum = x, s_lastv = INFINITY, s_lasti = -1;
  }
  __syncthreads();
  const float inv = 1.0f / s_sum;
  for (int r = 0; r < k; ++r) {
    const float lv = s_lastv;
    const int li = s_lasti;
    float bv = -INFINITY;
    int bi = 0x7fffffff;
    for (int c = tid; c < W; c += 1024) {
      const float v = row[c];
      const bool eligible = (v < lv) || (v == lv && c > li);   // strictly after the previous pick in (value desc, index asc)
      if (eligible && (v > bv || (v == bv && c < bi))) bv = v, bi = c;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) bv = ov, bi = oi;
    }
    __syncthreads();
    if (lane == 0) red_v[warp] = bv, red_i[warp] = bi;
    __syncthreads();
    if (warp == 0) {
      bv = red_v[lane], bi = red_i[lane];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (ov > bv || (ov == bv && oi < bi)) bv = ov, bi = oi;
      }
      if (lane == 0) {
        s_lastv = bv, s_lasti = bi;
        topv[(size_t)blockIdx.x * k + r] = __expf(bv - m) * inv;
        topi[(size_t)blockIdx.x * k + r] = bi;
      }
    }
    __syncthreads();
  }
}

// Single-pass softmax + top-k of one logits row per CTA.  Every thread streams its strided share of the row once
// (float4 loads), keeping an online (max, sum of exp) pair and its own TK_T best entries in registers; the k winners
// are then drawn by k block-wide arg-max rounds over the per-thread heads.  A thread whose LAST kept entry gets drawn
// might have dropped a better one, so it flags the row and gin_topk_kernel (k selection passes, exact for any input)
// redoes it -- with strided ownership that needs 4 of the top k in one of 1024 residue classes.  Order: value
// descending, ties to the lowest index, like the selection-pass kernel.
constexpr int TK_T = 4;

__global__ void __launch_bounds__(1024) gin_topk_stream_kernel(const float* __restrict__ logits, int ld, int W, int k,
                                                               float* __restrict__ topv, int32_t* __restrict__ topi,
                                                               int32_t* __restrict__ redo_flag, int only_flagged) {
  if (only_flagged && redo_flag[blockIdx.x] == 0) return;   // the threshold kernel already produced this row
  __shared__ float red_v[32];
  __shared__ float red_s[32];
  __shared__ float s_max, s_sum;
  __shared__ int s_redo;
  const float* row = logits + (size_t)blockIdx.x * ld;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float bv[TK_T];
  int bi[TK_T];
#pragma unroll
  for (int j = 0; j < TK_T; ++j) bv[j] = -INFINITY, bi[j] = 0x7fffffff;
  float lm = -INFINITY, ls = 0.f;
  auto visit = [&](float v, int c) {
    if (v > lm) {   // online softmax in base 2
      ls *= exp2f((lm - v) * 1.4426950408889634f);
      lm = v;
    }
    ls += exp2f((v - lm) * 1.4426950408889634f);
    if (v > bv[TK_T - 1]) {   // strict: among equal values the earlier (lower) index stays
      bv[TK_T - 1] = v, bi[TK_T - 1] = c;
#pragma unroll
      for (int j = TK_T - 1; j > 0; --j) {
        if (bv[j] > bv[j - 1]) {
          const float tv = bv[j]; bv[j] = bv[j - 1]; bv[j - 1] = tv;
          const int ti = bi[j]; bi[j] = bi[j - 1]; bi[j - 1] = ti;
        }
      }
    }
  };
  const bool vec = (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0);
  if (vec) {
    const int W4 = W >> 2;
    for (int c4 = tid; c4 < W4; c4 += 1024) {
      const float4 q = __ldcs(reinterpret_cast<const float4*>(row) + c4);   // streamed once: do not keep it in L2
      visit(q.x, 4 * c4), visit(q.y, 4 * c4 + 1), visit(q.z, 4 * c4 + 2), visit(q.w, 4 * c4 + 3);
    }
    for (int c = (W4 << 2) + tid; c < W; c += 1024) visit(row[c], c);
  } else {
    for (int c = tid; c < W; c += 1024) visit(row[c], c);
  }
  // block (max, sum)
  float m = warp_max(lm);
  if (lane == 0) red_v[warp] = m;
  if (tid == 0) s_redo = 0;
  __syncthreads();
  if (warp == 0) {
    const float x = warp_max(red_v[lane]);
    if (lane == 0) s_max = x;
  }
  __syncthreads();
  m = s_max;
  float s = (lm == -INFINITY) ? 0.f : ls * exp2f((lm - m) * 1.4426950408889634f);
  s = warp_sum(s);
  if (lane == 0) red_s[warp] = s;
  __syncthreads();
  if (warp == 0) {
    const float x = warp_sum(red_s[lane]);
    if (lane == 0) s_sum = x;
  }
  __syncthreads();
  const float inv = 1.0f / s_sum;
  // k arg-max rounds over the per-thread heads.  A candidate is one sortable 64-bit key (order-preserving float bits in
  // the high word, inverted index in the low word: larger key = larger value, ties to the lower index), so a warp
  // arg-max is two REDUX instructions and every warp reduces the 32 warp winners itself: one barrier per round.
  __shared__ uint32_t key_hi[2][32], key_lo[2][32];
  auto enc_hi = [](float v) {
    const uint32_t u = __float_as_uint(v);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  };
  int head = 0;
  for (int r = 0; r < k; ++r) {
    float cv = -INFINITY;
    int ci = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < TK_T; ++j)
      if (j == head) cv = bv[j], ci = bi[j];
    const uint32_t hi = enc_hi(cv), lo = 0xffffffffu - (uint32_t)ci;   // exhausted / empty slots: (-inf, index 2^31-1), loses to any real entry
    const uint32_t whi = __reduce_max_sync(0xffffffffu, hi);
    const uint32_t wlo = __reduce_max_sync(0xffffffffu, hi == whi ? lo : 0u);
    const int buf = r & 1;
    if (lane == 0) key_hi[buf][warp] = whi, key_lo[buf][warp] = wlo;
    __syncthreads();
    const uint32_t ghi = __reduce_max_sync(0xffffffffu, key_hi[buf][lane]);
    const uint32_t glo = __reduce_max_sync(0xffffffffu, key_hi[buf][lane] == ghi ? key_lo[buf][lane] : 0u);
    const int wi = (int)(0xffffffffu - glo);
    if (tid == 0) {
      const uint32_t ub = (ghi & 0x80000000u) ? (ghi & 0x7fffffffu) : ~ghi;
      const float wv = __uint_as_float(ub);
      topv[(size_t)blockIdx.x * k + r] = exp2f((wv - m) * 1.4426950408889634f) * inv;
      topi[(size_t)blockIdx.x * k + r] = wi;
    }
    if (ci == wi && ci != 0x7fffffff) {   // my head was drawn (indices are unique)
      ++head;
      if (head == TK_T) s_redo = 1;        // my kept list is exhausted: a dropped entry could have been next
    }
    // the other key buffer is rewritten next round; everybody has read this one before the barrier after that
  }
  __syncthreads();
  if (tid == 0) redo_flag[blockIdx.x] = s_redo;
}

// Threshold variant of the single-pass kernel for WIDE rows (the predictor's 180 576 templates).  In the kernel above
// every thread maintains its own sorted list, and the insertion branch diverges: a thread inserts ~19 times per row, but
// some lane of a warp inserts in ~600 of its 176 x 4 element steps, so the warp spends most of the pass in the
// insertion path (47 us per row instead of the ~7 us the row's bytes need).  Here the block first looks at a strided
// SAMPLE of 4096 elements (one float4 per thread), takes tau = the R-th largest of the 32 warp maxima (R ~ 7 k 4096 / W,
// so that ~7 k elements of the row are expected above tau) and m0 = the sample maximum, then streams the row once with
// a branch-free body -- sum += 2^((v - m0) log2 e), running max -- and pushes the rare elements v > tau into a
// shared-memory candidate list.  The top k of the row are the top k of the candidates (everything else is <= tau); each
// candidate finds its rank by counting (value descending, ties to the lower index), no barrier rounds.
// Exactness: if fewer than k candidates were found, the list overflowed, or the row maximum exceeds m0 by more than
// 2^60 (overflow guard of the fixed-reference sum), the row is flagged and redone by the kernels above.
constexpr int TKH_CAP = 2048;
__device__ __forceinline__ uint32_t tk_enc(float v) {
  const uint32_t u = __float_as_uint(v);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float tk_dec(uint32_t e) { return __uint_as_float((e & 0x80000000u) ? (e & 0x7fffffffu) : ~e); }

__global__ void __launch_bounds__(1024) gin_topk_thresh_kernel(const float* __restrict__ logits, int ld, int W, int k, int R,
                                                               float* __restrict__ topv, int32_t* __restrict__ topi,
                                                               int32_t* __restrict__ redo_flag) {
  __shared__ uint32_t wkey[32];
  __shared__ float red_m[32], red_s[32];
  __shared__ float2 cand[TKH_CAP];   // (value, index bits)
  __shared__ int s_cnt;
  const float* row = logits + (size_t)blockIdx.x * ld;
  const float4* row4 = reinterpret_cast<const float4*>(row);
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W4 = W >> 2;
  constexpr float LOG2E = 1.4426950408889634f;
  // ---- sample: float4 number tid * (W4 / 1024), spread over the whole row
  {
    const float4 q = __ldg(row4 + (size_t)tid * (W4 >> 10));
    const uint32_t key = tk_enc(fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
    const uint32_t wmax = __reduce_max_sync(0xffffffffu, key);
    if (lane == 0) wkey[warp] = wmax;
    if (tid == 0) s_cnt = 0;
  }
  __syncthreads();
  float tau, m0;
  {
    uint32_t cur = wkey[lane];
    m0 = tk_dec(__reduce_max_sync(0xffffffffu, cur));
    uint32_t t = 0;
    for (int r = 0; r < R; ++r) {   // R-th largest (with multiplicity) of the 32 warp maxima
      t = __reduce_max_sync(0xffffffffu, cur);
      const uint32_t holders = __ballot_sync(0xffffffffu, cur == t);
      if (lane == __ffs(holders) - 1) cur = 0u;   // 0 encodes below every float
    }
    tau = tk_dec(t);
  }
  // ---- one pass over the row
  const float m0c = m0 * LOG2E;
  float ls = 0.f, lm = -INFINITY;
  auto visit = [&](float v, int c) {
    ls += ex2_approx(fmaf(v, LOG2E, -m0c));
    lm = fmaxf(lm, v);
    if (v > tau) {
      const int p = atomicAdd(&s_cnt, 1);
      if (p < TKH_CAP) cand[p] = make_float2(v, __int_as_float(c));
    }
  };
  {
    int c4 = tid;
    for (; c4 + 1024 < W4; c4 += 2048) {
      const float4 q0 = __ldcs(row4 + c4), q1 = __ldcs(row4 + c4 + 1024);   // streamed once: do not keep it in L2
      visit(q0.x, 4 * c4), visit(q0.y, 4 * c4 + 1), visit(q0.z, 4 * c4 + 2), visit(q0.w, 4 * c4 + 3);
      visit(q1.x, 4 * c4 + 4096), visit(q1.y, 4 * c4 + 4097), visit(q1.z, 4 * c4 + 4098), visit(q1.w, 4 * c4 + 4099);
    }
    for (; c4 < W4; c4 += 1024) {
      const float4 q = __ldcs(row4 + c4);
      visit(q.x, 4 * c4), visit(q.y, 4 * c4 + 1), visit(q.z, 4 * c4 + 2), visit(q.w, 4 * c4 + 3);
    }
    for (int c = (W4 << 2) + tid; c < W; c += 1024) visit(row[c], c);
  }
  const float wm = warp_max(lm), wsum = warp_sum(ls);
  if (lane == 0) red_m[warp] = wm, red_s[warp] = wsum;
  __syncthreads();
  const float m = warp_max(red_m[lane]);
  const float sum = warp_sum(red_s[lane]);
  const int C = s_cnt;
  if (C < k || C > TKH_CAP || (m - m0) * LOG2E > 60.f || !(sum > 0.f)) {   // block-uniform
    if (tid == 0) redo_flag[blockIdx.x] = 1;
    return;
  }
  const float inv = 1.0f / sum;
  for (int t = tid; t < C; t += 1024) {
    const float2 me = cand[t];
    const int mi = __float_as_int(me.y);
    int rank = 0;
    for (int j = 0; j < C; ++j) {
      const float2 o = cand[j];   // same address for the whole warp: broadcast
      rank += (o.x > me.x || (o.x == me.x && __float_as_int(o.y) < mi)) ? 1 : 0;
    }
    if (rank < k) {
      topv[(size_t)blockIdx.x * k + rank] = ex2_approx(fmaf(me.x, LOG2E, -m0c)) * inv;
      topi[(size_t)blockIdx.x * k + rank] = mi;
    }
  }
  if (tid == 0) redo_flag[blockIdx.x] = 0;
}

// Rows per launch -> (threshold kernel | per-thread-list kernel) -> selection-pass kernel for whatever is still flagged.
static void launch_softmax_topk(const float* logits, int rows, int W, int ld, int k, float* topv, int32_t* topi, int32_t* flags,
                                cudaStream_t s) {
  const bool vec = (ld % 4 == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0);
  const long long r_need = ((long long)7 * k * 4096 + W - 1) / W;
  const int R = r_need < 4 ? 4 : (int)r_need;
  if (vec && W >= 16384 && R <= 32) {
    gin_topk_thresh_kernel<<<rows, 1024, 0, s>>>(logits, ld, W, k, R, topv, topi, flags);
    gin_topk_stream_kernel<<<rows, 1024, 0, s>>>(logits, ld, W, k, topv, topi, flags, 1);
  } else {
    gin_topk_stream_kernel<<<rows, 1024, 0, s>>>(logits, ld, W, k, topv, topi, flags, 0);
  }
  gin_topk_kernel<<<rows, 1024, 0, s>>>(logits, ld, W, k, topv, topi, flags);
}

// ---------------------------------------------------------------------------------------------
// Fused predictor head: template logits -> softmax -> top-k WITHOUT the (graphs, out_dim) logits matrix
// (graph_predictor/model.py:174-179; 5.9 GB written and read back per 8192 graphs at out_dim = 180 576 when materialised).
//   1. pilot GEMM: logits of every pilot_stride-th template (4096 columns, 2.3 % of the head) -> gin_head_pilot_kernel: per row
//      m0 = the sample maximum (reference of the softmax sum) and tau = the R-th largest of the sample's 32 warp maxima, R chosen
//      so that ~7 k templates of the full row are expected above tau (the rule of gin_topk_thresh_kernel);
//   2. head GEMM with EpiHeadTopk: no output matrix; thread = row adds 2^((x - m0) log2 e) over its columns and appends the
//      rare x > tau to the row's candidate list; per (N tile, column group) partial sums -> deterministic total;
//   3. gin_head_select_kernel: total, rank of every candidate by counting (value descending, ties to the lower index) -> top-k.
// Rows with fewer than k candidates, an overflowing list or a non-finite / zero sum are FLAGGED; the host reads the flag count
// (the one synchronisation of llb_gin_predictor_topk) and sends flagged rows through the exact materialising path.
// ---------------------------------------------------------------------------------------------
// W (rows, K) contiguous -> Wp (cols, K) with row stride ld (the padded head width)
__global__ void gin_pilot_pack_kernel(const float* __restrict__ W, const float* __restrict__ b, int K, int stride, int cols,
                                      __nv_bfloat16* __restrict__ Wp, int ld, float* __restrict__ bp) {
  const int j = blockIdx.x;
  const float* src = W + (size_t)j * stride * K;
  for (int k = threadIdx.x; k < K; k += blockDim.x) Wp[(size_t)j * ld + k] = __float2bfloat16(src[k]);
  if (threadIdx.x == 0) bp[j] = b[(size_t)j * stride];
}

// one CTA of 1024 threads per row of the (rows, 4096) pilot logits -> (tau, m0 * log2 e)
__global__ void __launch_bounds__(1024) gin_head_pilot_kernel(const float* __restrict__ pilot, int R, float2* __restrict__ rowtau) {
  __shared__ uint32_t wkey[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float4 q = __ldg(reinterpret_cast<const float4*>(pilot + (size_t)blockIdx.x * HEAD_PILOT_COLS) + tid);
  const uint32_t key = tk_enc(fmaxf(fmaxf(q.x, q.y), fmaxf(q.z, q.w)));
  const uint32_t wmax = __reduce_max_sync(0xffffffffu, key);
  if (lane == 0) wkey[warp] = wmax;
  __syncthreads();
  if (warp == 0) {
    uint32_t cur = wkey[lane];
    const float m0 = tk_dec(__reduce_max_sync(0xffffffffu, cur));
    uint32_t t = 0;
    for (int r = 0; r < R; ++r) {   // R-th largest (with multiplicity) of the 32 warp maxima
      t = __reduce_max_sync(0xffffffffu, cur);
      const uint32_t holders = __ballot_sync(0xffffffffu, cur == t);
      if (lane == __ffs(holders) - 1) cur = 0u;
    }
    if (lane == 0) rowtau[blockIdx.x] = make_float2(tk_dec(t), m0 * 1.4426950408889634f);
  }
}

struct EpiHeadTopk {
  static constexpr int CHUNK = 32;
  static constexpr bool OUT_F32 = true;
  static constexpr bool NO_STORE = true;
  void* C;     // unused
  int ldc;     // unused
  const float* bias;        // (N)
  const float2* rowtau;     // (M) threshold, m0 * log2 e
  float* part;              // (M, slots) partial softmax sums
  int slots;
  float2* cand;             // (M, HEAD_CAND_CAP) (value, column bits)
  int32_t* cnt;             // (M) candidates seen (may exceed the capacity)
  struct RowState {
    float tau, m0c, s;
  };
  __device__ __forceinline__ RowState row_begin(int row, int M) const {
    const float2 t = row < M ? __ldg(rowtau + row) : make_float2(INFINITY, 0.f);
    return RowState{t.x, t.y, 0.f};
  }
  __device__ __forceinline__ void transform(int row, int col0, float* v, int M, int N, RowState& st) const {
    constexpr float LOG2E = 1.4426950408889634f;
    float s0 = 0.f, s1 = 0.f;
    const bool full = col0 + 32 <= N;
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      float4 b;
      if (full) b = __ldg(reinterpret_cast<const float4*>(bias + col0 + i));
      else b = make_float4(col0 + i < N ? __ldg(bias + col0 + i) : 0.f, col0 + i + 1 < N ? __ldg(bias + col0 + i + 1) : 0.f,
                           col0 + i + 2 < N ? __ldg(bias + col0 + i + 2) : 0.f, col0 + i + 3 < N ? __ldg(bias + col0 + i + 3) : 0.f);
      const float x[4] = {v[i] + b.x, v[i + 1] + b.y, v[i + 2] + b.z, v[i + 3] + b.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const bool in = full || col0 + i + e < N;
        const float ex = in ? ex2_approx(fmaf(x[e], LOG2E, -st.m0c)) : 0.f;
        if (e & 1) s1 += ex; else s0 += ex;
        if (in && x[e] > st.tau && row < M) {   // rare (~350 of 180 576 columns per row)
          const int p = atomicAdd(cnt + row, 1);
          if (p < HEAD_CAND_CAP) cand[(size_t)row * HEAD_CAND_CAP + p] = make_float2(x[e], __int_as_float(col0 + i + e));
        }
      }
    }
    st.s += s0 + s1;
  }
  __device__ __forceinline__ void row_end(int row, int slot, RowState& st, int M) const {
    if (row < M) part[(size_t)row * slots + slot] = st.s;
  }
};

// one CTA per row: softmax denominator from the partial sums, top-k of the candidate list by a bitonic sort of 64-bit keys
// (order-preserving value bits | inverted column: descending key = value descending, ties to the lower column).  Ranking every
// candidate by counting was O(C^2) = 0.8 ms per 8192 rows at C ~ 350; the sort is O(C log^2 C).
__global__ void __launch_bounds__(256) gin_head_select_kernel(const float* __restrict__ part, int slots, const float2* __restrict__ rowtau,
                                                              const float2* __restrict__ cand, const int32_t* __restrict__ cnt, int k,
                                                              float* __restrict__ topv, int32_t* __restrict__ topi, int32_t* __restrict__ flagged,
                                                              int32_t* __restrict__ n_flagged) {
  __shared__ float red[8];
  __shared__ unsigned long long keys[HEAD_CAND_CAP];
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // fixed summation tree: thread t adds slots t, t + 256, ... in order, then warp / block trees
  float s = 0.f;
  for (int i = tid; i < slots; i += 256) s += part[(size_t)row * slots + i];
  s = warp_sum(s);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  float sum = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) sum += red[w];
  const int C = cnt[row];
  if (C < k || C > HEAD_CAND_CAP || !(sum > 0.f) || !(sum < 3.0e38f)) {   // block-uniform
    if (tid == 0) flagged[atomicAdd(n_flagged, 1)] = row;
    return;
  }
  int n = 64;
  while (n < C) n <<= 1;   // power of two >= C (<= HEAD_CAND_CAP)
  for (int i = tid; i < n; i += 256) {
    unsigned long long key = 0ull;   // padding sorts last
    if (i < C) {
      const float2 c = cand[(size_t)row * HEAD_CAND_CAP + i];
      key = ((unsigned long long)tk_enc(c.x) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)__float_as_int(c.y));
    }
    keys[i] = key;
  }
  __syncthreads();
  for (int size = 2; size <= n; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < (n >> 1); t += 256) {
        const int lo = 2 * t - (t & (stride - 1));   // index of the pair's first element
        const int hi = lo + stride;
        const bool desc = (lo & size) == 0;          // descending runs first -> whole array descending at the end
        const unsigned long long a = keys[lo], b2 = keys[hi];
        if ((a < b2) == desc) keys[lo] = b2, keys[hi] = a;
      }
      __syncthreads();
    }
  }
  const float m0c = rowtau[row].y;
  const float inv = 1.0f / sum;
  for (int r = tid; r < k; r += 256) {
    const unsigned long long key = keys[r];
    const float v = tk_dec((uint32_t)(key >> 32));
    topv[(size_t)row * k + r] = ex2_approx(fmaf(v, 1.4426950408889634f, -m0c)) * inv;
    topi[(size_t)row * k + r] = (int32_t)(0xffffffffu - (uint32_t)(key & 0xffffffffull));
  }
}

// flagged rows: gather their head inputs / scatter their exact results
__global__ void gin_gather_rows_kernel(const __nv_bfloat16* __restrict__ src, const int32_t* __restrict__ rows, int W, __nv_bfloat16* __restrict__ dst) {
  const int r = rows[blockIdx.x];
  const uint4* s4 = reinterpret_cast<const uint4*>(src + (size_t)r * W);
  uint4* d4 = reinterpret_cast<uint4*>(dst + (size_t)blockIdx.x * W);
  for (int i = threadIdx.x; i < W / 8; i += blockDim.x) d4[i] = s4[i];
}
__global__ void gin_scatter_topk_kernel(const float* __restrict__ v, const int32_t* __restrict__ i, const int32_t* __restrict__ rows, int k,
                                        float* __restrict__ topv, int32_t* __restrict__ topi) {
  const int r = rows[blockIdx.x];
  for (int j = threadIdx.x; j < k; j += blockDim.x) {
    topv[(size_t)r * k + j] = v[(size_t)blockIdx.x * k + j];
    topi[(size_t)r * k + j] = i[(size_t)blockIdx.x * k + j];
  }
}

__global__ void cost_mlp_kernel(const float* __restrict__ w0, const float* __restrict__ b0, const float* __restrict__ w1,
                                const float* __restrict__ b1, const float* __restrict__ fps, int fp_dim, int latent,
                                float* __restrict__ out) {
  extern __shared__ float hid[];
  const float* x = fps + (size_t)blockIdx.x * fp_dim;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  for (int o = warp; o < latent; o += nw) {
    float s = 0.f;
    for (int k = lane; k < fp_dim; k += 32) s = fmaf(x[k], w0[(size_t)o * fp_dim + k], s);
    s = warp_sum(s);
    if (lane == 0) hid[o] = fmaxf(s + b0[o], 0.f);
  }
  __syncthreads();
  if (warp == 0) {
    float s = 0.f;
    for (int k = lane; k < latent; k += 32) s = fmaf(hid[k], w1[k], s);
    s = warp_sum(s);
    if (lane == 0) out[blockIdx.x] = logf(1.0f + expf(s + b1[0]));
  }
}

}  // namespace
}  // namespace llb

using namespace llb;

static const int TOPK_CHUNK = 4096;

static int gin_carve(llb_gin* g, void* ws, size_t ws_bytes, int n, int e, int B, bool want_logits, size_t* need) {
  const GinLayout& G = g->G;
  const size_t H = G.Hp, I = G.I;
  Arena a(ws, ws_bytes);
  g->x32 = a.take<int32_t>(n), g->batch32 = a.take<int32_t>(n), g->graph_ptr = a.take<int32_t>(B + 1);
  g->rowptr = a.take<int32_t>(n + 1), g->col = a.take<int32_t>(e > 0 ? e : 1), g->eid = a.take<int32_t>(e > 0 ? e : 1);
  g->deg = a.take<int32_t>(n + 1);
  g->flags = a.take<int32_t>(4);
  const int nb = ceil_div(n + 1, 1024);
  g->blk = a.take<int32_t>(nb + 1), g->blk2 = a.take<int32_t>(ceil_div(nb, 1024) + 1);
  g->h = a.take<float>((size_t)n * H), g->hb = a.take<__nv_bfloat16>((size_t)n * H), g->agg = a.take<__nv_bfloat16>((size_t)n * H);
  g->z = a.take<__nv_bfloat16>((size_t)n * I);
  g->u = a.take<float>((size_t)n * H);
  g->ln_slots = ceil_div((int)H, 256) * (GEMM_EPI_WARPS / 4);
  g->ln_part = a.take<float>((size_t)n * g->ln_slots);   // analytic LayerNorm statistics
  g->vn_cur = a.take<float>((size_t)B * H), g->vn_next = a.take<float>((size_t)B * H), g->vu = a.take<float>((size_t)B * H);
  g->pool_b = a.take<__nv_bfloat16>((size_t)B * H), g->vz = a.take<__nv_bfloat16>((size_t)B * I);
  if (G.predictor) {
    g->mod = a.take<float>((size_t)G.L * B * 3 * H);
    g->ctext = a.take<__nv_bfloat16>((size_t)B * G.tdim);
  }
  g->pooled = a.take<float>((size_t)B * H), g->pooled_b = a.take<__nv_bfloat16>((size_t)B * H);
  g->pool_enc = a.take<uint32_t>((size_t)B * H);
  g->tail_sync = a.take<uint8_t>(gemm_ln_pair_workspace_bytes());
  g->hz = a.take<__nv_bfloat16>((size_t)B * G.HH);
  if (!G.predictor) g->head_out = a.take<float>((size_t)B * H);
  const bool fused_head = G.pilot_cols > 0 && B >= HEAD_FUSED_MIN_ROWS;
  // the materialising path serves small batches and the flagged rows of the fused path: a few hundred logit rows are enough then
  g->chunk_rows = fused_head ? HEAD_FUSED_MIN_ROWS : (B < TOPK_CHUNK ? B : TOPK_CHUNK);
  if (G.predictor && want_logits) {
    g->logits_ws = a.take<float>((size_t)g->chunk_rows * G.out_dim);
    g->topk_redo = a.take<int32_t>(g->chunk_rows);
    g->fused_rows = fused_head ? (B < HEAD_ROW_CHUNK ? B : HEAD_ROW_CHUNK) : 0;
    if (fused_head) {
      const size_t R = g->fused_rows;
      g->head_slots = ceil_div(G.out_dim, 256) * (GEMM_EPI_WARPS / 4);
      g->pilot_logits = a.take<float>(R * HEAD_PILOT_COLS);
      g->rowtau = a.take<float2>(R);
      g->head_part = a.take<float>(R * g->head_slots);
      g->head_cand = a.take<float2>(R * HEAD_CAND_CAP);
      g->head_cnt = a.take<int32_t>(R), g->head_flagged = a.take<int32_t>(R), g->head_nflag = a.take<int32_t>(4);
      g->redo_in = a.take<__nv_bfloat16>((size_t)g->chunk_rows * G.HH);
      g->max_k = 1024;
      g->redo_v = a.take<float>((size_t)g->chunk_rows * g->max_k), g->redo_i = a.take<int32_t>((size_t)g->chunk_rows * g->max_k);
    }
  }
  *need = align_up(a.off, 256);
  return LLB_OK;
}

static int gin_scan(llb_gin* g, const int32_t* deg, int32_t* rowptr, cudaStream_t s) {
  // rowptr[0..n] = exclusive scan of deg[0..n] (deg[n] = 0)
  const int cnt = g->n + 1;
  const int nb = ceil_div(cnt, 1024);
  scan_block_kernel<<<nb, 1024, 0, s>>>(deg, rowptr, g->blk, cnt);
  LLB_CUDA_OK(cudaGetLastError());
  if (nb > 1) {
    const int nb2 = ceil_div(nb, 1024);
    LLB_CHECK_ARG(nb2 <= 1024, "gin: too many nodes (%d)", g->n);
    scan_block_kernel<<<nb2, 1024, 0, s>>>(g->blk, g->blk, g->blk2, nb);
    LLB_CUDA_OK(cudaGetLastError());
    if (nb2 > 1) {
      scan_block_kernel<<<1, 1024, 0, s>>>(g->blk2, g->blk2, nullptr, nb2);
      scan_add_kernel<<<nb2, 1024, 0, s>>>(g->blk, g->blk2, nb);
      LLB_CUDA_OK(cudaGetLastError());
      g->launches += 2;
    }
    scan_add_kernel<<<nb, 1024, 0, s>>>(rowptr, g->blk, cnt);
    LLB_CUDA_OK(cudaGetLastError());
    g->launches += 2;
  }
  g->launches++;
  return LLB_OK;
}

namespace llb {
int gin_node_mlp(llb_gin* g, const __nv_bfloat16* in, int rows, int l, float* ln_part, __nv_bfloat16* zbuf, float* u, int u_ld,
                 bool first_half_only, int slot0, int slot4, cudaStream_t s) {
  // node MLP with analytic LayerNorm statistics: statistics GEMM (no output matrix) -> first linear with LayerNorm + GELU in
  // its epilogue -> second linear.  The un-normalised 4H-wide intermediate never exists.
  const GinLayout& G = g->G;
  const int H = G.Hp;
  g->ctr.slot = LLB_PROF_GIN_GEMM_STATS;
  EpiRowSq es{nullptr, 0, g->w<float>(G.mlp_stat[l]), ln_part, g->ln_slots};
  LLB_TRY((launch_gemm<256>(in, H, g->w<void>(G.mlp_chol[l]), H, rows, H, H, es, s, &g->ctr)));
  g->ctr.slot = slot0;
  EpiLnGelu el{zbuf, G.I, g->w<float>(G.mlp_ln_w[l]), g->w<float>(G.mlp_bg[l]), g->w<float>(G.mlp_ln_b[l]), ln_part, g->ln_slots,
               g->chol_c0[l], 1.0f / (float)(4 * G.H)};
  LLB_TRY((launch_gemm<256>(in, H, g->w<void>(G.mlp0_w[l]), H, rows, G.I, H, el, s, &g->ctr)));
  g->ctr.slot = slot4;
  if (first_half_only) return LLB_OK;   // the caller fuses the second linear with the layer tail
  GemmGroups f16;
  f16.ab_f16 = true;   // fp16 intermediate x fp16 weight
  return gemm_bias_act(zbuf, G.I, g->w<void>(G.mlp4_w[l]), G.I, g->w<float>(G.mlp4_b[l]), u, u_ld, rows, H, G.I, LLB_ACT_NONE, true, s, &g->ctr, f16);
}
}  // namespace llb

static int gin_mlp4(llb_gin* g, const __nv_bfloat16* in, int rows, size_t w0, size_t b0, size_t lnw, size_t lnb, size_t w4, size_t b4,
                    int hidden, int hidden_true, int out_f, __nv_bfloat16* zbuf, float* out, int out_ld, cudaStream_t s,
                    int slot0 = LLB_PROF_GIN_MISC, int slot4 = LLB_PROF_GIN_MISC, int gram_layer = -1, bool first_half_only = false) {
  // Linear -> LayerNorm(hidden_true) -> GELU -> Linear  (the 4H MLP of GINConv / virtual node / heads); `hidden` is the padded
  // width of the intermediate, the input width is Hp
  const int H = g->G.Hp;
  if (gram_layer >= 0) return gin_node_mlp(g, in, rows, gram_layer, g->ln_part, zbuf, out, out_ld, first_half_only, slot0, slot4, s);
  g->ctr.slot = slot0;
  LLB_TRY(gemm_bias_act(in, H, g->w<void>(w0), H, g->w<float>(b0), zbuf, hidden, rows, hidden, H, LLB_ACT_NONE, false, s, &g->ctr));
  RowLnArgs a;
  a.in = zbuf, a.in_ld = hidden, a.in_bf16 = true, a.rows = rows, a.width = hidden, a.valid = hidden_true;
  a.gamma = g->w<float>(lnw), a.beta = g->w<float>(lnb), a.act = LLB_ACT_GELU;
  a.out_bf16 = zbuf, a.out_bf16_ld = hidden;
  a.prof_slot = LLB_PROF_GIN_ROWLN;
  LLB_TRY(launch_row_ln(a, s));
  g->launches++;
  g->ctr.slot = slot4;
  return gemm_bias_act(zbuf, hidden, g->w<void>(w4), hidden, g->w<float>(b4), out, out_ld, rows, out_f, hidden, LLB_ACT_NONE, true, s, &g->ctr);
}

// Trunk up to the pooled graph vector (B,H), stored (B,Hp).  sv != null: also keep what the backward needs (GinSaved); the
// copies read the buffers the unchanged forward writes, so the computation itself is the same either way.
static int gin_trunk(llb_gin* g, const float* c, cudaStream_t s, const GinSaved* sv = nullptr) {
  const GinLayout& G = g->G;
  const int H = G.Hp, L = G.L, n = g->n, B = g->B;   // H: the padded width of every H-wide buffer here
  LLB_CHECK_ARG(n > 0 && B > 0, "gin: no graph batch bound");
  const int eb = (int)(((size_t)n * (H / 4) + 255) / 256 < 8192 ? ((size_t)n * (H / 4) + 255) / 256 : 8192);
  gin_embed_kernel<<<eb, 256, 0, s>>>(g->x32, g->w<float>(G.atom_emb), g->w<float>(G.vn_emb), g->h, g->hb, n, H);
  gin_broadcast_rows_kernel<<<ceil_div(B * H, 256) < 4096 ? ceil_div(B * H, 256) : 4096, 256, 0, s>>>(g->w<float>(G.vn_emb), g->vn_cur, B, H);
  LLB_CUDA_OK(cudaGetLastError());
  g->launches += 2;
  if (G.predictor) {
    gin_text_operand_kernel<<<ceil_div(B * G.tdim, 256) < 4096 ? ceil_div(B * G.tdim, 256) : 4096, 256, 0, s>>>(
        c, g->w<float>(G.text_drop), g->ctext, B, G.tdim);
    LLB_CUDA_OK(cudaGetLastError());
    g->launches++;
    g->ctr.slot = LLB_PROF_GIN_MISC;
    for (int l = 0; l < L; ++l)
      LLB_TRY(gemm_bias_act(g->ctext, G.tdim, g->w<void>(G.adapter_w[l]), G.tdim, g->w<float>(G.adapter_b[l]),
                            g->mod + (size_t)l * B * 3 * H, 3 * H, B, 3 * H, G.tdim, LLB_ACT_NONE, true, s, &g->ctr));
    if (sv) LLB_CUDA_OK(cudaMemcpyAsync(sv->mod, g->mod, (size_t)L * B * 3 * H * 4, cudaMemcpyDeviceToDevice, s));
  }
  for (int l = 0; l < L; ++l) {
    const bool last = (l == L - 1);
    if (sv && l > 0) LLB_CUDA_OK(cudaMemcpyAsync(sv->hin + (size_t)(l - 1) * n * H, g->h, (size_t)n * H * 4, cudaMemcpyDeviceToDevice, s));
    {
      ProfScope prof(LLB_PROF_GIN_AGGREGATE, s);
      const float* be = g->w<float>(G.bond_emb[l]);
      const float* ep = g->w<float>(G.eps[l]);
      const unsigned blocks = (unsigned)ceil_div(n, 8);
      switch (H) {   // width-specialised (neighbour-outer) kernel for the widths the checkpoints and fixtures use
        case 256: gin_aggregate_wide_kernel<1><<<blocks, 256, 0, s>>>(g->hb, g->rowptr, g->col, g->eid, be, ep, g->agg, n); break;
        case 512: gin_aggregate_wide_kernel<2><<<blocks, 256, 0, s>>>(g->hb, g->rowptr, g->col, g->eid, be, ep, g->agg, n); break;
        case 768: gin_aggregate_wide_kernel<3><<<blocks, 256, 0, s>>>(g->hb, g->rowptr, g->col, g->eid, be, ep, g->agg, n); break;
        case 1024: gin_aggregate_wide_kernel<4><<<blocks, 256, 0, s>>>(g->hb, g->rowptr, g->col, g->eid, be, ep, g->agg, n); break;
        default: gin_aggregate_kernel<<<blocks, 256, 0, s>>>(g->hb, g->rowptr, g->col, g->eid, be, ep, g->agg, n, H);
      }
    }
    LLB_CUDA_OK(cudaGetLastError());
    g->launches++;
    if (sv) LLB_CUDA_OK(cudaMemcpyAsync(sv->agg + (size_t)l * n * H, g->agg, (size_t)n * H * 2, cudaMemcpyDeviceToDevice, s));
    // LLB_GIN_FUSED_TAIL=0: second linear + row kernel instead of the fused GEMM + layer-tail kernel (launch_gin_tail)
    static const bool tail_env_off = getenv("LLB_GIN_FUSED_TAIL") && getenv("LLB_GIN_FUSED_TAIL")[0] == '0';
    const bool fused_tail = !tail_env_off && G.H == G.Hp && gin_tail_supported(H, G.I);   // the fused tail has no column mask
    if (!last) {
      // virtual node of the next layer from the max-pool of this layer's INPUT (model.py:148 / :343): the fused tail of the
      // previous layer has already accumulated it while it wrote that input; layer 0 (and the unfused path) pool explicitly
      {
        ProfScope prof(LLB_PROF_GIN_POOL, s);
        if (fused_tail && l > 0) {
          const size_t total = (size_t)B * H;
          gin_pool_decode_kernel<<<(unsigned)(ceil_div((int)(total / 4), 256) < 2048 ? ceil_div((int)(total / 4), 256) : 2048), 256, 0, s>>>(g->pool_enc, g->pool_b, total);
        } else {
          if (H % 2 == 0) gin_pool_max_bf16_kernel<<<dim3(B, ceil_div(H, 512)), 256, 0, s>>>(g->hb, g->graph_ptr, H, g->pool_b);
          else gin_pool_kernel<<<dim3(B, ceil_div(H, 256)), 256, 0, s>>>(nullptr, g->hb, g->graph_ptr, H, 1, nullptr, g->pool_b);
        }
      }
      LLB_CUDA_OK(cudaGetLastError());
      g->launches++;
      if (sv) LLB_CUDA_OK(cudaMemcpyAsync(sv->pool + (size_t)l * B * H, g->pool_b, (size_t)B * H * 2, cudaMemcpyDeviceToDevice, s));
      LLB_TRY(gin_mlp4(g, g->pool_b, B, G.vn0_w[l], G.vn0_b[l], G.vn_ln_w[l], G.vn_ln_b[l], G.vn4_w[l], G.vn4_b[l], G.I, 4 * G.H, H,
                       g->vz, g->vu, H, s));
      RowLnArgs a;
      a.in = g->vu, a.in_ld = H, a.rows = B, a.width = H, a.normalize = false;
      a.resid = g->vn_cur, a.resid_ld = H, a.out_f32 = g->vn_next, a.out_f32_ld = H;
      a.prof_slot = LLB_PROF_GIN_MISC;
      LLB_TRY(launch_row_ln(a, s));
      g->launches++;
    }
    // LayerNorm + GELU of the node MLP in the first linear's epilogue, from analytic row statistics (see EpiRowSq); the
    // intermediate is fp16 and the second linear multiplies it by the fp16 copy of its weight
    LLB_TRY(gin_mlp4(g, g->agg, n, G.mlp0_w[l], G.mlp0_b[l], G.mlp_ln_w[l], G.mlp_ln_b[l], G.mlp4_w[l], G.mlp4_b[l], G.I, 4 * G.H, H,
                     g->z, g->u, H, s, LLB_PROF_GIN_GEMM_MLP0, LLB_PROF_GIN_GEMM_MLP4, l, fused_tail));
    const float* mod = G.predictor ? g->mod + (size_t)l * B * 3 * H : nullptr;
    if (fused_tail) {
      // second linear + LayerNorm + affine / text-adaLN + GELU + gate + residual + next virtual node in ONE kernel; it also
      // accumulates the per-graph maxima of the rows it writes whenever the next layer has a virtual-node update to feed
      const bool want_pool = l + 1 < L - 1;
      if (want_pool) LLB_CUDA_OK(cudaMemsetAsync(g->pool_enc, 0, (size_t)B * H * 4, s));
      GinTailArgs t{};
      t.bias = g->w<float>(G.mlp4_b[l]), t.row_group = g->batch32;
      if (G.predictor) t.shift = mod, t.scale = mod + H, t.gate = mod + 2 * H, t.mod_ld = 3 * H;
      else t.gamma = g->w<float>(G.norm_w[l]), t.beta = g->w<float>(G.norm_b[l]);
      if (!last) t.addvec = g->vn_next, t.addvec_ld = H;
      t.act = last ? LLB_ACT_NONE : LLB_ACT_GELU;
      t.x = g->h, t.ldx = H, t.xb = g->hb, t.ldxb = H;
      t.pool_max = want_pool ? g->pool_enc : nullptr, t.pool_ld = H;
      t.a_f16 = 1;
      g->ctr.slot = LLB_PROF_GIN_GEMM_MLP4;
      LLB_TRY(launch_gin_tail(g->z, G.I, g->w<void>(G.mlp4_w[l]), G.I, n, H, G.I, t, g->tail_sync, gemm_ln_pair_workspace_bytes(), s, &g->ctr));
    } else {
      RowLnArgs a;
      a.in = g->u, a.in_ld = H, a.rows = n, a.width = H, a.valid = G.H;
      a.row_group = g->batch32;
      if (G.predictor) {
        a.shift = mod, a.scale = mod + H, a.gate = mod + 2 * H, a.mod_ld = 3 * H;
      } else {
        a.gamma = g->w<float>(G.norm_w[l]), a.beta = g->w<float>(G.norm_b[l]);
      }
      a.act = last ? LLB_ACT_NONE : LLB_ACT_GELU;
      a.resid = g->h, a.resid_ld = H;
      if (!last) a.addvec = g->vn_next, a.addvec_ld = H;
      a.out_f32 = g->h, a.out_f32_ld = H, a.out_bf16 = g->hb, a.out_bf16_ld = H;
      a.prof_slot = LLB_PROF_GIN_ROWLN;
      LLB_TRY(launch_row_ln(a, s));
      g->launches++;
    }
    if (!last) std::swap(g->vn_cur, g->vn_next);
  }
  {
    ProfScope prof(LLB_PROF_GIN_POOL, s);
    gin_pool_kernel<<<dim3(B, ceil_div(H, 256)), 256, 0, s>>>(g->h, nullptr, g->graph_ptr, H, 0, g->pooled, g->pooled_b);
  }
  LLB_CUDA_OK(cudaGetLastError());
  g->launches++;
  if (sv) LLB_CUDA_OK(cudaMemcpyAsync(sv->pooled_b, g->pooled_b, (size_t)B * H * 2, cudaMemcpyDeviceToDevice, s));
  return LLB_OK;
}

extern "C" {

int llb_gin_packed_bytes(const llb_gin_config* cfg, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes, "llb_gin_packed_bytes: null argument");
  GinLayout G;
  LLB_TRY(make_layout(*cfg, G));
  *bytes = G.total;
  return LLB_OK;
}

int llb_gin_pack_weights(const llb_gin_config* cfg, const llb_gin_weights* w, void* packed, size_t packed_bytes,
                         llb_stream_t stream) {
  LLB_TRY(require_sm100());
  LLB_CHECK_ARG(cfg && w && packed, "llb_gin_pack_weights: null argument");
  GinLayout G;
  LLB_TRY(make_layout(*cfg, G));
  if (packed_bytes < G.total) return fail(LLB_ERR_WORKSPACE, "gin: packed blob needs %zu bytes, got %zu", G.total, packed_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* base = (uint8_t*)packed;
  const int H = G.H, Hp = G.Hp, I = G.I;   // every tensor is written at its true shape into the padded strides (see GinLayout)
  auto bf = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(base + off); };
  auto cp = [&](size_t off, const float* src, size_t n) {
    return cudaMemcpyAsync(base + off, src, n * 4, cudaMemcpyDeviceToDevice, s);
  };
  auto cp_rows = [&](size_t off, int dst_ld, const float* src, int rows, int cols) {   // (rows, cols) -> row stride dst_ld
    return cudaMemcpy2DAsync(base + off, (size_t)dst_ld * 4, src, (size_t)cols * 4, (size_t)cols * 4, rows, cudaMemcpyDeviceToDevice, s);
  };
  LLB_CUDA_OK(cudaMemsetAsync(base, 0, G.total, s));   // the padding of every parameter is zero
  LLB_CUDA_OK(cp_rows(G.atom_emb, Hp, w->atom_emb, ATOM_VOCAB, H));
  LLB_CUDA_OK(cp(G.vn_emb, w->vn_emb, H));
  for (int l = 0; l < G.L; ++l) {
    gin_f32_to_f16_kernel<<<1024, 256, 0, s>>>(w->mlp4_w[l], 4 * H, reinterpret_cast<__half*>(base + G.mlp4_w[l]), I, H, 4 * H);   // fp16: see EpiLnGelu
    LLB_CUDA_OK(cudaGetLastError());
    LLB_CUDA_OK(cp(G.eps[l], w->eps[l], 1));
    LLB_CUDA_OK(cp(G.mlp_ln_w[l], w->mlp_ln_w[l], 4 * H));
    LLB_CUDA_OK(cp(G.mlp_ln_b[l], w->mlp_ln_b[l], 4 * H));
    LLB_CUDA_OK(cp(G.mlp4_b[l], w->mlp4_b[l], H));
    // first linear of the node MLP, CENTRED over its 4H outputs (LayerNorm is shift-invariant; see EpiRowSq), and the Cholesky
    // factor of its augmented Gram matrix for the analytic LayerNorm statistics: fp64 on the host, from the bf16-rounded
    // weight the tensor core multiplies by.  This is the one place where pack_weights synchronises the stream.
    // At a padded width the centring and the Gram matrix cover the true 4H rows and (H+1) columns only: the padded rows stay 0
    // (not centred), and a padded Gram matrix would be singular.
    {
      float* wbar = reinterpret_cast<float*>(base + G.chol_scratch);   // scratch doubles as the column-mean buffer first
      gin_colmean_kernel<<<ceil_div(H, 256), 256, 0, s>>>(w->mlp0_w[l], 4 * H, H, wbar);
      gin_center_weight_kernel<<<1024, 256, 0, s>>>(w->mlp0_w[l], wbar, 4 * H, H, bf(G.mlp0_w[l]), Hp);
      gin_center_bias_kernel<<<1, 1024, 0, s>>>(w->mlp0_b[l], w->mlp_ln_w[l], 4 * H, reinterpret_cast<float*>(base + G.mlp0_b[l]),
                                                 reinterpret_cast<float*>(base + G.mlp_bg[l]));
      double* Gd = reinterpret_cast<double*>(base + G.chol_scratch);
      gin_gram64_kernel<<<dim3(ceil_div(H + 1, 16), ceil_div(H + 1, 16)), 256, 0, s>>>(bf(G.mlp0_w[l]), Hp, reinterpret_cast<const float*>(base + G.mlp0_b[l]),
                                                                                      4 * H, H, Gd);
      LLB_CUDA_OK(cudaGetLastError());
      const int n1 = H + 1;
      std::vector<double> Gh((size_t)n1 * n1), Lh;
      LLB_CUDA_OK(cudaMemcpyAsync(Gh.data(), Gd, Gh.size() * 8, cudaMemcpyDeviceToHost, s));
      LLB_CUDA_OK(cudaStreamSynchronize(s));
      cholesky_lower_host(Gh, n1, Lh);
      // R[k][i] = L[i][k] (upper factor, k = output row of the statistics GEMM's weight), r[k] = L[H][k], c0 = L[H][H]^2.
      // R is stored (Hp, Hp) and r with Hp entries, zero past H; c0 sits at index Hp (EpiRowSq adds r_k to all Hp columns).
      std::vector<__nv_bfloat16> Rb((size_t)Hp * Hp, __float2bfloat16(0.f));
      std::vector<float> st(Hp + 4, 0.f);
      for (int k = 0; k < H; ++k) {
        for (int i = 0; i < H; ++i) Rb[(size_t)k * Hp + i] = __float2bfloat16(i >= k ? (float)Lh[(size_t)i * n1 + k] : 0.f);
        st[k] = (float)Lh[(size_t)H * n1 + k];
      }
      st[Hp] = (float)(Lh[(size_t)H * n1 + H] * Lh[(size_t)H * n1 + H]);
      LLB_CUDA_OK(cudaMemcpyAsync(base + G.mlp_chol[l], Rb.data(), Rb.size() * 2, cudaMemcpyHostToDevice, s));
      LLB_CUDA_OK(cudaMemcpyAsync(base + G.mlp_stat[l], st.data(), st.size() * 4, cudaMemcpyHostToDevice, s));
      LLB_CUDA_OK(cudaStreamSynchronize(s));   // Rb / st die with this scope
    }
    LLB_CUDA_OK(cp_rows(G.bond_emb[l], Hp, w->bond_emb[l], BOND_VOCAB, H));
    if (!G.predictor) {
      LLB_CHECK_ARG(w->norm_w && w->norm_b, "gin: the encoder needs norms.{l}.weight/bias");
      LLB_CUDA_OK(cp(G.norm_w[l], w->norm_w[l], H));
      LLB_CUDA_OK(cp(G.norm_b[l], w->norm_b[l], H));
    }
    if (l < G.L - 1) {
      LLB_TRY(launch_f32_to_bf16(w->vn0_w[l], H, bf(G.vn0_w[l]), Hp, 4 * H, H, Hp, s));
      LLB_TRY(launch_f32_to_bf16(w->vn4_w[l], 4 * H, bf(G.vn4_w[l]), I, H, 4 * H, I, s));
      LLB_CUDA_OK(cp(G.vn0_b[l], w->vn0_b[l], 4 * H));
      LLB_CUDA_OK(cp(G.vn_ln_w[l], w->vn_ln_w[l], 4 * H));
      LLB_CUDA_OK(cp(G.vn_ln_b[l], w->vn_ln_b[l], 4 * H));
      LLB_CUDA_OK(cp(G.vn4_b[l], w->vn4_b[l], H));
    }
    if (G.predictor) {
      // [shift | scale | gate] as three row blocks of Hp rows: the forward reads them at mod, mod + Hp, mod + 2 Hp
      for (int b = 0; b < 3; ++b) {
        LLB_TRY(launch_f32_to_bf16(w->adapter_w[l] + (size_t)b * H * G.tdim, G.tdim, bf(G.adapter_w[l]) + (size_t)b * Hp * G.tdim, G.tdim, H,
                                   G.tdim, G.tdim, s));
        LLB_CUDA_OK(cp(G.adapter_b[l] + (size_t)b * Hp * 4, w->adapter_b[l] + (size_t)b * H, H));
      }
    }
  }
  if (G.predictor) LLB_CUDA_OK(cp(G.text_drop, w->text_dropping, G.tdim));
  const int HOt = G.predictor ? G.out_dim : H;   // true output width of the head
  LLB_TRY(launch_f32_to_bf16(w->head0_w, H, bf(G.head0_w), Hp, G.HHt, H, Hp, s));
  LLB_TRY(launch_f32_to_bf16(w->head4_w, G.HHt, bf(G.head4_w), G.HH, HOt, G.HHt, G.HH, s));
  LLB_CUDA_OK(cp(G.head0_b, w->head0_b, G.HHt));
  LLB_CUDA_OK(cp(G.head_ln_w, w->head_ln_w, G.HHt));
  LLB_CUDA_OK(cp(G.head_ln_b, w->head_ln_b, G.HHt));
  LLB_CUDA_OK(cp(G.head4_b, w->head4_b, HOt));
  if (G.pilot_cols > 0) {
    gin_pilot_pack_kernel<<<G.pilot_cols, 256, 0, s>>>(w->head4_w, w->head4_b, G.HHt, G.pilot_stride, G.pilot_cols, bf(G.pilot_w), G.HH,
                                                       reinterpret_cast<float*>(base + G.pilot_b));
    LLB_CUDA_OK(cudaGetLastError());
  }
  return LLB_OK;
}

int llb_gin_create(const llb_gin_config* cfg, const void* packed, size_t packed_bytes, llb_gin** out) {
  LLB_TRY(require_sm100());
  LLB_CHECK_ARG(cfg && packed && out, "llb_gin_create: null argument");
  llb_gin* g = new llb_gin();
  g->cfg = *cfg;
  int st = make_layout(*cfg, g->G);
  if (st == LLB_OK && packed_bytes < g->G.total)
    st = fail(LLB_ERR_WORKSPACE, "gin: packed blob needs %zu bytes, got %zu", g->G.total, packed_bytes);
  if (st != LLB_OK) {
    delete g;
    return st;
  }
  g->blob = (const uint8_t*)packed;
  g->chol_c0.resize(g->G.L);
  for (int l = 0; l < g->G.L; ++l) {   // synchronous: create is not on the hot path
    cudaError_t e = cudaMemcpy(&g->chol_c0[l], g->blob + g->G.mlp_stat[l] + (size_t)g->G.Hp * 4, 4, cudaMemcpyDeviceToHost);
    if (e != cudaSuccess) {
      delete g;
      return fail(LLB_ERR_CUDA, "gin: reading the packed statistics back failed: %s", cudaGetErrorString(e));
    }
  }
  *out = g;
  return LLB_OK;
}

void llb_gin_destroy(llb_gin* g) { delete g; }

int llb_gin_workspace_bytes(const llb_gin_config* cfg, int num_nodes, int num_edges, int num_graphs, int want_logits,
                            size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes && num_nodes >= 1 && num_edges >= 0 && num_graphs >= 1, "llb_gin_workspace_bytes: bad argument");
  llb_gin tmp;
  tmp.cfg = *cfg;
  LLB_TRY(make_layout(*cfg, tmp.G));
  return gin_carve(&tmp, nullptr, 0, num_nodes, num_edges, num_graphs, want_logits != 0, bytes);
}

int llb_gin_bind(llb_gin* g, void* workspace, size_t workspace_bytes, int num_nodes, int num_edges, int num_graphs,
                 const int64_t* x, const int64_t* edge_index, const int64_t* edge_attr, const int64_t* batch,
                 llb_stream_t stream) {
  LLB_CHECK_ARG(g && workspace && x && batch && num_nodes >= 1 && num_graphs >= 1 && num_edges >= 0, "llb_gin_bind: bad argument");
  LLB_CHECK_ARG(num_edges == 0 || (edge_index && edge_attr), "llb_gin_bind: null edge arrays");
  LLB_CHECK_ARG(num_edges < (1 << 28), "llb_gin_bind: too many edges");
  cudaStream_t s = (cudaStream_t)stream;
  size_t need = 0;
  // logits scratch is carved whenever the workspace is large enough for it (top-k path); forward() writes to the caller's buffer
  LLB_TRY(gin_carve(g, workspace, workspace_bytes, num_nodes, num_edges, num_graphs, true, &need));
  g->want_logits = need <= workspace_bytes;
  if (!g->want_logits) {
    LLB_TRY(gin_carve(g, workspace, workspace_bytes, num_nodes, num_edges, num_graphs, false, &need));
    g->logits_ws = nullptr;
    if (need > workspace_bytes) return fail(LLB_ERR_WORKSPACE, "gin: workspace needs %zu bytes, got %zu", need, workspace_bytes);
  }
  g->n = num_nodes, g->e = num_edges, g->B = num_graphs;
  const int n = num_nodes, e = num_edges;
  LLB_CUDA_OK(cudaMemsetAsync(g->flags, 0, 16, s));
  gin_prep_nodes_kernel<<<ceil_div(n, 256), 256, 0, s>>>(x, batch, g->x32, g->batch32, g->graph_ptr, g->flags, n, num_graphs);
  LLB_CUDA_OK(cudaGetLastError());
  LLB_CUDA_OK(cudaMemsetAsync(g->deg, 0, (size_t)(n + 1) * 4, s));
  if (e > 0) {
    gin_degree_kernel<<<ceil_div(e, 256), 256, 0, s>>>(edge_index, edge_attr, g->deg, g->flags, e, n);
    LLB_CUDA_OK(cudaGetLastError());
  }
  LLB_TRY(gin_scan(g, g->deg, g->rowptr, s));
  LLB_CUDA_OK(cudaMemsetAsync(g->deg, 0, (size_t)(n + 1) * 4, s));
  if (e > 0) {
    gin_fill_kernel<<<ceil_div(e, 256), 256, 0, s>>>(edge_index, edge_attr, g->rowptr, g->deg, g->col, g->eid, e, n);
    gin_sort_rows_kernel<<<ceil_div(n, 256), 256, 0, s>>>(g->rowptr, g->col, g->eid, n);
    LLB_CUDA_OK(cudaGetLastError());
  }
  g->launches += 4;
  return LLB_OK;
}

int llb_gin_input_flags(llb_gin* g, int32_t* flags_host, llb_stream_t stream) {
  LLB_CHECK_ARG(g && flags_host && g->flags, "llb_gin_input_flags: no graph batch bound");
  cudaStream_t s = (cudaStream_t)stream;
  LLB_CUDA_OK(cudaMemcpyAsync(flags_host, g->flags, 4, cudaMemcpyDeviceToHost, s));
  LLB_CUDA_OK(cudaStreamSynchronize(s));
  return LLB_OK;
}

int llb_gin_encoder_forward(llb_gin* g, float* out, float* pooled_or_null, llb_stream_t stream) {
  LLB_CHECK_ARG(g && out && !g->G.predictor, "llb_gin_encoder_forward: needs an encoder handle and an output buffer");
  cudaStream_t s = (cudaStream_t)stream;
  const GinLayout& G = g->G;
  const int B = g->B;
  LLB_TRY(gin_trunk(g, nullptr, s));
  // the caller's (B,H) rows come out of the internal (B,Hp) ones
  if (pooled_or_null)
    LLB_CUDA_OK(cudaMemcpy2DAsync(pooled_or_null, (size_t)G.H * 4, g->pooled, (size_t)G.Hp * 4, (size_t)G.H * 4, B, cudaMemcpyDeviceToDevice, s));
  LLB_TRY(gin_mlp4(g, g->pooled_b, B, G.head0_w, G.head0_b, G.head_ln_w, G.head_ln_b, G.head4_w, G.head4_b, G.HH, G.HHt, G.HO, g->hz,
                   g->head_out, G.Hp, s, LLB_PROF_GIN_GEMM_HEAD, LLB_PROF_GIN_GEMM_HEAD));
  // L2 normalisation (the padded columns are 0 and add nothing): straight into the caller's rows when the row kernel can write
  // H columns (H % 4 == 0), else in place at the padded width and a strided copy
  const bool direct = G.H % 4 == 0;
  RowLnArgs a;
  a.in = g->head_out, a.in_ld = G.Hp, a.rows = B, a.width = direct ? G.H : G.Hp, a.normalize = false, a.l2_normalize = true;
  a.out_f32 = direct ? out : g->head_out, a.out_f32_ld = direct ? G.H : G.Hp;
  a.prof_slot = LLB_PROF_GIN_MISC;
  LLB_TRY(launch_row_ln(a, s));
  g->launches++;
  if (!direct)
    LLB_CUDA_OK(cudaMemcpy2DAsync(out, (size_t)G.H * 4, g->head_out, (size_t)G.Hp * 4, (size_t)G.H * 4, B, cudaMemcpyDeviceToDevice, s));
  return LLB_OK;
}

static int gin_head_hidden(llb_gin* g, cudaStream_t s) {
  // decoder.0 -> LayerNorm -> GELU, result (B,4H) bf16 in g->hz
  const GinLayout& G = g->G;
  g->ctr.slot = LLB_PROF_GIN_GEMM_HEAD;
  LLB_TRY(gemm_bias_act(g->pooled_b, G.Hp, g->w<void>(G.head0_w), G.Hp, g->w<float>(G.head0_b), g->hz, G.HH, g->B, G.HH, G.Hp,
                        LLB_ACT_NONE, false, s, &g->ctr));
  RowLnArgs a;
  a.in = g->hz, a.in_ld = G.HH, a.in_bf16 = true, a.rows = g->B, a.width = G.HH, a.valid = G.HHt;
  a.gamma = g->w<float>(G.head_ln_w), a.beta = g->w<float>(G.head_ln_b), a.act = LLB_ACT_GELU;
  a.out_bf16 = g->hz, a.out_bf16_ld = G.HH;
  a.prof_slot = LLB_PROF_GIN_ROWLN;
  LLB_TRY(launch_row_ln(a, s));
  g->launches++;
  return LLB_OK;
}

int llb_gin_predictor_forward(llb_gin* g, const float* c, float* logits, llb_stream_t stream) {
  LLB_CHECK_ARG(g && logits && g->G.predictor, "llb_gin_predictor_forward: needs a predictor handle and an output buffer");
  cudaStream_t s = (cudaStream_t)stream;
  const GinLayout& G = g->G;
  LLB_TRY(gin_trunk(g, c, s));
  LLB_TRY(gin_head_hidden(g, s));
  return gemm_bias_act(g->hz, G.HH, g->w<void>(G.head4_w), G.HH, g->w<float>(G.head4_b), logits, G.out_dim, g->B, G.out_dim, G.HH,
                       LLB_ACT_NONE, true, s, &g->ctr);
}

int llb_gin_saved_bytes(const llb_gin_config* cfg, int num_nodes, int num_edges, int num_graphs, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes && num_nodes >= 1 && num_edges >= 0 && num_graphs >= 1, "llb_gin_saved_bytes: bad argument");
  LLB_CHECK_ARG(cfg->predictor, "llb_gin_saved_bytes: only the predictor has a backward");
  GinLayout G;
  LLB_TRY(make_layout(*cfg, G));
  gin_saved_carve(G, nullptr, num_nodes, num_edges, num_graphs, nullptr, bytes);
  return LLB_OK;
}

int llb_gin_predictor_forward_saved(llb_gin* g, const float* c, float* logits, void* saved, size_t saved_bytes, llb_stream_t stream) {
  LLB_CHECK_ARG(g && logits && saved && g->G.predictor, "llb_gin_predictor_forward_saved: needs a predictor handle and output buffers");
  LLB_CHECK_ARG(g->n > 0 && g->B > 0, "gin: no graph batch bound");
  cudaStream_t s = (cudaStream_t)stream;
  const GinLayout& G = g->G;
  const int n = g->n, e = g->e, B = g->B;
  GinSaved sv;
  size_t need = 0;
  gin_saved_carve(G, saved, n, e, B, &sv, &need);
  if (saved_bytes < need) return fail(LLB_ERR_WORKSPACE, "gin: saved buffer needs %zu bytes, got %zu", need, saved_bytes);
  LLB_CUDA_OK(cudaMemcpyAsync(sv.graph_ptr, g->graph_ptr, (size_t)(B + 1) * 4, cudaMemcpyDeviceToDevice, s));
  LLB_CUDA_OK(cudaMemcpyAsync(sv.batch32, g->batch32, (size_t)n * 4, cudaMemcpyDeviceToDevice, s));
  // source-sorted CSR (the bound batch's degree scratch is free once llb_gin_bind has built the destination CSR)
  LLB_CUDA_OK(cudaMemsetAsync(g->deg, 0, (size_t)(n + 1) * 4, s));
  gin_csr_transpose_kernel<0><<<ceil_div(n, 256), 256, 0, s>>>(g->rowptr, g->col, g->eid, nullptr, g->deg, nullptr, nullptr, n);
  LLB_CUDA_OK(cudaGetLastError());
  LLB_TRY(gin_scan(g, g->deg, sv.srowptr, s));
  LLB_CUDA_OK(cudaMemsetAsync(g->deg, 0, (size_t)(n + 1) * 4, s));
  gin_csr_transpose_kernel<1><<<ceil_div(n, 256), 256, 0, s>>>(g->rowptr, g->col, g->eid, sv.srowptr, g->deg, sv.sdst, sv.seid, n);
  gin_sort_rows_kernel<<<ceil_div(n, 256), 256, 0, s>>>(sv.srowptr, sv.sdst, sv.seid, n);
  LLB_CUDA_OK(cudaGetLastError());
  g->launches += 3;
  // from here on exactly llb_gin_predictor_forward
  LLB_TRY(gin_trunk(g, c, s, &sv));
  LLB_TRY(gin_head_hidden(g, s));
  return gemm_bias_act(g->hz, G.HH, g->w<void>(G.head4_w), G.HH, g->w<float>(G.head4_b), logits, G.out_dim, B, G.out_dim, G.HH,
                       LLB_ACT_NONE, true, s, &g->ctr);
}

int llb_gin_predictor_topk(llb_gin* g, const float* c, int k, float* topk_prob, int32_t* topk_idx, llb_stream_t stream) {
  LLB_CHECK_ARG(g && topk_prob && topk_idx && g->G.predictor, "llb_gin_predictor_topk: needs a predictor handle and output buffers");
  const GinLayout& G = g->G;
  LLB_CHECK_ARG(k >= 1 && k <= G.out_dim, "llb_gin_predictor_topk: k=%d outside [1,%d]", k, G.out_dim);
  if (!g->logits_ws) return fail(LLB_ERR_WORKSPACE, "llb_gin_predictor_topk: bind the batch with a workspace sized with want_logits=1");
  cudaStream_t s = (cudaStream_t)stream;
  LLB_TRY(gin_trunk(g, c, s));
  LLB_TRY(gin_head_hidden(g, s));
  g->ctr.slot = LLB_PROF_GIN_GEMM_HEAD;
  // exact path over a range of head-input rows: materialise <= chunk_rows logit rows at a time, streaming softmax + top-k
  auto materialise = [&](const __nv_bfloat16* in, int nrows, float* outv, int32_t* outi) -> int {
    for (int r0 = 0; r0 < nrows; r0 += g->chunk_rows) {
      const int rows = nrows - r0 < g->chunk_rows ? nrows - r0 : g->chunk_rows;
      g->ctr.slot = LLB_PROF_GIN_GEMM_HEAD;
      LLB_TRY(gemm_bias_act(in + (size_t)r0 * G.HH, G.HH, g->w<void>(G.head4_w), G.HH, g->w<float>(G.head4_b), g->logits_ws, G.out_dim, rows,
                            G.out_dim, G.HH, LLB_ACT_NONE, true, s, &g->ctr));
      ProfScope prof(LLB_PROF_GIN_TOPK, s);
      launch_softmax_topk(g->logits_ws, rows, G.out_dim, G.out_dim, k, outv + (size_t)r0 * k, outi + (size_t)r0 * k, g->topk_redo, s);
      LLB_CUDA_OK(cudaGetLastError());
      g->launches += 3;
    }
    return LLB_OK;
  };
  g->head_flagged_rows = 0, g->head_fused_rows = 0;
  if (g->fused_rows == 0 || k > g->max_k) return materialise(g->hz, g->B, topk_prob, topk_idx);
  // ---- fused head + softmax + top-k (see EpiHeadTopk)
  const long long r_need = ((long long)7 * k * HEAD_PILOT_COLS + G.out_dim - 1) / G.out_dim;
  const int R = r_need < 4 ? 4 : (r_need > 32 ? 32 : (int)r_need);
  for (int r0 = 0; r0 < g->B; r0 += g->fused_rows) {
    const int rows = g->B - r0 < g->fused_rows ? g->B - r0 : g->fused_rows;
    const __nv_bfloat16* in = g->hz + (size_t)r0 * G.HH;
    LLB_CUDA_OK(cudaMemsetAsync(g->head_cnt, 0, (size_t)rows * 4, s));
    LLB_CUDA_OK(cudaMemsetAsync(g->head_nflag, 0, 16, s));
    g->ctr.slot = LLB_PROF_GIN_GEMM_HEAD;
    LLB_TRY(gemm_bias_act(in, G.HH, g->w<void>(G.pilot_w), G.HH, g->w<float>(G.pilot_b), g->pilot_logits, HEAD_PILOT_COLS, rows, HEAD_PILOT_COLS,
                          G.HH, LLB_ACT_NONE, true, s, &g->ctr));
    {
      ProfScope prof(LLB_PROF_GIN_TOPK, s);
      gin_head_pilot_kernel<<<rows, 1024, 0, s>>>(g->pilot_logits, R, g->rowtau);
    }
    LLB_CUDA_OK(cudaGetLastError());
    EpiHeadTopk eh{nullptr, 0, g->w<float>(G.head4_b), g->rowtau, g->head_part, g->head_slots, g->head_cand, g->head_cnt};
    g->ctr.slot = LLB_PROF_GIN_GEMM_HEAD;
    LLB_TRY((launch_gemm<256>(in, G.HH, g->w<void>(G.head4_w), G.HH, rows, G.out_dim, G.HH, eh, s, &g->ctr)));
    note_kernel(LLB_KERN_HEAD_TOPK);
    {
      ProfScope prof(LLB_PROF_GIN_TOPK, s);
      gin_head_select_kernel<<<rows, 256, 0, s>>>(g->head_part, g->head_slots, g->rowtau, g->head_cand, g->head_cnt, k, topk_prob + (size_t)r0 * k,
                                                  topk_idx + (size_t)r0 * k, g->head_flagged, g->head_nflag);
    }
    LLB_CUDA_OK(cudaGetLastError());
    g->launches += 2;
    // the one host synchronisation of this entry: did any row fall outside the threshold scheme's guarantees?
    int32_t nflag = 0;
    LLB_CUDA_OK(cudaMemcpyAsync(&nflag, g->head_nflag, 4, cudaMemcpyDeviceToHost, s));
    LLB_CUDA_OK(cudaStreamSynchronize(s));
    g->head_flagged_rows += nflag, g->head_fused_rows += rows;
    for (int f0 = 0; f0 < nflag; f0 += g->chunk_rows) {
      const int fr = nflag - f0 < g->chunk_rows ? nflag - f0 : g->chunk_rows;
      gin_gather_rows_kernel<<<fr, 128, 0, s>>>(in, g->head_flagged + f0, G.HH, g->redo_in);
      LLB_CUDA_OK(cudaGetLastError());
      LLB_TRY(materialise(g->redo_in, fr, g->redo_v, g->redo_i));
      gin_scatter_topk_kernel<<<fr, 64, 0, s>>>(g->redo_v, g->redo_i, g->head_flagged + f0, k, topk_prob + (size_t)r0 * k, topk_idx + (size_t)r0 * k);
      LLB_CUDA_OK(cudaGetLastError());
      g->launches += 2;
    }
  }
  return LLB_OK;
}

int64_t llb_gin_launch_count(const llb_gin* g) { return g ? g->launches + g->ctr.launches : 0; }

int64_t llb_gin_stat(const llb_gin* g, int which) {
  if (!g) return -1;
  switch (which) {
    case LLB_GIN_STAT_HEAD_FUSED_ROWS: return g->head_fused_rows;
    case LLB_GIN_STAT_HEAD_FLAGGED_ROWS: return g->head_flagged_rows;
    default: return -1;
  }
}

int llb_softmax_topk(const float* logits, int rows, int W, int ld, int k, float* topk_prob, int32_t* topk_idx, int32_t* scratch,
                     llb_stream_t stream) {
  LLB_TRY(require_sm100());
  LLB_CHECK_ARG(logits && topk_prob && topk_idx && scratch && rows >= 1 && W >= 1 && ld >= W && k >= 1 && k <= W,
                "llb_softmax_topk: bad argument (rows=%d W=%d ld=%d k=%d)", rows, W, ld, k);
  cudaStream_t s = (cudaStream_t)stream;
  launch_softmax_topk(logits, rows, W, ld, k, topk_prob, topk_idx, scratch, s);
  LLB_CUDA_OK(cudaGetLastError());
  return LLB_OK;
}

int llb_cost_mlp(const float* w0, const float* b0, const float* w1, const float* b1, const float* fps, int n, int fp_dim,
                 int latent, float* out, llb_stream_t stream) {
  LLB_TRY(require_sm100());
  LLB_CHECK_ARG(w0 && b0 && w1 && b1 && fps && out && n >= 1 && fp_dim >= 1 && latent >= 1 && latent <= 4096, "llb_cost_mlp: bad argument");
  cost_mlp_kernel<<<n, 256, latent * sizeof(float), (cudaStream_t)stream>>>(w0, b0, w1, b1, fps, fp_dim, latent, out);
  LLB_CUDA_OK(cudaGetLastError());
  return LLB_OK;
}

}  // extern "C"
