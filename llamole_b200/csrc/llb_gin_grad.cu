// Backward passes of the GIN modules (the forward is llb_gin.cu):
//   * the predictor with respect to the text condition c (graph_predictor/model.py:306-353 differentiated).  Only c is
//     differentiated: the parameters are constants, so every step that does not lie between c and the logits is skipped;
//   * the encoder (GraphCLIP, graph_encoder/model.py:37-41,124-205) with respect to every parameter.
// Both walk the same trunk backward (gin_trunk_backward).  Writing mod_l = Linear_l(SiLU(c)) = [shift | scale | gate] per graph
// (predictor) or the affine norms.{l} (encoder), the chain is
//   head      predictor: dhz = dlogits . W4 (split-K), LayerNorm + GELU backward, dpooled = dg . W0;
//             encoder:   L2-normalise backward -> fc2 -> GELU' + affine LayerNorm backward -> fc1;  then dh_L[i] = dpooled[batch[i]];
//   layer l   (l = L-1 .. 0) layer tail backward: GELU (not the last layer), gate, LayerNorm with (1 + scale) and shift (predictor:
//             per-graph sums give dmod_l) or with gamma, beta (encoder); the residual passes dh to dh_in_l;
//             node MLP backward du -> dz = du . W4 -> GELU' + LayerNorm(4H) backward -> da = dz_c . W0, then the transpose of the
//             aggregation over the source-sorted CSR, and the virtual node:
//             dvn_{l+1} = segsum(dh_in_{l+1}) + dvn_{l+2}, back through the virtual-node MLP to the max-pooled row, routed to
//             the node(s) that hold each column's maximum;
//   predictor: condition dctext = sum_l dmod_l . W_adapter_l (ONE GEMM: the layers' dmod side by side along K), dc = dctext * silu'(c).
//             Layer 0 stops after its tail: h_in_0 = atom_emb[x] + vn_emb, u_0's input and the layer-0 pool do not depend on c.
//   encoder:  layer 0 runs in full; dh_in_0 then gives the atom-embedding rows (sum by atom id) and, with dvn_1, the virtual-node
//             embedding (sum over graphs).
// Parameter gradients (encoder): weights dW = dY^T X over all rows (nodes or graphs) on the tcgen05 GEMM over bf16 transposes,
// split-K with the slices summed in index order (wgrad); biases and LayerNorm affines are fixed-order column sums (colsum) of
// dY and of the row products launch_row_ln_bwd writes; embedding rows and eps are per-chunk partial tables summed in chunk order.
// The 4H-wide intermediates z_l, u_l are recomputed with the forward's own kernels from the saved agg_l (storing them would
// cost 2 x 4H values per node and layer); h_in_l, agg_l, the pooled rows and mod are stored by the saved forward.
// Every sum runs in a fixed order (warp trees, segmented loops over contiguous node ranges, no float atomics), so the gradient
// is run-to-run bit-identical.  Padded columns (H % 64 != 0) stay exactly 0: the padded weights are 0 and the LayerNorm
// backward writes 0 past the true width; the parameter gradients are written at their true shapes.
#include <algorithm>
#include <initializer_list>

#include "llb_gin.cuh"
#include "llb_grad.cuh"
#include "llb_rowops.cuh"

namespace llb {
namespace {

constexpr int HEAD_GRAD_MAX_SPLIT = 32;     // K slices of the head's transposed product (dlogits . W4, K = out_dim) ...
constexpr int HEAD_GRAD_TARGET_TILES = 296; // ... halved until the slices' output tiles do not exceed two per SM (148 SMs)
constexpr int WGRAD_MAX_SPLIT = 16;         // K slices of a weight gradient (K = nodes or graphs) ...
constexpr int WGRAD_MIN_SLICE = 1024;       // ... doubled while the tiles stay within HEAD_GRAD_TARGET_TILES and a slice keeps this many rows
constexpr int GRAD_CHUNK = 256;             // rows per partial column sum (and source nodes per bond / eps partial table)
constexpr int ATOM_CHUNK = 512;             // nodes per partial atom-embedding table
constexpr int ATOM_VOCAB = 118;
constexpr int BOND_VOCAB = 5;

// Transposed bf16 copies of every weight the backward multiplies by, so that the backward GEMMs run on the forward's K-major
// tcgen05 kernels unchanged.  The predictor needs layers 1..L-1 (layer 0's MLPs do not lie between c and the logits) and the
// adapters; the encoder every layer and no adapter.
struct GinGradLayout {
  int kp;                                         // head K, padded (predictor: head_grad_kp; encoder: Hp)
  size_t head4t, head0t;                          // (HH, kp), (Hp, HH)
  std::vector<size_t> mlp4t, mlp0t;               // [l >= l0]: (I, Hp), (Hp, I)
  std::vector<size_t> vn4t, vn0t;                 // [l0 <= l < L-1]: (I, Hp), (Hp, I)
  size_t adaptert;                                // predictor: (tdim, L x 3Hp)
  size_t total;
};

void make_grad_layout(const GinLayout& G, GinGradLayout& R) {
  size_t off = 0;
  auto take = [&](size_t bytes) {
    off = align_up(off, 256);
    const size_t o = off;
    off += bytes;
    return o;
  };
  const size_t Hp = G.Hp, I = G.I;
  R.kp = G.predictor ? head_grad_kp(G) : G.HO;
  R.head4t = take((size_t)G.HH * R.kp * 2);
  R.head0t = take(Hp * G.HH * 2);
  R.mlp4t.assign(G.L, 0), R.mlp0t.assign(G.L, 0), R.vn4t.assign(G.L, 0), R.vn0t.assign(G.L, 0);
  for (int l = G.predictor ? 1 : 0; l < G.L; ++l) {
    R.mlp4t[l] = take(I * Hp * 2), R.mlp0t[l] = take(Hp * I * 2);
    if (l < G.L - 1) R.vn4t[l] = take(I * Hp * 2), R.vn0t[l] = take(Hp * I * 2);
  }
  R.adaptert = G.predictor ? take((size_t)G.tdim * G.L * 3 * Hp * 2) : 0;
  R.total = align_up(off, 256);
}

// out (n, W) = rows[batch[i]] (backward of the sum pool)
__global__ void gin_grad_gather_kernel(const float* __restrict__ rows, const int32_t* __restrict__ batch32, int n, int W,
                                       float* __restrict__ out) {
  const size_t total = (size_t)n * W;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x)
    out[idx] = rows[(size_t)batch32[idx / W] * W + idx % W];
}

// Transpose of gin_aggregate_kernel: agg_i = (1 + eps) hb_i + sum_{j->i} gelu(hb_j + bond[e_ji]) with hb = bf16(h_in), so
//   dh_in[j] += (1 + eps) da[j] + sum_{j->i} gelu'(hb_j + bond[e_ji]) da[i]
// over the source-sorted CSR (out-edges of j by edge id).  One warp per node; every warp writes only its own row.
__global__ void __launch_bounds__(256) gin_grad_aggregate_kernel(const float* __restrict__ hin, const float* __restrict__ da,
                                                                 const int32_t* __restrict__ srowptr, const int32_t* __restrict__ sdst,
                                                                 const int32_t* __restrict__ seid, const float* __restrict__ bond_emb,
                                                                 const float* __restrict__ eps_ptr, float* __restrict__ dh, int n, int W) {
  const int j = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (j >= n) return;
  const float one_eps = 1.0f + __ldg(eps_ptr);
  const int beg = srowptr[j], end = srowptr[j + 1];
  for (int c = lane; c < W; c += 32) {
    const float hb = __bfloat162float(__float2bfloat16(hin[(size_t)j * W + c]));
    float acc = dh[(size_t)j * W + c] + one_eps * da[(size_t)j * W + c];
    for (int k = beg; k < end; ++k) {
      const int i = __ldg(sdst + k), et = __ldg(seid + k) & 7;
      acc += gelu_erf_grad(hb + __ldg(bond_emb + (size_t)et * W + c)) * da[(size_t)i * W + c];
    }
    dh[(size_t)j * W + c] = acc;
  }
}

// The parameter side of the same transpose, per chunk of GRAD_CHUNK source nodes (grid (ceil(n/GRAD_CHUNK), ceil(W/256))):
//   part[chunk][t][c] = sum_{j in chunk} sum_{j->i, type t} gelu'(hb_j + bond[t]) da[i]   (t < 5: bond_encoder.{l} rows)
//   part[chunk][5][c] = sum_{j in chunk} hb_j da_j                                        (eps_l, before the sum over columns)
// Every thread owns one column of its chunk and walks the nodes and their out-edges in order.
__global__ void __launch_bounds__(256) gin_grad_bond_part_kernel(const float* __restrict__ hin, const float* __restrict__ da,
                                                                 const int32_t* __restrict__ srowptr, const int32_t* __restrict__ sdst,
                                                                 const int32_t* __restrict__ seid, const float* __restrict__ bond_emb,
                                                                 int n, int W, float* __restrict__ part) {
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= W) return;
  const int j0 = blockIdx.x * GRAD_CHUNK, j1 = j0 + GRAD_CHUNK < n ? j0 + GRAD_CHUNK : n;
  float b[BOND_VOCAB], acc[BOND_VOCAB + 1];
#pragma unroll
  for (int t = 0; t < BOND_VOCAB; ++t) b[t] = __ldg(bond_emb + (size_t)t * W + c), acc[t] = 0.f;
  acc[BOND_VOCAB] = 0.f;
  for (int j = j0; j < j1; ++j) {
    const float hb = __bfloat162float(__float2bfloat16(hin[(size_t)j * W + c]));
    acc[BOND_VOCAB] += hb * da[(size_t)j * W + c];
    for (int k = srowptr[j], end = srowptr[j + 1]; k < end; ++k) {
      const int i = __ldg(sdst + k), et = __ldg(seid + k) & 7;
      const float d = da[(size_t)i * W + c];
#pragma unroll
      for (int t = 0; t < BOND_VOCAB; ++t)
        if (et == t) acc[t] += gelu_erf_grad(hb + b[t]) * d;
    }
  }
#pragma unroll
  for (int t = 0; t <= BOND_VOCAB; ++t) part[((size_t)blockIdx.x * (BOND_VOCAB + 1) + t) * W + c] = acc[t];
}

// part[chunk][a][c] = sum_{i in chunk, x_i = a} dh[i][c] over ATOM_CHUNK nodes (grid (ceil(n/ATOM_CHUNK), ceil(W/128)), 128 threads):
// every thread accumulates its own column of a (118, 128) shared-memory table, nodes in order.
__global__ void __launch_bounds__(128) gin_grad_atom_part_kernel(const float* __restrict__ dh, const int32_t* __restrict__ x32, int n, int W,
                                                                 float* __restrict__ part) {
  extern __shared__ float tab[];
  const int t = threadIdx.x, c = blockIdx.y * 128 + t;
  for (int a = 0; a < ATOM_VOCAB; ++a) tab[a * 128 + t] = 0.f;
  if (c >= W) return;
  const int i0 = blockIdx.x * ATOM_CHUNK, i1 = i0 + ATOM_CHUNK < n ? i0 + ATOM_CHUNK : n;
  for (int i = i0; i < i1; ++i) tab[__ldg(x32 + i) * 128 + t] += dh[(size_t)i * W + c];
  for (int a = 0; a < ATOM_VOCAB; ++a) part[((size_t)blockIdx.x * ATOM_VOCAB + a) * W + c] = tab[a * 128 + t];
}

// Backward of the virtual node's max-pool (scatter_reduce amax, include_self with a -inf start): each column's gradient is split
// evenly over the nodes of the graph that hold the fp32 maximum, which is torch's rule for amax under autograd.  The forward
// pools the bf16 copy; rounding is monotone, so those nodes' bf16 value IS the pooled value.  Exact fp32 ties occur between
// automorphic nodes (the two methyls of an isopropyl group, the leaves of a star).  grid (B, ceil(W/256)).
__global__ void __launch_bounds__(256) gin_grad_route_max_kernel(const float* __restrict__ hin, const int32_t* __restrict__ graph_ptr,
                                                                 const float* __restrict__ dpool, float* __restrict__ dh, int W) {
  const int g = blockIdx.x;
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= W) return;
  const int beg = graph_ptr[g], end = graph_ptr[g + 1];
  if (beg == end) return;
  float bv = hin[(size_t)beg * W + c];
  int cnt = 1;
  for (int i = beg + 1; i < end; ++i) {
    const float v = hin[(size_t)i * W + c];
    if (v > bv) bv = v, cnt = 1;
    else if (v == bv) ++cnt;
  }
  const float share = dpool[(size_t)g * W + c] / (float)cnt;
  for (int i = beg; i < end; ++i)
    if (hin[(size_t)i * W + c] == bv) dh[(size_t)i * W + c] += share;
}

// dc = dctext * silu'(c), silu'(x) = s (1 + x (1 - s)), s = sigmoid(x)
__global__ void gin_grad_silu_kernel(const float* __restrict__ c, const float* __restrict__ dctext, float* __restrict__ dc, size_t total) {
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const float x = c[idx];
    const float sg = 1.0f / (1.0f + expf(-x));
    dc[idx] = dctext[idx] * sg * (1.0f + x * (1.0f - sg));
  }
}

// Backward of out = y / |y| (one warp per row): dy = (dout - out (out . dout)) / |y|; dout (B, H), y and dy (B, Hp), 0 past H.
__global__ void __launch_bounds__(256) gin_grad_l2norm_kernel(const float* __restrict__ y, const float* __restrict__ dout, int B, int H, int Hp,
                                                              float* __restrict__ dy, __nv_bfloat16* __restrict__ dy_b) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  const float* yr = y + (size_t)row * Hp;
  const float* dr = dout + (size_t)row * H;
  float q = 0.f, p = 0.f;
  for (int c = lane; c < H; c += 32) q += yr[c] * yr[c], p += yr[c] * dr[c];
  const float rs = rsqrtf(warp_sum(q));
  const float dot = warp_sum(p) * rs;   // out . dout
  for (int c = lane; c < Hp; c += 32) {
    const float v = c < H ? rs * (dr[c] - yr[c] * rs * dot) : 0.f;
    dy[(size_t)row * Hp + c] = v;
    dy_b[(size_t)row * Hp + c] = __float2bfloat16(v);
  }
}

// part[chunk][c] = sum of the chunk's GRAD_CHUNK rows of in (row stride ld), in row order.  grid (ceil(rows/GRAD_CHUNK), ceil(W/256)).
__global__ void __launch_bounds__(256) grad_colsum_part_kernel(const float* __restrict__ in, int ld, int rows, int W, float* __restrict__ part) {
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= W) return;
  const int r0 = blockIdx.x * GRAD_CHUNK, r1 = r0 + GRAD_CHUNK < rows ? r0 + GRAD_CHUNK : rows;
  float acc = 0.f;
  for (int r = r0; r < r1; ++r) acc += in[(size_t)r * ld + c];
  part[(size_t)blockIdx.x * W + c] = acc;
}

// out[k][c] = sum_r in[r * ld + off + k * seg + c] for k < nk, c < W, rows in order (out is (nk, W) row-major: a parameter's
// gradient at its true width).  grid ceil(nk * W / 256).
__global__ void __launch_bounds__(256) grad_colsum_kernel(const float* __restrict__ in, int rows, size_t ld, size_t off, int seg, int nk, int W,
                                                          float* __restrict__ out) {
  const int idx = blockIdx.x * 256 + threadIdx.x;
  if (idx >= nk * W) return;
  const int k = idx / W, c = idx % W;
  const float* p = in + off + (size_t)k * seg + c;
  float acc = 0.f;
  for (int r = 0; r < rows; ++r) acc += p[(size_t)r * ld];
  out[idx] = acc;
}

// out (rows_t, cols_t) = sum_s part[:, s N : s N + cols_t] in slice order (split-K partial products of a weight gradient)
__global__ void grad_slices_kernel(const float* __restrict__ part, int S, int N, int rows_t, int cols_t, float* __restrict__ out) {
  const size_t total = (size_t)rows_t * cols_t;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const size_t r = idx / cols_t, c = idx % cols_t;
    const float* p = part + r * (size_t)S * N + c;
    float acc = 0.f;
    for (int s = 0; s < S; ++s) acc += p[(size_t)s * N];
    out[idx] = acc;
  }
}

unsigned grid_for(size_t total) { return (unsigned)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096); }

// K slices of the weight gradient (M, N) = dY^T X over k rows: doubled while the output tiles of all slices fit two per SM and
// every slice keeps WGRAD_MIN_SLICE rows
int wgrad_split(int M, int N, int k) {
  const long long tiles = (long long)ceil_div(M, GEMM_BM) * ceil_div(N, 256);
  int s = 1;
  while (s < WGRAD_MAX_SPLIT && tiles * s * 2 <= HEAD_GRAD_TARGET_TILES && k >= 2 * s * WGRAD_MIN_SLICE) s *= 2;
  return s;
}

// The encoder backward's helpers over the saved buffer's scratch.
struct GradCtx {
  llb_gin* g;
  const GinSaved* sv;
  cudaStream_t s;
  LaunchCounter* ctr;

  // dst (cols, rows_out) bf16 <- src (rows, cols), zero in columns [rows, rows_out)
  template <class T>
  int tr(const T* src, int ld_s, int rows, int cols, __nv_bfloat16* dst, int rows_out) {
    return launch_kernel(ctr, NO_PROF, false, grad_transpose_kernel<T>, dim3(ceil_div(cols, 32), ceil_div(rows_out, 32)), dim3(32, 8), 0, s, src, ld_s,
                         rows, cols, dst, rows_out, rows_out);
  }
  // Column sums of in (rows, W) into the parameters' gradients: for every (off, Wt, out) of `outs`, out[c] = sum over the rows of
  // column off + c, c < Wt.  Partial sums over GRAD_CHUNK-row chunks, then the chunks in order.
  struct Out {
    int off, Wt;
    float* out;
  };
  int colsum(const float* in, int ld, int rows, int W, std::initializer_list<Out> outs) {
    const int nch = ceil_div(rows, GRAD_CHUNK);
    LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_colsum_part_kernel, dim3(nch, ceil_div(W, 256)), dim3(256), 0, s, in, ld, rows, W, sv->cpart));
    for (const Out& o : outs) LLB_TRY(sum_rows(sv->cpart, nch, W, o.off, 0, 1, o.Wt, o.out));
    return LLB_OK;
  }
  int sum_rows(const float* in, int rows, size_t ld, size_t off, int seg, int nk, int W, float* out) {
    return launch_kernel(ctr, NO_PROF, false, grad_colsum_kernel, dim3(ceil_div(nk * W, 256)), dim3(256), 0, s, in, rows, ld, off, seg, nk, W, out);
  }
  // out (rows_t, cols_t) fp32 = dY^T X over k rows: dY (k, M) row stride ldy, X (k, N) row stride ldx; M, N padded widths
  template <class TY, class TX>
  int wgrad(const TY* dY, int ldy, int M, const TX* X, int ldx, int N, int k, int rows_t, int cols_t, float* out) {
    const int S = wgrad_split(M, N, k);
    const int kp = (int)align_up((size_t)k, 64 * S);   // every slice a multiple of the K tile
    LLB_CHECK_ARG(kp <= sv->kmax, "gin: weight-gradient K %d exceeds the saved buffer's %d", kp, sv->kmax);
    LLB_TRY(tr(dY, ldy, k, M, sv->tA, kp));
    LLB_TRY(tr(X, ldx, k, N, sv->tW, kp));
    GemmGroups split;
    split.group_n = N, split.group_k = kp / S, split.split_k = true;
    LLB_TRY(gemm_bias_act(sv->tA, kp, sv->tW, kp, nullptr, sv->wpart, S * N, M, S * N, kp / S, LLB_ACT_NONE, true, s, ctr, split));
    return launch_kernel(ctr, NO_PROF, false, grad_slices_kernel, grid_for((size_t)rows_t * cols_t), dim3(256), 0, s, sv->wpart, S, N, rows_t,
                         cols_t, out);
  }
};

// Layers L-1 .. 0 of the backward, sv.dh = dL/d(trunk output) on entry.  P == null (predictor): the gradient with respect to c
// only (dmod in sv.dmod_b; layer 0 stops after its tail).  P != null (encoder): every parameter's gradient into P.
int gin_trunk_backward(GradCtx& X, const uint8_t* wt, const GinGradLayout& R, int n, int B, const llb_gin_encoder_grads* P) {
  llb_gin* g = X.g;
  const GinSaved& sv = *X.sv;
  const GinLayout& G = g->G;
  cudaStream_t s = X.s;
  LaunchCounter* ctr = X.ctr;
  const int L = G.L, H = G.H, Hp = G.Hp, I = G.I;
  auto gw = [&](size_t off) { return (const void*)(wt + off); };
  const dim3 seg_grid_h(B, ceil_div(Hp, 256));
  for (int l = L - 1; l >= 0; --l) {
    const bool last = l == L - 1;
    const float* hin = l >= sv.hin_l0 ? sv.hin + (size_t)(l - sv.hin_l0) * n * Hp : nullptr;
    if (!last) {
      // vn_{l+1} is added to every node of h_in_{l+1} and carried into vn_{l+2}
      LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, seg_grid_h, dim3(256), 0, s, sv.dh, Hp, sv.graph_ptr, Hp,
                            l < L - 2 ? sv.dvn : nullptr, sv.dvn, sv.dvn_b, Hp));
      if (l > 0 || P) {
        // vn_{l+1} = vn_l + MLP_l(maxpool(h_in_l)): back through the MLP to the pooled row (routed below)
        const __nv_bfloat16* pool = sv.pool + (size_t)l * B * Hp;
        g->ctr.slot = LLB_PROF_GIN_MISC;
        LLB_TRY(gemm_bias_act(pool, Hp, g->w<void>(G.vn0_w[l]), Hp, g->w<float>(G.vn0_b[l]), sv.vz, I, B, I, Hp, LLB_ACT_NONE, false, s, &g->ctr));
        LLB_TRY(gemm_bias_act(sv.dvn_b, Hp, gw(R.vn4t[l]), Hp, nullptr, sv.dvz, I, B, I, Hp, LLB_ACT_NONE, true, s, &g->ctr));
        if (P) {
          // fc2's input GELU(LN(vz)), recomputed with the forward's row kernel
          RowLnArgs f;
          f.in = sv.vz, f.in_ld = I, f.in_bf16 = true, f.rows = B, f.width = I, f.valid = 4 * H;
          f.gamma = g->w<float>(G.vn_ln_w[l]), f.beta = g->w<float>(G.vn_ln_b[l]), f.act = LLB_ACT_GELU;
          f.out_bf16 = sv.vz_post, f.out_bf16_ld = I;
          f.prof_slot = LLB_PROF_GIN_ROWLN;
          LLB_TRY(launch_row_ln(f, s, ctr));
          LLB_TRY(X.wgrad(sv.dvn, Hp, Hp, sv.vz_post, I, I, B, H, 4 * H, P->vn4_w[l]));
          LLB_TRY(X.colsum(sv.dvn, Hp, B, Hp, {{0, H, P->vn4_b[l]}}));
        }
        RowLnBwdArgs a;
        a.x = sv.vz, a.x_ld = I, a.x_bf16 = true, a.dy = sv.dvz, a.dy_ld = I;
        a.rows = B, a.width = I, a.valid = 4 * H;
        a.gamma = g->w<float>(G.vn_ln_w[l]), a.beta = g->w<float>(G.vn_ln_b[l]), a.gelu = true;
        a.out_bf16 = sv.dvz_b, a.out_ld = I;
        if (P) a.out_f32 = sv.dvz, a.prod = sv.prod, a.prod_ld = 2 * I, a.prod_sets = 2;
        LLB_TRY(launch_row_ln_bwd(a, s, ctr));
        if (P) {
          LLB_TRY(X.colsum(sv.prod, 2 * I, B, 2 * I, {{0, 4 * H, P->vn_ln_b[l]}, {I, 4 * H, P->vn_ln_w[l]}}));
          LLB_TRY(X.colsum(sv.dvz, I, B, I, {{0, 4 * H, P->vn0_b[l]}}));
          LLB_TRY(X.wgrad(sv.dvz, I, I, pool, Hp, Hp, B, 4 * H, H, P->vn0_w[l]));
        }
        LLB_TRY(gemm_bias_act(sv.dvz_b, I, gw(R.vn0t[l]), I, nullptr, sv.dpool, Hp, B, Hp, I, LLB_ACT_NONE, true, s, &g->ctr));
      }
    }
    // node MLP output u_l, recomputed from the saved aggregation with the forward's kernels
    const __nv_bfloat16* agg = sv.agg + (size_t)l * n * Hp;
    LLB_TRY(gin_node_mlp(g, agg, n, l, sv.ln_part, sv.z, sv.u, Hp, false, LLB_PROF_GIN_GEMM_MLP0, LLB_PROF_GIN_GEMM_MLP4, s));
    {
      // layer tail: h_out = gate * act(LN(u) (1 + scale) + shift) + h_in (+ vn_{l+1})   (predictor)
      //             h_out = act(LN(u) gamma + beta) + h_in (+ vn_{l+1})                  (encoder)
      RowLnBwdArgs a;
      a.x = sv.u, a.x_ld = Hp, a.dy = sv.dh, a.dy_ld = Hp;
      a.rows = n, a.width = Hp, a.valid = H;
      a.gelu = !last;
      if (G.predictor) {
        const float* mod = sv.mod + (size_t)l * B * 3 * Hp;
        a.row_group = sv.batch32, a.shift = mod, a.scale = mod + Hp, a.gate = mod + 2 * Hp, a.mod_ld = 3 * Hp;
        a.prod = sv.prod, a.prod_ld = 3 * Hp;
      } else {
        a.gamma = g->w<float>(G.norm_w[l]), a.beta = g->w<float>(G.norm_b[l]);
        a.prod = sv.prod, a.prod_ld = 2 * Hp, a.prod_sets = 2;
        a.out_f32 = sv.u;   // du over u, in place (u is not needed past this point)
      }
      if (l > 0 || P) a.out_bf16 = sv.du_b, a.out_ld = Hp;
      LLB_TRY(launch_row_ln_bwd(a, s, ctr));
      if (G.predictor)
        LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, dim3(B, ceil_div(3 * Hp, 256)), dim3(256), 0, s, sv.prod, 3 * Hp, sv.graph_ptr,
                              3 * Hp, nullptr, nullptr, sv.dmod_b + (size_t)l * 3 * Hp, L * 3 * Hp));
    }
    if (P) {
      LLB_TRY(X.colsum(sv.prod, 2 * Hp, n, 2 * Hp, {{0, H, P->norm_b[l]}, {Hp, H, P->norm_w[l]}}));
      LLB_TRY(X.colsum(sv.u, Hp, n, Hp, {{0, H, P->mlp4_b[l]}}));
      g->ctr.slot = LLB_PROF_GIN_GEMM_MLP4;
      LLB_TRY(X.wgrad(sv.u, Hp, Hp, reinterpret_cast<const __half*>(sv.z), I, I, n, H, 4 * H, P->mlp4_w[l]));
    } else if (l == 0) {
      break;   // nothing upstream of layer 0's tail depends on c
    }
    // node MLP: du -> dz = du . W4 -> GELU' + LayerNorm(4H) backward on the centred first linear's output -> da = dz_c . W0c
    // (the LayerNorm backward sums to zero over the 4H columns, so the centred weight gives the same product as W0)
    g->ctr.slot = LLB_PROF_GIN_GEMM_MLP0;
    LLB_TRY(gemm_bias_act(agg, Hp, g->w<void>(G.mlp0_w[l]), Hp, g->w<float>(G.mlp0_b[l]), sv.zpre, I, n, I, Hp, LLB_ACT_NONE, true, s, &g->ctr));
    g->ctr.slot = LLB_PROF_GIN_GEMM_MLP4;
    LLB_TRY(gemm_bias_act(sv.du_b, Hp, gw(R.mlp4t[l]), Hp, nullptr, sv.dz, I, n, I, Hp, LLB_ACT_NONE, true, s, &g->ctr));
    {
      RowLnBwdArgs a;
      a.x = sv.zpre, a.x_ld = I, a.dy = sv.dz, a.dy_ld = I;
      a.rows = n, a.width = I, a.valid = 4 * H;
      a.gamma = g->w<float>(G.mlp_ln_w[l]), a.beta = g->w<float>(G.mlp_ln_b[l]), a.gelu = true;
      a.out_bf16 = sv.dzpre_b, a.out_ld = I;
      if (P) a.out_f32 = sv.dz, a.prod = sv.prod, a.prod_ld = 2 * I, a.prod_sets = 2;
      LLB_TRY(launch_row_ln_bwd(a, s, ctr));
    }
    if (P) {
      LLB_TRY(X.colsum(sv.prod, 2 * I, n, 2 * I, {{0, 4 * H, P->mlp_ln_b[l]}, {I, 4 * H, P->mlp_ln_w[l]}}));
      LLB_TRY(X.colsum(sv.dz, I, n, I, {{0, 4 * H, P->mlp0_b[l]}}));
      g->ctr.slot = LLB_PROF_GIN_GEMM_MLP0;
      LLB_TRY(X.wgrad(sv.dz, I, I, agg, Hp, Hp, n, 4 * H, H, P->mlp0_w[l]));
    }
    g->ctr.slot = LLB_PROF_GIN_GEMM_MLP0;
    LLB_TRY(gemm_bias_act(sv.dzpre_b, I, gw(R.mlp0t[l]), I, nullptr, sv.da, Hp, n, Hp, I, LLB_ACT_NONE, true, s, &g->ctr));
    if (P) {
      // bond_encoder.{l} rows and eps_l: per-chunk tables, then the chunks in order (eps: then its columns in order)
      const int nch = ceil_div(n, GRAD_CHUNK);
      LLB_TRY(launch_kernel(ctr, LLB_PROF_GIN_AGGREGATE, false, gin_grad_bond_part_kernel, dim3(nch, ceil_div(Hp, 256)), dim3(256), 0, s, hin, sv.da,
                            sv.srowptr, sv.sdst, sv.seid, g->w<float>(G.bond_emb[l]), n, Hp, sv.bpart));
      LLB_TRY(X.sum_rows(sv.bpart, nch, (size_t)(BOND_VOCAB + 1) * Hp, 0, Hp, BOND_VOCAB, H, P->bond_emb[l]));
      LLB_TRY(X.sum_rows(sv.bpart, nch, (size_t)(BOND_VOCAB + 1) * Hp, (size_t)BOND_VOCAB * Hp, 0, 1, H, sv.evec));
      LLB_TRY(X.sum_rows(sv.evec, H, 1, 0, 0, 1, 1, P->eps[l]));
    }
    LLB_TRY(launch_kernel(ctr, LLB_PROF_GIN_AGGREGATE, false, gin_grad_aggregate_kernel, dim3(ceil_div(n, 8)), dim3(256), 0, s, hin, sv.da, sv.srowptr,
                          sv.sdst, sv.seid, g->w<float>(G.bond_emb[l]), g->w<float>(G.eps[l]), sv.dh, n, Hp));
    if (!last)
      LLB_TRY(launch_kernel(ctr, LLB_PROF_GIN_POOL, false, gin_grad_route_max_kernel, seg_grid_h, dim3(256), 0, s, hin, sv.graph_ptr, sv.dpool, sv.dh,
                            Hp));
  }
  if (!P) return LLB_OK;
  // h_in_0 = atom_emb[x] + vn_0[batch], vn_0 = vn_emb for every graph, vn_1 = vn_0 + MLP_0(...): sv.dh = dL/dh_in_0, sv.dvn = dL/dvn_1
  const int nca = ceil_div(n, ATOM_CHUNK);
  LLB_TRY(launch_kernel(ctr, NO_PROF, false, gin_grad_atom_part_kernel, dim3(nca, ceil_div(Hp, 128)), dim3(128), (size_t)ATOM_VOCAB * 128 * 4, s,
                        sv.dh, sv.x32, n, Hp, sv.apart));
  LLB_TRY(X.sum_rows(sv.apart, nca, (size_t)ATOM_VOCAB * Hp, 0, Hp, ATOM_VOCAB, H, P->atom_emb));
  LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, seg_grid_h, dim3(256), 0, s, sv.dh, Hp, sv.graph_ptr, Hp, sv.dvn, sv.dvn,
                        (__nv_bfloat16*)nullptr, Hp));
  return X.sum_rows(sv.dvn, B, Hp, 0, 0, 1, H, P->vn_emb);
}

}  // namespace

int head_grad_kp(const GinLayout& G) { return (int)align_up((size_t)G.out_dim, 64 * HEAD_GRAD_MAX_SPLIT); }

int head_grad_split(const GinLayout& G, int B) {
  const long long tiles = (long long)ceil_div(B, GEMM_BM) * ceil_div(G.HH, 256);
  int s = HEAD_GRAD_MAX_SPLIT;
  while (s > 1 && tiles * s > HEAD_GRAD_TARGET_TILES) s >>= 1;
  return s;
}

size_t gin_grad_weights_bytes(const GinLayout& G) {
  GinGradLayout R;
  make_grad_layout(G, R);
  return R.total;
}

int gin_pack_grad_weights(llb_gin* g, void* blob, cudaStream_t s) {
  const GinLayout& G = g->G;
  GinGradLayout R;
  make_grad_layout(G, R);
  uint8_t* base = (uint8_t*)blob;
  auto dst = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(base + off); };
  auto tr = [&](const auto* src, int ld_s, int rows, int cols, __nv_bfloat16* d, int ld_d) {
    using T = std::remove_const_t<std::remove_pointer_t<decltype(src)>>;
    return launch_kernel(&g->ctr, NO_PROF, false, grad_transpose_kernel<T>, dim3(ceil_div(cols, 32), ceil_div(rows, 32)), dim3(32, 8), 0, s, src,
                         ld_s, rows, cols, d, ld_d, rows);
  };
  const int Hp = G.Hp, I = G.I, HH = G.HH;
  LLB_CUDA_OK(cudaMemsetAsync(base, 0, R.total, s));   // the head's K padding past out_dim is zero
  LLB_TRY(tr(g->w<__nv_bfloat16>(G.head4_w), HH, G.HO, HH, dst(R.head4t), R.kp));
  LLB_TRY(tr(g->w<__nv_bfloat16>(G.head0_w), Hp, HH, Hp, dst(R.head0t), HH));
  for (int l = G.predictor ? 1 : 0; l < G.L; ++l) {
    LLB_TRY(tr(g->w<__half>(G.mlp4_w[l]), I, Hp, I, dst(R.mlp4t[l]), Hp));   // the forward's copy is fp16 (see EpiLnGelu)
    LLB_TRY(tr(g->w<__nv_bfloat16>(G.mlp0_w[l]), Hp, I, Hp, dst(R.mlp0t[l]), I));
    if (l < G.L - 1) {
      LLB_TRY(tr(g->w<__nv_bfloat16>(G.vn4_w[l]), I, Hp, I, dst(R.vn4t[l]), Hp));
      LLB_TRY(tr(g->w<__nv_bfloat16>(G.vn0_w[l]), Hp, I, Hp, dst(R.vn0t[l]), I));
    }
  }
  if (G.predictor)
    for (int l = 0; l < G.L; ++l)
      LLB_TRY(tr(g->w<__nv_bfloat16>(G.adapter_w[l]), G.tdim, 3 * Hp, G.tdim, dst(R.adaptert) + (size_t)l * 3 * Hp, G.L * 3 * Hp));
  return LLB_OK;
}

void gin_saved_carve(const GinLayout& G, void* saved, int n, int e, int B, GinSaved* sv, size_t* bytes) {
  GinSaved tmp{};
  GinSaved& v = sv ? *sv : tmp;
  v = GinSaved{};
  const bool P = G.predictor != 0;
  const size_t H = G.Hp, I = G.I, L = G.L, N = n, R = n > B ? n : B;
  Arena a(saved, 0);
  v.graph_ptr = a.take<int32_t>(B + 1), v.batch32 = a.take<int32_t>(N);
  v.srowptr = a.take<int32_t>(N + 1), v.sdst = a.take<int32_t>(e > 0 ? e : 1), v.seid = a.take<int32_t>(e > 0 ? e : 1);
  v.hin_l0 = P ? 1 : 0;
  v.hin = a.take<float>((L - v.hin_l0) * N * H);
  v.agg = a.take<__nv_bfloat16>(L * N * H);
  v.pool = a.take<__nv_bfloat16>((L - 1) * B * H);
  v.mod = a.take<float>(P ? L * B * 3 * H : 0);
  v.pooled_b = a.take<__nv_bfloat16>((size_t)B * H);
  v.head_split = P ? head_grad_split(G, B) : 1;
  v.dlog_b = a.take<__nv_bfloat16>(P ? (size_t)B * head_grad_kp(G) : 0);
  v.dhz_parts = a.take<float>((size_t)B * v.head_split * G.HH);   // the encoder's head: dL/d(fc2 input), then its LayerNorm input
  v.hz_pre = a.take<__nv_bfloat16>((size_t)B * G.HH), v.dhz_pre = a.take<__nv_bfloat16>((size_t)B * G.HH);
  v.dpooled = a.take<float>((size_t)B * H);
  v.dh = a.take<float>(N * H);
  v.dvn = a.take<float>((size_t)B * H), v.dpool = a.take<float>((size_t)B * H), v.dvn_b = a.take<__nv_bfloat16>((size_t)B * H);
  v.vz = a.take<__nv_bfloat16>((size_t)B * I), v.dvz_b = a.take<__nv_bfloat16>((size_t)B * I), v.dvz = a.take<float>((size_t)B * I);
  v.z = a.take<__nv_bfloat16>(N * I);
  v.u = a.take<float>(N * H);
  v.ln_part = a.take<float>(N * ceil_div((int)H, 256) * (GEMM_EPI_WARPS / 4));   // = llb_gin::ln_slots
  v.zpre = a.take<float>(N * I), v.dz = a.take<float>(N * I), v.dzpre_b = a.take<__nv_bfloat16>(N * I);
  v.prod = a.take<float>(P ? N * 3 * H : R * 2 * I);   // encoder: [dt | dt xh] of the 4H LayerNorms (and of the narrower ones)
  v.du_b = a.take<__nv_bfloat16>(N * H);
  v.da = a.take<float>(N * H);
  v.dmod_b = a.take<__nv_bfloat16>(P ? (size_t)B * L * 3 * H : 0);
  v.dctext = a.take<float>(P ? (size_t)B * G.tdim : 0);
  if (!P) {
    v.x32 = a.take<int32_t>(N);
    v.y = a.take<float>((size_t)B * H);
    v.wt = a.take<uint8_t>(gin_grad_weights_bytes(G));
    v.hz_post = a.take<__nv_bfloat16>((size_t)B * H), v.vz_post = a.take<__nv_bfloat16>((size_t)B * I);
    v.dyh = a.take<float>((size_t)B * H), v.dyh_b = a.take<__nv_bfloat16>((size_t)B * H);
    v.kmax = (int)align_up(R, 64 * WGRAD_MAX_SPLIT);
    v.tA = a.take<__nv_bfloat16>(I * v.kmax), v.tW = a.take<__nv_bfloat16>(I * v.kmax);
    // split-K partials: S x M x N <= (2 x 148 tiles of 128 x 256) once S > 1, M x N <= I x Hp at S = 1
    v.wpart = a.take<float>(std::max(I * H, (size_t)HEAD_GRAD_TARGET_TILES * GEMM_BM * 256));
    v.cpart = a.take<float>((size_t)ceil_div((int)R, GRAD_CHUNK) * 2 * I);
    v.apart = a.take<float>((size_t)ceil_div(n, ATOM_CHUNK) * ATOM_VOCAB * H);
    v.bpart = a.take<float>((size_t)ceil_div(n, GRAD_CHUNK) * (BOND_VOCAB + 1) * H);
    v.evec = a.take<float>(H);
  }
  *bytes = align_up(a.off, 256);
}

}  // namespace llb

using namespace llb;

extern "C" {

int llb_gin_grad_packed_bytes(const llb_gin_config* cfg, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes, "llb_gin_grad_packed_bytes: null argument");
  LLB_CHECK_ARG(cfg->predictor, "llb_gin_grad_packed_bytes: only the predictor has a backward");
  GinLayout G;
  LLB_TRY(make_layout(*cfg, G));
  *bytes = gin_grad_weights_bytes(G);
  return LLB_OK;
}

int llb_gin_pack_grad_weights(llb_gin* g, void* grad_blob, size_t grad_bytes, llb_stream_t stream) {
  LLB_CHECK_ARG(g && grad_blob && g->G.predictor, "llb_gin_pack_grad_weights: needs a predictor handle and a blob");
  const size_t need = gin_grad_weights_bytes(g->G);
  if (grad_bytes < need) return fail(LLB_ERR_WORKSPACE, "gin: grad blob needs %zu bytes, got %zu", need, grad_bytes);
  return gin_pack_grad_weights(g, grad_blob, (cudaStream_t)stream);
}

int llb_gin_predictor_backward_c(llb_gin* g, int num_nodes, int num_edges, int num_graphs, const float* c, const float* dlogits,
                                 void* saved, size_t saved_bytes, const void* grad_blob, size_t grad_bytes, float* dc,
                                 llb_stream_t stream) {
  LLB_CHECK_ARG(g && g->G.predictor && dlogits && saved && grad_blob && dc, "llb_gin_predictor_backward_c: null argument or not a predictor");
  if (!c) return fail(LLB_ERR_INVALID, "llb_gin_predictor_backward_c: c is NULL (the text_dropping row is a parameter, not an input)");
  LLB_CHECK_ARG(num_nodes >= 1 && num_edges >= 0 && num_graphs >= 1, "llb_gin_predictor_backward_c: bad batch size");
  const GinLayout& G = g->G;
  GinGradLayout R;
  make_grad_layout(G, R);
  if (grad_bytes < R.total) return fail(LLB_ERR_WORKSPACE, "gin: grad blob needs %zu bytes, got %zu", R.total, grad_bytes);
  const int n = num_nodes, B = num_graphs, L = G.L, Hp = G.Hp, HH = G.HH;
  GinSaved sv;
  size_t need = 0;
  gin_saved_carve(G, saved, n, num_edges, B, &sv, &need);
  if (saved_bytes < need) return fail(LLB_ERR_WORKSPACE, "gin: saved buffer needs %zu bytes, got %zu", need, saved_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  const uint8_t* gb = (const uint8_t*)grad_blob;
  auto gw = [&](size_t off) { return (const void*)(gb + off); };
  LaunchCounter* ctr = &g->ctr;
  ctr->slot = LLB_PROF_GIN_MISC;

  // ---- head: dhz = dlogits . W4 as head_split K slices (M = B is one or two row blocks; one slice would run on a few CTAs)
  {
    const int kp = R.kp, S = sv.head_split, kslice = kp / S;
    LLB_TRY(launch_f32_to_bf16(dlogits, G.out_dim, sv.dlog_b, kp, B, G.out_dim, kp, s, ctr));
    GemmGroups split;
    split.group_n = HH, split.group_k = kslice, split.split_k = true;
    g->ctr.slot = LLB_PROF_GIN_GEMM_HEAD;
    LLB_TRY(gemm_bias_act(sv.dlog_b, kp, gw(R.head4t), kp, nullptr, sv.dhz_parts, S * HH, B, S * HH, kslice, LLB_ACT_NONE, true, s, &g->ctr, split));
    // decoder.0's output (bf16, as the forward's row kernel read it), recomputed
    LLB_TRY(gemm_bias_act(sv.pooled_b, Hp, g->w<void>(G.head0_w), Hp, g->w<float>(G.head0_b), sv.hz_pre, HH, B, HH, Hp, LLB_ACT_NONE, false, s,
                          &g->ctr));
    RowLnBwdArgs a;
    a.x = sv.hz_pre, a.x_ld = HH, a.x_bf16 = true;
    a.dy = sv.dhz_parts, a.dy_ld = S * HH, a.dy_parts = S, a.dy_part_stride = HH;
    a.rows = B, a.width = HH, a.valid = G.HHt;
    a.gamma = g->w<float>(G.head_ln_w), a.beta = g->w<float>(G.head_ln_b), a.gelu = true;
    a.out_bf16 = sv.dhz_pre, a.out_ld = HH;
    LLB_TRY(launch_row_ln_bwd(a, s, ctr));
    LLB_TRY(gemm_bias_act(sv.dhz_pre, HH, gw(R.head0t), HH, nullptr, sv.dpooled, Hp, B, Hp, HH, LLB_ACT_NONE, true, s, &g->ctr));
    LLB_TRY(launch_kernel(ctr, NO_PROF, false, gin_grad_gather_kernel, grid_for((size_t)n * Hp), dim3(256), 0, s, sv.dpooled, sv.batch32, n, Hp,
                          sv.dh));
  }
  GradCtx X{g, &sv, s, ctr};
  LLB_TRY(gin_trunk_backward(X, gb, R, n, B, nullptr));
  // ---- condition: dctext = [dmod_0 | ... | dmod_{L-1}] . [W_adapter_0 | ... ]^T, dc = dctext * silu'(c)
  g->ctr.slot = LLB_PROF_GIN_MISC;
  LLB_TRY(gemm_bias_act(sv.dmod_b, L * 3 * Hp, gw(R.adaptert), L * 3 * Hp, nullptr, sv.dctext, G.tdim, B, G.tdim, L * 3 * Hp, LLB_ACT_NONE, true,
                        s, &g->ctr));
  return launch_kernel(ctr, NO_PROF, false, gin_grad_silu_kernel, grid_for((size_t)B * G.tdim), dim3(256), 0, s, c, sv.dctext, dc,
                       (size_t)B * G.tdim);
}

int llb_gin_encoder_backward(llb_gin* g, int num_nodes, int num_edges, int num_graphs, const float* d_out, void* saved, size_t saved_bytes,
                             const llb_gin_encoder_grads* grads, llb_stream_t stream) {
  LLB_CHECK_ARG(g && !g->G.predictor && d_out && saved && grads, "llb_gin_encoder_backward: null argument or not an encoder");
  LLB_CHECK_ARG(num_nodes >= 1 && num_edges >= 0 && num_graphs >= 1, "llb_gin_encoder_backward: bad batch size");
  const llb_gin_encoder_grads* P = grads;
  LLB_CHECK_ARG(P->atom_emb && P->vn_emb && P->eps && P->mlp0_w && P->mlp0_b && P->mlp_ln_w && P->mlp_ln_b && P->mlp4_w && P->mlp4_b &&
                    P->bond_emb && P->norm_w && P->norm_b && P->vn0_w && P->vn0_b && P->vn_ln_w && P->vn_ln_b && P->vn4_w && P->vn4_b &&
                    P->head0_w && P->head0_b && P->head_ln_w && P->head_ln_b && P->head4_w && P->head4_b,
                "llb_gin_encoder_backward: every gradient pointer (and per-layer array) must be set");
  const GinLayout& G = g->G;
  GinGradLayout R;
  make_grad_layout(G, R);
  const int n = num_nodes, B = num_graphs, H = G.H, Hp = G.Hp;
  GinSaved sv;
  size_t need = 0;
  gin_saved_carve(G, saved, n, num_edges, B, &sv, &need);
  if (saved_bytes < need) return fail(LLB_ERR_WORKSPACE, "gin: saved buffer needs %zu bytes, got %zu", need, saved_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  auto gw = [&](size_t off) { return (const void*)(sv.wt + off); };
  LaunchCounter* ctr = &g->ctr;
  GradCtx X{g, &sv, s, ctr};

  // ---- projection head: out = y / |y|, y = fc2(GELU(LN(fc1(pooled))))
  ctr->slot = LLB_PROF_GIN_GEMM_HEAD;
  LLB_TRY(launch_kernel(ctr, NO_PROF, false, gin_grad_l2norm_kernel, dim3(ceil_div(B, 8)), dim3(256), 0, s, sv.y, d_out, B, H, Hp, sv.dyh, sv.dyh_b));
  // fc1's output (bf16, as the forward's row kernel read it) and fc2's input GELU(LN(.)), recomputed with the forward's kernels
  LLB_TRY(gemm_bias_act(sv.pooled_b, Hp, g->w<void>(G.head0_w), Hp, g->w<float>(G.head0_b), sv.hz_pre, Hp, B, Hp, Hp, LLB_ACT_NONE, false, s, ctr));
  {
    RowLnArgs f;
    f.in = sv.hz_pre, f.in_ld = Hp, f.in_bf16 = true, f.rows = B, f.width = Hp, f.valid = H;
    f.gamma = g->w<float>(G.head_ln_w), f.beta = g->w<float>(G.head_ln_b), f.act = LLB_ACT_GELU;
    f.out_bf16 = sv.hz_post, f.out_bf16_ld = Hp;
    f.prof_slot = LLB_PROF_GIN_ROWLN;
    LLB_TRY(launch_row_ln(f, s, ctr));
  }
  LLB_TRY(X.wgrad(sv.dyh, Hp, Hp, sv.hz_post, Hp, Hp, B, H, H, P->head4_w));
  LLB_TRY(X.colsum(sv.dyh, Hp, B, Hp, {{0, H, P->head4_b}}));
  float* dhz = sv.dhz_parts;
  LLB_TRY(gemm_bias_act(sv.dyh_b, Hp, gw(R.head4t), Hp, nullptr, dhz, Hp, B, Hp, Hp, LLB_ACT_NONE, true, s, ctr));
  {
    RowLnBwdArgs a;
    a.x = sv.hz_pre, a.x_ld = Hp, a.x_bf16 = true, a.dy = dhz, a.dy_ld = Hp;
    a.rows = B, a.width = Hp, a.valid = H;
    a.gamma = g->w<float>(G.head_ln_w), a.beta = g->w<float>(G.head_ln_b), a.gelu = true;
    a.out_bf16 = sv.dhz_pre, a.out_f32 = dhz, a.out_ld = Hp;
    a.prod = sv.prod, a.prod_ld = 2 * Hp, a.prod_sets = 2;
    LLB_TRY(launch_row_ln_bwd(a, s, ctr));
  }
  LLB_TRY(X.colsum(sv.prod, 2 * Hp, B, 2 * Hp, {{0, H, P->head_ln_b}, {Hp, H, P->head_ln_w}}));
  LLB_TRY(X.colsum(dhz, Hp, B, Hp, {{0, H, P->head0_b}}));
  LLB_TRY(X.wgrad(dhz, Hp, Hp, sv.pooled_b, Hp, Hp, B, H, H, P->head0_w));
  LLB_TRY(gemm_bias_act(sv.dhz_pre, Hp, gw(R.head0t), Hp, nullptr, sv.dpooled, Hp, B, Hp, Hp, LLB_ACT_NONE, true, s, ctr));
  LLB_TRY(launch_kernel(ctr, NO_PROF, false, gin_grad_gather_kernel, grid_for((size_t)n * Hp), dim3(256), 0, s, sv.dpooled, sv.batch32, n, Hp, sv.dh));
  return gin_trunk_backward(X, sv.wt, R, n, B, P);
}

}  // extern "C"
