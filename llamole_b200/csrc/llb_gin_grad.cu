// Backward of the GIN predictor with respect to the text condition c (graph_predictor/model.py:306-353 differentiated; the
// forward is llb_gin.cu).  Only c is differentiated: the parameters are constants, so every step that does not lie between c
// and the logits is skipped.  Writing mod_l = Linear_l(SiLU(c)) = [shift | scale | gate] per graph, the chain is
//   head      dhz = dlogits . W4 (split-K), LayerNorm + GELU backward, dpooled = dg . W0, dh_L[i] = dpooled[batch[i]];
//   layer l   (l = L-1 .. 0) layer tail backward: GELU (not the last layer), gate, non-affine LayerNorm with (1 + scale) and shift;
//             per-graph sums give dmod_l; the residual passes dh to dh_in_l;
//             (l >= 1) node MLP backward du -> dz = du . W4 -> GELU' + LayerNorm(4H) backward -> da = dz_c . W0, then the
//             transpose of the aggregation over the source-sorted CSR, and the virtual node:
//             dvn_{l+1} = segsum(dh_in_{l+1}) + dvn_{l+2}, back through the virtual-node MLP to the max-pooled row, routed to
//             the node that holds each column's maximum;
//   condition dctext = sum_l dmod_l . W_adapter_l (ONE GEMM: the layers' dmod side by side along K), dc = dctext * silu'(c).
// Layer 0 stops after its tail: h_in_0 = atom_emb[x] + vn_emb, u_0's input and the layer-0 pool do not depend on c.
// The 4H-wide intermediates z_l, u_l are recomputed with the forward's own kernels from the saved agg_l (storing them would
// cost 2 x 4H values per node and layer); h_in_l, agg_l, the pooled rows and mod are stored by the saved forward.
// Every sum runs in a fixed order (warp trees, segmented loops over contiguous node ranges, no float atomics), so the gradient
// is run-to-run bit-identical.  Padded columns (H % 64 != 0) stay exactly 0: the padded weights are 0 and the LayerNorm
// backward writes 0 past the true width.
#include "llb_gin.cuh"
#include "llb_grad.cuh"
#include "llb_rowops.cuh"

namespace llb {
namespace {

constexpr int HEAD_GRAD_MAX_SPLIT = 32;     // K slices of the head's transposed product (dlogits . W4, K = out_dim) ...
constexpr int HEAD_GRAD_TARGET_TILES = 296; // ... halved until the slices' output tiles do not exceed two per SM (148 SMs)

// Transposed bf16 copies of every weight the backward multiplies by, so that the backward GEMMs run on the forward's K-major
// tcgen05 kernels unchanged.
struct GinGradLayout {
  int kp;                                         // head K, padded (head_grad_kp)
  size_t head4t, head0t;                          // (HH, kp), (Hp, HH)
  std::vector<size_t> mlp4t, mlp0t;               // [l >= 1]: (I, Hp), (Hp, I)
  std::vector<size_t> vn4t, vn0t;                 // [1 <= l < L-1]: (I, Hp), (Hp, I)
  size_t adaptert;                                // (tdim, L x 3Hp)
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
  R.kp = head_grad_kp(G);
  R.head4t = take((size_t)G.HH * R.kp * 2);
  R.head0t = take(Hp * G.HH * 2);
  R.mlp4t.assign(G.L, 0), R.mlp0t.assign(G.L, 0), R.vn4t.assign(G.L, 0), R.vn0t.assign(G.L, 0);
  for (int l = 1; l < G.L; ++l) {
    R.mlp4t[l] = take(I * Hp * 2), R.mlp0t[l] = take(Hp * I * 2);
    if (l < G.L - 1) R.vn4t[l] = take(I * Hp * 2), R.vn0t[l] = take(Hp * I * 2);
  }
  R.adaptert = take((size_t)G.tdim * G.L * 3 * Hp * 2);
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

// Backward of the virtual node's max-pool (scatter_reduce amax): each column's gradient goes to the node of the graph that holds
// the fp32 maximum, the lowest node index on exact ties.  The forward pools the bf16 copy; rounding is monotone, so that node's
// bf16 value IS the pooled value.  Exact fp32 ties occur between automorphic nodes (the two methyls of an isopropyl group, the
// leaves of a star): such nodes have identical dh/dc, so sending the whole gradient to one of them gives the same dc as the
// reference's even split.  grid (B, ceil(W/256)).
__global__ void __launch_bounds__(256) gin_grad_route_max_kernel(const float* __restrict__ hin, const int32_t* __restrict__ graph_ptr,
                                                                 const float* __restrict__ dpool, float* __restrict__ dh, int W) {
  const int g = blockIdx.x;
  const int c = blockIdx.y * 256 + threadIdx.x;
  if (c >= W) return;
  const int beg = graph_ptr[g], end = graph_ptr[g + 1];
  if (beg == end) return;
  int best = beg;
  float bv = hin[(size_t)beg * W + c];
  for (int i = beg + 1; i < end; ++i) {
    const float v = hin[(size_t)i * W + c];
    if (v > bv) bv = v, best = i;
  }
  dh[(size_t)best * W + c] += dpool[(size_t)g * W + c];
}

// dc = dctext * silu'(c), silu'(x) = s (1 + x (1 - s)), s = sigmoid(x)
__global__ void gin_grad_silu_kernel(const float* __restrict__ c, const float* __restrict__ dctext, float* __restrict__ dc, size_t total) {
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const float x = c[idx];
    const float sg = 1.0f / (1.0f + expf(-x));
    dc[idx] = dctext[idx] * sg * (1.0f + x * (1.0f - sg));
  }
}

unsigned grid_for(size_t total) { return (unsigned)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096); }

}  // namespace

int head_grad_kp(const GinLayout& G) { return (int)align_up((size_t)G.out_dim, 64 * HEAD_GRAD_MAX_SPLIT); }

int head_grad_split(const GinLayout& G, int B) {
  const long long tiles = (long long)ceil_div(B, GEMM_BM) * ceil_div(G.HH, 256);
  int s = HEAD_GRAD_MAX_SPLIT;
  while (s > 1 && tiles * s > HEAD_GRAD_TARGET_TILES) s >>= 1;
  return s;
}

void gin_saved_carve(const GinLayout& G, void* saved, int n, int e, int B, GinSaved* sv, size_t* bytes) {
  GinSaved tmp{};
  GinSaved& v = sv ? *sv : tmp;
  const size_t H = G.Hp, I = G.I, L = G.L, N = n;
  Arena a(saved, 0);
  v.graph_ptr = a.take<int32_t>(B + 1), v.batch32 = a.take<int32_t>(N);
  v.srowptr = a.take<int32_t>(N + 1), v.sdst = a.take<int32_t>(e > 0 ? e : 1), v.seid = a.take<int32_t>(e > 0 ? e : 1);
  v.hin = a.take<float>((L - 1) * N * H);
  v.agg = a.take<__nv_bfloat16>(L * N * H);
  v.pool = a.take<__nv_bfloat16>((L - 1) * B * H);
  v.mod = a.take<float>(L * B * 3 * H);
  v.pooled_b = a.take<__nv_bfloat16>((size_t)B * H);
  v.head_split = head_grad_split(G, B);
  v.dlog_b = a.take<__nv_bfloat16>((size_t)B * head_grad_kp(G));
  v.dhz_parts = a.take<float>((size_t)B * v.head_split * G.HH);
  v.hz_pre = a.take<__nv_bfloat16>((size_t)B * G.HH), v.dhz_pre = a.take<__nv_bfloat16>((size_t)B * G.HH);
  v.dpooled = a.take<float>((size_t)B * H);
  v.dh = a.take<float>(N * H);
  v.dvn = a.take<float>((size_t)B * H), v.dpool = a.take<float>((size_t)B * H), v.dvn_b = a.take<__nv_bfloat16>((size_t)B * H);
  v.vz = a.take<__nv_bfloat16>((size_t)B * I), v.dvz_b = a.take<__nv_bfloat16>((size_t)B * I), v.dvz = a.take<float>((size_t)B * I);
  v.z = a.take<__nv_bfloat16>(N * I);
  v.u = a.take<float>(N * H);
  v.ln_part = a.take<float>(N * ceil_div((int)H, 256) * (GEMM_EPI_WARPS / 4));   // = llb_gin::ln_slots
  v.zpre = a.take<float>(N * I), v.dz = a.take<float>(N * I), v.dzpre_b = a.take<__nv_bfloat16>(N * I);
  v.prod = a.take<float>(N * 3 * H);
  v.du_b = a.take<__nv_bfloat16>(N * H);
  v.da = a.take<float>(N * H);
  v.dmod_b = a.take<__nv_bfloat16>((size_t)B * L * 3 * H);
  v.dctext = a.take<float>((size_t)B * G.tdim);
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
  GinGradLayout R;
  make_grad_layout(G, R);
  *bytes = R.total;
  return LLB_OK;
}

int llb_gin_pack_grad_weights(llb_gin* g, void* grad_blob, size_t grad_bytes, llb_stream_t stream) {
  LLB_CHECK_ARG(g && grad_blob && g->G.predictor, "llb_gin_pack_grad_weights: needs a predictor handle and a blob");
  const GinLayout& G = g->G;
  GinGradLayout R;
  make_grad_layout(G, R);
  if (grad_bytes < R.total) return fail(LLB_ERR_WORKSPACE, "gin: grad blob needs %zu bytes, got %zu", R.total, grad_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* base = (uint8_t*)grad_blob;
  auto dst = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(base + off); };
  auto tr = [&](const auto* src, int ld_s, int rows, int cols, __nv_bfloat16* d, int ld_d) {
    using T = std::remove_const_t<std::remove_pointer_t<decltype(src)>>;
    return launch_kernel(&g->ctr, NO_PROF, false, grad_transpose_kernel<T>, dim3(ceil_div(cols, 32), ceil_div(rows, 32)), dim3(32, 8), 0, s, src,
                         ld_s, rows, cols, d, ld_d);
  };
  const int Hp = G.Hp, I = G.I, HH = G.HH;
  LLB_CUDA_OK(cudaMemsetAsync(base, 0, R.total, s));   // the head's K padding past out_dim is zero
  LLB_TRY(tr(g->w<__nv_bfloat16>(G.head4_w), HH, G.out_dim, HH, dst(R.head4t), R.kp));
  LLB_TRY(tr(g->w<__nv_bfloat16>(G.head0_w), Hp, HH, Hp, dst(R.head0t), HH));
  for (int l = 1; l < G.L; ++l) {
    LLB_TRY(tr(g->w<__half>(G.mlp4_w[l]), I, Hp, I, dst(R.mlp4t[l]), Hp));   // the forward's copy is fp16 (see EpiLnGelu)
    LLB_TRY(tr(g->w<__nv_bfloat16>(G.mlp0_w[l]), Hp, I, Hp, dst(R.mlp0t[l]), I));
    if (l < G.L - 1) {
      LLB_TRY(tr(g->w<__nv_bfloat16>(G.vn4_w[l]), I, Hp, I, dst(R.vn4t[l]), Hp));
      LLB_TRY(tr(g->w<__nv_bfloat16>(G.vn0_w[l]), Hp, I, Hp, dst(R.vn0t[l]), I));
    }
  }
  for (int l = 0; l < G.L; ++l)
    LLB_TRY(tr(g->w<__nv_bfloat16>(G.adapter_w[l]), G.tdim, 3 * Hp, G.tdim, dst(R.adaptert) + (size_t)l * 3 * Hp, G.L * 3 * Hp));
  return LLB_OK;
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
  const int n = num_nodes, B = num_graphs, L = G.L, Hp = G.Hp, I = G.I, HH = G.HH;
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
  // ---- layers, last to first; sv.dh holds dL/d(output of layer l) = dL/d(h_in_{l+1}) on entry
  const dim3 seg_grid_h(B, ceil_div(Hp, 256));
  for (int l = L - 1; l >= 0; --l) {
    const bool last = l == L - 1;
    const float* hin = l > 0 ? sv.hin + (size_t)(l - 1) * n * Hp : nullptr;
    if (!last) {
      // vn_{l+1} is added to every node of h_in_{l+1} and carried into vn_{l+2}
      LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, seg_grid_h, dim3(256), 0, s, sv.dh, Hp, sv.graph_ptr, Hp,
                            l < L - 2 ? sv.dvn : nullptr, sv.dvn, sv.dvn_b, Hp));
      if (l > 0) {
        // vn_{l+1} = vn_l + MLP_l(maxpool(h_in_l)): back through the MLP to the pooled row (routed below)
        g->ctr.slot = LLB_PROF_GIN_MISC;
        LLB_TRY(gemm_bias_act(sv.pool + (size_t)l * B * Hp, Hp, g->w<void>(G.vn0_w[l]), Hp, g->w<float>(G.vn0_b[l]), sv.vz, I, B, I, Hp,
                              LLB_ACT_NONE, false, s, &g->ctr));
        LLB_TRY(gemm_bias_act(sv.dvn_b, Hp, gw(R.vn4t[l]), Hp, nullptr, sv.dvz, I, B, I, Hp, LLB_ACT_NONE, true, s, &g->ctr));
        RowLnBwdArgs a;
        a.x = sv.vz, a.x_ld = I, a.x_bf16 = true, a.dy = sv.dvz, a.dy_ld = I;
        a.rows = B, a.width = I, a.valid = 4 * G.H;
        a.gamma = g->w<float>(G.vn_ln_w[l]), a.beta = g->w<float>(G.vn_ln_b[l]), a.gelu = true;
        a.out_bf16 = sv.dvz_b, a.out_ld = I;
        LLB_TRY(launch_row_ln_bwd(a, s, ctr));
        LLB_TRY(gemm_bias_act(sv.dvz_b, I, gw(R.vn0t[l]), I, nullptr, sv.dpool, Hp, B, Hp, I, LLB_ACT_NONE, true, s, &g->ctr));
      }
    }
    // node MLP output u_l, recomputed from the saved aggregation with the forward's kernels
    const __nv_bfloat16* agg = sv.agg + (size_t)l * n * Hp;
    LLB_TRY(gin_node_mlp(g, agg, n, l, sv.ln_part, sv.z, sv.u, Hp, false, LLB_PROF_GIN_GEMM_MLP0, LLB_PROF_GIN_GEMM_MLP4, s));
    {
      // layer tail: h_out = gate * act(LN(u) (1 + scale) + shift) + h_in (+ vn_{l+1})
      const float* mod = sv.mod + (size_t)l * B * 3 * Hp;
      RowLnBwdArgs a;
      a.x = sv.u, a.x_ld = Hp, a.dy = sv.dh, a.dy_ld = Hp;
      a.rows = n, a.width = Hp, a.valid = G.H;
      a.row_group = sv.batch32, a.shift = mod, a.scale = mod + Hp, a.gate = mod + 2 * Hp, a.mod_ld = 3 * Hp;
      a.gelu = !last;
      a.prod = sv.prod, a.prod_ld = 3 * Hp;
      if (l > 0) a.out_bf16 = sv.du_b, a.out_ld = Hp;
      LLB_TRY(launch_row_ln_bwd(a, s, ctr));
      LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, dim3(B, ceil_div(3 * Hp, 256)), dim3(256), 0, s, sv.prod, 3 * Hp, sv.graph_ptr,
                            3 * Hp, nullptr, nullptr, sv.dmod_b + (size_t)l * 3 * Hp, L * 3 * Hp));
    }
    if (l == 0) break;   // nothing upstream of layer 0's tail depends on c
    // node MLP: du -> dz = du . W4 -> GELU' + LayerNorm(4H) backward on the centred first linear's output -> da = dz_c . W0c
    // (the LayerNorm backward sums to zero over the 4H columns, so the centred weight gives the same product as W0)
    g->ctr.slot = LLB_PROF_GIN_GEMM_MLP0;
    LLB_TRY(gemm_bias_act(agg, Hp, g->w<void>(G.mlp0_w[l]), Hp, g->w<float>(G.mlp0_b[l]), sv.zpre, I, n, I, Hp, LLB_ACT_NONE, true, s, &g->ctr));
    g->ctr.slot = LLB_PROF_GIN_GEMM_MLP4;
    LLB_TRY(gemm_bias_act(sv.du_b, Hp, gw(R.mlp4t[l]), Hp, nullptr, sv.dz, I, n, I, Hp, LLB_ACT_NONE, true, s, &g->ctr));
    {
      RowLnBwdArgs a;
      a.x = sv.zpre, a.x_ld = I, a.dy = sv.dz, a.dy_ld = I;
      a.rows = n, a.width = I, a.valid = 4 * G.H;
      a.gamma = g->w<float>(G.mlp_ln_w[l]), a.beta = g->w<float>(G.mlp_ln_b[l]), a.gelu = true;
      a.out_bf16 = sv.dzpre_b, a.out_ld = I;
      LLB_TRY(launch_row_ln_bwd(a, s, ctr));
    }
    g->ctr.slot = LLB_PROF_GIN_GEMM_MLP0;
    LLB_TRY(gemm_bias_act(sv.dzpre_b, I, gw(R.mlp0t[l]), I, nullptr, sv.da, Hp, n, Hp, I, LLB_ACT_NONE, true, s, &g->ctr));
    LLB_TRY(launch_kernel(ctr, LLB_PROF_GIN_AGGREGATE, false, gin_grad_aggregate_kernel, dim3(ceil_div(n, 8)), dim3(256), 0, s, hin, sv.da, sv.srowptr,
                          sv.sdst, sv.seid, g->w<float>(G.bond_emb[l]), g->w<float>(G.eps[l]), sv.dh, n, Hp));
    if (!last)
      LLB_TRY(launch_kernel(ctr, LLB_PROF_GIN_POOL, false, gin_grad_route_max_kernel, seg_grid_h, dim3(256), 0, s, hin, sv.graph_ptr, sv.dpool, sv.dh,
                            Hp));
  }
  // ---- condition: dctext = [dmod_0 | ... | dmod_{L-1}] . [W_adapter_0 | ... ]^T, dc = dctext * silu'(c)
  g->ctr.slot = LLB_PROF_GIN_MISC;
  LLB_TRY(gemm_bias_act(sv.dmod_b, L * 3 * Hp, gw(R.adaptert), L * 3 * Hp, nullptr, sv.dctext, G.tdim, B, G.tdim, L * 3 * Hp, LLB_ACT_NONE, true,
                        s, &g->ctr));
  return launch_kernel(ctr, NO_PROF, false, gin_grad_silu_kernel, grid_for((size_t)B * G.tdim), dim3(256), 0, s, c, sv.dctext, dc,
                       (size_t)B * G.tdim);
}

}  // extern "C"

