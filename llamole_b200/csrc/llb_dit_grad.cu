// Backward of the GraphDiT denoiser with respect to its condition vector c = t_emb + y_emb + txt_emb (transformer.py:93-187
// differentiated; the forward is dit_body in llb_dit.cu).  The parameters are constants.  Writing mod_l = softsign(ada2_l(silu(
// ada0_l(c)))) = [sh_a | sc_a | g_a | sh_m | sc_m | g_m] per molecule and [shift | scale] = ada2_out(silu(ada0_out(c))), the chain is
//   output    dlogits -> symmetrised, masked d(out) -> LayerNorm(d0) backward with (1 + scale): dshift, dscale per molecule,
//             -> . W_out_fc2 -> GELU' -> . W_out_fc1 = dx;
//   block l   (l = D-1 .. 0) MLP half: LayerNorm backward with gate, (1 + sc_m), sh_m (row products -> dmod), . W_fc2, GELU',
//             . W_fc1 added to dx (the residual passes dx through); attention half: the same tail backward (-> dmod), . W_proj,
//             attention backward with the per-head q/k LayerNorms (dit_grad_attention_kernel), . W_qkv added to dx;
//   condition dz = dmod (1 - |mod|)^2, dhid = [dz_l . W_ada2_l]_l | dmodout . W_out_ada2 (one grouped launch + one),
//             dpre = dhid silu'(pre), dc = dpre . [W_ada0_0 | ... | W_ada0_D] (ONE split-K product, slices summed in order).
// Block 0 stops after its attention tail: its input is the token embedding, which does not depend on c.
// Every block intermediate is recomputed from the saved residual stream with the forward's GEMMs run unfused (fp32 output
// where a LayerNorm needs statistics); the fused forward kernels never materialise the pre-LayerNorm rows, the raw q/k, or the
// fc1 pre-activation, and storing them would cost (6H + 2F) values per token and block.  No float atomics, every sum in a
// fixed order: the gradient is run-to-run bit-identical.
#include <algorithm>

#include "llb_dit.cuh"
#include "llb_grad.cuh"
#include "llb_rowops.cuh"

namespace llb {
namespace {

constexpr int COND_GRAD_MAX_SPLIT = 32;      // K slices of the condition product (dc = dpre . W_ada0, K = (D+1) H) ...
constexpr int COND_GRAD_TARGET_TILES = 296;  // ... halved until the slices' output tiles do not exceed two per SM (148 SMs)

// Transposed bf16 copies of every weight the backward multiplies by (the forward's K-major tcgen05 kernels then serve the
// transposed products unchanged).  (rows, cols) below are the stored shapes.
struct DitGradLayout {
  std::vector<size_t> qkvt, projt, fc1t, fc2t;   // [l]: (H, 3H), (H, H), (H, F), (F, H)
  size_t ada2t;                                  // (D H, 6H): layer l at rows [l H, (l+1) H)
  size_t ada0t;                                  // (H, KA): the D+1 adaLN.0 weights side by side along K, zero past (D+1) H
  size_t out_fc1t, out_fc2t, out_ada2t;          // (H, H), (H, K0o), (H, KO), zero past d0 / 2 d0
  size_t total;
};

void make_grad_layout(const DitLayout& L, DitGradLayout& R) {
  size_t off = 0;
  auto take = [&](size_t bytes) {
    off = align_up(off, 256);
    const size_t o = off;
    off += bytes;
    return o;
  };
  const size_t H = L.H, F = L.F, D = L.D;
  for (size_t l = 0; l < D; ++l) {
    R.qkvt.push_back(take(H * 3 * H * 2));
    R.projt.push_back(take(H * H * 2));
    R.fc1t.push_back(take(H * F * 2));
    R.fc2t.push_back(take(F * H * 2));
  }
  R.ada2t = take(D * H * 6 * H * 2);
  R.ada0t = take(H * (size_t)dit_grad_ka(L) * 2);
  R.out_fc1t = take(H * H * 2);
  R.out_fc2t = take(H * (size_t)dit_grad_k0o(L) * 2);
  R.out_ada2t = take(H * (size_t)dit_grad_ko(L) * 2);
  R.total = align_up(off, 256);
}

unsigned grid_for(size_t total) { return (unsigned)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096); }

// Output-layer tail, one CTA per molecule.  The forward (dit_step_kernel) computes T = LN(raw) (1 + scale) + shift (+ the one-hot
// input), adds, zeroes the diagonal and the padded pairs, symmetrises the valid pairs as 0.5 (T_ij + T_ji) and writes the masked
// dense logits.  Backward: dT_ij = 0.5 (dE_ij + dE_ji) on valid pairs i != j, 0 elsewhere, dT = dX on the atom columns; then the
// LayerNorm backward over d0 -> draw (bf16, zero past d0) and the per-molecule sums dshift = sum_i dT, dscale = sum_i dT xh.
__global__ void __launch_bounds__(256) dit_grad_out_tail_kernel(const float* __restrict__ raw, int raw_ld, const float* __restrict__ modout,
                                                                const int32_t* __restrict__ mol_off, const float* __restrict__ dX,
                                                                const float* __restrict__ dE, int N, __nv_bfloat16* __restrict__ draw,
                                                                int draw_ld, float* __restrict__ dmodout) {
  __shared__ float s_mean[DIT_GRAD_MAXN], s_rstd[DIT_GRAD_MAXN];
  const int b = blockIdx.x;
  const int d0 = DIT_XC + DIT_EC * N;
  const int off = mol_off[b], n = mol_off[b + 1] - off;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* shift = modout + (size_t)b * 2 * d0;
  const float* scale = shift + d0;
  const float* dXb = dX + (size_t)b * N * DIT_XC;
  const float* dEb = dE + (size_t)b * N * N * DIT_EC;
  auto dT = [&](int i, int k) -> float {
    if (k < DIT_XC) return dXb[i * DIT_XC + k];
    const int j = (k - DIT_XC) / DIT_EC, e = (k - DIT_XC) % DIT_EC;
    if (j >= n || j == i) return 0.f;
    return 0.5f * (dEb[((size_t)i * N + j) * DIT_EC + e] + dEb[((size_t)j * N + i) * DIT_EC + e]);
  };
  for (int i = warp; i < n; i += 8) {
    const float* src = raw + (size_t)(off + i) * raw_ld;
    float s = 0.f;
    for (int k = lane; k < d0; k += 32) s += src[k];
    const float mean = warp_sum(s) / (float)d0;
    float q = 0.f;
    for (int k = lane; k < d0; k += 32) {
      const float d = src[k] - mean;
      q = fmaf(d, d, q);
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)d0 + 1e-5f);
    float s1 = 0.f, s2 = 0.f;
    for (int k = lane; k < d0; k += 32) {
      const float xh = (src[k] - mean) * rstd, g = dT(i, k) * (1.0f + scale[k]);
      s1 += g, s2 += g * xh;
    }
    s1 = warp_sum(s1) / (float)d0, s2 = warp_sum(s2) / (float)d0;
    __nv_bfloat16* dst = draw + (size_t)(off + i) * draw_ld;
    for (int k = lane; k < draw_ld; k += 32) {
      float v = 0.f;
      if (k < d0) {
        const float xh = (src[k] - mean) * rstd;
        v = rstd * (dT(i, k) * (1.0f + scale[k]) - s1 - xh * s2);
      }
      dst[k] = __float2bfloat16(v);
    }
    if (lane == 0) s_mean[i] = mean, s_rstd[i] = rstd;
  }
  __syncthreads();
  for (int k = tid; k < d0; k += blockDim.x) {
    float dsh = 0.f, dsc = 0.f;
    for (int i = 0; i < n; ++i) {
      const float g = dT(i, k);
      dsh += g;
      dsc += g * (raw[(size_t)(off + i) * raw_ld + k] - s_mean[i]) * s_rstd[i];
    }
    dmodout[(size_t)b * 2 * d0 + k] = dsh;
    dmodout[(size_t)b * 2 * d0 + d0 + k] = dsc;
  }
}

// out = bf16(g * gelu'(pre)) (the exact erf derivative)
__global__ void dit_grad_gelu_kernel(const float* __restrict__ g, const float* __restrict__ pre, __nv_bfloat16* __restrict__ out, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
    out[i] = __float2bfloat16(g[i] * gelu_erf_grad(pre[i]));
}

__global__ void dit_grad_add_kernel(float* __restrict__ acc, const float* __restrict__ v, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) acc[i] += v[i];
}

// dz = bf16(dmod * softsign'(z)), softsign'(z) = 1 / (1 + |z|)^2 = (1 - |mod|)^2 from the forward's output mod = softsign(z)
__global__ void dit_grad_softsign_kernel(const float* __restrict__ dmod, const float* __restrict__ mod, __nv_bfloat16* __restrict__ dz, size_t total) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const float u = 1.0f - fabsf(mod[i]);
    dz[i] = __float2bfloat16(dmod[i] * u * u);
  }
}

// dpre (B, ld) bf16 = dhid * silu'(pre) on the first W columns, 0 up to ld
__global__ void dit_grad_silu_kernel(const float* __restrict__ dhid, const float* __restrict__ pre, int W, __nv_bfloat16* __restrict__ dpre,
                                     int ld, int B) {
  const size_t total = (size_t)B * ld;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / ld), k = (int)(i % ld);
    float v = 0.f;
    if (k < W) {
      const float x = pre[(size_t)b * W + k];
      const float sg = 1.0f / (1.0f + expf(-x));
      v = dhid[(size_t)b * W + k] * sg * (1.0f + x * (1.0f - sg));
    }
    dpre[i] = __float2bfloat16(v);
  }
}

// dc[b] = sum_s parts[b, s H : (s+1) H], slices in index order
__global__ void dit_grad_sum_slices_kernel(const float* __restrict__ parts, int S, int H, int B, float* __restrict__ dc) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B * H; i += gridDim.x * blockDim.x) {
    const int b = i / H, h = i % H;
    float acc = 0.f;
    for (int s = 0; s < S; ++s) acc += parts[((size_t)b * S + s) * H + h];
    dc[i] = acc;
  }
}

// Attention backward over one (molecule, head): n <= 64 tokens, dh = 64, the varlen layout of the forward (rows mol_off[b] ..).
// Recomputes the per-head affine LayerNorms of q and k (eps 1e-5) from the raw qkv rows, S = q^ k^T dh^-1/2 and P = softmax(S)
// over the molecule's keys, then
//   dV = P^T dO,  dP = dO V^T,  dS = P (dP - rowsum(P dP))  (rowsum(P dP) = rowsum(dO . O)),
//   dq^ = dS k^ dh^-1/2,  dk^ = dS^T q^ dh^-1/2,  back through both LayerNorms,
// and writes dqkv (rows, 3H) bf16 in the [q | k | v] head-major layout of the qkv linear.  fp32 throughout, in shared memory.
constexpr int AG_LD = DIT_DH + 1;
constexpr int AG_SMEM = (8 * DIT_GRAD_MAXN * AG_LD + 4 * DIT_DH + 4 * DIT_GRAD_MAXN) * 4;

__global__ void __launch_bounds__(256) dit_grad_attention_kernel(const float* __restrict__ qkv_raw, const __nv_bfloat16* __restrict__ v_b,
                                                                 const __nv_bfloat16* __restrict__ dO, const int32_t* __restrict__ mol_off,
                                                                 int H, int heads, const float* __restrict__ qw, const float* __restrict__ qb,
                                                                 const float* __restrict__ kw, const float* __restrict__ kb,
                                                                 __nv_bfloat16* __restrict__ dqkv) {
  extern __shared__ float ag[];
  float* Qx = ag;                         // normalised q (xh), then dq^
  float* Kx = Qx + DIT_GRAD_MAXN * AG_LD; // normalised k, then dk^
  float* Qh = Kx + DIT_GRAD_MAXN * AG_LD; // q^ = xh w + b
  float* Kh = Qh + DIT_GRAD_MAXN * AG_LD;
  float* V = Kh + DIT_GRAD_MAXN * AG_LD;
  float* G = V + DIT_GRAD_MAXN * AG_LD;   // dO
  float* P = G + DIT_GRAD_MAXN * AG_LD;
  float* dS = P + DIT_GRAD_MAXN * AG_LD;
  float* wq = dS + DIT_GRAD_MAXN * AG_LD; // qw, qb, kw, kb
  float* st = wq + 4 * DIT_DH;            // q rstd, k rstd, rowsum(P dP), spare
  const int b = blockIdx.x / heads, hd = blockIdx.x % heads;
  const int off = mol_off[b], n = mol_off[b + 1] - off;
  if (n == 0) return;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int ld3 = 3 * H, c0 = hd * DIT_DH;
  const float scl = rsqrtf((float)DIT_DH);
  if (tid < DIT_DH) wq[tid] = qw[tid], wq[DIT_DH + tid] = qb[tid], wq[2 * DIT_DH + tid] = kw[tid], wq[3 * DIT_DH + tid] = kb[tid];
  for (int idx = tid; idx < n * DIT_DH; idx += 256) {
    const int i = idx / DIT_DH, d = idx % DIT_DH;
    const size_t r = (size_t)(off + i);
    Qx[i * AG_LD + d] = qkv_raw[r * ld3 + c0 + d];
    Kx[i * AG_LD + d] = qkv_raw[r * ld3 + H + c0 + d];
    V[i * AG_LD + d] = __bfloat162float(v_b[r * ld3 + 2 * H + c0 + d]);   // the forward's v operand (bf16)
    G[i * AG_LD + d] = __bfloat162float(dO[r * H + c0 + d]);
  }
  __syncthreads();
  // per-head LayerNorms: one warp per (row, q|k)
  for (int task = warp; task < 2 * n; task += 8) {
    const int i = task >> 1, which = task & 1;
    float* x = (which ? Kx : Qx) + i * AG_LD;
    float* y = (which ? Kh : Qh) + i * AG_LD;
    const float a0 = x[lane], a1 = x[lane + 32];
    const float mean = warp_sum(a0 + a1) * (1.0f / DIT_DH);
    const float d0 = a0 - mean, d1 = a1 - mean;
    const float rstd = rsqrtf(warp_sum(d0 * d0 + d1 * d1) * (1.0f / DIT_DH) + 1e-5f);
    const float* w = wq + which * 2 * DIT_DH;
    x[lane] = d0 * rstd, x[lane + 32] = d1 * rstd;
    y[lane] = fmaf(d0 * rstd, w[lane], w[DIT_DH + lane]);
    y[lane + 32] = fmaf(d1 * rstd, w[lane + 32], w[DIT_DH + lane + 32]);
    if (lane == 0) st[which * DIT_GRAD_MAXN + i] = rstd;
  }
  __syncthreads();
  // S -> P (row-wise softmax over the n keys), dP = dO V^T
  for (int idx = tid; idx < n * n; idx += 256) {
    const int i = idx / n, j = idx % n;
    float s = 0.f, dp = 0.f;
#pragma unroll 16
    for (int d = 0; d < DIT_DH; ++d) {
      s = fmaf(Qh[i * AG_LD + d], Kh[j * AG_LD + d], s);
      dp = fmaf(G[i * AG_LD + d], V[j * AG_LD + d], dp);
    }
    P[i * AG_LD + j] = s * scl;
    dS[i * AG_LD + j] = dp;
  }
  __syncthreads();
  for (int i = warp; i < n; i += 8) {
    float* p = P + i * AG_LD;
    const float s0 = lane < n ? p[lane] : -INFINITY, s1 = lane + 32 < n ? p[lane + 32] : -INFINITY;
    const float m = warp_max(fmaxf(s0, s1));
    const float e0 = lane < n ? expf(s0 - m) : 0.f, e1 = lane + 32 < n ? expf(s1 - m) : 0.f;
    const float inv = 1.0f / warp_sum(e0 + e1);
    const float p0 = e0 * inv, p1 = e1 * inv;
    float* ds = dS + i * AG_LD;
    const float dp0 = lane < n ? ds[lane] : 0.f, dp1 = lane + 32 < n ? ds[lane + 32] : 0.f;
    const float rs = warp_sum(p0 * dp0 + p1 * dp1);
    if (lane < n) p[lane] = p0, ds[lane] = p0 * (dp0 - rs);
    if (lane + 32 < n) p[lane + 32] = p1, ds[lane + 32] = p1 * (dp1 - rs);
  }
  __syncthreads();
  // dV = P^T dO -> dqkv; dq^ = dS k^ scl, dk^ = dS^T q^ scl (into registers, then over the normalised rows once all are read)
  for (int idx = tid; idx < n * DIT_DH; idx += 256) {
    const int j = idx / DIT_DH, d = idx % DIT_DH;
    float dv = 0.f;
    for (int i = 0; i < n; ++i) dv = fmaf(P[i * AG_LD + j], G[i * AG_LD + d], dv);
    dqkv[(size_t)(off + j) * ld3 + 2 * H + c0 + d] = __float2bfloat16(dv);
  }
  float dq[DIT_GRAD_MAXN * DIT_DH / 256], dk[DIT_GRAD_MAXN * DIT_DH / 256];
#pragma unroll
  for (int r = 0; r < DIT_GRAD_MAXN * DIT_DH / 256; ++r) {
    const int idx = tid + 256 * r;
    const int i = idx / DIT_DH, d = idx % DIT_DH;
    float aq = 0.f, ak = 0.f;
    if (i < n) {
      for (int j = 0; j < n; ++j) {
        aq = fmaf(dS[i * AG_LD + j], Kh[j * AG_LD + d], aq);
        ak = fmaf(dS[j * AG_LD + i], Qh[j * AG_LD + d], ak);
      }
    }
    dq[r] = aq * scl, dk[r] = ak * scl;
  }
  __syncthreads();
  // the LayerNorm backward needs the whole row: park dq^ (times gamma) in Qh, dk^ in Kh
#pragma unroll
  for (int r = 0; r < DIT_GRAD_MAXN * DIT_DH / 256; ++r) {
    const int idx = tid + 256 * r;
    const int i = idx / DIT_DH, d = idx % DIT_DH;
    if (i < n) Qh[i * AG_LD + d] = dq[r] * wq[d], Kh[i * AG_LD + d] = dk[r] * wq[2 * DIT_DH + d];
  }
  __syncthreads();
  for (int task = warp; task < 2 * n; task += 8) {
    const int i = task >> 1, which = task & 1;
    const float* x = (which ? Kx : Qx) + i * AG_LD;
    const float* g = (which ? Kh : Qh) + i * AG_LD;
    const float g0 = g[lane], g1 = g[lane + 32], x0 = x[lane], x1 = x[lane + 32];
    const float m1 = warp_sum(g0 + g1) * (1.0f / DIT_DH), m2 = warp_sum(g0 * x0 + g1 * x1) * (1.0f / DIT_DH);
    const float rstd = st[which * DIT_GRAD_MAXN + i];
    __nv_bfloat16* o = dqkv + (size_t)(off + i) * ld3 + which * H + c0;
    o[lane] = __float2bfloat16(rstd * (g0 - m1 - x0 * m2));
    o[lane + 32] = __float2bfloat16(rstd * (g1 - m1 - x1 * m2));
  }
}

}  // namespace

int dit_grad_k0o(const DitLayout& L) { return (int)align_up((size_t)L.d0, 64); }
int dit_grad_ko(const DitLayout& L) { return (int)align_up((size_t)2 * L.d0, 64); }
int dit_grad_ka(const DitLayout& L) { return (int)align_up((size_t)(L.D + 1) * L.H, 64 * COND_GRAD_MAX_SPLIT); }

int dit_grad_split(const DitLayout& L, int B) {
  const long long tiles = (long long)ceil_div(B, GEMM_BM) * ceil_div(L.H, 256);
  int s = COND_GRAD_MAX_SPLIT;
  while (s > 1 && tiles * s > COND_GRAD_TARGET_TILES) s >>= 1;
  return s;
}

void dit_saved_carve(const DitLayout& L, void* saved, int B, int Mtok, DitSaved* sv, size_t* bytes) {
  DitSaved tmp{};
  DitSaved& v = sv ? *sv : tmp;
  const size_t H = L.H, F = L.F, D = L.D, M = Mtok > 0 ? Mtok : 1;
  const size_t wmax = std::max<size_t>(std::max<size_t>(F, 3 * H), (size_t)dit_grad_k0o(L));
  Arena a(saved, 0);
  v.mol_off = a.take<int32_t>(B + 1), v.row_mol = a.take<int32_t>(M);
  v.cvec = a.take<__nv_bfloat16>((size_t)B * H);
  v.xs = a.take<float>((2 * D + 1) * M * H);
  v.mod = a.take<float>((size_t)B * D * 6 * H);
  v.modout = a.take<float>((size_t)B * 2 * L.d0);
  v.split = dit_grad_split(L, B);
  v.xb = a.take<__nv_bfloat16>(M * H), v.qkv = a.take<__nv_bfloat16>(M * 3 * H), v.attn = a.take<__nv_bfloat16>(M * H);
  v.hb = a.take<__nv_bfloat16>(M * F);
  v.qkv_raw = a.take<float>(M * 3 * H), v.y = a.take<float>(M * H), v.pre = a.take<float>(M * F);
  v.raw = a.take<float>(M * align_up(L.d0, 4));
  v.dx = a.take<float>(M * H), v.tmp = a.take<float>(M * F);
  v.db = a.take<__nv_bfloat16>(M * wmax), v.dvec = a.take<__nv_bfloat16>(M * H);
  v.prod = a.take<float>(M * 3 * H);
  v.dmod = a.take<float>((size_t)B * D * 6 * H), v.dmodout = a.take<float>((size_t)B * 2 * L.d0);
  v.dz_b = a.take<__nv_bfloat16>((size_t)B * D * 6 * H), v.dmodout_b = a.take<__nv_bfloat16>((size_t)B * dit_grad_ko(L));
  v.dhid = a.take<float>((size_t)B * (D + 1) * H), v.pre0 = a.take<float>((size_t)B * (D + 1) * H);
  v.dpre_b = a.take<__nv_bfloat16>((size_t)B * dit_grad_ka(L));
  v.dc_parts = a.take<float>((size_t)B * v.split * H);
  *bytes = align_up(a.off, 256);
}

int dit_grad_check_n(const DitLayout& L, const char* entry) {
  LLB_CHECK_ARG(L.N <= DIT_GRAD_MAXN, "%s: max_nodes=%d must be in [1,%d] (the denoiser's backward)", entry, L.N, DIT_GRAD_MAXN);
  return LLB_OK;
}

}  // namespace llb

using namespace llb;

extern "C" {

int llb_dit_grad_packed_bytes(const llb_dit_config* cfg, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes, "llb_dit_grad_packed_bytes: null argument");
  DitLayout L;
  LLB_TRY(make_layout(*cfg, L));
  LLB_TRY(dit_grad_check_n(L, "llb_dit_grad_packed_bytes"));
  DitGradLayout R;
  make_grad_layout(L, R);
  *bytes = R.total;
  return LLB_OK;
}

int llb_dit_train_saved_bytes(const llb_dit_config* cfg, int B, int num_tokens, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes && B >= 1 && num_tokens >= 0, "llb_dit_train_saved_bytes: bad argument");
  DitLayout L;
  LLB_TRY(make_layout(*cfg, L));
  LLB_TRY(dit_grad_check_n(L, "llb_dit_train_saved_bytes"));
  LLB_CHECK_ARG(num_tokens <= B * L.N, "llb_dit_train_saved_bytes: %d tokens exceed %d molecules of at most %d atoms", num_tokens, B, L.N);
  dit_saved_carve(L, nullptr, B, num_tokens, nullptr, bytes);
  return LLB_OK;
}

int llb_dit_pack_grad_weights(llb_dit* h, void* grad_blob, size_t grad_bytes, llb_stream_t stream) {
  LLB_CHECK_ARG(h && grad_blob, "llb_dit_pack_grad_weights: null argument");
  const DitLayout& L = h->L;
  LLB_TRY(dit_grad_check_n(L, "llb_dit_pack_grad_weights"));
  DitGradLayout R;
  make_grad_layout(L, R);
  if (grad_bytes < R.total) return fail(LLB_ERR_WORKSPACE, "dit: grad blob needs %zu bytes, got %zu", R.total, grad_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* base = (uint8_t*)grad_blob;
  auto dst = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(base + off); };
  auto tr = [&](size_t src, int rows, int cols, __nv_bfloat16* d, int ld_d) {
    return launch_kernel(&h->ctr, NO_PROF, false, grad_transpose_kernel<__nv_bfloat16>, dim3(ceil_div(cols, 32), ceil_div(rows, 32)), dim3(32, 8), 0, s,
                         h->w<__nv_bfloat16>(src), cols, rows, cols, d, ld_d, rows);
  };
  const int H = L.H, F = L.F, D = L.D;
  LLB_CUDA_OK(cudaMemsetAsync(base, 0, R.total, s));   // the K padding of the out-layer and condition operands is zero
  for (int l = 0; l < D; ++l) {
    LLB_TRY(tr(L.qkv_w[l], 3 * H, H, dst(R.qkvt[l]), 3 * H));
    LLB_TRY(tr(L.proj_w[l], H, H, dst(R.projt[l]), H));
    LLB_TRY(tr(L.fc1_w[l], F, H, dst(R.fc1t[l]), F));
    LLB_TRY(tr(L.fc2_w[l], H, F, dst(R.fc2t[l]), H));
    LLB_TRY(tr(L.ada2_w[l], 6 * H, H, dst(R.ada2t) + (size_t)l * H * 6 * H, 6 * H));
  }
  LLB_TRY(tr(L.ada0_w, (D + 1) * H, H, dst(R.ada0t), dit_grad_ka(L)));
  LLB_TRY(tr(L.out_fc1_w, H, H, dst(R.out_fc1t), H));
  LLB_TRY(tr(L.out_fc2_w, L.d0, H, dst(R.out_fc2t), dit_grad_k0o(L)));
  LLB_TRY(tr(L.out_ada2_w, 2 * L.d0, H, dst(R.out_ada2t), dit_grad_ko(L)));
  return LLB_OK;
}

int llb_dit_backward_c(llb_dit* h, int B, int num_tokens, void* saved, size_t saved_bytes, const void* grad_blob, size_t grad_bytes,
                       const float* dlogits_X, const float* dlogits_E, float* dc, llb_stream_t stream) {
  LLB_CHECK_ARG(h && saved && grad_blob && dlogits_X && dlogits_E && dc, "llb_dit_backward_c: null argument");
  LLB_CHECK_ARG(B >= 1 && num_tokens >= 0 && num_tokens <= B * h->L.N, "llb_dit_backward_c: bad batch size");
  const DitLayout& L = h->L;
  LLB_TRY(dit_grad_check_n(L, "llb_dit_backward_c"));
  DitGradLayout R;
  make_grad_layout(L, R);
  if (grad_bytes < R.total) return fail(LLB_ERR_WORKSPACE, "dit: grad blob needs %zu bytes, got %zu", R.total, grad_bytes);
  DitSaved sv;
  size_t need = 0;
  dit_saved_carve(L, saved, B, num_tokens, &sv, &need);
  if (saved_bytes < need) return fail(LLB_ERR_WORKSPACE, "dit: saved buffer needs %zu bytes, got %zu", need, saved_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  const int H = L.H, F = L.F, D = L.D, M = num_tokens, d0 = L.d0;
  const int K0o = dit_grad_k0o(L), KO = dit_grad_ko(L), KA = dit_grad_ka(L), ldm = D * 6 * H;
  const int raw_ld = (int)align_up(d0, 4);
  const uint8_t* gb = (const uint8_t*)grad_blob;
  auto gw = [&](size_t off) { return (const void*)(gb + off); };
  LaunchCounter* ctr = &h->ctr;
  ctr->slot = LLB_PROF_GEMM_OTHER;
  auto gemm = [&](const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int rows, int N, int K, int act,
                  bool f32, GemmGroups grp = GemmGroups()) {
    return gemm_bias_act(A, lda, W, ldw, bias, C, ldc, rows, N, K, act, f32, s, ctr, grp);
  };
  auto to_bf16 = [&](const float* x) -> int {   // sv.xb = bf16(x), the forward's GEMM operand of that residual row
    return launch_f32_to_bf16(x, H, sv.xb, H, M, H, H, s, ctr);
  };
  auto gelu_bwd = [&](const float* g, const float* pre, __nv_bfloat16* out, size_t total) -> int {
    return launch_kernel(ctr, NO_PROF, false, dit_grad_gelu_kernel, grid_for(total), dim3(256), 0, s, g, pre, out, total);
  };
  auto add_dx = [&](const float* v) -> int {
    return launch_kernel(ctr, NO_PROF, false, dit_grad_add_kernel, grid_for((size_t)M * H), dim3(256), 0, s, sv.dx, v, (size_t)M * H);
  };
  if (M > 0) {
    // ---- output layer
    LLB_TRY(to_bf16(sv.xs + (size_t)2 * D * M * H));
    LLB_TRY(gemm(sv.xb, H, h->w<void>(L.out_fc1_w), H, h->w<float>(L.out_fc1_b), sv.hb, H, M, H, H, LLB_ACT_GELU, false));
    LLB_TRY(gemm(sv.hb, H, h->w<void>(L.out_fc2_w), H, h->w<float>(L.out_fc2_b), sv.raw, raw_ld, M, d0, H, LLB_ACT_NONE, true));
    LLB_TRY(launch_kernel(ctr, NO_PROF, false, dit_grad_out_tail_kernel, dim3(B), dim3(256), 0, s, sv.raw, raw_ld, sv.modout, sv.mol_off, dlogits_X,
                          dlogits_E, L.N, sv.db, K0o, sv.dmodout));
    LLB_TRY(gemm(sv.db, K0o, gw(R.out_fc2t), K0o, nullptr, sv.tmp, H, M, H, K0o, LLB_ACT_NONE, true));
    LLB_TRY(gemm(sv.xb, H, h->w<void>(L.out_fc1_w), H, h->w<float>(L.out_fc1_b), sv.pre, H, M, H, H, LLB_ACT_NONE, true));
    LLB_TRY(gelu_bwd(sv.tmp, sv.pre, sv.dvec, (size_t)M * H));
    LLB_TRY(gemm(sv.dvec, H, gw(R.out_fc1t), H, nullptr, sv.dx, H, M, H, H, LLB_ACT_NONE, true));
    // ---- blocks, last to first; sv.dx = dL/d(residual stream after block l)
    const dim3 seg_grid(B, ceil_div(3 * H, 256));
    for (int l = D - 1; l >= 0; --l) {
      const float* mod = sv.mod + (size_t)l * 6 * H;
      const float* x_in = sv.xs + (size_t)(2 * l) * M * H;
      const float* x_mid = x_in + (size_t)M * H;
      // MLP half: x_out = x_mid + g_m (LN(m) (1 + sc_m) + sh_m), m = fc2(gelu(fc1(x_mid)))
      LLB_TRY(to_bf16(x_mid));
      ctr->slot = LLB_PROF_GEMM_FC1;
      LLB_TRY(gemm(sv.xb, H, h->w<void>(L.fc1_w[l]), H, h->w<float>(L.fc1_b[l]), sv.hb, F, M, F, H, LLB_ACT_GELU, false));
      ctr->slot = LLB_PROF_GEMM_FC2;
      LLB_TRY(gemm(sv.hb, F, h->w<void>(L.fc2_w[l]), F, h->w<float>(L.fc2_b[l]), sv.y, H, M, H, F, LLB_ACT_NONE, true));
      RowLnBwdArgs t;
      t.x = sv.y, t.x_ld = H, t.dy = sv.dx, t.dy_ld = H;
      t.rows = M, t.width = H, t.valid = H;
      t.row_group = sv.row_mol, t.mod_ld = ldm;
      t.prod = sv.prod, t.prod_ld = 3 * H;
      t.out_bf16 = sv.dvec, t.out_ld = H;
      t.prof_slot = LLB_PROF_LN_MOD_RES;
      {
        RowLnBwdArgs a = t;
        a.shift = mod + 3 * H, a.scale = mod + 4 * H, a.gate = mod + 5 * H;
        LLB_TRY(launch_row_ln_bwd(a, s, ctr));
      }
      LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, seg_grid, dim3(256), 0, s, sv.prod, 3 * H, sv.mol_off, 3 * H, nullptr,
                            sv.dmod + (size_t)l * 6 * H + 3 * H, nullptr, ldm));
      ctr->slot = LLB_PROF_GEMM_FC2;
      LLB_TRY(gemm(sv.dvec, H, gw(R.fc2t[l]), H, nullptr, sv.tmp, F, M, F, H, LLB_ACT_NONE, true));
      ctr->slot = LLB_PROF_GEMM_FC1;
      LLB_TRY(gemm(sv.xb, H, h->w<void>(L.fc1_w[l]), H, h->w<float>(L.fc1_b[l]), sv.pre, F, M, F, H, LLB_ACT_NONE, true));
      LLB_TRY(gelu_bwd(sv.tmp, sv.pre, sv.db, (size_t)M * F));
      LLB_TRY(gemm(sv.db, F, gw(R.fc1t[l]), F, nullptr, sv.y, H, M, H, F, LLB_ACT_NONE, true));
      LLB_TRY(add_dx(sv.y));
      // attention half: x_mid = x_in + g_a (LN(a) (1 + sc_a) + sh_a), a = proj(attention(qkv(x_in)))
      LLB_TRY(to_bf16(x_in));
      ctr->slot = LLB_PROF_GEMM_QKV;
      const float q_scale = 1.4426950408889634f / sqrtf((float)DIT_DH);
      EpiQKV eq{sv.qkv, 3 * H, H, h->w<float>(L.qn_w[l]), h->w<float>(L.qn_b[l]), h->w<float>(L.kn_w[l]), h->w<float>(L.kn_b[l]), q_scale};
      LLB_TRY((launch_gemm<128>(sv.xb, H, h->w<void>(L.qkv_w[l]), H, M, 3 * H, H, eq, s, ctr)));
      {
        CUtensorMap tmQKV;
        LLB_TRY(make_tensor_map_2d(&tmQKV, sv.qkv, 2, M, 3 * H, 3 * H, DIT_DH, 64, 128));
        LLB_TRY(launch_kernel(ctr, LLB_PROF_ATTENTION, true, dit_attention_tma_kernel<64>, dim3((unsigned)(B * L.heads)), dim3(128), 0, s, tmQKV, sv.attn,
                              sv.mol_off, B, M, H, L.heads));
      }
      ctr->slot = LLB_PROF_GEMM_PROJ;
      LLB_TRY(gemm(sv.attn, H, h->w<void>(L.proj_w[l]), H, h->w<float>(L.proj_b[l]), sv.y, H, M, H, H, LLB_ACT_NONE, true));
      {
        RowLnBwdArgs a = t;
        a.shift = mod, a.scale = mod + H, a.gate = mod + 2 * H;
        if (l == 0) a.out_bf16 = nullptr;
        LLB_TRY(launch_row_ln_bwd(a, s, ctr));
      }
      LLB_TRY(launch_kernel(ctr, NO_PROF, false, grad_segsum_kernel, seg_grid, dim3(256), 0, s, sv.prod, 3 * H, sv.mol_off, 3 * H, nullptr,
                            sv.dmod + (size_t)l * 6 * H, nullptr, ldm));
      if (l == 0) break;   // block 0's input is the token embedding: nothing upstream depends on c
      LLB_TRY(gemm(sv.dvec, H, gw(R.projt[l]), H, nullptr, sv.attn, H, M, H, H, LLB_ACT_NONE, false));   // dO (bf16)
      ctr->slot = LLB_PROF_GEMM_QKV;
      LLB_TRY(gemm(sv.xb, H, h->w<void>(L.qkv_w[l]), H, nullptr, sv.qkv_raw, 3 * H, M, 3 * H, H, LLB_ACT_NONE, true));
      LLB_TRY(launch_kernel(ctr, LLB_PROF_ATTENTION, false, dit_grad_attention_kernel, dim3(B * L.heads), dim3(256), AG_SMEM, s, sv.qkv_raw, sv.qkv,
                            sv.attn, sv.mol_off, H, L.heads, h->w<float>(L.qn_w[l]), h->w<float>(L.qn_b[l]), h->w<float>(L.kn_w[l]),
                            h->w<float>(L.kn_b[l]), sv.db));
      LLB_TRY(gemm(sv.db, 3 * H, gw(R.qkvt[l]), 3 * H, nullptr, sv.y, H, M, H, 3 * H, LLB_ACT_NONE, true));
      LLB_TRY(add_dx(sv.y));
    }
  } else {   // no atoms at all: the logits do not depend on c
    LLB_CUDA_OK(cudaMemsetAsync(sv.dmod, 0, (size_t)B * ldm * 4, s));
    LLB_CUDA_OK(cudaMemsetAsync(sv.dmodout, 0, (size_t)B * 2 * d0 * 4, s));
  }
  // ---- condition
  ctr->slot = LLB_PROF_GEMM_ADALN;
  const size_t nmod = (size_t)B * ldm;
  LLB_TRY(launch_kernel(ctr, NO_PROF, false, dit_grad_softsign_kernel, grid_for(nmod), dim3(256), 0, s, sv.dmod, sv.mod, sv.dz_b, nmod));
  const int ldh = (D + 1) * H;
  {
    GemmGroups grp;
    grp.group_n = H, grp.group_k = 6 * H;
    LLB_TRY(gemm(sv.dz_b, ldm, gw(R.ada2t), 6 * H, nullptr, sv.dhid, ldh, B, D * H, 6 * H, LLB_ACT_NONE, true, grp));
  }
  LLB_TRY(launch_f32_to_bf16(sv.dmodout, 2 * d0, sv.dmodout_b, KO, B, 2 * d0, KO, s, ctr));
  LLB_TRY(gemm(sv.dmodout_b, KO, gw(R.out_ada2t), KO, nullptr, sv.dhid + (size_t)D * H, ldh, B, H, KO, LLB_ACT_NONE, true));
  LLB_TRY(gemm(sv.cvec, H, h->w<void>(L.ada0_w), H, h->w<float>(L.ada0_b), sv.pre0, ldh, B, ldh, H, LLB_ACT_NONE, true));
  LLB_TRY(launch_kernel(ctr, NO_PROF, false, dit_grad_silu_kernel, grid_for((size_t)B * KA), dim3(256), 0, s, sv.dhid, sv.pre0, ldh, sv.dpre_b, KA,
                        B));
  {
    const int S = sv.split, ks = KA / S;
    GemmGroups split;
    split.group_n = H, split.group_k = ks, split.split_k = true;
    LLB_TRY(gemm(sv.dpre_b, KA, gw(R.ada0t), KA, nullptr, sv.dc_parts, S * H, B, S * H, ks, LLB_ACT_NONE, true, split));
    return launch_kernel(ctr, NO_PROF, false, dit_grad_sum_slices_kernel, grid_for((size_t)B * H), dim3(256), 0, s, sv.dc_parts, S, H, B, dc);
  }
}

}  // extern "C"
