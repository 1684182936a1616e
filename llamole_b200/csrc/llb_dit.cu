// GraphDiT sampler: weight packing, batch binding, denoiser pass and the reverse-diffusion loop.
// Reference: graph_decoder/diffusion_model.py:252-399, transformer.py:93-187 (see include/llamole_b200.h).
#include <math.h>
#include <stdlib.h>

#include <vector>

// split-K factor of the latency-regime fc2 (K = F): F / 4 per slice, partial products summed by the row kernel
#define LLB_DIT_SPLITK 4

#ifndef LLB_ATTN_DEFAULT
#define LLB_ATTN_DEFAULT 3
#endif

#include "llb_dit.cuh"
#include "llb_gemm_ln.cuh"
#include "llb_rowops.cuh"

namespace llb {

int make_layout(const llb_dit_config& c, DitLayout& L) {
  LLB_CHECK_ARG(c.hidden > 0 && c.hidden % 64 == 0, "dit: hidden=%d must be a positive multiple of 64", c.hidden);
  LLB_CHECK_ARG(c.heads > 0 && c.hidden == c.heads * DIT_DH, "dit: head dim must be 64 (hidden=%d heads=%d)", c.hidden, c.heads);
  LLB_CHECK_ARG(c.mlp_hidden > 0 && c.mlp_hidden % 64 == 0, "dit: mlp_hidden=%d must be a multiple of 64", c.mlp_hidden);
  LLB_CHECK_ARG(c.max_nodes >= 1 && c.max_nodes <= DIT_MAXN, "dit: max_nodes=%d must be in [1,%d]", c.max_nodes, DIT_MAXN);
  LLB_CHECK_ARG(c.depth >= 1 && c.timesteps >= 1 && c.y_dim >= 0 && c.y_dim <= 32, "dit: bad depth/timesteps/y_dim");
  LLB_CHECK_ARG(c.text_dim > 0 && c.text_dim % 64 == 0, "dit: text_dim=%d must be a multiple of 64", c.text_dim);
  L.H = c.hidden, L.D = c.depth, L.heads = c.heads, L.F = c.mlp_hidden, L.N = c.max_nodes, L.T = c.timesteps;
  L.ydim = c.y_dim, L.tdim = c.text_dim;
  L.d0 = DIT_XC + DIT_EC * L.N;
  L.K0 = (int)align_up(L.d0, 64);
  L.KC = L.ydim * L.H + L.tdim;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    off = align_up(off, 256);
    size_t o = off;
    off += bytes;
    return o;
  };
  const size_t H = L.H, F = L.F, D = L.D;
  L.x_embed_w = take(H * L.K0 * 2);
  L.cond_w = take(H * (size_t)L.KC * 2);
  L.ada0_w = take((D + 1) * H * H * 2);
  L.out_fc1_w = take(H * H * 2);
  L.out_fc2_w = take((size_t)L.d0 * H * 2);
  L.out_ada2_w = take((size_t)2 * L.d0 * H * 2);
  for (size_t l = 0; l < D; ++l) {
    L.qkv_w.push_back(take(3 * H * H * 2));
    L.proj_w.push_back(take(H * H * 2));
    L.fc1_w.push_back(take(F * H * 2));
    L.fc2_w.push_back(take(H * F * 2));
  }
  for (size_t l = 0; l < D; ++l) L.ada2_w.push_back(take(6 * H * H * 2));   // contiguous: one (D 6H, H) operand of the grouped launch
  L.x_ln_w = take(H * 4), L.x_ln_b = take(H * 4);
  L.ada0_b = take((D + 1) * H * 4);
  L.out_fc1_b = take(H * 4), L.out_fc2_b = take((size_t)L.d0 * 4), L.out_ada2_b = take((size_t)2 * L.d0 * 4);
  for (size_t l = 0; l < D; ++l) {
    L.qn_w.push_back(take(DIT_DH * 4)), L.qn_b.push_back(take(DIT_DH * 4));
    L.kn_w.push_back(take(DIT_DH * 4)), L.kn_b.push_back(take(DIT_DH * 4));
    L.proj_b.push_back(take(2 * H * 4)), L.fc1_b.push_back(take(F * 4));   // proj: H values, then zeros (bias of the 2-slice split-K launch)
    L.fc2_b.push_back(take(LLB_DIT_SPLITK * H * 4));   // H values, then zeros: bias of the split-K launch (slice 0 carries it)
  }
  for (size_t l = 0; l < D; ++l) L.ada2_b.push_back(take(6 * H * 4));   // contiguous, like the weights
  L.y_mlp0_w = take((size_t)L.ydim * H * 4), L.y_mlp0_b = take((size_t)L.ydim * H * 4), L.y_drop = take((size_t)L.ydim * H * 4);
  L.txt_drop = take(H * 4), L.txt_b = take(H * 4);
  L.c1_table = take((size_t)(L.T + 1) * H * 4);
  L.c_unc = take(H * 4);
  L.tables = take((DIT_XC + DIT_EC + 2 * DIT_XC * DIT_EC) * 4);
  L.betas = take((size_t)(L.T + 1) * 4), L.abar = take((size_t)(L.T + 1) * 4);
  L.setup_scratch = take((size_t)(L.T + 1) * (256 + H) * 4);
  L.total = align_up(off, 256);
  return LLB_OK;
}

namespace {

// timestep features on normalised t = i / T (conditions.py:33-51)
__global__ void dit_tfeat_kernel(float* __restrict__ feat, int T) {
  const int i = blockIdx.x;  // 0..T
  const int k = threadIdx.x;  // 0..127
  const float tn = (float)i / (float)T;
  const float f = expf(-logf(10000.0f) * (float)k / 128.0f);
  const float arg = tn * f;
  feat[(size_t)i * 256 + k] = cosf(arg);
  feat[(size_t)i * 256 + 128 + k] = sinf(arg);
}

__global__ void dit_cunc_kernel(const float* __restrict__ y_drop, const float* __restrict__ txt_drop, float* __restrict__ c_unc,
                                int ydim, int H) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= H) return;
  float s = txt_drop[h];
  for (int d = 0; d < ydim; ++d) s += y_drop[(size_t)d * H + h];
  c_unc[h] = s;
}

// A_cond row b = [softmax_H(y[b,d] w0_d + b0_d) for d (zeros if NaN) | txt[b] (zeros if any NaN)]
// (conditions.py:76-98, 108-123).  grid (B, ydim+1), 256 threads.
__global__ void __launch_bounds__(256) dit_cond_operand_kernel(const float* __restrict__ props, const float* __restrict__ txt,
                                                               const float* __restrict__ w0, const float* __restrict__ b0,
                                                               __nv_bfloat16* __restrict__ A, uint8_t* __restrict__ missing,
                                                               int ydim, int tdim, int H, int KC) {
  __shared__ float red[32];
  __shared__ float bcast;
  const int b = blockIdx.x, d = blockIdx.y;
  const int tid = threadIdx.x;
  __nv_bfloat16* out = A + (size_t)b * KC;
  auto block_reduce = [&](float v, bool is_max) {
    v = is_max ? warp_max(v) : warp_sum(v);
    if ((tid & 31) == 0) red[tid >> 5] = v;
    __syncthreads();
    if (tid < 32) {
      float x = tid < (int)(blockDim.x >> 5) ? red[tid] : (is_max ? -INFINITY : 0.f);
      x = is_max ? warp_max(x) : warp_sum(x);
      if (tid == 0) bcast = x;
    }
    __syncthreads();
    const float r = bcast;
    __syncthreads();
    return r;
  };
  if (d < ydim) {
    const float y = props[(size_t)b * ydim + d];
    const bool miss = isnan(y);
    if (tid == 0) missing[(size_t)b * (ydim + 1) + d] = miss ? 1 : 0;
    out += (size_t)d * H;
    if (miss) {
      for (int h = tid; h < H; h += blockDim.x) out[h] = __float2bfloat16(0.f);
      return;
    }
    const float* w = w0 + (size_t)d * H;
    const float* bb = b0 + (size_t)d * H;
    float m = -INFINITY;
    for (int h = tid; h < H; h += blockDim.x) m = fmaxf(m, fmaf(y, w[h], bb[h]));
    m = block_reduce(m, true);
    float s = 0.f;
    for (int h = tid; h < H; h += blockDim.x) s += expf(fmaf(y, w[h], bb[h]) - m);
    s = block_reduce(s, false);
    const float inv = 1.0f / s;
    for (int h = tid; h < H; h += blockDim.x) out[h] = __float2bfloat16(expf(fmaf(y, w[h], bb[h]) - m) * inv);
  } else {
    const float* t = txt + (size_t)b * tdim;
    float bad = 0.f;
    for (int k = tid; k < tdim; k += blockDim.x) bad += isnan(t[k]) ? 1.f : 0.f;
    bad = block_reduce(bad, false);
    const bool miss = bad > 0.f;
    if (tid == 0) missing[(size_t)b * (ydim + 1) + ydim] = miss ? 1 : 0;
    out += (size_t)ydim * H;
    for (int k = tid; k < tdim; k += blockDim.x) out[k] = __float2bfloat16(miss ? 0.f : t[k]);
  }
}

// cinv[b] += sum over missing properties of the drop rows + (text missing ? txt_drop : txt bias)
__global__ void dit_cond_fixup_kernel(float* __restrict__ cinv, const uint8_t* __restrict__ missing, const float* __restrict__ y_drop,
                                      const float* __restrict__ txt_drop, const float* __restrict__ txt_b, int B, int ydim, int H) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * H) return;
  const int b = i / H, h = i % H;
  const uint8_t* ms = missing + (size_t)b * (ydim + 1);
  float v = cinv[i];
  for (int d = 0; d < ydim; ++d)
    if (ms[d]) v += y_drop[(size_t)d * H + h];
  v += ms[ydim] ? txt_drop[h] : txt_b[h];
  cinv[i] = v;
}

}  // namespace
}  // namespace llb

using namespace llb;

// t_in_smem = false: the T_GLOBAL step kernel, whose logit rows T stay in global memory
static size_t dit_step_smem(int N, int passes, bool t_in_smem = true) {
  const int d0 = DIT_XC + DIT_EC * N;
  return (t_in_smem ? (size_t)passes * N * d0 * 4 : 0) + (size_t)passes * N * sizeof(NodeStats) + (size_t)N * DIT_EC * 4 +
         ((N + 15) & ~15) + (size_t)N * N + 16;
}

static int smem_per_block_optin() {
  static int bytes = 0;
  if (bytes == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&bytes, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (bytes <= 0) bytes = 48 * 1024;
  }
  return bytes;
}

static int dit_carve(llb_dit* h, void* ws, size_t ws_bytes, int B, int Mtok, size_t* need) {
  const DitLayout& L = h->L;
  const size_t passes = 2;
  const size_t M = passes * (size_t)Mtok;
  Arena a(ws, ws_bytes);
  h->x = a.take<float>(M * L.H);
  h->xb = a.take<__nv_bfloat16>(M * L.H);
  h->y = a.take<__nv_bfloat16>(M * L.H);
  h->qkv = a.take<__nv_bfloat16>(M * 3 * L.H);
  h->attn = a.take<__nv_bfloat16>(M * L.H);
  h->hbuf = a.take<__nv_bfloat16>(M * L.F > (size_t)Mtok * L.H * 2 ? M * L.F : (size_t)Mtok * L.H * 2);
  h->tok = a.take<__nv_bfloat16>((size_t)Mtok * L.K0);
  h->raw_ld = (int)align_up(L.d0, 4);
  h->raw = a.take<float>(M * h->raw_ld);
  h->cvec = a.take<__nv_bfloat16>((size_t)(B + 1) * L.H);
  h->hid = a.take<__nv_bfloat16>((size_t)(B + 1) * (L.D + 1) * L.H);
  h->mod = a.take<float>((size_t)L.D * (B + 1) * 6 * L.H);
  h->modout = a.take<float>((size_t)(B + 1) * 2 * L.d0);
  h->cinv = a.take<float>((size_t)B * L.H);
  h->acond = a.take<__nv_bfloat16>((size_t)B * L.KC);
  h->missing = a.take<uint8_t>((size_t)B * (L.ydim + 1));
  h->stX = a.take<int8_t>((size_t)B * L.N);
  h->stE = a.take<int8_t>((size_t)B * L.N * L.N);
  h->mol_off = a.take<int32_t>(B + 1);
  h->row_mol = a.take<int32_t>(Mtok > 0 ? Mtok : 1);
  h->row_group = a.take<int32_t>(M > 0 ? M : 1);
  h->ln_sync = a.take<uint8_t>(gemm_ln_pair_workspace_bytes());
  h->part = a.take<float>((M < 640 ? M : 640) * (size_t)LLB_DIT_SPLITK * L.H);   // split-K partials (latency regime, <= 640 rows)
  *need = align_up(a.off, 256);
  return LLB_OK;
}

static bool dit_latency_regime(const llb_dit* h) {
  static const bool ln_env_set = getenv("LLB_FUSED_LN") != nullptr;
  return !ln_env_set && h->passes * h->Mtok < 2048;
}

// The t-independent part of a denoiser pass: token embedding, every adaLN modulation (from h->cvec), the transformer blocks and the
// output MLP, up to the raw output-layer rows (h->raw).
static int dit_body(llb_dit* h, cudaStream_t s) {
  const DitLayout& L = h->L;
  const int H = L.H, F = L.F, D = L.D, B = h->B, Mtok = h->Mtok;
  const int M = h->passes * Mtok;
  LaunchCounter* ctr = &h->ctr;
  // 1. tokens -> embedding -> LayerNorm (shared by both halves)
  LLB_TRY(launch_kernel(ctr, LLB_PROF_DIT_MISC, false, dit_tokens_kernel, dim3(ceil_div(Mtok, 8)), dim3(256), 0, s, h->stX, h->stE, h->mol_off,
                        h->row_mol, h->tok, Mtok, L.N, L.K0));
  ctr->slot = LLB_PROF_GEMM_OTHER;
  float* emb = reinterpret_cast<float*>(h->hbuf);
  LLB_TRY(gemm_bias_act(h->tok, L.K0, h->w<void>(L.x_embed_w), L.K0, nullptr, emb, H, Mtok, H, L.K0, LLB_ACT_NONE, true, s, ctr));
  {
    RowLnArgs a;
    a.in = emb, a.in_ld = H, a.in_bf16 = false, a.rows = Mtok, a.width = H;
    a.gamma = h->w<float>(L.x_ln_w), a.beta = h->w<float>(L.x_ln_b);
    a.out_f32 = h->x, a.out_f32_ld = H, a.out_bf16 = h->xb, a.out_bf16_ld = H;
    a.dup_rows = h->passes == 2 ? Mtok : 0;
    a.prof_slot = LLB_PROF_DIT_MISC;
    LLB_TRY(launch_row_ln(a, s, ctr));
  }
  // a saved pass (llb_dit_denoise_c) keeps the residual stream at every block-half boundary for its backward
  auto save_x = [&](int k) -> int {
    if (h->save_x) LLB_CUDA_OK(cudaMemcpyAsync(h->save_x + (size_t)k * M * H, h->x, (size_t)M * H * 4, cudaMemcpyDeviceToDevice, s));
    return LLB_OK;
  };
  LLB_TRY(save_x(0));
  // 2. all adaLN modulations of this step from the conditioning vector
  ctr->slot = LLB_PROF_GEMM_ADALN;
  const int ldh = (D + 1) * H;
  LLB_TRY(gemm_bias_act(h->cvec, H, h->w<void>(L.ada0_w), H, h->w<float>(L.ada0_b), h->hid, ldh, B + 1, ldh, H, LLB_ACT_SILU, false, s, ctr));
  // the D modulation linears depend only on the condition: ONE launch grouped along N (group l reads hid[:, l H : (l+1) H],
  // its 6H x H weight is rows [l 6H, (l+1) 6H) of the stacked operand); mod is (B+1, D, 6H).
  const int ldm = D * 6 * H;
  // the stacked operand needs the D weights (and biases) back to back in the blob: true whenever 6 H H 2 and 6 H 4 bytes are
  // multiples of the blob's 256-byte alignment; checked rather than assumed
  const bool stacked = D == 1 || (L.ada2_w[1] - L.ada2_w[0] == (size_t)6 * H * H * 2 && L.ada2_b[1] - L.ada2_b[0] == (size_t)6 * H * 4);
  if (stacked && (6 * H) % 256 == 0) {
    GemmGroups grp;
    grp.group_n = 6 * H, grp.group_k = H;
    LLB_TRY(gemm_bias_act(h->hid, ldh, h->w<void>(L.ada2_w[0]), H, h->w<float>(L.ada2_b[0]), h->mod, ldm, B + 1, ldm, H, LLB_ACT_SOFTSIGN, true, s,
                          ctr, grp));
  } else {
    for (int l = 0; l < D; ++l)
      LLB_TRY(gemm_bias_act(h->hid + (size_t)l * H, ldh, h->w<void>(L.ada2_w[l]), H, h->w<float>(L.ada2_b[l]), h->mod + (size_t)l * 6 * H, ldm,
                            B + 1, 6 * H, H, LLB_ACT_SOFTSIGN, true, s, ctr));
  }
  LLB_TRY(gemm_bias_act(h->hid + (size_t)D * H, ldh, h->w<void>(L.out_ada2_w), H, h->w<float>(L.out_ada2_b), h->modout, 2 * L.d0,
                        B + 1, 2 * L.d0, H, LLB_ACT_NONE, true, s, ctr));
  // 3. transformer blocks
  const float q_scale = 1.4426950408889634f / sqrtf((float)DIT_DH);
  // Latency regime (a handful of molecules, e.g. the reference's per-prompt batches of 6): below ~2000 token rows the
  // fused block tails occupy only 2 M / 256 row groups of 8 SMs each and stream their weights through too few TMA rings
  // (fc2 + LN 33 us vs 19 + 9 us for GEMM<64> + row kernel at 406 rows), so the unfused pair is used unless
  // LLB_FUSED_LN says otherwise.  Measured cross-over: 978 rows 2.54 vs 3.06 ms/step, 3870 rows 4.45 vs 4.20.
  const bool latency_regime = dit_latency_regime(h);
  const bool fused_ln = gemm_ln_supported(H, H) && gemm_ln_supported(H, F) && gemm_ln_enabled() && !latency_regime;
  // LLB_FUSED_LN=0: GEMM + row kernel everywhere; default: both block halves fused on the CTA-pair kernel when H = 1024
  // (other widths have no fused kernel: a full row must fit four pairs' tensor memory).
  // LLB_ATTN=2: tcgen05 attention (two heads per 128-row tile, P in tensor memory; needs an even head count and molecules of at
  // most 64 atoms); default: mma.sync attention fed by TMA, on a 64-row tile unless a molecule of the batch has more atoms.
  static const bool attn_umma_env = getenv("LLB_ATTN") && getenv("LLB_ATTN")[0] == '2';
  const bool attn_umma = attn_umma_env && L.heads % 2 == 0;
  const bool fused_pair = fused_ln;
  const size_t part_rows = (size_t)(M < 640 ? M : 640) * LLB_DIT_SPLITK;   // rows x slices the split-K buffer h->part holds (dit_carve)
  const size_t ln_sync_bytes = gemm_ln_pair_workspace_bytes();
  for (int l = 0; l < D; ++l) {
    const float* mod = h->mod + (size_t)l * 6 * H;   // row stride ldm
    // Block 0 sees the SAME token embedding in the conditional and the unconditional half and attention has no
    // conditioning, so its qkv GEMM and attention run once on Mtok rows; the halves part ways at the first modulation.
    const bool share0 = l == 0 && h->passes == 2 && fused_ln;
    ctr->slot = LLB_PROF_GEMM_QKV;
    EpiQKV eq{h->qkv, 3 * H, H, h->w<float>(L.qn_w[l]), h->w<float>(L.qn_b[l]), h->w<float>(L.kn_w[l]), h->w<float>(L.kn_b[l]), q_scale};
    // The first kernel of the blocks is launched the ordinary way: the row kernels prefetch their modulation vectors AHEAD of
    // their dependency wait, and with a full dependency here everything the adaLN GEMMs wrote is complete before any kernel of a
    // block can run any code at all -- by construction, not by the SMs happening to be full.
    if (l == 0) pdl_full_barrier_next() = true;
    // latency regime: 128-wide tiles while they fit one wave (twice the CTAs streaming the weight, half the MMAs per CTA)
    if (latency_regime && ceil_div(M, 128) * ceil_div(3 * H, 128) <= num_sms())
      LLB_TRY((launch_gemm<128>(h->xb, H, h->w<void>(L.qkv_w[l]), H, M, 3 * H, H, eq, s, ctr)));
    else
      LLB_TRY((launch_gemm<256>(h->xb, H, h->w<void>(L.qkv_w[l]), H, share0 ? Mtok : M, 3 * H, H, eq, s, ctr)));
    pdl_full_barrier_next() = false;   // (the CTA-pair kernel is launched the ordinary way anyway and does not consume the flag)
    {
      const int seqs = (share0 ? 1 : h->passes) * B;
      CUtensorMap tmQKV;
      LLB_TRY(make_tensor_map_2d(&tmQKV, h->qkv, 2, seqs / B * Mtok, 3 * H, 3 * H, DIT_DH, 64, 128));
      if (attn_umma && h->max_n <= 64) {
        const int units = seqs * (L.heads / 2);
        LLB_TRY(launch_kernel(ctr, LLB_PROF_ATTENTION, false, dit_attention_umma4_kernel, dim3(units < num_sms() ? units : num_sms()),
                              dim3(ATT4_THREADS), ATT4_SMEM, s, tmQKV, h->attn, h->mol_off, B, Mtok, H, L.heads, units));
      } else if (h->max_n <= 64) {
        LLB_TRY(launch_kernel(ctr, LLB_PROF_ATTENTION, true, dit_attention_tma_kernel<64>, dim3((unsigned)(seqs * L.heads)), dim3(128), 0, s, tmQKV,
                              h->attn, h->mol_off, B, Mtok, H, L.heads));
      } else {
        LLB_TRY(launch_kernel(ctr, LLB_PROF_ATTENTION, true, dit_attention_tma_kernel<128>, dim3((unsigned)(seqs * L.heads)), dim3(256),
                              ATTT_SMEM128, s, tmQKV, h->attn, h->mol_off, B, Mtok, H, L.heads));
      }
    }
    // x += gate * (LN(linear(.)) (1 + scale) + shift): fused into the GEMM epilogue when a cluster can hold a full row
    RowLnArgs a;
    a.in = h->y, a.in_ld = H, a.in_bf16 = true, a.rows = M, a.width = H;
    a.row_group = h->row_group, a.mod_ld = ldm;
    a.resid = h->x, a.resid_ld = H, a.out_f32 = h->x, a.out_f32_ld = H, a.out_bf16 = h->xb, a.out_bf16_ld = H;
    GemmLnArgs f{nullptr, h->row_group, nullptr, nullptr, nullptr, ldm, h->x, H, h->xb, H};
    ctr->slot = LLB_PROF_GEMM_PROJ;
    if (fused_ln) {
      f.bias = h->w<float>(L.proj_b[l]), f.shift = mod, f.scale = mod + H, f.gate = mod + 2 * H;
      // with the shared block-0 attention both halves project the same Mtok attention rows onto their own residual rows
      for (int part = 0; part < (share0 ? 2 : 1); ++part) {
        GemmLnArgs fp = f;
        const int rows = share0 ? Mtok : M;
        fp.row_group = f.row_group + (size_t)part * Mtok, fp.x = f.x + (size_t)part * Mtok * H, fp.xb = f.xb + (size_t)part * Mtok * H;
        LLB_TRY(launch_gemm_ln_pair(h->attn, H, h->w<void>(L.proj_w[l]), H, rows, H, H, fp, h->ln_sync, ln_sync_bytes, s, ctr));
      }
    } else {
      // latency regime: K = H in two slices (twice the CTAs streaming the weight, half the k-blocks each: the k-loop is paced by
      // the bytes one SM's TMA ring can take, 406 rows: 16 blocks 3.0 us), partial products summed by the row kernel
      static const bool no_splitk_p = getenv("LLB_SPLITK") && getenv("LLB_SPLITK")[0] == '0';
      // (while the two slices' 128-wide tiles fit one wave -- up to 9 row blocks -- and the slice buffer)
      if (latency_regime && !no_splitk_p && H % 128 == 0 && ceil_div(M, 128) * (2 * H / 128) <= num_sms() && 2 * (size_t)M <= part_rows) {
        GemmGroups grp;
        grp.group_n = H, grp.group_k = H / 2, grp.split_k = true;
        LLB_TRY(gemm_bias_act(h->attn, H, h->w<void>(L.proj_w[l]), H, h->w<float>(L.proj_b[l]), h->part, 2 * H, M, 2 * H, H / 2, LLB_ACT_NONE, true, s,
                              ctr, grp));
        RowLnArgs ap = a;
        ap.in = h->part, ap.in_ld = 2 * H, ap.in_bf16 = false, ap.in_parts = 2, ap.in_part_stride = H;
        ap.shift = mod, ap.scale = mod + H, ap.gate = mod + 2 * H;
        LLB_TRY(launch_row_ln(ap, s, ctr));
      } else {
        LLB_TRY(gemm_bias_act(h->attn, H, h->w<void>(L.proj_w[l]), H, h->w<float>(L.proj_b[l]), h->y, H, M, H, H, LLB_ACT_NONE, false, s, ctr));
        a.shift = mod, a.scale = mod + H, a.gate = mod + 2 * H;
        LLB_TRY(launch_row_ln(a, s, ctr));
      }
    }
    LLB_TRY(save_x(2 * l + 1));
    ctr->slot = LLB_PROF_GEMM_FC1;
    LLB_TRY(gemm_bias_act(h->xb, H, h->w<void>(L.fc1_w[l]), H, h->w<float>(L.fc1_b[l]), h->hbuf, F, M, F, H, LLB_ACT_GELU, false, s, ctr));
    ctr->slot = LLB_PROF_GEMM_FC2;
    if (fused_pair) {
      f.bias = h->w<float>(L.fc2_b[l]), f.shift = mod + 3 * H, f.scale = mod + 4 * H, f.gate = mod + 5 * H;
      LLB_TRY(launch_gemm_ln_pair(h->hbuf, F, h->w<void>(L.fc2_w[l]), F, M, H, F, f, h->ln_sync, ln_sync_bytes, s, ctr));
    } else {
      // latency regime: K = F is cut into LLB_DIT_SPLITK slices that run as groups of one launch (4x the CTAs streaming the
      // weights, a quarter of the k-blocks each); the row kernel adds the fp32 partial products in slice order
      static const bool no_splitk = getenv("LLB_SPLITK") && getenv("LLB_SPLITK")[0] == '0';
      // four slices up to 640 rows (measured: 406 rows 2.16 -> 2.05 ms/step); beyond that four slices no longer fit one wave
      // (978 rows: 2.40 -> 2.42) but TWO do up to 9 row blocks, and a CTA's k-loop is paced by its K / 16 MMA issues (256 of them
      // for the whole K at 978 rows: the long pole of the block)
      int parts = 1;
      if (latency_regime && !no_splitk && H % 128 == 0) {
        if (M <= 640 && F % (LLB_DIT_SPLITK * 64) == 0) parts = LLB_DIT_SPLITK;
        else if (F % 128 == 0 && ceil_div(M, 128) * (2 * H / 128) <= num_sms() && 2 * (size_t)M <= part_rows) parts = 2;
      }
      const int Ks = F / parts;
      if (parts > 1) {
        GemmGroups grp;
        grp.group_n = H, grp.group_k = Ks, grp.split_k = true;
        LLB_TRY(gemm_bias_act(h->hbuf, F, h->w<void>(L.fc2_w[l]), F, h->w<float>(L.fc2_b[l]), h->part, parts * H, M, parts * H,
                              Ks, LLB_ACT_NONE, true, s, ctr, grp));
        RowLnArgs ap = a;
        ap.in = h->part, ap.in_ld = parts * H, ap.in_bf16 = false, ap.in_parts = parts, ap.in_part_stride = H;
        ap.shift = mod + 3 * H, ap.scale = mod + 4 * H, ap.gate = mod + 5 * H;
        LLB_TRY(launch_row_ln(ap, s, ctr));
      } else {
        LLB_TRY(gemm_bias_act(h->hbuf, F, h->w<void>(L.fc2_w[l]), F, h->w<float>(L.fc2_b[l]), h->y, H, M, H, F, LLB_ACT_NONE, false, s, ctr));
        a.shift = mod + 3 * H, a.scale = mod + 4 * H, a.gate = mod + 5 * H;
        LLB_TRY(launch_row_ln(a, s, ctr));
      }
    }
    LLB_TRY(save_x(2 * l + 2));
  }
  // 4. output MLP (the LayerNorm / modulation / symmetrisation tail lives in the step kernel)
  ctr->slot = LLB_PROF_GEMM_OTHER;
  LLB_TRY(gemm_bias_act(h->xb, H, h->w<void>(L.out_fc1_w), H, h->w<float>(L.out_fc1_b), h->y, H, M, H, H, LLB_ACT_GELU, false, s, ctr));
  LLB_TRY(gemm_bias_act(h->y, H, h->w<void>(L.out_fc2_w), H, h->w<float>(L.out_fc2_b), h->raw, h->raw_ld, M, L.d0, H, LLB_ACT_NONE, true, s, ctr));
  return LLB_OK;
}

static bool dit_graph_enabled() {
  static const bool on = !(getenv("LLB_GRAPH") && getenv("LLB_GRAPH")[0] == '0');
  return on;
}

// Capture dit_body on the handle's own stream (the caller's may be the legacy default stream, which cannot be captured) and
// instantiate it; the executable graph is then launched into the caller's stream.
static int dit_build_graph(llb_dit* h) {
  h->graph_state = -1;
  // a capture that cannot even begin (the caller is capturing this thread's work itself, say) is not an error of the pass either
  if (!h->capture_stream && cudaStreamCreateWithFlags(&h->capture_stream, cudaStreamNonBlocking) != cudaSuccess) {
    (void)cudaGetLastError();
    h->capture_stream = nullptr;
    return LLB_OK;
  }
  int64_t kern0[LLB_KERN_FAMILIES];
  for (int f = 0; f < LLB_KERN_FAMILIES; ++f) kern0[f] = llb_kernel_launches(f);
  const int64_t launches0 = h->ctr.launches;
  if (cudaStreamBeginCapture(h->capture_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    (void)cudaGetLastError();
    return LLB_OK;
  }
  const int rc = dit_body(h, h->capture_stream);
  cudaGraph_t g = nullptr;
  const cudaError_t e = cudaStreamEndCapture(h->capture_stream, &g);
  // the capture issued nothing: take its launches back out of the counter, replays add them
  h->graph_launches = h->ctr.launches - launches0;
  h->ctr.launches = launches0;
  for (int f = 0; f < LLB_KERN_FAMILIES; ++f) {
    h->graph_kern[f] = llb_kernel_launches(f) - kern0[f];
    note_kernel(f, -h->graph_kern[f]);
  }
  if (rc != LLB_OK || e != cudaSuccess || !g) {
    if (g) cudaGraphDestroy(g);
    (void)cudaGetLastError();
    return rc != LLB_OK ? rc : LLB_OK;   // an un-capturable launch is not an error of the pass: it runs eagerly
  }
  const cudaError_t ei = cudaGraphInstantiate(&h->body_graph, g, 0);
  cudaGraphDestroy(g);
  if (ei != cudaSuccess) {
    (void)cudaGetLastError();
    h->body_graph = nullptr;
    return LLB_OK;
  }
  h->graph_state = 1;
  return LLB_OK;
}

// One full denoiser pass over both CFG halves up to the raw output-layer rows (h->raw).
static int dit_forward(llb_dit* h, int t, cudaStream_t s) {
  const DitLayout& L = h->L;
  if (h->Mtok == 0) return LLB_OK;
  LLB_TRY(launch_kernel(&h->ctr, LLB_PROF_DIT_MISC, false, dit_cvec_kernel, dim3(ceil_div((h->B + 1) * L.H, 256)), dim3(256), 0, s,
                        h->w<float>(L.c1_table) + (size_t)t * L.H, h->cinv, h->w<float>(L.c_unc), h->cvec, h->B, L.H));
  const bool want_graph = dit_latency_regime(h) && dit_graph_enabled() && !profile_on() && h->passes_run >= 1;
  h->passes_run++;
  if (want_graph && h->graph_state == 0) LLB_TRY(dit_build_graph(h));
  if (want_graph && h->graph_state == 1) {
    LLB_CUDA_OK(cudaGraphLaunch(h->body_graph, s));
    h->ctr.launches += h->graph_launches;
    for (int f = 0; f < LLB_KERN_FAMILIES; ++f) note_kernel(f, h->graph_kern[f]);
    return LLB_OK;
  }
  return dit_body(h, s);
}

static int dit_launch_step(llb_dit* h, DitStepArgs& a, cudaStream_t s) {
  const size_t smem = dit_step_smem(h->L.N, a.passes);
  if (smem > (size_t)smem_per_block_optin()) {
    // T does not fit (N > 71 with guidance): its home is the raw output-layer rows, row (p, atom i) = raw row p Mtok + off + i
    // (raw_ld >= d0).  Nothing reads those rows after the step kernel: the next denoiser pass rewrites them, the logits dump
    // returns T itself, and the backward recomputes its own copy from the saved residual stream.
    a.tg = h->raw, a.tg_ld = h->raw_ld;
    const size_t gsmem = dit_step_smem(h->L.N, a.passes, false);
    if (h->B <= num_sms())
      return launch_kernel(&h->ctr, LLB_PROF_DIT_STEP, false, dit_step_kernel<512, true>, dim3(h->B), dim3(512), gsmem, s, a, h->tables);
    return launch_kernel(&h->ctr, LLB_PROF_DIT_STEP, false, dit_step_kernel<256, true>, dim3(h->B), dim3(256), gsmem, s, a, h->tables);
  }
  if (h->B <= num_sms())   // fewer molecules than SMs: wider CTAs
    return launch_kernel(&h->ctr, LLB_PROF_DIT_STEP, false, dit_step_kernel<512>, dim3(h->B), dim3(512), smem, s, a, h->tables);
  return launch_kernel(&h->ctr, LLB_PROF_DIT_STEP, false, dit_step_kernel<256>, dim3(h->B), dim3(256), smem, s, a, h->tables);
}

static void dit_fill_step(llb_dit* h, DitStepArgs& a, int t) {
  a = DitStepArgs{};
  a.mol_off = h->mol_off;
  a.B = h->B, a.N = h->L.N, a.Mtok = h->Mtok, a.passes = h->passes;
  a.X = h->stX, a.E = h->stE;
  a.beta_t = h->betas[t], a.abar_s = h->abar[t - 1], a.abar_t = h->abar[t];
  a.guide_scale = h->cfg.guide_scale;
  a.stream_id = (uint32_t)(t - 1);
  a.mol_base = h->mol_base;
}

// Batch binding shared by llb_dit_begin and llb_dit_denoise_c: workspace carve-up and the varlen row bookkeeping.
static int dit_bind(llb_dit* h, void* workspace, size_t workspace_bytes, int B, const int32_t* n_nodes_host, int64_t mol_index_base,
                    cudaStream_t s) {
  const DitLayout& L = h->L;
  std::vector<int32_t> off(B + 1, 0);
  for (int b = 0; b < B; ++b) {
    LLB_CHECK_ARG(n_nodes_host[b] >= 0 && n_nodes_host[b] <= L.N, "dit: n_nodes[%d]=%d outside [0,%d]", b, n_nodes_host[b], L.N);
    off[b + 1] = off[b] + n_nodes_host[b];
  }
  const int Mtok = off[B];
  int max_n = 0;
  for (int b = 0; b < B; ++b) max_n = n_nodes_host[b] > max_n ? n_nodes_host[b] : max_n;
  size_t need = 0;
  LLB_TRY(dit_carve(h, workspace, workspace_bytes, B, Mtok, &need));
  if (need > workspace_bytes) return fail(LLB_ERR_WORKSPACE, "dit: workspace needs %zu bytes, got %zu", need, workspace_bytes);
  h->drop_graph();   // the captured launches carry the previous binding's pointers and sizes
  h->B = B, h->Mtok = Mtok, h->mol_base = mol_index_base, h->max_n = max_n;
  std::vector<int32_t> row_mol(Mtok > 0 ? Mtok : 1), row_group(h->passes * Mtok > 0 ? h->passes * Mtok : 1);
  for (int b = 0; b < B; ++b)
    for (int r = off[b]; r < off[b + 1]; ++r) {
      row_mol[r] = b;
      row_group[r] = b;
      if (h->passes == 2) row_group[Mtok + r] = B;
    }
  LLB_CUDA_OK(cudaMemcpyAsync(h->mol_off, off.data(), (B + 1) * 4, cudaMemcpyHostToDevice, s));
  if (Mtok > 0) {
    LLB_CUDA_OK(cudaMemcpyAsync(h->row_mol, row_mol.data(), (size_t)Mtok * 4, cudaMemcpyHostToDevice, s));
    LLB_CUDA_OK(cudaMemcpyAsync(h->row_group, row_group.data(), (size_t)h->passes * Mtok * 4, cudaMemcpyHostToDevice, s));
  }
  LLB_CUDA_OK(cudaMemsetAsync(h->ln_sync, 0, gemm_ln_pair_workspace_bytes(), s));   // mailbox tags start from a known state
  return LLB_OK;
}

extern "C" {

int llb_dit_packed_bytes(const llb_dit_config* cfg, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes, "llb_dit_packed_bytes: null argument");
  DitLayout L;
  LLB_TRY(make_layout(*cfg, L));
  *bytes = L.total;
  return LLB_OK;
}

int llb_dit_pack_weights(const llb_dit_config* cfg, const llb_dit_weights* w, void* packed, size_t packed_bytes,
                         llb_stream_t stream) {
  LLB_TRY(require_sm100());
  LLB_CHECK_ARG(cfg && w && packed, "llb_dit_pack_weights: null argument");
  DitLayout L;
  LLB_TRY(make_layout(*cfg, L));
  if (packed_bytes < L.total) return fail(LLB_ERR_WORKSPACE, "dit: packed blob needs %zu bytes, got %zu", L.total, packed_bytes);
  cudaStream_t s = (cudaStream_t)stream;
  uint8_t* base = (uint8_t*)packed;
  const int H = L.H, F = L.F, D = L.D;
  auto bf = [&](size_t off) { return reinterpret_cast<__nv_bfloat16*>(base + off); };
  auto f32 = [&](size_t off) { return reinterpret_cast<float*>(base + off); };
  auto cp = [&](size_t off, const float* src, size_t n) {
    return cudaMemcpyAsync(base + off, src, n * 4, cudaMemcpyDeviceToDevice, s);
  };
  LLB_TRY(launch_f32_to_bf16(w->x_embed_w, L.d0, bf(L.x_embed_w), L.K0, H, L.d0, L.K0, s, nullptr));
  for (int d = 0; d < L.ydim; ++d)
    LLB_TRY(launch_f32_to_bf16(w->y_mlp2_w[d], H, bf(L.cond_w) + (size_t)d * H, L.KC, H, H, H, s, nullptr));
  LLB_TRY(launch_f32_to_bf16(w->txt_w, L.tdim, bf(L.cond_w) + (size_t)L.ydim * H, L.KC, H, L.tdim, L.tdim, s, nullptr));
  for (int l = 0; l < D; ++l) {
    LLB_TRY(launch_f32_to_bf16(w->ada0_w[l], H, bf(L.ada0_w) + (size_t)l * H * H, H, H, H, H, s, nullptr));
    LLB_CUDA_OK(cp(L.ada0_b + (size_t)l * H * 4, w->ada0_b[l], H));
    LLB_TRY(launch_f32_to_bf16(w->qkv_w[l], H, bf(L.qkv_w[l]), H, 3 * H, H, H, s, nullptr));
    LLB_TRY(launch_f32_to_bf16(w->proj_w[l], H, bf(L.proj_w[l]), H, H, H, H, s, nullptr));
    LLB_TRY(launch_f32_to_bf16(w->fc1_w[l], H, bf(L.fc1_w[l]), H, F, H, H, s, nullptr));
    LLB_TRY(launch_f32_to_bf16(w->fc2_w[l], F, bf(L.fc2_w[l]), F, H, F, F, s, nullptr));
    LLB_TRY(launch_f32_to_bf16(w->ada2_w[l], H, bf(L.ada2_w[l]), H, 6 * H, H, H, s, nullptr));
    LLB_CUDA_OK(cp(L.qn_w[l], w->q_norm_w[l], DIT_DH));
    LLB_CUDA_OK(cp(L.qn_b[l], w->q_norm_b[l], DIT_DH));
    LLB_CUDA_OK(cp(L.kn_w[l], w->k_norm_w[l], DIT_DH));
    LLB_CUDA_OK(cp(L.kn_b[l], w->k_norm_b[l], DIT_DH));
    LLB_CUDA_OK(cp(L.proj_b[l], w->proj_b[l], H));
    LLB_CUDA_OK(cudaMemsetAsync(static_cast<uint8_t*>(packed) + L.proj_b[l] + H * 4, 0, (size_t)H * 4, s));
    LLB_CUDA_OK(cp(L.fc1_b[l], w->fc1_b[l], F));
    LLB_CUDA_OK(cp(L.fc2_b[l], w->fc2_b[l], H));
    LLB_CUDA_OK(cudaMemsetAsync(static_cast<uint8_t*>(packed) + L.fc2_b[l] + H * 4, 0, (size_t)(LLB_DIT_SPLITK - 1) * H * 4, s));
    LLB_CUDA_OK(cp(L.ada2_b[l], w->ada2_b[l], 6 * H));
  }
  LLB_TRY(launch_f32_to_bf16(w->out_ada0_w, H, bf(L.ada0_w) + (size_t)D * H * H, H, H, H, H, s, nullptr));
  LLB_CUDA_OK(cp(L.ada0_b + (size_t)D * H * 4, w->out_ada0_b, H));
  LLB_TRY(launch_f32_to_bf16(w->out_fc1_w, H, bf(L.out_fc1_w), H, H, H, H, s, nullptr));
  LLB_TRY(launch_f32_to_bf16(w->out_fc2_w, H, bf(L.out_fc2_w), H, L.d0, H, H, s, nullptr));
  LLB_TRY(launch_f32_to_bf16(w->out_ada2_w, H, bf(L.out_ada2_w), H, 2 * L.d0, H, H, s, nullptr));
  LLB_CUDA_OK(cp(L.out_fc1_b, w->out_fc1_b, H));
  LLB_CUDA_OK(cp(L.out_fc2_b, w->out_fc2_b, L.d0));
  LLB_CUDA_OK(cp(L.out_ada2_b, w->out_ada2_b, 2 * L.d0));
  LLB_CUDA_OK(cp(L.x_ln_w, w->x_embed_ln_w, H));
  LLB_CUDA_OK(cp(L.x_ln_b, w->x_embed_ln_b, H));
  for (int d = 0; d < L.ydim; ++d) {
    LLB_CUDA_OK(cp(L.y_mlp0_w + (size_t)d * H * 4, w->y_mlp0_w[d], H));
    LLB_CUDA_OK(cp(L.y_mlp0_b + (size_t)d * H * 4, w->y_mlp0_b[d], H));
  }
  LLB_CUDA_OK(cp(L.y_drop, w->y_drop, (size_t)L.ydim * H));
  LLB_CUDA_OK(cp(L.txt_drop, w->txt_drop, H));
  LLB_CUDA_OK(cp(L.txt_b, w->txt_b, H));
  LLB_CUDA_OK(cp(L.tables, w->x_marg, DIT_XC));
  LLB_CUDA_OK(cp(L.tables + DIT_XC * 4, w->e_marg, DIT_EC));
  LLB_CUDA_OK(cp(L.tables + (DIT_XC + DIT_EC) * 4, w->xe, DIT_XC * DIT_EC));
  LLB_CUDA_OK(cp(L.tables + (DIT_XC + DIT_EC + DIT_XC * DIT_EC) * 4, w->ex, DIT_XC * DIT_EC));
  LLB_CUDA_OK(cp(L.betas, w->betas, L.T + 1));
  LLB_CUDA_OK(cp(L.abar, w->alphas_bar, L.T + 1));
  // timestep-embedding table for t = 0..T (t_embedder, conditions.py:53-58), fp32 on CUDA cores (set-up only)
  {
    float* feat = f32(L.setup_scratch);                  // (T+1,256)
    float* hidden = feat + (size_t)(L.T + 1) * 256;      // (T+1,H)
    LLB_TRY(launch_kernel(nullptr, NO_PROF, false, dit_tfeat_kernel, dim3(L.T + 1), dim3(128), 0, s, feat, L.T));
    LLB_TRY(launch_linear_f32(feat, 256, w->t_mlp0_w, 256, w->t_mlp0_b, hidden, H, L.T + 1, H, 256, LLB_ACT_SILU, s, nullptr));
    LLB_TRY(launch_linear_f32(hidden, H, w->t_mlp2_w, H, w->t_mlp2_b, f32(L.c1_table), H, L.T + 1, H, H, LLB_ACT_NONE, s, nullptr));
  }
  return launch_kernel(nullptr, NO_PROF, false, dit_cunc_kernel, dim3(ceil_div(H, 256)), dim3(256), 0, s, w->y_drop, w->txt_drop, f32(L.c_unc),
                       L.ydim, H);
}

int llb_dit_create(const llb_dit_config* cfg, const void* packed, size_t packed_bytes, llb_dit** out) {
  LLB_TRY(require_sm100());
  LLB_CHECK_ARG(cfg && packed && out, "llb_dit_create: null argument");
  llb_dit* h = new llb_dit();
  h->cfg = *cfg;
  int st = make_layout(*cfg, h->L);
  if (st != LLB_OK) {
    delete h;
    return st;
  }
  if (packed_bytes < h->L.total) {
    size_t need = h->L.total;
    delete h;
    return fail(LLB_ERR_WORKSPACE, "dit: packed blob needs %zu bytes, got %zu", need, packed_bytes);
  }
  h->blob = (const uint8_t*)packed;
  h->passes = (cfg->guide_scale != 1.0f) ? 2 : 1;
  // host copies of the small tables (synchronous: create is not on the hot path)
  h->betas.resize(cfg->timesteps + 1);
  h->abar.resize(cfg->timesteps + 1);
  cudaError_t e = cudaMemcpy(h->betas.data(), h->blob + h->L.betas, (cfg->timesteps + 1) * 4, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(h->abar.data(), h->blob + h->L.abar, (cfg->timesteps + 1) * 4, cudaMemcpyDeviceToHost);
  float tb[DIT_XC + DIT_EC + 2 * DIT_XC * DIT_EC];
  if (e == cudaSuccess) e = cudaMemcpy(tb, h->blob + h->L.tables, sizeof(tb), cudaMemcpyDeviceToHost);
  if (e != cudaSuccess) {
    delete h;
    return fail(LLB_ERR_CUDA, "dit: reading tables back failed: %s", cudaGetErrorString(e));
  }
  memcpy(h->tables.x_marg, tb, DIT_XC * 4);
  memcpy(h->tables.e_marg, tb + DIT_XC, DIT_EC * 4);
  memcpy(h->tables.xe, tb + DIT_XC + DIT_EC, DIT_XC * DIT_EC * 4);
  memcpy(h->tables.ex, tb + DIT_XC + DIT_EC + DIT_XC * DIT_EC, DIT_XC * DIT_EC * 4);
  *out = h;
  return LLB_OK;
}

void llb_dit_destroy(llb_dit* h) { delete h; }

int llb_dit_workspace_bytes(const llb_dit_config* cfg, int max_molecules, size_t* bytes) {
  LLB_CHECK_ARG(cfg && bytes && max_molecules >= 1, "llb_dit_workspace_bytes: bad argument");
  llb_dit tmp;
  tmp.cfg = *cfg;
  LLB_TRY(make_layout(*cfg, tmp.L));
  return dit_carve(&tmp, nullptr, 0, max_molecules, max_molecules * cfg->max_nodes, bytes);
}

int llb_dit_begin(llb_dit* h, void* workspace, size_t workspace_bytes, int B, const int32_t* n_nodes_host,
                  const float* props, const float* txt, int64_t mol_index_base, llb_stream_t stream) {
  LLB_CHECK_ARG(h && workspace && n_nodes_host && props && txt && B >= 1, "llb_dit_begin: bad argument");
  cudaStream_t s = (cudaStream_t)stream;
  const DitLayout& L = h->L;
  LLB_TRY(dit_bind(h, workspace, workspace_bytes, B, n_nodes_host, mol_index_base, s));
  // the copies above read pageable host memory: they have been staged by the time cudaMemcpyAsync returns
  LLB_TRY(launch_kernel(&h->ctr, NO_PROF, false, dit_cond_operand_kernel, dim3(B, L.ydim + 1), dim3(256), 0, s, props, txt,
                        h->w<float>(L.y_mlp0_w), h->w<float>(L.y_mlp0_b), h->acond, h->missing, L.ydim, L.tdim, L.H, L.KC));
  LLB_TRY(gemm_bias_act(h->acond, L.KC, h->w<void>(L.cond_w), L.KC, nullptr, h->cinv, L.H, B, L.H, L.KC, LLB_ACT_NONE, true, s, &h->ctr));
  return launch_kernel(&h->ctr, NO_PROF, false, dit_cond_fixup_kernel, dim3(ceil_div(B * L.H, 256)), dim3(256), 0, s, h->cinv, h->missing,
                       h->w<float>(L.y_drop), h->w<float>(L.txt_drop), h->w<float>(L.txt_b), B, L.ydim, L.H);
}

int llb_dit_set_state(llb_dit* h, const int8_t* X, const int8_t* E, llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0 && X && E, "llb_dit_set_state: no batch bound or null state");
  cudaStream_t s = (cudaStream_t)stream;
  LLB_CUDA_OK(cudaMemcpyAsync(h->stX, X, (size_t)h->B * h->L.N, cudaMemcpyDeviceToDevice, s));
  LLB_CUDA_OK(cudaMemcpyAsync(h->stE, E, (size_t)h->B * h->L.N * h->L.N, cudaMemcpyDeviceToDevice, s));
  return LLB_OK;
}

int llb_dit_get_state(llb_dit* h, int8_t* X, int8_t* E, llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0 && X && E, "llb_dit_get_state: no batch bound or null state");
  cudaStream_t s = (cudaStream_t)stream;
  LLB_CUDA_OK(cudaMemcpyAsync(X, h->stX, (size_t)h->B * h->L.N, cudaMemcpyDeviceToDevice, s));
  LLB_CUDA_OK(cudaMemcpyAsync(E, h->stE, (size_t)h->B * h->L.N * h->L.N, cudaMemcpyDeviceToDevice, s));
  return LLB_OK;
}

int llb_dit_init_state(llb_dit* h, uint64_t seed, const float* qX0, const float* qE0, llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0, "llb_dit_init_state: no batch bound");
  LLB_CHECK_ARG((qX0 == nullptr) == (qE0 == nullptr), "llb_dit_init_state: pass both noise tensors or neither");
  return launch_kernel(&h->ctr, NO_PROF, false, dit_init_state_kernel, dim3(h->B), dim3(256), 0, (cudaStream_t)stream, h->stX, h->stE, h->mol_off,
                       h->L.N, qX0, qE0, seed, (uint32_t)h->L.T, h->mol_base, h->tables);
}

int llb_dit_denoise(llb_dit* h, int t, int unconditioned, float* logits_X, float* logits_E, llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0 && logits_X && logits_E, "llb_dit_denoise: no batch bound or null output");
  LLB_CHECK_ARG(t >= 1 && t <= h->L.T, "llb_dit_denoise: t=%d outside [1,%d]", t, h->L.T);
  LLB_CHECK_ARG(!unconditioned || h->passes == 2, "llb_dit_denoise: guide_scale == 1 has no unconditional pass");
  cudaStream_t s = (cudaStream_t)stream;
  LLB_TRY(dit_forward(h, t, s));
  DitStepArgs a;
  dit_fill_step(h, a, t);
  a.raw = h->raw, a.raw_ld = h->raw_ld, a.modout = h->modout;
  a.sample = 0, a.dump_logits = 1, a.dump_pass = unconditioned ? 1 : 0, a.dumpX = logits_X, a.dumpE = logits_E;
  return dit_launch_step(h, a, s);
}

int llb_dit_denoise_c(llb_dit* h, void* workspace, size_t workspace_bytes, int B, const int32_t* n_nodes_host, const int8_t* X,
                      const int8_t* E, const float* c, float* logits_X, float* logits_E, void* saved, size_t saved_bytes,
                      llb_stream_t stream) {
  LLB_CHECK_ARG(h && workspace && n_nodes_host && X && E && c && logits_X && logits_E && B >= 1, "llb_dit_denoise_c: bad argument");
  LLB_CHECK_ARG(h->passes == 1, "llb_dit_denoise_c: needs a handle created with guide_scale == 1 (one pass)");
  cudaStream_t s = (cudaStream_t)stream;
  const DitLayout& L = h->L;
  const int H = L.H;
  if (saved) LLB_TRY(dit_grad_check_n(L, "llb_dit_denoise_c with a saved buffer"));
  LLB_TRY(dit_bind(h, workspace, workspace_bytes, B, n_nodes_host, 0, s));
  const int Mtok = h->Mtok;
  DitSaved sv{};
  if (saved) {
    size_t need = 0;
    dit_saved_carve(L, saved, B, Mtok, &sv, &need);
    if (saved_bytes < need) return fail(LLB_ERR_WORKSPACE, "dit: saved buffer needs %zu bytes, got %zu", need, saved_bytes);
  }
  LLB_CUDA_OK(cudaMemcpyAsync(h->stX, X, (size_t)B * L.N, cudaMemcpyDeviceToDevice, s));
  LLB_CUDA_OK(cudaMemcpyAsync(h->stE, E, (size_t)B * L.N * L.N, cudaMemcpyDeviceToDevice, s));
  // the caller's c replaces cinv + the timestep table; row B (the unconditional row of a guided pass) feeds nothing here
  LLB_TRY(launch_f32_to_bf16(c, H, h->cvec, H, B, H, H, s, &h->ctr));
  LLB_CUDA_OK(cudaMemsetAsync(h->cvec + (size_t)B * H, 0, (size_t)H * 2, s));
  if (Mtok > 0) {
    h->save_x = saved ? sv.xs : nullptr;
    const int rc = dit_body(h, s);
    h->save_x = nullptr;
    LLB_TRY(rc);
  }
  if (saved) {
    LLB_CUDA_OK(cudaMemcpyAsync(sv.mol_off, h->mol_off, (size_t)(B + 1) * 4, cudaMemcpyDeviceToDevice, s));
    if (Mtok > 0) LLB_CUDA_OK(cudaMemcpyAsync(sv.row_mol, h->row_mol, (size_t)Mtok * 4, cudaMemcpyDeviceToDevice, s));
    LLB_CUDA_OK(cudaMemcpyAsync(sv.cvec, h->cvec, (size_t)B * H * 2, cudaMemcpyDeviceToDevice, s));
    LLB_CUDA_OK(cudaMemcpyAsync(sv.mod, h->mod, (size_t)B * L.D * 6 * H * 4, cudaMemcpyDeviceToDevice, s));
    LLB_CUDA_OK(cudaMemcpyAsync(sv.modout, h->modout, (size_t)B * 2 * L.d0 * 4, cudaMemcpyDeviceToDevice, s));
  }
  // the step kernel's logits dump only (no schedule lookup: t reaches the denoiser through c alone)
  DitStepArgs a{};
  a.mol_off = h->mol_off;
  a.B = B, a.N = L.N, a.Mtok = Mtok, a.passes = 1;
  a.X = h->stX, a.E = h->stE;
  a.raw = h->raw, a.raw_ld = h->raw_ld, a.modout = h->modout;
  a.sample = 0, a.dump_logits = 1, a.dump_pass = 0, a.dumpX = logits_X, a.dumpE = logits_E;
  return dit_launch_step(h, a, s);
}

int llb_dit_step(llb_dit* h, int t, uint64_t seed, const float* qX, const float* qE, float* prob_X, float* prob_E,
                 llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0, "llb_dit_step: no batch bound");
  LLB_CHECK_ARG(t >= 1 && t <= h->L.T, "llb_dit_step: t=%d outside [1,%d]", t, h->L.T);
  LLB_CHECK_ARG((qX == nullptr) == (qE == nullptr), "llb_dit_step: pass both noise tensors or neither");
  cudaStream_t s = (cudaStream_t)stream;
  LLB_TRY(dit_forward(h, t, s));
  DitStepArgs a;
  dit_fill_step(h, a, t);
  a.raw = h->raw, a.raw_ld = h->raw_ld, a.modout = h->modout;
  a.sample = 1, a.seed = seed, a.qX = qX, a.qE = qE, a.dumpX = prob_X, a.dumpE = prob_E;
  return dit_launch_step(h, a, s);
}

int llb_dit_sample(llb_dit* h, int t_first, int t_last, uint64_t seed, const float* qX_all, const float* qE_all,
                   llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0, "llb_dit_sample: no batch bound");
  LLB_CHECK_ARG(t_first <= h->L.T && t_last >= 1 && t_first >= t_last, "llb_dit_sample: bad range %d..%d", t_first, t_last);
  const size_t nx = (size_t)h->B * h->L.N * DIT_XC, ne = (size_t)h->B * h->L.N * h->L.N * DIT_EC;
  for (int t = t_first; t >= t_last; --t) {
    const float* qx = qX_all ? qX_all + (size_t)(t - 1) * nx : nullptr;
    const float* qe = qE_all ? qE_all + (size_t)(t - 1) * ne : nullptr;
    LLB_TRY(llb_dit_step(h, t, seed, qx, qe, nullptr, nullptr, stream));
  }
  return LLB_OK;
}

int64_t llb_dit_launch_count(const llb_dit* h) { return h ? h->ctr.launches : 0; }

int llb_dit_graph_state(const llb_dit* h) { return h ? h->graph_state : 0; }

int llb_dit_posterior_sample(llb_dit* h, int t, const float* lc_X, const float* lc_E, const float* lu_X,
                             const float* lu_E, uint64_t seed, const float* qX, const float* qE, float* prob_X,
                             float* prob_E, llb_stream_t stream) {
  LLB_CHECK_ARG(h && h->B > 0 && lc_X && lc_E, "llb_dit_posterior_sample: no batch bound or null logits");
  LLB_CHECK_ARG(h->passes == 1 || (lu_X && lu_E), "llb_dit_posterior_sample: guidance needs the unconditional logits");
  LLB_CHECK_ARG(t >= 1 && t <= h->L.T, "llb_dit_posterior_sample: t=%d outside [1,%d]", t, h->L.T);
  DitStepArgs a;
  dit_fill_step(h, a, t);
  a.lcX = lc_X, a.lcE = lc_E, a.luX = lu_X, a.luE = lu_E;
  a.sample = 1, a.seed = seed, a.qX = qX, a.qE = qE, a.dumpX = prob_X, a.dumpE = prob_E;
  return dit_launch_step(h, a, (cudaStream_t)stream);
}

}  // extern "C"

LLB_STEP_TRACE_INSTALL(llb_trace_install_dit)
