#include "llb_rowops.cuh"

namespace llb {

namespace {

struct RowLnDev {
  const void* in;
  int in_ld, in_bf16, rows, width, normalize, in_parts, in_part_stride;
  const float *gamma, *beta;
  const int32_t* row_group;
  const float *shift, *scale, *gate;
  int mod_ld, act;
  const float* resid;
  int resid_ld;
  const float* addvec;
  int addvec_ld;
  float* out_f32;
  int out_f32_ld;
  __nv_bfloat16* out_bf16;
  int out_bf16_ld, dup_rows, l2_normalize;
  int valid;   // row_ln_kernel only (the register-resident kernel runs valid == width)
};

// Compile-time feature mask of the register-resident kernel.  F_RUNTIME keeps every test on the runtime
// descriptor (cold variants); the hot variants are instantiated with the exact mask so that the body is
// straight-line code and the compiler can hoist every load above the reductions.
enum : unsigned {
  F_IN_BF16 = 1u << 0, F_NORM = 1u << 1, F_GAMMA = 1u << 2, F_MOD = 1u << 3, F_GELU = 1u << 4, F_GATE = 1u << 5,
  F_RESID = 1u << 6, F_ADDVEC = 1u << 7, F_OUT_F32 = 1u << 8, F_OUT_BF16 = 1u << 9, F_RUNTIME = 1u << 31
};

__device__ __forceinline__ float4 load4(const void* base, bool is_bf16, size_t idx) {
  if (is_bf16) {
    const uint2 u = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(base) + idx);
    return make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
  }
  return *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(base) + idx);
}

__device__ __forceinline__ float act_rt(float x, int act) {
  switch (act) {
    case LLB_ACT_GELU: return gelu_fast(x);
    case LLB_ACT_SILU: return silu(x);
    case LLB_ACT_SOFTSIGN: return softsign(x);
  }
  return x;
}

// Fallback for widths that are not a multiple of 128, and for rows whose last width - valid columns are padding: one warp per row,
// three sweeps over L1/L2.  Statistics over the first `valid` columns; the padding columns are written as 0.
__global__ void __launch_bounds__(256) row_ln_kernel(RowLnDev a) {
  pdl_launch_dependents();
  pdl_wait();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= a.rows) return;
  const size_t in_off = (size_t)row * a.in_ld;
  const int W = a.width, V = a.valid;
  float mean = 0.f, rstd = 1.f;
  if (a.normalize || a.l2_normalize) {
    float s = 0.f;
    if (a.normalize) {
      for (int c = lane * 4; c < W; c += 128) {
        const float4 v = load4(a.in, a.in_bf16, in_off + c);
        s += ((c < V ? v.x : 0.f) + (c + 1 < V ? v.y : 0.f)) + ((c + 2 < V ? v.z : 0.f) + (c + 3 < V ? v.w : 0.f));
      }
      mean = warp_sum(s) / (float)V;
    }
    float q = 0.f;
    for (int c = lane * 4; c < W; c += 128) {
      const float4 v = load4(a.in, a.in_bf16, in_off + c);
      const float d0 = c < V ? v.x - mean : 0.f, d1 = c + 1 < V ? v.y - mean : 0.f;
      const float d2 = c + 2 < V ? v.z - mean : 0.f, d3 = c + 3 < V ? v.w - mean : 0.f;
      q += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
    q = warp_sum(q);
    rstd = a.l2_normalize ? rsqrtf(q) : rsqrtf(q / (float)V + 1e-5f);
  }
  const int g = a.row_group ? a.row_group[row] : row;
  const float* sh = a.shift ? a.shift + (size_t)g * a.mod_ld : nullptr;
  const float* sc = a.scale ? a.scale + (size_t)g * a.mod_ld : nullptr;
  const float* gt = a.gate ? a.gate + (size_t)g * a.mod_ld : nullptr;
  const float* av = a.addvec ? a.addvec + (size_t)g * a.addvec_ld : nullptr;
  for (int c = lane * 4; c < W; c += 128) {
    const float4 v4 = load4(a.in, a.in_bf16, in_off + c);
    float v[4] = {v4.x, v4.y, v4.z, v4.w};
    float r[4] = {0.f, 0.f, 0.f, 0.f};
    if (a.resid) {
      const float4 r4 = *reinterpret_cast<const float4*>(a.resid + (size_t)row * a.resid_ld + c);
      r[0] = r4.x, r[1] = r4.y, r[2] = r4.z, r[3] = r4.w;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float x = (v[i] - mean) * rstd;
      if (a.gamma) x = x * __ldg(a.gamma + c + i) + __ldg(a.beta + c + i);
      if (sc) x = x * (1.0f + __ldg(sc + c + i)) + __ldg(sh + c + i);
      x = act_rt(x, a.act);
      if (gt) x *= __ldg(gt + c + i);
      if (a.resid) x += r[i];
      if (av) x += __ldg(av + c + i);
      v[i] = c + i < V ? x : 0.f;
    }
    if (a.out_f32) {
      const float4 o = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(a.out_f32 + (size_t)row * a.out_f32_ld + c) = o;
      if (a.dup_rows) *reinterpret_cast<float4*>(a.out_f32 + (size_t)(row + a.dup_rows) * a.out_f32_ld + c) = o;
    }
    if (a.out_bf16) {
      const uint2 o = make_uint2(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]));
      *reinterpret_cast<uint2*>(a.out_bf16 + (size_t)row * a.out_bf16_ld + c) = o;
      if (a.dup_rows) *reinterpret_cast<uint2*>(a.out_bf16 + (size_t)(row + a.dup_rows) * a.out_bf16_ld + c) = o;
    }
  }
}

// Backward of row_ln_kernel (see RowLnBwdArgs).  Three sweeps over the row: statistics, the two sums of the LayerNorm backward,
// output.  Any width; columns past `valid` are written as 0.
__global__ void __launch_bounds__(256) row_ln_bwd_kernel(RowLnBwdArgs a) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= a.rows) return;
  const int W = a.width, V = a.valid;
  const size_t xo = (size_t)row * a.x_ld, yo = (size_t)row * a.dy_ld;
  auto xv = [&](int c) {
    return a.x_bf16 ? __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(a.x)[xo + c]) : reinterpret_cast<const float*>(a.x)[xo + c];
  };
  float s = 0.f;
  for (int c = lane; c < V; c += 32) s += xv(c);
  const float mean = warp_sum(s) / (float)V;
  float q = 0.f;
  for (int c = lane; c < V; c += 32) {
    const float d = xv(c) - mean;
    q += d * d;
  }
  const float rstd = rsqrtf(warp_sum(q) / (float)V + 1e-5f);
  const int g = a.row_group ? a.row_group[row] : row;
  const float* sh = a.shift ? a.shift + (size_t)g * a.mod_ld : nullptr;
  const float* sc = a.scale ? a.scale + (size_t)g * a.mod_ld : nullptr;
  const float* gt = a.gate ? a.gate + (size_t)g * a.mod_ld : nullptr;
  // column c -> xh, dy, dt (gradient at t), and the factor d(t)/d(xh)
  auto col = [&](int c, float& xh, float& dyv, float& t, float& dt, float& mul) {
    xh = (xv(c) - mean) * rstd;
    if (a.gamma) mul = __ldg(a.gamma + c), t = fmaf(xh, mul, __ldg(a.beta + c));
    else if (sc) mul = 1.0f + __ldg(sc + c), t = fmaf(xh, mul, __ldg(sh + c));
    else mul = 1.0f, t = xh;
    dyv = a.dy[yo + c];
    for (int p = 1; p < a.dy_parts; ++p) dyv += a.dy[yo + (size_t)p * a.dy_part_stride + c];
    const float da = gt ? dyv * __ldg(gt + c) : dyv;
    dt = a.gelu ? da * gelu_erf_grad(t) : da;
  };
  float s1 = 0.f, s2 = 0.f;
  for (int c = lane; c < V; c += 32) {
    float xh, dyv, t, dt, mul;
    col(c, xh, dyv, t, dt, mul);
    const float dxh = dt * mul;
    s1 += dxh, s2 += dxh * xh;
  }
  s1 = warp_sum(s1) / (float)V, s2 = warp_sum(s2) / (float)V;
  for (int c = lane; c < W; c += 32) {
    float dx = 0.f, p0 = 0.f, p1 = 0.f, p2 = 0.f;
    if (c < V) {
      float xh, dyv, t, dt, mul;
      col(c, xh, dyv, t, dt, mul);
      dx = rstd * (dt * mul - s1 - xh * s2);
      p0 = dt, p1 = dt * xh, p2 = dyv * (a.gelu ? gelu_erf(t) : t);
    }
    if (a.out_bf16) a.out_bf16[(size_t)row * a.out_ld + c] = __float2bfloat16(dx);
    if (a.prod) {
      float* pr = a.prod + (size_t)row * a.prod_ld + c;
      pr[0] = p0, pr[W] = p1, pr[2 * W] = p2;
    }
  }
}

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }

// Register-resident variant: the row (NCH float4 per lane, width = 128 * NCH) is read from global exactly once.
template <int NCH, unsigned F>
__global__ void __launch_bounds__(256) row_ln_reg_kernel(RowLnDev a) {
  pdl_launch_dependents();   // the next kernel's prologue (and its weight prefetch) may overlap this memory-bound pass
  LLB_STAMP(0x1B, a.in_parts, threadIdx.x == 0);
  constexpr bool RT = (F & F_RUNTIME) != 0;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  // Ahead of the dependency wait: the row's modulation vectors into L1.  They (and row_group) are constants of the step, written
  // by a launch that is NOT programmatic and lies before this one in the stream, so they are complete whenever this kernel runs at
  // all; the dependent round trips row_group -> vectors then overlap the tail of the GEMM this kernel waits for.
  if (!RT && (F & F_MOD) && (F & F_GATE) && row < a.rows) {
    const int g0 = a.row_group ? __ldg(a.row_group + row) : row;
    const float* m0 = a.shift + (size_t)g0 * a.mod_ld + lane * 4;
    const float* m1 = a.scale + (size_t)g0 * a.mod_ld + lane * 4;
    const float* m2 = a.gate + (size_t)g0 * a.mod_ld + lane * 4;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      asm volatile("prefetch.global.L1 [%0];" ::"l"(m0 + k * 128));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(m1 + k * 128));
      asm volatile("prefetch.global.L1 [%0];" ::"l"(m2 + k * 128));
    }
  }
  pdl_wait();
  LLB_STAMP(0x2B, a.in_parts, threadIdx.x == 0);
  if (row >= a.rows) return;
  const bool in_bf16 = RT ? a.in_bf16 != 0 : (F & F_IN_BF16) != 0;
  const bool norm = RT ? a.normalize != 0 : (F & F_NORM) != 0;
  const bool l2n = RT ? a.l2_normalize != 0 : false;
  const bool has_gamma = RT ? a.gamma != nullptr : (F & F_GAMMA) != 0;
  const bool has_mod = RT ? a.scale != nullptr : (F & F_MOD) != 0;
  const bool has_gate = RT ? a.gate != nullptr : (F & F_GATE) != 0;
  const bool has_resid = RT ? a.resid != nullptr : (F & F_RESID) != 0;
  const bool has_add = RT ? a.addvec != nullptr : (F & F_ADDVEC) != 0;
  const bool out32 = RT ? a.out_f32 != nullptr : (F & F_OUT_F32) != 0;
  const bool out16 = RT ? a.out_bf16 != nullptr : (F & F_OUT_BF16) != 0;
  const int dup = RT ? a.dup_rows : 0;
  const size_t in_off = (size_t)row * a.in_ld;
  float4 v[NCH];
#pragma unroll
  for (int k = 0; k < NCH; ++k) v[k] = load4(a.in, in_bf16, in_off + lane * 4 + k * 128);
  // split-K partial products, summed in index order
  if (NCH <= 8 && (a.in_parts == 4 || a.in_parts == 2)) {   // all loads of the slices in flight together (one exposed round trip)
    constexpr int NQ = NCH <= 8 ? NCH : 1;
    float4 q[3][NQ];
    const int extra = a.in_parts - 1;
#pragma unroll
    for (int p = 0; p < 3; ++p)
      if (p < extra) {
#pragma unroll
        for (int k = 0; k < NQ; ++k) q[p][k] = load4(a.in, in_bf16, in_off + (size_t)(p + 1) * a.in_part_stride + lane * 4 + k * 128);
      }
#pragma unroll
    for (int p = 0; p < 3; ++p)
      if (p < extra) {
#pragma unroll
        for (int k = 0; k < NQ; ++k) v[k].x += q[p][k].x, v[k].y += q[p][k].y, v[k].z += q[p][k].z, v[k].w += q[p][k].w;
      }
  } else {
    for (int p = 1; p < a.in_parts; ++p) {
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        const float4 q = load4(a.in, in_bf16, in_off + (size_t)p * a.in_part_stride + lane * 4 + k * 128);
        v[k].x += q.x, v[k].y += q.y, v[k].z += q.z, v[k].w += q.w;
      }
    }
  }
  // the residual is fetched together with the row (one exposed DRAM latency per row)
  constexpr int NRES = (NCH <= 8 && !RT && (F & F_RESID)) ? NCH : 1;
  float4 res[NRES];
  if (NRES == NCH && has_resid) {
#pragma unroll
    for (int k = 0; k < NRES; ++k) res[k] = *reinterpret_cast<const float4*>(a.resid + (size_t)row * a.resid_ld + lane * 4 + k * 128);
  }
  const int g = a.row_group ? a.row_group[row] : row;
  float mean = 0.f, rstd = 1.f;
  if (norm || l2n) {
    if (norm) {
      float s = 0.f;
#pragma unroll
      for (int k = 0; k < NCH; ++k) s += (v[k].x + v[k].y) + (v[k].z + v[k].w);
      mean = warp_sum(s) * (1.0f / (128.0f * NCH));
    }
    float q = 0.f;
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      const float d0 = v[k].x - mean, d1 = v[k].y - mean, d2 = v[k].z - mean, d3 = v[k].w - mean;
      q += (d0 * d0 + d1 * d1) + (d2 * d2 + d3 * d3);
    }
    q = warp_sum(q);
    rstd = l2n ? rsqrtf(q) : rsqrtf(q * (1.0f / (128.0f * NCH)) + 1e-5f);
  }
  const float* sh = has_mod ? a.shift + (size_t)g * a.mod_ld : nullptr;
  const float* sc = has_mod ? a.scale + (size_t)g * a.mod_ld : nullptr;
  const float* gt = has_gate ? a.gate + (size_t)g * a.mod_ld : nullptr;
  const float* av = has_add ? a.addvec + (size_t)g * a.addvec_ld : nullptr;
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    const int c = lane * 4 + k * 128;
    float x[4] = {(v[k].x - mean) * rstd, (v[k].y - mean) * rstd, (v[k].z - mean) * rstd, (v[k].w - mean) * rstd};
    if (has_gamma) {
      const float4 gm = ldg4(a.gamma + c), bt = ldg4(a.beta + c);
      x[0] = fmaf(x[0], gm.x, bt.x), x[1] = fmaf(x[1], gm.y, bt.y), x[2] = fmaf(x[2], gm.z, bt.z), x[3] = fmaf(x[3], gm.w, bt.w);
    }
    if (has_mod) {
      const float4 s4 = ldg4(sc + c), h4 = ldg4(sh + c);
      x[0] = fmaf(x[0], 1.0f + s4.x, h4.x), x[1] = fmaf(x[1], 1.0f + s4.y, h4.y);
      x[2] = fmaf(x[2], 1.0f + s4.z, h4.z), x[3] = fmaf(x[3], 1.0f + s4.w, h4.w);
    }
    if (RT) {
      if (a.act != LLB_ACT_NONE) {
#pragma unroll
        for (int i = 0; i < 4; ++i) x[i] = act_rt(x[i], a.act);
      }
    } else if (F & F_GELU) {
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = gelu_fast(x[i]);
    }
    if (has_gate) {
      const float4 g4 = ldg4(gt + c);
      x[0] *= g4.x, x[1] *= g4.y, x[2] *= g4.z, x[3] *= g4.w;
    }
    if (has_resid) {
      const float4 r4 = (NRES == NCH) ? res[NRES == NCH ? k : 0] : *reinterpret_cast<const float4*>(a.resid + (size_t)row * a.resid_ld + c);
      x[0] += r4.x, x[1] += r4.y, x[2] += r4.z, x[3] += r4.w;
    }
    if (has_add) {
      const float4 a4 = ldg4(av + c);
      x[0] += a4.x, x[1] += a4.y, x[2] += a4.z, x[3] += a4.w;
    }
    if (out32) {
      const float4 o = make_float4(x[0], x[1], x[2], x[3]);
      *reinterpret_cast<float4*>(a.out_f32 + (size_t)row * a.out_f32_ld + c) = o;
      if (dup) *reinterpret_cast<float4*>(a.out_f32 + (size_t)(row + dup) * a.out_f32_ld + c) = o;
    }
    if (out16) {
      const uint2 o = make_uint2(pack_bf16x2(x[0], x[1]), pack_bf16x2(x[2], x[3]));
      *reinterpret_cast<uint2*>(a.out_bf16 + (size_t)row * a.out_bf16_ld + c) = o;
      if (dup) *reinterpret_cast<uint2*>(a.out_bf16 + (size_t)(row + dup) * a.out_bf16_ld + c) = o;
    }
  }
}

template <unsigned F>
bool launch_reg(int nch, int grid, const RowLnDev& d, cudaStream_t stream) {
  switch (nch) {
    case 1: return launch_pdl(row_ln_reg_kernel<1, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 2: return launch_pdl(row_ln_reg_kernel<2, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 4: return launch_pdl(row_ln_reg_kernel<4, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 6: return launch_pdl(row_ln_reg_kernel<6, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 8: return launch_pdl(row_ln_reg_kernel<8, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 12: return launch_pdl(row_ln_reg_kernel<12, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 16: return launch_pdl(row_ln_reg_kernel<16, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 24: return launch_pdl(row_ln_reg_kernel<24, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
    case 32: return launch_pdl(row_ln_reg_kernel<32, F>, dim3(grid), dim3(256), 0, stream, d) == cudaSuccess;
  }
  return false;
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ src, int src_ld, __nv_bfloat16* __restrict__ dst, int dst_ld,
                                   int rows, int cols, int pad_cols) {
  const size_t total = (size_t)rows * pad_cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / pad_cols), c = (int)(i % pad_cols);
    dst[(size_t)r * dst_ld + c] = __float2bfloat16(c < cols ? src[(size_t)r * src_ld + c] : 0.0f);
  }
}

// One warp per output element (set-up only: timestep-embedding table and friends).
__global__ void __launch_bounds__(256) linear_f32_kernel(const float* __restrict__ in, int in_ld, const float* __restrict__ W,
                                                         int w_ld, const float* __restrict__ b, float* __restrict__ out,
                                                         int out_ld, int rows, int out_f, int in_f, int act) {
  const size_t widx = (size_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (widx >= (size_t)rows * out_f) return;
  const int r = (int)(widx / out_f), o = (int)(widx % out_f);
  const float* x = in + (size_t)r * in_ld;
  const float* w = W + (size_t)o * w_ld;
  float s = 0.f;
  for (int k = lane; k < in_f; k += 32) s = fmaf(x[k], w[k], s);
  s = warp_sum(s);
  if (lane == 0) {
    float y = s + (b ? b[o] : 0.0f);
    if (act == LLB_ACT_SILU) y = y / (1.0f + expf(-y));   // accurate form: this feeds the timestep table
    else y = act_rt(y, act);
    out[(size_t)r * out_ld + o] = y;
  }
}

}  // namespace

int launch_row_ln(const RowLnArgs& a, cudaStream_t stream) {
  if (a.rows <= 0) return LLB_OK;
  LLB_CHECK_ARG(a.width % 4 == 0 && a.in_ld % 4 == 0, "row_ln: width %d / ld %d must be multiples of 4", a.width, a.in_ld);
  LLB_CHECK_ARG((a.shift == nullptr) == (a.scale == nullptr), "row_ln: shift and scale come together");
  LLB_CHECK_ARG(a.in_parts >= 1 && (a.in_parts == 1 || (a.width % 128 == 0 && a.in_part_stride % 4 == 0)),
                "row_ln: summed input parts need a width that is a multiple of 128 (width %d, parts %d)", a.width, a.in_parts);
  const int valid = a.valid > 0 ? a.valid : a.width;
  LLB_CHECK_ARG(valid <= a.width && (valid == a.width || a.in_parts == 1), "row_ln: valid=%d outside [1, width=%d] or with summed parts", valid,
                a.width);
  RowLnDev d{a.in, a.in_ld, a.in_bf16 ? 1 : 0, a.rows, a.width, a.normalize ? 1 : 0, a.in_parts, a.in_part_stride, a.gamma, a.beta, a.row_group,
             a.shift, a.scale, a.gate, a.mod_ld, a.act, a.resid, a.resid_ld, a.addvec, a.addvec_ld, a.out_f32,
             a.out_f32_ld, a.out_bf16, a.out_bf16_ld, a.dup_rows, a.l2_normalize ? 1 : 0, valid};
  ProfScope prof(a.prof_slot, stream);
  const int grid = ceil_div(a.rows, 8);
  // all vector operands of the register path are read as float4
  const bool vec_ok = a.mod_ld % 4 == 0 && a.addvec_ld % 4 == 0 && a.resid_ld % 4 == 0 && a.out_f32_ld % 4 == 0 && a.out_bf16_ld % 4 == 0;
  const int nch = (a.width % 128 == 0 && vec_ok && valid == a.width) ? a.width / 128 : 0;   // padded rows: row_ln_kernel
  unsigned f = 0;
  f |= a.in_bf16 ? F_IN_BF16 : 0, f |= a.normalize ? F_NORM : 0, f |= a.gamma ? F_GAMMA : 0, f |= a.scale ? F_MOD : 0;
  f |= a.act == LLB_ACT_GELU ? F_GELU : 0, f |= a.gate ? F_GATE : 0, f |= a.resid ? F_RESID : 0, f |= a.addvec ? F_ADDVEC : 0;
  f |= a.out_f32 ? F_OUT_F32 : 0, f |= a.out_bf16 ? F_OUT_BF16 : 0;
  const bool plain = !a.l2_normalize && a.dup_rows == 0 && (a.act == LLB_ACT_NONE || a.act == LLB_ACT_GELU);
  // hot variants (compile-time masks)
  constexpr unsigned V_DIT = F_IN_BF16 | F_NORM | F_MOD | F_GATE | F_RESID | F_OUT_F32 | F_OUT_BF16;       // x += g (LN(y)(1+s)+b)
  constexpr unsigned V_MLP = F_IN_BF16 | F_NORM | F_GAMMA | F_GELU | F_OUT_BF16;                            // GELU(LN_affine(z))
  constexpr unsigned V_ENC = F_NORM | F_GAMMA | F_GELU | F_RESID | F_ADDVEC | F_OUT_F32 | F_OUT_BF16;       // GIN encoder layer tail
  constexpr unsigned V_ENC_LAST = F_NORM | F_GAMMA | F_RESID | F_OUT_F32 | F_OUT_BF16;
  constexpr unsigned V_PRED = F_NORM | F_MOD | F_GELU | F_GATE | F_RESID | F_ADDVEC | F_OUT_F32 | F_OUT_BF16;  // GIN predictor layer tail
  constexpr unsigned V_PRED_LAST = F_NORM | F_MOD | F_GATE | F_RESID | F_OUT_F32 | F_OUT_BF16;
  bool done = false;
  if (nch > 0 && plain) {
    if (f == V_DIT) done = launch_reg<V_DIT>(nch, grid, d, stream);
    else if (f == V_MLP) done = launch_reg<V_MLP>(nch, grid, d, stream);
    else if (f == V_ENC) done = launch_reg<V_ENC>(nch, grid, d, stream);
    else if (f == V_ENC_LAST) done = launch_reg<V_ENC_LAST>(nch, grid, d, stream);
    else if (f == V_PRED) done = launch_reg<V_PRED>(nch, grid, d, stream);
    else if (f == V_PRED_LAST) done = launch_reg<V_PRED_LAST>(nch, grid, d, stream);
  }
  if (!done && nch > 0) done = launch_reg<F_RUNTIME>(nch, grid, d, stream);
  if (!done) (void)launch_pdl(row_ln_kernel, dim3(grid), dim3(256), 0, stream, d);
  LLB_CUDA_OK(cudaGetLastError());
  return LLB_OK;
}

int launch_row_ln_bwd(const RowLnBwdArgs& a, cudaStream_t stream) {
  if (a.rows <= 0) return LLB_OK;
  LLB_CHECK_ARG(a.x && a.dy && a.valid >= 1 && a.valid <= a.width && a.dy_parts >= 1, "row_ln_bwd: bad argument (width %d, valid %d)",
                a.width, a.valid);
  LLB_CHECK_ARG((a.shift == nullptr) == (a.scale == nullptr) && (a.gamma == nullptr) == (a.beta == nullptr) && !(a.gamma && a.scale),
                "row_ln_bwd: gamma/beta or shift/scale, in pairs");
  ProfScope prof(a.prof_slot, stream);
  row_ln_bwd_kernel<<<ceil_div(a.rows, 8), 256, 0, stream>>>(a);
  LLB_CUDA_OK(cudaGetLastError());
  return LLB_OK;
}

int launch_f32_to_bf16(const float* src, int src_ld, __nv_bfloat16* dst, int dst_ld, int rows, int cols, int pad_cols,
                       cudaStream_t stream) {
  if (rows <= 0) return LLB_OK;
  const size_t total = (size_t)rows * pad_cols;
  const int blocks = (int)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
  f32_to_bf16_kernel<<<blocks, 256, 0, stream>>>(src, src_ld, dst, dst_ld, rows, cols, pad_cols);
  LLB_CUDA_OK(cudaGetLastError());
  return LLB_OK;
}

int launch_linear_f32(const float* in, int in_ld, const float* W, int w_ld, const float* b, float* out, int out_ld,
                      int rows, int out_f, int in_f, int act, cudaStream_t stream) {
  if (rows <= 0) return LLB_OK;
  const size_t warps = (size_t)rows * out_f;
  linear_f32_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, stream>>>(in, in_ld, W, w_ld, b, out, out_ld, rows, out_f, in_f, act);
  LLB_CUDA_OK(cudaGetLastError());
  return LLB_OK;
}

}  // namespace llb

LLB_STEP_TRACE_INSTALL(llb_trace_install_rowops)
