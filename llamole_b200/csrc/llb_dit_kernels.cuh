// Device kernels of the GraphDiT sampler that are not GEMMs: token one-hot builder, QKV epilogue (per-head
// LayerNorm), small-sequence attention on mma.sync, and the fused per-molecule step kernel
// (output-layer LN/modulate/symmetrise -> softmax -> closed-form posterior -> guidance -> categorical sample).
// The non-template kernels are static: the sampler (llb_dit.cu) and the denoiser's backward (llb_dit_grad.cu) both include this.
#pragma once
#include "llb_common.cuh"

namespace llb {

constexpr int DIT_XC = 16;  // atom classes
constexpr int DIT_EC = 5;   // bond classes
constexpr int DIT_DH = 64;  // head dim (fixed)
constexpr int DIT_MAXN = 128;        // atoms per molecule of the sampler
constexpr int DIT_GRAD_MAXN = 64;    // atoms per molecule of the denoiser's backward (llb_dit_grad.cu)

// ------------------------------------------------------------------------------------------------
// QKV GEMM epilogue: per-head affine LayerNorm on q and k (layers.py:49-50,66), softmax scale folded into q.
// ------------------------------------------------------------------------------------------------
struct EpiQKV {
  static constexpr int CHUNK = 64;
  static constexpr bool OUT_F32 = false;
  void* C;  // (M, 3H) bf16
  int ldc;
  int H;
  const float *qw, *qb, *kw, *kb;  // (64) each
  float q_scale;                   // dh^-0.5 * log2(e)
  __device__ __forceinline__ void transform(int row, int col0, float* v, int M, int N) const {
    const int which = col0 / H;  // 0 q, 1 k, 2 v
    if (which < 2) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 64; ++i) s += v[i];
      const float mean = s * (1.0f / 64.0f);
      float q = 0.f;
#pragma unroll
      for (int i = 0; i < 64; ++i) {
        const float d = v[i] - mean;
        q = fmaf(d, d, q);
      }
      const float rstd = rsqrtf(q * (1.0f / 64.0f) + 1e-5f);
      const float4* w = reinterpret_cast<const float4*>(which == 0 ? qw : kw);
      const float4* b = reinterpret_cast<const float4*>(which == 0 ? qb : kb);
      const float post = which == 0 ? q_scale : 1.0f;
#pragma unroll
      for (int i = 0; i < 16; ++i) {
        const float4 w4 = __ldg(w + i), b4 = __ldg(b + i);
        v[4 * i] = ((v[4 * i] - mean) * rstd * w4.x + b4.x) * post;
        v[4 * i + 1] = ((v[4 * i + 1] - mean) * rstd * w4.y + b4.y) * post;
        v[4 * i + 2] = ((v[4 * i + 2] - mean) * rstd * w4.z + b4.z) * post;
        v[4 * i + 3] = ((v[4 * i + 3] - mean) * rstd * w4.w + b4.w) * post;
      }
    }
  }
};

// ------------------------------------------------------------------------------------------------
// Token builder: one-hot joint rows [X_t | E_t row] for the valid tokens (transformer.py:94-95).
// tok (Mtok, K0) bf16; one warp per token.
// ------------------------------------------------------------------------------------------------
static __global__ void __launch_bounds__(256) dit_tokens_kernel(const int8_t* __restrict__ X, const int8_t* __restrict__ E,
                                                         const int32_t* __restrict__ mol_off, const int32_t* __restrict__ row_mol,
                                                         __nv_bfloat16* __restrict__ tok, int Mtok, int N, int K0) {
  const int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (r >= Mtok) return;
  const int b = row_mol[r];
  const int i = r - mol_off[b];
  const int n = mol_off[b + 1] - mol_off[b];
  const int xt = X[(size_t)b * N + i];
  const int8_t* erow = E + ((size_t)b * N + i) * N;
  __nv_bfloat16* o = tok + (size_t)r * K0;
  const __nv_bfloat16 one = __float2bfloat16(1.0f), zero = __float2bfloat16(0.0f);
  for (int k = lane; k < K0; k += 32) {
    bool hot = false;
    if (k < DIT_XC) {
      hot = (k == xt);
    } else {
      const int j = (k - DIT_XC) / DIT_EC, a = (k - DIT_XC) % DIT_EC;
      if (j < n) hot = (erow[j] == a);
    }
    o[k] = hot ? one : zero;
  }
}

// c (B+1, H) bf16 = timestep table row t + step-invariant part (cond rows) / drop vector (last row).
static __global__ void dit_cvec_kernel(const float* __restrict__ c1_t, const float* __restrict__ cinv,
                                const float* __restrict__ c_unc, __nv_bfloat16* __restrict__ cvec, int B, int H) {
  const int total = (B + 1) * H;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / H, h = i % H;
    const float v = c1_t[h] + (b < B ? cinv[(size_t)b * H + h] : c_unc[h]);
    cvec[i] = __float2bfloat16(v);
  }
}

// ------------------------------------------------------------------------------------------------
// Attention over one (sequence, head): n <= ROWS tokens, dh = 64 (layers.py:68-81; only valid tokens exist
// in the packed layout, which is output-identical to the reference's masking, SURVEY.md section 8a-6).
// ROWS / 16 warps, warp w owns query rows [16w, 16w+16).  S = Q K^T and O = P V on mma.sync.m16n8k16 (bf16, fp32 acc).
// q is pre-scaled by dh^-0.5 * log2(e) so the softmax is exp2(s - max).
// ------------------------------------------------------------------------------------------------
constexpr int ATT_LD = 72;  // padded smem row (bf16 elements): conflict-free ldmatrix

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_bf16_16816(float* c, uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

// ------------------------------------------------------------------------------------------------
// Default attention kernel: operands delivered by TMA.  (A first version staged q/k/v through registers -- 12 LDG.128 + 12
// STS.128 per thread, a third of its shared-memory wavefronts -- and ran 15.8 instead of 12.5 ms/step; removed in round 2.)
// One thread issues three 64 x 64 box loads of the qkv matrix (128-byte swizzle, so ldmatrix stays conflict-free
// without padding) and the CTA waits on one mbarrier.  Rows past the end of the sequence hold the next sequence's
// tokens (or zeros past the end of the matrix): keys >= n are masked to -inf exactly as before, so they contribute
// p = 0 times a finite value; queries >= n are never stored.
// ROWS = 64 is the kernel of every batch whose molecules have at most 64 atoms.  ROWS = 128 (a batch with a larger molecule):
// 8 warps, 128 keys, each operand two 64-row boxes stacked in a 16 KB tile (the 128-byte swizzle repeats every 8 rows, so the
// stacked boxes are one 128-row swizzled tile); the second box is loaded only for a molecule of more than 64 atoms, since rows
// >= 64 of a smaller one are never read.  Its three tiles exceed the 48 KB of static shared memory: dynamic, ATTT_SMEM128 bytes.
// ------------------------------------------------------------------------------------------------
constexpr int ATTT_TILE = 64 * DIT_DH * 2;   // one 64-row operand box (8 KB)
constexpr int ATTT_SMEM128 = 3 * 2 * ATTT_TILE + 1024;   // dynamic shared memory of the 128-row kernel (+ slack to align to 1 KB)

__device__ __forceinline__ uint32_t attt_swz(int row, int chunk) { return (uint32_t)(row * 128 + ((chunk ^ (row & 7)) << 4)); }

template <int ROWS>
static __global__ void __launch_bounds__(2 * ROWS) dit_attention_tma_kernel(const __grid_constant__ CUtensorMap tmQKV, __nv_bfloat16* __restrict__ out,
                                                                     const int32_t* __restrict__ mol_off, int B, int Mtok, int H, int heads) {
  static_assert(ROWS == 64 || ROWS == 128, "dit attention: 64- or 128-row tile");
  constexpr int TILE = ROWS * DIT_DH * 2;   // one operand tile
  constexpr int KT = ROWS / 8;              // key tiles of 8
  pdl_launch_dependents();
  LLB_STAMP(0x1A, 0, threadIdx.x == 0);
  // (the 64-row tile is static shared memory, declared ahead of the barrier as it always was)
  __shared__ __align__(1024) uint8_t tiles64[ROWS == 64 ? 3 * TILE : 1];
  __shared__ __align__(8) uint64_t bar;
  uint8_t* tiles = tiles64;
  if constexpr (ROWS == 128) {
    extern __shared__ uint8_t att_dyn_smem[];
    tiles = att_dyn_smem + ((1024u - (smem_u32(att_dyn_smem) & 1023u)) & 1023u);
  }
  const int head = blockIdx.x % heads;
  const int seq = blockIdx.x / heads;  // pass * B + molecule
  const int b = seq % B, pass = seq / B;
  // the molecule offsets are constants of the batch binding (copied in by llb_dit_begin): read, like the barrier set-up, ahead of
  // the dependency wait
  const int row0 = pass * Mtok + __ldg(mol_off + b);
  const int n = __ldg(mol_off + b + 1) - __ldg(mol_off + b);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (tid == 0) {
    tma_prefetch_desc(&tmQKV);
    mbar_init(&bar, 1);
    fence_mbar_init();
  }
  __syncthreads();
  pdl_wait();   // qkv comes from the previous kernel of the stream
  LLB_STAMP(0x2A, 0, threadIdx.x == 0);
  if (n == 0) return;
  if (tid == 0) {
    if constexpr (ROWS == 64) {
      mbar_arrive_expect_tx(&bar, 3 * ATTT_TILE);
#pragma unroll
      for (int mat = 0; mat < 3; ++mat) tma_load_2d(tiles + mat * ATTT_TILE, &tmQKV, &bar, mat * H + head * DIT_DH, row0);
    } else {
      const int boxes = n > 64 ? 2 : 1;
      mbar_arrive_expect_tx(&bar, 3 * boxes * ATTT_TILE);
      for (int mat = 0; mat < 3; ++mat)
        for (int hb = 0; hb < boxes; ++hb)
          tma_load_2d(tiles + mat * TILE + hb * ATTT_TILE, &tmQKV, &bar, mat * H + head * DIT_DH, row0 + 64 * hb);
    }
  }
  if (warp * 16 >= n) return;
  const uint32_t sQ = smem_u32(tiles), sK = sQ + TILE, sV = sK + TILE;
  const int npad = (n + 15) & ~15;
  const int ntiles = npad >> 3;  // key tiles of 8
  mbar_wait(&bar, 0);
  // ---- S = Q K^T
  float s[KT][4];
#pragma unroll
  for (int j = 0; j < KT; ++j) s[j][0] = s[j][1] = s[j][2] = s[j][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    uint32_t a0, a1, a2, a3;
    ldsm_x4(sQ + attt_swz(warp * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, ks * 2 + (lane >> 4)), a0, a1, a2, a3);
#pragma unroll
    for (int jp = 0; jp < KT / 2; ++jp) {
      if (jp * 2 < ntiles) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4(sK + attt_swz(jp * 16 + (lane & 7) + (lane >> 4) * 8, ks * 2 + ((lane >> 3) & 1)), b0, b1, b2, b3);
        mma_bf16_16816(s[2 * jp], a0, a1, a2, a3, b0, b1);
        mma_bf16_16816(s[2 * jp + 1], a0, a1, a2, a3, b2, b3);
      }
    }
  }
  // ---- softmax over keys < n (rows g and g+8 of this warp's 16)
  const int t4 = lane & 3;
  float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
  for (int j = 0; j < KT; ++j) {
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const int key = j * 8 + t4 * 2 + e;
      if (key >= n) s[j][e] = s[j][2 + e] = -INFINITY;
      m0 = fmaxf(m0, s[j][e]);
      m1 = fmaxf(m1, s[j][2 + e]);
    }
  }
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 1));
  m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 2));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 1));
  m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 2));
  float l0 = 0.f, l1 = 0.f;
  uint32_t p[KT][2];
#pragma unroll
  for (int j = 0; j < KT; ++j) {
    const float e0 = ex2_approx(s[j][0] - m0), e1 = ex2_approx(s[j][1] - m0);   // MUFU.EX2 alone: exp2f adds a range fix-up per call
    const float e2 = ex2_approx(s[j][2] - m1), e3 = ex2_approx(s[j][3] - m1);
    l0 += e0 + e1;
    l1 += e2 + e3;
    p[j][0] = pack_bf16x2(e0, e1);
    p[j][1] = pack_bf16x2(e2, e3);
  }
  l0 += __shfl_xor_sync(0xffffffffu, l0, 1);
  l0 += __shfl_xor_sync(0xffffffffu, l0, 2);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 1);
  l1 += __shfl_xor_sync(0xffffffffu, l1, 2);
  // ---- O = P V
  float o[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f;
#pragma unroll
  for (int ks = 0; ks < KT / 2; ++ks) {
    if (ks * 16 < npad) {
      const uint32_t a0 = p[2 * ks][0], a1 = p[2 * ks][1], a2 = p[2 * ks + 1][0], a3 = p[2 * ks + 1][1];
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        uint32_t b0, b1, b2, b3;
        ldsm_x4_t(sV + attt_swz(ks * 16 + (lane & 7) + ((lane >> 3) & 1) * 8, dp * 2 + (lane >> 4)), b0, b1, b2, b3);
        mma_bf16_16816(o[2 * dp], a0, a1, a2, a3, b0, b1);
        mma_bf16_16816(o[2 * dp + 1], a0, a1, a2, a3, b2, b3);
      }
    }
  }
  const float inv0 = 1.0f / l0, inv1 = 1.0f / l1;
  const int g = lane >> 2;
  // stage the warp's 16 x 64 output tile in its own (already consumed) Q rows (same swizzle), then write 16-byte
  // pieces so that 8 lanes cover one 128-byte row segment
  __syncwarp();
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(sQ + attt_swz(warp * 16 + g, j) + t4 * 4), "r"(pack_bf16x2(o[j][0] * inv0, o[j][1] * inv0)) : "memory");
    asm volatile("st.shared.b32 [%0], %1;" ::"r"(sQ + attt_swz(warp * 16 + g + 8, j) + t4 * 4), "r"(pack_bf16x2(o[j][2] * inv1, o[j][3] * inv1))
                 : "memory");
  }
  __syncwarp();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int pp = lane + 32 * i;
    const int r = pp >> 3, ch = pp & 7;
    const int grow = warp * 16 + r;
    uint4 v4;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v4.x), "=r"(v4.y), "=r"(v4.z), "=r"(v4.w) : "r"(sQ + attt_swz(grow, ch)));
    if (grow < n) *reinterpret_cast<uint4*>(out + (size_t)(row0 + grow) * H + head * DIT_DH + ch * 8) = v4;
  }
}

// ------------------------------------------------------------------------------------------------
// Attention on tcgen05 (LLB_ATTN=2, opt-in; needs an even head count).  The mma.sync kernels above re-read K and V with
// ldmatrix in every warp; here the tensor core reads its operands straight from the tiles TMA wrote:
//   unit      = (sequence, pair of heads).  Q2 / K2 / V2 are 128-row tiles: rows 0..63 head h0, rows 64..127 head h1
//               (six 64 x 64 TMA boxes of the qkv matrix, 128-byte swizzle; rows past the sequence end belong to the
//               next sequence or are zero-filled, and are masked).
//   S         = Q2 . K2^T  (M128 x N128 x K64, fp32 in TMEM): the two diagonal 64 x 64 blocks are the two heads' scores.
//   softmax   = thread r owns row r: tcgen05.ld of its block's 64 columns, exp2 (q carries dh^-0.5 log2 e), masked keys
//               contribute exactly 0.
//   P         never touches shared memory: the bf16 row of the block-diagonal P goes back into TENSOR memory, columns
//               [0,64) of the unit's 128 (32-bit column c = keys 2c, 2c+1 of the stacked 128 keys; the other head's half
//               is written as zeros).  A first design staged P in swizzled shared memory (64 KB of P tiles, 192 TMEM
//               columns per unit): two units in flight per SM, 18.8 ms/step.
//   O         = P . V2 (M128 x N64 x K128) is a tcgen05.mma with the A operand in tensor memory and V2 as an MN-major
//               shared-memory operand (exactly the [key][dh] tile TMA delivered, no transposition); it lands in columns
//               [64,128), which S no longer needs.  O / row-sum -> bf16 -> each thread stores its row's 128 bytes.
// Four units are in flight (4 x 128 columns), fed by a 4-stage ring of 48 KB TMA stages; 16 softmax / epilogue warps
// (4 per unit), one TMA warp, one MMA warp that issues S of unit k, then P V of unit k - 2.
// Measured: 15.2 ms/step (335 us per launch under ncu, 60 % DRAM, issue slots 59 % busy) against 13.2 ms for the
// TMA-fed mma.sync kernel; with molecules of 5..50 atoms the fixed 128-row unit costs more (11.4 vs 8.1 ms/step).
// ------------------------------------------------------------------------------------------------
constexpr int ATTU_TILE = 128 * 64 * 2;                       // one 128-row operand tile (16 KB)
constexpr int ATTU_STAGE_BYTES = 3 * ATTU_TILE;               // Q2 | K2 | V2
constexpr int ATT4_STAGES = 4;
constexpr int ATT4_GROUPS = 4;
constexpr int ATT4_OFF_BARS = ATT4_STAGES * ATTU_STAGE_BYTES;
constexpr int ATT4_SMEM = ATT4_OFF_BARS + 512 + 1024;
constexpr int ATT4_THREADS = (4 * ATT4_GROUPS + 2) * 32;

static __global__ void __launch_bounds__(ATT4_THREADS, 1)
dit_attention_umma4_kernel(const __grid_constant__ CUtensorMap tmQKV, __nv_bfloat16* __restrict__ out, const int32_t* __restrict__ mol_off,
                           int B, int Mtok, int H, int heads, int num_units) {
  extern __shared__ uint8_t att4_raw[];
  uint8_t* smem = att4_raw + ((1024u - (smem_u32(att4_raw) & 1023u)) & 1023u);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ATT4_OFF_BARS);
  uint64_t* full = bars;                        // [STAGES] TMA -> MMA
  uint64_t* empty = full + ATT4_STAGES;         // [STAGES] P V done -> TMA
  uint64_t* s_full = empty + ATT4_STAGES;       // [GROUPS] S in TMEM
  uint64_t* p_full = s_full + ATT4_GROUPS;      // [GROUPS] P in TMEM (and S consumed)
  uint64_t* o_full = p_full + ATT4_GROUPS;      // [GROUPS] O in TMEM
  uint64_t* o_empty = o_full + ATT4_GROUPS;     // [GROUPS] O consumed: the unit's 128 columns are free
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_empty + ATT4_GROUPS);
  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int hpairs = heads >> 1;
  constexpr int W_TMA = 4 * ATT4_GROUPS, W_MMA = W_TMA + 1;

  if (warp == W_TMA && elect_one()) {
    tma_prefetch_desc(&tmQKV);
    for (int i = 0; i < ATT4_STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int g = 0; g < ATT4_GROUPS; ++g) {
      mbar_init(&s_full[g], 1);
      mbar_init(&p_full[g], 4);
      mbar_init(&o_full[g], 1);
      mbar_init(&o_empty[g], 4);
    }
    fence_mbar_init();
  }
  if (warp == W_MMA) tmem_alloc(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == W_TMA) {
    // ---------------- TMA producer ----------------
    int st = 0;
    uint32_t ph = 0;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      const int seq = u / hpairs, hp = u % hpairs;
      const int b = seq % B, pass = seq / B;
      const int n = mol_off[b + 1] - mol_off[b];
      if (n == 0) continue;
      const int row0 = pass * Mtok + mol_off[b];
      mbar_wait(&empty[st], ph ^ 1);
      if (elect_one()) {
        uint8_t* base = smem + st * ATTU_STAGE_BYTES;
        mbar_arrive_expect_tx(&full[st], ATTU_STAGE_BYTES);
#pragma unroll
        for (int mat = 0; mat < 3; ++mat)
#pragma unroll
          for (int hl = 0; hl < 2; ++hl)
            tma_load_2d(base + mat * ATTU_TILE + hl * (ATTU_TILE / 2), &tmQKV, &full[st], mat * H + (2 * hp + hl) * DIT_DH, row0);
      }
      __syncwarp();
      if (++st == ATT4_STAGES) {
        st = 0;
        ph ^= 1;
      }
    }
  } else if (warp == W_MMA) {
    // ---------------- MMA issuer ----------------
    constexpr uint32_t idesc_s = umma_idesc_bf16(128, 128);
    constexpr uint32_t idesc_o = umma_idesc_bf16(128, 64) | (1u << 16);   // B (= V2) is MN-major
    auto issue_pv = [&](int j) {   // unit j of this CTA: group j & 3, stage j & 3, use number j >> 2 of both
      const int g = j & 3, st = j & 3;
      mbar_wait(&p_full[g], (uint32_t)((j >> 2) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint32_t t_p = tmem_base + g * 128, t_o = t_p + 64;
        const uint64_t v_desc = umma_desc_k128(smem_u32(smem + st * ATTU_STAGE_BYTES + 2 * ATTU_TILE));
#pragma unroll
        for (int kk = 0; kk < 8; ++kk)   // 16 keys per step: 8 columns of P; V2 16 rows = 2 KB further down
          umma_bf16_ts(t_o, t_p + kk * 8, v_desc + (uint64_t)(kk * 128), idesc_o, kk != 0 ? 1u : 0u);
        umma_commit(&o_full[g]);
        umma_commit(&empty[st]);
      }
      __syncwarp();
    };
    int k = 0;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      const int seq = u / hpairs;
      const int b = seq % B;
      if (mol_off[b + 1] - mol_off[b] == 0) continue;
      const int g = k & 3, st = k & 3;
      const uint32_t use = (uint32_t)((k >> 2) & 1);
      const uint64_t q_desc = umma_desc_k128(smem_u32(smem + st * ATTU_STAGE_BYTES));
      const uint64_t k_desc = q_desc + (ATTU_TILE >> 4);
      mbar_wait(&full[st], use);
      mbar_wait(&o_empty[g], use ^ 1);   // the previous unit of this group has read its O: the 128 columns are free
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int kq = 0; kq < 4; ++kq) umma_bf16(tmem_base + g * 128, q_desc + 2 * kq, k_desc + 2 * kq, idesc_s, kq != 0 ? 1u : 0u);
        umma_commit(&s_full[g]);
      }
      __syncwarp();
      if (k >= 2) issue_pv(k - 2);
      ++k;
    }
    if (k >= 2) issue_pv(k - 2);
    if (k >= 1) issue_pv(k - 1);
  } else {
    // ---------------- softmax + epilogue: group = warp / 4, thread = row of the stacked 128-row tile ----------------
    const int grp = warp >> 2, wq = warp & 3;
    const int r = wq * 32 + lane;            // TMEM lane
    const int hl = wq >> 1;                  // head of the pair (warp-uniform)
    const uint32_t t_grp = tmem_base + ((uint32_t)(wq * 32) << 16) + grp * 128;
    const uint32_t t_s = t_grp + hl * 64;
    const uint32_t t_o = t_grp + 64;
    int k = 0;
    uint32_t up = 0;
    for (int u = blockIdx.x; u < num_units; u += gridDim.x) {
      const int seq = u / hpairs, hp = u % hpairs;
      const int b = seq % B, pass = seq / B;
      const int n = mol_off[b + 1] - mol_off[b];
      if (n == 0) continue;
      if (((k++) & 3) != grp) continue;      // another group's unit
      const int row0 = pass * Mtok + mol_off[b];
      mbar_wait(&s_full[grp], up);
      tc_fence_after();
      float sc[64];
      tmem_ld32(t_s, sc);
      tmem_ld32(t_s + 32, sc + 32);
      tmem_ld_wait();
      float m = -INFINITY;
#pragma unroll
      for (int j = 0; j < 64; ++j) m = fmaxf(m, j < n ? sc[j] : -INFINITY);
      float l = 0.f;
      const uint32_t zeros[16] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int c = 0; c < 2; ++c) {          // 32 keys -> 16 packed columns per store
        uint32_t pk[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const int j = c * 32 + 2 * i;
          const float e0 = j < n ? ex2_approx(sc[j] - m) : 0.f;
          const float e1 = j + 1 < n ? ex2_approx(sc[j + 1] - m) : 0.f;
          l += e0 + e1;
          pk[i] = pack_bf16x2(e0, e1);
        }
        tmem_st16(t_grp + hl * 32 + c * 16, pk);
        tmem_st16(t_grp + (1 - hl) * 32 + c * 16, zeros);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[grp]);
      const float inv = 1.0f / l;
      mbar_wait(&o_full[grp], up);
      tc_fence_after();
      tmem_ld32(t_o, sc);
      tmem_ld32(t_o + 32, sc + 32);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&o_empty[grp]);
      const int q_idx = r & 63;
      if (q_idx < n) {
        uint4* dst = reinterpret_cast<uint4*>(out + (size_t)(row0 + q_idx) * H + (2 * hp + hl) * DIT_DH);
#pragma unroll
        for (int c = 0; c < 8; ++c)
          dst[c] = make_uint4(pack_bf16x2(sc[c * 8] * inv, sc[c * 8 + 1] * inv), pack_bf16x2(sc[c * 8 + 2] * inv, sc[c * 8 + 3] * inv),
                              pack_bf16x2(sc[c * 8 + 4] * inv, sc[c * 8 + 5] * inv), pack_bf16x2(sc[c * 8 + 6] * inv, sc[c * 8 + 7] * inv));
      }
      up ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------
// Fused per-molecule step kernel.
// ------------------------------------------------------------------------------------------------
struct DitTablesDev {
  float x_marg[DIT_XC];
  float e_marg[DIT_EC];
  float xe[DIT_XC][DIT_EC];
  float ex[DIT_EC][DIT_XC];
};

struct DitStepArgs {
  // logits source A: raw output-layer rows (M, raw_ld) fp32 + modulation (B+1, 2*d0) fp32
  const float* raw;
  int raw_ld;
  const float* modout;
  // logits source B: dense masked logits in the reference layout (parity entry)
  const float *lcX, *lcE, *luX, *luE;
  const int32_t* mol_off;
  int B, N, Mtok, passes;
  // state (in place)
  int8_t* X;
  int8_t* E;
  // schedule scalars for this step
  float beta_t, abar_s, abar_t, guide_scale;
  // noise
  const float* qX;  // (B,N,16) or null
  const float* qE;  // (B,N,N,5) or null
  uint64_t seed;
  uint32_t stream_id;  // counter-RNG stream (= s, the index of the state being produced)
  int64_t mol_base;
  // outputs
  int sample;        // 1: write the new state
  float* dumpX;      // optional (B,N,16): logits of pass `dump_pass` (sample==0) or guided probs (sample==1)
  float* dumpE;      // optional (B,N,N,5)
  int dump_pass;
  int dump_logits;
  // T_GLOBAL step kernel only: T's rows in global memory, row (pass p, atom i of molecule b) at (p Mtok + mol_off[b] + i) tg_ld
  float* tg;
  int tg_ld;
};

// Per-node statistics of one pass kept in shared memory.
struct NodeStats {
  float pX[DIT_XC];   // softmax of the atom logits
  float S[DIT_EC];    // sum_j softmax(E logits)[i,j,:] over all N slots (masked / diagonal slots give 0.2)
  float A[DIT_EC];    // sum_c pX[c] * xe[c,:]
};

__device__ __forceinline__ void softmax5(const float* l, float* p) {
  const float m = fmaxf(fmaxf(fmaxf(l[0], l[1]), fmaxf(l[2], l[3])), l[4]);
  float e[5], s = 0.f;
#pragma unroll
  for (int a = 0; a < 5; ++a) {
    e[a] = __expf(l[a] - m);
    s += e[a];
  }
  const float inv = 1.0f / s;
#pragma unroll
  for (int a = 0; a < 5; ++a) p[a] = e[a] * inv;
}

// Closed form of reverse_diffusion with Q = a I + (1-a) U (SURVEY.md section 8a-5; diffusion_utils.py:476-492):
//   out[k] = ((1-beta) v[k] + beta UX[k]) * (abar_s p[k] + (1-abar_s) PU[k]) / max(abar_t v[k] + (1-abar_t) UX[k], 1e-5)
__device__ __forceinline__ float post_term(float v, float ux, float p, float pu, float beta, float abar_s, float abar_t) {
  const float left = (1.0f - beta) * v + beta * ux;
  const float right = abar_s * p + (1.0f - abar_s) * pu;
  const float den = fmaxf(abar_t * v + (1.0f - abar_t) * ux, 1e-5f);
  return left * right / den;
}

// Dynamic shared memory: T[pass][n][d0] logits rows (fp32), then NodeStats[pass][n], then small arrays.
// T_GLOBAL (T does not fit a block's shared memory: 2 N d0 4 bytes is 186 KB at N = 64, 701 KB at N = 128): T lives in
// global memory at a.tg and shared memory starts at NodeStats.  A template parameter rather than a pointer chosen at run time,
// so that the shared-memory instantiations keep shared-memory (not generic) loads and stores.
// THREADS = 256 (two CTAs per SM at throughput batch sizes) or 512 (a handful of molecules: one CTA per molecule is all the
// parallelism there is, so each gets more threads); every loop strides by blockDim.x.
template <int THREADS, bool T_GLOBAL = false>
static __global__ void __launch_bounds__(THREADS) dit_step_kernel(DitStepArgs a, const __grid_constant__ DitTablesDev tb) {
  LLB_STAMP(0x1C, 0, threadIdx.x == 0);
  extern __shared__ __align__(16) float sm[];
  const int b = blockIdx.x;
  const int N = a.N, d0 = DIT_XC + DIT_EC * N;
  const int off = a.mol_off[b];
  const int n = a.mol_off[b + 1] - off;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nthreads = blockDim.x;
  int8_t* Xg = a.X + (size_t)b * N;
  int8_t* Eg = a.E + (size_t)b * N * N;

  float* T = sm;                                                       // passes * N * d0
  const int ld = T_GLOBAL ? a.tg_ld : d0;                              // row stride of T
  auto tpass = [&](int p) -> float* {                                  // row 0 of pass p
    return T_GLOBAL ? a.tg + ((size_t)p * a.Mtok + off) * ld : T + (size_t)p * N * d0;
  };
  auto trow = [&](int p, int i) -> float* {                            // row i of pass p
    return T_GLOBAL ? a.tg + ((size_t)p * a.Mtok + off + i) * ld : T + ((size_t)p * N + i) * d0;
  };
  NodeStats* stats = reinterpret_cast<NodeStats*>(T_GLOBAL ? sm : T + (size_t)a.passes * N * d0);   // passes * N
  float* cnt = reinterpret_cast<float*>(stats + a.passes * N);         // N * 5
  int8_t* sX = reinterpret_cast<int8_t*>(cnt + N * DIT_EC);            // N
  int8_t* sE = sX + ((N + 15) & ~15);                                  // N * N

  if (n == 0) {
    if (a.sample) {
      for (int i = tid; i < N; i += nthreads) Xg[i] = -1;
      for (int i = tid; i < N * N; i += nthreads) Eg[i] = -1;
    }
    return;
  }
  for (int i = tid; i < N; i += nthreads) sX[i] = Xg[i];
  for (int i = tid; i < N * N; i += nthreads) sE[i] = Eg[i];
  __syncthreads();

  // ---------------- logits into T ----------------
  if (a.raw != nullptr) {
    // output layer tail (transformer.py:166-187): LN(d0) -> modulate -> + one-hot input -> zero diag/masked -> symmetrise
    for (int p = 0; p < a.passes; ++p) {
      const float* shift = a.modout + (size_t)(p == 0 ? b : a.B) * (2 * d0);
      const float* scale = shift + d0;
      for (int i = warp; i < n; i += nthreads / 32) {
        const float* src = a.raw + (size_t)(p * a.Mtok + off + i) * a.raw_ld;
        float* dst = trow(p, i);   // with T_GLOBAL: src itself
        float s = 0.f;
        for (int k = lane; k < d0; k += 32) {
          const float v = src[k];
          if constexpr (!T_GLOBAL) dst[k] = v;
          s += v;
        }
        const float mean = warp_sum(s) / (float)d0;
        float q = 0.f;
        for (int k = lane; k < d0; k += 32) {
          const float d = dst[k] - mean;
          q = fmaf(d, d, q);
        }
        const float rstd = rsqrtf(warp_sum(q) / (float)d0 + 1e-5f);
        for (int k = lane; k < d0; k += 32) dst[k] = (dst[k] - mean) * rstd * (1.0f + scale[k]) + shift[k];
      }
    }
    __syncthreads();
    // atoms: + one-hot; bonds: symmetrise valid off-diagonal pairs, zero the rest
    for (int p = 0; p < a.passes; ++p) {
      float* Tp = tpass(p);
      for (int idx = tid; idx < n * DIT_XC; idx += nthreads) {
        const int i = idx / DIT_XC, c = idx % DIT_XC;
        Tp[i * ld + c] += (sX[i] == c) ? 1.0f : 0.0f;
      }
      for (int idx = tid; idx < n * N; idx += nthreads) {
        const int i = idx / N, j = idx % N;
        float* tij = Tp + i * ld + DIT_XC + DIT_EC * j;
        if (j >= n || j == i) {
#pragma unroll
          for (int e = 0; e < DIT_EC; ++e) tij[e] = 0.f;
        } else if (i < j) {
          float* tji = Tp + j * ld + DIT_XC + DIT_EC * i;
          const int et = sE[i * N + j];
#pragma unroll
          for (int e = 0; e < DIT_EC; ++e) {
            const float m = 0.5f * ((tij[e] + (et == e ? 1.0f : 0.0f)) + (tji[e] + (et == e ? 1.0f : 0.0f)));
            tij[e] = m;
            tji[e] = m;
          }
        }
      }
    }
    __syncthreads();
  } else {
    for (int p = 0; p < a.passes; ++p) {
      const float* lX = (p == 0 ? a.lcX : a.luX) + (size_t)b * N * DIT_XC;
      const float* lE = (p == 0 ? a.lcE : a.luE) + (size_t)b * N * N * DIT_EC;
      float* Tp = tpass(p);
      for (int idx = tid; idx < n * d0; idx += nthreads) {
        const int i = idx / d0, k = idx % d0;
        Tp[i * ld + k] = k < DIT_XC ? lX[i * DIT_XC + k] : lE[(size_t)i * N * DIT_EC + (k - DIT_XC)];
      }
    }
    __syncthreads();
  }

  if (a.dump_logits) {
    // masked logits in the reference's dense layout (zeros outside the valid block)
    const float* Tp = tpass(a.dump_pass);
    float* oX = a.dumpX + (size_t)b * N * DIT_XC;
    float* oE = a.dumpE + (size_t)b * N * N * DIT_EC;
    for (int idx = tid; idx < N * DIT_XC; idx += nthreads) {
      const int i = idx / DIT_XC;
      oX[idx] = i < n ? Tp[i * ld + idx % DIT_XC] : 0.f;
    }
    for (int idx = tid; idx < N * N * DIT_EC; idx += nthreads) {
      const int i = idx / (N * DIT_EC), k = idx % (N * DIT_EC);
      oE[idx] = (i < n && k / DIT_EC < n) ? Tp[i * ld + DIT_XC + k] : 0.f;
    }
    if (!a.sample) return;
  }

  // ---------------- per-node statistics ----------------
  // cnt_i[e] = number of slots j with E_t[i,j] == e (masked slots and the z_T diagonal hold no class)
  for (int idx = tid; idx < n * DIT_EC; idx += nthreads) {
    const int i = idx / DIT_EC, e = idx % DIT_EC;
    int c = 0;
    for (int j = 0; j < n; ++j) c += (sE[i * N + j] == e);
    cnt[idx] = (float)c;
  }
  for (int idx = warp; idx < a.passes * n; idx += nthreads / 32) {
    const int p = idx / n, i = idx % n;
    const float* ti = trow(p, i);
    NodeStats& st = stats[p * N + i];
    // atom softmax (16 logits: lanes 0..15)
    float l = lane < DIT_XC ? ti[lane] : -INFINITY;
    const float m = warp_max(l);
    const float e = lane < DIT_XC ? __expf(l - m) : 0.f;
    const float sum = warp_sum(e);
    const float px = e / sum;
    if (lane < DIT_XC) st.pX[lane] = px;
    // S over all N slots: valid off-diagonal slots from the logits, the others contribute 0.2 each
    float Sa[DIT_EC] = {0.f, 0.f, 0.f, 0.f, 0.f};
    for (int j = lane; j < n; j += 32) {
      if (j != i) {
        float pe[DIT_EC];
        softmax5(ti + DIT_XC + DIT_EC * j, pe);
#pragma unroll
        for (int q = 0; q < DIT_EC; ++q) Sa[q] += pe[q];
      }
    }
    const float rest = 0.2f * (float)(N - n + 1);
#pragma unroll
    for (int q = 0; q < DIT_EC; ++q) {
      const float v = warp_sum(Sa[q]) + rest;
      if (lane == 0) st.S[q] = v;
    }
#pragma unroll
    for (int q = 0; q < DIT_EC; ++q) {
      const float v = warp_sum(lane < DIT_XC ? px * tb.xe[lane][q] : 0.f);
      if (lane == 0) st.A[q] = v;
    }
  }
  __syncthreads();

  const float beta = a.beta_t, as_ = a.abar_s, at_ = a.abar_t, gs = a.guide_scale;
  const uint2 key = make_uint2((uint32_t)(a.seed & 0xffffffffu), (uint32_t)(a.seed >> 32));
  const uint32_t molid = (uint32_t)(a.mol_base + b);

  // ---------------- atoms ----------------
  for (int i = tid; i < n; i += nthreads) {
    const int xt = sX[i];
    float prob[DIT_XC];
    for (int p = 0; p < a.passes; ++p) {
      const NodeStats& st = stats[p * N + i];
      float un[DIT_XC], sum = 0.f;
      float sumpx = 0.f;
#pragma unroll
      for (int c = 0; c < DIT_XC; ++c) sumpx += st.pX[c];
#pragma unroll
      for (int c = 0; c < DIT_XC; ++c) {
        float ux = tb.x_marg[xt];
        float pu = sumpx * tb.x_marg[c];
#pragma unroll
        for (int e = 0; e < DIT_EC; ++e) {
          ux = fmaf(cnt[i * DIT_EC + e], tb.xe[c][e], ux);
          pu = fmaf(st.S[e], tb.ex[e][c], pu);
        }
        un[c] = post_term(xt == c ? 1.0f : 0.0f, ux, st.pX[c], pu, beta, as_, at_);
        sum += un[c];
      }
      if (sum == 0.f) {
#pragma unroll
        for (int c = 0; c < DIT_XC; ++c) un[c] = 1e-5f;
        sum = 1e-5f * DIT_XC;
      }
      if (p == 0) {
#pragma unroll
        for (int c = 0; c < DIT_XC; ++c) prob[c] = un[c] / sum;
      } else {
        float gsum = 0.f;
#pragma unroll
        for (int c = 0; c < DIT_XC; ++c) {
          const float pu_ = un[c] / sum;
          prob[c] = pu_ * powf(prob[c] / fmaxf(pu_, 1e-5f), gs);
          gsum += prob[c];
        }
        gsum = fmaxf(gsum, 1e-5f);
#pragma unroll
        for (int c = 0; c < DIT_XC; ++c) prob[c] /= gsum;
      }
    }
    if (a.dumpX && !a.dump_logits) {
#pragma unroll
      for (int c = 0; c < DIT_XC; ++c) a.dumpX[((size_t)b * N + i) * DIT_XC + c] = prob[c];
    }
    if (a.sample) {
      float q[DIT_XC];
      if (a.qX) {
#pragma unroll
        for (int c = 0; c < DIT_XC; ++c) q[c] = a.qX[((size_t)b * N + i) * DIT_XC + c];
      } else {
#pragma unroll
        for (int g = 0; g < DIT_XC / 4; ++g) {
          const uint4 r = philox4x32_10(make_uint4((uint32_t)i, molid, a.stream_id, (uint32_t)g), key);
          q[4 * g] = exp1_from_bits(r.x), q[4 * g + 1] = exp1_from_bits(r.y);
          q[4 * g + 2] = exp1_from_bits(r.z), q[4 * g + 3] = exp1_from_bits(r.w);
        }
      }
      // clamp_min(1e-5) -> (renormalisation does not move the argmax) -> argmax(p / q)  (diffusion_utils.py:392-395)
      int best = 0;
      float bv = -1.f;
#pragma unroll
      for (int c = 0; c < DIT_XC; ++c) {
        const float v = fmaxf(prob[c], 1e-5f) / q[c];
        if (v > bv) bv = v, best = c;
      }
      Xg[i] = (int8_t)best;
    }
  }
  if (a.sample) {
    for (int i = n + tid; i < N; i += nthreads) Xg[i] = -1;
  }

  // ---------------- bonds: pairs i < j of valid nodes (the reference keeps triu(1) and mirrors it) ----------------
  const int npairs = n * (n - 1) / 2;
  for (int pidx = tid; pidx < npairs; pidx += nthreads) {
    // unrank pidx -> (i, j), i < j
    int i = (int)((2.0f * n - 1.0f - sqrtf((2.0f * n - 1.0f) * (2.0f * n - 1.0f) - 8.0f * (float)pidx)) * 0.5f);
    while (i > 0 && (i * (2 * n - i - 1)) / 2 > pidx) --i;
    while (((i + 1) * (2 * n - i - 2)) / 2 <= pidx) ++i;
    const int j = pidx - (i * (2 * n - i - 1)) / 2 + i + 1;
    const int et = sE[i * N + j];
    const int xt = sX[i];
    float cm = 0.f;
#pragma unroll
    for (int e = 0; e < DIT_EC; ++e) cm = fmaf(cnt[i * DIT_EC + e], tb.e_marg[e], cm);
    float prob[DIT_EC];
    for (int p = 0; p < a.passes; ++p) {
      const NodeStats& st = stats[p * N + i];
      float pe[DIT_EC];
      softmax5(trow(p, i) + DIT_XC + DIT_EC * j, pe);
      const float Ssum = (st.S[0] + st.S[1]) + (st.S[2] + st.S[3]) + st.S[4];
      float un[DIT_EC], sum = 0.f;
#pragma unroll
      for (int e = 0; e < DIT_EC; ++e) {
        const float ux = tb.ex[e][xt] + cm;
        const float pu = st.A[e] + Ssum * tb.e_marg[e];
        un[e] = post_term(et == e ? 1.0f : 0.0f, ux, pe[e], pu, beta, as_, at_);
        sum += un[e];
      }
      if (sum == 0.f) {
#pragma unroll
        for (int e = 0; e < DIT_EC; ++e) un[e] = 1e-5f;
        sum = 1e-5f * DIT_EC;
      }
      if (p == 0) {
#pragma unroll
        for (int e = 0; e < DIT_EC; ++e) prob[e] = un[e] / sum;
      } else {
        float gsum = 0.f;
#pragma unroll
        for (int e = 0; e < DIT_EC; ++e) {
          const float pu_ = un[e] / sum;
          prob[e] = pu_ * powf(prob[e] / fmaxf(pu_, 1e-5f), gs);
          gsum += prob[e];
        }
        gsum = fmaxf(gsum, 1e-5f);
#pragma unroll
        for (int e = 0; e < DIT_EC; ++e) prob[e] /= gsum;
      }
    }
    if (a.dumpE && !a.dump_logits) {
#pragma unroll
      for (int e = 0; e < DIT_EC; ++e) a.dumpE[(((size_t)b * N + i) * N + j) * DIT_EC + e] = prob[e];
    }
    if (a.sample) {
      float q[8];
      if (a.qE) {
#pragma unroll
        for (int e = 0; e < DIT_EC; ++e) q[e] = a.qE[(((size_t)b * N + i) * N + j) * DIT_EC + e];
      } else {
        const uint32_t pos = (uint32_t)(N + i * N + j);
        const uint4 r0 = philox4x32_10(make_uint4(pos, molid, a.stream_id, 0u), key);
        const uint4 r1 = philox4x32_10(make_uint4(pos, molid, a.stream_id, 1u), key);
        q[0] = exp1_from_bits(r0.x), q[1] = exp1_from_bits(r0.y), q[2] = exp1_from_bits(r0.z), q[3] = exp1_from_bits(r0.w);
        q[4] = exp1_from_bits(r1.x);
      }
      int best = 0;
      float bv = -1.f;
#pragma unroll
      for (int e = 0; e < DIT_EC; ++e) {
        const float v = fmaxf(prob[e], 1e-5f) / q[e];
        if (v > bv) bv = v, best = e;
      }
      Eg[i * N + j] = (int8_t)best;
      Eg[j * N + i] = (int8_t)best;
    }
  }
  if (a.sample) {
    // diagonal of valid nodes: class 0 (triu(1)+transpose leaves 0 there); everything touching a masked node: none
    for (int idx = tid; idx < N * N; idx += nthreads) {
      const int i = idx / N, j = idx % N;
      if (i >= n || j >= n) Eg[idx] = -1;
      else if (i == j) Eg[idx] = 0;
    }
  }
}

// z_T from the limit marginals (diffusion_utils.py:495-518): argmax(marg / q); strict upper triangle mirrored,
// diagonal and masked entries hold no class (-1).
static __global__ void __launch_bounds__(256) dit_init_state_kernel(int8_t* __restrict__ X, int8_t* __restrict__ E,
                                                             const int32_t* __restrict__ mol_off, int N, const float* __restrict__ qX0,
                                                             const float* __restrict__ qE0, uint64_t seed, uint32_t stream_id,
                                                             int64_t mol_base, const __grid_constant__ DitTablesDev tb) {
  const int b = blockIdx.x;
  const int n = mol_off[b + 1] - mol_off[b];
  const uint2 key = make_uint2((uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32));
  const uint32_t molid = (uint32_t)(mol_base + b);
  for (int i = threadIdx.x; i < N; i += blockDim.x) {
    int best = -1;
    if (i < n) {
      float bv = -1.f;
      for (int g = 0; g < DIT_XC / 4; ++g) {
        float q[4];
        if (qX0) {
          for (int e = 0; e < 4; ++e) q[e] = qX0[((size_t)b * N + i) * DIT_XC + 4 * g + e];
        } else {
          const uint4 r = philox4x32_10(make_uint4((uint32_t)i, molid, stream_id, (uint32_t)g), key);
          q[0] = exp1_from_bits(r.x), q[1] = exp1_from_bits(r.y), q[2] = exp1_from_bits(r.z), q[3] = exp1_from_bits(r.w);
        }
        for (int e = 0; e < 4; ++e) {
          const float v = tb.x_marg[4 * g + e] / q[e];
          if (v > bv) bv = v, best = 4 * g + e;
        }
      }
    }
    X[(size_t)b * N + i] = (int8_t)best;
  }
  for (int idx = threadIdx.x; idx < N * N; idx += blockDim.x) {
    const int i = idx / N, j = idx % N;
    if (i >= n || j >= n || i == j) {
      E[(size_t)b * N * N + idx] = -1;
    } else if (i < j) {
      float q[8];
      if (qE0) {
        for (int e = 0; e < DIT_EC; ++e) q[e] = qE0[(((size_t)b * N + i) * N + j) * DIT_EC + e];
      } else {
        const uint32_t pos = (uint32_t)(N + i * N + j);
        const uint4 r0 = philox4x32_10(make_uint4(pos, molid, stream_id, 0u), key);
        const uint4 r1 = philox4x32_10(make_uint4(pos, molid, stream_id, 1u), key);
        q[0] = exp1_from_bits(r0.x), q[1] = exp1_from_bits(r0.y), q[2] = exp1_from_bits(r0.z), q[3] = exp1_from_bits(r0.w);
        q[4] = exp1_from_bits(r1.x);
      }
      int best = 0;
      float bv = -1.f;
      for (int e = 0; e < DIT_EC; ++e) {
        const float v = tb.e_marg[e] / q[e];
        if (v > bv) bv = v, best = e;
      }
      E[(size_t)b * N * N + i * N + j] = (int8_t)best;
      E[(size_t)b * N * N + j * N + i] = (int8_t)best;
    }
  }
}

}  // namespace llb
