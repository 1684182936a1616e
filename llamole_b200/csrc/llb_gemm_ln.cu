// CTA-pair GEMMs with a LayerNorm tail fused into the epilogue: GraphDiT block tails (N = 1024) and GIN layer tails (N = 768 / 1024); see llb_gemm_ln.cuh.
#include <stdlib.h>

#include <atomic>

#include "llb_gemm_ln.cuh"

namespace llb {

namespace {

#ifdef LLB_GEMM_TRACE
__device__ long long* g_gln_trace = nullptr;   // [tile][16] stamps of CTA 0 (tools/gemm_ln_trace.cu)
__device__ int g_gln_exp = 0;                  // knock-outs: 1 no x store, 2 no xb store, 4 no residual reload, 8 no pass 2, 16 empty epilogue (pair kernel)
#define GLN_TRACE(tile_idx, slot, value) \
  do { if (g_gln_trace && blockIdx.x == 0 && (tile_idx) < 64) g_gln_trace[(size_t)(tile_idx) * 16 + (slot)] = (value); } while (0)
#define GLN_EXP(bit) ((g_gln_exp & (bit)) != 0)
#else
#define GLN_EXP(bit) false
#define GLN_TRACE(tile_idx, slot, value) do { } while (0)
#endif

__device__ __forceinline__ uint32_t cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(32 * GEMM_EPI_WARPS) : "memory"); }

struct GlnPass2 {
  uint32_t t_row;        // TMEM address of this warp's first column
  uint32_t xstg, xbstg;  // shared addresses of the warp's fp32 / bf16 staging tiles
  uint32_t bias_s;       // shared address of bias[cbase]
  uint32_t mod_s;        // shared address of the row's staged modulation (STAGED only), at column cbase
  const float* g_shift;  // global modulation rows of this thread's group, at column n0 + cbase (slow path)
  const float* g_scale;
  const float* g_gate;
  const float* xrow;     // e.x + (first coalesced row) * ldx + n0 + cbase + 4 * slot
  size_t xstride;        // 4 rows further down
  int rows_left;         // valid rows from this lane's first coalesced row (row 4 it is valid iff 4 it < rows_left)
  int gcol, grow;        // global column / row of the warp's 32 x 128 block (TMA store coordinates)
  float rstd, nmr;
  int trace_tile;        // debug builds only
};

// Pass 2 with the residual travelling through TMA in BOTH directions (CTA-pair kernel): the residual box of a chunk is
// TMA-loaded into the warp's swizzled staging tile, each thread (= TMEM lane = row) adds its 32 normalised, modulated
// values to its own row IN PLACE and packs the bf16 copy, and the same tile is TMA-stored back.  No transposition, no
// generic global access (generic loads from 8 warps crawl once shared memory has taken the whole L1), 20 instead of 40
// shared-memory instructions per chunk.  With NXB = 2 staging tiles the next chunk's load is issued a chunk ahead;
// with NXB = 1 (long K, where the epilogue has slack) load and store of consecutive chunks serialise.
template <bool STAGED, int NXB>
__device__ __forceinline__ void gln_pass2_tma(const GlnPass2& a, const CUtensorMap* tmX, const CUtensorMap* tmXb, uint64_t* res_full,
                                              uint32_t& res_phase, int lane) {
  float v[32];
#ifdef LLB_GEMM_TRACE
  long long tt0 = 0, tt1 = 0, tt2 = 0, tt3 = 0;
#endif
#pragma unroll 1
  for (int ci = 0; ci < GLN_BN / 2 / 32; ++ci) {
    const int c = ci * 32;
    const int b = NXB == 2 ? (ci & 1) : 0;
#ifdef LLB_GEMM_TRACE
    const long long k0 = clock64();
#endif
    tmem_ld32(a.t_row + c, v);
    tmem_ld_wait();
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      const float4 bb = lds128(a.bias_s + (c + 4 * p) * 4);
      float4 s1, sh;
      if (STAGED) {
        s1 = lds128(a.mod_s + (c + 4 * p) * 4);
        sh = lds128(a.mod_s + (GLN_BN + c + 4 * p) * 4);
      } else {
        const float4 gt = __ldg(reinterpret_cast<const float4*>(a.g_gate + c + 4 * p));
        s1 = __ldg(reinterpret_cast<const float4*>(a.g_scale + c + 4 * p));
        sh = __ldg(reinterpret_cast<const float4*>(a.g_shift + c + 4 * p));
        s1.x = (1.0f + s1.x) * gt.x, s1.y = (1.0f + s1.y) * gt.y, s1.z = (1.0f + s1.z) * gt.z, s1.w = (1.0f + s1.w) * gt.w;
        sh.x *= gt.x, sh.y *= gt.y, sh.z *= gt.z, sh.w *= gt.w;
      }
      v[4 * p] = fmaf(fmaf(v[4 * p] + bb.x, a.rstd, a.nmr), s1.x, sh.x);
      v[4 * p + 1] = fmaf(fmaf(v[4 * p + 1] + bb.y, a.rstd, a.nmr), s1.y, sh.y);
      v[4 * p + 2] = fmaf(fmaf(v[4 * p + 2] + bb.z, a.rstd, a.nmr), s1.z, sh.z);
      v[4 * p + 3] = fmaf(fmaf(v[4 * p + 3] + bb.w, a.rstd, a.nmr), s1.w, sh.w);
    }
#ifdef LLB_GEMM_TRACE
    const long long k1 = clock64();
#endif
    // the previous chunk's stores have read their staging tiles: the bf16 tile and the other fp32 tile are free
    if (elect_one()) {
      bulk_wait_read<0>();
      if (NXB == 2 && ci + 1 < GLN_BN / 2 / 32) {
        mbar_arrive_expect_tx(&res_full[b ^ 1], 4096);
        tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(a.xstg + (b ^ 1) * 4096)), tmX, &res_full[b ^ 1], a.gcol + c + 32, a.grow);
      }
    }
    __syncwarp();
#ifdef LLB_GEMM_TRACE
    const long long k2 = clock64();
#endif
    mbar_wait(&res_full[b], (res_phase >> b) & 1u);
    res_phase ^= 1u << b;
#ifdef LLB_GEMM_TRACE
    const long long k3 = clock64();
#endif
    const uint32_t xs = a.xstg + b * 4096 + lane * 128;
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      const uint32_t addr = xs + ((p ^ (lane & 7)) << 4);
      const float4 r = lds128(addr);
      v[4 * p] += r.x, v[4 * p + 1] += r.y, v[4 * p + 2] += r.z, v[4 * p + 3] += r.w;
      sts128(addr, make_float4(v[4 * p], v[4 * p + 1], v[4 * p + 2], v[4 * p + 3]));
    }
    const uint32_t xbs = a.xbstg + lane * 64;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float4 q;
      q.x = __uint_as_float(pack_bf16x2(v[8 * j], v[8 * j + 1])), q.y = __uint_as_float(pack_bf16x2(v[8 * j + 2], v[8 * j + 3]));
      q.z = __uint_as_float(pack_bf16x2(v[8 * j + 4], v[8 * j + 5])), q.w = __uint_as_float(pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
      sts128(xbs + ((j ^ ((lane >> 1) & 3)) << 4), q);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (elect_one()) {
      if (!GLN_EXP(1)) tma_store_2d(tmX, reinterpret_cast<const void*>(__cvta_shared_to_generic(a.xstg + b * 4096)), a.gcol + c, a.grow);
      if (!GLN_EXP(2)) tma_store_2d(tmXb, reinterpret_cast<const void*>(__cvta_shared_to_generic(a.xbstg)), a.gcol + c, a.grow);
      bulk_commit();
      if (NXB == 1 && ci + 1 < GLN_BN / 2 / 32) {   // single tile: reload it as soon as the store has read it
        bulk_wait_read<0>();
        mbar_arrive_expect_tx(&res_full[0], 4096);
        tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(a.xstg)), tmX, &res_full[0], a.gcol + c + 32, a.grow);
      }
    }
#ifdef LLB_GEMM_TRACE
    const long long k4 = clock64();
    tt0 += k1 - k0, tt1 += k2 - k1, tt2 += k3 - k2, tt3 += k4 - k3;
#endif
  }
#ifdef LLB_GEMM_TRACE
  if (a.trace_tile >= 0) {
    GLN_TRACE(a.trace_tile, 11, tt0);   // tmem + math
    GLN_TRACE(a.trace_tile, 12, tt1);   // wait for the previous stores' smem reads
    GLN_TRACE(a.trace_tile, 13, tt2);   // wait for the residual load
    GLN_TRACE(a.trace_tile, 14, tt3);   // add, pack, fence, store issue
  }
#endif
}

// Pass 2 of the GIN layer tail (GinTailArgs): same data path as gln_pass2_tma -- the residual chunk arrives by TMA in the warp's
// staging tile, thread = row adds its 32 values in place, the tile goes back by TMA -- with the GIN arithmetic in between.  The
// per-graph vectors (text-adaLN shift / scale / gate, next virtual node) are read straight from global memory: the 32 rows of a
// warp belong to a handful of graphs, so these are mostly same-address loads, and with K = 4 H the epilogue has ~12k cycles.
struct GinRow {
  const float* sc;   // scale row of this thread's graph at the warp's first column (null: affine gamma / beta from shared memory)
  const float* sh;
  const float* gt;   // gate row or null
  const float* av;   // addvec row or null
  uint32_t gamma_s, beta_s;   // shared addresses at the warp's first column
  int group;         // graph of this thread's row
  int nvalid;        // rows of this warp's 32 that exist (row < M): 0..32, warp-uniform
  uint32_t heads;    // bit r: row r of the warp starts a new graph (bit 0 unused), warp-uniform
};
template <int NXB>
__device__ __forceinline__ void gin_pass2_tma(const GlnPass2& a, const GinRow& gr, const GinTailArgs& t, const CUtensorMap* tmX,
                                              const CUtensorMap* tmXb, uint64_t* res_full, uint32_t& res_phase, int lane) {
  float v[32];
#pragma unroll 1
  for (int ci = 0; ci < GLN_BN / 2 / 32; ++ci) {
    const int c = ci * 32;
    const int b = NXB == 2 ? (ci & 1) : 0;
    tmem_ld32(a.t_row + c, v);
    tmem_ld_wait();
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      const float4 bb = lds128(a.bias_s + (c + 4 * p) * 4);
      float4 s1, sh;
      if (gr.sc != nullptr) {
        s1 = __ldg(reinterpret_cast<const float4*>(gr.sc + c + 4 * p));
        sh = __ldg(reinterpret_cast<const float4*>(gr.sh + c + 4 * p));
        s1.x += 1.0f, s1.y += 1.0f, s1.z += 1.0f, s1.w += 1.0f;
      } else {
        s1 = lds128(gr.gamma_s + (c + 4 * p) * 4);
        sh = lds128(gr.beta_s + (c + 4 * p) * 4);
      }
      float x0 = fmaf(fmaf(v[4 * p] + bb.x, a.rstd, a.nmr), s1.x, sh.x);
      float x1 = fmaf(fmaf(v[4 * p + 1] + bb.y, a.rstd, a.nmr), s1.y, sh.y);
      float x2 = fmaf(fmaf(v[4 * p + 2] + bb.z, a.rstd, a.nmr), s1.z, sh.z);
      float x3 = fmaf(fmaf(v[4 * p + 3] + bb.w, a.rstd, a.nmr), s1.w, sh.w);
      if (t.act == LLB_ACT_GELU) x0 = gelu_fast(x0), x1 = gelu_fast(x1), x2 = gelu_fast(x2), x3 = gelu_fast(x3);
      if (gr.gt != nullptr) {
        const float4 g4 = __ldg(reinterpret_cast<const float4*>(gr.gt + c + 4 * p));
        x0 *= g4.x, x1 *= g4.y, x2 *= g4.z, x3 *= g4.w;
      }
      if (gr.av != nullptr) {
        const float4 a4 = __ldg(reinterpret_cast<const float4*>(gr.av + c + 4 * p));
        x0 += a4.x, x1 += a4.y, x2 += a4.z, x3 += a4.w;
      }
      v[4 * p] = x0, v[4 * p + 1] = x1, v[4 * p + 2] = x2, v[4 * p + 3] = x3;
    }
    // the previous chunk's stores have read their staging tiles: the bf16 tile and the other fp32 tile are free
    if (elect_one()) {
      bulk_wait_read<0>();
      if (NXB == 2 && ci + 1 < GLN_BN / 2 / 32) {
        mbar_arrive_expect_tx(&res_full[b ^ 1], 4096);
        tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(a.xstg + (b ^ 1) * 4096)), tmX, &res_full[b ^ 1], a.gcol + c + 32, a.grow);
      }
    }
    __syncwarp();
    mbar_wait(&res_full[b], (res_phase >> b) & 1u);
    res_phase ^= 1u << b;
    const uint32_t xs = a.xstg + b * 4096 + lane * 128;
#pragma unroll
    for (int p = 0; p < 8; ++p) {
      const uint32_t addr = xs + ((p ^ (lane & 7)) << 4);
      const float4 r = lds128(addr);
      v[4 * p] += r.x, v[4 * p + 1] += r.y, v[4 * p + 2] += r.z, v[4 * p + 3] += r.w;
      sts128(addr, make_float4(v[4 * p], v[4 * p + 1], v[4 * p + 2], v[4 * p + 3]));
    }
    const uint32_t xbs = a.xbstg + lane * 64;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float4 q;
      q.x = __uint_as_float(pack_bf16x2(v[8 * j], v[8 * j + 1])), q.y = __uint_as_float(pack_bf16x2(v[8 * j + 2], v[8 * j + 3]));
      q.z = __uint_as_float(pack_bf16x2(v[8 * j + 4], v[8 * j + 5])), q.w = __uint_as_float(pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
      sts128(xbs + ((j ^ ((lane >> 1) & 3)) << 4), q);
    }
    fence_proxy_async_smem();
    __syncwarp();
    if (elect_one()) {
      tma_store_2d(tmX, reinterpret_cast<const void*>(__cvta_shared_to_generic(a.xstg + b * 4096)), a.gcol + c, a.grow);
      tma_store_2d(tmXb, reinterpret_cast<const void*>(__cvta_shared_to_generic(a.xbstg)), a.gcol + c, a.grow);
      bulk_commit();
    }
    if (t.pool_max != nullptr && gr.nvalid > 0) {
      // per-graph column maxima of the new rows: lane = column of the chunk, reading the warp's 32 rows back from the staging
      // tile (the swizzle spreads a row's 32 columns over the 32 banks: conflict-free).  The rows' graph boundaries are a
      // tile-constant bit mask, so the scan is 32 independent loads and a chain of uniform selects; every run of equal graph ids
      // ends in ONE 128-byte atomicMax (order-independent, hence deterministic).
      const uint32_t xt = a.xstg + b * 4096;
      const int cq = lane >> 2, cw = lane & 3;
      float vals[32];
#pragma unroll
      for (int r = 0; r < 32; ++r)
        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(vals[r]) : "r"(xt + r * 128 + ((cq ^ (r & 7)) << 4) + cw * 4));
      uint32_t* pcol = t.pool_max + a.gcol + c + lane;
      float run = vals[0];
#pragma unroll
      for (int r = 1; r < 32; ++r) {
        if (r < gr.nvalid) {                 // warp-uniform
          if ((gr.heads >> r) & 1u) {        // warp-uniform: row r starts a new graph -> flush the finished one
            atomicMax(pcol + (size_t)__shfl_sync(0xffffffffu, gr.group, r - 1) * t.pool_ld, float_order_enc(__float_as_uint(run)));
            run = vals[r];
          } else {
            run = fmaxf(run, vals[r]);
          }
        }
      }
      atomicMax(pcol + (size_t)__shfl_sync(0xffffffffu, gr.group, gr.nvalid - 1) * t.pool_ld, float_order_enc(__float_as_uint(run)));
      __syncwarp();
    }
    if (NXB == 1 && ci + 1 < GLN_BN / 2 / 32) {   // single tile: reload it as soon as the store has read it
      if (elect_one()) {
        bulk_wait_read<0>();
        mbar_arrive_expect_tx(&res_full[0], 4096);
        tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(a.xstg)), tmX, &res_full[0], a.gcol + c + 32, a.grow);
      }
      __syncwarp();
    }
  }
}

// Modulation stager, one warp, one tile: which modulation rows do the tile's 128 token rows use (runs of equal
// row_group), stage gate*(1+scale) and gate*shift of those rows (this CTA's 256 columns) in shared memory, and pull the
// CTA's block of the residual stream into L2 for the epilogue's pass 2.
__device__ __forceinline__ void gln_stage_tile(const GemmLnArgs& e, const CUtensorMap* tmXpf, float* mod_dst, int2* rowinfo, int* glist,
                                               int m0, int n0, int M, int lane) {
  constexpr int BN = GLN_BN;
  int cnt = 0;
#pragma unroll
  for (int seg = 0; seg < 4; ++seg) {
    const int r = m0 + seg * 32 + lane;
    const int rc = r < M ? r : M - 1;
    const int g = __ldg(e.row_group + rc);
    const int gp = (rc > m0) ? __ldg(e.row_group + rc - 1) : g;
    const int flag = (r < M && g != gp) ? 1 : 0;
    const uint32_t mask = __ballot_sync(0xffffffffu, flag);
    const int gi = cnt + __popc(mask & (0xffffffffu >> (31 - lane)));
    cnt += __popc(mask);
    rowinfo[seg * 32 + lane] = make_int2(gi, g);
    if ((flag || (seg == 0 && lane == 0)) && gi < GLN_MAX_GROUPS) glist[gi] = g;
  }
  const int ngroups = cnt + 1;
  if (lane == 0) {
    glist[4] = ngroups;
    if (m0 < M && tmXpf != nullptr && !GLN_EXP(32)) l2_prefetch_tile(tmXpf, n0, m0);   // this CTA's 128 x 256 block of the residual stream
  }
  __syncwarp();
  if (ngroups <= GLN_MAX_GROUPS) {
    // mod_dst[k][0][col] = gate * (1 + scale), [k][1][col] = gate * shift; each lane owns 8 columns per group
    float4 sh[GLN_MAX_GROUPS][2], sc[GLN_MAX_GROUPS][2], gt[GLN_MAX_GROUPS][2];
#pragma unroll
    for (int k = 0; k < GLN_MAX_GROUPS; ++k) {
      if (k < ngroups) {
        const size_t off = (size_t)glist[k] * e.mod_ld + n0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int col = h * 128 + lane * 4;
          sh[k][h] = __ldg(reinterpret_cast<const float4*>(e.shift + off + col));
          sc[k][h] = __ldg(reinterpret_cast<const float4*>(e.scale + off + col));
          gt[k][h] = __ldg(reinterpret_cast<const float4*>(e.gate + off + col));
        }
      }
    }
#pragma unroll
    for (int k = 0; k < GLN_MAX_GROUPS; ++k) {
      if (k < ngroups) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int col = h * 128 + lane * 4;
          const float4 g4 = gt[k][h], s4 = sc[k][h], h4 = sh[k][h];
          *reinterpret_cast<float4*>(mod_dst + (k * 2 + 0) * BN + col) =
              make_float4((1.0f + s4.x) * g4.x, (1.0f + s4.y) * g4.y, (1.0f + s4.z) * g4.z, (1.0f + s4.w) * g4.w);
          *reinterpret_cast<float4*>(mod_dst + (k * 2 + 1) * BN + col) = make_float4(h4.x * g4.x, h4.y * g4.y, h4.z * g4.z, h4.w * g4.w);
        }
      }
    }
  }
  __syncwarp();
}

// Pass 1 of the epilogue: sum and sum of squares of (accumulator + bias) over this warp's 128 columns of its row.
__device__ __forceinline__ float2 gln_pass1(uint32_t t_row, uint32_t bias_s) {
  float v[32];
  float s = 0.f, ss = 0.f;
#pragma unroll 1
  for (int c = 0; c < GLN_BN / 2; c += 32) {
    tmem_ld32(t_row + c, v);
    tmem_ld_wait();
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      const float4 b = lds128(bias_s + (c + i) * 4);
      const float a0 = v[i] + b.x, a1 = v[i + 1] + b.y, a2 = v[i + 2] + b.z, a3 = v[i + 3] + b.w;
      s += (a0 + a1) + (a2 + a3);
      ss = fmaf(a0, a0, ss), ss = fmaf(a1, a1, ss), ss = fmaf(a2, a2, ss), ss = fmaf(a3, a3, ss);
    }
  }
  return make_float2(s, ss);
}

// ------------------------------------------------------------------------------------------------------------------
// N = 1024 variant on the CTA-pair (cta_group::2) main loop.
//
// The cluster kernel above cannot use tcgen05.mma.cta_group::2: a pair splits the M dimension, so one pair owns a
// 256-row x 256-column block, a full 1024-column row then spans four pairs = a cluster of 8, and only 15 such clusters
// fit the B200 (120 of 148 SMs).  Here FOUR INDEPENDENT PAIRS (four 2-CTA clusters, 72 of 74 pairs in use) form a
// group that owns one 256-row block; CTA (slice s, rank r) holds rows [128 r, +128) x columns [256 s, +256).  The row
// statistics are exchanged between the four CTAs of equal rank through global memory (L2): every statistics warp
// writes its 32 rows, releases a per-(group, rank) counter (fence + atomic add) and every epilogue warp polls the
// counter with acquire loads.  The ~2.5k cycles of round trips sit inside the epilogue, which the second TMEM
// accumulator stage overlaps with the next tile's MMAs.  All CTAs of the persistent grid must be co-resident (the grid
// is launched cooperatively, never larger than the device holds).
// ------------------------------------------------------------------------------------------------------------------
// (STAGES, MODST, NXB): (4, 1, 2) for short K -- the epilogue is the long pole, so every warp gets two fp32 staging tiles and
// loads the next chunk's residual a chunk ahead; (5, 1, 1) for long K -- the main loop is, and one more 32 KB ring stage
// rides out the DRAM latency jitter the epilogue's own traffic causes.
template <int STAGES_, int MODST_, int NXB_>
struct GlnPairSmemT {
  static constexpr int STAGES = STAGES_;
  static constexpr int MODST = MODST_;
  static constexpr int NXB = NXB_;   // fp32 staging tiles per epilogue warp
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;            // 16 KB: this CTA's 128 rows
  static constexpr int B_BYTES = (GLN_BN / 2) * GEMM_BK * 2;       // 16 KB: this CTA's half of the pair's 256 W rows
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int XSTG_PER_WARP = NXB * 32 * 32 * 4;
  static constexpr int XBSTG_PER_WARP = 32 * 32 * 2;
  static constexpr int MOD_STAGE_FLOATS = GLN_MAX_GROUPS * 2 * GLN_BN;
  static constexpr int OFF_XSTG = STAGES * STAGE_BYTES;
  static constexpr int OFF_XBSTG = OFF_XSTG + GEMM_EPI_WARPS * XSTG_PER_WARP;
  static constexpr int OFF_MOD = OFF_XBSTG + GEMM_EPI_WARPS * XBSTG_PER_WARP;
  static constexpr int OFF_BIAS = OFF_MOD + MODST * MOD_STAGE_FLOATS * 4;
  static constexpr int OFF_PART = OFF_BIAS + GLN_BN * 4;
  static constexpr int OFF_ROWINFO = OFF_PART + 2 * GEMM_BM * 8;
  static constexpr int OFF_GLIST = OFF_ROWINFO + MODST * GEMM_BM * 8;
  static constexpr int OFF_BARS = OFF_GLIST + 64;
  static constexpr int TOTAL = OFF_BARS + 512 + 1024;
};
static_assert(GlnPairSmemT<4, 1, 2>::TOTAL <= 232448 && GlnPairSmemT<5, 1, 1>::TOTAL <= 232448,
              "gemm_ln pair kernel shared memory exceeds the 227 KB per-CTA limit");

// Statistics mailbox entry: {sum, tag, sum of squares, tag}.  Data and flag travel in the same 8-byte halves (each
// half is an atomic access), so the exchange needs no fence, no atomic and no counter: a reader simply re-reads until both
// tags carry the value expected for this launch and tile.
__device__ __forceinline__ void st_mailbox(uint4* p, float s, float ss, uint32_t tag) {
  asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(__float_as_uint(s)), "r"(tag), "r"(__float_as_uint(ss)), "r"(tag)
               : "memory");
}
__device__ __forceinline__ uint4 ld_mailbox(const uint4* p) {
  uint4 v;
  asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
  return v;
}

// Epilogue payload of the pair kernel: the GraphDiT block tail (GemmLnArgs) or the GIN layer tail (GinTailArgs).
template <bool GIN>
struct PairTail {
  using type = GemmLnArgs;
};
template <>
struct PairTail<true> {
  using type = GinTailArgs;
};

template <int STAGES_, int MODST_, int NXB_, int NS, bool GIN>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_ln_pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmBh,
                    const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmXb,
                    const __grid_constant__ CUtensorMap tmXpf, int M, int K, int G, typename PairTail<GIN>::type e, uint4* sync_stats,
                    uint32_t tag_base, int prefetch_x) {
  using S = GlnPairSmemT<STAGES_, MODST_, NXB_>;
  constexpr int STAGES = S::STAGES;
  constexpr int MODST = S::MODST;
  constexpr int NXB = S::NXB;
  constexpr int BN = GLN_BN;
  // NS column slices of 256 = pairs per group
  const uint32_t rank = cluster_rank();
  const int pair = blockIdx.x >> 1;
  const int grp = pair / NS, slice = pair % NS;
  if (grp >= G) return;   // spare pair(s): both CTAs leave together, nothing was set up yet

  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* smA = smem;
  uint8_t* smB = smem + STAGES * S::A_BYTES;
  float* modS = reinterpret_cast<float*>(smem + S::OFF_MOD);
  float* biasS = reinterpret_cast<float*>(smem + S::OFF_BIAS);
  float2* partS = reinterpret_cast<float2*>(smem + S::OFF_PART);
  int2* rowinfoS = reinterpret_cast<int2*>(smem + S::OFF_ROWINFO);
  int* glistS = reinterpret_cast<int*>(smem + S::OFF_GLIST);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + S::OFF_BARS);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;
  uint64_t* mod_full = bars + 2 * STAGES + 4;
  uint64_t* mod_empty = bars + 2 * STAGES + 6;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 8);
  uint64_t* res_full = bars + 2 * STAGES + 10;   // [epilogue warp][2]: residual chunk landed in the warp's staging tile

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int num_mb = (M + 2 * GEMM_BM - 1) / (2 * GEMM_BM);
  const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;
  const int n0 = slice * BN;

  if (warp == GEMM_EPI_WARPS && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmBh);
    tma_prefetch_desc(&tmX);
    tma_prefetch_desc(&tmXb);
    tma_prefetch_desc(&tmXpf);
    for (int st = 0; st < STAGES; ++st) {
      mbar_init(&full[st], 1);
      mbar_init(&empty[st], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 2 * GEMM_EPI_WARPS);
    }
    for (int a = 0; a < MODST; ++a) {
      mbar_init(&mod_full[a], 1);
      mbar_init(&mod_empty[a], GEMM_EPI_WARPS);
    }
    for (int a = 0; a < 2 * GEMM_EPI_WARPS; ++a) mbar_init(&res_full[a], 1);
    fence_mbar_init();
  }
  if (threadIdx.x < BN) {
    biasS[threadIdx.x] = e.bias ? e.bias[n0 + threadIdx.x] : 0.0f;
    if constexpr (GIN) {   // affine LayerNorm weight / bias of this CTA's columns live where the DiT variant stages its modulations
      modS[threadIdx.x] = e.gamma ? e.gamma[n0 + threadIdx.x] : 1.0f;
      modS[BN + threadIdx.x] = e.beta ? e.beta[n0 + threadIdx.x] : 0.0f;
    }
  }
  cluster_sync_all();
  if (warp == GEMM_EPI_WARPS + 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)(2 * BN))
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == GEMM_EPI_WARPS) {
    // ---------------- TMA producer (both CTAs; completion bytes go to the leader's full[]) ----------------
    int stage = 0;
    uint32_t phase = 0;
    const int nB = n0 + (int)rank * (BN / 2);
    for (int mb = grp; mb < num_mb; mb += G) {
      const int m0 = mb * 2 * GEMM_BM + (int)rank * GEMM_BM;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * S::STAGE_BYTES);
          tma_load_2d_2sm(smA + stage * S::A_BYTES, &tmA, &full[stage], kb * GEMM_BK, m0);
          tma_load_2d_2sm(smB + stage * S::B_BYTES, &tmBh, &full[stage], kb * GEMM_BK, nB);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == GEMM_EPI_WARPS + 1) {
    // ---------------- MMA issuer (leader CTA only; converged warp, one elected lane issues) ----------------
    if (rank == 0) {
      const uint32_t idesc = umma_idesc_ab(2 * GEMM_BM, BN, GIN && (prefetch_x & 2) != 0);   // GIN tail: bit 1 = fp16 operands
      const uint64_t a_desc0 = umma_desc_k128(smem_u32(smA));
      const uint64_t b_desc0 = umma_desc_k128(smem_u32(smB));
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int tcount = 0;
      for (int mb = grp; mb < num_mb; mb += G, ++tcount) {
        if (lane == 0) GLN_TRACE(tcount, 8, clock64());
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        if (lane == 0) GLN_TRACE(tcount, 9, clock64());
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a_desc = a_desc0 + (uint64_t)(stage * (S::A_BYTES >> 4));
            const uint64_t b_desc = b_desc0 + (uint64_t)(stage * (S::B_BYTES >> 4));
#pragma unroll
            for (int k = 0; k < GEMM_BK / 16; ++k) umma_bf16_2sm(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_commit_2sm(&empty[stage]);
          }
          __syncwarp();
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (elect_one()) umma_commit_2sm(&tmem_full[acc]);
        __syncwarp();
        if (lane == 0) GLN_TRACE(tcount, 10, clock64());
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp == GEMM_EPI_WARPS + 3) {
    // ---------------- modulation stager (GraphDiT tail only) ----------------
    if constexpr (!GIN) {
      int st = 0;
      uint32_t ph = 0;
      for (int mb = grp; mb < num_mb; mb += G) {
        const int m0 = mb * 2 * GEMM_BM + (int)rank * GEMM_BM;
        mbar_wait(&mod_empty[st], ph ^ 1);
        gln_stage_tile(e, prefetch_x ? &tmXpf : nullptr, modS + (size_t)st * S::MOD_STAGE_FLOATS, rowinfoS + st * GEMM_BM, glistS + st * 8, m0, n0, M,
                       lane);
        if (lane == 0) mbar_arrive(&mod_full[st]);
        if (++st == MODST) {
          st = 0;
          ph ^= 1;
        }
      }
    }
  } else if (warp < GEMM_EPI_WARPS) {
    // ---------------- epilogue ----------------
    const int q = warp & 3, ch = warp >> 2;
    const int rloc = q * 32 + lane;
    const int cbase = ch * (BN / 2);
    const float inv_n = 1.0f / (float)(NS * BN);
    GlnPass2 a;
    a.xstg = smem_u32(smem + S::OFF_XSTG + warp * S::XSTG_PER_WARP);
    a.xbstg = smem_u32(smem + S::OFF_XBSTG + warp * S::XBSTG_PER_WARP);
    a.bias_s = smem_u32(biasS + cbase);
    a.gcol = n0 + cbase;
    int acc = 0;
    uint32_t acc_phase = 0;
    int ms = 0;           // modulation stage / phase (MODST stages)
    uint32_t mph = 0;
    uint32_t res_phase = 0;   // bit b: phase of this warp's res_full[b]
    int tcount = 0;
    const bool tr = warp == 0 && lane == 0;
    for (int mb = grp; mb < num_mb; mb += G, ++tcount) {
      const int m0 = mb * 2 * GEMM_BM + (int)rank * GEMM_BM;
      if (tr) GLN_TRACE(tcount, 0, clock64());
      if constexpr (GIN) {   // pull the NEXT tile's block of the node features into L2 while this tile is being finished
        const int m0n = m0 + G * 2 * GEMM_BM;
        if ((prefetch_x & 1) && warp == 0 && lane == 0 && m0n < M) l2_prefetch_tile(&tmXpf, n0, m0n);
      }
      // the tile's first residual chunk starts its way into the staging tile now (the previous tile's stores have read it)
      a.grow = m0 + q * 32;
      if (elect_one()) {
        bulk_wait_read<0>();
        mbar_arrive_expect_tx(&res_full[warp * 2], 4096);
        tma_load_2d(reinterpret_cast<void*>(__cvta_shared_to_generic(a.xstg)), &tmX, &res_full[warp * 2], a.gcol, a.grow);
      }
      __syncwarp();
      if (tr) GLN_TRACE(tcount, 1, clock64());
      mbar_wait(&tmem_full[acc], acc_phase);
      if (tr) GLN_TRACE(tcount, 2, clock64());
      tc_fence_after();
      a.t_row = tmem_base + acc * BN + ((uint32_t)(q * 32) << 16) + cbase;
      if (!GIN && GLN_EXP(16)) {   // knock-out: empty epilogue (main loop alone)
        mbar_wait(&res_full[warp * 2], res_phase & 1u);
        res_phase ^= 1u;
        mbar_wait(&mod_full[ms], mph);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_cluster(&tmem_empty[acc], 0);
          mbar_arrive(&mod_empty[ms]);
        }
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
        if (++ms == MODST) {
          ms = 0;
          mph ^= 1;
        }
        continue;
      }
      partS[ch * GEMM_BM + rloc] = gln_pass1(a.t_row, a.bias_s);
      epi_bar_sync();
      // statistics mailboxes: [group][tile parity][rank][slice][128 rows]
      uint4* gstats = sync_stats + (size_t)((grp * 2 + (tcount & 1)) * 2 + rank) * NS * GEMM_BM;
      const uint32_t tag = tag_base + (uint32_t)(tcount + 1);
      if (ch == 0) {
        const float2 p0 = partS[rloc], p1 = partS[GEMM_BM + rloc];
        st_mailbox(gstats + slice * GEMM_BM + rloc, p0.x + p1.x, p0.y + p1.y, tag);
      }
      if (tr) GLN_TRACE(tcount, 3, clock64());
      // poll this row's four mailboxes (one per column slice) until all carry this tile's tag
      {
        // the partial sums are kept per source and added in slice order once all four are in: adding them in ARRIVAL
        // order made the fp32 row statistics -- and through them a few sampled categories per step -- vary from run to run
        float sv[NS], ssv[NS];
        uint32_t pending = (1u << NS) - 1u;
        const long long start = clock64();
        while (pending) {
#pragma unroll
          for (int src = 0; src < NS; ++src) {
            if (pending & (1u << src)) {
              const uint4 v = ld_mailbox(gstats + src * GEMM_BM + rloc);
              if (v.y == tag && v.w == tag) {
                sv[src] = __uint_as_float(v.x), ssv[src] = __uint_as_float(v.z);
                pending &= ~(1u << src);
              }
            }
          }
          if (pending && clock64() - start > 8000000000ll) {
            printf("llamole_b200: statistics exchange timed out (block %d thread %d)\n", blockIdx.x, threadIdx.x);
            __trap();
          }
        }
        if (tr) GLN_TRACE(tcount, 4, clock64());
        float s = 0.f, ss = 0.f;
#pragma unroll
        for (int src = 0; src < NS; ++src) s += sv[src], ss += ssv[src];
        const float mean = s * inv_n;
        const float var = fmaxf(ss * inv_n - mean * mean, 0.0f);
        a.rstd = rsqrtf(var + 1e-5f);
        a.nmr = -mean * a.rstd;
      }
      a.trace_tile = tr ? tcount : -1;
      if constexpr (GIN) {
        const int row = m0 + rloc;
        GinRow gr;
        gr.group = __ldg(e.row_group + (row < M ? row : M - 1));
        gr.nvalid = M - (m0 + q * 32) < 32 ? (M - (m0 + q * 32) > 0 ? M - (m0 + q * 32) : 0) : 32;
        {
          const int gup = __shfl_up_sync(0xffffffffu, gr.group, 1);
          gr.heads = __ballot_sync(0xffffffffu, lane > 0 && gr.group != gup);
        }
        const size_t moff = (size_t)gr.group * e.mod_ld + n0 + cbase;
        gr.sc = e.scale ? e.scale + moff : nullptr;
        gr.sh = e.shift ? e.shift + moff : nullptr;
        gr.gt = e.gate ? e.gate + moff : nullptr;
        gr.av = e.addvec ? e.addvec + (size_t)gr.group * e.addvec_ld + n0 + cbase : nullptr;
        gr.gamma_s = smem_u32(modS + cbase), gr.beta_s = smem_u32(modS + BN + cbase);
        gin_pass2_tma<NXB>(a, gr, e, &tmX, &tmXb, &res_full[warp * 2], res_phase, lane);
      } else {
        // the tile's modulation rows are staged (the stager had pass 1 and the exchange to do it)
        mbar_wait(&mod_full[ms], mph);
        const int2 info = rowinfoS[ms * GEMM_BM + rloc];
        const bool staged = glistS[ms * 8 + 4] <= GLN_MAX_GROUPS;
        if (GLN_EXP(8)) {
          mbar_wait(&res_full[warp * 2], res_phase & 1u);
          res_phase ^= 1u;
        } else if (staged) {
          a.mod_s = smem_u32(modS + (size_t)ms * S::MOD_STAGE_FLOATS + (size_t)info.x * 2 * BN + cbase);
          gln_pass2_tma<true, NXB>(a, &tmX, &tmXb, &res_full[warp * 2], res_phase, lane);
        } else {
          const size_t off = (size_t)info.y * e.mod_ld + n0 + cbase;
          a.g_shift = e.shift + off, a.g_scale = e.scale + off, a.g_gate = e.gate + off;
          gln_pass2_tma<false, NXB>(a, &tmX, &tmXb, &res_full[warp * 2], res_phase, lane);
        }
      }
      if (tr) GLN_TRACE(tcount, 5, clock64());
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_cluster(&tmem_empty[acc], 0);
        if (!GIN) mbar_arrive(&mod_empty[ms]);
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
      if (++ms == MODST) {
        ms = 0;
        mph ^= 1;
      }
    }
    if (lane == 0) bulk_wait_all();
  }
  tc_fence_before();
  cluster_sync_all();
  if (warp == GEMM_EPI_WARPS + 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * BN)) : "memory");
  }
}

}  // namespace

bool gemm_ln_enabled() {
  static int mode = -1;
  if (mode < 0) {
    const char* v = getenv("LLB_FUSED_LN");
    mode = (v && v[0] == '0') ? 0 : 1;
  }
  return mode != 0;
}

size_t gemm_ln_pair_workspace_bytes() {
  // statistics mailboxes: [group][2 tile parities][2 ranks][4 slices][128 rows] x 16 bytes
  return (size_t)GLN_PAIR_MAX_GROUPS * 2 * 2 * 4 * GEMM_BM * sizeof(uint4);
}

int launch_gemm_ln_pair(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const GemmLnArgs& e, void* sync_ws,
                        size_t sync_bytes, cudaStream_t stream, LaunchCounter* ctr) {
  if (M <= 0) return LLB_OK;
  LLB_CHECK_ARG(N == 4 * GLN_BN && K % 8 == 0, "gemm_ln_pair: N=%d must be 1024 and K=%d a multiple of 8", N, K);
  LLB_CHECK_ARG(lda % 8 == 0 && ldw % 8 == 0 && e.ldx % 4 == 0 && e.ldxb % 8 == 0 && e.mod_ld % 4 == 0,
                "gemm_ln_pair: leading dimensions must keep rows 16-byte aligned");
  LLB_CHECK_ARG(e.row_group && e.shift && e.scale && e.gate && e.x && e.xb, "gemm_ln_pair: null operand");
  LLB_CHECK_ARG(sync_ws && sync_bytes >= gemm_ln_pair_workspace_bytes() && (reinterpret_cast<uintptr_t>(sync_ws) & 127) == 0,
                "gemm_ln_pair: the exchange workspace needs %zu bytes, 128-byte aligned", gemm_ln_pair_workspace_bytes());
  LLB_CHECK_ARG(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(e.x) |
                  reinterpret_cast<uintptr_t>(e.xb) | reinterpret_cast<uintptr_t>(e.shift) | reinterpret_cast<uintptr_t>(e.scale) |
                  reinterpret_cast<uintptr_t>(e.gate)) & 15) == 0,
                "gemm_ln_pair: operands must be 16-byte aligned");
  LLB_CHECK_ARG(A != (const void*)e.xb, "gemm_ln_pair: the A operand must not alias the bf16 output");
  CUtensorMap tmA, tmBh, tmX, tmXb, tmXpf;
  LLB_TRY(make_tensor_map_2d(&tmA, A, 2, M, K, lda, GEMM_BK, GEMM_BM, 128));
  LLB_TRY(make_tensor_map_2d(&tmBh, W, 2, N, K, ldw, GEMM_BK, GLN_BN / 2, 128));
  LLB_TRY(make_tensor_map_2d(&tmX, e.x, 4, M, N, e.ldx, 32, 32, 128));
  LLB_TRY(make_tensor_map_2d(&tmXb, e.xb, 2, M, N, e.ldxb, 32, 32, 64));
  LLB_TRY(make_tensor_map_2d(&tmXpf, e.x, 4, M, N, e.ldx, GLN_BN, GEMM_BM, 0));
  // long K: the main loop is the long pole -> 5-stage ring, single modulation stage, no L2 prefetch of the residual (its
  // 128 KB TMA prefetch per tile delays the ring's loads; the residual reads hide behind the MMAs anyway);
  // short K: the epilogue is -> modulation stager two tiles ahead, residual prefetched.
  const bool long_k = K > 2048;
  auto kern = long_k ? gemm_ln_pair_kernel<5, 1, 1, 4, false> : gemm_ln_pair_kernel<4, 1, 2, 4, false>;
  const int smem_bytes = long_k ? GlnPairSmemT<5, 1, 1>::TOTAL : GlnPairSmemT<4, 1, 2>::TOTAL;
  static bool configured[2] = {false, false};
  static int max_groups_v[2] = {0, 0};
  static bool cooperative = true;
  if (!configured[long_k]) {
    LLB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    cudaLaunchConfig_t q = {};
    q.blockDim = dim3(GEMM_THREADS), q.dynamicSmemBytes = smem_bytes, q.gridDim = dim3(2 * (num_sms() / 2));
    int n = 0;
    LLB_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &q));
    max_groups_v[long_k] = n / 4 < GLN_PAIR_MAX_GROUPS ? n / 4 : GLN_PAIR_MAX_GROUPS;
    LLB_CHECK_ARG(max_groups_v[long_k] > 0, "gemm_ln_pair: fewer than four CTA pairs fit on this device");
    configured[long_k] = true;
  }
  const int max_groups = max_groups_v[long_k];
  const int num_mb = ceil_div(M, 2 * GEMM_BM);
  const int G = num_mb < max_groups ? num_mb : max_groups;
  uint4* stats = reinterpret_cast<uint4*>(sync_ws);
  // launch-unique tag prefix: stale mailboxes of earlier launches (or whatever the workspace held before) never match
  static std::atomic<uint32_t> epoch{0x5eed};
  LLB_CHECK_ARG(ceil_div(num_mb, G) < 4096, "gemm_ln_pair: M=%d is too large for the mailbox tags", M);
  const uint32_t tag_base = epoch.fetch_add(1) << 12;
  const int prefetch_x = long_k ? 0 : 1;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;   // every CTA of the grid is resident: the groups spin on each other
  attr[0].val.cooperative = 1;
  cfg.blockDim = dim3(GEMM_THREADS), cfg.dynamicSmemBytes = smem_bytes, cfg.stream = stream, cfg.attrs = attr;
  cfg.gridDim = dim3(2 * 4 * G);
  {
    ProfScope prof(ctr ? ctr->slot : LLB_PROF_GEMM_OTHER, stream);
    cudaError_t err = cudaErrorNotSupported;
    if (cooperative) {
      cfg.numAttrs = 1;
      err = cudaLaunchKernelEx(&cfg, kern, tmA, tmBh, tmX, tmXb, tmXpf, M, K, G, e, stats, tag_base, prefetch_x);
      if (err != cudaSuccess) {
        (void)cudaGetLastError();
        cooperative = false;   // this driver does not combine clusters with cooperative launch; the grid still fits the device
      }
    }
    if (!cooperative) {
      cfg.numAttrs = 0;
      err = cudaLaunchKernelEx(&cfg, kern, tmA, tmBh, tmX, tmXb, tmXpf, M, K, G, e, stats, tag_base, prefetch_x);
    }
    LLB_CUDA_OK(err);
    note_kernel(LLB_KERN_GEMM_LN_PAIR);
  }
  LLB_CUDA_OK(cudaGetLastError());
  if (ctr) ctr->launches++;
  return LLB_OK;
}

template <int NS>
static int launch_gin_tail_ns(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const GinTailArgs& t, void* sync_ws,
                              cudaStream_t stream, LaunchCounter* ctr) {
  CUtensorMap tmA, tmBh, tmX, tmXb, tmXpf;
  LLB_TRY(make_tensor_map_2d(&tmA, A, 2, M, K, lda, GEMM_BK, GEMM_BM, 128));
  LLB_TRY(make_tensor_map_2d(&tmBh, W, 2, N, K, ldw, GEMM_BK, GLN_BN / 2, 128));
  LLB_TRY(make_tensor_map_2d(&tmX, t.x, 4, M, N, t.ldx, 32, 32, 128));
  LLB_TRY(make_tensor_map_2d(&tmXb, t.xb, 2, M, N, t.ldxb, 32, 32, 64));
  LLB_TRY(make_tensor_map_2d(&tmXpf, t.x, 4, M, N, t.ldx, GLN_BN, GEMM_BM, 0));
  // long K: (5 stages, one staging tile); short K: (4 stages, two staging tiles, the next chunk's residual loaded a chunk ahead).
  // Measured at K = 3072 (ncu, tensor pipe active): 67 % vs 60 %, and an L2 prefetch of the next tile's residual block loses too.
  const bool long_k = K > 2048;
  const int prefetch_x = t.a_f16 ? 2 : 0;
  auto kern = long_k ? gemm_ln_pair_kernel<5, 1, 1, NS, true> : gemm_ln_pair_kernel<4, 1, 2, NS, true>;
  const int smem_bytes = long_k ? GlnPairSmemT<5, 1, 1>::TOTAL : GlnPairSmemT<4, 1, 2>::TOTAL;
  static bool configured[2] = {false, false};
  static int max_groups_v[2] = {0, 0};
  static bool cooperative = true;
  if (!configured[long_k]) {
    LLB_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    cudaLaunchConfig_t q = {};
    q.blockDim = dim3(GEMM_THREADS), q.dynamicSmemBytes = smem_bytes, q.gridDim = dim3(2 * (num_sms() / 2));
    int n = 0;
    LLB_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, kern, &q));
    // the mailbox area holds GLN_PAIR_MAX_GROUPS x 4 slices = 72 (group, slice) columns
    const int cap = GLN_PAIR_MAX_GROUPS * 4 / NS;
    max_groups_v[long_k] = n / NS < cap ? n / NS : cap;
    LLB_CHECK_ARG(max_groups_v[long_k] > 0, "gin_tail: fewer than %d CTA pairs fit on this device", NS);
    configured[long_k] = true;
  }
  const int max_groups = max_groups_v[long_k];
  const int num_mb = ceil_div(M, 2 * GEMM_BM);
  const int G = num_mb < max_groups ? num_mb : max_groups;
  uint4* stats = reinterpret_cast<uint4*>(sync_ws);
  static std::atomic<uint32_t> epoch{0x9117};
  LLB_CHECK_ARG(ceil_div(num_mb, G) < 4096, "gin_tail: M=%d is too large for the mailbox tags", M);
  const uint32_t tag_base = epoch.fetch_add(1) << 12;
  cudaLaunchConfig_t cfg = {};
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;   // every CTA of the grid is resident: the pairs of a group spin on each other
  attr[0].val.cooperative = 1;
  cfg.blockDim = dim3(GEMM_THREADS), cfg.dynamicSmemBytes = smem_bytes, cfg.stream = stream, cfg.attrs = attr;
  cfg.gridDim = dim3(2 * NS * G);
  {
    ProfScope prof(ctr ? ctr->slot : LLB_PROF_GEMM_OTHER, stream);
    cudaError_t err = cudaErrorNotSupported;
    if (cooperative) {
      cfg.numAttrs = 1;
      err = cudaLaunchKernelEx(&cfg, kern, tmA, tmBh, tmX, tmXb, tmXpf, M, K, G, t, stats, tag_base, prefetch_x);
      if (err != cudaSuccess) {
        (void)cudaGetLastError();
        cooperative = false;
      }
    }
    if (!cooperative) {
      cfg.numAttrs = 0;
      err = cudaLaunchKernelEx(&cfg, kern, tmA, tmBh, tmX, tmXb, tmXpf, M, K, G, t, stats, tag_base, prefetch_x);
    }
    LLB_CUDA_OK(err);
    note_kernel(LLB_KERN_GIN_FUSED_MLP);
  }
  LLB_CUDA_OK(cudaGetLastError());
  if (ctr) ctr->launches++;
  return LLB_OK;
}

int launch_gin_tail(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const GinTailArgs& t, void* sync_ws, size_t sync_bytes,
                    cudaStream_t stream, LaunchCounter* ctr) {
  if (M <= 0) return LLB_OK;
  LLB_CHECK_ARG(gin_tail_supported(N, K), "gin_tail: N=%d must be 768 or 1024 and K=%d a multiple of 8", N, K);
  LLB_CHECK_ARG(lda % 8 == 0 && ldw % 8 == 0 && t.ldx % 4 == 0 && t.ldxb % 8 == 0 && t.mod_ld % 4 == 0 && t.addvec_ld % 4 == 0,
                "gin_tail: leading dimensions must keep rows 16-byte aligned");
  LLB_CHECK_ARG(t.row_group && t.x && t.xb && ((t.gamma && t.beta) || (t.shift && t.scale)), "gin_tail: null operand");
  LLB_CHECK_ARG(sync_ws && sync_bytes >= gemm_ln_pair_workspace_bytes() && (reinterpret_cast<uintptr_t>(sync_ws) & 127) == 0,
                "gin_tail: the exchange workspace needs %zu bytes, 128-byte aligned", gemm_ln_pair_workspace_bytes());
  LLB_CHECK_ARG(((reinterpret_cast<uintptr_t>(A) | reinterpret_cast<uintptr_t>(W) | reinterpret_cast<uintptr_t>(t.x) | reinterpret_cast<uintptr_t>(t.xb) |
                  reinterpret_cast<uintptr_t>(t.shift) | reinterpret_cast<uintptr_t>(t.scale) | reinterpret_cast<uintptr_t>(t.gate) |
                  reinterpret_cast<uintptr_t>(t.addvec)) & 15) == 0,
                "gin_tail: operands must be 16-byte aligned");
  LLB_CHECK_ARG(A != (const void*)t.xb, "gin_tail: the A operand must not alias the bf16 output");
  if (N == 3 * GLN_BN) return launch_gin_tail_ns<3>(A, lda, W, ldw, M, N, K, t, sync_ws, stream, ctr);
  return launch_gin_tail_ns<4>(A, lda, W, ldw, M, N, K, t, sync_ws, stream, ctr);
}

}  // namespace llb

#ifdef LLB_GEMM_TRACE
extern "C" void llb_gln_set_trace(long long* p) { cudaMemcpyToSymbol(llb::g_gln_trace, &p, sizeof(p)); }
extern "C" void llb_gln_set_exp(int m) { cudaMemcpyToSymbol(llb::g_gln_exp, &m, sizeof(m)); }
#endif

extern "C" int llb_gemm_ln_workspace_bytes(size_t* bytes) {
  LLB_CHECK_ARG(bytes, "llb_gemm_ln_workspace_bytes: null argument");
  *bytes = llb::gemm_ln_pair_workspace_bytes();
  return LLB_OK;
}

extern "C" int llb_gemm_ln_residual_ws(const void* A, int lda, const void* W, int ldw, const float* bias, const int32_t* row_group,
                                       const float* shift, const float* scale, const float* gate, int mod_ld, float* x, int ldx,
                                       void* xb, int ldxb, int M, int N, int K, void* workspace, size_t workspace_bytes,
                                       llb_stream_t stream) {
  LLB_TRY(llb::require_sm100());
  LLB_CHECK_ARG(A && W, "llb_gemm_ln_residual_ws: null operand");
  llb::GemmLnArgs e{bias, row_group, shift, scale, gate, mod_ld, x, ldx, reinterpret_cast<__nv_bfloat16*>(xb), ldxb};
  return llb::launch_gemm_ln_pair(A, lda, W, ldw, M, N, K, e, workspace, workspace_bytes, (cudaStream_t)stream, nullptr);
}
