// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[M,N] = epilogue(A[M,K] . W[N,K]^T)
//
// A (activations) and W (nn.Linear weight, (out,in)) are both K-major bf16, so both operands go through TMA
// with the 128-byte swizzle straight into the UMMA shared-memory layout.
//
// Persistent, warp-specialised CTA (one per SM), 12 warps:
//   warps 0..7  epilogue: tcgen05.ld their TMEM lane quarter (warp % 4), run the fused epilogue functor, stage the
//               converted chunk in swizzled shared memory and hand it to a TMA store (full 128-byte lines, no LSU
//               pressure), then release the accumulator stage (tmem_empty[acc]) so the next tile's MMAs overlap
//   warp 8      TMA producer: fills a ring of STAGES {A 128x64, W BNx64} tiles, arms full[] with expect_tx
//   warp 9      MMA issuer: one elected lane issues tcgen05.mma (M=128, N=BN, K=16) x4 per stage and
//               tcgen05.commit's the stage's empty[] barrier; after the last k-block commits tmem_full[acc]
//   warp 10     TMEM allocator (2 accumulator stages x BN fp32 columns)
// The producer / issuer warps carry the highest warp ids on their scheduler: the issue arbiter prefers high ids,
// so a busy epilogue can never starve the single thread that feeds the tensor pipe.
// Tiles are walked n-fastest so that the CTAs in flight share A tiles through L2 and W stays L2-resident.
#pragma once
#include <type_traits>
#include "llb_common.cuh"

namespace llb {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_EPI_WARPS = 8;
constexpr int GEMM_THREADS = 32 * (GEMM_EPI_WARPS + 4);
constexpr int GEMM_STAGING_PER_WARP = 8192;  // ring of 32-row staging boxes: 4 x (32 x 64 B) or 2 x (32 x 128 B)

template <int BN>
struct GemmCfg {
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;
  static constexpr int B_BYTES = BN * GEMM_BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (BN == 256) ? 3 : (BN == 128 ? 5 : 6);
  static constexpr int TMEM_COLS = 2 * BN;  // 512 / 256 / 128
  static constexpr int STAGING_BYTES = GEMM_EPI_WARPS * GEMM_STAGING_PER_WARP;
  static constexpr int BAR_BYTES = 256;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + BAR_BYTES + 1024;  // +1024: alignment slack
};

__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

#ifdef LLB_GEMM_TRACE
// Debug-only instrumentation (tools/gemm_trace.cu, never compiled into the library): per-tile cycle stamps of every
// role of CTA pair 0, and an experiment mask that switches single pipeline stages off to find the binding one
// (1 = no MMA issue, 2 = no epilogue at all, 4 = no epilogue math, 8 = no epilogue store).
__device__ long long* g_gemm_trace = nullptr;   // [tile][16]
__device__ int g_gemm_exp = 0;
#define LLB_TRACE(tile_idx, slot, value) \
  do { if (g_gemm_trace && blockIdx.x < 2) g_gemm_trace[((size_t)(tile_idx) * 2 + blockIdx.x) * 16 + (slot)] = (value); } while (0)
#define LLB_EXP(bit) ((g_gemm_exp & (bit)) != 0)
#else
#define LLB_TRACE(tile_idx, slot, value) do { } while (0)
#define LLB_EXP(bit) false
#endif

// Epilogue functors that only reduce (no C matrix) declare `static constexpr bool NO_STORE = true`.
template <class E, class = void>
struct epi_no_store : std::false_type {};
template <class E>
struct epi_no_store<E, std::void_t<decltype(E::NO_STORE)>> : std::integral_constant<bool, E::NO_STORE> {};

// Epilogue functors may carry per-ROW state across the column chunks of a tile (a running reduction, a row statistic looked up
// once): they declare `struct RowState` and the three-call protocol below.
template <class E, class = void>
struct epi_row_state : std::false_type {};
template <class E>
struct epi_row_state<E, std::void_t<typename E::RowState>> : std::true_type {};
// Functors that produce their 16-bit output already PACKED (half2 arithmetic) declare `static constexpr bool PACKS_OUTPUT = true`
// and implement transform_pack(row, col0, const float* v, uint32_t* out16, M, N[, RowState&]): 32 accumulators -> 16 words.
template <class E, class = void>
struct epi_packs : std::false_type {};
template <class E>
struct epi_packs<E, std::void_t<decltype(E::PACKS_OUTPUT)>> : std::integral_constant<bool, E::PACKS_OUTPUT> {};
// Functors that read per-COLUMN vectors (LayerNorm weights, biases) can have their warp's slice of up to three of them staged in
// WARP-PRIVATE shared memory: `static constexpr int WARP_VECS = k` and `const float* warp_vec(int i) const`.  Every epilogue warp
// loads the 128 columns it will work on (lane l: columns 4 l .. 4 l + 3 of each vector) BEFORE it waits for the tile's
// accumulators and reads them back as broadcast LDS per chunk: one exposed L2 round trip per tile instead of one per
// 32-column chunk (shared memory leaves this kernel next to no L1), and no barrier between warps -- a block-wide staging
// behind a named barrier put the eight warps in lockstep and cost more than it saved.
template <class E, class = void>
struct epi_warp_vecs : std::integral_constant<int, 0> {};
template <class E>
struct epi_warp_vecs<E, std::void_t<decltype(E::WARP_VECS)>> : std::integral_constant<int, E::WARP_VECS> {};
struct EpiNoRowState {};
template <class E, bool HAS = epi_row_state<E>::value>
struct epi_row_state_of { using type = EpiNoRowState; };
template <class E>
struct epi_row_state_of<E, true> { using type = typename E::RowState; };

// One epilogue warp's share of a 128 x BN accumulator tile: warp % 4 selects the TMEM lane quarter (32 rows), the
// warps sharing a quarter split the columns.  tcgen05.ld -> fused functor -> swizzled smem staging -> TMA store.
// The per-row state of this thread's row of tile row-block m0: computed BEFORE the thread waits for the tile's accumulators, so
// that whatever the functor looks up for the row (e.g. its LayerNorm statistics) travels while the tile's MMAs still run.
template <class Epi>
__device__ __forceinline__ typename epi_row_state_of<Epi>::type gemm_epilogue_row_begin(const Epi& epi, int m0, int M) {
  if constexpr (epi_row_state<Epi>::value) {
    return epi.row_begin(m0 + (uniform_warp_idx() & 3) * 32 + (int)(threadIdx.x & 31), M);
  } else {
    return EpiNoRowState{};
  }
}

// per-warp staging area: a ring of 32-row output boxes, minus 2 KB for the staged column vectors of functors that ask for them
template <class Epi>
struct GemmWarpStaging {
  static constexpr int NV = epi_warp_vecs<Epi>::value;
  static constexpr int RING_BYTES = NV > 0 ? GEMM_STAGING_PER_WARP - 2048 : GEMM_STAGING_PER_WARP;
  static_assert(NV <= 3, "at most three staged vectors (3 x 128 floats = 1.5 KB per warp)");
};
// this warp's 128-column slices of the functor's vectors -> its private shared memory (call before waiting for the accumulators)
template <int BN, class Epi>
__device__ __forceinline__ void gemm_stage_warp_vectors(const Epi& epi, uint8_t* stg, int n0, int N) {
  constexpr int NV = epi_warp_vecs<Epi>::value;
  if constexpr (NV > 0) {
    constexpr int COLS_PER_WARP = BN / (GEMM_EPI_WARPS / 4);
    static_assert(COLS_PER_WARP == 128, "warp-staged vectors assume 128 columns per epilogue warp");
    const int lane = threadIdx.x & 31, cg = uniform_warp_idx() >> 2;
    const uint32_t wv = smem_u32(stg) + GemmWarpStaging<Epi>::RING_BYTES;
    const int col = n0 + cg * COLS_PER_WARP + 4 * lane;
    __syncwarp();   // the previous tile's reads of this area are done
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const float* src = epi.warp_vec(i);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (col + 3 < N) v = __ldg(reinterpret_cast<const float4*>(src + col));
      else if (col < N) v = make_float4(__ldg(src + col), col + 1 < N ? __ldg(src + col + 1) : 0.f, col + 2 < N ? __ldg(src + col + 2) : 0.f, 0.f);
      sts128(wv + (i * COLS_PER_WARP + 4 * lane) * 4, v);
    }
    __syncwarp();
  }
}

template <int BN, bool TMA_STORE, class Epi>
__device__ __forceinline__ void gemm_epilogue_tile(const Epi& epi, const CUtensorMap* tmC, uint32_t tmem_acc, int m0, int n0, int M,
                                                   int N, uint8_t* stg, int& buf, typename epi_row_state_of<Epi>::type rst) {
  constexpr int ELEM = Epi::OUT_F32 ? 4 : 2;
  constexpr int ROW_BYTES = Epi::CHUNK * ELEM;
  constexpr int NBUF = GemmWarpStaging<Epi>::RING_BYTES / (32 * ROW_BYTES);
  constexpr bool WV = epi_warp_vecs<Epi>::value > 0;
  static_assert(NBUF >= 1, "staging ring too small for this epilogue");
  constexpr int COLS_PER_WARP = BN / (GEMM_EPI_WARPS / 4);
  constexpr bool ROW_STATE = epi_row_state<Epi>::value;
  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  const int quarter = warp & 3, cg = warp >> 2;
  const int row = m0 + quarter * 32 + lane;
  const uint32_t t_row = tmem_acc + ((uint32_t)(quarter * 32) << 16) + cg * COLS_PER_WARP;
  constexpr bool PACKS = epi_packs<Epi>::value;
  static_assert(!PACKS || (!Epi::OUT_F32 && Epi::CHUNK == 32), "packed epilogues produce 32 16-bit columns per call");
  float v[Epi::CHUNK];
  [[maybe_unused]] uint32_t packed[PACKS ? 16 : 1];
#pragma unroll 1
  for (int c = 0; c < COLS_PER_WARP; c += Epi::CHUNK) {
    const int col0 = n0 + cg * COLS_PER_WARP + c;
    if (col0 >= N) break;   // warp-uniform
    tmem_ld32(t_row + c, v);
    if (Epi::CHUNK == 64) tmem_ld32(t_row + c + 32, v + 32);
    tmem_ld_wait();
    if (!LLB_EXP(4)) {
      if constexpr (PACKS && WV) {
        epi.transform_pack(row, col0, v, packed, M, N, rst, smem_u32(stg) + GemmWarpStaging<Epi>::RING_BYTES + c * 4);
      } else if constexpr (PACKS) {
        if constexpr (ROW_STATE) epi.transform_pack(row, col0, v, packed, M, N, rst);
        else epi.transform_pack(row, col0, v, packed, M, N);
      } else if constexpr (ROW_STATE) {
        epi.transform(row, col0, v, M, N, rst);
      } else {
        epi.transform(row, col0, v, M, N);
      }
    }
    if (LLB_EXP(8) || epi_no_store<Epi>::value) continue;
    if (TMA_STORE) {
      uint8_t* dst = stg + buf * (32 * ROW_BYTES);
      if (elect_one()) bulk_wait_read<NBUF - 1>();   // the buffer about to be overwritten has been read out
      __syncwarp();
      // row `lane` of the staging tile, 16-byte pieces XOR-swizzled exactly like the C tensor map
      uint8_t* rowp = dst + lane * ROW_BYTES;
      const int sw = ROW_BYTES == 128 ? (lane & 7) : ((lane >> 1) & 3);
#pragma unroll
      for (int p = 0; p < ROW_BYTES / 16; ++p) {
        uint4 q;
        if constexpr (PACKS) {
          q = make_uint4(packed[4 * p], packed[4 * p + 1], packed[4 * p + 2], packed[4 * p + 3]);
        } else if (Epi::OUT_F32) {
          q = make_uint4(__float_as_uint(v[4 * p]), __float_as_uint(v[4 * p + 1]), __float_as_uint(v[4 * p + 2]),
                         __float_as_uint(v[4 * p + 3]));
        } else {
          q = make_uint4(pack_bf16x2(v[8 * p], v[8 * p + 1]), pack_bf16x2(v[8 * p + 2], v[8 * p + 3]),
                         pack_bf16x2(v[8 * p + 4], v[8 * p + 5]), pack_bf16x2(v[8 * p + 6], v[8 * p + 7]));
        }
        *reinterpret_cast<uint4*>(rowp + ((p ^ sw) << 4)) = q;
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        tma_store_2d(tmC, dst, col0, m0 + quarter * 32);
        bulk_commit();
      }
      buf = (buf + 1) % NBUF;
    } else if (row < M) {
      if constexpr (PACKS) {   // unaligned C: pairs of 16-bit values through generic stores (ldc and N even)
        uint32_t* out = reinterpret_cast<uint32_t*>(reinterpret_cast<uint16_t*>(epi.C) + (size_t)row * epi.ldc + col0);
        for (int i = 0; i < 16; ++i)
          if (col0 + 2 * i < N) out[i] = packed[i];
      } else if (Epi::OUT_F32) {
        float* out = reinterpret_cast<float*>(epi.C) + (size_t)row * epi.ldc + col0;
        for (int i = 0; i < Epi::CHUNK; ++i)
          if (col0 + i < N) out[i] = v[i];
      } else {
        __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(epi.C) + (size_t)row * epi.ldc + col0;
        for (int i = 0; i < Epi::CHUNK; ++i)
          if (col0 + i < N) out[i] = __float2bfloat16(v[i]);
      }
    }
  }
  // slot = which (N tile, column group) of the row this warp covered: (N / BN rounded up) * (epilogue warps / 4) slots per row
  if constexpr (ROW_STATE) epi.row_end(row, (n0 / BN) * (GEMM_EPI_WARPS / 4) + cg, rst, M);
}

// Epilogue functor contract:
//   static constexpr int  CHUNK   (32 or 64): consecutive accumulator columns handed over per call
//   static constexpr bool OUT_F32 : element type of C (fp32 or bf16); CHUNK * sizeof(elem) <= 128
//   void* C; int ldc;              output matrix (row-major)
//   __device__ void transform(int row, int col0, float* v, int M, int N) const   -- in place on v[CHUNK];
//     called for every row of the tile, including rows >= M (their results are never stored).
//   optional per-row state (struct RowState): RowState row_begin(row, M); transform(..., RowState&); row_end(row, slot, RowState&, M)
//     -- row_begin once per (tile, thread) BEFORE the thread waits for the accumulators, row_end after the last chunk, slot as above.
template <int BN, bool TMA_STORE, class Epi>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmC, int M, int N, int K, Epi epi, int group_n, int group_k, int group_w, int opts) {
  using Cfg = GemmCfg<BN>;
  const int ab_f16 = opts & 1;
  const bool m_fast = (opts & 2) != 0;   // walk the tiles m-fastest: a narrow A stays in L2 while a wide W is streamed once
  constexpr int STAGES = Cfg::STAGES;
  constexpr int ELEM = Epi::OUT_F32 ? 4 : 2;
  constexpr int ROW_BYTES = Epi::CHUNK * ELEM;            // 64 or 128
  static_assert(ROW_BYTES == 64 || ROW_BYTES == 128, "epilogue chunk must be 64 or 128 bytes per row");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smA = smem;
  uint8_t* smB = smem + STAGES * Cfg::A_BYTES;
  uint8_t* smStage = smem + STAGES * Cfg::STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smStage + Cfg::STAGING_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int num_m = (M + GEMM_BM - 1) / GEMM_BM;
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;

  if (warp == GEMM_EPI_WARPS && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (TMA_STORE) tma_prefetch_desc(&tmC);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], GEMM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == GEMM_EPI_WARPS + 2) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();   // the next kernel of the stream may begin its own prologue on SMs this grid leaves free
  LLB_STAMP(0x10 + BN / 64, ((unsigned long long)N << 32) | (unsigned)K, threadIdx.x == 0);

  if (warp == GEMM_EPI_WARPS) {
    // ---------------- TMA producer: the whole warp walks the ring (uniform control flow), one elected lane issues ----------------
    int stage = 0;
    uint32_t phase = 0;
    // The WEIGHT tiles of the first ring stages do not depend on the previous kernel of the stream: they are requested before the
    // dependency wait (programmatic dependent launch), so at small batch sizes -- where a step is a chain of ~170 short kernels,
    // each waiting for its first weight bytes -- that latency overlaps the predecessor's tail.  Activations follow after the wait.
    int hoisted = 0;
    if (blockIdx.x < num_tiles) {
      const int tile = blockIdx.x;
      const int n0 = (m_fast ? tile / num_m : tile % num_n) * BN;
      const int grp_i = group_n > 0 ? n0 / group_n : 0;
      const int kw0 = group_w ? grp_i * group_k : 0, wn0 = group_w ? n0 - grp_i * group_n : n0;
      hoisted = num_kb < STAGES ? num_kb : STAGES;
      if (elect_one()) {
        for (int kb = 0; kb < hoisted; ++kb) {
          mbar_arrive_expect_tx(&full[kb], Cfg::STAGE_BYTES);
          tma_load_2d(smB + kb * Cfg::B_BYTES, &tmB, &full[kb], kw0 + kb * GEMM_BK, wn0);
        }
      }
      __syncwarp();
    }
    pdl_wait();
    LLB_STAMP(0x20 + BN / 64, ((unsigned long long)N << 32) | (unsigned)K, lane == 0);
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = (m_fast ? tile % num_m : tile / num_n) * GEMM_BM;
      const int n0 = (m_fast ? tile / num_m : tile % num_n) * BN;
      // grouped along N: group g reads A columns [g group_k, +K); split-K flavour (group_w): it also reads the SAME W rows
      // at columns [g group_k, +K), i.e. the groups are the K-slices of one linear and C holds their partial products
      const int grp_i = group_n > 0 ? n0 / group_n : 0;
      const int ka0 = grp_i * group_k;
      const int kw0 = group_w ? ka0 : 0, wn0 = group_w ? n0 - grp_i * group_n : n0;
      for (int kb = 0; kb < num_kb; ++kb) {
        const bool pre = hoisted > 0;   // this stage's barrier is armed and its weight tile is on its way already
        if (!pre) mbar_wait(&empty[stage], phase ^ 1);
        if (elect_one()) {
          if (!pre) mbar_arrive_expect_tx(&full[stage], Cfg::STAGE_BYTES);
          tma_load_2d(smA + stage * Cfg::A_BYTES, &tmA, &full[stage], ka0 + kb * GEMM_BK, m0);
          if (!pre) tma_load_2d(smB + stage * Cfg::B_BYTES, &tmB, &full[stage], kw0 + kb * GEMM_BK, wn0);
        }
        if (pre) --hoisted;
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
    }
  } else if (warp == GEMM_EPI_WARPS + 1) {
    // ---------------- MMA issuer: converged warp, one elected lane issues (operands stay in uniform registers) ----------------
    pdl_wait();
    const uint32_t idesc = umma_idesc_ab(GEMM_BM, BN, ab_f16 != 0);
    const uint64_t a_desc0 = umma_desc_k128(smem_u32(smA));   // stage 0, k-step 0; stages / k-steps are plain adds
    const uint64_t b_desc0 = umma_desc_k128(smem_u32(smB));
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + acc * BN;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full[stage], phase);
        if (kb == 0 || kb == num_kb - 1) LLB_STAMP(kb == 0 ? 0x40 : 0x50, ((unsigned long long)N << 32) | (unsigned)K, lane == 0);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t a_desc = a_desc0 + (uint64_t)(stage * (Cfg::A_BYTES >> 4));
          const uint64_t b_desc = b_desc0 + (uint64_t)(stage * (Cfg::B_BYTES >> 4));
#pragma unroll
          for (int k = 0; k < GEMM_BK / 16; ++k) umma_bf16(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      if (elect_one()) umma_commit(&tmem_full[acc]);
      __syncwarp();
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
  } else if (warp < GEMM_EPI_WARPS) {
    // ---------------- epilogue ----------------
    pdl_wait();   // the functor may read what the previous kernel wrote (row statistics), and C may be a buffer it still reads
    uint8_t* stg = smStage + warp * GEMM_STAGING_PER_WARP;
    int buf = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = (m_fast ? tile % num_m : tile / num_n) * GEMM_BM;
      const int n0 = (m_fast ? tile / num_m : tile % num_n) * BN;
      const auto rst = gemm_epilogue_row_begin(epi, m0, M);
      gemm_stage_warp_vectors<BN>(epi, stg, n0, N);
      mbar_wait(&tmem_full[acc], acc_phase);
      LLB_STAMP(0x60, ((unsigned long long)N << 32) | (unsigned)K, threadIdx.x == 0);
      tc_fence_after();
      gemm_epilogue_tile<BN, TMA_STORE>(epi, &tmC, tmem_base + acc * BN, m0, n0, M, N, stg, buf, rst);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    // the staging buffers must have been read before the CTA retires its shared memory; the global writes themselves are part of
    // the grid's completion like any other store
    if (TMA_STORE && lane == 0) bulk_wait_read<0>();
  }
  tc_fence_before();
  __syncthreads();
  LLB_STAMP(0x30 + BN / 64, ((unsigned long long)N << 32) | (unsigned)K, threadIdx.x == 0);
  if (warp == GEMM_EPI_WARPS + 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// cta_group::2 variant: a CTA PAIR (cluster of 2, same TPC) computes a 256 x 256 tile.  CTA r owns rows
// [m0 + 128 r, +128) and loads only HALF of the W tile (rows n0 + 128 r ..); tcgen05.mma.cta_group::2 (issued by the
// leader CTA's single thread) makes both tensor cores read the concatenated B operand, so per SM the shared-memory
// and L2->SM traffic per MMA drops by a third (A 16 KB + B 16 KB per 64-wide k-block instead of 16 + 32) and the
// ring deepens to 6 stages.  Barriers: full[] lives in the leader (both CTAs' TMA loads complete_tx on it),
// empty[] / tmem_full[] are signalled in both CTAs by a multicast tcgen05.commit, tmem_empty[] lives in the leader and
// collects the epilogue warps of both CTAs.
// ------------------------------------------------------------------------------------------------

struct Gemm2Cfg {
  static constexpr int BN = 256;
  static constexpr int A_BYTES = GEMM_BM * GEMM_BK * 2;        // 16 KB
  static constexpr int B_BYTES = (BN / 2) * GEMM_BK * 2;       // 16 KB (this CTA's half of the W tile)
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = 5;
  static constexpr int TMEM_COLS = 2 * BN;
  static constexpr int STAGING_BYTES = GEMM_EPI_WARPS * GEMM_STAGING_PER_WARP;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STAGING_BYTES + 256 + 1024;
};

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load whose completion bytes are credited to the LEADER CTA's mbarrier (peer bit of the cluster address cleared).
__device__ __forceinline__ void tma_load_2d_2sm(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accum)
      : "memory");
}
// Arrives (once the issued MMAs have completed) on the barrier at this offset in BOTH CTAs of the pair.
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3)
               : "memory");
}
// Arrive on an mbarrier of CTA `cta` of the cluster.  Relaxed: the accumulator hand-over it signals is ordered by
// tcgen05.wait::ld + tcgen05.fence::before_thread_sync, and a release at cluster scope costs a MEMBAR.GPU per arrive.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

template <bool TMA_STORE, class Epi>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
gemm_tcgen05_2cta_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                         const __grid_constant__ CUtensorMap tmC, int M, int N, int K, Epi epi, int group_n, int group_k, int group_w, int opts) {
  using Cfg = Gemm2Cfg;
  const int ab_f16 = opts & 1;
  const bool m_fast = (opts & 2) != 0;   // walk the tiles m-fastest: a narrow A stays in L2 while a wide W is streamed once
  constexpr int STAGES = Cfg::STAGES;
  constexpr int BN = Cfg::BN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* smA = smem;
  uint8_t* smB = smem + STAGES * Cfg::A_BYTES;
  uint8_t* smStage = smem + STAGES * Cfg::STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smStage + Cfg::STAGING_BYTES);
  uint64_t* full = bars;
  uint64_t* empty = bars + STAGES;
  uint64_t* tmem_full = bars + 2 * STAGES;
  uint64_t* tmem_empty = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;
  const int num_m = (M + 2 * GEMM_BM - 1) / (2 * GEMM_BM);
  const int num_n = (N + BN - 1) / BN;
  const int num_tiles = num_m * num_n;
  const int num_kb = (K + GEMM_BK - 1) / GEMM_BK;

  if (warp == GEMM_EPI_WARPS && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    if (TMA_STORE) tma_prefetch_desc(&tmC);
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tmem_full[a], 1);
      mbar_init(&tmem_empty[a], 2 * GEMM_EPI_WARPS);
    }
    fence_mbar_init();
  }
  cluster_sync_all();
  if (warp == GEMM_EPI_WARPS + 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  LLB_STAMP(0x1D, ((unsigned long long)N << 32) | (unsigned)K, threadIdx.x == 0);

  if (warp == GEMM_EPI_WARPS) {
    // ---------------- TMA producer (both CTAs; completion bytes go to the leader's full[]) ----------------
    // the whole warp walks the ring (uniform control flow); one elected lane issues
    int stage = 0;
    uint32_t phase = 0;
    int tcount = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs, ++tcount) {
      const int m0 = (m_fast ? tile % num_m : tile / num_n) * (2 * GEMM_BM) + rank * GEMM_BM;
      const int n0 = (m_fast ? tile / num_m : tile % num_n) * BN + rank * (BN / 2);
      const int grp_i = group_n > 0 ? n0 / group_n : 0;   // grouped along N (group_n is a multiple of BN), see the single-CTA kernel
      const int ka0 = grp_i * group_k;
      const int kw0 = group_w ? ka0 : 0, wn0 = group_w ? n0 - grp_i * group_n : n0;
      long long wsum = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
#ifdef LLB_GEMM_TRACE
        const long long w0 = clock64();
#endif
        mbar_wait(&empty[stage], phase ^ 1);
#ifdef LLB_GEMM_TRACE
        wsum += clock64() - w0;
        if (kb == num_kb - 1 && lane == 0) { LLB_TRACE(tcount, 0, wsum); LLB_TRACE(tcount, 1, clock64()); }
#endif
        if (elect_one()) {
          if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * Cfg::STAGE_BYTES);
          tma_load_2d_2sm(smA + stage * Cfg::A_BYTES, &tmA, &full[stage], ka0 + kb * GEMM_BK, m0);
          tma_load_2d_2sm(smB + stage * Cfg::B_BYTES, &tmB, &full[stage], kw0 + kb * GEMM_BK, wn0);
        }
        __syncwarp();
        if (++stage == STAGES) {
          stage = 0;
          phase ^= 1;
        }
      }
      (void)wsum;
    }
  } else if (warp == GEMM_EPI_WARPS + 1) {
    // ---------------- MMA issuer (leader CTA only): converged warp, one elected lane issues ----------------
    if (rank == 0) {
      const uint32_t idesc = umma_idesc_ab(2 * GEMM_BM, BN, ab_f16 != 0);
      const uint64_t a_desc0 = umma_desc_k128(smem_u32(smA));   // stage 0, k-step 0; stages / k-steps are plain adds
      const uint64_t b_desc0 = umma_desc_k128(smem_u32(smB));
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      int tcount = 0;
      for (int tile = pair; tile < num_tiles; tile += num_pairs, ++tcount) {
        if (lane == 0) LLB_TRACE(tcount, 2, clock64());
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        if (lane == 0) LLB_TRACE(tcount, 3, clock64());
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        long long fsum = 0;
        for (int kb = 0; kb < num_kb; ++kb) {
#ifdef LLB_GEMM_TRACE
          const long long w0 = clock64();
#endif
          mbar_wait(&full[stage], phase);
#ifdef LLB_GEMM_TRACE
          fsum += clock64() - w0;
          if (kb == num_kb - 1 && lane == 0) { LLB_TRACE(tcount, 4, fsum); LLB_TRACE(tcount, 5, clock64()); }
#endif
          tc_fence_after();
          if (elect_one()) {
            const uint64_t a_desc = a_desc0 + (uint64_t)(stage * (Cfg::A_BYTES >> 4));
            const uint64_t b_desc = b_desc0 + (uint64_t)(stage * (Cfg::B_BYTES >> 4));
#pragma unroll
            for (int k = 0; k < GEMM_BK / 16; ++k) {
              if (!LLB_EXP(1)) umma_bf16_2sm(d_tmem, a_desc + 2 * k, b_desc + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            }
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
        (void)fsum;
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      }
    }
  } else if (warp < GEMM_EPI_WARPS) {
    // ---------------- epilogue (each CTA drains its own 128 x 256 half) ----------------
    uint8_t* stg = smStage + warp * GEMM_STAGING_PER_WARP;
    int buf = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    int tcount = 0;
    for (int tile = pair; tile < num_tiles; tile += num_pairs, ++tcount) {
      const int m0 = (m_fast ? tile % num_m : tile / num_n) * (2 * GEMM_BM) + rank * GEMM_BM;
      const int n0 = (m_fast ? tile / num_m : tile % num_n) * BN;
      if (warp == 0 && lane == 0) LLB_TRACE(tcount, 6, clock64());
      const auto rst = gemm_epilogue_row_begin(epi, m0, M);
      gemm_stage_warp_vectors<BN>(epi, stg, n0, N);
      mbar_wait(&tmem_full[acc], acc_phase);
      if (warp == 0 && lane == 0) LLB_TRACE(tcount, 7, clock64());
      tc_fence_after();
      if (!LLB_EXP(2)) gemm_epilogue_tile<BN, TMA_STORE>(epi, &tmC, tmem_base + acc * BN, m0, n0, M, N, stg, buf, rst);
      tc_fence_before();
      __syncwarp();
      if (warp == 0 && lane == 0) LLB_TRACE(tcount, 8, clock64());
      if (lane == 0) mbar_arrive_cluster(&tmem_empty[acc], 0);
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    }
    if (TMA_STORE && lane == 0) bulk_wait_all();
  }
  tc_fence_before();
  LLB_STAMP(0x3D, ((unsigned long long)N << 32) | (unsigned)K, threadIdx.x == 0);
  cluster_sync_all();   // nobody leaves while the peer may still signal its barriers / read its operand half
  if (warp == GEMM_EPI_WARPS + 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------------
// 2-D tensor map: inner dim = cols (contiguous), outer dim = rows; box = box_cols x box_rows;
// swizzle_bytes in {64, 128} must equal box_cols * elem_bytes; 0 = no swizzle (prefetch-only maps).
int make_tensor_map_2d(CUtensorMap* out, const void* ptr, int elem_bytes, int rows, int cols, int ld_elems, int box_cols,
                       int box_rows, int swizzle_bytes);


// Grouped along N (group_n > 0): output columns [g group_n, (g+1) group_n) are A[:, g group_k : g group_k + K] . W[g group_n ..]^T,
// i.e. G independent linears that share their rows, with their (N_g, K) weights stacked and their inputs side by side --
// one launch instead of G (the 28 adaLN modulation linears of a reverse step).
// split_k: the groups are the K-slices of ONE linear (W is (group_n, G group_k); group g multiplies A[:, g group_k : +K] with
// W[:, g group_k : +K]) and C (M, G group_n) holds the G partial products, to be summed by the consumer in a fixed order.
struct GemmGroups {
  int group_n = 0, group_k = 0;
  bool split_k = false;
  bool ab_f16 = false;   // both operands are IEEE fp16 instead of bf16 (same tile shapes, same descriptors otherwise)
  bool m_fastest = false;   // tile order: consecutive CTAs share a W tile (narrow A resident in L2, wide W streamed from HBM once)
};

template <int BN, class Epi>
int launch_gemm(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const Epi& epi,
                cudaStream_t stream, LaunchCounter* ctr = nullptr, GemmGroups grp = GemmGroups()) {
  using Cfg = GemmCfg<BN>;
  if (M <= 0 || N <= 0) return LLB_OK;
  LLB_CHECK_ARG(K > 0 && lda % 8 == 0 && ldw % 8 == 0, "gemm: K=%d lda=%d ldw=%d (ld must be a multiple of 8)", K, lda, ldw);
  LLB_CHECK_ARG((reinterpret_cast<uintptr_t>(A) & 15) == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0,
                "gemm: operands must be 16-byte aligned");
  constexpr int ELEM = Epi::OUT_F32 ? 4 : 2;
  CUtensorMap tmA, tmB, tmC;
  LLB_CHECK_ARG(grp.group_n == 0 || (grp.group_n % BN == 0 && grp.group_k >= K && grp.group_k % 8 == 0 && N % grp.group_n == 0),
                "gemm: grouped call needs group_n=%d a multiple of the N tile %d dividing N=%d and group_k=%d >= K", grp.group_n, BN, N,
                grp.group_k);
  LLB_CHECK_ARG(!grp.split_k || grp.group_n > 0, "gemm: split_k needs groups");
  const int a_cols = grp.group_n ? (N / grp.group_n - 1) * grp.group_k + K : K;
  const int w_rows = grp.split_k ? grp.group_n : N, w_cols = grp.split_k ? a_cols : K;
  LLB_TRY(make_tensor_map_2d(&tmA, A, 2, M, a_cols, lda, GEMM_BK, GEMM_BM, 128));
  LLB_TRY(make_tensor_map_2d(&tmB, W, 2, w_rows, w_cols, ldw, GEMM_BK, BN, 128));
  const bool tma_store = !epi_no_store<Epi>::value && ((size_t)epi.ldc * ELEM) % 16 == 0 && (reinterpret_cast<uintptr_t>(epi.C) & 15) == 0;
  if (tma_store) LLB_TRY(make_tensor_map_2d(&tmC, epi.C, ELEM, M, N, epi.ldc, Epi::CHUNK, 32, Epi::CHUNK * ELEM));
  else tmC = tmA;
  const int tiles = ceil_div(M, GEMM_BM) * ceil_div(N, BN);
  const int grid = tiles < num_sms() ? tiles : num_sms();
  // m-fastest automatically when A fits the L2 comfortably and W does not (the predictor head: 50 MB of activations against a
  // 1.1 GB weight, which the n-fastest walk would stream from HBM once per 256-row block); never for grouped launches
  const bool m_fast = grp.group_n == 0 && (grp.m_fastest || ((size_t)M * K * 2 <= ((size_t)64 << 20) && (size_t)N * K * 2 >= ((size_t)256 << 20)));
  // CTA-pair kernel: wide problems whose 256 x 256 pair-tiles fill the machine
  const int pair_tiles = ceil_div(M, 2 * GEMM_BM) * ceil_div(N, 256);
  // (not for a single row block: the pair's second CTA would multiply nothing but padding, and a skinny GEMM -- the adaLN
  // modulations of a handful of molecules, 352 MB of weights against 7 rows -- wants every SM streaming its own weight tiles)
  const bool use_pair = BN == 256 && M > GEMM_BM && pair_tiles >= num_sms() / 2 && grp.group_n % 256 == 0;
  const int slot = ctr ? ctr->slot : LLB_PROF_GEMM_OTHER;
  const int flags = (grp.ab_f16 ? 1 : 0) | (m_fast ? 2 : 0);
  if (use_pair) {
    // the cluster shape is the kernel's __cluster_dims__; an ordinary launch
    CUtensorMap tmBh;
    LLB_TRY(make_tensor_map_2d(&tmBh, W, 2, w_rows, w_cols, ldw, GEMM_BK, 128, 128));
    const int pairs = pair_tiles < num_sms() / 2 ? pair_tiles : num_sms() / 2;
    auto launch2 = [&](auto kern) -> int {
      return launch_kernel(ctr, slot, false, kern, dim3(2 * pairs), dim3(GEMM_THREADS), (size_t)Gemm2Cfg::SMEM_BYTES, stream, tmA, tmBh, tmC, M, N,
                           K, epi, grp.group_n, grp.group_k, grp.split_k ? 1 : 0, flags);
    };
    LLB_TRY(tma_store ? launch2(gemm_tcgen05_2cta_kernel<true, Epi>) : launch2(gemm_tcgen05_2cta_kernel<false, Epi>));
    note_kernel(LLB_KERN_GEMM_2CTA);
    return LLB_OK;
  }
  auto launch1 = [&](auto kern) -> int {
    return launch_kernel(ctr, slot, true, kern, dim3(grid), dim3(GEMM_THREADS), (size_t)Cfg::SMEM_BYTES, stream, tmA, tmB, tmC, M, N, K, epi,
                         grp.group_n, grp.group_k, grp.split_k ? 1 : 0, flags);
  };
  LLB_TRY(tma_store ? launch1(gemm_tcgen05_kernel<BN, true, Epi>) : launch1(gemm_tcgen05_kernel<BN, false, Epi>));
  note_kernel(LLB_KERN_GEMM_1CTA);
  return LLB_OK;
}

// ------------------------------------------------------------------------------------------------
// Epilogues
// ------------------------------------------------------------------------------------------------
template <int ACT, bool F32 = true>
__device__ __forceinline__ float apply_act(float x) {
  if (ACT == LLB_ACT_GELU) return F32 ? gelu_fast(x) : gelu_bf16(x);   // bf16 output: the cheaper fit is far below the rounding
  if (ACT == 9) return gelu_fma_only(x);   // experiment variants (tools/gemm_trace.cu only)
  if (ACT == 10) {
    float y = x;
#pragma unroll
    for (int i = 0; i < 8; ++i) y = fmaf(y, 0.999f, 0.001f);
    return y;
  }
  if (ACT == LLB_ACT_SILU) return silu(x);
  if (ACT == LLB_ACT_SOFTSIGN) return softsign(x);
  return x;
}

// C = act(acc + bias) -> bf16 or fp32 row-major.
template <int ACT, bool F32>
struct EpiBiasAct {
  static constexpr int CHUNK = 32;
  static constexpr bool OUT_F32 = F32;
  void* C;
  int ldc;
  const float* bias;  // may be null
  __device__ __forceinline__ void transform(int row, int col0, float* v, int M, int N) const {
    if (bias != nullptr) {
      if (col0 + 32 <= N) {
#pragma unroll
        for (int i = 0; i < 32; i += 4) {
          const float4 b = __ldg(reinterpret_cast<const float4*>(bias + col0 + i));
          v[i] += b.x, v[i + 1] += b.y, v[i + 2] += b.z, v[i + 3] += b.w;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 32; ++i) v[i] += (col0 + i < N) ? __ldg(bias + col0 + i) : 0.0f;
      }
    }
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = apply_act<ACT, F32>(v[i]);
  }
};

// Generic runtime-dispatched GEMM used by the small / non-critical linears.
int gemm_bias_act(const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int M, int N,
                  int K, int act, bool out_f32, cudaStream_t stream, LaunchCounter* ctr = nullptr, GemmGroups grp = GemmGroups());

}  // namespace llb
