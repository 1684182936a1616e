// Fused   x += gate[g] * ( LN(A . W^T + bias) * (1 + scale[g]) + shift[g] )   ->  x (fp32, in place) and xb (bf16)
//
// This is the tail of both halves of a GraphDiT block (transformer.py:143-144: attention projection and MLP fc2, each
// followed by a non-affine LayerNorm, the adaLN modulation, the gate and the residual add).  Unfused, the GEMM writes
// y (bf16) and a row kernel re-reads it together with x: 14 bytes per element of HBM traffic and a memory-bound
// kernel between two GEMMs.  Here the LayerNorm runs on the fp32 accumulators in TMEM: 10 bytes per element, all of
// it overlapped with the next tile's MMAs.
//
// A full output row (N = H columns) has to be visible to normalise it, and 1024 fp32 accumulator columns are twice one SM's
// tensor memory, so a row is shared: FOUR independent CTA pairs (cta_group::2) form a group that owns a 256-row block, CTA
// (slice s, rank r) holds rows [128 r, +128) x columns [256 s, +256).  The epilogue
//   pass 1  tcgen05.ld -> per-row sum / sum of squares over the CTA's 256 columns; the four CTAs of equal rank exchange them
//           through mailboxes in L2 (data and tag in the same atomic 8-byte halves: no fence, no counter);
//   pass 2  tcgen05.ld again (TMEM reads are cheap) -> normalise, modulate with the tile's (<= 4) modulation rows staged
//           in shared memory, gate -> residual chunk in and result out through TMA, in the thread = row layout.
// (A 4-CTA-cluster variant with the statistics in distributed shared memory existed in round 1; it lost to this kernel at every
// shape the sampler uses and was removed.)
#pragma once
#include "llb_gemm.cuh"

namespace llb {

constexpr int GLN_BN = 256;
constexpr int GLN_PAIR_MAX_GROUPS = 18;   // 4-pair groups of the CTA-pair variant (72 of the B200's 74 pairs)
constexpr int GLN_MAX_GROUPS = 4;   // modulation rows staged per tile (a 128-row tile of 50-atom molecules touches <= 4)

struct GemmLnArgs {
  const float* bias;            // (N) or null
  const int32_t* row_group;     // (M) modulation row of each token row, non-decreasing runs
  const float* shift;           // modulation vectors: v[g * mod_ld + col]
  const float* scale;
  const float* gate;
  int mod_ld;
  float* x;                     // (M, ldx) fp32 residual stream, updated in place
  int ldx;
  __nv_bfloat16* xb;            // (M, ldxb) bf16 copy of the new x
  int ldxb;
};

// Fused GEMM + LayerNorm tails exist for N = 1024 (four CTA pairs per 256-row block, GraphDiT) and N = 768 (three, GIN):
// a full output row has to fit the pairs' tensor memory.  Other widths use GEMM + row kernel.
inline bool gemm_ln_supported(int N, int K) { return N == 4 * GLN_BN && K % 8 == 0; }
bool gemm_ln_enabled();   // LLB_FUSED_LN=0 selects GEMM + row kernel for the GraphDiT block tails (A-B comparison, pinned multi-GPU tests)

// Tail of a GIN layer fused into the second linear of the node MLP (graph_encoder/model.py:131-149, graph_predictor/model.py:318-348):
//   h[r,:] = gate_g * act( LN(A[r,:] . W^T + bias) * s1 + sh ) + h[r,:] + addvec_g      g = row_group[r] (graph of node r)
// with (s1, sh) = (gamma, beta) per column (encoder: affine LayerNorm) or (1 + scale_g, shift_g) per graph (predictor: text-adaLN);
// gate / addvec optional.  h (fp32, in place) and hb (its bf16 copy) are written through TMA; optionally the per-graph column
// MAXIMUM of the new h is accumulated into pool_max (order-preserving uint encoding, atomicMax: order-independent, hence
// deterministic) -- the next layer's virtual-node update pools exactly this matrix (model.py:148).
struct GinTailArgs {
  const float* bias;          // (N)
  const int32_t* row_group;   // (M) graph id per node row, non-decreasing
  const float* gamma;         // (N) or null
  const float* beta;          // (N) or null
  const float* shift;         // (graphs, mod_ld) or null
  const float* scale;
  const float* gate;
  int mod_ld;
  const float* addvec;        // (graphs, addvec_ld) or null
  int addvec_ld;
  int act;                    // LLB_ACT_NONE or LLB_ACT_GELU
  float* x;                   // (M, ldx) fp32 node features, updated in place
  int ldx;
  __nv_bfloat16* xb;          // (M, ldxb)
  int ldxb;
  uint32_t* pool_max;         // (graphs, pool_ld) encoded running maxima (cleared to 0 by the caller) or null
  int pool_ld;
  int a_f16;                  // A and W are IEEE fp16 instead of bf16
};
// N = 768 (three CTA pairs per 256-row block) or 1024 (four); needs the same exchange workspace as launch_gemm_ln_pair.
inline bool gin_tail_supported(int N, int K) { return (N == 3 * GLN_BN || N == 4 * GLN_BN) && K % 8 == 0; }
int launch_gin_tail(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const GinTailArgs& t, void* sync_ws, size_t sync_bytes,
                    cudaStream_t stream, LaunchCounter* ctr);
// order-preserving encoding of a float for unsigned atomicMax (0 = below every float)
__host__ __device__ inline uint32_t float_order_enc(uint32_t bits) { return (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u); }
__host__ __device__ inline uint32_t float_order_dec(uint32_t e) { return (e & 0x80000000u) ? (e & 0x7fffffffu) : ~e; }

// CTA-pair variant for N = 1024 (see llb_gemm_ln.cu): needs a caller-provided exchange workspace (any contents; the launch
// clears its counters with a stream-ordered memset) that no other launch uses concurrently.
size_t gemm_ln_pair_workspace_bytes();
int launch_gemm_ln_pair(const void* A, int lda, const void* W, int ldw, int M, int N, int K, const GemmLnArgs& e, void* sync_ws,
                        size_t sync_bytes, cudaStream_t stream, LaunchCounter* ctr);

}  // namespace llb
