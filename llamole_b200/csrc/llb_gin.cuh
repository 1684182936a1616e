// State shared by the GIN forward (llb_gin.cu) and the predictor's backward with respect to the text condition
// (llb_gin_grad.cu): the packed-weight layout, the handle, and the buffers a saved forward leaves for its backward.
#pragma once
#include <vector>

#include "llb_gemm.cuh"

namespace llb {

// Widths.  H is the model's hidden size, any H >= 1.  Every H-wide operand and activation is stored with Hp = round_up(H, 64)
// columns and every 4H-wide one with I = round_up(4H, 64); the padding of the parameters is zero, so the padded columns of every
// activation stay exactly 0 through embeddings, GEMMs, biases, GELU (gelu(0) = 0), residuals, pooling and the virtual node.  The
// only code that must know the true width is the LayerNorm statistics (divide by H / 4H) and the predictor's non-affine
// LayerNorm, which would otherwise write -mean * rstd into the padded columns (row LayerNorms get `valid` = the true width).
// When H % 64 == 0, Hp == H and I == 4H.  Below, "(4H,H)" etc. name the true shape and the stored shape is (I,Hp).
struct GinLayout {
  int H, Hp, I, L, predictor, out_dim, tdim;
  int HH, HHt, HO;   // head: hidden width (padded, true), output width (padded: Hp for the encoder, out_dim for the predictor)
  std::vector<size_t> mlp0_w, mlp4_w, vn0_w, vn4_w, adapter_w;   // bf16
  std::vector<size_t> mlp_chol;                                    // bf16 (H,H): Cholesky factor of the node MLP's first linear (analytic LayerNorm)
  std::vector<size_t> mlp_stat;                                    // fp32 [r (Hp, 0 past H) | c0 at Hp, 0, 0, 0]: bias column and constant of that factor
  std::vector<size_t> mlp_bg;                                      // fp32 (4H): centred bias x LayerNorm gamma
  size_t chol_scratch;                                             // fp64 (H+1, H+1) Gram matrix (true H), pack time only
  size_t head0_w, head4_w;
  size_t pilot_w, pilot_b;     // (pilot_cols, HH) bf16 / (pilot_cols) fp32: every pilot_stride-th template of the head (fused top-k)
  int pilot_cols, pilot_stride;
  size_t atom_emb, vn_emb, text_drop;                             // fp32
  std::vector<size_t> eps, mlp0_b, mlp_ln_w, mlp_ln_b, mlp4_b, bond_emb, norm_w, norm_b;
  std::vector<size_t> vn0_b, vn_ln_w, vn_ln_b, vn4_b, adapter_b;
  size_t head0_b, head_ln_w, head_ln_b, head4_b;
  size_t total;
};

int make_layout(const llb_gin_config& c, GinLayout& G);

// What llb_gin_predictor_forward_saved keeps for llb_gin_predictor_backward_c, carved from the caller's `saved` buffer.  The
// first group is written by the forward; the rest is scratch of the backward.  The batch bookkeeping is copied too, so that a
// later llb_gin_bind on the same handle cannot change the gradient of an earlier forward.
struct GinSaved {
  // written by the forward
  int32_t *graph_ptr, *batch32;          // (B+1), (n)
  int32_t *srowptr, *sdst, *seid;        // SOURCE-sorted CSR: out-edges of every node, ordered by edge id (n+1), (e), (e)
  float* hin;                            // (L-1, n, Hp) fp32: the input h_in_l of layers 1..L-1
  __nv_bfloat16* agg;                    // (L, n, Hp): the node MLP's input of every layer
  __nv_bfloat16* pool;                   // (L-1, B, Hp): max-pooled rows that feed the virtual-node MLPs
  float* mod;                            // (L, B, 3Hp): [shift | scale | gate] of every layer
  __nv_bfloat16* pooled_b;               // (B, Hp): the head's input
  // backward scratch
  int head_split;                        // K slices of the head's transposed product (see head_grad_split)
  __nv_bfloat16* dlog_b;                 // (B, Kp) bf16 copy of dlogits, zero past out_dim
  float* dhz_parts;                      // (B, head_split x HH) split-K partial products
  __nv_bfloat16 *hz_pre, *dhz_pre;       // (B, HH) head pre-LayerNorm row and its gradient
  float* dpooled;                        // (B, Hp)
  float* dh;                             // (n, Hp) gradient of the current layer's node rows
  float *dvn, *dpool;                    // (B, Hp)
  __nv_bfloat16* dvn_b;                  // (B, Hp)
  __nv_bfloat16 *vz, *dvz_b;             // (B, I) virtual-node MLP pre-LayerNorm row and its gradient
  float* dvz;                            // (B, I)
  __nv_bfloat16* z;                      // (n, I) recomputed node MLP intermediate (fp16 bits)
  float* u;                              // (n, Hp) recomputed node MLP output
  float* ln_part;                        // (n, ln_slots) analytic LayerNorm partial sums of the recomputation
  float* zpre;                           // (n, I) node MLP pre-LayerNorm row (centred first linear)
  float* dz;                             // (n, I)
  __nv_bfloat16* dzpre_b;                // (n, I)
  float* prod;                           // (n, 3Hp) per-node products of the modulation gradients
  __nv_bfloat16* du_b;                   // (n, Hp)
  float* da;                             // (n, Hp)
  __nv_bfloat16* dmod_b;                 // (B, L x 3Hp) all layers' modulation gradients side by side
  float* dctext;                         // (B, text_dim)
};
// Carves `saved` (nullptr: sizing only) for a batch of n nodes, e edges, B graphs; *bytes receives the size.
void gin_saved_carve(const GinLayout& G, void* saved, int n, int e, int B, GinSaved* sv, size_t* bytes);
// Padded K of the head's transposed product: out_dim rounded up so that every split of head_grad_split divides it into
// multiples of 64.
int head_grad_kp(const GinLayout& G);
int head_grad_split(const GinLayout& G, int B);

}  // namespace llb

struct llb_gin {
  llb_gin_config cfg;
  llb::GinLayout G;
  const uint8_t* blob = nullptr;
  llb::GemmCounters ctr;
  int64_t launches = 0;
  int n = 0, e = 0, B = 0;
  bool want_logits = false;
  int32_t *x32 = nullptr, *batch32 = nullptr, *graph_ptr = nullptr, *rowptr = nullptr, *col = nullptr, *eid = nullptr;
  int32_t *deg = nullptr, *blk = nullptr, *blk2 = nullptr;
  int32_t* flags = nullptr;   // input-defect bits of the bound batch (LLB_GIN_BAD_*)
  float* h = nullptr;
  __nv_bfloat16* hb = nullptr;
  __nv_bfloat16* agg = nullptr;
  __nv_bfloat16* z = nullptr;
  float* u = nullptr;
  float* ln_part = nullptr;   // (n, ln_slots) partial |zc|^2 sums of the node MLP (analytic LayerNorm)
  int ln_slots = 0;
  std::vector<float> chol_c0;   // per layer: constant of the Cholesky factor (host copy)
  float *vn_cur = nullptr, *vn_next = nullptr, *vu = nullptr;
  __nv_bfloat16 *pool_b = nullptr, *vz = nullptr;
  float* mod = nullptr;
  __nv_bfloat16* ctext = nullptr;
  float* pooled = nullptr;
  __nv_bfloat16* pooled_b = nullptr;
  __nv_bfloat16* hz = nullptr;
  float* head_out = nullptr;
  float* logits_ws = nullptr;
  int32_t* topk_redo = nullptr;   // per row of a logits chunk: redo with the selection-pass kernel
  // fused head + top-k
  float* pilot_logits = nullptr;   // (fused rows, HEAD_PILOT_COLS)
  float2* rowtau = nullptr;        // (fused rows)
  float* head_part = nullptr;      // (fused rows, head_slots)
  int head_slots = 0, fused_rows = 0;
  float2* head_cand = nullptr;     // (fused rows, HEAD_CAND_CAP)
  int32_t *head_cnt = nullptr, *head_flagged = nullptr, *head_nflag = nullptr;
  __nv_bfloat16* redo_in = nullptr;   // (chunk_rows, HH) gathered head inputs of flagged rows
  float* redo_v = nullptr;
  int32_t* redo_i = nullptr;
  int max_k = 0;
  int64_t head_flagged_rows = 0, head_fused_rows = 0;   // statistics of the last llb_gin_predictor_topk call
  uint32_t* pool_enc = nullptr;   // (B,H) per-graph maxima from the fused layer tail (encoded)
  void* tail_sync = nullptr;      // statistics-exchange workspace of the fused layer tail
  int chunk_rows = 0;
  template <class T>
  const T* w(size_t off) const { return reinterpret_cast<const T*>(blob + off); }
};

namespace llb {
// Node MLP of layer l with analytic LayerNorm statistics (see EpiRowSq in llb_gin.cu): statistics GEMM -> first linear with
// LayerNorm + GELU in its epilogue -> zbuf (rows, I) fp16 -> second linear -> u (rows, Hp) fp32 unless first_half_only.
int gin_node_mlp(llb_gin* g, const __nv_bfloat16* in, int rows, int l, float* ln_part, __nv_bfloat16* zbuf, float* u, int u_ld,
                 bool first_half_only, int slot0, int slot4, cudaStream_t s);
}  // namespace llb
