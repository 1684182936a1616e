// State shared by the GraphDiT sampler (llb_dit.cu) and the backward of its denoiser with respect to the condition vector
// (llb_dit_grad.cu): the packed-weight layout, the handle, and the buffers a saved forward leaves for its backward.
#pragma once
#include <vector>

#include "llb_dit_kernels.cuh"
#include "llb_gemm.cuh"

namespace llb {

struct DitLayout {
  int H, D, heads, F, N, T, ydim, tdim, d0, K0, KC;
  // bf16 matrices (byte offsets)
  size_t x_embed_w, cond_w, ada0_w, out_fc1_w, out_fc2_w, out_ada2_w;
  std::vector<size_t> qkv_w, proj_w, fc1_w, fc2_w, ada2_w;
  // fp32 vectors
  size_t x_ln_w, x_ln_b, ada0_b, out_fc1_b, out_fc2_b, out_ada2_b;
  std::vector<size_t> qn_w, qn_b, kn_w, kn_b, proj_b, fc1_b, fc2_b, ada2_b;
  size_t y_mlp0_w, y_mlp0_b, y_drop, txt_drop, txt_b;   // (ydim,H) x3, (H), (H)
  size_t c1_table;   // (T+1, H): timestep embedding for t = 0..T
  size_t c_unc;      // (H): sum of the drop embeddings
  size_t tables;     // x_marg(16) e_marg(5) xe(80) ex(80)
  size_t betas, abar;  // (T+1) each
  size_t setup_scratch;  // (T+1, 256 + H) fp32, used by pack_weights only
  size_t total;
};

int make_layout(const llb_dit_config& c, DitLayout& L);
// The backward of the denoiser (and the saved forward that feeds it) is built for at most DIT_GRAD_MAXN atoms per molecule.
int dit_grad_check_n(const DitLayout& L, const char* entry);

// What llb_dit_denoise_c keeps for llb_dit_backward_c, carved from the caller's `saved` buffer (dit_saved_carve).  The first
// group is written by the forward; the rest is scratch of the backward.  The batch bookkeeping is copied too, so that a later
// call on the same handle cannot change the gradient of an earlier forward.
struct DitSaved {
  // written by the forward
  int32_t *mol_off, *row_mol;            // (B+1), (Mtok)
  __nv_bfloat16* cvec;                   // (B, H): the condition as the adaLN GEMM read it
  float* xs;                             // (2D+1, Mtok, H): the residual stream after the embedding and after every block half
  float* mod;                            // (B, D 6H): softsign outputs [sh_a | sc_a | g_a | sh_m | sc_m | g_m] of every block
  float* modout;                         // (B, 2 d0): [shift | scale] of the output layer
  // backward scratch
  int split;                             // K slices of the condition product (dit_grad_split)
  __nv_bfloat16 *xb, *qkv, *attn, *hb;   // (Mtok, H), (Mtok, 3H), (Mtok, H), (Mtok, F): recomputed forward operands
  float *qkv_raw, *y, *pre, *raw;        // (Mtok, 3H) pre-LayerNorm q/k/v, (Mtok, H), (Mtok, F), (Mtok, d0 padded to 4)
  float *dx, *tmp;                       // (Mtok, H) gradient of the residual stream, (Mtok, F) scratch
  __nv_bfloat16* db;                     // (Mtok, max(F, 3H, K0o)) bf16 gradient operand of the next transposed product
  __nv_bfloat16* dvec;                   // (Mtok, H) bf16 gradient operand
  float* prod;                           // (Mtok, 3H) row products of the LayerNorm backward
  float *dmod, *dmodout;                 // (B, D 6H), (B, 2 d0)
  __nv_bfloat16 *dz_b, *dmodout_b;       // (B, D 6H), (B, KO)
  float *dhid, *pre0;                    // (B, (D+1) H): gradient and pre-activation of the stacked adaLN.0 outputs
  __nv_bfloat16* dpre_b;                 // (B, KA)
  float* dc_parts;                       // (B, split H)
};

// Widths of the backward's padded operands: K0o = d0 and KO = 2 d0 rounded up to 64 (the out-layer products), KA = (D+1) H
// rounded up so that every split-K slice of the condition product is a multiple of 64.
int dit_grad_k0o(const DitLayout& L);
int dit_grad_ko(const DitLayout& L);
int dit_grad_ka(const DitLayout& L);
int dit_grad_split(const DitLayout& L, int B);
// sv == nullptr: only the size
void dit_saved_carve(const DitLayout& L, void* saved, int B, int Mtok, DitSaved* sv, size_t* bytes);

}  // namespace llb

struct llb_dit {
  llb_dit_config cfg;
  llb::DitLayout L;
  const uint8_t* blob = nullptr;
  std::vector<float> betas, abar;   // host copies of the schedule
  llb::DitTablesDev tables;
  llb::LaunchCounter ctr;
  // batch binding
  int B = 0, Mtok = 0, passes = 2;
  int max_n = 0;                 // atoms of the batch's largest molecule: picks the attention tile
  int64_t mol_base = 0;
  // workspace carve-up
  float* x = nullptr;            // (M,H) residual stream fp32
  __nv_bfloat16* xb = nullptr;   // (M,H) bf16 copy (GEMM A operand)
  __nv_bfloat16* y = nullptr;    // (M,H)
  __nv_bfloat16* qkv = nullptr;  // (M,3H)
  __nv_bfloat16* attn = nullptr; // (M,H)
  __nv_bfloat16* hbuf = nullptr; // (M,F)  (also fp32 scratch (Mtok,H) for the token embedding)
  __nv_bfloat16* tok = nullptr;  // (Mtok,K0)
  float* raw = nullptr;          // (M, raw_ld)
  int raw_ld = 0;
  __nv_bfloat16* cvec = nullptr; // (B+1,H)
  __nv_bfloat16* hid = nullptr;  // (B+1,(D+1)H)
  float* mod = nullptr;          // (D, B+1, 6H)
  float* modout = nullptr;       // (B+1, 2 d0)
  float* part = nullptr;         // (min(2M, 640), SPLITK, H) split-K partial products of fc2
  float* cinv = nullptr;         // (B,H)
  __nv_bfloat16* acond = nullptr;  // (B,KC)
  uint8_t* missing = nullptr;    // (B, ydim+1)
  int8_t* stX = nullptr;         // (B,N)
  int8_t* stE = nullptr;         // (B,N,N)
  int32_t* mol_off = nullptr;    // (B+1)
  int32_t* row_mol = nullptr;    // (Mtok)
  int32_t* row_group = nullptr;  // (M): modulation row of each token row
  void* ln_sync = nullptr;       // statistics-exchange workspace of the CTA-pair GEMM + LayerNorm kernel
  float* save_x = nullptr;       // set by a saved pass only: (2D+1, M, H), the residual stream after the embedding and every block half
  // Latency regime: everything of a denoiser pass that does not depend on t (all but the conditioning-vector kernel) is captured
  // once per batch binding and replayed as ONE CUDA graph launch; the programmatic-dependent-launch edges are kept by the capture.
  cudaGraphExec_t body_graph = nullptr;
  cudaStream_t capture_stream = nullptr;
  int graph_state = 0;           // 0 not built, 1 ready, -1 capture / instantiation failed for this binding (eager launches)
  int passes_run = 0;            // denoiser passes since llb_dit_begin (the first one runs eagerly: lazy one-time set-up is not capturable)
  int64_t graph_launches = 0;    // kernel launches one replay stands for
  int64_t graph_kern[LLB_KERN_FAMILIES] = {};
  void drop_graph() {
    if (body_graph) cudaGraphExecDestroy(body_graph);
    body_graph = nullptr, graph_state = 0, passes_run = 0;
  }
  ~llb_dit() {
    drop_graph();
    if (capture_stream) cudaStreamDestroy(capture_stream);
  }
  template <class T>
  const T* w(size_t off) const { return reinterpret_cast<const T*>(blob + off); }
};

