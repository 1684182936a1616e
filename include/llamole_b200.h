/*
 * llamole_b200 -- C ABI of the B200-native (sm_100a) graph-module hot path of Llamole.
 *
 * The reference (liugangcode/Llamole) is pure Python and has no FFI layer of its own; its boundary for this
 * path is the three nn.Module classes under src/model (SURVEY.md section 8b).  This header is the boundary
 * between those classes (re-hosted in llamole_b200/graph_{decoder,encoder,predictor}.py, bound with ctypes)
 * and the hand-written CUDA.  Each entry names the reference code it replaces (paths relative to
 * /root/reference/src/model).
 *
 * Conventions
 *   - plain pointers and sizes only; `*_dev` / unmarked pointers are device memory, `*_host` are host memory;
 *   - every call is asynchronous on `stream`, never synchronises the device and allocates nothing the caller
 *     can see: weights are packed into a caller-allocated blob, scratch comes from a caller-allocated
 *     workspace (sizes from the *_bytes functions);
 *   - return value: LLB_OK or a negative status; llb_last_error() gives the message of the calling thread's
 *     last failure;
 *   - sm_100 (B200) only.  There is no fallback path: other devices get LLB_ERR_ARCH.
 */
#ifndef LLAMOLE_B200_H
#define LLAMOLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* llb_stream_t; /* == cudaStream_t */

enum {
  LLB_OK = 0,
  LLB_ERR_INVALID = -1,   /* bad argument / unsupported shape */
  LLB_ERR_ARCH = -2,      /* not an sm_100 device */
  LLB_ERR_CUDA = -3,      /* CUDA runtime / driver error */
  LLB_ERR_WORKSPACE = -4  /* workspace or blob too small */
};

enum { LLB_ACT_NONE = 0, LLB_ACT_GELU = 1, LLB_ACT_SILU = 2, LLB_ACT_SOFTSIGN = 3 };

const char* llb_last_error(void);
int llb_version(void);
/* Refuses anything but compute capability 10.x (no fallback by design). */
int llb_arch_check(int device);

/* ------------------------------------------------------------------------------------------------------
 * Live kernel timing (bench.py's roofline): when enabled, every kernel launch of the library is bracketed by
 * CUDA events on the launching stream and accumulated per slot.  llb_profile_read synchronises on the recorded
 * events, returns the slot's total device time and launch count since the last reset, and clears it.
 * ---------------------------------------------------------------------------------------------------- */
enum {
  LLB_PROF_GEMM_QKV = 0, LLB_PROF_GEMM_PROJ, LLB_PROF_GEMM_FC1, LLB_PROF_GEMM_FC2, LLB_PROF_GEMM_ADALN,
  LLB_PROF_GEMM_OTHER, LLB_PROF_ATTENTION, LLB_PROF_LN_MOD_RES, LLB_PROF_DIT_STEP, LLB_PROF_DIT_MISC,
  LLB_PROF_GIN_AGGREGATE, LLB_PROF_GIN_POOL, LLB_PROF_GIN_GEMM_MLP0, LLB_PROF_GIN_GEMM_MLP4, LLB_PROF_GIN_ROWLN,
  LLB_PROF_GIN_MISC, LLB_PROF_GIN_GEMM_HEAD, LLB_PROF_GIN_TOPK, LLB_PROF_GIN_GEMM_STATS, LLB_PROF_SLOTS
};
int llb_profile_enable(int on);
int llb_profile_read(int slot, double* total_ms, int64_t* launches);
const char* llb_profile_slot_name(int slot);
/* Launch counters per kernel FAMILY since the library was loaded (process-wide).  The parity tests use them to assert that
 * a shape really reached the kernel it is meant to cover (e.g. the CTA-pair GEMM, which only runs on wide problems). */
enum {
  LLB_KERN_GEMM_1CTA = 0,    /* gemm_tcgen05_kernel */
  LLB_KERN_GEMM_2CTA,        /* gemm_tcgen05_2cta_kernel (cta_group::2) */
  LLB_KERN_GEMM_LN_PAIR,     /* gemm_ln_pair_kernel<..., GIN = 0>: GraphDiT block tail (GEMM + LayerNorm + modulation + residual) */
  LLB_KERN_GEMM_LN_CLUSTER,  /* retired in round 2 (the thread-block-cluster variant of the above); always 0, slot kept for ABI stability */
  LLB_KERN_GIN_FUSED_MLP,    /* gemm_ln_pair_kernel<..., GIN = 1>: second GIN linear + LayerNorm + layer tail + max-pooling */
  LLB_KERN_HEAD_TOPK,        /* gemm_tcgen05_2cta_kernel<EpiHeadTopk>: predictor head GEMM + softmax partial sums + top-k candidates */
  LLB_KERN_FAMILIES
};
int64_t llb_kernel_launches(int family);

/* ------------------------------------------------------------------------------------------------------
 * tcgen05 GEMM building block:  C[M,N] = act(A[M,K] . W[N,K]^T + bias[N])
 * A, W: bf16 row-major (K contiguous; lda, ldw in elements, multiples of 8); C: bf16 or fp32 row-major.
 * Replaces every nn.Linear on the path (cuBLAS in the reference): graph_decoder/layers.py:47,52,108-111,
 * transformer.py:41-44,125-130,158-162; graph_encoder/model.py:111,163,191-195; graph_predictor/model.py:258-263.
 * ---------------------------------------------------------------------------------------------------- */
int llb_gemm_bf16(const void* A, int lda, const void* W, int ldw, const float* bias, void* C, int ldc, int M,
                  int N, int K, int act, int out_fp32, llb_stream_t stream);

/* Fused tail of a GraphDiT block half (transformer.py:143-144):
 *   x[r,:] += gate[g] * ( LayerNorm(A[r,:] . W^T + bias) * (1 + scale[g]) + shift[g] ),  g = row_group[r]
 * LayerNorm over the N = 1024 output columns (eps 1e-5, no affine) on the fp32 accumulators; x (M, ldx) fp32 is updated in
 * place and xb (M, ldxb) receives its bf16 copy (the next GEMM's operand; must not alias A).  shift / scale / gate point at
 * (groups, mod_ld) fp32 matrices.  Runs on CTA pairs (tcgen05.mma.cta_group::2): four pairs share a 256-row block and exchange
 * the LayerNorm statistics through `workspace` (llb_gemm_ln_workspace_bytes bytes, 128-byte aligned, owned by the caller, not
 * shared with a concurrent launch).  Other widths return LLB_ERR_INVALID (the sampler then uses GEMM + row kernel). */
int llb_gemm_ln_workspace_bytes(size_t* bytes);
int llb_gemm_ln_residual_ws(const void* A, int lda, const void* W, int ldw, const float* bias, const int32_t* row_group,
                            const float* shift, const float* scale, const float* gate, int mod_ld, float* x, int ldx,
                            void* xb, int ldxb, int M, int N, int K, void* workspace, size_t workspace_bytes,
                            llb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * GraphDiT sampler  (graph_decoder/diffusion_model.py:252-399, transformer.py:93-187, layers.py:56-116,
 * conditions.py:19-123, diffusion_utils.py:93-108,316-349,376-413,476-518)
 * ---------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t hidden;      /* H, multiple of 64 */
  int32_t depth;       /* transformer blocks */
  int32_t heads;       /* H / heads must be 64 */
  int32_t mlp_hidden;  /* int(H * mlp_ratio), multiple of 64 */
  int32_t max_nodes;   /* N <= 128 for sampling, <= 64 for the training entries below; joint token width d0 = 16 + 5 N */
  int32_t timesteps;   /* T */
  int32_t y_dim;       /* 10 */
  int32_t text_dim;    /* 768 */
  float guide_scale;   /* classifier-free guidance scale; 1 disables the unconditional pass */
} llb_dit_config;

/* fp32 device pointers in the reference's state_dict layout (SURVEY.md section 8b), row-major (out, in). */
typedef struct {
  const float* x_embed_w;                  /* x_embedder.0.weight (H, d0) */
  const float *x_embed_ln_w, *x_embed_ln_b; /* x_embedder.1 */
  const float *t_mlp0_w, *t_mlp0_b;        /* t_embedder.mlp.0 (H,256) */
  const float *t_mlp2_w, *t_mlp2_b;        /* t_embedder.mlp.2 (H,H) */
  const float* y_drop;                     /* y_embedder.embedding_drop.weight (y_dim, H) */
  const float* const* y_mlp0_w;            /* [y_dim] (H,1) */
  const float* const* y_mlp0_b;            /* [y_dim] (H) */
  const float* const* y_mlp2_w;            /* [y_dim] (H,H), no bias */
  const float* txt_drop;                   /* txt_embedder.embedding_drop.weight (1,H) */
  const float *txt_w, *txt_b;              /* txt_embedder.linear (H, text_dim) */
  /* per block, arrays of `depth` device pointers */
  const float* const* qkv_w;               /* (3H,H) rows [q|k|v], head-major */
  const float* const* q_norm_w;
  const float* const* q_norm_b;            /* (64) */
  const float* const* k_norm_w;
  const float* const* k_norm_b;
  const float* const* proj_w;
  const float* const* proj_b;              /* (H,H),(H) */
  const float* const* fc1_w;
  const float* const* fc1_b;               /* (F,H),(F) */
  const float* const* fc2_w;
  const float* const* fc2_b;               /* (H,F),(H) */
  const float* const* ada0_w;
  const float* const* ada0_b;              /* adaLN_modulation.0 (H,H) */
  const float* const* ada2_w;
  const float* const* ada2_b;              /* adaLN_modulation.2 (6H,H) */
  /* output layer */
  const float *out_fc1_w, *out_fc1_b;      /* (H,H) */
  const float *out_fc2_w, *out_fc2_b;      /* (d0,H) */
  const float *out_ada0_w, *out_ada0_b;    /* (H,H) */
  const float *out_ada2_w, *out_ada2_b;    /* (2 d0,H) */
  /* diffusion tables (diffusion_model.py:78-93, diffusion_utils.py:172-185) */
  const float* x_marg;                     /* (16) */
  const float* e_marg;                     /* (5) */
  const float* xe;                         /* (16,5) */
  const float* ex;                         /* (5,16) */
  const float* betas;                      /* (T+1) */
  const float* alphas_bar;                 /* (T+1) */
} llb_dit_weights;

typedef struct llb_dit llb_dit;

/* Size of the packed (bf16 GEMM operands + fp32 vectors + pre-computed tables) weight blob. */
int llb_dit_packed_bytes(const llb_dit_config* cfg, size_t* bytes);
/* Converts/packs the checkpoint and pre-computes the step-invariant tables (timestep embeddings for
 * t = 0..T, unconditional drop vector).  Replaces GraphDiT.init_model's placement of the denoiser
 * (diffusion_model.py:105-110; loader.py:245-247). */
int llb_dit_pack_weights(const llb_dit_config* cfg, const llb_dit_weights* w, void* packed, size_t packed_bytes,
                         llb_stream_t stream);
int llb_dit_create(const llb_dit_config* cfg, const void* packed, size_t packed_bytes, llb_dit** out);
void llb_dit_destroy(llb_dit* h);
int llb_dit_workspace_bytes(const llb_dit_config* cfg, int max_molecules, size_t* bytes);

/* Binds a batch: node counts (HOST array, the reference draws them on the host too,
 * diffusion_utils.py:160-162), conditions on the device (props: NaN = missing property,
 * diffusion_model.py:259; txt: a row containing NaN = missing text).  Computes the step-invariant part of
 * the conditioning vector (conditions.py:76-98,108-123).  `mol_index_base` is the global index of molecule 0
 * (keys the counter RNG so that results do not depend on how a batch is sharded over GPUs). */
int llb_dit_begin(llb_dit* h, void* workspace, size_t workspace_bytes, int B, const int32_t* n_nodes_host,
                  const float* props, const float* txt, int64_t mol_index_base, llb_stream_t stream);

/* State: X (B,N) int8 atom class or -1 (masked); E (B,N,N) int8 bond class, -1 = all-zero vector
 * (masked pair, or the diagonal of z_T; diffusion_utils.py:509-518). */
int llb_dit_set_state(llb_dit* h, const int8_t* X, const int8_t* E, llb_stream_t stream);
int llb_dit_get_state(llb_dit* h, int8_t* X, int8_t* E, llb_stream_t stream);
/* z_T ~ limit marginals (diffusion_utils.py:495-518).  qX0 (B,N,16) / qE0 (B,N,N,5): pre-drawn Exp(1) noise,
 * or NULL for the counter RNG keyed by `seed`. */
int llb_dit_init_state(llb_dit* h, uint64_t seed, const float* qX0, const float* qE0, llb_stream_t stream);

/* Parity entry: masked denoiser logits of the current state at integer time t (1..T).
 * == Transformer.forward(...).mask(node_mask) (transformer.py:93-108).  logits_X (B,N,16), logits_E (B,N,N,5). */
int llb_dit_denoise(llb_dit* h, int t, int unconditioned, float* logits_X, float* logits_E, llb_stream_t stream);

/* One reverse step t -> t-1 in place (sample_p_zs_given_zt, diffusion_model.py:309-399): conditional and
 * unconditional denoiser pass, closed-form posterior, guidance, categorical sampling.
 * qX (B,N,16), qE (B,N,N,5): pre-drawn Exp(1) noise for this step or NULL (counter RNG).
 * prob_X / prob_E: optional dumps of the guided probabilities (B,N,16) / (B,N,N,5) (only i<j pairs are written). */
int llb_dit_step(llb_dit* h, int t, uint64_t seed, const float* qX, const float* qE, float* prob_X, float* prob_E,
                 llb_stream_t stream);
/* The loop of GraphDiT.generate (diffusion_model.py:279-289) for t = t_first .. t_last (descending, inclusive).
 * qX_all (T,B,N,16) / qE_all (T,B,N,N,5) indexed by s = t-1, or NULL. */
int llb_dit_sample(llb_dit* h, int t_first, int t_last, uint64_t seed, const float* qX_all, const float* qE_all,
                   llb_stream_t stream);
/* Number of kernel launches issued by this handle so far (bench.py's gpu_launches). */
/* Backward of the denoiser with respect to its condition vector c = t_emb + y_emb + txt_emb (B,H) (the SFT loss of
 * GraphDiT.forward; the parameters are constants).  Uses a handle created with guide_scale == 1 (one pass, no unconditional
 * half), so a sampler's handle, workspace and captured graph are never touched.
 *   llb_dit_grad_packed_bytes / llb_dit_pack_grad_weights: a second, caller-owned blob of transposed bf16 copies of every
 *     weight the backward multiplies by (qkv, proj, fc1, fc2, adaLN.2 of every block, the D+1 adaLN.0 weights stacked along K,
 *     the output layer's fc1, fc2, adaLN.2), built on the device from the handle's packed blob (~1.1 GB at H = 1024, depth 28).
 *   llb_dit_train_saved_bytes / llb_dit_denoise_c: one denoiser pass over the int8 states X (B,N), E (B,N,N) of the molecules of
 *     n_nodes_host[b] atoms with the caller's fp32 c in place of the timestep table + conditions; writes the same masked dense
 *     logits as llb_dit_denoise (logits_X (B,N,16), logits_E (B,N,N,5), zero outside each molecule; a molecule of 0 atoms is not
 *     written).  t reaches the denoiser only through c: nothing indexes the schedule.  With `saved` (NULL: inference) it also
 *     keeps the residual stream at every block-half boundary, the modulations, c and the batch bookkeeping, so a later call on
 *     the handle cannot change this forward's gradient; the buffer also holds the backward's scratch (one per forward).
 *   llb_dit_backward_c: dlogits (same shapes, fp32) -> dc (B,H) fp32 for the forward that filled `saved` (pass that forward's
 *     B and atom total).  Run-to-run bit-identical.
 * These entries (and llb_dit_denoise_c with a `saved` buffer) need max_nodes <= 64; llb_dit_denoise_c without one takes
 * max_nodes up to 128, like the sampler. */
int llb_dit_grad_packed_bytes(const llb_dit_config* cfg, size_t* bytes);
int llb_dit_pack_grad_weights(llb_dit* h, void* grad_blob, size_t grad_bytes, llb_stream_t stream);
int llb_dit_train_saved_bytes(const llb_dit_config* cfg, int B, int num_tokens, size_t* bytes);
int llb_dit_denoise_c(llb_dit* h, void* workspace, size_t workspace_bytes, int B, const int32_t* n_nodes_host, const int8_t* X,
                      const int8_t* E, const float* c, float* logits_X, float* logits_E, void* saved, size_t saved_bytes,
                      llb_stream_t stream);
int llb_dit_backward_c(llb_dit* h, int B, int num_tokens, void* saved, size_t saved_bytes, const void* grad_blob, size_t grad_bytes,
                       const float* dlogits_X, const float* dlogits_E, float* dc, llb_stream_t stream);
/* Kernels this handle has issued since it was created, replayed graph nodes included (one replay counts every kernel it runs). */
int64_t llb_dit_launch_count(const llb_dit* h);
/* Small batches (fewer than 2048 token rows, e.g. the reference's per-prompt batches of 6, modeling_llamole.py:653): from the
 * second denoiser pass of a batch binding on, the t-independent launches of a pass are replayed as one CUDA graph (a launch
 * count still reports the kernels executed).  1 = the graph is in use, 0 = not built (large batch, first pass, profiling on,
 * LLB_GRAPH=0), -1 = capture or instantiation failed and the pass is issued launch by launch. */
int llb_dit_graph_state(const llb_dit* h);

/* Standalone fused posterior + guidance + sampling (K8-K10) from given dense masked logits; used by the
 * parity tests to check categories bit-exactly against the oracle on identical logits and noise. */
int llb_dit_posterior_sample(llb_dit* h, int t, const float* lc_X, const float* lc_E, const float* lu_X,
                             const float* lu_E, uint64_t seed, const float* qX, const float* qE, float* prob_X,
                             float* prob_E, llb_stream_t stream);

/* ------------------------------------------------------------------------------------------------------
 * GIN encoder / predictor  (graph_encoder/model.py:37-41,124-205; graph_predictor/model.py:306-353,387-391)
 * ---------------------------------------------------------------------------------------------------- */
typedef struct {
  int32_t hidden;      /* H >= 1, any value: stored zero-padded to a multiple of 64 (and 4H likewise), so a width that is not a
                          multiple of 64 costs the FLOPs and bytes of the padded one */
  int32_t layers;      /* L >= 2 */
  int32_t predictor;   /* 0 = GraphCLIP encoder, 1 = GNNRetrosynthsizer */
  int32_t out_dim;     /* predictor: template classes; encoder: ignored */
  int32_t text_dim;    /* predictor: 768 */
} llb_gin_config;

typedef struct {
  const float* atom_emb;                 /* (118,H) */
  const float* vn_emb;                   /* (1,H) */
  /* per layer arrays [L] */
  const float* const* eps;               /* (1) */
  const float* const* mlp0_w;
  const float* const* mlp0_b;            /* (4H,H) */
  const float* const* mlp_ln_w;
  const float* const* mlp_ln_b;          /* (4H) */
  const float* const* mlp4_w;
  const float* const* mlp4_b;            /* (H,4H) */
  const float* const* bond_emb;          /* (5,H) */
  const float* const* norm_w;            /* encoder: (H); predictor: NULL array */
  const float* const* norm_b;
  /* virtual-node MLPs, arrays [L-1] */
  const float* const* vn0_w;
  const float* const* vn0_b;
  const float* const* vn_ln_w;
  const float* const* vn_ln_b;
  const float* const* vn4_w;
  const float* const* vn4_b;
  /* predictor only */
  const float* const* adapter_w;         /* [L] (3H,text_dim) */
  const float* const* adapter_b;
  const float* text_dropping;            /* (1,text_dim) */
  /* head: encoder = ProjectionHead fc1/norm1/fc2 (H,H); predictor = decoder.0/.1/.4 */
  const float *head0_w, *head0_b;
  const float *head_ln_w, *head_ln_b;
  const float *head4_w, *head4_b;
} llb_gin_weights;

typedef struct llb_gin llb_gin;

int llb_gin_packed_bytes(const llb_gin_config* cfg, size_t* bytes);
int llb_gin_pack_weights(const llb_gin_config* cfg, const llb_gin_weights* w, void* packed, size_t packed_bytes,
                         llb_stream_t stream);
int llb_gin_create(const llb_gin_config* cfg, const void* packed, size_t packed_bytes, llb_gin** out);
void llb_gin_destroy(llb_gin* h);
int llb_gin_workspace_bytes(const llb_gin_config* cfg, int num_nodes, int num_edges, int num_graphs, int want_logits,
                            size_t* bytes);

/* Destination-sorted CSR of the directed edge list + per-graph node ranges (replaces PyG's
 * propagate/scatter bookkeeping, graph_encoder/model.py:169).  edge_index (2,E) int64, edge_attr (E) int64,
 * batch (n) int64 sorted ascending.  Results live in the workspace bound by llb_gin_bind. */
int llb_gin_bind(llb_gin* h, void* workspace, size_t workspace_bytes, int num_nodes, int num_edges, int num_graphs,
                 const int64_t* x, const int64_t* edge_index, const int64_t* edge_attr, const int64_t* batch,
                 llb_stream_t stream);
/* Input defects of the batch bound last, as a bit mask written to *flags_host (the one call of this header that SYNCHRONISES
 * the stream: it is how the Python classes raise the IndexError the reference raises for such inputs, graph_encoder/model.py:125,
 * :169).  The kernels themselves clamp / skip the offending entries and never index out of bounds. */
enum {
  LLB_GIN_BAD_ATOM_ID = 1,  /* x outside [0,118) */
  LLB_GIN_BAD_BATCH = 2,    /* batch not ascending or outside [0,num_graphs) */
  LLB_GIN_BAD_EDGE = 4,     /* edge endpoint outside [0,num_nodes) */
  LLB_GIN_BAD_BOND_ID = 8   /* edge_attr outside [0,5) */
};
int llb_gin_input_flags(llb_gin* h, int32_t* flags_host, llb_stream_t stream);
/* GraphCLIP.forward: unit-norm embeddings (B,H) fp32. */
int llb_gin_encoder_forward(llb_gin* h, float* out, float* pooled_or_null, llb_stream_t stream);
/* GNNRetrosynthsizer.forward: logits (B,out_dim) fp32.  c (B,text_dim) fp32 or NULL (= text_dropping row). */
int llb_gin_predictor_forward(llb_gin* h, const float* c, float* logits, llb_stream_t stream);
/* Device part of sample_templates (graph_predictor/model.py:176-179): softmax over out_dim + top-k, without
 * materialising the logits for the caller.  topk_prob (B,k) fp32, topk_idx (B,k) int32, sorted descending. */
int llb_gin_predictor_topk(llb_gin* h, const float* c, int k, float* topk_prob, int32_t* topk_idx,
                           llb_stream_t stream);
/* Backward of GNNRetrosynthsizer.forward with respect to c (the text condition; the parameters are constants).
 *   llb_gin_grad_packed_bytes / llb_gin_pack_grad_weights: a second, caller-owned blob of transposed bf16 copies of every
 *     weight the backward multiplies by, built on the device from the handle's packed blob (the predictor head's copy is
 *     out_dim x 4H: 1.1 GB at 180 576 templates and H = 768).  Only a caller that differentiates needs it.
 *   llb_gin_saved_bytes / llb_gin_predictor_forward_saved: llb_gin_predictor_forward (the same kernels: bit-identical logits)
 *     that also stores what the backward needs into the caller's `saved` buffer, including the batch bookkeeping, so a later
 *     llb_gin_bind on the same handle does not change the gradient.  The buffer also holds the backward's scratch: one buffer
 *     per forward whose gradient is wanted.
 *   llb_gin_predictor_backward_c: dlogits (B,out_dim) fp32 -> dc (B,text_dim) fp32, for the forward that filled `saved` (pass
 *     that forward's batch sizes).  c must be the forward's c; a NULL c is LLB_ERR_INVALID.  Run-to-run bit-identical.
 * The *_bytes entries reject encoder configs. */
int llb_gin_grad_packed_bytes(const llb_gin_config* cfg, size_t* bytes);
int llb_gin_pack_grad_weights(llb_gin* h, void* grad_blob, size_t grad_bytes, llb_stream_t stream);
int llb_gin_saved_bytes(const llb_gin_config* cfg, int num_nodes, int num_edges, int num_graphs, size_t* bytes);
int llb_gin_predictor_forward_saved(llb_gin* h, const float* c, float* logits, void* saved, size_t saved_bytes,
                                    llb_stream_t stream);
int llb_gin_predictor_backward_c(llb_gin* h, int num_nodes, int num_edges, int num_graphs, const float* c,
                                 const float* dlogits, void* saved, size_t saved_bytes, const void* grad_blob,
                                 size_t grad_bytes, float* dc, llb_stream_t stream);
/* Backward of GraphCLIP.forward with respect to every parameter of the encoder (GNNEncoder + ProjectionHead).
 *   llb_gin_encoder_saved_bytes / llb_gin_encoder_forward_saved: llb_gin_encoder_forward (the same kernels: bit-identical
 *     embeddings, fused layer tail included) that also stores what the backward needs into the caller's `saved` buffer: the
 *     batch bookkeeping and atom ids, every layer's input and aggregation, the virtual node's pooled rows, the read-out, the head's
 *     output before the L2 normalisation, and transposed bf16 copies of the weights the backward multiplies by (about 90 MB at
 *     H = 768, L = 5).  A later llb_gin_bind therefore does not change this forward's gradient.  The buffer also holds the
 *     backward's scratch: one buffer per forward whose gradient is wanted.
 *   llb_gin_encoder_backward: d_out (B,H) fp32 = dL/d(embeddings) -> the fp32 gradient of every parameter, written (not
 *     accumulated) at the parameter's true shape through `grads`, for the forward that filled `saved` (pass that forward's batch
 *     sizes).  Dropout is not applied (the forward never applies it).  Run-to-run bit-identical.
 * These entries reject predictor configs; llb_gin_grad_packed_bytes / llb_gin_saved_bytes reject encoder configs. */
typedef struct {
  float* atom_emb;                 /* (118,H) */
  float* vn_emb;                   /* (1,H) */
  /* per layer arrays [L] */
  float* const* eps;               /* (1) */
  float* const* mlp0_w;            /* (4H,H) */
  float* const* mlp0_b;            /* (4H) */
  float* const* mlp_ln_w;
  float* const* mlp_ln_b;          /* (4H) */
  float* const* mlp4_w;            /* (H,4H) */
  float* const* mlp4_b;            /* (H) */
  float* const* bond_emb;          /* (5,H) */
  float* const* norm_w;
  float* const* norm_b;            /* (H) */
  /* virtual-node MLPs, arrays [L-1] */
  float* const* vn0_w;
  float* const* vn0_b;
  float* const* vn_ln_w;
  float* const* vn_ln_b;
  float* const* vn4_w;
  float* const* vn4_b;
  /* ProjectionHead fc1 / norm1 / fc2 (H,H) */
  float *head0_w, *head0_b;
  float *head_ln_w, *head_ln_b;
  float *head4_w, *head4_b;
} llb_gin_encoder_grads;
int llb_gin_encoder_saved_bytes(const llb_gin_config* cfg, int num_nodes, int num_edges, int num_graphs, size_t* bytes);
int llb_gin_encoder_forward_saved(llb_gin* h, float* out, void* saved, size_t saved_bytes, llb_stream_t stream);
int llb_gin_encoder_backward(llb_gin* h, int num_nodes, int num_edges, int num_graphs, const float* d_out, void* saved,
                             size_t saved_bytes, const llb_gin_encoder_grads* grads, llb_stream_t stream);
/* Kernels this handle has issued since it was created. */
int64_t llb_gin_launch_count(const llb_gin* h);
/* Statistics of the last llb_gin_predictor_topk call on this handle: rows that went through the fused head + softmax + top-k
 * kernel, and how many of those fell back to the exact materialising path (expected: none). */
enum { LLB_GIN_STAT_HEAD_FUSED_ROWS = 0, LLB_GIN_STAT_HEAD_FLAGGED_ROWS = 1 };
int64_t llb_gin_stat(const llb_gin* h, int which);
/* The softmax + top-k stage on its own (graph_predictor/model.py:177-179: F.softmax(logits, dim=1) then torch.topk):
 * logits (rows, ld) fp32 with W valid columns -> topk_prob / topk_idx (rows, k), value descending, ties to the lowest
 * index.  One streaming pass per row, plus an exact selection-pass redo of the rows flagged in `scratch` (rows int32). */
int llb_softmax_topk(const float* logits, int rows, int W, int ld, int k, float* topk_prob, int32_t* topk_idx,
                     int32_t* scratch, llb_stream_t stream);

/* CostMLP.forward (graph_predictor/model.py:387-391): softplus(W1 relu(W0 fp + b0) + b1).
 * fps (n,2048) fp32, out (n) fp32. */
int llb_cost_mlp(const float* w0, const float* b0, const float* w1, const float* b1, const float* fps, int n,
                 int fp_dim, int latent, float* out, llb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LLAMOLE_B200_H */
