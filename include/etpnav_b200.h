/* etpnav_b200 — C ABI of the B200-native ETPNav planner hot path.
 *
 * The reference (MarSaKi/ETPNav) is pure Python and has no FFI: its planner is reached as three
 * methods of one torch.nn.Module,
 *     GlocalTextPathNavCMT.forward_txt        vlnce_baselines/models/etp/vilmodel_cmt.py:684
 *     GlocalTextPathNavCMT.forward_panorama   vlnce_baselines/models/etp/vilmodel_cmt.py:690
 *     GlocalTextPathNavCMT.forward_navigation vlnce_baselines/models/etp/vilmodel_cmt.py:721
 * called from ETP.forward (vlnce_baselines/models/Policy_ViewSelection_ETP.py:167,346,352-357).
 * This header is the boundary a binding for that module sits on: plain pointers and sizes, no torch
 * types.  All pointers are DEVICE pointers unless stated; the caller (PyTorch in the shipped host
 * module etpnav_b200/planner.py) owns every buffer; every call is asynchronous on `stream`
 * (a cudaStream_t passed as void*) and never synchronises.  Return value: 0 = ok, negative = error
 * (see etp_last_error()).  bf16 tensors are raw uint16 storage (`void*` here).
 *
 * Two layers are exported:
 *   (1) step level  — etp_forward_panorama / etp_forward_navigation / etp_forward_txt and their
 *       backward twins: one call = one reference method (INTEGRATION.md shows the binding).
 *   (2) operator level — the fused kernels the step level is made of (GEMM+epilogue, attention,
 *       LayerNorm, token packing, SAP head, AdamW); exported for the parity tests and for hosts that
 *       want to compose them differently.
 * Two further groups at the end of the file cover the rows SURVEY.md §8f calls "next":
 *   (3) the pre-training twin GlocalTextPathCMT (pretrain_src/pretrain_src/model/vilmodel.py:656-754):
 *       etp_segment_gather(_rows), etp_forward_lang2visn / etp_backward_lang2visn;
 *   (4) the trainer's per-step map packing (vlnce_baselines/ss_trainer_ETP.py:344-417): etp_gmap_pack;
 *   (5) the data-parallel update over NVLink peer memory (ss_trainer_ETP.py:211-213): etp_ipc_*, etp_peer_*.
 */
#ifndef ETPNAV_B200_H_
#define ETPNAV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ETP_OK 0
#define ETP_ERR_INVALID (-1)
#define ETP_ERR_CUDA (-2)
#define ETP_ERR_NO_DEVICE (-3)

/* ---------------------------------------------------------------------------------------------
 * library
 * ------------------------------------------------------------------------------------------- */
int etp_version(void);                /* 100 * major + minor */
/* sizeof() of the public structs of this header (gemm_args, attn_args, attn_bwd_args, pano_pack_args, node_pack_args,
 * dropout, layer_weights, nav_weights, nav_inputs, pano_layer_weights, pano_weights, pano_inputs, txt_weights): returns how
 * many there are and fills out[0..n); a binding compares them with its own struct mirrors. */
int etp_struct_sizes(int32_t* out, int32_t n);
const char* etp_last_error(void);     /* text of the last error on this thread */
/* 0 if the current CUDA device is sm_100 (B200); ETP_ERR_NO_DEVICE otherwise. */
int etp_check_device(void);
/* thin CUDA event helpers for hosts without their own bindings (used for the gradient-bucket overlap) */
void* etp_event_create(void);                       /* cudaEventCreateWithFlags(disable timing); NULL on error */
void etp_event_destroy(void* event);
int etp_event_record(void* event, void* stream);        /* cudaEventRecord */
int etp_stream_wait_event(void* stream, void* event);   /* cudaStreamWaitEvent */
/* Leave `n` SMs to other kernels: the library's persistent grids (one CTA or CTA pair per SM) size themselves for the
 * remaining ones.  A data-parallel host sets this to the CTA count of its gradient all-reduce (NCCL_MAX_CTAS) so the
 * collective and the backward GEMMs do not queue for the same SMs; 0 (default) = use every SM. */
void etp_set_sm_reserve(int32_t n);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
long long etp_launch_count(void);
/* CUDA-event timing of every tcgen05 GEMM launch (for the roofline line of bench.py): enable, run steps,
 * collect = synchronise and return total milliseconds / algorithmic flops / launch count, then reset. */
void etp_prof_gemm_enable(int on);
int etp_prof_gemm_collect(double* total_ms, double* total_flops, long long* launches);
/* same records as a text table, one line per (kernel, shape tag): count \t total_ms \t flops \t kernel \t tag;
 * every kernel of the library is timed while profiling is enabled.  Resets the records. */
int etp_prof_report(char* buf, size_t cap);

/* ---------------------------------------------------------------------------------------------
 * operator level
 * ------------------------------------------------------------------------------------------- */

/* D[M,N] = epilogue(alpha * A.B^T) on tcgen05 tensor cores; replaces torch.nn.Linear / matmul on the
 * reference path (vilmodel_cmt.py:108-110,326-328,151,178,190,654; common/transformer.py:174-181).
 * a_mn/b_mn = 0: operand stored [rows, K] (K contiguous); 1: stored [K, rows] (rows contiguous).
 * epilogue: x = alpha*acc + bias[n]; out_pre = bf16(x) (or bf16(gelu'(x)) if pre_mode); x = act(x); x *= f(aux); x += resid;
 *           x = dropout(x) (before the residual; also applied to the saved gelu');
 *           out_f32 (=, or += atomically) x; out_bf16 = bf16(x); colsum[n] += sum_m x (bias gradients). */
typedef struct {
  int32_t M, N, K;
  const void* A; int32_t lda; int32_t a_mn;
  const void* B; int32_t ldb; int32_t b_mn;
  float alpha;
  const float* bias;
  int32_t act;        /* 0 none, 1 gelu(erf), 2 relu */
  int32_t aux_mode;   /* 0 none, 1: *= gelu'(aux), 2: *= (aux > 0), 3: *= aux */
  const void* aux; int32_t ld_aux;
  const float* resid; int32_t ld_resid;
  float* out_f32; int32_t ld_f32; int32_t atomic;
  void* out_bf16; int32_t ld_bf16;
  void* out_pre; int32_t ld_pre;
  int32_t k_splits;   /* >1 requires atomic */
  int32_t block_n;    /* 0 auto, 128, 256 */
  float* colsum;      /* optional fp32 [N]: += column sums of the final value x */
  int32_t pre_mode;   /* 0: out_pre = pre-activation, 1: out_pre = gelu'(pre-activation) (act must be 1) */
  uint32_t drop_key, drop_thr;  /* dropout of the activated value before the residual add; thr = 0: off (see etp_dropout) */
  float drop_scale;
} etp_gemm_args;
int etp_gemm(const etp_gemm_args* args, void* stream);

/* softmax(scale*q.k^T + bias).v, head dim 64; bias = (key_valid ? 0 : mask_value) + pair_w*pair + pair_b.
 * BertOutAttention (vilmodel_cmt.py:325-352), BertSelfAttention (:103-141, graph bias :391-393),
 * nn.MultiheadAttention in the pano encoder (common/transformer.py:176).  impl: 0 auto, 1 CUDA-core,
 * 2 tcgen05 (3 / 4 force its two-CTAs-per-SM / one-CTA-per-SM generation; 2 follows ETP_ATTN_V2, default the former). */
typedef struct {
  int32_t B, heads, Sq, Sk;
  const void* q; int32_t ldq;
  const void* k; int32_t ldk;
  const void* v; int32_t ldv;
  float scale;
  const uint8_t* key_valid;  /* [B,Sk] or NULL */
  float mask_value;
  const float* pair;         /* [B,Sq,Sk] or NULL */
  float pair_w, pair_b;
  const float* pair_w_dev;   /* optional DEVICE scalars overriding pair_w / pair_b (sprel_linear params) */
  const float* pair_b_dev;
  void* out; int32_t ldo;
  float* lse;                /* [B,heads,Sq] or NULL */
  int32_t impl;
} etp_attn_args;
int etp_attention_fwd(const etp_attn_args* args, void* stream);

/* Backward of etp_attention_fwd (same q/k/v/out/lse): dq, dk, dv (bf16) and, when `pair` is given, the
 * sprel_linear gradients accumulated into the device scalars dpair_w / dpair_b.  dvec: fp32 scratch
 * [B,heads,Sq].  impl: 0 auto, 1 CUDA-core, 2 tcgen05 (Sq <= 128). */
typedef struct {
  int32_t B, heads, Sq, Sk;
  const void* q; const void* k; const void* v;
  int32_t ldq, ldk, ldv;
  const void* out; int32_t ldo;
  const void* dout; int32_t lddo;
  const float* lse;
  float* dvec;
  float scale;
  const uint8_t* key_valid;
  float mask_value;
  const float* pair;
  float pair_w, pair_b;
  void* dq; void* dk; void* dv;
  int32_t lddq, lddk, lddv;
  float* dpair_w; float* dpair_b;
  int32_t impl;
} etp_attn_bwd_args;
int etp_attention_bwd(const etp_attn_bwd_args* args, void* stream);

/* LayerNorm over the last dim (768), biased variance (torch.nn.LayerNorm / BertLayerNorm,
 * vilmodel_cmt.py:24-28). */
int etp_layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, int32_t rows, int32_t H,
                      float* y_f32, void* y_bf16, float* mean, float* rstd, void* stream);
int etp_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                      int32_t rows, int32_t H, float* dx_f32, int32_t accumulate_dx, void* dx_bf16, float* dgamma,
                      float* dbeta, void* stream);
int etp_colsum_bf16(const void* x, int32_t rows, int32_t cols, int32_t ld, float* out, void* stream);
int etp_colsum_f32(const float* x, int32_t rows, int32_t cols, int32_t ld, float* out, void* stream);
int etp_cast_f32_to_bf16(const float* x, void* y, int64_t n, void* stream);

/* view-token packing, vilmodel_cmt.py:695-711 */
typedef struct {
  int32_t rows;
  const float* rgb_lin; const float* dep_lin; const float* loc_fts; const int64_t* nav_types;
  const float* loc_w; const float* loc_b;
  const float* img_g; const float* img_b; const float* dep_g; const float* dep_b;
  const float* loc_g; const float* loc_bb; const float* out_g; const float* out_b;
  const float* nav_emb; const float* tok_emb1;
  float* x_f32; float* loc_lin; float* sum_pre; float* stats;
} etp_pano_pack_args;
int etp_pano_pack_fwd(const etp_pano_pack_args* args, void* stream);

/* node-token packing, vilmodel_cmt.py:728-730 */
typedef struct {
  int32_t rows;
  const float* img_fts; const int64_t* step_ids; const float* pos_fts;
  const float* pos_w; const float* pos_b; const float* pos_g; const float* pos_bb;
  const float* step_emb;
  float* x_f32; void* x_bf16; float* pos_lin; float* stats;
} etp_node_pack_args;
int etp_node_pack_fwd(const etp_node_pack_args* args, void* stream);

/* SAP head tail, vilmodel_cmt.py:654-658 (net.2, net.4) and :742-744 */
int etp_sap_tail_fwd(const float* relu_out, const float* gamma, const float* beta, const float* w4, const float* b4,
                     const uint8_t* visited, const uint8_t* valid, int32_t rows, int32_t H, float* logits,
                     float* mean, float* rstd, void* stream);

/* Caller-side loss of one step, fused: softmax / cross-entropy(sum, ignore_index) / its gradient / greedy action
 * over the node logits (ss_trainer_ETP.py:879-900: F.softmax, F.cross_entropy(reduction='sum', ignore_index=-100),
 * argmax).  loss_sum (device scalar) is ADDED to; dlogits = grad_scale * d(sum CE)/d logits; probs, argmax optional. */
int etp_step_loss(const float* logits, const int64_t* labels, int32_t B, int32_t N, int64_t ignore_index,
                  float grad_scale, float* loss_sum, float* dlogits, float* probs, int64_t* argmax, void* stream);

/* ---------------------------------------------------------------------------------------------
 * step level: one call = one reference method
 * ------------------------------------------------------------------------------------------- */

/* Dropout of the reference's train() mode (config.hidden_dropout_prob after every dense / embedding LayerNorm,
 * config.attention_probs_dropout_prob on the attention probabilities, pred_head_dropout_prob in the SAP head;
 * vilmodel_cmt.py:76,133,153,192,349,656; common/transformer.py:176-181).  A keep flag is a pure function of
 * (seed, site, element index): pass the SAME struct to the backward call and it regenerates the forward's masks —
 * nothing is stored.  NULL pointer or p == 0: no dropout (eval()).  Draw a fresh seed for every forward call. */
typedef struct {
  uint64_t seed;
  float p_hidden, p_attn, p_head;
} etp_dropout;
/* keep flags (1 / 0) of elements [0, n) of `site` as the kernels compute them (tests build the matching oracle masks) */
int etp_dropout_mask(const etp_dropout* d, float p, uint32_t site, int64_t n, uint8_t* out, void* stream);

/* One post-LN BERT-style block.  Used three ways:
 *   - GraphLXRTXLayer (vilmodel_cmt.py:365-398): cross-attention (x*) + self-attention (s*) + FFN (f*)
 *   - BertLayer of the language encoder (vilmodel_cmt.py:195-208): x* pointers NULL
 * GEMM weights are bf16 [out,in] row-major; q|k|v (and key|value) are concatenated along `out`
 * by the host at weight-cache time (the fp32 master parameters keep the reference's separate names).
 * biases / LayerNorm affine are fp32. */
typedef struct {
  const void* xq_w;   const float* xq_b;    /* visual_attention.att.query            [768,768]  */
  const void* xkv_w;  const float* xkv_b;   /* visual_attention.att.key|value        [1536,768] */
  const void* xo_w;   const float* xo_b;    /* visual_attention.output.dense         [768,768]  */
  const float* xln_g; const float* xln_b;   /* visual_attention.output.LayerNorm                */
  const void* sqkv_w; const float* sqkv_b;  /* (visn_self_att.self|attention.self).query|key|value [2304,768] */
  const void* so_w;   const float* so_b;    /* (visn_self_att|attention).output.dense           */
  const float* sln_g; const float* sln_b;
  const void* f1_w;   const float* f1_b;    /* (visn_inter|intermediate).dense       [3072,768] */
  const void* f2_w;   const float* f2_b;    /* (visn_output|output).dense            [768,3072] */
  const float* fln_g; const float* fln_b;
} etp_layer_weights;

/* GlobalMapEncoder + CrossmodalEncoder + NextActionPrediction (vilmodel_cmt.py:566-579,435-452,651-661) */
typedef struct {
  int32_t num_x_layers;
  float ln_eps;                       /* config.layer_norm_eps: 1e-12 BERT, 1e-5 XLM-R */
  const etp_layer_weights* layers;    /* HOST array [num_x_layers] */
  const float* pos_w; const float* pos_b; const float* pos_g; const float* pos_bb;  /* gmap_pos_embeddings.{0,1} */
  const float* step_emb;              /* gmap_step_embeddings.weight [100,768] */
  const float* sprel_w; const float* sprel_b;  /* sprel_linear scalars (device) or NULL when !use_sprels */
  const void* sap0_w; const float* sap0_b;     /* global_sap_head.net.0 [768,768] bf16 */
  const float* sap_g; const float* sap_bb;     /* global_sap_head.net.2 LayerNorm */
  const float* sap4_w; const float* sap4_b;    /* global_sap_head.net.4 [1,768], [1] */
  /* key|value projections of ALL x-layers stacked: bf16 [num_x_layers*1536, 768] and fp32 [num_x_layers*1536]
   * (layers[i].xkv_w == xkv_all_w + i*1536*768): the text K/V of every layer come out of one GEMM. */
  const void* xkv_all_w; const float* xkv_all_b;
} etp_nav_weights;

typedef struct {
  int32_t B, N, L;
  const float* txt_embeds;            /* [B,L,768] */
  const uint8_t* txt_masks;           /* [B,L] 1 = token */
  const int64_t* gmap_step_ids;       /* [B,N] */
  const float* gmap_img_fts;          /* [B,N,768] */
  const float* gmap_pos_fts;          /* [B,N,7] */
  const uint8_t* gmap_masks;          /* [B,N] */
  const uint8_t* gmap_visited_masks;  /* [B,N] */
  const float* gmap_pair_dists;       /* [B,N,N] */
  const etp_dropout* dropout;         /* train() mode dropout, or NULL */
  /* backward only, optional: HOST array of num_x_layers + 1 cudaEvent_t (entries may be NULL); event i < X is recorded
   * on the stream when every parameter gradient of x-layer i is complete (layers finish in the order X-1 ... 0),
   * event X when the whole navigation group is, so the caller can start the all-reduce of those gradient slices on
   * another stream while the rest of the backward runs */
  void* const* layer_done_events;
  /* optional: bf16 image of txt_embeds [B,L,768] (raw uint16 storage).  When non-NULL the navigation forward / backward
   * read the instruction through it (their first act on txt_embeds is a cast to bf16 for TMA anyway) and txt_embeds may be
   * NULL: a host that keeps, or stages across PCIe, the instruction embeddings in bf16 saves the cast and half the bytes. */
  const void* txt_embeds_bf16;
  /* optional: the instruction's key|value projections of ALL x-layers, computed once per episode by
   * etp_encode_text_kv (bf16 [txt_kv_batch * L, num_x_layers * 1536]).  The reference recomputes them at every step of
   * every layer although txt_embeds is constant over the episode (vilmodel_cmt.py:326-328; 24 % of the forward FLOPs at
   * B64/N80/L200).  txt_kv_rows (device int32 [B], or NULL = identity) maps the step's batch rows to rows of the
   * episode batch the cache was built for: the trainer shrinks the batch as episodes finish
   * (all_txt_embeds[not_done_index], ss_trainer_ETP.py:819-821).  With txt_kv_all set, txt_embeds may be NULL.
   * In training the record then has no text side (etp_nav_kv_saved_bytes) and the backward needs txt_kv_grad. */
  const void* txt_kv_all;
  const int32_t* txt_kv_rows;
  int32_t txt_kv_batch;
  /* optional, for a host that runs the panorama branch on a second stream next to the instruction-side work of this
   * call (the 768 view rows keep ~130 SMs idle; the text K|V projection and its weight gradient are the only node-
   * independent GEMMs of the step):
   *   side_sm_reserve  SMs the text-side GEMMs of this call (all-layer K|V projection forward; its weight / data
   *                    gradient backward) leave free for that other stream (0 = none)
   *   img_ready_event  forward: cudaEvent_t the stream waits for right before gmap_img_fts is first read (node packing),
   *                    i.e. AFTER the text K|V projection has been issued
   *   img_grad_event   backward: cudaEvent_t recorded as soon as d_gmap_img_fts is final, BEFORE the text-side gradient
   *                    GEMMs are issued */
  int32_t side_sm_reserve;
  void* img_ready_event;
  void* img_grad_event;
  /* backward only, required with txt_kv_all (training rollout through the text K|V cache): fp32 accumulator
   * [txt_kv_batch * L, num_x_layers * 1536] of the rollout's dK|dV.  The backward adds this step's dK|dV into row
   * txt_kv_rows[b] * L + l (no text-side weight / data gradient GEMM runs; d_txt_embeds must be NULL); the per-layer
   * value-bias gradients are still taken here.  After the last step, etp_backward_text_kv turns the accumulator into the
   * key|value weight gradient and d txt_embeds.  Steps must run in order on one stream (plain read-add-write). */
  float* txt_kv_grad;
} etp_nav_inputs;

/* Bytes of the activation record forward_navigation writes (and backward reads) when training != 0;
 * with training == 0 the size of the scratch the forward needs. */
size_t etp_nav_saved_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers, int32_t training);
/* The same with etp_nav_inputs.txt_kv_all set: no bf16 txt_embeds and no K|V of the step in the record, i.e.
 * B*L*(num_x_layers*1536 + 768)*2 bytes less than etp_nav_saved_bytes. */
size_t etp_nav_kv_saved_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers, int32_t training);
/* GlocalTextPathNavCMT.forward_navigation (vilmodel_cmt.py:721-750).
 * outputs: gmap_embeds fp32 [B,N,768], global_logits fp32 [B,N] (-inf at visited / padded nodes). */
int etp_forward_navigation(const etp_nav_weights* w, const etp_nav_inputs* in, float* gmap_embeds,
                           float* global_logits, void* saved, size_t saved_bytes, int32_t training, void* stream);
/* Episode-level text K|V cache of a rollout (inference, or training with etp_nav_inputs.txt_kv_grad):
 * kv_all[b*L + l, i*1536 : (i+1)*1536] = key|value projection of x-layer i of token (b, l)
 * (visual_attention.att.{key,value}, vilmodel_cmt.py:327-328), bf16.  txt_embeds fp32 [B,L,768]
 * (or txt_embeds_bf16, the other NULL); work: B*L*768 bf16 of scratch (unused with the bf16 input). */
int etp_encode_text_kv(const etp_nav_weights* w, const float* txt_embeds, const void* txt_embeds_bf16, int32_t B, int32_t L,
                       void* kv_all, void* work, void* stream);
/* Backward of etp_encode_text_kv after a training rollout: dkv_acc = the etp_nav_inputs.txt_kv_grad accumulator
 * [B*L, num_x_layers*1536] fp32.  Casts it to bf16, ACCUMULATES (+=) its weight gradient into grads->xkv_all_w (one GEMM) and,
 * when d_txt_embeds [B,L,768] fp32 is non-NULL, overwrites it with the data gradient (one GEMM).  txt_embeds fp32 or
 * txt_embeds_bf16 (the other NULL) are the embeddings the cache was built from; work: etp_text_kv_bwd_work_bytes. */
size_t etp_text_kv_bwd_work_bytes(int32_t B, int32_t L, int32_t num_x_layers);
int etp_backward_text_kv(const etp_nav_weights* w, const etp_nav_weights* grads, const float* txt_embeds,
                         const void* txt_embeds_bf16, int32_t B, int32_t L, const float* dkv_acc, float* d_txt_embeds,
                         void* work, void* stream);

/* ImageEmbeddings + pano encoder (vilmodel_cmt.py:454-486; common/transformer.py:127-182) */
typedef struct {
  const void* in_w;  const float* in_b;    /* self_attn.in_proj_weight [2304,768] bf16, in_proj_bias */
  const void* out_w; const float* out_b;   /* self_attn.out_proj */
  const void* l1_w;  const float* l1_b;    /* linear1 [3072,768] */
  const void* l2_w;  const float* l2_b;    /* linear2 [768,3072] */
  const float* n1_g; const float* n1_b; const float* n2_g; const float* n2_b;  /* norm1, norm2 (eps 1e-5) */
} etp_pano_layer_weights;

typedef struct {
  int32_t num_pano_layers;
  float layer_eps;                          /* 1e-5: nn.LayerNorm default inside the pano layers */
  const etp_pano_layer_weights* layers;     /* HOST array */
  const void* img_w; const float* img_b;    /* img_linear [768,512] bf16 */
  const void* dep_w; const float* dep_b;    /* dep_linear [768,128] bf16 or NULL (use_depth_embedding false) */
  const float* loc_w; const float* loc_b;   /* loc_linear [768,4] fp32 */
  const float* img_g; const float* img_bb; const float* dep_g; const float* dep_bb;
  const float* loc_g; const float* loc_bb; const float* out_g; const float* out_bb;  /* 4 LayerNorms, eps 1e-12 */
  const float* nav_emb;                     /* nav_type_embedding.weight [2,768] */
  const float* tok_emb1;                    /* embeddings.token_type_embeddings.weight row 1 */
  const float* fin_g; const float* fin_b;   /* pano_encoder.norm (eps 1e-12) */
} etp_pano_weights;

typedef struct {
  int32_t B, V;
  const float* rgb_fts;       /* [B,V,512] */
  const float* dep_fts;       /* [B,V,128] */
  const float* loc_fts;       /* [B,V,4]   */
  const int64_t* nav_types;   /* [B,V]     */
  const int64_t* view_lens;   /* [B]       */
  const etp_dropout* dropout; /* train() mode dropout, or NULL */
  /* optional, etp_backward_panorama: num_pano_layers cudaEvent_t; event i (i >= 1) is recorded on the stream when every
   * parameter gradient of pano layer i (and, for the last layer, of pano_encoder.norm) is complete — layers finish in
   * the order P-1 ... 1; layer 0 and the view embeddings are final when the call is.  Entry 0 is ignored. */
  void* const* layer_done_events;
} etp_pano_inputs;

size_t etp_pano_saved_bytes(int32_t B, int32_t V, int32_t num_pano_layers, int32_t training);
/* GlocalTextPathNavCMT.forward_panorama (vilmodel_cmt.py:690-719).
 * outputs: pano_embeds fp32 [B,V,768], pano_masks uint8 [B,V] (= arange(V) < view_lens, common/ops.py:36-44). */
int etp_forward_panorama(const etp_pano_weights* w, const etp_pano_inputs* in, float* pano_embeds,
                         uint8_t* pano_masks, void* saved, size_t saved_bytes, int32_t training, void* stream);

/* BertEmbeddings + LanguageEncoder (vilmodel_cmt.py:48-77,413-433) */
typedef struct {
  int32_t num_l_layers;
  float ln_eps;
  const etp_layer_weights* layers;  /* HOST array; x* members NULL */
  const float* word_emb; const float* pos_emb; const float* type_emb0;  /* fp32 tables; type row 0 */
  const float* emb_g; const float* emb_b;
} etp_txt_weights;

size_t etp_txt_saved_bytes(int32_t B, int32_t L, int32_t num_l_layers, int32_t training);
/* GlocalTextPathNavCMT.forward_txt (vilmodel_cmt.py:684-688): txt_ids int64 [B,L], txt_masks uint8 [B,L]
 * -> txt_embeds fp32 [B,L,768]. */
int etp_forward_txt(const etp_txt_weights* w, const int64_t* txt_ids, const uint8_t* txt_masks, int32_t B, int32_t L,
                    float* txt_embeds, void* saved, size_t saved_bytes, int32_t training, void* stream,
                    const etp_dropout* dropout);

/* ---------------------------------------------------------------------------------------------
 * high-precision forward mode (inference): what the reference's eval()/inference() rollouts compute in fp32
 * (ss_trainer_ETP.py:513-756, no autocast) and what BASELINE.json's parity band (rtol 1e-3 / atol 1e-4) needs.
 * Every contraction stays on tcgen05 as a SPLIT-bf16 x3 product realised by tripling K:
 *   A' = [A_hi | A_lo | A_hi] (etp_split3 form 0),  B' = [B_hi | B_hi | B_lo] (form 1),  D = A'.B'^T = etp_gemm(K' = 3K);
 * attention runs in fp32 on the CUDA cores (etp_attention_f32_fwd: etp_attn_args with q/k/v/out FLOAT pointers, lse and
 * impl ignored); activations stay fp32.  The weight structs are the ones of the bf16 mode with every GEMM-weight
 * pointer redirected to the form-1 image of that weight ([out, 3*in] bf16).  `work`: scratch of etp_hp_*_work_bytes.
 * No activation record, no backward.
 * ------------------------------------------------------------------------------------------- */
int etp_split3(const float* x, void* y_bf16, int64_t rows, int32_t K, int32_t form, void* stream);
int etp_attention_f32_fwd(const etp_attn_args* args, void* stream);
size_t etp_hp_nav_work_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers);
size_t etp_hp_pano_work_bytes(int32_t B, int32_t V);
size_t etp_hp_txt_work_bytes(int32_t B, int32_t L);
int etp_forward_navigation_hp(const etp_nav_weights* w, const etp_nav_inputs* in, float* gmap_embeds,
                              float* global_logits, void* work, size_t work_bytes, void* stream);
int etp_forward_panorama_hp(const etp_pano_weights* w, const etp_pano_inputs* in, float* pano_embeds,
                            uint8_t* pano_masks, void* work, size_t work_bytes, void* stream);
int etp_forward_txt_hp(const etp_txt_weights* w, const int64_t* txt_ids, const uint8_t* txt_masks, int32_t B, int32_t L,
                       float* txt_embeds, void* work, size_t work_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * step level, backward (autograd counterparts; the reference gets these from torch autograd via
 * scaler.scale(loss).backward(), ss_trainer_ETP.py:504).
 * `grads` is the same struct type as the weights with EVERY pointer redirected into a flat fp32
 * gradient buffer laid out like the parameters; parameter gradients are ACCUMULATED (+=) there.
 * `saved` is the record the matching forward call wrote with training != 0; `work` is scratch.
 * ------------------------------------------------------------------------------------------- */
size_t etp_nav_bwd_work_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers);
size_t etp_pano_bwd_work_bytes(int32_t B, int32_t V);
size_t etp_txt_bwd_work_bytes(int32_t B, int32_t L);
/* d_gmap_embeds [B,N,768] and/or d_global_logits [B,N] (either may be NULL) -> d_txt_embeds [B,L,768],
 * d_gmap_img_fts [B,N,768] (overwritten; either may be NULL) + parameter gradients. */
int etp_backward_navigation(const etp_nav_weights* w, const etp_nav_weights* grads, const etp_nav_inputs* in,
                            const float* d_gmap_embeds, const float* d_global_logits, void* saved, size_t saved_bytes,
                            void* work, size_t work_bytes, float* d_txt_embeds, float* d_gmap_img_fts, void* stream);
/* d_pano_embeds [B,V,768] -> d_rgb_fts [B,V,512], d_dep_fts [B,V,128] (either may be NULL) + parameter gradients. */
int etp_backward_panorama(const etp_pano_weights* w, const etp_pano_weights* grads, const etp_pano_inputs* in,
                          const uint8_t* pano_masks, const float* d_pano_embeds, void* saved, size_t saved_bytes,
                          void* work, size_t work_bytes, float* d_rgb_fts, float* d_dep_fts, void* stream);
int etp_backward_txt(const etp_txt_weights* w, const etp_txt_weights* grads, const int64_t* txt_ids,
                     const uint8_t* txt_masks, int32_t B, int32_t L, const float* d_txt_embeds, void* saved,
                     size_t saved_bytes, void* work, size_t work_bytes, void* stream, const etp_dropout* dropout);

/* torch.optim.AdamW semantics (ss_trainer_ETP.py:213) over flat fp32 buffers; also rewrites the bf16 image of
 * the parameters.  grad_scale multiplies the gradient first (1/world_size after the gradient all-reduce). */
int etp_adamw_step(float* param, void* param_bf16, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                   float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                   void* stream);

/* The same update with the knobs of the reference's pre-training optimizer (pretrain_src/pretrain_src/optim/misc.py:14-20:
 * no weight decay for biases / LayerNorm; train_r2r.py:279-284: clip_grad_norm_) and of frozen parameters
 * (vilmodel_cmt.py:675-682; torch's AdamW skips parameters without a gradient).  flags: one byte per 64 elements of the
 * flat layout (every tensor starts on a 64-element boundary): bit 0 = trainable, bit 1 = weight decay applies; NULL = all.
 * normsq: DEVICE scalar = sum of g^2 over the trainable blocks (etp_grad_sumsq ADDS to it; zero it first); with
 * max_norm > 0 the gradient is scaled by min(1, max_norm / (grad_scale * sqrt(normsq) + 1e-6)).  n % 64 == 0 with flags. */
int etp_adamw_step_ex(float* param, void* param_bf16, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                      float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                      const uint8_t* flags, const float* normsq, float max_norm, void* stream);
int etp_grad_sumsq(const float* grad, int64_t n, const uint8_t* flags, float* out, void* stream);
/* CTAs per SM of the update kernel: 16 (default: the update alone runs at the HBM roofline) down to 1 (a host that runs it
 * on a side stream under the backward pass: a small grid-striding grid leaves the SM resources to the GEMM CTAs). */
void etp_set_adamw_ctas_per_sm(int32_t n);

/* ---------------------------------------------------------------------------------------------
 * pre-training twin (SURVEY.md §8f N2): GlocalTextPathCMT of pretrain_src/pretrain_src/model/vilmodel.py:656-754.
 * Its `forward` is the composition etp_forward_txt -> etp_forward_panorama over the (sum of steps) x views
 * trajectory batch (ImageEmbeddings.forward, :488-534) -> etp_segment_gather (_aggregate_gmap_features, :585-619)
 * -> etp_forward_navigation; `forward_mlm` (:713-754) replaces the last call by etp_forward_lang2visn.
 * ------------------------------------------------------------------------------------------- */
/* out[s, :] = sum_{k in [seg_ptr[s], seg_ptr[s+1])} weight[k] * src[index[k], :]   (rows of `width` floats, width % 4 == 0;
 * an empty segment writes zeros).  Forward of _aggregate_gmap_features with the host-built CSR of the reference's
 * visited / unvisited dictionaries (weight = 1/len), its backward with the transposed structure, and the
 * masked-token gather of _compute_masked_hidden (pretrain_cmt.py:160-164) with unit weights. */
int etp_segment_gather(const float* src, const int32_t* seg_ptr, const int32_t* index, const float* weight,
                       int32_t num_segments, int32_t width, float* out, void* stream);

/* The same gather with one device pointer per source row (`rows[index[k]]`, each `width` floats, 16-byte aligned): reads
 * the per-node tensors of a GraphMap where they live (inference path of the map image features, no stacking copy). */
int etp_segment_gather_rows(const float* const* rows, const int32_t* seg_ptr, const int32_t* index, const float* weight,
                            int32_t num_segments, int32_t width, float* out, void* stream);

/* GraphLXRTXLayer.forward_lang2visn stacked over the x-layers as GlocalTextPathCMT.forward_mlm drives it
 * (vilmodel.py:400-411,733-741): the instruction tokens query the packed map nodes (visual_attention weights,
 * key mask = gmap_masks), then lang_self_att / lang_inter / lang_output over the tokens.
 * `w` is an etp_nav_weights whose layers[i].{sqkv,so,sln,f1,f2,fln}* point at the lang_* parameters of x-layer i
 * (x* members: visual_attention, as for navigation); sap* / sprel* are ignored.  `in` is the navigation input
 * struct (gmap_visited_masks / gmap_pair_dists ignored).  Output: lang_embeds fp32 [B,L,768]. */
size_t etp_l2v_saved_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers, int32_t training);
int etp_forward_lang2visn(const etp_nav_weights* w, const etp_nav_inputs* in, float* lang_embeds, void* saved,
                          size_t saved_bytes, int32_t training, void* stream);
size_t etp_l2v_bwd_work_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers);
/* d_lang_embeds [B,L,768] -> d_txt_embeds [B,L,768], d_gmap_img_fts [B,N,768] (overwritten; either may be NULL)
 * + parameter gradients accumulated through `grads`. */
int etp_backward_lang2visn(const etp_nav_weights* w, const etp_nav_weights* grads, const etp_nav_inputs* in,
                           const float* d_lang_embeds, void* saved, size_t saved_bytes, void* work, size_t work_bytes,
                           float* d_txt_embeds, float* d_gmap_img_fts, void* stream);

/* ---------------------------------------------------------------------------------------------
 * caller-side packing (SURVEY.md §8f N3): the numeric half of ETPTrainer._nav_gmap_variable
 * (vlnce_baselines/ss_trainer_ETP.py:344-417) with GraphMap.get_pos_fts / front_to_ghost_dist
 * (vlnce_baselines/models/graph_utils.py:258-322), one launch for the whole batch of environments.
 * The host flattens each GraphMap into two blobs (etpnav_b200/packing.py shows the layout a binding produces):
 *   meta[env]  = {n_nodes, n_ghosts, cur_node, off_f64, off_i32, nnz_fronts, 0, 0}          (int32, device)
 *   f64 @off   = cur_pos[3], base_heading, node_pos[3n], ghost_aug_pos[3g], shortest_dist[n*n]
 *   i32 @off   = node_stepId[n], front_ptr[g+1], front_idx[nnz], len(shortest_path)[n*n]
 * Outputs are the padded tensors of the reference, [B, n_max] / [B, n_max, 7] / [B, n_max, n_max], rows
 * [stop], nodes, ghosts, zero padding: gmap_step_ids int64, gmap_visited_masks / gmap_masks uint8 (bool storage),
 * gmap_pos_fts and gmap_pair_dists fp32.  Distances are bit-identical to the reference's numpy (double arithmetic in
 * the same operation order, rounded once to fp32); sin / cos of the float32-rounded angles are within 1 ulp.
 * The image-feature half (stack / pad of node and ghost embeddings, :362-366,399) is etp_segment_gather. */
int etp_gmap_pack(const int32_t* meta, const double* f64_blob, const int32_t* i32_blob, int32_t B, int32_t n_max,
                  int32_t max_ghosts, int64_t* gmap_step_ids, uint8_t* gmap_visited_masks, uint8_t* gmap_masks,
                  float* gmap_pos_fts, float* gmap_pair_dists, void* stream);

/* ---------------------------------------------------------------------------------------------
 * data-parallel update over NVLink peer memory (SURVEY.md §8e): the exchange step of the reference's
 * DistributedDataParallel + torch.optim.AdamW (vlnce_baselines/ss_trainer_ETP.py:211-213) as ONE kernel per gradient
 * bucket — reduce-scatter (peer loads), AdamW on the owned 1/world sub-slice, all-gather of the new parameters and their
 * bf16 image (peer stores).  One process per GPU; every rank maps the other ranks' flat buffers through CUDA IPC.
 * ------------------------------------------------------------------------------------------- */
/* IPC plumbing for hosts without their own: handle (64 bytes) + byte offset of `ptr` inside its allocation;
 * etp_ipc_open maps a peer's allocation (peer access enabled lazily) and returns its base in this process. */
int etp_ipc_export(const void* ptr, void* handle64, int64_t* offset);
int etp_ipc_open(const void* handle64, void** base_out);
int etp_ipc_close(void* base);

#define ETP_PEER_MAX_RANKS 8
#define ETP_PEER_MAX_BUCKETS 32
#define ETP_PEER_FLAG_WORDS (2 * ETP_PEER_MAX_BUCKETS * ETP_PEER_MAX_RANKS)
typedef struct {
  int32_t world, rank;
  float* grad[ETP_PEER_MAX_RANKS];      /* base of every rank's flat fp32 gradient buffer (own entry = local pointer) */
  float* param[ETP_PEER_MAX_RANKS];     /* ... flat fp32 parameter buffer */
  uint16_t* image[ETP_PEER_MAX_RANKS];  /* ... bf16 image of the parameters (what the GEMMs read) */
  uint32_t* flags[ETP_PEER_MAX_RANKS];  /* ... flag block, ETP_PEER_FLAG_WORDS zero-initialised words: [kind][bucket][rank] */
} etp_peer_group;
/* kind 0 = READY (this rank's gradients of `bucket` are final for step `value`), 1 = DONE (this rank has read the bucket's
 * gradients from, and written its new parameters to, every rank).  Signal: this rank's word at EVERY rank := value, after
 * all work already in `stream`.  Wait: spin (device side, own flag block) until the words of all ranks for buckets
 * [bucket_lo, bucket_hi) reach `value`; after `timeout_s` (<= 0: 10 s) the wait gives up and etp_peer_error reports it. */
int etp_peer_signal(const etp_peer_group* g, int32_t kind, int32_t bucket, uint32_t value, void* stream);
int etp_peer_wait(const etp_peer_group* g, int32_t kind, int32_t bucket_lo, int32_t bucket_hi, uint32_t value,
                  double timeout_s, void* stream);
/* The fused kernel over this rank's OWNED sub-slice [offset, offset + n) of the flat buffers (elements, multiples of 4):
 * g = sum_r grad_r (rank order), AdamW with grad_scale 1/world (torch.optim.AdamW, as etp_adamw_step) on exp_avg /
 * exp_avg_sq [n] (owner-local), result stored to param_r / image_r of every rank.  write_reduced != 0 also leaves the
 * summed gradient in the owner's own gradient buffer (self-checks).  ctas: grid size (<= 0: 64). */
int etp_peer_reduce_adamw(const etp_peer_group* g, int64_t offset, int64_t n, float* exp_avg, float* exp_avg_sq, float lr,
                          float beta1, float beta2, float eps, float weight_decay, int32_t step, int32_t write_reduced,
                          int32_t ctas, void* stream);
int etp_peer_error(int32_t* out);   /* 0, or 1 + kind of a wait that timed out (synchronises the device) */

#ifdef __cplusplus
}
#endif
#endif /* ETPNAV_B200_H_ */
