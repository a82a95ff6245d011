// Internal C++ interface of the kernel launchers (the public C ABI is include/etpnav_b200.h).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "host.h"

namespace etp {

typedef __nv_bfloat16 bf16;

struct GemmArgs {
  int M = 0, N = 0, K = 0;
  const bf16* A = nullptr;  // a_mn == 0: [M, K] row-major (pitch lda);  a_mn == 1: [K, M] row-major
  int lda = 0;
  int a_mn = 0;
  const bf16* B = nullptr;  // b_mn == 0: [N, K] row-major (pitch ldb);  b_mn == 1: [K, N] row-major
  int ldb = 0;
  int b_mn = 0;
  float alpha = 1.0f;
  const float* bias = nullptr;  // [N]
  int act = 0;                  // 0 none, 1 gelu(erf), 2 relu
  int aux_mode = 0;             // 0 none, 1: *= gelu'(aux), 2: *= (aux > 0), 3: *= aux
  const bf16* aux = nullptr;
  int ld_aux = 0;
  const float* resid = nullptr;  // fp32 [M, N] added after activation
  int ld_resid = 0;
  float* out_f32 = nullptr;
  int ld_f32 = 0;
  int atomic = 0;  // out_f32 += result (atomicAdd); required for k_splits > 1
  bf16* out_bf16 = nullptr;
  int ld_bf16 = 0;
  bf16* out_pre = nullptr;  // bf16 copy of the pre-activation value (alpha*acc + bias) ...
  int ld_pre = 0;
  int pre_mode = 0;         // ... or, if 1 (with act = gelu), of the activation derivative gelu'(pre) for the backward
  int k_splits = 1;
  int block_n = 0;  // 0 = auto, else 128 or 256
  float* colsum = nullptr;  // fp32 [N]: += column sums of the final value (bias gradient of the producing Linear)
  // dropout applied to the activated value (and to the saved derivative) BEFORE the residual add: nn.Dropout after a
  // dense layer (BertSelfOutput / BertOutput, vilmodel_cmt.py:150-154,189-193; transformer.py:176-181).  thr 0 = off.
  uint32_t drop_key = 0, drop_thr = 0;
  float drop_scale = 1.0f;
};
int gemm(const GemmArgs& a, cudaStream_t stream);
// n <= 8 weight-gradient problems (a_mn = b_mn = 1, out_f32 += A^T.B, nothing else) in one persistent launch
int gemm_grouped_wgrad(const GemmArgs* a, int n, cudaStream_t stream);

// ---- row-wise kernels (elementwise.cu) ------------------------------------------------------------
// y = LayerNorm(x) * gamma + beta over the last dim (H = 768), biased variance, eps inside sqrt.
// Writes any of: y_f32, y_bf16; saves mean / rstd (fp32 [rows]) when non-null.
int layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, int rows, int H, float* y_f32,
                  bf16* y_bf16, float* mean, float* rstd, cudaStream_t stream);
// dx = LN backward (dy fp32 [rows,H], x fp32, mean, rstd); accumulates dgamma/dbeta (fp32 [H], atomicAdd).
// dx is written to dx_f32 (fp32; if accumulate_dx != 0 it is added to the existing content) and,
// if non-null, a bf16 copy to dx_bf16.  dxsum (fp32 [H], optional) += column sums of the written dx: the bias
// gradient of the Linear feeding this LayerNorm, fused here instead of a separate column-sum pass.
int layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd, int rows,
                  int H, float* dx_f32, int accumulate_dx, bf16* dx_bf16, float* dgamma, float* dbeta,
                  cudaStream_t stream, float* dxsum = nullptr, DropHost drop = DropHost{0u, 0u, 1.0f});
// out[c] += sum_r x[r, c]   (bias gradients)
int colsum_bf16(const bf16* x, int rows, int cols, int ld, float* out, cudaStream_t stream);
int colsum_f32(const float* x, int rows, int cols, int ld, float* out, cudaStream_t stream);
// up to 8 of them in one launch (jobs with out == nullptr are skipped); cols, ld multiples of 8, x 16-byte aligned
struct ColsumJob {
  const bf16* x = nullptr;
  int rows = 0, cols = 0, ld = 0;
  float* out = nullptr;
};
int colsum_bf16_grouped(const ColsumJob* jobs, int n, cudaStream_t stream);
int cast_f32_to_bf16(const float* x, bf16* y, int64_t n, cudaStream_t stream);
int dropout_mask(DropHost d, int64_t n, uint8_t* out, cudaStream_t stream);  // keep flags of one site (tests)
int add_f32(float* dst, const float* src, int64_t n, cudaStream_t stream);  // dst += src
// acc[rows[b]*L + l, :] += dkv[b*L + l, :] over b < B, l < L (fp32 += bf16; rows == nullptr: identity; width % 8 == 0).
// The rows of one call must be distinct: there are no atomics.
int kv_grad_accumulate(const bf16* dkv, const int32_t* rows, int B, int L, int width, float* acc, cudaStream_t stream);

// ---- token packing (pack.cu) ----------------------------------------------------------------------
struct PanoPackArgs {
  int rows = 0;                       // B*V
  const float* rgb_lin = nullptr;     // [rows,768] = rgb_fts @ W_img^T + b (GEMM output)
  const float* dep_lin = nullptr;     // [rows,768] or null (use_depth_embedding false)
  const float* loc_fts = nullptr;     // [rows,4]
  const int64_t* nav_types = nullptr; // [rows]
  const float *loc_w = nullptr, *loc_b = nullptr;  // [768,4], [768]
  const float *img_g = nullptr, *img_b = nullptr, *dep_g = nullptr, *dep_b = nullptr, *loc_g = nullptr,
              *loc_bb = nullptr, *out_g = nullptr, *out_b = nullptr;
  const float* nav_emb = nullptr;  // [2,768]
  const float* tok_emb1 = nullptr; // token_type_embeddings row 1, [768]
  float* x_f32 = nullptr;          // [rows,768] packed view tokens (fp32 residual stream)
  // saved for backward (may be null in inference)
  float* loc_lin = nullptr;  // [rows,768]
  float* sum_pre = nullptr;  // [rows,768] value before the final layer_norm
  float* stats = nullptr;    // [rows,8]: mean/rstd of img, dep, loc, out LayerNorms
  DropHost drop{0u, 0u, 1.0f};  // dropout after the final LayerNorm (vilmodel_cmt.py:710-711), train mode
};
int pano_pack_fwd(const PanoPackArgs& a, cudaStream_t stream);

struct NodePackArgs {
  int rows = 0;                         // B*N
  const float* img_fts = nullptr;       // [rows,768]
  const int64_t* step_ids = nullptr;    // [rows]
  const float* pos_fts = nullptr;       // [rows,7]
  const float *pos_w = nullptr, *pos_b = nullptr, *pos_g = nullptr, *pos_bb = nullptr;  // [768,7],[768],[768],[768]
  const float* step_emb = nullptr;      // [100,768]
  float* x_f32 = nullptr;
  bf16* x_bf16 = nullptr;
  float* pos_lin = nullptr;  // saved [rows,768] (null in inference)
  float* stats = nullptr;    // saved [rows,2]
};
int node_pack_fwd(const NodePackArgs& a, cudaStream_t stream);

// SAP head tail: h = LN_1e-12(relu_out) ; logit = h . w4 + b4 ; -inf where visited or padded.
// (vilmodel_cmt.py:654-658 net.2..net.4, :742-744)
// word + position + token-type-0 embedding gather and LayerNorm (BertEmbeddings.forward, vilmodel_cmt.py:62-77)
int embed_txt_fwd(const int64_t* ids, const float* word_emb, const float* pos_emb, const float* type_emb0,
                  const float* gamma, const float* beta, float eps, int B, int L, float* x_f32, bf16* x_bf16,
                  float* sum_pre, float* stats, cudaStream_t stream, DropHost drop = DropHost{0u, 0u, 1.0f});
int seq_mask(const int64_t* lens, int B, int V, uint8_t* mask, cudaStream_t stream);  // mask[b,v] = v < lens[b]

// fused caller-side loss of one step (ss_trainer_ETP.py:879-900): see pack.cu:step_loss_kernel
int step_loss(const float* logits, const int64_t* labels, int B, int N, int64_t ignore_index, float grad_scale,
              float* loss_sum, float* dlogits, float* probs, int64_t* argmax, cudaStream_t stream);

int sap_tail_fwd(const float* relu_out, const float* gamma, const float* beta, const float* w4, const float* b4,
                 const uint8_t* visited, const uint8_t* valid, int rows, int H, float* logits, float* mean,
                 float* rstd, cudaStream_t stream, DropHost drop = DropHost{0u, 0u, 1.0f});

// ---- attention (attention.cu) ---------------------------------------------------------------------
struct AttnArgs {
  int B = 0, heads = 12, Sq = 0, Sk = 0;
  const bf16* q = nullptr;  // [B, Sq, ldq] head h at column h*64
  int ldq = 0;
  const bf16* k = nullptr;  // [B, Sk, ldk]
  int ldk = 0;
  const bf16* v = nullptr;
  int ldv = 0;
  float scale = 0.125f;              // applied to q.k^T
  const uint8_t* key_valid = nullptr;  // [B, Sk] 1 = real token
  float mask_value = -10000.0f;        // added where key_valid == 0 (use -inf for nn.MultiheadAttention semantics)
  const float* pair = nullptr;         // [B, Sq, Sk] or null: bias += pair_w * pair + pair_b
  float pair_w = 0.0f, pair_b = 0.0f;
  const float* pair_w_dev = nullptr;  // optional device scalars overriding pair_w / pair_b
  const float* pair_b_dev = nullptr;
  bf16* out = nullptr;  // [B, Sq, ldo]
  int ldo = 0;
  float* lse = nullptr;  // [B, heads, Sq] log-sum-exp of the biased scores (saved for backward), may be null
  // dropout of the attention probabilities (train mode; thr 0 = off): element index ((b*heads+h)*Sq+q)*Sk+k
  uint32_t drop_key = 0, drop_thr = 0;
  float drop_scale = 1.0f;
  // optional: K / V live in a tensor of kv_B batch rows and query batch b reads row kv_rows[b] of it (device int32 [B]);
  // the episode-level text K|V cache of a rollout whose batch shrinks (etp_nav_inputs.txt_kv_rows)
  const int32_t* kv_rows = nullptr;
  int kv_B = 0;
};
int attention_fwd(const AttnArgs& a, cudaStream_t stream);

struct AttnBwdArgs {
  int B = 0, heads = 12, Sq = 0, Sk = 0;
  const bf16 *q = nullptr, *k = nullptr, *v = nullptr;  // as in the forward
  int ldq = 0, ldk = 0, ldv = 0;
  const bf16* out = nullptr;   // forward output (context), [B,Sq,ldo]
  int ldo = 0;
  const bf16* dout = nullptr;  // gradient of the context
  int lddo = 0;
  const float* lse = nullptr;  // [B,heads,Sq] from the forward
  float* dvec = nullptr;       // scratch [B,heads,Sq]: D_i = sum_d dO*O
  float scale = 0.125f;
  const uint8_t* key_valid = nullptr;
  float mask_value = -10000.0f;
  const float* pair = nullptr;
  float pair_w = 0.0f, pair_b = 0.0f;
  const float* pair_w_dev = nullptr;
  const float* pair_b_dev = nullptr;
  bf16 *dq = nullptr, *dk = nullptr, *dv = nullptr;
  int lddq = 0, lddk = 0, lddv = 0;
  float* dpair_w = nullptr;  // += sum dS * pair   (sprel_linear.weight grad), device scalar or null
  float* dpair_b = nullptr;  // += sum dS          (sprel_linear.bias grad)
  uint32_t drop_key = 0, drop_thr = 0;  // the forward's attention-probability dropout (same key)
  float drop_scale = 1.0f;
  // optional, as in AttnArgs: K / V are READ from row kv_rows[b] of a kv_B-row tensor; dK / dV are still written compact
  // (batch b at row b) — the training rollout's text K|V cache, whose gradient is gathered by kv_grad_accumulate
  const int32_t* kv_rows = nullptr;
  int kv_B = 0;
};
int attention_bwd(const AttnBwdArgs& a, cudaStream_t stream);      // CUDA-core, any shape
int attention_bwd_dispatch(const AttnBwdArgs& a, cudaStream_t stream);

// ---- backward of the packing / head kernels (pack_bwd.cu) -------------------------------------------
// SAP tail backward: dlogits [rows] (entries of dead nodes are ignored) -> d(relu pre-activation) as bf16
// [rows,768] (ReLU mask applied), accumulates dgamma/dbeta [768], dw4 [768], db4 [1].
int sap_tail_bwd(const float* dlogits, const float* relu_out, const float* gamma, const float* beta, const float* w4,
                 const float* mean, const float* rstd, const uint8_t* visited, const uint8_t* valid, int rows,
                 bf16* dpre_bf16, float* dgamma, float* dbeta, float* dw4, float* db4, cudaStream_t stream,
                 DropHost drop = DropHost{0u, 0u, 1.0f});
// node packing backward: dx [rows,768] -> dstep_emb (scatter-add), LN/Linear7 grads. d(img_fts) == dx.
int node_pack_bwd(const float* dx, const int64_t* step_ids, const float* pos_fts, const float* pos_lin,
                  const float* stats, const float* pos_g, int rows, float* dstep_emb, float* dpos_w, float* dpos_b,
                  float* dpos_g, float* dpos_bb, cudaStream_t stream);
struct PanoPackBwdArgs {
  int rows = 0;
  const float* dx = nullptr;        // grad of the packed token [rows,768]
  const float *rgb_lin = nullptr, *dep_lin = nullptr, *loc_lin = nullptr, *sum_pre = nullptr, *stats = nullptr;
  const float* loc_fts = nullptr;
  const int64_t* nav_types = nullptr;
  const float *img_g = nullptr, *dep_g = nullptr, *loc_g = nullptr, *out_g = nullptr;
  bf16 *drgb_lin = nullptr, *ddep_lin = nullptr;  // grads of the two GEMM outputs (bf16, for dgrad/wgrad)
  float *dimg_g = nullptr, *dimg_b = nullptr, *ddep_g = nullptr, *ddep_b = nullptr, *dloc_g = nullptr, *dloc_b = nullptr,
        *dout_g = nullptr, *dout_b = nullptr;
  float *dloc_w = nullptr, *dloc_bias = nullptr;  // [768,4], [768]
  float *dnav_emb = nullptr, *dtok_emb1 = nullptr;
  DropHost drop{0u, 0u, 1.0f};  // the forward's dropout after the final LayerNorm
};
int pano_pack_bwd(const PanoPackBwdArgs& a, cudaStream_t stream);
// embedding + LN backward of forward_txt: dx [rows,768] -> scatter-add into word / position / type-0 tables
int embed_txt_bwd(const float* dx, const int64_t* ids, const float* sum_pre, const float* stats, const float* gamma,
                  int B, int L, float* dword, float* dpos, float* dtype0, float* dgamma, float* dbeta,
                  cudaStream_t stream, DropHost drop = DropHost{0u, 0u, 1.0f});

// ---- optimizer (adamw.cu) ----------------------------------------------------------------------------
// torch.optim.AdamW semantics (decoupled weight decay, bias correction) over flat fp32 buffers; also refreshes
// the bf16 image of the parameters.  grad_scale multiplies the gradient first (1/world_size after all-reduce).
int adamw_step(float* param, bf16* param_bf16, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
               float lr, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
               cudaStream_t stream, const uint8_t* flags = nullptr, const float* normsq = nullptr, float max_norm = 0.0f);
void set_adamw_ctas_per_sm(int n);  // grid size of the update kernel: 16 (default, alone at the HBM roofline) .. 1 (background)
// out[0] += sum g^2 over the blocks whose flag bit 0 is set (all of them when flags == nullptr)
int grad_sumsq(const float* grad, int64_t n, const uint8_t* flags, float* out, cudaStream_t stream);

}  // namespace etp
