// Step-level backward sequencing: the autograd counterparts of forward_navigation / forward_panorama /
// forward_txt (planner.cu).  Reads the activation record the forward wrote, produces
//   - parameter gradients, ACCUMULATED (+=) into a flat fp32 gradient buffer laid out like the parameters
//     (the `g` structs below are the weight structs with every pointer redirected into that buffer),
//   - gradients w.r.t. the live activations of the caller (txt_embeds, gmap_img_fts, rgb_fts, dep_fts).
// dgrad = tcgen05 GEMM with the weight consumed MN-major as stored; wgrad = tcgen05 GEMM with both operands
// MN-major, split-K, fp32 atomic accumulation; bias grads = column sums; LayerNorm / GELU / ReLU / softmax
// backward fused into the neighbouring kernels where the data is already in registers.
#include "../../include/etpnav_b200.h"
#include "planner.h"

namespace etp {

#define ETP_TRY(expr)              \
  do {                             \
    int _rc = (expr);              \
    if (_rc != ETP_OK) return _rc; \
  } while (0)

struct BwdScratch {
  float *g0 = nullptr, *g1 = nullptr, *g2 = nullptr;  // fp32 [rows,768]
  bf16 *gb = nullptr, *gb2 = nullptr, *gb3 = nullptr;  // bf16 [rows,768]: dY of the three 768-wide Linears of a layer,
                                                        // kept until the layer's weight gradients run as one launch
  bf16 *dctx = nullptr, *dq = nullptr;                  // bf16 [rows,768]
  bf16* dqkv = nullptr;                                 // bf16 [rows,2304]
  bf16* dpre = nullptr;                                 // bf16 [rows,3072]
  bf16* dkv = nullptr;                                  // bf16 [kv_rows,1536]
  float* dvec = nullptr;                                // fp32 [B,heads,S]
  float* dtxt = nullptr;                                // fp32 [kv_rows,768]
  void carve(Arena& ar, size_t rows, size_t kv_rows, size_t bhs, size_t kv_layers = 1) {
    g0 = ar.take<float>(rows * kH); g1 = ar.take<float>(rows * kH); g2 = ar.take<float>(rows * kH);
    gb = ar.take<bf16>(rows * kH); gb2 = ar.take<bf16>(rows * kH); gb3 = ar.take<bf16>(rows * kH);
    dctx = ar.take<bf16>(rows * kH); dq = ar.take<bf16>(rows * kH);
    dqkv = ar.take<bf16>(rows * 3 * kH);
    dpre = ar.take<bf16>(rows * kI);
    dkv = ar.take<bf16>(kv_rows * 2 * kH * kv_layers);  // all layers' dK|dV side by side
    dvec = ar.take<float>(bhs);
    dtxt = ar.take<float>(kv_rows * kH);
  }
};

// dX[rows, K_in] = dY[rows, N_out] . W[N_out, K_in]  (+ resid)   — W consumed MN-major as stored
static int dgrad(const bf16* dY, int rows, int N_out, int ldy, const void* W, int K_in, const float* resid, float* out_f32,
                 bf16* out_bf16, int aux_mode, const bf16* aux, cudaStream_t s, const void* colsum = nullptr) {
  GemmArgs g;
  g.M = rows; g.N = K_in; g.K = N_out;
  g.A = dY; g.lda = ldy;
  g.B = static_cast<const bf16*>(W); g.ldb = K_in; g.b_mn = 1;
  g.resid = resid; g.ld_resid = K_in;
  g.out_f32 = out_f32; g.ld_f32 = K_in;
  g.out_bf16 = out_bf16; g.ld_bf16 = K_in;
  g.aux_mode = aux_mode; g.aux = aux; g.ld_aux = K_in;
  g.colsum = static_cast<float*>(const_cast<void*>(colsum));  // bias gradient of the layer that produced dX's pre-image
  return gemm(g, s);
}

// dW[N_out, K_in] += dY[rows, N_out]^T . X[rows, K_in]   — both operands MN-major as stored; split-K atomics
static int wgrad(const bf16* dY, int rows, int N_out, int ldy, const bf16* X, int K_in, int ldx, void* dW, cudaStream_t s) {
  if (dW == nullptr) return ETP_OK;
  GemmArgs g;
  g.M = N_out; g.N = K_in; g.K = rows;
  g.A = dY; g.lda = ldy; g.a_mn = 1;
  g.B = X; g.ldb = ldx; g.b_mn = 1;
  g.out_f32 = static_cast<float*>(dW); g.ld_f32 = K_in;
  // Few output tiles (256 x bn per CTA pair), long reduction (rows = tokens): pick the tile width and the number of
  // token-axis splits that minimise  waves x (k-blocks per split + epilogue), in units of one 256x256x64 MMA block.
  // One split: every tile owns its output and accumulates with a plain read-add-write (resid = out); otherwise the
  // partial tiles are added with fp32 reductions.
  const int pairs = num_sms() / 2;
  const int kb = (rows + 63) / 64;
  double best = 1e30;
  int best_bn = 128, best_splits = 1;
  for (int bn = 128; bn <= 256; bn += 128) {
    if (bn == 256 && K_in % 256 != 0) continue;
    const int tiles = ((N_out + 255) / 256) * ((K_in + bn - 1) / bn);
    const double w = bn / 256.0;
    for (int splits = 1; splits <= 32 && splits * 4 <= kb; ++splits) {
      const int total = tiles * splits;
      const int waves = (total + pairs - 1) / pairs;
      const int kbs = (kb + splits - 1) / splits;
      const double cost = waves * (kbs * w + 8.0 * w + 4.0);
      if (cost < best) { best = cost; best_bn = bn; best_splits = splits; }
    }
  }
  g.block_n = best_bn;
  g.k_splits = best_splits;
  if (best_splits > 1) {
    g.atomic = 1;
  } else {
    g.resid = g.out_f32; g.ld_resid = K_in;  // dW = acc + dW
  }
  return gemm(g, s);
}

// The weight gradients of one layer do not feed anything else in the backward pass: they are collected here and run
// as ONE grouped launch when the layer's data gradients are done (gemm_grouped_wgrad).  The dY operands must stay
// untouched until flush().
struct WgradBatch {
  GemmArgs a[8];
  int n = 0;
  int add(const bf16* dY, int rows, int N_out, int ldy, const bf16* X, int K_in, int ldx, const void* dW, cudaStream_t s) {
    if (dW == nullptr) return ETP_OK;
    if (n == 8) ETP_TRY(flush(s));
    GemmArgs& g = a[n++];
    g = GemmArgs();
    g.M = N_out; g.N = K_in; g.K = rows;
    g.A = dY; g.lda = ldy; g.a_mn = 1;
    g.B = X; g.ldb = ldx; g.b_mn = 1;
    g.out_f32 = static_cast<float*>(const_cast<void*>(dW)); g.ld_f32 = K_in;
    return ETP_OK;
  }
  int flush(cudaStream_t s) {
    int rc = ETP_OK;
    if (n == 1) rc = wgrad(a[0].A, a[0].K, a[0].M, a[0].lda, a[0].B, a[0].N, a[0].ldb, a[0].out_f32, s);
    else if (n > 1) rc = gemm_grouped_wgrad(a, n, s);
    n = 0;
    return rc;
  }
};

// Bias gradients that need their own pass (d b_q, and d b_v under attention dropout) are collected per layer and run as
// ONE grouped column-sum launch at the layer's end, where every dY operand is still intact (the layer's weight
// gradients, flushed right after, read the same buffers).
struct BiasBatch {
  ColsumJob j[8];
  int n = 0;
  int add(const bf16* dY, int rows, int cols, int ld, const void* db, cudaStream_t s) {
    if (db == nullptr) return ETP_OK;
    if (n == 8) ETP_TRY(flush(s));
    ColsumJob& q = j[n++];
    q.x = dY; q.rows = rows; q.cols = cols; q.ld = ld; q.out = static_cast<float*>(const_cast<void*>(db));
    return ETP_OK;
  }
  int flush(cudaStream_t s) {
    int rc = n > 0 ? colsum_bf16_grouped(j, n, s) : ETP_OK;
    n = 0;
    return rc;
  }
};

static int bias_grad(const bf16* dY, int rows, int cols, int ld, const void* db, cudaStream_t s) {
  if (db == nullptr) return ETP_OK;
  return colsum_bf16(dY, rows, cols, ld, static_cast<float*>(const_cast<void*>(db)), s);
}
static inline float* F(const void* p) { return static_cast<float*>(const_cast<void*>(p)); }

// Backward of self_ffn_block (planner.cu): dx_out = grad of the block output; writes grad of the block input
// (the LayerNorm output `a`) to `da`.  `da` may alias neither sc.g0 nor sc.g1.
static int self_ffn_block_bwd(const etp_layer_weights& w, const etp_layer_weights& g, const LayerRecord& rec,
                              const bf16* a_bf16, const float* dx_out, float* da, int B, int S, const uint8_t* key_valid,
                              const float* pair, const float* pair_w, const float* pair_b, float* dpair_w, float* dpair_b,
                              BwdScratch& sc, WgradBatch& wb, BiasBatch& bb, cudaStream_t s, const DropCtx& dc,
                              uint32_t site_base, int layer) {
  const int rows = B * S;
  // x = LN(t3)
  // (bias gradients ride along: column sums of dt3 inside the LayerNorm backward, of dpre inside the dgrad epilogue)
  ETP_TRY(layernorm_bwd(dx_out, rec.t3, w.fln_g, rec.st3, rec.st3 + rows, rows, kH, sc.g0, 0, sc.gb3, F(g.fln_g), F(g.fln_b), s,
                        F(g.f2_b), dc.hidden(drop_site(site_base, layer, kDropFfnOut))));
  // t3 = h.W2^T + b2 + c
  ETP_TRY(wb.add(sc.gb3, rows, kH, kH, rec.h, kI, kI, g.f2_w, s));
  ETP_TRY(dgrad(sc.gb3, rows, kH, kH, w.f2_w, kI, nullptr, nullptr, sc.dpre, 3, rec.pre, s, g.f1_b));  // * gelu'(pre), saved by the forward
  // pre = c.W1^T + b1
  ETP_TRY(wb.add(sc.dpre, rows, kI, kI, rec.cb, kH, kH, g.f1_w, s));
  ETP_TRY(dgrad(sc.dpre, rows, kI, kI, w.f1_w, kH, sc.g0, sc.g1, nullptr, 0, nullptr, s));  // dc = dpre.W1 + dt3
  // c = LN(t2)
  ETP_TRY(layernorm_bwd(sc.g1, rec.t2, w.sln_g, rec.st2, rec.st2 + rows, rows, kH, sc.g0, 0, sc.gb2, F(g.sln_g), F(g.sln_b), s,
                        F(g.so_b), dc.hidden(drop_site(site_base, layer, kDropSOut))));
  // t2 = ctx2.Wo^T + bo + a
  ETP_TRY(wb.add(sc.gb2, rows, kH, kH, rec.ctx2, kH, kH, g.so_w, s));
  // Bias gradients of the fused q|k|v projection, without touching dK / dV:  the context is  P.(x.Wv + b_v)  and the
  // rows of P sum to one, so  d b_v = column sums of dctx  (taken in this dgrad's epilogue);  a key bias shifts all
  // scores of a query row equally, which softmax ignores, so  d b_k = 0  exactly;  only  d b_q = column sums of dQ
  // needs a pass over the attention backward's output.
  // (with dropout on the attention probabilities the rows of the dropped P no longer sum to one: then d b_v is taken
  // from dV below, as column sums)
  const bool pdrop = dc.attn(0).thr != 0;
  ETP_TRY(dgrad(sc.gb2, rows, kH, kH, w.so_w, kH, nullptr, nullptr, sc.dctx, 0, nullptr, s,
                (g.sqkv_b && !pdrop) ? F(g.sqkv_b) + 2 * kH : nullptr));
  // attention
  AttnBwdArgs at;
  at.B = B; at.heads = kHeads; at.Sq = S; at.Sk = S;
  at.q = rec.qkv; at.k = rec.qkv + kH; at.v = rec.qkv + 2 * kH; at.ldq = at.ldk = at.ldv = 3 * kH;
  at.out = rec.ctx2; at.ldo = kH; at.dout = sc.dctx; at.lddo = kH; at.lse = rec.lse2; at.dvec = sc.dvec;
  at.scale = 0.125f; at.key_valid = key_valid; at.mask_value = -10000.0f;
  at.pair = pair; at.pair_w_dev = pair_w; at.pair_b_dev = pair_b; at.dpair_w = pair ? dpair_w : nullptr;
  at.dpair_b = pair ? dpair_b : nullptr;
  at.dq = sc.dqkv; at.dk = sc.dqkv + kH; at.dv = sc.dqkv + 2 * kH; at.lddq = at.lddk = at.lddv = 3 * kH;
  {
    const DropHost d = dc.attn(drop_site(site_base, layer, kDropSAttn));
    at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
  }
  ETP_TRY(attention_bwd_dispatch(at, s));
  // qkv = a.Wqkv^T + b
  ETP_TRY(bb.add(sc.dqkv, rows, kH, 3 * kH, g.sqkv_b, s));  // query part only (see above)
  if (pdrop && g.sqkv_b) ETP_TRY(bb.add(sc.dqkv + 2 * kH, rows, kH, 3 * kH, F(g.sqkv_b) + 2 * kH, s));
  ETP_TRY(wb.add(sc.dqkv, rows, 3 * kH, 3 * kH, a_bf16, kH, kH, g.sqkv_w, s));
  ETP_TRY(dgrad(sc.dqkv, rows, 3 * kH, 3 * kH, w.sqkv_w, kH, sc.g0, da, nullptr, 0, nullptr, s));  // da = dqkv.Wqkv + dt2
  return ETP_OK;
}

int backward_navigation(const etp_nav_weights& w, const etp_nav_weights& g, const etp_nav_inputs& in,
                        const float* d_gmap_embeds, const float* d_logits, void* saved, size_t saved_bytes, void* work,
                        size_t work_bytes, float* d_txt_embeds, float* d_gmap_img_fts, cudaStream_t s) {
  const int B = in.B, N = in.N, L = in.L, X = w.num_x_layers;
  const int rows = B * N, kv_rows = B * L;
  // episode-level text K|V cache (training rollout): K / V are read from the cache through the row map, and dK|dV of all
  // layers are added into the caller's accumulator instead of becoming this step's text-side weight / data gradients
  const bf16* kv_cache = static_cast<const bf16*>(in.txt_kv_all);
  float* kv_grad = in.txt_kv_grad;
  if (kv_cache || kv_grad) {
    ETP_REQUIRE(kv_cache && kv_grad, "backward_navigation: txt_kv_all and txt_kv_grad go together (the record of a cached "
                                     "forward has no text side)");
    ETP_REQUIRE(X > 0, "backward_navigation: a text K|V cache needs at least one x-layer");
    ETP_REQUIRE(d_txt_embeds == nullptr, "backward_navigation: with txt_kv_grad, d_txt_embeds comes from etp_backward_text_kv");
    ETP_REQUIRE(in.txt_kv_rows == nullptr || in.txt_kv_batch > 0, "backward_navigation: txt_kv_batch must be given with txt_kv_rows");
  }
  Arena ar(saved, saved_bytes);
  NavRecord rec;
  rec.carve(ar, B, N, L, X, true, kv_cache != nullptr);
  ETP_REQUIRE(ar.off <= saved_bytes, "backward_navigation: saved buffer too small");
  Arena wa(work, work_bytes);
  BwdScratch sc;
  sc.carve(wa, rows, kv_rows, static_cast<size_t>(B) * kHeads * (N > L ? N : L), X > 0 ? X : 1);
  float* P = wa.take<float>(static_cast<size_t>(rows) * kH);
  float* Q = wa.take<float>(static_cast<size_t>(rows) * kH);
  ETP_REQUIRE(wa.off <= work_bytes, "backward_navigation: workspace too small");
  ETP_REQUIRE(d_gmap_embeds || d_logits, "backward_navigation: no incoming gradient");
  DropCtx dc;
  if (in.dropout) { dc.seed = in.dropout->seed; dc.p_hidden = in.dropout->p_hidden; dc.p_attn = in.dropout->p_attn; dc.p_head = in.dropout->p_head; }

  const bf16* x_last = X > 0 ? rec.layers[X - 1].xb : rec.x0b;
  if (d_logits) {
    ETP_TRY(sap_tail_bwd(d_logits, rec.relu, w.sap_g, w.sap_bb, w.sap4_w, rec.sap_stats, rec.sap_stats + rows,
                         in.gmap_visited_masks, in.gmap_masks, rows, sc.gb, F(g.sap_g), F(g.sap_bb), F(g.sap4_w), F(g.sap4_b), s,
                         dc.head(kSiteNav + kSiteHead)));
    ETP_TRY(bias_grad(sc.gb, rows, kH, kH, g.sap0_b, s));
    ETP_TRY(wgrad(sc.gb, rows, kH, kH, x_last, kH, kH, const_cast<void*>(g.sap0_w), s));
    ETP_TRY(dgrad(sc.gb, rows, kH, kH, w.sap0_w, kH, d_gmap_embeds, P, nullptr, 0, nullptr, s));
  } else {
    ETP_CHECK_CUDA(cudaMemcpyAsync(P, d_gmap_embeds, static_cast<size_t>(rows) * kH * 4, cudaMemcpyDeviceToDevice, s));
  }
  float* dtxt = d_txt_embeds ? d_txt_embeds : sc.dtxt;
  const int ldkv = X * 2 * kH;
  for (int i = X - 1; i >= 0; --i) {
    const etp_layer_weights& lw = w.layers[i];
    const etp_layer_weights& lg = g.layers[i];
    const LayerRecord& r = rec.layers[i];
    const bf16* x_in = i > 0 ? rec.layers[i - 1].xb : rec.x0b;
    WgradBatch wb;
    BiasBatch bb;
    ETP_TRY(self_ffn_block_bwd(lw, lg, r, r.ab, P, Q, B, N, in.gmap_masks, w.sprel_w ? in.gmap_pair_dists : nullptr, w.sprel_w,
                               w.sprel_b, F(g.sprel_w), F(g.sprel_b), sc, wb, bb, s, dc, kSiteNav, i));
    // a = LN(t1),  t1 = ctx1.Wo^T + bo + x_in
    ETP_TRY(layernorm_bwd(Q, r.t1, lw.xln_g, r.st1, r.st1 + rows, rows, kH, sc.g0, 0, sc.gb, F(lg.xln_g), F(lg.xln_b), s,
                          F(lg.xo_b), dc.hidden(drop_site(kSiteNav, i, kDropXOut))));
    ETP_TRY(wb.add(sc.gb, rows, kH, kH, r.ctx1, kH, kH, lg.xo_w, s));
    // d b_v (text value bias of this layer) = column sums of dctx; d b_k = 0 (see self_ffn_block_bwd)
    const bool pdrop = dc.attn(0).thr != 0;  // dropped P rows do not sum to one: d b_v from dV after the attention backward
    ETP_TRY(dgrad(sc.gb, rows, kH, kH, lw.xo_w, kH, nullptr, nullptr, sc.dctx, 0, nullptr, s,
                  (lg.xkv_b && !pdrop) ? F(lg.xkv_b) + kH : nullptr));
    AttnBwdArgs at;
    at.B = B; at.heads = kHeads; at.Sq = N; at.Sk = L;
    at.q = r.q; at.ldq = kH; at.k = r.kv; at.ldk = r.ldkv; at.v = r.kv + kH; at.ldv = r.ldkv;
    if (kv_cache) {  // as in the forward: layer i's slice of the cached rows, read through the batch-row map
      at.k = kv_cache + static_cast<size_t>(i) * 2 * kH; at.v = at.k + kH;
      at.ldk = at.ldv = ldkv;
      at.kv_rows = in.txt_kv_rows; at.kv_B = in.txt_kv_rows ? in.txt_kv_batch : B;
    }
    at.out = r.ctx1; at.ldo = kH; at.dout = sc.dctx; at.lddo = kH; at.lse = r.lse1; at.dvec = sc.dvec;
    at.scale = 0.125f; at.key_valid = in.txt_masks; at.mask_value = -10000.0f;
    bf16* dkv_i = sc.dkv + static_cast<size_t>(i) * 2 * kH;  // this layer's slice of [B*L, X*1536]
    at.dq = sc.dq; at.lddq = kH; at.dk = dkv_i; at.lddk = ldkv; at.dv = dkv_i + kH; at.lddv = ldkv;
    {
      const DropHost d = dc.attn(drop_site(kSiteNav, i, kDropXAttn));
      at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
    }
    ETP_TRY(attention_bwd_dispatch(at, s));
    ETP_TRY(bb.add(sc.dq, rows, kH, kH, lg.xq_b, s));
    if (pdrop && lg.xkv_b) ETP_TRY(bb.add(dkv_i + kH, kv_rows, kH, ldkv, F(lg.xkv_b) + kH, s));
    ETP_TRY(wb.add(sc.dq, rows, kH, kH, x_in, kH, kH, lg.xq_w, s));
    ETP_TRY(dgrad(sc.dq, rows, kH, kH, lw.xq_w, kH, sc.g0, P, nullptr, 0, nullptr, s));  // dx_in = dq.Wq + dt1
    ETP_TRY(bb.flush(s));  // the layer's bias gradients that need a pass of their own, one launch
    ETP_TRY(wb.flush(s));  // the layer's six weight gradients, one launch
    if (in.layer_done_events && in.layer_done_events[i])
      ETP_CHECK_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(in.layer_done_events[i]), s));
  }
  // node packing: x0 = img_fts + E_step[ids] + LN(pos_fts.W^T + b).  Done BEFORE the text-side GEMMs: d_gmap_img_fts is
  // what the panorama branch's backward waits for (img_grad_event), and nothing below touches it.
  ETP_TRY(node_pack_bwd(P, in.gmap_step_ids, in.gmap_pos_fts, rec.pos_lin, rec.pos_stats, w.pos_g, rows, F(g.step_emb),
                        F(g.pos_w), F(g.pos_b), F(g.pos_g), F(g.pos_bb), s));
  if (d_gmap_img_fts)
    ETP_CHECK_CUDA(cudaMemcpyAsync(d_gmap_img_fts, P, static_cast<size_t>(rows) * kH * 4, cudaMemcpyDeviceToDevice, s));
  if (in.img_grad_event) ETP_CHECK_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(in.img_grad_event), s));
  // text side, all layers at once: kv_all = txt . Wkv_all^T + b  ->  one wgrad, one dgrad (bias grads: above); they leave
  // side_sm_reserve SMs to the stream that now runs the panorama backward
  if (kv_grad) {
    ETP_TRY(kv_grad_accumulate(sc.dkv, in.txt_kv_rows, B, L, ldkv, kv_grad, s));
  } else if (X > 0) {
    const bf16* txtb = in.txt_embeds_bf16 ? static_cast<const bf16*>(in.txt_embeds_bf16) : rec.txtb;
    const int prev = get_sm_reserve();
    if (in.side_sm_reserve > 0) set_sm_reserve(prev + in.side_sm_reserve);
    int rc = wgrad(sc.dkv, kv_rows, ldkv, ldkv, txtb, kH, kH, const_cast<void*>(g.xkv_all_w), s);
    if (rc == ETP_OK && d_txt_embeds) rc = dgrad(sc.dkv, kv_rows, ldkv, ldkv, w.xkv_all_w, kH, nullptr, dtxt, nullptr, 0, nullptr, s);
    set_sm_reserve(prev);
    ETP_TRY(rc);
  } else if (d_txt_embeds) {
    ETP_CHECK_CUDA(cudaMemsetAsync(d_txt_embeds, 0, static_cast<size_t>(kv_rows) * kH * 4, s));
  }
  // entry X of the optional event array: every gradient of the navigation group is complete
  if (in.layer_done_events && in.layer_done_events[X])
    ETP_CHECK_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(in.layer_done_events[X]), s));
  return ETP_OK;
}

// Backward of forward_lang2visn (planner.cu).  Same skeleton as backward_navigation with the roles swapped: the token
// stream carries the residual gradient (P), the node side receives dK|dV of all layers, which become one wgrad and one
// dgrad of the stacked key|value projection, and then flow into the node-packing backward.
int backward_lang2visn(const etp_nav_weights& w, const etp_nav_weights& g, const etp_nav_inputs& in,
                       const float* d_lang_embeds, void* saved, size_t saved_bytes, void* work, size_t work_bytes,
                       float* d_txt_embeds, float* d_gmap_img_fts, cudaStream_t s) {
  const int B = in.B, N = in.N, L = in.L, X = w.num_x_layers;
  ETP_REQUIRE(X >= 1, "backward_lang2visn: needs at least one x-layer");
  const int rows = B * L, kv_rows = B * N;
  Arena ar(saved, saved_bytes);
  L2VRecord rec;
  rec.carve(ar, B, N, L, X, true);
  ETP_REQUIRE(ar.off <= saved_bytes, "backward_lang2visn: saved buffer too small");
  Arena wa(work, work_bytes);
  BwdScratch sc;
  sc.carve(wa, rows, kv_rows, static_cast<size_t>(B) * kHeads * (N > L ? N : L), X);
  float* P = wa.take<float>(static_cast<size_t>(rows) * kH);
  float* Q = wa.take<float>(static_cast<size_t>(rows) * kH);
  ETP_REQUIRE(wa.off <= work_bytes, "backward_lang2visn: workspace too small");
  DropCtx dc;
  if (in.dropout) { dc.seed = in.dropout->seed; dc.p_hidden = in.dropout->p_hidden; dc.p_attn = in.dropout->p_attn; dc.p_head = in.dropout->p_head; }

  const float* dx = d_lang_embeds;
  const int ldkv = X * 2 * kH;
  for (int i = X - 1; i >= 0; --i) {
    const etp_layer_weights& lw = w.layers[i];
    const etp_layer_weights& lg = g.layers[i];
    const LayerRecord& r = rec.layers[i];
    const bf16* x_in = i > 0 ? rec.layers[i - 1].xb : rec.txtb;
    WgradBatch wb;
    BiasBatch bb;
    ETP_TRY(self_ffn_block_bwd(lw, lg, r, r.ab, dx, Q, B, L, in.txt_masks, nullptr, nullptr, nullptr, nullptr, nullptr, sc, wb,
                               bb, s, dc, kSiteL2V, i));
    ETP_TRY(layernorm_bwd(Q, r.t1, lw.xln_g, r.st1, r.st1 + rows, rows, kH, sc.g0, 0, sc.gb, F(lg.xln_g), F(lg.xln_b), s,
                          F(lg.xo_b), dc.hidden(drop_site(kSiteL2V, i, kDropXOut))));
    ETP_TRY(wb.add(sc.gb, rows, kH, kH, r.ctx1, kH, kH, lg.xo_w, s));
    const bool pdrop = dc.attn(0).thr != 0;
    ETP_TRY(dgrad(sc.gb, rows, kH, kH, lw.xo_w, kH, nullptr, nullptr, sc.dctx, 0, nullptr, s,
                  (lg.xkv_b && !pdrop) ? F(lg.xkv_b) + kH : nullptr));
    AttnBwdArgs at;
    at.B = B; at.heads = kHeads; at.Sq = L; at.Sk = N;
    at.q = r.q; at.ldq = kH; at.k = r.kv; at.ldk = r.ldkv; at.v = r.kv + kH; at.ldv = r.ldkv;
    at.out = r.ctx1; at.ldo = kH; at.dout = sc.dctx; at.lddo = kH; at.lse = r.lse1; at.dvec = sc.dvec;
    at.scale = 0.125f; at.key_valid = in.gmap_masks; at.mask_value = -10000.0f;
    bf16* dkv_i = sc.dkv + static_cast<size_t>(i) * 2 * kH;
    at.dq = sc.dq; at.lddq = kH; at.dk = dkv_i; at.lddk = ldkv; at.dv = dkv_i + kH; at.lddv = ldkv;
    {
      const DropHost d = dc.attn(drop_site(kSiteL2V, i, kDropXAttn));
      at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
    }
    ETP_TRY(attention_bwd_dispatch(at, s));
    ETP_TRY(bb.add(sc.dq, rows, kH, kH, lg.xq_b, s));
    if (pdrop && lg.xkv_b) ETP_TRY(bb.add(dkv_i + kH, kv_rows, kH, ldkv, F(lg.xkv_b) + kH, s));
    ETP_TRY(wb.add(sc.dq, rows, kH, kH, x_in, kH, kH, lg.xq_w, s));
    // dx_in = dq.Wq + dt1; the first layer's input is the caller's txt_embeds
    float* dst = (i == 0 && d_txt_embeds) ? d_txt_embeds : P;
    ETP_TRY(dgrad(sc.dq, rows, kH, kH, lw.xq_w, kH, sc.g0, dst, nullptr, 0, nullptr, s));
    ETP_TRY(bb.flush(s));
    ETP_TRY(wb.flush(s));
    dx = P;
  }
  // node side, all layers at once: kv_all = nodes . Wkv_all^T + b
  ETP_TRY(wgrad(sc.dkv, kv_rows, ldkv, ldkv, rec.nodeb, kH, kH, const_cast<void*>(g.xkv_all_w), s));
  ETP_TRY(dgrad(sc.dkv, kv_rows, ldkv, ldkv, w.xkv_all_w, kH, nullptr, sc.dtxt, nullptr, 0, nullptr, s));  // d(packed nodes)
  ETP_TRY(node_pack_bwd(sc.dtxt, in.gmap_step_ids, in.gmap_pos_fts, rec.pos_lin, rec.pos_stats, w.pos_g, kv_rows, F(g.step_emb),
                        F(g.pos_w), F(g.pos_b), F(g.pos_g), F(g.pos_bb), s));
  if (d_gmap_img_fts)
    ETP_CHECK_CUDA(cudaMemcpyAsync(d_gmap_img_fts, sc.dtxt, static_cast<size_t>(kv_rows) * kH * 4, cudaMemcpyDeviceToDevice, s));
  return ETP_OK;
}

int backward_panorama(const etp_pano_weights& w, const etp_pano_weights& g, const etp_pano_inputs& in,
                      const uint8_t* pano_masks, const float* d_pano_embeds, void* saved, size_t saved_bytes, void* work,
                      size_t work_bytes, float* d_rgb_fts, float* d_dep_fts, cudaStream_t s) {
  const int B = in.B, V = in.V, Pn = w.num_pano_layers;
  const int rows = B * V;
  Arena ar(saved, saved_bytes);
  PanoRecord rec;
  rec.carve(ar, B, V, Pn, true);
  ETP_REQUIRE(ar.off <= saved_bytes, "backward_panorama: saved buffer too small");
  Arena wa(work, work_bytes);
  BwdScratch sc;
  sc.carve(wa, rows, 0, static_cast<size_t>(B) * kHeads * V);
  ETP_REQUIRE(wa.off <= work_bytes, "backward_panorama: workspace too small");
  DropCtx dc;
  if (in.dropout) { dc.seed = in.dropout->seed; dc.p_hidden = in.dropout->p_hidden; dc.p_attn = in.dropout->p_attn; dc.p_head = in.dropout->p_head; }
  float* A = sc.g0;
  float* Bf = sc.g1;
  if (Pn > 0) {
    ETP_TRY(layernorm_bwd(d_pano_embeds, rec.xs[2 * Pn], w.fin_g, rec.fin_stats, rec.fin_stats + rows, rows, kH, A, 0, sc.gb,
                          F(g.fin_g), F(g.fin_b), s, F(g.layers[Pn - 1].l2_b),
                          dc.hidden(drop_site(kSitePano, Pn - 1, kDropPFfnOut))));  // bf16 copy = d linear2 output of the last layer
  } else {
    ETP_CHECK_CUDA(cudaMemcpyAsync(A, d_pano_embeds, static_cast<size_t>(rows) * kH * 4, cudaMemcpyDeviceToDevice, s));
  }
  for (int i = Pn - 1; i >= 0; --i) {
    const etp_pano_layer_weights& lw = w.layers[i];
    const etp_pano_layer_weights& lg = g.layers[i];
    const PanoLayerRecord& r = rec.layers[i];
    const float* x = rec.xs[2 * i];
    const float* x_mid = rec.xs[2 * i + 1];
    // x_out = x_mid + gelu(LN2(x_mid).W1^T + b1).W2^T + b2      (A = dx_out, sc.gb = bf16(A); the linear2 bias
    // gradient = column sums of A was accumulated by the LayerNorm backward that produced A)
    WgradBatch wb;
    ETP_TRY(wb.add(sc.gb, rows, kH, kH, r.h, kI, kI, lg.l2_w, s));
    ETP_TRY(dgrad(sc.gb, rows, kH, kH, lw.l2_w, kI, nullptr, nullptr, sc.dpre, 3, r.pre, s, lg.l1_b));
    ETP_TRY(wb.add(sc.dpre, rows, kI, kI, r.y2b, kH, kH, lg.l1_w, s));
    ETP_TRY(dgrad(sc.dpre, rows, kI, kI, lw.l1_w, kH, nullptr, Bf, nullptr, 0, nullptr, s));  // dy2
    ETP_TRY(layernorm_bwd(Bf, x_mid, lw.n2_g, r.st2, r.st2 + rows, rows, kH, A, 1, sc.gb2, F(lg.n2_g), F(lg.n2_b), s,
                          F(lg.out_b), dc.hidden(drop_site(kSitePano, i, kDropPOut))));  // A = dx_mid
    // x_mid = x + attn(LN1(x)).Wout^T + bout
    ETP_TRY(wb.add(sc.gb2, rows, kH, kH, r.ctx, kH, kH, lg.out_w, s));
    const bool pdrop = dc.hidden(0).thr != 0;  // MHA dropout on: d b_v from dV below
    ETP_TRY(dgrad(sc.gb2, rows, kH, kH, lw.out_w, kH, nullptr, nullptr, sc.dctx, 0, nullptr, s,
                  (lg.in_b && !pdrop) ? F(lg.in_b) + 2 * kH : nullptr));  // d b_v of in_proj_bias (q|k|v); d b_k = 0
    AttnBwdArgs at;
    at.B = B; at.heads = kHeads; at.Sq = V; at.Sk = V;
    at.q = r.qkv; at.k = r.qkv + kH; at.v = r.qkv + 2 * kH; at.ldq = at.ldk = at.ldv = 3 * kH;
    at.out = r.ctx; at.ldo = kH; at.dout = sc.dctx; at.lddo = kH; at.lse = r.lse; at.dvec = sc.dvec;
    at.scale = 0.125f; at.key_valid = pano_masks; at.mask_value = -INFINITY;
    at.dq = sc.dqkv; at.dk = sc.dqkv + kH; at.dv = sc.dqkv + 2 * kH; at.lddq = at.lddk = at.lddv = 3 * kH;
    {
      const DropHost d = dc.hidden(drop_site(kSitePano, i, kDropPAttn));  // MHA dropout = hidden_dropout_prob (common/ops.py:15)
      at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
    }
    ETP_TRY(attention_bwd(at, s));
    BiasBatch bb;
    ETP_TRY(bb.add(sc.dqkv, rows, kH, 3 * kH, lg.in_b, s));  // query part
    if (pdrop && lg.in_b) ETP_TRY(bb.add(sc.dqkv + 2 * kH, rows, kH, 3 * kH, F(lg.in_b) + 2 * kH, s));
    ETP_TRY(bb.flush(s));
    ETP_TRY(wb.add(sc.dqkv, rows, 3 * kH, 3 * kH, r.y1b, kH, kH, lg.in_w, s));
    ETP_TRY(dgrad(sc.dqkv, rows, 3 * kH, 3 * kH, lw.in_w, kH, nullptr, Bf, nullptr, 0, nullptr, s));  // dy1
    ETP_TRY(wb.flush(s));  // the layer's four weight gradients, one launch (sc.gb is rewritten just below)
    ETP_TRY(layernorm_bwd(Bf, x, lw.n1_g, r.st1, r.st1 + rows, rows, kH, A, 1, sc.gb, F(lg.n1_g), F(lg.n1_b), s,
                          i > 0 ? F(g.layers[i - 1].l2_b) : nullptr,
                          i > 0 ? dc.hidden(drop_site(kSitePano, i - 1, kDropPFfnOut)) : DropHost{0u, 0u, 1.0f}));  // A = dx (= dx_out of layer i-1)
    if (i > 0 && in.layer_done_events && in.layer_done_events[i])   // layer i's gradient slice is final: its exchange may start
      ETP_CHECK_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(in.layer_done_events[i]), s));
  }
  PanoPackBwdArgs pb;
  pb.rows = rows; pb.dx = A; pb.rgb_lin = rec.rgb_lin; pb.dep_lin = w.dep_w ? rec.dep_lin : nullptr; pb.loc_lin = rec.loc_lin;
  pb.sum_pre = rec.sum_pre; pb.stats = rec.stats; pb.loc_fts = in.loc_fts; pb.nav_types = in.nav_types;
  pb.img_g = w.img_g; pb.dep_g = w.dep_g; pb.loc_g = w.loc_g; pb.out_g = w.out_g;
  pb.drgb_lin = sc.dq; pb.ddep_lin = sc.dctx;
  pb.dimg_g = F(g.img_g); pb.dimg_b = F(g.img_bb); pb.ddep_g = F(g.dep_g); pb.ddep_b = F(g.dep_bb);
  pb.dloc_g = F(g.loc_g); pb.dloc_b = F(g.loc_bb); pb.dout_g = F(g.out_g); pb.dout_b = F(g.out_bb);
  pb.dloc_w = F(g.loc_w); pb.dloc_bias = F(g.loc_b); pb.dnav_emb = F(g.nav_emb); pb.dtok_emb1 = F(g.tok_emb1);
  pb.drop = dc.hidden(kSitePano + kSiteEmbed);
  ETP_TRY(pano_pack_bwd(pb, s));
  ETP_TRY(bias_grad(sc.dq, rows, kH, kH, g.img_b, s));
  ETP_TRY(wgrad(sc.dq, rows, kH, kH, rec.rgbb, 512, 512, const_cast<void*>(g.img_w), s));
  if (d_rgb_fts) ETP_TRY(dgrad(sc.dq, rows, kH, kH, w.img_w, 512, nullptr, d_rgb_fts, nullptr, 0, nullptr, s));
  if (w.dep_w) {
    ETP_TRY(bias_grad(sc.dctx, rows, kH, kH, g.dep_b, s));
    ETP_TRY(wgrad(sc.dctx, rows, kH, kH, rec.depb, 128, 128, const_cast<void*>(g.dep_w), s));
    if (d_dep_fts) ETP_TRY(dgrad(sc.dctx, rows, kH, kH, w.dep_w, 128, nullptr, d_dep_fts, nullptr, 0, nullptr, s));
  }
  return ETP_OK;
}

int backward_txt(const etp_txt_weights& w, const etp_txt_weights& g, const int64_t* txt_ids, const uint8_t* txt_masks, int B,
                 int L, const float* d_txt_embeds, void* saved, size_t saved_bytes, void* work, size_t work_bytes,
                 cudaStream_t s, const etp_dropout* dropout) {
  DropCtx dc;
  if (dropout) { dc.seed = dropout->seed; dc.p_hidden = dropout->p_hidden; dc.p_attn = dropout->p_attn; dc.p_head = dropout->p_head; }
  const int NL = w.num_l_layers, rows = B * L;
  Arena ar(saved, saved_bytes);
  TxtRecord rec;
  rec.carve(ar, B, L, NL, true);
  ETP_REQUIRE(ar.off <= saved_bytes, "backward_txt: saved buffer too small");
  Arena wa(work, work_bytes);
  BwdScratch sc;
  sc.carve(wa, rows, 0, static_cast<size_t>(B) * kHeads * L);
  float* P = wa.take<float>(static_cast<size_t>(rows) * kH);
  float* Q = wa.take<float>(static_cast<size_t>(rows) * kH);
  ETP_REQUIRE(wa.off <= work_bytes, "backward_txt: workspace too small");
  const float* dx = d_txt_embeds;
  for (int i = NL - 1; i >= 0; --i) {
    const bf16* a_bf16 = i > 0 ? rec.layers[i - 1].xb : rec.x0b;
    float* da = (dx == P) ? Q : P;
    WgradBatch wb;
    BiasBatch bb;
    ETP_TRY(self_ffn_block_bwd(w.layers[i], g.layers[i], rec.layers[i], a_bf16, dx, da, B, L, txt_masks, nullptr, nullptr,
                               nullptr, nullptr, nullptr, sc, wb, bb, s, dc, kSiteTxt, i));
    ETP_TRY(bb.flush(s));
    ETP_TRY(wb.flush(s));
    dx = da;
  }
  ETP_TRY(embed_txt_bwd(dx, txt_ids, rec.sum_pre, rec.emb_stats, w.emb_g, B, L, F(g.word_emb), F(g.pos_emb), F(g.type_emb0),
                        F(g.emb_g), F(g.emb_b), s, dc.hidden(kSiteTxt + kSiteEmbed)));
  return ETP_OK;
}

// Backward of etp_encode_text_kv for a training rollout: the accumulated dK|dV of every step, cast to bf16 once, make ONE
// weight gradient of the stacked key|value projection and (optionally) ONE data gradient of txt_embeds.  (The value-bias
// gradients were taken step by step by backward_navigation; the key-bias gradient is zero.)
int backward_text_kv(const etp_nav_weights& w, const etp_nav_weights& g, const float* txt_embeds, const bf16* txt_embeds_bf16,
                     int B, int L, const float* dkv_acc, float* d_txt_embeds, void* work, cudaStream_t s) {
  const int X = w.num_x_layers;
  ETP_REQUIRE(B > 0 && L > 0 && X > 0, "backward_text_kv: bad shape");
  const size_t rows = static_cast<size_t>(B) * L, ldkv = static_cast<size_t>(X) * 2 * kH;
  Arena wa(work, ~size_t(0));
  bf16* dkvb = wa.take<bf16>(rows * ldkv);
  const bf16* txtb = txt_embeds_bf16;
  if (txtb == nullptr) {
    bf16* t = wa.take<bf16>(rows * kH);
    ETP_TRY(cast_f32_to_bf16(txt_embeds, t, static_cast<int64_t>(rows) * kH, s));
    txtb = t;
  }
  ETP_TRY(cast_f32_to_bf16(dkv_acc, dkvb, static_cast<int64_t>(rows * ldkv), s));
  ETP_TRY(wgrad(dkvb, static_cast<int>(rows), static_cast<int>(ldkv), static_cast<int>(ldkv), txtb, kH, kH,
                const_cast<void*>(g.xkv_all_w), s));
  if (d_txt_embeds)
    ETP_TRY(dgrad(dkvb, static_cast<int>(rows), static_cast<int>(ldkv), static_cast<int>(ldkv), w.xkv_all_w, kH, nullptr,
                  d_txt_embeds, nullptr, 0, nullptr, s));
  return ETP_OK;
}

static size_t work_bytes_for(size_t rows, size_t kv_rows, size_t bhs, size_t kv_layers = 1) {
  Arena wa(nullptr, ~size_t(0));
  BwdScratch sc;
  sc.carve(wa, rows, kv_rows, bhs, kv_layers);
  wa.take<float>(rows * kH);
  wa.take<float>(rows * kH);
  return wa.off;
}

}  // namespace etp

using namespace etp;
#define ETP_API __attribute__((visibility("default")))
static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

ETP_API size_t etp_nav_bwd_work_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers) {
  return work_bytes_for(static_cast<size_t>(B) * N, static_cast<size_t>(B) * L, static_cast<size_t>(B) * kHeads * (N > L ? N : L),
                        num_x_layers > 0 ? num_x_layers : 1);
}
ETP_API size_t etp_text_kv_bwd_work_bytes(int32_t B, int32_t L, int32_t num_x_layers) {
  Arena wa(nullptr, ~size_t(0));
  const size_t rows = static_cast<size_t>(B) * L;
  wa.take<bf16>(rows * 2 * kH * (num_x_layers > 0 ? num_x_layers : 1));
  wa.take<bf16>(rows * kH);
  return wa.off;
}
ETP_API size_t etp_pano_bwd_work_bytes(int32_t B, int32_t V) {
  return work_bytes_for(static_cast<size_t>(B) * V, 0, static_cast<size_t>(B) * kHeads * V);
}
ETP_API size_t etp_txt_bwd_work_bytes(int32_t B, int32_t L) {
  return work_bytes_for(static_cast<size_t>(B) * L, 0, static_cast<size_t>(B) * kHeads * L);
}

ETP_API size_t etp_l2v_bwd_work_bytes(int32_t B, int32_t N, int32_t L, int32_t num_x_layers) {
  return work_bytes_for(static_cast<size_t>(B) * L, static_cast<size_t>(B) * N, static_cast<size_t>(B) * kHeads * (N > L ? N : L),
                        num_x_layers > 0 ? num_x_layers : 1);
}
ETP_API int etp_backward_lang2visn(const etp_nav_weights* w, const etp_nav_weights* grads, const etp_nav_inputs* in,
                                   const float* d_lang_embeds, void* saved, size_t saved_bytes, void* work,
                                   size_t work_bytes, float* d_txt_embeds, float* d_gmap_img_fts, void* stream) {
  ETP_REQUIRE(w && grads && in && d_lang_embeds && saved && work, "etp_backward_lang2visn: null argument");
  return backward_lang2visn(*w, *grads, *in, d_lang_embeds, saved, saved_bytes, work, work_bytes, d_txt_embeds,
                            d_gmap_img_fts, S(stream));
}

ETP_API int etp_backward_navigation(const etp_nav_weights* w, const etp_nav_weights* grads, const etp_nav_inputs* in,
                                    const float* d_gmap_embeds, const float* d_global_logits, void* saved,
                                    size_t saved_bytes, void* work, size_t work_bytes, float* d_txt_embeds,
                                    float* d_gmap_img_fts, void* stream) {
  ETP_REQUIRE(w && grads && in && saved && work, "etp_backward_navigation: null argument");
  return backward_navigation(*w, *grads, *in, d_gmap_embeds, d_global_logits, saved, saved_bytes, work, work_bytes,
                             d_txt_embeds, d_gmap_img_fts, S(stream));
}
ETP_API int etp_backward_text_kv(const etp_nav_weights* w, const etp_nav_weights* grads, const float* txt_embeds,
                                 const void* txt_embeds_bf16, int32_t B, int32_t L, const float* dkv_acc, float* d_txt_embeds,
                                 void* work, void* stream) {
  ETP_REQUIRE(w && grads && dkv_acc && work && (txt_embeds || txt_embeds_bf16), "etp_backward_text_kv: null argument");
  return backward_text_kv(*w, *grads, txt_embeds, static_cast<const bf16*>(txt_embeds_bf16), B, L, dkv_acc, d_txt_embeds,
                          work, S(stream));
}
ETP_API int etp_backward_panorama(const etp_pano_weights* w, const etp_pano_weights* grads, const etp_pano_inputs* in,
                                  const uint8_t* pano_masks, const float* d_pano_embeds, void* saved, size_t saved_bytes,
                                  void* work, size_t work_bytes, float* d_rgb_fts, float* d_dep_fts, void* stream) {
  ETP_REQUIRE(w && grads && in && pano_masks && d_pano_embeds && saved && work, "etp_backward_panorama: null argument");
  return backward_panorama(*w, *grads, *in, pano_masks, d_pano_embeds, saved, saved_bytes, work, work_bytes, d_rgb_fts,
                           d_dep_fts, S(stream));
}
ETP_API int etp_backward_txt(const etp_txt_weights* w, const etp_txt_weights* grads, const int64_t* txt_ids,
                             const uint8_t* txt_masks, int32_t B, int32_t L, const float* d_txt_embeds, void* saved,
                             size_t saved_bytes, void* work, size_t work_bytes, void* stream, const etp_dropout* dropout) {
  ETP_REQUIRE(w && grads && txt_ids && txt_masks && d_txt_embeds && saved && work, "etp_backward_txt: null argument");
  return backward_txt(*w, *grads, txt_ids, txt_masks, B, L, d_txt_embeds, saved, saved_bytes, work, work_bytes, S(stream),
                      dropout);
}

ETP_API int etp_adamw_step(float* param, void* param_bf16, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                           float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step, float grad_scale,
                           void* stream) {
  return adamw_step(param, static_cast<bf16*>(param_bf16), grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                    step, grad_scale, S(stream));
}

/* AdamW with per-block flags (one byte per 64 elements: bit 0 trainable, bit 1 weight decay; NULL = all set) and optional
 * global-norm clipping: normsq = device scalar with sum g^2 (etp_grad_sumsq), max_norm <= 0 disables it. */
ETP_API int etp_adamw_step_ex(float* param, void* param_bf16, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                              float lr, float beta1, float beta2, float eps, float weight_decay, int32_t step,
                              float grad_scale, const uint8_t* flags, const float* normsq, float max_norm, void* stream) {
  return adamw_step(param, static_cast<bf16*>(param_bf16), grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, weight_decay,
                    step, grad_scale, S(stream), flags, normsq, max_norm);
}
ETP_API void etp_set_adamw_ctas_per_sm(int32_t n) { set_adamw_ctas_per_sm(n); }
ETP_API int etp_grad_sumsq(const float* grad, int64_t n, const uint8_t* flags, float* out, void* stream) {
  return grad_sumsq(grad, n, flags, out, S(stream));
}

}  // extern "C"
