// Step-level host sequencing: one C-ABI call = one method of the reference planner
// (GlocalTextPathNavCMT.forward_txt / forward_panorama / forward_navigation, vilmodel_cmt.py:684,690,721).
// Pure launch code: every op is one of the kernels in gemm.cu / attention*.cu / elementwise.cu / pack.cu,
// issued back-to-back on the caller's stream with no host synchronisation, so a whole step can be
// captured in a CUDA graph by the host.  Activations that the backward pass needs are laid out in a
// caller-owned "saved" record (layout = the *Record structs below, identical for forward and backward).
#include "../../include/etpnav_b200.h"
#include "planner.h"

namespace etp {

// ---------------------------------------------------------------------------------------------------
// saved-activation records
// ---------------------------------------------------------------------------------------------------
void LayerRecord::carve(Arena& ar, int rows, int kv_rows, int B, int Sq, bool cross) {
  const size_t r = rows;
  if (cross) {
    q = ar.take<bf16>(r * kH);
    if (kv_rows > 0) { kv = ar.take<bf16>(static_cast<size_t>(kv_rows) * 2 * kH); ldkv = 2 * kH; }
    ctx1 = ar.take<bf16>(r * kH);
    lse1 = ar.take<float>(static_cast<size_t>(B) * kHeads * Sq);
    t1 = ar.take<float>(r * kH);
    st1 = ar.take<float>(r * 2);
    ab = ar.take<bf16>(r * kH);
  }
  qkv = ar.take<bf16>(r * 3 * kH);
  ctx2 = ar.take<bf16>(r * kH);
  lse2 = ar.take<float>(static_cast<size_t>(B) * kHeads * Sq);
  t2 = ar.take<float>(r * kH);
  st2 = ar.take<float>(r * 2);
  cb = ar.take<bf16>(r * kH);
  pre = ar.take<bf16>(r * kI);
  h = ar.take<bf16>(r * kI);
  t3 = ar.take<float>(r * kH);
  st3 = ar.take<float>(r * 2);
  xb = ar.take<bf16>(r * kH);
}

void NavRecord::carve(Arena& ar, int B, int N, int L, int X, bool training, bool txt_cached) {
  const size_t rows = static_cast<size_t>(B) * N;
  if (!txt_cached) {
    txtb = ar.take<bf16>(static_cast<size_t>(B) * L * kH);
    kv_all = ar.take<bf16>(static_cast<size_t>(B) * L * 2 * kH * (X > 0 ? X : 1));
  }
  x0b = ar.take<bf16>(rows * kH);
  pos_lin = ar.take<float>(rows * kH);
  pos_stats = ar.take<float>(rows * 2);
  xa = ar.take<float>(rows * kH);
  xc = ar.take<float>(rows * kH);
  xf = ar.take<float>(rows * kH);
  relu = ar.take<float>(rows * kH);
  sap_stats = ar.take<float>(rows * 2);
  layers.resize(X);
  const size_t mark = ar.off;
  for (int i = 0; i < X; ++i) {
    if (!training) ar.off = mark;  // inference: all layers alias one scratch record
    layers[i].carve(ar, static_cast<int>(rows), 0, B, N, true);
    if (kv_all) layers[i].kv = kv_all + static_cast<size_t>(i) * 2 * kH;  // slice of the all-layer K|V buffer
    layers[i].ldkv = X * 2 * kH;
  }
}

void L2VRecord::carve(Arena& ar, int B, int N, int L, int X, bool training) {
  const size_t rows = static_cast<size_t>(B) * L, nrows = static_cast<size_t>(B) * N;
  nodeb = ar.take<bf16>(nrows * kH);
  pos_lin = ar.take<float>(nrows * kH);
  pos_stats = ar.take<float>(nrows * 2);
  nodef = ar.take<float>(nrows * kH);
  kv_all = ar.take<bf16>(nrows * 2 * kH * (X > 0 ? X : 1));
  txtb = ar.take<bf16>(rows * kH);
  xa = ar.take<float>(rows * kH);
  xc = ar.take<float>(rows * kH);
  xf = ar.take<float>(rows * kH);
  layers.resize(X);
  const size_t mark = ar.off;
  for (int i = 0; i < X; ++i) {
    if (!training) ar.off = mark;
    layers[i].carve(ar, static_cast<int>(rows), 0, B, L, true);
    layers[i].kv = kv_all + static_cast<size_t>(i) * 2 * kH;
    layers[i].ldkv = X * 2 * kH;
  }
}

void PanoRecord::carve(Arena& ar, int B, int V, int P, bool training) {
  const size_t rows = static_cast<size_t>(B) * V;
  rgbb = ar.take<bf16>(rows * 512);
  depb = ar.take<bf16>(rows * 128);
  rgb_lin = ar.take<float>(rows * kH);
  dep_lin = ar.take<float>(rows * kH);
  loc_lin = ar.take<float>(rows * kH);
  sum_pre = ar.take<float>(rows * kH);
  stats = ar.take<float>(rows * 8);
  xs.resize(2 * P + 1);
  for (auto& p : xs) p = ar.take<float>(rows * kH);
  fin_stats = ar.take<float>(rows * 2);
  layers.resize(P);
  const size_t mark = ar.off;
  for (int i = 0; i < P; ++i) {
    if (!training) ar.off = mark;
    auto& l = layers[i];
    l.y1b = ar.take<bf16>(rows * kH);
    l.st1 = ar.take<float>(rows * 2);
    l.qkv = ar.take<bf16>(rows * 3 * kH);
    l.ctx = ar.take<bf16>(rows * kH);
    l.lse = ar.take<float>(static_cast<size_t>(B) * kHeads * V);
    l.y2b = ar.take<bf16>(rows * kH);
    l.st2 = ar.take<float>(rows * 2);
    l.pre = ar.take<bf16>(rows * kI);
    l.h = ar.take<bf16>(rows * kI);
  }
}

void TxtRecord::carve(Arena& ar, int B, int L, int NL, bool training) {
  const size_t rows = static_cast<size_t>(B) * L;
  sum_pre = ar.take<float>(rows * kH);
  emb_stats = ar.take<float>(rows * 2);
  x0b = ar.take<bf16>(rows * kH);
  xa = ar.take<float>(rows * kH);
  xc = ar.take<float>(rows * kH);
  layers.resize(NL);
  const size_t mark = ar.off;
  for (int i = 0; i < NL; ++i) {
    if (!training) ar.off = mark;
    layers[i].carve(ar, static_cast<int>(rows), 0, B, L, false);
  }
}

// ---------------------------------------------------------------------------------------------------
// building blocks
// ---------------------------------------------------------------------------------------------------
// out = A[rows,K] . W[N,K]^T + bias  with the usual epilogue options
static int linear(const bf16* A, int rows, int K, const void* W, int N, const float* bias, int act, const float* resid,
                  float* out_f32, bf16* out_bf16, bf16* out_dact, cudaStream_t s, DropHost drop = DropHost{0u, 0u, 1.0f}) {
  GemmArgs g;
  g.M = rows; g.N = N; g.K = K;
  g.A = A; g.lda = K;
  g.B = static_cast<const bf16*>(W); g.ldb = K;
  g.bias = bias; g.act = act;
  g.resid = resid; g.ld_resid = N;
  g.out_f32 = out_f32; g.ld_f32 = N;
  g.out_bf16 = out_bf16; g.ld_bf16 = N;
  g.out_pre = out_dact; g.ld_pre = N; g.pre_mode = out_dact ? 1 : 0;  // saved for backward: gelu'(pre-activation)
  g.drop_key = drop.key; g.drop_thr = drop.thr; g.drop_scale = drop.scale;
  return gemm(g, s);
}

#define ETP_TRY(expr)            \
  do {                           \
    int _rc = (expr);            \
    if (_rc != ETP_OK) return _rc; \
  } while (0)

// self-attention + FFN half of a post-LN block (BertAttention + BertIntermediate + BertOutput,
// vilmodel_cmt.py:156-193): in = (a_f32, a_bf16) -> out x (fp32 into x_out, bf16 into rec.xb)
static int self_ffn_block(const etp_layer_weights& w, float eps, LayerRecord& rec, const float* a_f32, const bf16* a_bf16,
                          int B, int S, const uint8_t* key_valid, const float* pair, const float* pair_w,
                          const float* pair_b, float* c_f32, float* x_out, bool training, cudaStream_t s,
                          const DropCtx& dc, uint32_t site_base, int layer) {
  const int rows = B * S;
  ETP_TRY(linear(a_bf16, rows, kH, w.sqkv_w, 3 * kH, w.sqkv_b, 0, nullptr, nullptr, rec.qkv, nullptr, s));
  AttnArgs at;
  at.B = B; at.heads = kHeads; at.Sq = S; at.Sk = S;
  at.q = rec.qkv; at.ldq = 3 * kH;
  at.k = rec.qkv + kH; at.ldk = 3 * kH;
  at.v = rec.qkv + 2 * kH; at.ldv = 3 * kH;
  at.scale = 0.125f; at.key_valid = key_valid; at.mask_value = -10000.0f;
  at.pair = pair; at.pair_w_dev = pair_w; at.pair_b_dev = pair_b;
  at.out = rec.ctx2; at.ldo = kH; at.lse = rec.lse2;
  {
    const DropHost d = dc.attn(drop_site(site_base, layer, kDropSAttn));
    at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
  }
  ETP_TRY(attention_dispatch(at, s));
  ETP_TRY(linear(rec.ctx2, rows, kH, w.so_w, kH, w.so_b, 0, a_f32, rec.t2, nullptr, nullptr, s,
                 dc.hidden(drop_site(site_base, layer, kDropSOut))));
  ETP_TRY(layernorm_fwd(rec.t2, w.sln_g, w.sln_b, eps, rows, kH, c_f32, rec.cb, rec.st2, rec.st2 + rows, s));
  ETP_TRY(linear(rec.cb, rows, kH, w.f1_w, kI, w.f1_b, 1, nullptr, nullptr, rec.h, training ? rec.pre : nullptr, s));
  ETP_TRY(linear(rec.h, rows, kI, w.f2_w, kH, w.f2_b, 0, c_f32, rec.t3, nullptr, nullptr, s,
                 dc.hidden(drop_site(site_base, layer, kDropFfnOut))));
  ETP_TRY(layernorm_fwd(rec.t3, w.fln_g, w.fln_b, eps, rows, kH, x_out, rec.xb, rec.st3, rec.st3 + rows, s));
  return ETP_OK;
}

int forward_navigation(const etp_nav_weights& w, const etp_nav_inputs& in, float* gmap_embeds, float* global_logits,
                       void* saved, size_t saved_bytes, bool training, cudaStream_t s) {
  const int B = in.B, N = in.N, L = in.L, X = w.num_x_layers;
  ETP_REQUIRE(B > 0 && N > 0 && L > 0 && X >= 0, "forward_navigation: bad shape");
  ETP_REQUIRE(N <= 1024 && L <= 1024, "forward_navigation: at most 1024 nodes / tokens");
  const bf16* kv_cache = static_cast<const bf16*>(in.txt_kv_all);
  if (kv_cache) {
    ETP_REQUIRE(X > 0, "forward_navigation: a text K|V cache needs at least one x-layer");
    ETP_REQUIRE(in.txt_kv_rows == nullptr || in.txt_kv_batch > 0, "forward_navigation: txt_kv_batch must be given with txt_kv_rows");
  }
  // with the cache the record has no text-side part: the backward reads K|V from the cache and hands dK|dV to the
  // caller's accumulator (etp_nav_inputs.txt_kv_grad), whose one weight / data gradient runs after the rollout
  Arena ar(saved, saved_bytes);
  NavRecord rec;
  rec.carve(ar, B, N, L, X, training, kv_cache != nullptr);
  ETP_REQUIRE(ar.off <= saved_bytes, "forward_navigation: saved buffer too small");
  const int rows = B * N;
  DropCtx dc;
  if (in.dropout) { dc.seed = in.dropout->seed; dc.p_hidden = in.dropout->p_hidden; dc.p_attn = in.dropout->p_attn; dc.p_head = in.dropout->p_head; }

  const bf16* txtb = static_cast<const bf16*>(in.txt_embeds_bf16);
  if (txtb == nullptr && kv_cache == nullptr) {
    ETP_REQUIRE(in.txt_embeds != nullptr, "forward_navigation: txt_embeds (fp32) or txt_embeds_bf16 is required");
    ETP_TRY(cast_f32_to_bf16(in.txt_embeds, rec.txtb, static_cast<int64_t>(B) * L * kH, s));
    txtb = rec.txtb;
  }
  // text K|V of every layer in ONE GEMM: [B*L,768] x [X*1536,768]^T (they depend only on txt_embeds).  Issued FIRST: it is
  // the one node-independent GEMM of the call, so a host may still be producing gmap_img_fts on another stream
  // (img_ready_event) while it runs, on the SMs side_sm_reserve leaves to that stream.
  if (X > 0 && kv_cache == nullptr) {
    const int prev = get_sm_reserve();
    if (in.side_sm_reserve > 0) set_sm_reserve(prev + in.side_sm_reserve);
    const int rc = linear(txtb, B * L, kH, w.xkv_all_w, X * 2 * kH, w.xkv_all_b, 0, nullptr, nullptr, rec.kv_all, nullptr, s);
    set_sm_reserve(prev);
    ETP_TRY(rc);
  }
  if (in.img_ready_event) ETP_CHECK_CUDA(cudaStreamWaitEvent(s, static_cast<cudaEvent_t>(in.img_ready_event), 0));
  NodePackArgs np;
  np.rows = rows; np.img_fts = in.gmap_img_fts; np.step_ids = in.gmap_step_ids; np.pos_fts = in.gmap_pos_fts;
  np.pos_w = w.pos_w; np.pos_b = w.pos_b; np.pos_g = w.pos_g; np.pos_bb = w.pos_bb; np.step_emb = w.step_emb;
  np.x_f32 = X > 0 ? rec.xf : gmap_embeds; np.x_bf16 = rec.x0b;
  np.pos_lin = training ? rec.pos_lin : nullptr; np.stats = rec.pos_stats;
  ETP_TRY(node_pack_fwd(np, s));
  const float* x_f32 = np.x_f32;
  const bf16* x_bf16 = rec.x0b;
  for (int i = 0; i < X; ++i) {
    const etp_layer_weights& lw = w.layers[i];
    LayerRecord& r = rec.layers[i];
    // cross-attention: nodes query the instruction (BertXAttention, vilmodel_cmt.py:354-363,325-352)
    ETP_TRY(linear(x_bf16, rows, kH, lw.xq_w, kH, lw.xq_b, 0, nullptr, nullptr, r.q, nullptr, s));
    AttnArgs at;
    at.B = B; at.heads = kHeads; at.Sq = N; at.Sk = L;
    at.q = r.q; at.ldq = kH;
    at.k = r.kv; at.ldk = r.ldkv;
    at.v = r.kv + kH; at.ldv = r.ldkv;
    if (kv_cache) {   // episode-level cache: layer i's slice of the cached [., X*1536] rows, read through the batch-row map
      at.k = kv_cache + static_cast<size_t>(i) * 2 * kH; at.v = at.k + kH;
      at.ldk = at.ldv = X * 2 * kH;
      at.kv_rows = in.txt_kv_rows; at.kv_B = in.txt_kv_rows ? in.txt_kv_batch : B;
    }
    at.scale = 0.125f; at.key_valid = in.txt_masks; at.mask_value = -10000.0f;
    at.out = r.ctx1; at.ldo = kH; at.lse = r.lse1;
    {
      const DropHost d = dc.attn(drop_site(kSiteNav, i, kDropXAttn));
      at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
    }
    ETP_TRY(attention_dispatch(at, s));
    ETP_TRY(linear(r.ctx1, rows, kH, lw.xo_w, kH, lw.xo_b, 0, x_f32, r.t1, nullptr, nullptr, s,
                   dc.hidden(drop_site(kSiteNav, i, kDropXOut))));
    ETP_TRY(layernorm_fwd(r.t1, lw.xln_g, lw.xln_b, w.ln_eps, rows, kH, rec.xa, r.ab, r.st1, r.st1 + rows, s));
    // graph-aware self-attention + FFN (vilmodel_cmt.py:391-396)
    float* x_out = (i == X - 1) ? gmap_embeds : rec.xf;
    ETP_TRY(self_ffn_block(lw, w.ln_eps, r, rec.xa, r.ab, B, N, in.gmap_masks, w.sprel_w ? in.gmap_pair_dists : nullptr,
                           w.sprel_w, w.sprel_b, rec.xc, x_out, training, s, dc, kSiteNav, i));
    x_f32 = x_out;
    x_bf16 = r.xb;
  }
  // SAP head (NextActionPrediction, vilmodel_cmt.py:651-661) + masking (:743-744)
  ETP_TRY(linear(x_bf16, rows, kH, w.sap0_w, kH, w.sap0_b, 2, nullptr, rec.relu, nullptr, nullptr, s));
  ETP_TRY(sap_tail_fwd(rec.relu, w.sap_g, w.sap_bb, w.sap4_w, w.sap4_b, in.gmap_visited_masks, in.gmap_masks, rows, kH,
                       global_logits, rec.sap_stats, rec.sap_stats + rows, s, dc.head(kSiteNav + kSiteHead)));
  return ETP_OK;
}

int forward_panorama(const etp_pano_weights& w, const etp_pano_inputs& in, float* pano_embeds, uint8_t* pano_masks,
                     void* saved, size_t saved_bytes, bool training, cudaStream_t s) {
  const int B = in.B, V = in.V, P = w.num_pano_layers;
  ETP_REQUIRE(B > 0 && V > 0 && P >= 0, "forward_panorama: bad shape");
  Arena ar(saved, saved_bytes);
  PanoRecord rec;
  rec.carve(ar, B, V, P, training);
  ETP_REQUIRE(ar.off <= saved_bytes, "forward_panorama: saved buffer too small");
  const int rows = B * V;
  DropCtx dc;
  if (in.dropout) { dc.seed = in.dropout->seed; dc.p_hidden = in.dropout->p_hidden; dc.p_attn = in.dropout->p_attn; dc.p_head = in.dropout->p_head; }
  ETP_TRY(seq_mask(in.view_lens, B, V, pano_masks, s));
  ETP_TRY(cast_f32_to_bf16(in.rgb_fts, rec.rgbb, static_cast<int64_t>(rows) * 512, s));
  ETP_TRY(linear(rec.rgbb, rows, 512, w.img_w, kH, w.img_b, 0, nullptr, rec.rgb_lin, nullptr, nullptr, s));
  if (w.dep_w) {
    ETP_TRY(cast_f32_to_bf16(in.dep_fts, rec.depb, static_cast<int64_t>(rows) * 128, s));
    ETP_TRY(linear(rec.depb, rows, 128, w.dep_w, kH, w.dep_b, 0, nullptr, rec.dep_lin, nullptr, nullptr, s));
  }
  float* x = (P == 0) ? pano_embeds : rec.xs[0];
  PanoPackArgs pp;
  pp.rows = rows; pp.rgb_lin = rec.rgb_lin; pp.dep_lin = w.dep_w ? rec.dep_lin : nullptr; pp.loc_fts = in.loc_fts;
  pp.nav_types = in.nav_types; pp.loc_w = w.loc_w; pp.loc_b = w.loc_b;
  pp.img_g = w.img_g; pp.img_b = w.img_bb; pp.dep_g = w.dep_g; pp.dep_b = w.dep_bb; pp.loc_g = w.loc_g; pp.loc_bb = w.loc_bb;
  pp.out_g = w.out_g; pp.out_b = w.out_bb; pp.nav_emb = w.nav_emb; pp.tok_emb1 = w.tok_emb1;
  pp.x_f32 = x; pp.loc_lin = training ? rec.loc_lin : nullptr; pp.sum_pre = training ? rec.sum_pre : nullptr;
  pp.stats = rec.stats;
  pp.drop = dc.hidden(kSitePano + kSiteEmbed);
  ETP_TRY(pano_pack_fwd(pp, s));
  // pre-norm encoder layers (TransformerEncoderLayer.forward_pre, common/transformer.py:170-182)
  for (int i = 0; i < P; ++i) {
    const etp_pano_layer_weights& lw = w.layers[i];
    auto& r = rec.layers[i];
    float* x_mid = rec.xs[2 * i + 1];
    float* x_out = rec.xs[2 * i + 2];
    ETP_TRY(layernorm_fwd(x, lw.n1_g, lw.n1_b, w.layer_eps, rows, kH, nullptr, r.y1b, r.st1, r.st1 + rows, s));
    ETP_TRY(linear(r.y1b, rows, kH, lw.in_w, 3 * kH, lw.in_b, 0, nullptr, nullptr, r.qkv, nullptr, s));
    AttnArgs at;
    at.B = B; at.heads = kHeads; at.Sq = V; at.Sk = V;
    at.q = r.qkv; at.ldq = 3 * kH; at.k = r.qkv + kH; at.ldk = 3 * kH; at.v = r.qkv + 2 * kH; at.ldv = 3 * kH;
    at.scale = 0.125f; at.key_valid = pano_masks; at.mask_value = -INFINITY;
    at.out = r.ctx; at.ldo = kH; at.lse = r.lse;
    {
      const DropHost d = dc.hidden(drop_site(kSitePano, i, kDropPAttn));  // MHA dropout = hidden_dropout_prob (common/ops.py:15)
      at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
    }
    ETP_TRY(attention_fwd(at, s));  // <= 16 views: CUDA-core kernel
    ETP_TRY(linear(r.ctx, rows, kH, lw.out_w, kH, lw.out_b, 0, x, x_mid, nullptr, nullptr, s,
                   dc.hidden(drop_site(kSitePano, i, kDropPOut))));
    ETP_TRY(layernorm_fwd(x_mid, lw.n2_g, lw.n2_b, w.layer_eps, rows, kH, nullptr, r.y2b, r.st2, r.st2 + rows, s));
    // dropout(gelu(.)) inside the FFN (transformer.py:180): the saved derivative carries the same mask
    ETP_TRY(linear(r.y2b, rows, kH, lw.l1_w, kI, lw.l1_b, 1, nullptr, nullptr, r.h, training ? r.pre : nullptr, s,
                   dc.hidden(drop_site(kSitePano, i, kDropPFfn))));
    ETP_TRY(linear(r.h, rows, kI, lw.l2_w, kH, lw.l2_b, 0, x_mid, x_out, nullptr, nullptr, s,
                   dc.hidden(drop_site(kSitePano, i, kDropPFfnOut))));
    x = x_out;
  }
  if (P > 0)
    ETP_TRY(layernorm_fwd(x, w.fin_g, w.fin_b, 1e-12f, rows, kH, pano_embeds, nullptr, rec.fin_stats, rec.fin_stats + rows, s));
  return ETP_OK;
}

int forward_txt(const etp_txt_weights& w, const int64_t* txt_ids, const uint8_t* txt_masks, int B, int L,
                float* txt_embeds, void* saved, size_t saved_bytes, bool training, cudaStream_t s, const etp_dropout* dropout) {
  DropCtx dc;
  if (dropout) { dc.seed = dropout->seed; dc.p_hidden = dropout->p_hidden; dc.p_attn = dropout->p_attn; dc.p_head = dropout->p_head; }
  const int NL = w.num_l_layers;
  ETP_REQUIRE(B > 0 && L > 0 && NL >= 0, "forward_txt: bad shape");
  ETP_REQUIRE(L <= 1024, "forward_txt: at most 1024 tokens");
  Arena ar(saved, saved_bytes);
  TxtRecord rec;
  rec.carve(ar, B, L, NL, training);
  ETP_REQUIRE(ar.off <= saved_bytes, "forward_txt: saved buffer too small");
  float* x = NL > 0 ? rec.xa : txt_embeds;
  ETP_TRY(embed_txt_fwd(txt_ids, w.word_emb, w.pos_emb, w.type_emb0, w.emb_g, w.emb_b, w.ln_eps, B, L, x, rec.x0b,
                        training ? rec.sum_pre : nullptr, rec.emb_stats, s, dc.hidden(kSiteTxt + kSiteEmbed)));
  const bf16* xb = rec.x0b;
  for (int i = 0; i < NL; ++i) {
    float* x_out = (i == NL - 1) ? txt_embeds : rec.xa;
    // BertLayer.forward (vilmodel_cmt.py:202-208): self-attention over tokens + FFN.  In-place on xa is safe:
    // the block reads a_f32 only as the residual of the first GEMM, before x_out is written.
    ETP_TRY(self_ffn_block(w.layers[i], w.ln_eps, rec.layers[i], x, xb, B, L, txt_masks, nullptr, nullptr, nullptr,
                           rec.xc, x_out, training, s, dc, kSiteTxt, i));
    x = x_out;
    xb = rec.layers[i].xb;
  }
  return ETP_OK;
}

// GlocalTextPathCMT.forward_mlm's cross-modal part (pretrain_src/pretrain_src/model/vilmodel.py:733-741): node packing
// (gmap_input_embedding, :621-632) then, per x-layer, GraphLXRTXLayer.forward_lang2visn (:400-411): tokens query the
// nodes through visual_attention, lang_self_att over the tokens, lang_inter / lang_output.  The node K|V of every
// layer depend only on the packed nodes, so they come out of one GEMM, like the text K|V of forward_navigation.
int forward_lang2visn(const etp_nav_weights& w, const etp_nav_inputs& in, float* lang_embeds, void* saved,
                      size_t saved_bytes, bool training, cudaStream_t s) {
  const int B = in.B, N = in.N, L = in.L, X = w.num_x_layers;
  ETP_REQUIRE(B > 0 && N > 0 && L > 0 && X >= 1, "forward_lang2visn: bad shape");
  ETP_REQUIRE(N <= 1024 && L <= 1024, "forward_lang2visn: at most 1024 nodes / tokens");
  ETP_REQUIRE(in.txt_embeds != nullptr, "forward_lang2visn: fp32 txt_embeds required (the tokens are the residual stream)");
  Arena ar(saved, saved_bytes);
  L2VRecord rec;
  rec.carve(ar, B, N, L, X, training);
  ETP_REQUIRE(ar.off <= saved_bytes, "forward_lang2visn: saved buffer too small");
  const int rows = B * L, nrows = B * N;
  DropCtx dc;
  if (in.dropout) { dc.seed = in.dropout->seed; dc.p_hidden = in.dropout->p_hidden; dc.p_attn = in.dropout->p_attn; dc.p_head = in.dropout->p_head; }

  NodePackArgs np;
  np.rows = nrows; np.img_fts = in.gmap_img_fts; np.step_ids = in.gmap_step_ids; np.pos_fts = in.gmap_pos_fts;
  np.pos_w = w.pos_w; np.pos_b = w.pos_b; np.pos_g = w.pos_g; np.pos_bb = w.pos_bb; np.step_emb = w.step_emb;
  np.x_f32 = rec.nodef; np.x_bf16 = rec.nodeb;
  np.pos_lin = training ? rec.pos_lin : nullptr; np.stats = rec.pos_stats;
  ETP_TRY(node_pack_fwd(np, s));
  ETP_TRY(cast_f32_to_bf16(in.txt_embeds, rec.txtb, static_cast<int64_t>(rows) * kH, s));
  ETP_TRY(linear(rec.nodeb, nrows, kH, w.xkv_all_w, X * 2 * kH, w.xkv_all_b, 0, nullptr, nullptr, rec.kv_all, nullptr, s));
  const float* x_f32 = in.txt_embeds;
  const bf16* x_bf16 = rec.txtb;
  for (int i = 0; i < X; ++i) {
    const etp_layer_weights& lw = w.layers[i];
    LayerRecord& r = rec.layers[i];
    ETP_TRY(linear(x_bf16, rows, kH, lw.xq_w, kH, lw.xq_b, 0, nullptr, nullptr, r.q, nullptr, s));
    AttnArgs at;
    at.B = B; at.heads = kHeads; at.Sq = L; at.Sk = N;
    at.q = r.q; at.ldq = kH;
    at.k = r.kv; at.ldk = r.ldkv;
    at.v = r.kv + kH; at.ldv = r.ldkv;
    at.scale = 0.125f; at.key_valid = in.gmap_masks; at.mask_value = -10000.0f;
    at.out = r.ctx1; at.ldo = kH; at.lse = r.lse1;
    {
      const DropHost d = dc.attn(drop_site(kSiteL2V, i, kDropXAttn));
      at.drop_key = d.key; at.drop_thr = d.thr; at.drop_scale = d.scale;
    }
    ETP_TRY(attention_dispatch(at, s));
    ETP_TRY(linear(r.ctx1, rows, kH, lw.xo_w, kH, lw.xo_b, 0, x_f32, r.t1, nullptr, nullptr, s,
                   dc.hidden(drop_site(kSiteL2V, i, kDropXOut))));
    ETP_TRY(layernorm_fwd(r.t1, lw.xln_g, lw.xln_b, w.ln_eps, rows, kH, rec.xa, r.ab, r.st1, r.st1 + rows, s));
    float* x_out = (i == X - 1) ? lang_embeds : rec.xf;
    ETP_TRY(self_ffn_block(lw, w.ln_eps, r, rec.xa, r.ab, B, L, in.txt_masks, nullptr, nullptr, nullptr, rec.xc, x_out,
                           training, s, dc, kSiteL2V, i));
    x_f32 = x_out;
    x_bf16 = r.xb;
  }
  return ETP_OK;
}

static size_t record_bytes_nav(int B, int N, int L, int X, bool training, bool txt_cached) {
  Arena ar(nullptr, ~size_t(0));
  NavRecord r;
  r.carve(ar, B, N, L, X, training, txt_cached);
  return ar.off;
}

}  // namespace etp

using namespace etp;
#define ETP_API __attribute__((visibility("default")))
static inline cudaStream_t S(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

ETP_API size_t etp_nav_saved_bytes(int32_t B, int32_t N, int32_t L, int32_t X, int32_t training) {
  return record_bytes_nav(B, N, L, X, training != 0, false);
}
ETP_API size_t etp_nav_kv_saved_bytes(int32_t B, int32_t N, int32_t L, int32_t X, int32_t training) {
  return record_bytes_nav(B, N, L, X, training != 0, true);
}
ETP_API size_t etp_pano_saved_bytes(int32_t B, int32_t V, int32_t P, int32_t training) {
  Arena ar(nullptr, ~size_t(0));
  PanoRecord r;
  r.carve(ar, B, V, P, training != 0);
  return ar.off;
}
ETP_API size_t etp_txt_saved_bytes(int32_t B, int32_t L, int32_t NL, int32_t training) {
  Arena ar(nullptr, ~size_t(0));
  TxtRecord r;
  r.carve(ar, B, L, NL, training != 0);
  return ar.off;
}

ETP_API size_t etp_l2v_saved_bytes(int32_t B, int32_t N, int32_t L, int32_t X, int32_t training) {
  Arena ar(nullptr, ~size_t(0));
  L2VRecord r;
  r.carve(ar, B, N, L, X, training != 0);
  return ar.off;
}
ETP_API int etp_forward_lang2visn(const etp_nav_weights* w, const etp_nav_inputs* in, float* lang_embeds, void* saved,
                                  size_t saved_bytes, int32_t training, void* stream) {
  ETP_REQUIRE(w && in && lang_embeds && saved, "etp_forward_lang2visn: null argument");
  return forward_lang2visn(*w, *in, lang_embeds, saved, saved_bytes, training != 0, S(stream));
}

ETP_API int etp_forward_navigation(const etp_nav_weights* w, const etp_nav_inputs* in, float* gmap_embeds,
                                   float* global_logits, void* saved, size_t saved_bytes, int32_t training, void* stream) {
  ETP_REQUIRE(w && in && gmap_embeds && global_logits && saved, "etp_forward_navigation: null argument");
  return forward_navigation(*w, *in, gmap_embeds, global_logits, saved, saved_bytes, training != 0, S(stream));
}
ETP_API int etp_encode_text_kv(const etp_nav_weights* w, const float* txt_embeds, const void* txt_embeds_bf16, int32_t B,
                               int32_t L, void* kv_all, void* work, void* stream) {
  ETP_REQUIRE(w && kv_all && (txt_embeds || txt_embeds_bf16), "etp_encode_text_kv: null argument");
  ETP_REQUIRE(B > 0 && L > 0 && w->num_x_layers > 0, "etp_encode_text_kv: bad shape");
  const bf16* tb = static_cast<const bf16*>(txt_embeds_bf16);
  if (tb == nullptr) {
    ETP_REQUIRE(work != nullptr, "etp_encode_text_kv: scratch needed for the fp32 input");
    ETP_TRY(cast_f32_to_bf16(txt_embeds, static_cast<bf16*>(work), static_cast<int64_t>(B) * L * kH, S(stream)));
    tb = static_cast<const bf16*>(work);
  }
  return linear(tb, B * L, kH, w->xkv_all_w, w->num_x_layers * 2 * kH, w->xkv_all_b, 0, nullptr, nullptr,
                static_cast<bf16*>(kv_all), nullptr, S(stream));
}

ETP_API int etp_forward_panorama(const etp_pano_weights* w, const etp_pano_inputs* in, float* pano_embeds,
                                 uint8_t* pano_masks, void* saved, size_t saved_bytes, int32_t training, void* stream) {
  ETP_REQUIRE(w && in && pano_embeds && pano_masks && saved, "etp_forward_panorama: null argument");
  return forward_panorama(*w, *in, pano_embeds, pano_masks, saved, saved_bytes, training != 0, S(stream));
}
ETP_API int etp_forward_txt(const etp_txt_weights* w, const int64_t* txt_ids, const uint8_t* txt_masks, int32_t B,
                            int32_t L, float* txt_embeds, void* saved, size_t saved_bytes, int32_t training, void* stream,
                            const etp_dropout* dropout) {
  ETP_REQUIRE(w && txt_ids && txt_masks && txt_embeds && saved, "etp_forward_txt: null argument");
  return forward_txt(*w, txt_ids, txt_masks, B, L, txt_embeds, saved, saved_bytes, training != 0, S(stream), dropout);
}

}  // extern "C"
