// Saved-activation records and helpers shared by the step-level forward (planner.cu) and backward
// (planner_bwd.cu) sequencing code.
#pragma once
#include <vector>

#include "host.h"
#include "ops.h"

namespace etp {

constexpr int kH = 768;      // hidden size
constexpr int kI = 3072;     // FFN intermediate size
constexpr int kHeads = 12;   // heads of 64

// Bump allocator over a caller-owned device buffer (256-byte aligned slices).  With base == nullptr it
// only measures.
struct Arena {
  uint8_t* base;
  size_t cap;
  size_t off = 0;
  Arena(void* b, size_t c) : base(static_cast<uint8_t*>(b)), cap(c) {}
  template <typename T>
  T* take(size_t n) {
    const size_t bytes = (n * sizeof(T) + 255) & ~size_t(255);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += bytes;
    return p;
  }
};

// One post-LN block (cross-attention part only when `cross`): everything backward needs.
struct LayerRecord {
  bf16 *q = nullptr, *kv = nullptr, *ctx1 = nullptr;  // cross-attn: q [rows,768], k|v [kv_rows,1536], context
  float* lse1 = nullptr;
  float* t1 = nullptr;   // pre-LayerNorm sum (fp32)
  float* st1 = nullptr;  // mean[rows], rstd[rows]
  bf16* ab = nullptr;    // LN output (bf16) = input of the self-attention block
  bf16 *qkv = nullptr, *ctx2 = nullptr;
  float* lse2 = nullptr;
  float* t2 = nullptr;
  float* st2 = nullptr;
  bf16* cb = nullptr;
  bf16 *pre = nullptr, *h = nullptr;  // FFN: gelu'(pre-activation) for the backward / GELU output [rows,3072]
  float* t3 = nullptr;
  float* st3 = nullptr;
  bf16* xb = nullptr;  // block output (bf16)
  int ldkv = 0;        // row pitch of kv (elements): 2*768 when owned, X*1536 when it is a slice of NavRecord::kv_all
  void carve(Arena& ar, int rows, int kv_rows, int B, int Sq, bool cross);
};

struct NavRecord {
  bf16* txtb = nullptr;    // (both left out when the text K|V come from an episode-level cache, etp_nav_inputs.txt_kv_all)
  bf16* kv_all = nullptr;  // text K|V of all layers, [B*L, X*1536]
  bf16* x0b = nullptr;
  float *pos_lin = nullptr, *pos_stats = nullptr;
  float *xa = nullptr, *xc = nullptr, *xf = nullptr;  // fp32 residual-stream scratch
  float *relu = nullptr, *sap_stats = nullptr;
  std::vector<LayerRecord> layers;
  void carve(Arena& ar, int B, int N, int L, int X, bool training, bool txt_cached);
};

// forward_lang2visn (pre-training twin, forward_mlm): the instruction tokens are the query stream, the packed map
// nodes the (layer-invariant) context
struct L2VRecord {
  bf16* nodeb = nullptr;    // packed nodes gmap_input_embeds (bf16) [B*N,768]
  float *pos_lin = nullptr, *pos_stats = nullptr;
  bf16* kv_all = nullptr;   // node K|V of all layers, [B*N, X*1536]
  bf16* txtb = nullptr;     // bf16 copy of the incoming txt_embeds [B*L,768]
  float *xa = nullptr, *xc = nullptr, *xf = nullptr, *nodef = nullptr;
  std::vector<LayerRecord> layers;
  void carve(Arena& ar, int B, int N, int L, int X, bool training);
};

struct PanoLayerRecord {
  bf16* y1b = nullptr;
  float* st1 = nullptr;
  bf16 *qkv = nullptr, *ctx = nullptr;
  float* lse = nullptr;
  bf16* y2b = nullptr;
  float* st2 = nullptr;
  bf16 *pre = nullptr, *h = nullptr;
};
struct PanoRecord {
  bf16 *rgbb = nullptr, *depb = nullptr;
  float *rgb_lin = nullptr, *dep_lin = nullptr, *loc_lin = nullptr, *sum_pre = nullptr, *stats = nullptr;
  std::vector<float*> xs;  // fp32 residual stream after packing / after each half-layer
  float* fin_stats = nullptr;
  std::vector<PanoLayerRecord> layers;
  void carve(Arena& ar, int B, int V, int P, bool training);
};

struct TxtRecord {
  float *sum_pre = nullptr, *emb_stats = nullptr;
  bf16* x0b = nullptr;
  float *xa = nullptr, *xc = nullptr;
  std::vector<LayerRecord> layers;
  void carve(Arena& ar, int B, int L, int NL, bool training);
};

// Dropout of one step-level call: seed + probabilities (include/etpnav_b200.h: etp_dropout) -> per-site kernel
// parameters.  Sites: one id per nn.Dropout instance of the reference; forward and backward use the same ids.
struct DropCtx {
  uint64_t seed = 0;
  float p_hidden = 0.f, p_attn = 0.f, p_head = 0.f;
  DropHost hidden(uint32_t site) const { return make_drop_host(seed, p_hidden, site); }
  DropHost attn(uint32_t site) const { return make_drop_host(seed, p_attn, site); }
  DropHost head(uint32_t site) const { return make_drop_host(seed, p_head, site); }
};
// site = base + 16 * layer + k
constexpr uint32_t kSiteNav = 1000, kSitePano = 2000, kSiteTxt = 3000, kSiteL2V = 4000;
constexpr uint32_t kSiteEmbed = 900;  // + base: dropout after the packing / embedding LayerNorm
constexpr uint32_t kSiteHead = 901;   // + kSiteNav: NextActionPrediction
// post-LN blocks (x-layers, BERT layers): k =
constexpr uint32_t kDropXAttn = 0, kDropXOut = 1, kDropSAttn = 2, kDropSOut = 3, kDropFfnOut = 4;
// pre-LN pano layers (common/transformer.py:170-182): k =
constexpr uint32_t kDropPAttn = 0, kDropPOut = 1, kDropPFfn = 2, kDropPFfnOut = 3;
inline uint32_t drop_site(uint32_t base, int layer, uint32_t k) { return base + 16u * static_cast<uint32_t>(layer) + k; }

// tcgen05 kernel when the shape allows it, CUDA-core kernel otherwise
int attention_dispatch(const AttnArgs& a, cudaStream_t stream);

}  // namespace etp
