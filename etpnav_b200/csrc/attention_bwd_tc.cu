// Attention backward (head dim 64) on tcgen05 tensor cores, for query sequences that fit one 128-row tile
// (graph nodes: <= 128).  PERSISTENT: one CTA per SM walks over (batch, head) items; keys in blocks of 128.
//
//   per key block ("step"):  S = Q.K^T, dP = dO.V^T                 (2 x [M=128,N=128,K=64] into TMEM)
//     16 softmax-backward warps — thread = (query row, 32-key slice): P = exp2(s2 - lse2), dS = P * (dP - D) (x scale),
//     both written to shared memory as bf16 in the 128B-swizzled [query, key] layout, which the tensor core
//     reads K-major (dQ += dS.K) AND MN-major (dV = P^T.dO, dK = dS^T.Q) — the same bytes, two descriptors;
//     sprel_linear gradients (sum dS*pair, sum dS) accumulate per thread over the CTA's whole item list;
//   then  dV_blk = P^T.dO, dK_blk = dS^T.Q  ([M=128 keys, N=64, K=128 queries]),  dQ += dS.K  (accumulating
//   in TMEM across key blocks); dK/dV rows are read back (thread = key; one warp group takes dV, the other dK)
//   and stored as bf16; dQ after the last block.  Q and dO tiles double as MN-major B operands, K as both
//   K-major (S) and MN-major (dQ) B.
//
// The control thread runs one step ahead of the math: Q/dO and K/V tiles are double-buffered, so the TMA
// loads of step s+1 (possibly the next item) are in flight while the warps work on step s, and S/dP of
// step s+1 are issued right behind the dV/dK/dQ MMAs of step s.  TMEM allocation, barrier set-up and the
// launch are paid once per CTA instead of once per (batch, head).
// Gradient counterpart of BertOutAttention / BertSelfAttention (vilmodel_cmt.py:325-352, 103-141, 391-393).
#include "common.cuh"
#include "host.h"
#include "ops.h"

namespace etp {

namespace {

constexpr int kBQ = 128;
constexpr int kBK = 128;
constexpr int kD = 64;
constexpr int kTile = kBQ * kD * 2;     // 16 KB: Q, dO, K, V tiles
constexpr int kPBytes = kBQ * kBK * 2;  // 32 KB: P and dS
constexpr int kWQ = 4;                  // warps per TMEM lane quadrant: each owns 32 of the block's 128 keys
constexpr int kWarps = 4 * kWQ;         // softmax-backward warps
constexpr int kMathThreads = kWarps * 32;
constexpr int kThreads = kMathThreads + 32;  // + control warp
constexpr int kSmemBytes = 8 * kTile + 2 * kPBytes + 2 * kBK * 4 + kWQ * kBQ * 4 + 256 + 1024 + 256;
constexpr uint32_t kTmemCols = 512;  // S [0,128) dP [128,256) dV [256,320) dK [320,384) dQ [384,448)
constexpr float kLog2e = 1.4426950408889634f;

struct BwdDev {
  int B, heads, Sq, Sk;
  float scale;
  const uint8_t* key_valid;
  float mask_value;
  const float* pair;
  float pair_w, pair_b;
  const float* pair_w_dev;
  const float* pair_b_dev;
  const bf16* out; int ldo;
  const bf16* dout; int lddo;
  const float* lse;
  bf16 *dq, *dk, *dv;
  int lddq, lddk, lddv;
  float *dpair_w, *dpair_b;
  Drop drop;  // the forward's attention-probability dropout (thr 0 = off)
  const int32_t* kv_rows;  // optional batch-row map of the K / V tensor (see AttnBwdArgs)
  unsigned long long* dbg;  // optional timeline of CTA 0 (globaltimer ns): [0,64) control thread, [64,128) math thread 0
};

ETP_DEVICE unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define ETP_DBG(slot)                                                      \
  do {                                                                     \
    if (p.dbg && blockIdx.x == 0 && (slot) < 64) p.dbg[dbg_base + (slot)] = gtime(); \
  } while (0)

ETP_DEVICE uint4 pack8(const float* f) {
  return make_uint4(pack_bf16x2(f[0], f[1]), pack_bf16x2(f[2], f[3]), pack_bf16x2(f[4], f[5]), pack_bf16x2(f[6], f[7]));
}
ETP_DEVICE uint4 pack8u(const uint32_t* u) {
  return make_uint4(pack_bf16x2(__uint_as_float(u[0]), __uint_as_float(u[1])),
                    pack_bf16x2(__uint_as_float(u[2]), __uint_as_float(u[3])),
                    pack_bf16x2(__uint_as_float(u[4]), __uint_as_float(u[5])),
                    pack_bf16x2(__uint_as_float(u[6]), __uint_as_float(u[7])));
}
ETP_DEVICE float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
ETP_DEVICE float dot8(const uint4& a, const uint4& c) {
  const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&a);
  const __nv_bfloat162* hc = reinterpret_cast<const __nv_bfloat162*>(&c);
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const float2 fa = __bfloat1622float2(ha[t]), fc = __bfloat1622float2(hc[t]);
    s = fmaf(fa.x, fc.x, s);
    s = fmaf(fa.y, fc.y, s);
  }
  return s;
}

// batch row of the K / V tensor that query batch b reads (kept out of line: inlined, its load lengthens live ranges
// in the control loop enough to add spills)
__device__ __noinline__ int kv_row_of(const int32_t* kv_rows, int b) { return __ldg(kv_rows + b); }

template <bool kPair>
__global__ void __launch_bounds__(kThreads, 1)
attention_bwd_tc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmDO,
                        const __grid_constant__ CUtensorMap tmK, const __grid_constant__ CUtensorMap tmV,
                        const __grid_constant__ CUtensorMap tmDQ, const __grid_constant__ CUtensorMap tmDK,
                        const __grid_constant__ CUtensorMap tmDV, const BwdDev p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                 // [2][16 KB]
  uint8_t* sDO = sQ + 2 * kTile;      // [2][16 KB]
  uint8_t* sK = sDO + 2 * kTile;      // [2][16 KB]
  uint8_t* sV = sK + 2 * kTile;       // [2][16 KB]
  uint8_t* sP = sV + 2 * kTile;
  uint8_t* sDS = sP + kPBytes;
  float* sKb = reinterpret_cast<float*>(sDS + kPBytes);  // [2][128] per-key additive bias (log2 domain)
  float* sDp = sKb + 2 * kBK;                             // [kWQ][128] partial row dots of dO.O
  float* sRed = sDp + kWQ * kBQ;                          // [2 * kWarps]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRed + 2 * kWarps);
  uint64_t* q_full = bars + 0;    // [2]
  uint64_t* kv_full = bars + 2;   // [2]
  uint64_t* sdp_ready = bars + 4;
  uint64_t* pds_ready = bars + 5;
  uint64_t* g_ready = bars + 6;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 7);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nblk = (p.Sk + kBK - 1) / kBK;
  const int n_items = p.B * p.heads;

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmDO); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV);
    tma_prefetch_desc(&tmDQ); tma_prefetch_desc(&tmDK); tma_prefetch_desc(&tmDV);
    mbar_init(&q_full[0], 1); mbar_init(&q_full[1], 1);
    mbar_init(&kv_full[0], 1); mbar_init(&kv_full[1], 1);
    mbar_init(sdp_ready, 1);
    mbar_init(pds_ready, kMathThreads);
    mbar_init(g_ready, 1);
    fence_barrier_init();
    fence_proxy_async();
  }
  griddep_launch();  // PDL: the next kernel may start its own prologue
  griddep_wait();    // previous kernel complete; nothing above touched global memory or TMEM
  if (warp == kWarps) {
    tmem_alloc(tmem_ptr, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tm = *tmem_ptr;
  const uint32_t tS = tm, tDP = tm + 128, tDV = tm + 256, tDK = tm + 320, tDQ = tm + 384;

  if (warp == kWarps) {
    // ======================= control warp: TMA + MMA issue (one lane), one step ahead =======================
    if (lane == 0 && static_cast<int>(blockIdx.x) < n_items) {
      constexpr uint32_t id_s = make_idesc_bf16(128, 128, 0, 0);   // [q, d] x [key, d]^T
      constexpr uint32_t id_kv = make_idesc_bf16(128, 64, 1, 1);   // A = P/dS read MN-major, B = dO/Q MN-major
      constexpr uint32_t id_q = make_idesc_bf16(128, 64, 0, 1);    // A = dS K-major, B = K MN-major
      const uint32_t aP = smem_u32(sP), aDS = smem_u32(sDS);
      auto load_q = [&](int item, int st) {
        const int b = item / p.heads, h = item % p.heads;
        mbar_arrive_expect_tx(&q_full[st], 2 * kTile);
        tma_load_3d(sQ + st * kTile, &tmQ, &q_full[st], h * kD, 0, b);
        tma_load_3d(sDO + st * kTile, &tmDO, &q_full[st], h * kD, 0, b);
      };
      auto load_kv = [&](int item, int j, int st) {
        const int b = item / p.heads, h = item % p.heads;
        const int kvb = p.kv_rows ? kv_row_of(p.kv_rows, b) : b;
        mbar_arrive_expect_tx(&kv_full[st], 2 * kTile);
        tma_load_3d(sK + st * kTile, &tmK, &kv_full[st], h * kD, j * kBK, kvb);
        tma_load_3d(sV + st * kTile, &tmV, &kv_full[st], h * kD, j * kBK, kvb);
      };
      const int dbg_base = 0;
      ETP_DBG(0);
      load_q(blockIdx.x, 0);
      load_kv(blockIdx.x, 0, 0);
      int s = 0;   // step counter (item, key block) of this CTA
      int ii = 0;  // item counter of this CTA
      for (int item = blockIdx.x; item < n_items; item += gridDim.x, ++ii) {
        const int qst = ii & 1;
        const uint32_t aQ = smem_u32(sQ + qst * kTile), aDO = smem_u32(sDO + qst * kTile);
        for (int j = 0; j < nblk; ++j, ++s) {
          const int kst = s & 1;
          const uint32_t aK = smem_u32(sK + kst * kTile), aV = smem_u32(sV + kst * kTile);
          if (j == 0) mbar_wait(&q_full[qst], (ii >> 1) & 1);
          mbar_wait(&kv_full[kst], (s >> 1) & 1);
          tc_fence_after();
          ETP_DBG(1 + 4 * s);  // tiles landed
          {
            // descriptor low words advance by (bytes >> 4) per MMA; high words are loop constants
            const uint64_t dq0 = make_smem_desc(aQ, 16, 1024), dk0 = make_smem_desc(aK, 16, 1024);
            const uint64_t do0 = make_smem_desc(aDO, 16, 1024), dv0 = make_smem_desc(aV, 16, 1024);
#pragma unroll
            for (int k = 0; k < kD / 16; ++k)
              umma_bf16_lh(tS, desc_lo(dq0) + 2 * k, desc_hi(dq0), desc_lo(dk0) + 2 * k, desc_hi(dk0), id_s, k > 0 ? 1u : 0u);
#pragma unroll
            for (int k = 0; k < kD / 16; ++k)
              umma_bf16_lh(tDP, desc_lo(do0) + 2 * k, desc_hi(do0), desc_lo(dv0) + 2 * k, desc_hi(dv0), id_s, k > 0 ? 1u : 0u);
          }
          umma_commit(sdp_ready);
          // prefetch the tiles of the next step; its buffers were last read by the MMAs of step s-1
          const bool more_blocks = j + 1 < nblk;
          const int next_item = item + gridDim.x;
          if (more_blocks || next_item < n_items) {
            if (s >= 1) mbar_wait(g_ready, (s - 1) & 1);
            if (more_blocks) {
              load_kv(item, j + 1, (s + 1) & 1);
            } else {
              load_q(next_item, (ii + 1) & 1);
              load_kv(next_item, 0, (s + 1) & 1);
            }
          }
          ETP_DBG(2 + 4 * s);  // S/dP issued, next tiles requested
          mbar_wait(pds_ready, s & 1);
          tc_fence_after();
          ETP_DBG(3 + 4 * s);  // P/dS ready
          // dV / dK: reduction over the 128 queries, 16 per MMA: A panels are [query rows of 128 B] -> advance 16 rows =
          // 2048 B, two 64-key panels 16 KB apart (LBO), 8-row groups 1 KB apart (SBO); B = dO / Q tile read MN-major.
          {
            const uint64_t dpm = make_smem_desc(aP, 16384, 1024), dsm = make_smem_desc(aDS, 16384, 1024);   // MN-major A
            const uint64_t dom = make_smem_desc(aDO, 8192, 1024), dqm = make_smem_desc(aQ, 8192, 1024);     // MN-major B
            const uint64_t dsk = make_smem_desc(aDS, 16, 1024);                                             // K-major A
            const uint64_t dkm = make_smem_desc(aK, 8192, 1024);                                            // MN-major B
            // reductions only over the query / key groups that exist (the rest of the tiles is zero padding)
            const int qgroups = (min(kBQ, p.Sq) + 15) >> 4;
            const int kgroups = (min(kBK, p.Sk - j * kBK) + 15) >> 4;
#pragma unroll
            for (int k = 0; k < kBQ / 16; ++k) {
              if (k >= qgroups) break;
              umma_bf16_lh(tDV, desc_lo(dpm) + 128 * k, desc_hi(dpm), desc_lo(dom) + 128 * k, desc_hi(dom), id_kv, k > 0 ? 1u : 0u);
              umma_bf16_lh(tDK, desc_lo(dsm) + 128 * k, desc_hi(dsm), desc_lo(dqm) + 128 * k, desc_hi(dqm), id_kv, k > 0 ? 1u : 0u);
            }
            // dQ += dS.K : reduction over the 128 keys of this block
#pragma unroll
            for (int k = 0; k < kBK / 16; ++k)
              if (k < kgroups)
              umma_bf16_lh(tDQ, desc_lo(dsk) + (k >> 2) * 1024 + (k & 3) * 2, desc_hi(dsk), desc_lo(dkm) + 128 * k, desc_hi(dkm),
                           id_q, (j > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit(g_ready);
          ETP_DBG(4 + 4 * s);  // dV/dK/dQ issued
        }
      }
    }
  } else {
    // ======================= softmax-backward warps: thread = (query row, 32-key slice) =======================
    const int quad = warp & 3;            // TMEM lane quadrant
    const int wq = warp >> 2;             // which 32 keys of the block (softmax phase) / which read-back slice
    const int r = quad * 32 + lane;       // query row (softmax phase) / key row of the block (dK, dV read-back)
    const bool qv = r < p.Sq;
    const bool warp_live = quad * 32 < p.Sq;  // some row of this warp is a real query (warp-uniform)
    const uint32_t lane_sel = static_cast<uint32_t>(quad * 32) << 16;
    const float pw2 = (p.pair_w_dev ? __ldg(p.pair_w_dev) : p.pair_w) * kLog2e;
    const float pb2 = (p.pair_b_dev ? __ldg(p.pair_b_dev) : p.pair_b) * kLog2e;
    const float sl2 = p.scale * kLog2e;
    const float mask2 = p.mask_value * kLog2e;
    const bool pair_vec = (p.Sk & 3) == 0;  // rows of the pair bias are 16-byte aligned
    const int dbg_base = 64;
    const bool dbg_thread = threadIdx.x == 0;
    float wsum = 0.f, bsum = 0.f;           // sum dS*scale*pair, sum dS*scale over everything this thread sees
    int s = 0;
    // O / dO slices and lse of the row for the NEXT item are requested one item ahead (their latency hides behind
    // the current item's math); D = sum_d dO * O: each of the row's four threads takes 16 of the 64 dims
    uint4 nO0, nO1, nD0, nD1;
    float n_lse = 0.f;
    auto request_item = [&](int item) {
      if (qv && item < n_items) {
        const int b = item / p.heads, h = item % p.heads;
        const size_t row = static_cast<size_t>(b) * p.Sq + r;
        const uint4* po = reinterpret_cast<const uint4*>(p.out + row * p.ldo + h * kD + wq * 16);
        const uint4* pd = reinterpret_cast<const uint4*>(p.dout + row * p.lddo + h * kD + wq * 16);
        nO0 = __ldg(po); nO1 = __ldg(po + 1); nD0 = __ldg(pd); nD1 = __ldg(pd + 1);
        n_lse = p.lse[(static_cast<size_t>(b) * p.heads + h) * p.Sq + r];
      }
    };
    // per-step inputs fetched one step ahead as well: validity of key (k0 + tid) for the mask, and the first 16 pair
    // biases of this thread's row
    uint8_t kv_next = 1;
    float pv[16];
    auto load_pair_at = [&](const float* row_ptr, int key0) {
      if constexpr (kPair) {
        if (qv) {
          if (pair_vec) {
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
              if (key0 + i < p.Sk) f = __ldg(reinterpret_cast<const float4*>(row_ptr + key0 + i));
              pv[i] = f.x; pv[i + 1] = f.y; pv[i + 2] = f.z; pv[i + 3] = f.w;
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) pv[i] = (key0 + i < p.Sk) ? __ldg(row_ptr + key0 + i) : 0.f;
          }
        } else {
#pragma unroll
          for (int i = 0; i < 16; ++i) pv[i] = 0.f;
        }
      }
    };
    auto request_step = [&](int item, int j) {
      if (item >= n_items) return;
      const int b = item / p.heads;
      if (threadIdx.x < kBK) {
        const int k = j * kBK + static_cast<int>(threadIdx.x);
        kv_next = (p.key_valid && k < p.Sk) ? __ldg(p.key_valid + static_cast<size_t>(b) * p.Sk + k) : 1;
      }
      if constexpr (kPair) load_pair_at(p.pair + (static_cast<size_t>(b) * p.Sq + r) * p.Sk, j * kBK + wq * 32);
    };
    request_item(blockIdx.x);
    request_step(blockIdx.x, 0);
    for (int item = blockIdx.x; item < n_items; item += gridDim.x) {
      const int b = item / p.heads, h = item % p.heads;
      const float* pair_row = kPair ? p.pair + (static_cast<size_t>(b) * p.Sq + r) * p.Sk : nullptr;
      const uint32_t e_row = static_cast<uint32_t>(((static_cast<size_t>(b) * p.heads + h) * p.Sq + r) * p.Sk);
      float nlse2 = -INFINITY, Ds = 0.f;  // -lse (log2 domain): -inf kills padding rows
      {
        float part = 0.f;
        if (qv) {
          part = dot8(nO0, nD0) + dot8(nO1, nD1);
          nlse2 = -n_lse * kLog2e;
        }
        sDp[wq * kBQ + r] = part;
      }

      for (int j = 0; j < nblk; ++j, ++s) {
        const uint32_t ph = s & 1;
        const int k0 = j * kBK;
        float* kb = sKb + (s & 1) * kBK;
        if (threadIdx.x < kBK) {
          const int k = k0 + static_cast<int>(threadIdx.x);
          float v = -INFINITY;
          if (k < p.Sk) v = (kv_next ? 0.f : mask2) + (kPair ? pb2 : 0.f);
          kb[threadIdx.x] = v;
        }
        if (dbg_thread) ETP_DBG(0 + 6 * s);  // step begins
        if (threadIdx.x == 0) tma_store_wait_read();  // the previous step's output tiles have left P / dS
        named_bar_sync(1, kMathThreads);  // key bias (and, for j == 0, the partial row dots) visible
        if (j == 0) Ds = (sDp[r] + sDp[kBQ + r] + sDp[2 * kBQ + r] + sDp[3 * kBQ + r]) * p.scale;
        if (dbg_thread) ETP_DBG(1 + 6 * s);  // past the CTA barrier
        mbar_wait(sdp_ready, ph);
        tc_fence_after();
        if (dbg_thread) ETP_DBG(2 + 6 * s);  // S/dP ready
#pragma unroll
        for (int sub = 0; sub < 2; ++sub) {
          const int c = wq * 32 + sub * 16;  // first key column of this 16-key piece inside the block
          float pe[16], de[16];
          if (warp_live) {  // warp-uniform: tcgen05.ld is a warp-collective instruction
            uint32_t vs[16], vd[16];
            tmem_ld16(tS + lane_sel + c, vs);
            tmem_ld16(tDP + lane_sel + c, vd);
            // dropout multipliers of these 16 probabilities: one hash per aligned pair when the key count is even
            float dm[16];
            if (p.drop.thr) {
              const uint32_t e0 = e_row + static_cast<uint32_t>(k0 + c);
              if ((p.Sk & 1) == 0) {
#pragma unroll
                for (int i = 0; i < 16; i += 2) drop_mul2(p.drop, e0 + i, dm[i], dm[i + 1]);
              } else {
#pragma unroll
                for (int i = 0; i < 16; ++i) dm[i] = drop_mul(p.drop, e0 + i);
              }
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) dm[i] = 1.0f;
            }
            tmem_ld_wait();
#pragma unroll
            for (int i = 0; i < 16; i += 4) {
              const float4 kb4 = *reinterpret_cast<const float4*>(kb + c + i);
              const float kbv[4] = {kb4.x, kb4.y, kb4.z, kb4.w};
#pragma unroll
              for (int t = 0; t < 4; ++t) {
                float sc = fmaf(__uint_as_float(vs[i + t]), sl2, kbv[t]);
                if constexpr (kPair) sc = fmaf(pw2, pv[i + t], sc);
                const float pr = ex2_approx(sc + nlse2);                            // P (0 on padding rows)
                const float mk = dm[i + t];  // forward dropout multiplier of this probability (1, or 0 / 1/(1-p))
                // dP = mask * d(dropped P);  dS = P * (dP - D)  (x scale);  dV uses the dropped P
                const float dss = pr * fmaf(__uint_as_float(vd[i + t]) * mk, p.scale, -Ds);
                if constexpr (kPair) { wsum = fmaf(dss, pv[i + t], wsum); bsum += dss; }
                pe[i + t] = pr * mk;
                de[i + t] = dss;
              }
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) { pe[i] = 0.f; de[i] = 0.f; }
          }
          if (sub == 0) load_pair_at(pair_row, k0 + wq * 32 + 16);  // next piece's bias while this one is packed
          uint8_t* prow = sP + (c >> 6) * 16384 + r * 128;
          uint8_t* drow = sDS + (c >> 6) * 16384 + r * 128;
          const int ch0 = (c & 63) >> 3;
#pragma unroll
          for (int g = 0; g < 2; ++g) {
            const int off = (((ch0 + g) ^ (r & 7)) << 4);
            *reinterpret_cast<uint4*>(prow + off) = pack8(pe + 8 * g);
            *reinterpret_cast<uint4*>(drow + off) = pack8(de + 8 * g);
          }
        }
        fence_proxy_async();
        tc_fence_before();
        mbar_arrive(pds_ready);
        if (dbg_thread) ETP_DBG(3 + 6 * s);  // P/dS written
        // next step's mask / bias and, at an item boundary, the next item's O / dO / lse: in flight during the read-back
        if (j == nblk - 1) {
          request_item(item + gridDim.x);
          request_step(item + gridDim.x, 0);
        } else {
          request_step(item, j + 1);
        }
        // dK / dV of this key block (thread r now owns key k0 + r; slices 0,1 take dV columns, slices 2,3 dK columns)
        // and, after the last block, dQ: TMEM -> bf16 -> the (now idle) P / dS buffers in the TMA 128B-swizzled
        // layout -> one TMA store per tile.  Row-per-thread global stores would touch 32 cache lines per warp
        // instruction; the TMA store is asynchronous and clips rows past the sequence end.
        mbar_wait(g_ready, ph);
        tc_fence_after();
        if (dbg_thread) ETP_DBG(4 + 6 * s);  // dV/dK/dQ ready
        {
          const int cs = (wq & 1) * 32;
          uint32_t vv[32];
          tmem_ld32((wq < 2 ? tDV : tDK) + lane_sel + cs, vv);
          tmem_ld_wait();
          uint8_t* trow = sP + (wq < 2 ? 0 : kTile) + r * 128;
#pragma unroll
          for (int g = 0; g < 4; ++g)
            *reinterpret_cast<uint4*>(trow + ((((wq & 1) * 4 + g) ^ (r & 7)) << 4)) = pack8u(vv + 8 * g);
        }
        if (j == nblk - 1 && wq < 2) {
          uint32_t v[32];
          tmem_ld32(tDQ + lane_sel + wq * 32, v);
          tmem_ld_wait();
          uint8_t* trow = sDS + r * 128;
#pragma unroll
          for (int g = 0; g < 4; ++g) *reinterpret_cast<uint4*>(trow + (((wq * 4 + g) ^ (r & 7)) << 4)) = pack8u(v + 8 * g);
        }
        fence_proxy_async();
        tc_fence_before();
        named_bar_sync(2, kMathThreads);  // tiles complete
        if (threadIdx.x == 0) {
          tma_store_3d(&tmDV, sP, h * kD, k0, b);
          tma_store_3d(&tmDK, sP + kTile, h * kD, k0, b);
          if (j == nblk - 1) tma_store_3d(&tmDQ, sDS, h * kD, 0, b);
          tma_store_commit();
        }
        if (dbg_thread) ETP_DBG(5 + 6 * s);  // read-back stored
      }
    }
    if (threadIdx.x == 0) tma_store_wait_all();
    if (kPair && p.dpair_w) {
      wsum = warp_sum(wsum);
      bsum = warp_sum(bsum);
      if (lane == 0) { sRed[warp] = wsum; sRed[kWarps + warp] = bsum; }
      named_bar_sync(1, kMathThreads);
      if (threadIdx.x == 0) {
        float a = 0.f, c = 0.f;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) { a += sRed[w]; c += sRed[kWarps + w]; }
        const float inv = 1.0f / p.scale;  // the sums were taken over dS * scale
        atomicAdd(p.dpair_w, a * inv);
        atomicAdd(p.dpair_b, c * inv);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kWarps) {
    tc_fence_after();
    tmem_dealloc(tm, kTmemCols);
  }
}

}  // namespace

// debug timeline buffer (device, 128 x u64) of the next launches; null = off
static unsigned long long* g_attn_bwd_dbg = nullptr;
void attention_bwd_tc_set_debug(void* dev_buf) { g_attn_bwd_dbg = static_cast<unsigned long long*>(dev_buf); }

bool attention_bwd_tc_supported(const AttnBwdArgs& a) {
  if (a.Sq > kBQ) return false;
  if (a.Sq < 32 && a.Sk < 32) return false;  // tiny problems: CUDA-core kernels
  if (a.ldq % 8 || a.ldk % 8 || a.ldv % 8 || a.lddo % 8 || a.ldo % 8 || a.lddq % 8 || a.lddk % 8 || a.lddv % 8) return false;
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  return al16(a.q) && al16(a.k) && al16(a.v) && al16(a.out) && al16(a.dout) && al16(a.dq) && al16(a.dk) && al16(a.dv) &&
         (a.pair == nullptr || al16(a.pair));
}

int attention_bwd_tc(const AttnBwdArgs& a, cudaStream_t stream) {
  ETP_REQUIRE(attention_bwd_tc_supported(a), "attention_bwd_tc: unsupported shape / layout");
  CUtensorMap tq, tdo, tk, tv;
  const uint64_t W = static_cast<uint64_t>(a.heads) * kD;
  int rc = get_tmap_3d(a.q, W, a.Sq, a.B, a.ldq, static_cast<uint64_t>(a.Sq) * a.ldq, kD, kBQ, &tq);
  if (rc) return rc;
  rc = get_tmap_3d(a.dout, W, a.Sq, a.B, a.lddo, static_cast<uint64_t>(a.Sq) * a.lddo, kD, kBQ, &tdo);
  if (rc) return rc;
  const int kvB = a.kv_rows ? a.kv_B : a.B;
  ETP_REQUIRE(kvB > 0, "attention_bwd_tc: kv_B must be given with kv_rows");
  rc = get_tmap_3d(a.k, W, a.Sk, kvB, a.ldk, static_cast<uint64_t>(a.Sk) * a.ldk, kD, kBK, &tk);
  if (rc) return rc;
  rc = get_tmap_3d(a.v, W, a.Sk, kvB, a.ldv, static_cast<uint64_t>(a.Sk) * a.ldv, kD, kBK, &tv);
  if (rc) return rc;
  CUtensorMap tdq, tdk, tdv;
  rc = get_tmap_3d(a.dq, W, a.Sq, a.B, a.lddq, static_cast<uint64_t>(a.Sq) * a.lddq, kD, kBQ, &tdq);
  if (rc) return rc;
  rc = get_tmap_3d(a.dk, W, a.Sk, a.B, a.lddk, static_cast<uint64_t>(a.Sk) * a.lddk, kD, kBK, &tdk);
  if (rc) return rc;
  rc = get_tmap_3d(a.dv, W, a.Sk, a.B, a.lddv, static_cast<uint64_t>(a.Sk) * a.lddv, kD, kBK, &tdv);
  if (rc) return rc;
  static bool attr_set = false;
  if (!attr_set) {
    ETP_CHECK_CUDA(cudaFuncSetAttribute(attention_bwd_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    ETP_CHECK_CUDA(cudaFuncSetAttribute(attention_bwd_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  BwdDev d;
  d.B = a.B; d.heads = a.heads; d.Sq = a.Sq; d.Sk = a.Sk; d.scale = a.scale; d.key_valid = a.key_valid;
  d.mask_value = a.mask_value; d.pair = a.pair; d.pair_w = a.pair_w; d.pair_b = a.pair_b; d.pair_w_dev = a.pair_w_dev;
  d.pair_b_dev = a.pair_b_dev; d.out = a.out; d.ldo = a.ldo; d.dout = a.dout; d.lddo = a.lddo; d.lse = a.lse;
  d.dq = a.dq; d.dk = a.dk; d.dv = a.dv; d.lddq = a.lddq; d.lddk = a.lddk; d.lddv = a.lddv;
  d.dpair_w = a.dpair_w; d.dpair_b = a.dpair_b;
  d.drop = Drop{a.drop_key, a.drop_thr, a.drop_scale};
  d.kv_rows = a.kv_rows;
  d.dbg = g_attn_bwd_dbg;
  const int items = a.B * a.heads;
  const int grid = items < num_sms() ? items : num_sms();
  if (a.pair)
    ETP_CHECK_CUDA(launch_pdl(attention_bwd_tc_kernel<true>, dim3(grid), dim3(kThreads), kSmemBytes, stream, tq, tdo, tk, tv, tdq, tdk, tdv, d));
  else
    ETP_CHECK_CUDA(launch_pdl(attention_bwd_tc_kernel<false>, dim3(grid), dim3(kThreads), kSmemBytes, stream, tq, tdo, tk, tv, tdq, tdk, tdv, d));
  ETP_LAUNCHED();
  return ETP_OK;
}

}  // namespace etp
