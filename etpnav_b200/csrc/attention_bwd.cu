// Attention backward, head dim 64, CUDA-core variant (any shape; the tensor-core variant in
// attention_bwd_tc.cu takes over when a whole query sequence fits one 128-row tile).
//   P = exp(s - lse),  s = scale * q.k^T + bias        (lse saved by the forward kernel)
//   D_i = sum_d dO_id * O_id ;  dP = dO.V^T ;  dS = P * (dP - D)
//   dQ = scale * dS.K ;  dK = scale * dS^T.Q ;  dV = P^T.dO
//   sprel_linear grads (vilmodel_cmt.py:732-734): dw += sum dS * pair, db += sum dS
// Two kernels, each recomputing P from q, k and the saved log-sum-exp:
//   A: one warp per query row (keys across lanes)  -> dQ, D, sprel sums
//   B: one warp per key row   (queries across lanes) -> dK, dV
// Autograd counterpart of BertSelfAttention / BertOutAttention (vilmodel_cmt.py:103-141,325-352) and of
// nn.MultiheadAttention in the pano encoder (common/transformer.py:176).
#include "common.cuh"
#include "host.h"
#include "ops.h"

namespace etp {

namespace {
constexpr int kD = 64;
constexpr int kStr = 66;  // bf16 row stride in smem (33 words)
constexpr int kTile = 16;

ETP_DEVICE float dot64(const float* a, const bf16* row) {
  const uint32_t* r = reinterpret_cast<const uint32_t*>(row);
  float acc = 0.f;
#pragma unroll
  for (int d = 0; d < kD / 2; ++d) {
    const uint32_t u = r[d];
    const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u));
    acc += a[2 * d] * f.x + a[2 * d + 1] * f.y;
  }
  return acc;
}
ETP_DEVICE void stage_rows(bf16* dst, const bf16* src, int rows, int ld) {
  for (int i = threadIdx.x; i < rows * 8; i += blockDim.x) {
    const int r = i >> 3, c = (i & 7) * 8;
    const uint4 t = *reinterpret_cast<const uint4*>(src + static_cast<size_t>(r) * ld + c);
    uint32_t* d = reinterpret_cast<uint32_t*>(dst + r * kStr + c);
    d[0] = t.x; d[1] = t.y; d[2] = t.z; d[3] = t.w;
  }
}

__global__ void __launch_bounds__(256) attn_bwd_dq_kernel(const AttnBwdArgs a, int sk_pad) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  extern __shared__ uint8_t smem[];
  bf16* Ks = reinterpret_cast<bf16*>(smem);
  bf16* Vs = Ks + static_cast<size_t>(sk_pad) * kStr;
  float* qs = reinterpret_cast<float*>(Vs + static_cast<size_t>(sk_pad) * kStr);
  float* dos = qs + 8 * kD;
  float* dss = dos + 8 * kD;
  float* kb = dss + 8 * sk_pad;
  __shared__ float red[2][8];
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * kTile;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Sk = a.Sk;
  const int kvb = a.kv_rows ? __ldg(a.kv_rows + b) : b;  // row of the K / V tensor this batch element reads
  stage_rows(Ks, a.k + static_cast<size_t>(kvb) * Sk * a.ldk + h * kD, Sk, a.ldk);
  stage_rows(Vs, a.v + static_cast<size_t>(kvb) * Sk * a.ldv + h * kD, Sk, a.ldv);
  for (int j = threadIdx.x; j < sk_pad; j += 256) {
    float m = -INFINITY;
    if (j < Sk) m = (a.key_valid == nullptr || a.key_valid[static_cast<size_t>(b) * Sk + j]) ? 0.f : a.mask_value;
    kb[j] = m;
  }
  __syncthreads();
  const float pw = a.pair_w_dev ? __ldg(a.pair_w_dev) : a.pair_w;
  const float pb = a.pair_b_dev ? __ldg(a.pair_b_dev) : a.pair_b;
  float* myq = qs + warp * kD;
  float* mydo = dos + warp * kD;
  float* myds = dss + warp * sk_pad;
  float wsum = 0.f, bsum = 0.f;
  for (int qi = warp; qi < kTile; qi += 8) {
    const int q = q0 + qi;
    if (q >= a.Sq) break;
    const size_t row = static_cast<size_t>(b) * a.Sq + q;
    const float2 fq = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a.q + row * a.ldq + h * kD + lane * 2));
    const float2 fd = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a.dout + row * a.lddo + h * kD + lane * 2));
    const float2 fo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a.out + row * a.ldo + h * kD + lane * 2));
    myq[lane * 2] = fq.x * a.scale; myq[lane * 2 + 1] = fq.y * a.scale;
    mydo[lane * 2] = fd.x; mydo[lane * 2 + 1] = fd.y;
    const float Dv = warp_sum(fd.x * fo.x + fd.y * fo.y);
    const float lse = a.lse[(static_cast<size_t>(b) * a.heads + h) * a.Sq + q];
    if (lane == 0) a.dvec[(static_cast<size_t>(b) * a.heads + h) * a.Sq + q] = Dv;
    __syncwarp();
    const float* pair = a.pair ? a.pair + row * Sk : nullptr;
    for (int t = 0; t < sk_pad / 32; ++t) {
      const int j = t * 32 + lane;
      float ds = 0.f;
      if (j < Sk) {
        float s = dot64(myq, Ks + j * kStr) + kb[j];
        float pv = 0.f;
        if (pair) { pv = pair[j]; s += pw * pv + pb; }
        const float p = __expf(s - lse);
        float dp = dot64(mydo, Vs + j * kStr);  // d(dropped P); back through the dropout mask
        if (a.drop_thr) dp *= drop_mul(Drop{a.drop_key, a.drop_thr, a.drop_scale}, static_cast<uint32_t>(((static_cast<size_t>(b) * a.heads + h) * a.Sq + q) * Sk + j));
        ds = p * (dp - Dv);
        wsum += ds * pv;
        bsum += ds;
      }
      myds[j] = ds;
    }
    __syncwarp();
    float o0 = 0.f, o1 = 0.f;
    for (int j = 0; j < Sk; ++j) {
      const float dsj = myds[j];
      const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(Ks + j * kStr + lane * 2));
      o0 += dsj * f.x; o1 += dsj * f.y;
    }
    *reinterpret_cast<uint32_t*>(a.dq + row * a.lddq + h * kD + lane * 2) = pack_bf16x2(o0 * a.scale, o1 * a.scale);
    __syncwarp();
  }
  if (a.dpair_w) {  // block-level reduction, one atomic pair per CTA
    wsum = warp_sum(wsum); bsum = warp_sum(bsum);
    if (lane == 0) { red[0][warp] = wsum; red[1][warp] = bsum; }
    __syncthreads();
    if (threadIdx.x == 0) {
      float w = 0.f, bb = 0.f;
      for (int i = 0; i < 8; ++i) { w += red[0][i]; bb += red[1][i]; }
      atomicAdd(a.dpair_w, w);
      atomicAdd(a.dpair_b, bb);
    }
  }
}

__global__ void __launch_bounds__(256) attn_bwd_dkv_kernel(const AttnBwdArgs a, int sq_pad) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  extern __shared__ uint8_t smem[];
  bf16* Qs = reinterpret_cast<bf16*>(smem);
  bf16* dOs = Qs + static_cast<size_t>(sq_pad) * kStr;
  float* lses = reinterpret_cast<float*>(dOs + static_cast<size_t>(sq_pad) * kStr);
  float* Ds = lses + sq_pad;
  float* ks = Ds + sq_pad;
  float* vs = ks + 8 * kD;
  float* ps = vs + 8 * kD;
  float* dss = ps + 8 * sq_pad;
  const int b = blockIdx.z, h = blockIdx.y, k0 = blockIdx.x * kTile;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int Sq = a.Sq, Sk = a.Sk;
  const size_t kvb = a.kv_rows ? __ldg(a.kv_rows + b) : b;  // K / V are read from this row; dK / dV go to row b
  stage_rows(Qs, a.q + static_cast<size_t>(b) * Sq * a.ldq + h * kD, Sq, a.ldq);
  stage_rows(dOs, a.dout + static_cast<size_t>(b) * Sq * a.lddo + h * kD, Sq, a.lddo);
  for (int i = threadIdx.x; i < sq_pad; i += 256) {
    const size_t o = (static_cast<size_t>(b) * a.heads + h) * Sq + i;
    lses[i] = i < Sq ? a.lse[o] : 0.f;
    Ds[i] = i < Sq ? a.dvec[o] : 0.f;
  }
  __syncthreads();
  const float pw = a.pair_w_dev ? __ldg(a.pair_w_dev) : a.pair_w;
  const float pb = a.pair_b_dev ? __ldg(a.pair_b_dev) : a.pair_b;
  float* myk = ks + warp * kD;
  float* myv = vs + warp * kD;
  float* myp = ps + warp * sq_pad;
  float* myds = dss + warp * sq_pad;
  for (int ki = warp; ki < kTile; ki += 8) {
    const int j = k0 + ki;
    if (j >= Sk) break;
    const size_t krow = static_cast<size_t>(b) * Sk + j;
    const size_t kvrow = kvb * Sk + j;
    const float2 fk = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a.k + kvrow * a.ldk + h * kD + lane * 2));
    const float2 fv = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(a.v + kvrow * a.ldv + h * kD + lane * 2));
    myk[lane * 2] = fk.x * a.scale; myk[lane * 2 + 1] = fk.y * a.scale;
    myv[lane * 2] = fv.x; myv[lane * 2 + 1] = fv.y;
    const float kbias = (a.key_valid == nullptr || a.key_valid[krow]) ? 0.f : a.mask_value;
    __syncwarp();
    for (int t = 0; t < sq_pad / 32; ++t) {
      const int i = t * 32 + lane;
      float p = 0.f, ds = 0.f;
      if (i < Sq) {
        float s = dot64(myk, Qs + i * kStr) + kbias;
        if (a.pair) s += pw * a.pair[(static_cast<size_t>(b) * Sq + i) * Sk + j] + pb;
        p = __expf(s - lses[i]);
        float dp = dot64(myv, dOs + i * kStr);
        float mk = 1.0f;
        if (a.drop_thr)
          mk = drop_mul(Drop{a.drop_key, a.drop_thr, a.drop_scale},
                        static_cast<uint32_t>(((static_cast<size_t>(b) * a.heads + h) * Sq + i) * Sk + j));
        ds = p * (dp * mk - Ds[i]);
        p *= mk;  // dV = (dropped P)^T . dO
      }
      myp[i] = p;
      myds[i] = ds;
    }
    __syncwarp();
    float v0 = 0.f, v1 = 0.f, g0 = 0.f, g1 = 0.f;
    for (int i = 0; i < Sq; ++i) {
      const float pi = myp[i], dsi = myds[i];
      const float2 fo = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(dOs + i * kStr + lane * 2));
      const float2 fq = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(Qs + i * kStr + lane * 2));
      v0 += pi * fo.x; v1 += pi * fo.y;
      g0 += dsi * fq.x; g1 += dsi * fq.y;
    }
    *reinterpret_cast<uint32_t*>(a.dv + krow * a.lddv + h * kD + lane * 2) = pack_bf16x2(v0, v1);
    *reinterpret_cast<uint32_t*>(a.dk + krow * a.lddk + h * kD + lane * 2) = pack_bf16x2(g0 * a.scale, g1 * a.scale);
    __syncwarp();
  }
}

}  // namespace

int attention_bwd(const AttnBwdArgs& a, cudaStream_t stream) {
  ETP_REQUIRE(a.B > 0 && a.Sq > 0 && a.Sk > 0 && a.heads > 0, "attention_bwd: empty problem");
  ETP_REQUIRE(a.q && a.k && a.v && a.out && a.dout && a.lse && a.dvec && a.dq && a.dk && a.dv, "attention_bwd: null argument");
  ETP_REQUIRE(a.ldq % 8 == 0 && a.ldk % 8 == 0 && a.ldv % 8 == 0 && a.lddo % 8 == 0 && a.ldo % 2 == 0 && a.lddq % 2 == 0 &&
                  a.lddk % 2 == 0 && a.lddv % 2 == 0, "attention_bwd: pitches");
  ETP_REQUIRE(a.kv_rows == nullptr || a.kv_B > 0, "attention_bwd: kv_B must be given with kv_rows");
  const int sk_pad = (a.Sk + 31) / 32 * 32, sq_pad = (a.Sq + 31) / 32 * 32;
  const size_t smem_a = static_cast<size_t>(sk_pad) * kStr * 2 * 2 + 2 * 8 * kD * 4 + 8 * static_cast<size_t>(sk_pad) * 4 +
                        static_cast<size_t>(sk_pad) * 4;
  const size_t smem_b = static_cast<size_t>(sq_pad) * kStr * 2 * 2 + 2 * static_cast<size_t>(sq_pad) * 4 + 2 * 8 * kD * 4 +
                        2 * 8 * static_cast<size_t>(sq_pad) * 4;
  ETP_REQUIRE(smem_a <= 220 * 1024 && smem_b <= 220 * 1024, "attention_bwd: sequence too long for shared memory");
  static bool attr = false;
  if (!attr) {
    ETP_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dq_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    ETP_CHECK_CUDA(cudaFuncSetAttribute(attn_bwd_dkv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    attr = true;
  }
  ETP_CHECK_CUDA(launch_pdl(attn_bwd_dq_kernel, dim3(dim3((a.Sq + kTile - 1) / kTile, a.heads, a.B)), dim3(256), smem_a, stream, a, sk_pad));
  ETP_LAUNCHED();
  ETP_CHECK_CUDA(launch_pdl(attn_bwd_dkv_kernel, dim3(dim3((a.Sk + kTile - 1) / kTile, a.heads, a.B)), dim3(256), smem_b, stream, a, sq_pad));
  ETP_LAUNCHED();
  return ETP_OK;
}

bool attention_bwd_tc_supported(const AttnBwdArgs& a);          // attention_bwd_tc.cu
int attention_bwd_tc(const AttnBwdArgs& a, cudaStream_t stream);

int attention_bwd_dispatch(const AttnBwdArgs& a, cudaStream_t stream) {
  if (attention_bwd_tc_supported(a)) return attention_bwd_tc(a, stream);
  return attention_bwd(a, stream);
}

}  // namespace etp
