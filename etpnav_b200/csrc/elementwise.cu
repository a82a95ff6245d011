// Row-wise HBM-bound kernels: LayerNorm forward/backward, column sums (bias gradients), casts.
// One warp owns one 768-wide row: 24 values per lane as six 128-bit loads, warp-shuffle reductions,
// fp32 statistics.  Replaces torch.nn.LayerNorm / BertLayerNorm on the reference path
// (vilmodel_cmt.py:24-28,151-153,190-192; common/transformer.py:144-145,174,178; common/ops.py:20).
#include "common.cuh"
#include "host.h"
#include "ops.h"

namespace etp {

constexpr int kH = 768;
constexpr int kVec = kH / 128;  // float4 per lane

ETP_DEVICE void load_row(const float* p, int lane, float (&v)[24]) {
#pragma unroll
  for (int i = 0; i < kVec; ++i) {
    const float4 t = *reinterpret_cast<const float4*>(p + (i * 32 + lane) * 4);
    v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
  }
}
ETP_DEVICE void store_row(float* p, int lane, const float (&v)[24]) {
#pragma unroll
  for (int i = 0; i < kVec; ++i)
    *reinterpret_cast<float4*>(p + (i * 32 + lane) * 4) = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
ETP_DEVICE void store_row_bf16(bf16* p, int lane, const float (&v)[24]) {
#pragma unroll
  for (int i = 0; i < kVec; ++i)
    *reinterpret_cast<uint2*>(p + (i * 32 + lane) * 4) =
        make_uint2(pack_bf16x2(v[4 * i], v[4 * i + 1]), pack_bf16x2(v[4 * i + 2], v[4 * i + 3]));
}
// mean and 1/sqrt(var + eps) of a row held across the warp (two-pass: exact like torch's LayerNorm)
ETP_DEVICE void row_stats(const float (&v)[24], float eps, float& mean, float& rstd) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) s += v[i];
  mean = warp_sum(s) * (1.0f / kH);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 24; ++i) { const float d = v[i] - mean; q += d * d; }
  rstd = rsqrtf(warp_sum(q) * (1.0f / kH) + eps);
}

__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ x, const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, float eps, int rows,
                                                             float* __restrict__ y_f32, bf16* __restrict__ y_bf16,
                                                             float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  float v[24], g[24], b[24];
  load_row(x + static_cast<size_t>(row) * kH, lane, v);
  load_row(gamma, lane, g);
  load_row(beta, lane, b);
  float mean, rstd;
  row_stats(v, eps, mean, rstd);
#pragma unroll
  for (int i = 0; i < 24; ++i) v[i] = (v[i] - mean) * rstd * g[i] + b[i];
  if (y_f32) store_row(y_f32 + static_cast<size_t>(row) * kH, lane, v);
  if (y_bf16) store_row_bf16(y_bf16 + static_cast<size_t>(row) * kH, lane, v);
  if (lane == 0) {
    if (mean_out) mean_out[row] = mean;
    if (rstd_out) rstd_out[row] = rstd;
  }
}

int layernorm_fwd(const float* x, const float* gamma, const float* beta, float eps, int rows, int H, float* y_f32,
                  bf16* y_bf16, float* mean, float* rstd, cudaStream_t stream) {
  ETP_REQUIRE(H == kH, "layernorm: hidden size must be 768");
  if (rows <= 0) return ETP_OK;
  ETP_CHECK_CUDA(launch_pdl(layernorm_fwd_kernel, dim3((rows + 7) / 8), dim3(256), 0, stream, x, gamma, beta, eps, rows, y_f32, y_bf16, mean, rstd));
  ETP_LAUNCHED();
  return ETP_OK;
}

// Backward: dx = rstd * (g - mean(g) - xhat * mean(g * xhat)),  g = dy * gamma,  xhat = (x - mean) * rstd.
// dgamma += sum_rows dy * xhat, dbeta += sum_rows dy, dxsum += sum_rows dx: per-lane partials over a grid-stride loop of
// rows.  The three partial rows live in SHARED memory (each lane owns its own float4 slots, so no synchronisation is
// needed inside the loop): keeping them in registers cost 72 registers per thread and limited the kernel to ONE 8-warp CTA
// per SM (178 registers), i.e. 8 warps of loads in flight; with them in shared memory two CTAs fit and the 2 x 148 CTA grid
// is a single wave.  At the end the 8 warps' partials are summed and leave as one vector reduction per 4 columns per CTA.
constexpr int kLnBwdSmem = (3 * 8 + 1) * (kH / 4) * 16;  // [dgamma | dbeta | dxsum][warp][192] float4 + gamma = 76,800 B
ETP_DEVICE void red_add_v4(float* p, float4 v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__global__ void __launch_bounds__(256, 2) layernorm_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                                const float* __restrict__ gamma, const float* __restrict__ mean,
                                                                const float* __restrict__ rstd, int rows, float* __restrict__ dx_f32,
                                                                int accumulate_dx, bf16* __restrict__ dx_bf16,
                                                                float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                                float* __restrict__ dxsum, const Drop drop) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  extern __shared__ float4 ln_acc[];
  constexpr int kQ = kH / 4;  // float4 slots per row
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float4* adg = ln_acc + (0 * 8 + warp) * kQ;
  float4* adb = ln_acc + (1 * 8 + warp) * kQ;
  float4* ads = ln_acc + (2 * 8 + warp) * kQ;
  float4* sgam = ln_acc + 3 * 8 * kQ;  // gamma, read per chunk (kept out of the registers)
#pragma unroll
  for (int i = 0; i < kVec; ++i) {
    adg[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    adb[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    ads[i * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int c = threadIdx.x; c < kQ; c += 256) sgam[c] = reinterpret_cast<const float4*>(gamma)[c];
  __syncthreads();
  for (int row = blockIdx.x * 8 + warp; row < rows; row += gridDim.x * 8) {
    float d[24], v[24];
    load_row(dy + static_cast<size_t>(row) * kH, lane, d);
    load_row(x + static_cast<size_t>(row) * kH, lane, v);
    const float mu = mean[row], rs = rstd[row];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      float4 tg = adg[i * 32 + lane], tb = adb[i * 32 + lane];
      const float4 gi = sgam[i * 32 + lane];
      const float gg[4] = {gi.x, gi.y, gi.z, gi.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) v[4 * i + j] = (v[4 * i + j] - mu) * rs;  // xhat
      tg.x += d[4 * i] * v[4 * i]; tg.y += d[4 * i + 1] * v[4 * i + 1];
      tg.z += d[4 * i + 2] * v[4 * i + 2]; tg.w += d[4 * i + 3] * v[4 * i + 3];
      tb.x += d[4 * i]; tb.y += d[4 * i + 1]; tb.z += d[4 * i + 2]; tb.w += d[4 * i + 3];
      adg[i * 32 + lane] = tg;
      adb[i * 32 + lane] = tb;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        d[4 * i + j] *= gg[j];  // g
        s1 += d[4 * i + j];
        s2 += d[4 * i + j] * v[4 * i + j];
      }
    }
    s1 = warp_sum(s1) * (1.0f / kH);
    s2 = warp_sum(s2) * (1.0f / kH);
    float* o = dx_f32 + static_cast<size_t>(row) * kH;
#pragma unroll
    for (int i = 0; i < kVec; ++i) {
      float4 t;
      t.x = rs * (d[4 * i] - s1 - v[4 * i] * s2);
      t.y = rs * (d[4 * i + 1] - s1 - v[4 * i + 1] * s2);
      t.z = rs * (d[4 * i + 2] - s1 - v[4 * i + 2] * s2);
      t.w = rs * (d[4 * i + 3] - s1 - v[4 * i + 3] * s2);
      float4* o4 = reinterpret_cast<float4*>(o + (i * 32 + lane) * 4);
      if (accumulate_dx) {
        const float4 prev = *o4;
        t.x += prev.x; t.y += prev.y; t.z += prev.z; t.w += prev.w;
      }
      *o4 = t;
      if (drop.thr) {
        // the Linear whose output this LayerNorm normalised went through dropout before the residual add: ITS output
        // gradient (the bf16 copy the dgrad / wgrad GEMMs read, and the bias gradient) carries the mask; the fp32
        // dx written above is the residual branch and does not.  Element index = row * 768 + column (drop_row24).
        const uint32_t e = static_cast<uint32_t>(row) * 768u + static_cast<uint32_t>((i * 32 + lane) * 4);
        float m0, m1, m2, m3;
        drop_mul2(drop, e, m0, m1);
        drop_mul2(drop, e + 2, m2, m3);
        t.x *= m0; t.y *= m1; t.z *= m2; t.w *= m3;
      }
      if (dx_bf16)
        *reinterpret_cast<uint2*>(dx_bf16 + static_cast<size_t>(row) * kH + (i * 32 + lane) * 4) =
            make_uint2(pack_bf16x2(t.x, t.y), pack_bf16x2(t.z, t.w));
      if (dxsum != nullptr) {
        float4 ts = ads[i * 32 + lane];
        ts.x += t.x; ts.y += t.y; ts.z += t.z; ts.w += t.w;
        ads[i * 32 + lane] = ts;
      }
    }
  }
  __syncthreads();
  // CTA reduction of the 8 warps' partial rows; one vector reduction per 4 columns per CTA and quantity
  for (int c = threadIdx.x; c < kQ; c += 256) {
    if (dgamma != nullptr) {
      float4 sg = make_float4(0.f, 0.f, 0.f, 0.f), sb = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const float4 a = ln_acc[(0 * 8 + w) * kQ + c], b2 = ln_acc[(1 * 8 + w) * kQ + c];
        sg.x += a.x; sg.y += a.y; sg.z += a.z; sg.w += a.w;
        sb.x += b2.x; sb.y += b2.y; sb.z += b2.z; sb.w += b2.w;
      }
      red_add_v4(dgamma + 4 * c, sg);
      red_add_v4(dbeta + 4 * c, sb);
    }
    if (dxsum != nullptr) {
      float4 ss = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int w = 0; w < 8; ++w) {
        const float4 a = ln_acc[(2 * 8 + w) * kQ + c];
        ss.x += a.x; ss.y += a.y; ss.z += a.z; ss.w += a.w;
      }
      red_add_v4(dxsum + 4 * c, ss);
    }
  }
}

int layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd, int rows,
                  int H, float* dx_f32, int accumulate_dx, bf16* dx_bf16, float* dgamma, float* dbeta,
                  cudaStream_t stream, float* dxsum, DropHost drop) {

  ETP_REQUIRE(H == kH, "layernorm: hidden size must be 768");
  if (rows <= 0) return ETP_OK;
  ETP_REQUIRE((dgamma == nullptr) == (dbeta == nullptr), "layernorm_bwd: dgamma and dbeta come together");
  ETP_REQUIRE(((reinterpret_cast<uintptr_t>(dgamma) | reinterpret_cast<uintptr_t>(dbeta) | reinterpret_cast<uintptr_t>(dxsum)) & 15) == 0,
              "layernorm_bwd: dgamma / dbeta / dxsum must be 16-byte aligned");
  static bool attr = false;
  if (!attr) {
    ETP_CHECK_CUDA(cudaFuncSetAttribute(layernorm_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kLnBwdSmem));
    attr = true;
  }
  int grid = (rows + 7) / 8;
  if (grid > 2 * num_sms()) grid = 2 * num_sms();  // two resident CTAs per SM: one wave
  ETP_CHECK_CUDA(launch_pdl(layernorm_bwd_kernel, dim3(grid), dim3(256), kLnBwdSmem, stream, dy, x, gamma, mean, rstd, rows, dx_f32, accumulate_dx, dx_bf16, dgamma,
                                                 dbeta, dxsum, Drop{drop.key, drop.thr, drop.scale}));
  ETP_LAUNCHED();
  return ETP_OK;
}

// out[c] += sum_r x[r, c].  Each CTA covers 64 columns x a slab of rows; threads (32 x 8): lane-pairs of columns,
// 8 row lanes, 4 rows in flight per thread; shared-memory reduce over the 8 row lanes; one atomicAdd per column per CTA.
template <typename T>
__global__ void __launch_bounds__(256) colsum_kernel(const T* __restrict__ x, int rows, int cols, int ld, int rows_per_cta,
                                                      float* __restrict__ out) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  __shared__ float red[8][64];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int c = blockIdx.x * 64 + tx * 2;
  const int r0 = blockIdx.y * rows_per_cta;
  const int r1 = min(rows, r0 + rows_per_cta);
  float s0 = 0.f, s1 = 0.f;
  if (c < cols) {
    auto ld2 = [&](int r) -> float2 {
      const T* p = x + static_cast<size_t>(r) * ld + c;
      if constexpr (sizeof(T) == 2) return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p));
      else return *reinterpret_cast<const float2*>(p);
    };
    int r = r0 + ty;
    for (; r + 24 < r1; r += 32) {
      const float2 a = ld2(r), b = ld2(r + 8), d = ld2(r + 16), e = ld2(r + 24);
      s0 += (a.x + b.x) + (d.x + e.x);
      s1 += (a.y + b.y) + (d.y + e.y);
    }
    for (; r < r1; r += 8) {
      const float2 a = ld2(r);
      s0 += a.x; s1 += a.y;
    }
  }
  red[ty][tx * 2] = s0;
  red[ty][tx * 2 + 1] = s1;
  __syncthreads();
  if (threadIdx.x < 64) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][threadIdx.x];
    const int cc = blockIdx.x * 64 + threadIdx.x;
    if (cc < cols) atomicAdd(out + cc, s);
  }
}

template <typename T>
static int colsum_impl(const T* x, int rows, int cols, int ld, float* out, cudaStream_t stream) {
  ETP_REQUIRE(cols % 2 == 0 && ld % 2 == 0, "colsum: even cols/ld required");
  if (rows <= 0) return ETP_OK;
  const int gx = (cols + 63) / 64;
  int gy = (4 * num_sms() + gx - 1) / gx;  // ~4 CTAs per SM: the kernel is pure streaming
  int rpc = (rows + gy - 1) / gy;
  if (rpc < 64) rpc = 64;
  gy = (rows + rpc - 1) / rpc;
  ETP_CHECK_CUDA(launch_pdl(colsum_kernel<T>, dim3(dim3(gx, gy)), dim3(256), 0, stream, x, rows, cols, ld, rpc, out));
  ETP_LAUNCHED();
  return ETP_OK;
}
int colsum_bf16(const bf16* x, int rows, int cols, int ld, float* out, cudaStream_t stream) {
  return colsum_impl<bf16>(x, rows, cols, ld, out, stream);
}
int colsum_f32(const float* x, int rows, int cols, int ld, float* out, cudaStream_t stream) {
  return colsum_impl<float>(x, rows, cols, ld, out, stream);
}

// Several column sums in ONE launch (the bias gradients of one transformer layer: d b_q, d b_v of the cross- and the
// self-attention): out_j[c] += sum_r x_j[r, c] for up to 8 bf16 matrices.  A CTA = (job, 64-column block, row slab);
// thread = (8 columns as one 16-byte load, one of 32 row lanes), four rows in flight per thread.
struct ColsumJobs {
  int n, total_ctas;
  const bf16* x[8];
  float* out[8];
  int rows[8], cols[8], ld[8], gx[8], rpc[8], cta_start[8];
};
__global__ void __launch_bounds__(256) colsum_grouped_kernel(const ColsumJobs jb) {
  griddep_launch();
  griddep_wait();
  __shared__ float red[32][65];
  int j = 0;
  while (j + 1 < jb.n && static_cast<int>(blockIdx.x) >= jb.cta_start[j + 1]) ++j;
  const int local = blockIdx.x - jb.cta_start[j];
  const int cb = local % jb.gx[j], rb = local / jb.gx[j];
  const int tc = threadIdx.x & 7, tr = threadIdx.x >> 3;
  const int c = cb * 64 + tc * 8;
  const int r0 = rb * jb.rpc[j], r1 = min(jb.rows[j], r0 + jb.rpc[j]);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  if (c < jb.cols[j]) {
    const bf16* base = jb.x[j] + c;
    const size_t ld = jb.ld[j];
    auto add8 = [&](const uint4& u) {
      const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(h[i]);
        acc[2 * i] += f.x; acc[2 * i + 1] += f.y;
      }
    };
    int r = r0 + tr;
    for (; r + 96 < r1; r += 128) {
      const uint4 a = __ldg(reinterpret_cast<const uint4*>(base + r * ld));
      const uint4 b = __ldg(reinterpret_cast<const uint4*>(base + (r + 32) * ld));
      const uint4 d = __ldg(reinterpret_cast<const uint4*>(base + (r + 64) * ld));
      const uint4 e = __ldg(reinterpret_cast<const uint4*>(base + (r + 96) * ld));
      add8(a); add8(b); add8(d); add8(e);
    }
    for (; r < r1; r += 32) add8(__ldg(reinterpret_cast<const uint4*>(base + r * ld)));
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) red[tr][tc * 8 + i] = acc[i];
  __syncthreads();
  if (threadIdx.x < 64) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 32; ++w) s += red[w][threadIdx.x];
    const int cc = cb * 64 + threadIdx.x;
    if (cc < jb.cols[j]) atomicAdd(jb.out[j] + cc, s);
  }
}

int colsum_bf16_grouped(const ColsumJob* jobs, int n, cudaStream_t stream) {
  ETP_REQUIRE(jobs != nullptr && n >= 0 && n <= 8, "colsum_grouped: 0..8 jobs");
  ColsumJobs jb;
  jb.n = 0;
  long long work = 0;
  for (int i = 0; i < n; ++i) {
    if (jobs[i].out == nullptr || jobs[i].rows <= 0) continue;
    ETP_REQUIRE(jobs[i].cols % 8 == 0 && jobs[i].ld % 8 == 0 && (reinterpret_cast<uintptr_t>(jobs[i].x) & 15) == 0,
                "colsum_grouped: 16-byte aligned rows of a multiple of 8 columns required");
    const int k = jb.n++;
    jb.x[k] = jobs[i].x; jb.out[k] = jobs[i].out; jb.rows[k] = jobs[i].rows; jb.cols[k] = jobs[i].cols; jb.ld[k] = jobs[i].ld;
    jb.gx[k] = (jobs[i].cols + 63) / 64;
    work += static_cast<long long>(jb.gx[k]) * jobs[i].rows;
  }
  if (jb.n == 0) return ETP_OK;
  // ~6 CTAs per SM over all jobs: rows per CTA from the total (64-column x row) work, at least 128 rows
  long long rpc = (work + 6LL * num_sms() - 1) / (6LL * num_sms());
  if (rpc < 128) rpc = 128;
  int start = 0;
  for (int k = 0; k < jb.n; ++k) {
    jb.rpc[k] = static_cast<int>(rpc);
    jb.cta_start[k] = start;
    start += jb.gx[k] * ((jb.rows[k] + jb.rpc[k] - 1) / jb.rpc[k]);
  }
  jb.total_ctas = start;
  ETP_CHECK_CUDA(launch_pdl(colsum_grouped_kernel, dim3(start), dim3(256), 0, stream, jb));
  ETP_LAUNCHED();
  return ETP_OK;
}

__global__ void cast_kernel(const float* __restrict__ x, bf16* __restrict__ y, int64_t n4) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const float4 t = reinterpret_cast<const float4*>(x)[i];
    reinterpret_cast<uint2*>(y)[i] = make_uint2(pack_bf16x2(t.x, t.y), pack_bf16x2(t.z, t.w));
  }
}
__global__ void cast_tail_kernel(const float* __restrict__ x, bf16* __restrict__ y, int64_t start, int64_t n) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  const int64_t i = start + threadIdx.x;
  if (i < n) y[i] = __float2bfloat16(x[i]);
}
int cast_f32_to_bf16(const float* x, bf16* y, int64_t n, cudaStream_t stream) {
  if (n <= 0) return ETP_OK;
  ETP_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 7) == 0, "cast: alignment");
  const int64_t n4 = n / 4;
  if (n4 > 0) {
    int64_t blocks = (n4 + 255) / 256;
    if (blocks > 8 * num_sms()) blocks = 8 * num_sms();
    ETP_CHECK_CUDA(launch_pdl(cast_kernel, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, x, y, n4));
  }
  if (n4 * 4 < n) ETP_CHECK_CUDA(launch_pdl(cast_tail_kernel, dim3(1), dim3(32), 0, stream, x, y, n4 * 4, n));
  ETP_LAUNCHED();
  return ETP_OK;
}

__global__ void add_kernel(float* __restrict__ dst, const float* __restrict__ src, int64_t n) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x)
    dst[i] += src[i];
}
int add_f32(float* dst, const float* src, int64_t n, cudaStream_t stream) {
  if (n <= 0) return ETP_OK;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 8 * num_sms()) blocks = 8 * num_sms();
  ETP_CHECK_CUDA(launch_pdl(add_kernel, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, dst, src, n));
  ETP_LAUNCHED();
  return ETP_OK;
}

// One thread per 8 columns of a row: a 16-byte bf16 load, two 16-byte fp32 read-modify-writes.  HBM-bound.
__global__ void kv_grad_accumulate_kernel(const bf16* __restrict__ dkv, const int32_t* __restrict__ rows, int L,
                                          int w8, int64_t n8, float* __restrict__ acc) {
  griddep_launch();  // PDL (common.cuh): let the next kernel get scheduled ...
  griddep_wait();    // ... and wait for the previous one before touching memory
  for (int64_t i = blockIdx.x * static_cast<int64_t>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<int64_t>(gridDim.x) * blockDim.x) {
    const int64_t r = i / w8;
    const int c = static_cast<int>(i - r * w8);
    const int b = static_cast<int>(r / L), l = static_cast<int>(r - static_cast<int64_t>(b) * L);
    const int64_t dst = (static_cast<int64_t>(rows ? __ldg(rows + b) : b) * L + l) * w8 + c;
    const uint4 g = __ldg(reinterpret_cast<const uint4*>(dkv) + i);
    float4* a = reinterpret_cast<float4*>(acc) + 2 * dst;
    float4 a0 = a[0], a1 = a[1];
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&g);
    float2 f;
    f = __bfloat1622float2(h[0]); a0.x += f.x; a0.y += f.y;
    f = __bfloat1622float2(h[1]); a0.z += f.x; a0.w += f.y;
    f = __bfloat1622float2(h[2]); a1.x += f.x; a1.y += f.y;
    f = __bfloat1622float2(h[3]); a1.z += f.x; a1.w += f.y;
    a[0] = a0; a[1] = a1;
  }
}
int kv_grad_accumulate(const bf16* dkv, const int32_t* rows, int B, int L, int width, float* acc, cudaStream_t stream) {
  ETP_REQUIRE(B > 0 && L > 0 && width > 0 && width % 8 == 0, "kv_grad_accumulate: bad shape");
  ETP_REQUIRE((reinterpret_cast<uintptr_t>(dkv) & 15) == 0 && (reinterpret_cast<uintptr_t>(acc) & 15) == 0,
              "kv_grad_accumulate: alignment");
  const int64_t n8 = static_cast<int64_t>(B) * L * (width / 8);
  int64_t blocks = (n8 + 255) / 256;
  if (blocks > 8 * num_sms()) blocks = 8 * num_sms();
  ETP_CHECK_CUDA(launch_pdl(kv_grad_accumulate_kernel, dim3(static_cast<int>(blocks)), dim3(256), 0, stream, dkv, rows, L,
                            width / 8, n8, acc));
  ETP_LAUNCHED();
  return ETP_OK;
}

// keep flags of elements [0, n) of one dropout site, exactly as the fused kernels evaluate them (test utility)
__global__ void dropout_mask_kernel(const Drop d, int64_t n, uint8_t* __restrict__ out) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (d.thr == 0 || drop_mul(d, static_cast<uint32_t>(i)) != 0.0f) ? 1 : 0;
}
int dropout_mask(DropHost d, int64_t n, uint8_t* out, cudaStream_t stream) {
  ETP_REQUIRE(out != nullptr && n >= 0 && n < (int64_t(1) << 32), "dropout_mask: bad arguments");
  if (n == 0) return ETP_OK;
  dropout_mask_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, stream>>>(Drop{d.key, d.thr, d.scale}, n, out);
  ETP_LAUNCHED();
  return ETP_OK;
}

}  // namespace etp
