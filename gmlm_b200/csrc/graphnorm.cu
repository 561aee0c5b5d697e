// graphnorm.cu — whole-graph column statistics + normalisation (SURVEY §8a row A7:
// [PyG] GraphNorm(batch=None), called main.py:273,286,299,309), its backward, the optional
// fused exact-erf GELU of the layer closure (main.py:274), and the soft node masking of
// main.py:92-99 (row A11) with its masked column-sum backward.
//
// All of it is HBM-bound streaming over an [N, C] matrix: 128-bit loads along the channel
// dimension, every thread owns a fixed pack of channels and strides over rows, so the
// per-channel constants live in registers.  Column reductions are two-stage and
// order-fixed (per-CTA fp64 partials, then one in-order pass): no atomics, run-to-run
// deterministic.  The variance is one-pass,
//   E[(x - a*mu)^2] = (sum x^2 - sum x * mu * (2a - a^2)) / N,
// which cancels when the column's offset is large against its spread (worst at a = 1, PyG's init).
// For fp32 activations the column sums are therefore taken about a pivot, the column's first row p:
// d = x - p (exact), d^2 (one fp64 rounding) and both sums are formed in fp64, and sum x = sum d + N p,
// sum x^2 = sum d^2 + 2 p sum d + N p^2 are rebuilt once per column at the end.  A constant column
// then gives sum x^2 == fl(sum x * mu) bit for bit, so its variance is exactly 0 and rstd exactly
// 1/sqrt(eps); an offset column keeps about the two-pass form's accuracy up to offset/spread ~ 1e3,
// beyond which the fp32 mean the forward stores is the limit.  bf16 activations (8-bit mantissa, exact
// squares in fp32) keep fp32 running sums per thread.
#include <algorithm>

#include <type_traits>

#include "common.cuh"

namespace gmlm {
namespace {

constexpr int kCta = 256;
constexpr int kU = 4;    // row loads in flight per thread

struct Tile {
  int tpr;        // threads along the channel dimension (power of two <= 256)
  int rpc;        // rows covered by one CTA pass
  int64_t packs;  // packs per row
  dim3 grid;
};

inline Tile make_tile(int64_t num_rows, int64_t channels, int vec, int max_row_blocks) {
  Tile t;
  t.packs = (channels + vec - 1) / vec;
  int tpr = 1;
  while (tpr < t.packs && tpr < kCta) tpr <<= 1;
  t.tpr = tpr;
  t.rpc = kCta / tpr;
  int64_t col_tiles = (t.packs + tpr - 1) / tpr;
  int64_t row_blocks = (num_rows + t.rpc - 1) / t.rpc;
  int64_t want = std::max<int64_t>(1, int64_t(max_row_blocks) / col_tiles);
  if (row_blocks > want) row_blocks = want;
  if (row_blocks < 1) row_blocks = 1;
  t.grid = dim3((unsigned)col_tiles, (unsigned)row_blocks);
  return t;
}

// Exact-erf GELU (main.py:274, F.gelu default).  fp32 activations use erff/expf; bf16 activations
// (resolution 2^-8) use the Abramowitz-Stegun 7.1.26 rational form on MUFU.RCP/EX2: |error| of
// gelu and gelu' <= 5e-7 absolute (checked against fp64 over [-9, 9]) for a third of the
// instructions -- these kernels are issue-bound on the transcendental, not on HBM, otherwise.
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void phi_fast(float n, float& cdf, float& e) {
  const float t = rcp_approx(fmaf(0.3275911f * 0.70710678118654752440f, fabsf(n), 1.0f));
  float p = fmaf(t, 1.061405429f, -1.453152027f);
  p = fmaf(p, t, 1.421413741f);
  p = fmaf(p, t, -0.284496736f);
  p = fmaf(p, t, 0.254829592f);
  e = ex2_approx((n * n) * (-0.5f * 1.4426950408889634f));   // exp(-n^2/2)
  const float h = 0.5f * (p * t) * e;
  cdf = n >= 0.f ? 1.0f - h : h;
}
template <typename T>
__device__ __forceinline__ float gelu_f(float n) {
  if constexpr (sizeof(T) == 4) {
    return 0.5f * n * (1.0f + erff(n * 0.70710678118654752440f));
  } else {
    float cdf, e;
    phi_fast(n, cdf, e);
    return n * cdf;
  }
}
template <typename T>
__device__ __forceinline__ float gelu_grad_f(float n) {
  if constexpr (sizeof(T) == 4) {
    const float cdf = 0.5f * (1.0f + erff(n * 0.70710678118654752440f));
    const float pdf = 0.39894228040143267794f * expf(-0.5f * n * n);
    return cdf + n * pdf;
  } else {
    float cdf, e;
    phi_fast(n, cdf, e);
    return fmaf(n * 0.39894228040143267794f, e, cdf);
  }
}

// ---------------------------------------------------------------- column sums
// partial[(by * 2 + k) * C + c], k = 0: sum, k = 1: sum of squares; for fp32 taken about pivot[c] when
// pivot is given (colstats_final_kernel adds it back).  Optional row mask.
template <typename T, int VEC>
__global__ void __launch_bounds__(kCta) colstats_kernel(const T* __restrict__ x, int64_t num_rows, int64_t C,
                                                        int64_t ldx, const uint8_t* __restrict__ mask,
                                                        const float* __restrict__ pivot, int tpr,
                                                        double* __restrict__ partial) {
  __shared__ double sh[2][kCta];
  const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr, rpc = kCta / tpr;
  const int64_t cp = int64_t(blockIdx.x) * tpr + tx;
  const int64_t c0 = cp * VEC;
  const bool cvalid = c0 < C;
  // per-thread running sums: fp64 for fp32 activations; bf16 activations (resolution 4e-3, ~100 rows per
  // thread) keep them in fp32 and widen only for the cross-thread / cross-CTA reduction
  using AccT = typename std::conditional<sizeof(T) == 2, float, double>::type;
  AccT s[VEC], q[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) s[k] = q[k] = AccT(0);
  if constexpr (sizeof(T) == 4) {
    if (cvalid) {
      double p[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) p[k] = pivot ? double(pivot[c0 + k]) : 0.0;
      const int64_t stride = int64_t(gridDim.y) * rpc;
      for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += stride * kU) {
        Pack<T, VEC> v[kU];
        bool ok[kU];
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          const int64_t rr = r + u * stride;
          ok[u] = rr < num_rows && (mask == nullptr || mask[rr] != 0);
          if (ok[u]) v[u].load(x + rr * ldx + c0);
        }
#pragma unroll
        for (int u = 0; u < kU; ++u) {
          if (!ok[u]) continue;
          float f[VEC];
          v[u].unpack(f);
#pragma unroll
          for (int k = 0; k < VEC; ++k) {
            const double d = double(f[k]) - p[k];   // exact for fp32 values less than 2^29 apart in scale
            s[k] += d;
            q[k] = fma(d, d, q[k]);
          }
        }
      }
    }
  } else if (cvalid) {
    // kU row loads in flight per thread (latency, not issue, bounds a one-load loop); fp32 partials
    // over those rows, flushed into the fp64 accumulators: error of a partial <= kU ulp(fp32)
    const int64_t stride = int64_t(gridDim.y) * rpc;
    for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += stride * kU) {
      Pack<T, VEC> p[kU];
      bool ok[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int64_t rr = r + u * stride;
        ok[u] = rr < num_rows && (mask == nullptr || mask[rr] != 0);
        if (ok[u]) p[u].load(x + rr * ldx + c0);
      }
      float ps[VEC], pq[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) ps[k] = pq[k] = 0.f;
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (!ok[u]) continue;
        float f[VEC];
        p[u].unpack(f);
#pragma unroll
        for (int k = 0; k < VEC; ++k) { ps[k] += f[k]; pq[k] = fmaf(f[k], f[k], pq[k]); }
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) { s[k] += AccT(ps[k]); q[k] += AccT(pq[k]); }
    }
  }
  // reduce over ty in fixed order
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    sh[0][threadIdx.x] = double(s[k]);
    sh[1][threadIdx.x] = double(q[k]);
    __syncthreads();
    if (ty == 0 && cvalid) {
      double a = 0.0, b = 0.0;
      for (int y = 0; y < rpc; ++y) { a += sh[0][y * tpr + tx]; b += sh[1][y * tpr + tx]; }
      partial[(int64_t(blockIdx.y) * 2 + 0) * C + c0 + k] = a;
      partial[(int64_t(blockIdx.y) * 2 + 1) * C + c0 + k] = b;
    }
    __syncthreads();
  }
}

// 32 channels x 8 row-block ranges per CTA: group g sums the partials y in [g*span, (g+1)*span) in order (eight
// independent loads ahead of the adds), the eight range sums are combined in group order: a fixed summation tree
// (deterministic) whose serial chain is row_blocks / 8 long (one thread per channel walking all ~1000 partials made
// this tiny kernel cost as much as the statistics pass on L2-resident graphs).  With a pivot p (colstats of fp32
// rows) the sums are of d = x - p over num_rows rows and are turned back into sums of x and x^2 here; for a
// constant column (d == 0) that leaves out0 = N p exactly and out1 = fl(N p * p).
constexpr int kFinalGroups = 8;
__global__ void __launch_bounds__(32 * kFinalGroups) colstats_final_kernel(const double* __restrict__ partial,
                                                                           int row_blocks, int64_t C,
                                                                           const float* __restrict__ pivot,
                                                                           int64_t num_rows,
                                                                           double* __restrict__ out0,
                                                                           double* __restrict__ out1) {
  __shared__ double sh[2][kFinalGroups][32];
  const int cx = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int64_t c = int64_t(blockIdx.x) * 32 + cx;
  const int span = (row_blocks + kFinalGroups - 1) / kFinalGroups;
  const int y0 = g * span, y1 = min(row_blocks, y0 + span);
  double a = 0.0, b = 0.0;
  if (c < C) {
    int y = y0;
    for (; y + 4 <= y1; y += 4) {
      double va[4], vb[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        va[k] = partial[(int64_t(y + k) * 2 + 0) * C + c];
        vb[k] = partial[(int64_t(y + k) * 2 + 1) * C + c];
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) { a += va[k]; b += vb[k]; }
    }
    for (; y < y1; ++y) {
      a += partial[(int64_t(y) * 2 + 0) * C + c];
      b += partial[(int64_t(y) * 2 + 1) * C + c];
    }
  }
  sh[0][g][cx] = a;
  sh[1][g][cx] = b;
  __syncthreads();
  if (g == 0 && c < C) {
    double ta = 0.0, tb = 0.0;
#pragma unroll
    for (int k = 0; k < kFinalGroups; ++k) { ta += sh[0][k][cx]; tb += sh[1][k][cx]; }
    if (pivot) {
      const double p = pivot[c], np = double(num_rows) * p;
      tb = (tb + 2.0 * p * ta) + np * p;
      ta = ta + np;
    }
    if (out0) out0[c] = ta;
    if (out1) out1[c] = tb;
  }
}

// ---------------------------------------------------------------- forward
__global__ void graphnorm_prepare_kernel(const double* __restrict__ colsum, const double* __restrict__ colsq,
                                         const float* __restrict__ mean_scale, int64_t num_rows, int64_t C, float eps,
                                         float* __restrict__ mean_out, float* __restrict__ rstd_out) {
  const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double n = double(num_rows);
  const double mu = colsum[c] / n;
  const double a = double(mean_scale[c]);
  // sum x^2 - fl(sum x * mu): exactly 0 for a constant column whose sums colstats formed about a pivot
  double var = (colsq[c] - __dmul_rn(colsum[c], mu) * (2.0 * a - a * a)) / n;
  if (var < 0.0) var = 0.0;
  mean_out[c] = float(mu);
  rstd_out[c] = float(1.0 / sqrt(var + double(eps)));
}

template <typename T, int VEC>
__global__ void __launch_bounds__(kCta) graphnorm_fwd_kernel(const T* __restrict__ x, int64_t num_rows, int64_t C,
                                                             int64_t ldx, const float* __restrict__ mean,
                                                             const float* __restrict__ rstd,
                                                             const float* __restrict__ weight,
                                                             const float* __restrict__ bias,
                                                             const float* __restrict__ mean_scale, int fuse_gelu,
                                                             int tpr, T* __restrict__ y, int64_t ldy) {
  const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr, rpc = kCta / tpr;
  const int64_t c0 = (int64_t(blockIdx.x) * tpr + tx) * VEC;
  if (c0 >= C) return;
  float shift[VEC], k1[VEC], b[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    shift[k] = mean[c0 + k] * mean_scale[c0 + k];
    k1[k] = weight[c0 + k] * rstd[c0 + k];
    b[k] = bias[c0 + k];
  }
  const int64_t stride = int64_t(gridDim.y) * rpc;
  for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += stride * kU) {
    Pack<T, VEC> p[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u)
      if (r + u * stride < num_rows) p[u].load(x + (r + u * stride) * ldx + c0);
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int64_t rr = r + u * stride;
      if (rr >= num_rows) break;
      float f[VEC];
      p[u].unpack(f);
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const float n = (f[k] - shift[k]) * k1[k] + b[k];
        f[k] = fuse_gelu ? gelu_f<T>(n) : n;
      }
      p[u].pack(f);
      p[u].store(y + rr * ldy + c0);
    }
  }
}

// ---------------------------------------------------------------- backward
// dn = gy * gelu'(n) (or gy); partial sums of dn and dn*ohat
template <typename T, int VEC>
__global__ void __launch_bounds__(kCta, 2) graphnorm_bwd_stats_kernel(
    const T* __restrict__ x, const T* __restrict__ gy, int64_t num_rows, int64_t C, int64_t ldx, int64_t ldg,
    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ weight,
    const float* __restrict__ bias, const float* __restrict__ mean_scale, int fuse_gelu, int tpr,
    double* __restrict__ partial) {
  __shared__ double sh[2][kCta];
  const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr, rpc = kCta / tpr;
  const int64_t c0 = (int64_t(blockIdx.x) * tpr + tx) * VEC;
  const bool cvalid = c0 < C;
  double s[VEC], q[VEC];
  float shift[VEC], rs[VEC], wv[VEC], b[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    s[k] = q[k] = 0.0;
    shift[k] = rs[k] = wv[k] = b[k] = 0.f;
  }
  if (cvalid) {
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      shift[k] = mean[c0 + k] * mean_scale[c0 + k];
      rs[k] = rstd[c0 + k];
      wv[k] = weight[c0 + k];
      b[k] = bias[c0 + k];
    }
    const int64_t stride = int64_t(gridDim.y) * rpc;
    for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += stride * kU) {
      Pack<T, VEC> px[kU], pg[kU];
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        const int64_t rr = r + u * stride;
        if (rr < num_rows) {
          px[u].load(x + rr * ldx + c0);
          pg[u].load(gy + rr * ldg + c0);
        }
      }
      float ps[VEC], pq[VEC];
#pragma unroll
      for (int k = 0; k < VEC; ++k) ps[k] = pq[k] = 0.f;
#pragma unroll
      for (int u = 0; u < kU; ++u) {
        if (r + u * stride >= num_rows) break;
        float fx[VEC], fg[VEC];
        px[u].unpack(fx);
        pg[u].unpack(fg);
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          const float oh = (fx[k] - shift[k]) * rs[k];
          float dn = fg[k];
          if (fuse_gelu) dn *= gelu_grad_f<T>(oh * wv[k] + b[k]);
          ps[k] += dn;
          pq[k] = fmaf(dn, oh, pq[k]);
        }
      }
#pragma unroll
      for (int k = 0; k < VEC; ++k) { s[k] += double(ps[k]); q[k] += double(pq[k]); }
    }
  }
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    sh[0][threadIdx.x] = s[k];
    sh[1][threadIdx.x] = q[k];
    __syncthreads();
    if (ty == 0 && cvalid) {
      double a = 0.0, bb = 0.0;
      for (int y = 0; y < rpc; ++y) { a += sh[0][y * tpr + tx]; bb += sh[1][y * tpr + tx]; }
      partial[(int64_t(blockIdx.y) * 2 + 0) * C + c0 + k] = a;
      partial[(int64_t(blockIdx.y) * 2 + 1) * C + c0 + k] = bb;
    }
    __syncthreads();
  }
}

// per-channel constants of the input gradient + parameter gradients
//   dx = k1 * (dn - ohat * k2) - k3,  k1 = w*rstd, k2 = S2/N, k3 = (a/N) * sum(do)
__global__ void graphnorm_bwd_params_kernel(const double* __restrict__ sum_g, const double* __restrict__ sum_go,
                                            const float* __restrict__ mean, const float* __restrict__ rstd,
                                            const float* __restrict__ weight, const float* __restrict__ mean_scale,
                                            int64_t num_rows, int64_t C, float* __restrict__ g_weight,
                                            float* __restrict__ g_bias, float* __restrict__ g_mean_scale) {
  const int64_t c = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const double s1 = sum_g[c], s2 = sum_go[c];
  const double mu = mean[c], rs = rstd[c], w = weight[c], a = mean_scale[c];
  const double sum_do = w * rs * (s1 - s2 * rs * mu * (1.0 - a));
  if (g_weight) g_weight[c] = float(s2);
  if (g_bias) g_bias[c] = float(s1);
  if (g_mean_scale) g_mean_scale[c] = float(-mu * sum_do);
}

template <typename T, int VEC>
__global__ void __launch_bounds__(kCta, 2) graphnorm_bwd_apply_kernel(
    const T* __restrict__ x, const T* __restrict__ gy, int64_t num_rows, int64_t C, int64_t ldx, int64_t ldg,
    const float* __restrict__ mean, const float* __restrict__ rstd, const float* __restrict__ weight,
    const float* __restrict__ bias, const float* __restrict__ mean_scale, int fuse_gelu,
    const double* __restrict__ sum_g, const double* __restrict__ sum_go, int64_t stat_rows, int tpr,
    T* __restrict__ gx, int64_t ldgx) {
  const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr, rpc = kCta / tpr;
  const int64_t c0 = (int64_t(blockIdx.x) * tpr + tx) * VEC;
  if (c0 >= C) return;
  float shift[VEC], rs[VEC], wv[VEC], b[VEC], k1[VEC], k2[VEC], k3[VEC];
  const double n = double(stat_rows);
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    const double mu = mean[c0 + k], r = rstd[c0 + k], w = weight[c0 + k], a = mean_scale[c0 + k];
    const double s1 = sum_g[c0 + k], s2 = sum_go[c0 + k];
    const double sum_do = w * r * (s1 - s2 * r * mu * (1.0 - a));
    shift[k] = float(mu) * float(a);
    rs[k] = float(r);
    wv[k] = float(w);
    b[k] = bias[c0 + k];
    k1[k] = float(w * r);
    k2[k] = float(s2 / n);
    k3[k] = float(a * sum_do / n);
  }
  const int64_t stride = int64_t(gridDim.y) * rpc;
  for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += stride * kU) {
    Pack<T, VEC> px[kU], pg[kU];
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int64_t rr = r + u * stride;
      if (rr < num_rows) {
        px[u].load(x + rr * ldx + c0);
        pg[u].load(gy + rr * ldg + c0);
      }
    }
#pragma unroll
    for (int u = 0; u < kU; ++u) {
      const int64_t rr = r + u * stride;
      if (rr >= num_rows) break;
      float fx[VEC], fg[VEC];
      px[u].unpack(fx);
      pg[u].unpack(fg);
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const float oh = (fx[k] - shift[k]) * rs[k];
        float dn = fg[k];
        if (fuse_gelu) dn *= gelu_grad_f<T>(oh * wv[k] + b[k]);
        fg[k] = k1[k] * (dn - oh * k2[k]) - k3[k];
      }
      pg[u].pack(fg);
      pg[u].store(gx + rr * ldgx + c0);
    }
  }
}

// ---------------------------------------------------------------- soft masking (A11)
template <typename T, int VEC>
__global__ void __launch_bounds__(kCta) soft_mask_fwd_kernel(const T* __restrict__ x, int64_t num_rows, int64_t F,
                                                             int64_t ldx, const uint8_t* __restrict__ mask,
                                                             const float* __restrict__ token, float beta,
                                                             float one_minus_beta, int tpr, T* __restrict__ y,
                                                             int64_t ldy) {
  const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr, rpc = kCta / tpr;
  const int64_t c0 = (int64_t(blockIdx.x) * tpr + tx) * VEC;
  if (c0 >= F) return;
  float bt[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) bt[k] = __fmul_rn(beta, token[c0 + k]);
  for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += int64_t(gridDim.y) * rpc) {
    Pack<T, VEC> p;
    p.load(x + r * ldx + c0);
    if (mask[r]) {
      float f[VEC];
      p.unpack(f);
      // (1-beta)*x + beta*t with the reference's rounding sequence (no FMA contraction)
#pragma unroll
      for (int k = 0; k < VEC; ++k) f[k] = __fadd_rn(__fmul_rn(one_minus_beta, f[k]), bt[k]);
      p.pack(f);
    }
    p.store(y + r * ldy + c0);
  }
}

template <typename T, int VEC>
__global__ void __launch_bounds__(kCta) soft_mask_gx_kernel(const T* __restrict__ gy, int64_t num_rows, int64_t F,
                                                            int64_t ldg, const uint8_t* __restrict__ mask,
                                                            float one_minus_beta, int tpr, T* __restrict__ gx,
                                                            int64_t ldgx) {
  const int tx = threadIdx.x % tpr, ty = threadIdx.x / tpr, rpc = kCta / tpr;
  const int64_t c0 = (int64_t(blockIdx.x) * tpr + tx) * VEC;
  if (c0 >= F) return;
  for (int64_t r = int64_t(blockIdx.y) * rpc + ty; r < num_rows; r += int64_t(gridDim.y) * rpc) {
    Pack<T, VEC> p;
    p.load(gy + r * ldg + c0);
    if (mask[r]) {
      float f[VEC];
      p.unpack(f);
#pragma unroll
      for (int k = 0; k < VEC; ++k) f[k] = __fmul_rn(one_minus_beta, f[k]);
      p.pack(f);
    }
    p.store(gx + r * ldgx + c0);
  }
}

__global__ void scale_to_f32_kernel(const double* __restrict__ in, float scale, int64_t n, float* __restrict__ out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) out[i] = float(double(scale) * in[i]);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

constexpr int kMaxRowBlocks = 148 * 8;

// CTAs of `kernel` that are resident at once on the whole device: the streaming kernels run exactly one
// wave of them (each thread strides over the rows), so there is no partial last wave.
template <auto Kernel>
int resident_ctas() {
  static int cached[kMaxDevices] = {};   // per kernel instantiation and device; benign race (same value)
  const int dev = current_device();
  if (cached[dev] == 0) {
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, Kernel, kCta, 0) != cudaSuccess || occ < 1) occ = 1;
    cached[dev] = std::min(occ * num_sms(), kMaxRowBlocks);
  }
  return cached[dev];
}

// dispatch helper: calls fn.template operator()<T, VEC>()
template <typename Fn>
int dispatch(int dtype, bool vec_ok, Fn&& fn) {
  if (dtype == GMLM_F32) return vec_ok ? fn.template operator()<float, 4>() : fn.template operator()<float, 1>();
  if (dtype == GMLM_BF16)
    return vec_ok ? fn.template operator()<__nv_bfloat16, 8>() : fn.template operator()<__nv_bfloat16, 1>();
  return fail(GMLM_ERR_INVALID, "dtype must be GMLM_F32 or GMLM_BF16");
}

inline bool vec_ok(int dtype, int64_t C, std::initializer_list<const void*> ptrs, std::initializer_list<int64_t> lds) {
  const int v = dtype == GMLM_F32 ? 4 : 8;
  if (C % v) return false;
  for (const void* p : ptrs) if (!aligned16(p)) return false;
  for (int64_t l : lds) if (l % v) return false;
  return true;
}

size_t partial_bytes(int64_t C) { return size_t(kMaxRowBlocks) * 2 * size_t(C) * sizeof(double) + 256; }

}  // namespace
}  // namespace gmlm

using namespace gmlm;

extern "C" {

size_t gmlm_colstats_workspace_bytes(int64_t /*num_rows*/, int64_t channels) { return partial_bytes(channels); }

static int colstats_impl(const void* x, int dtype, int64_t N, int64_t C, int64_t ldx, const uint8_t* mask,
                         double* out0, double* out1, void* ws, size_t ws_bytes, cudaStream_t st) {
  GMLM_REQUIRE(N >= 0 && C >= 0 && ldx >= C, "colstats: bad sizes");
  if (C == 0) return GMLM_OK;
  GMLM_REQUIRE(ws && ws_bytes >= partial_bytes(C), "colstats: workspace too small");
  double* partial = static_cast<double*>(ws);
  const bool v = vec_ok(dtype, C, {x}, {ldx});
  // fp32 sums are taken about the first row (a row mask would leave the pivoted row count unknown)
  const float* pivot = dtype == GMLM_F32 && N > 0 && mask == nullptr ? static_cast<const float*>(x) : nullptr;
  int row_blocks = 1;
  int rc = dispatch(dtype, v, [&]<typename T, int VEC>() -> int {
    Tile t = make_tile(N, C, VEC, resident_ctas<colstats_kernel<T, VEC>>());
    row_blocks = int(t.grid.y);
    colstats_kernel<T, VEC><<<t.grid, kCta, 0, st>>>(static_cast<const T*>(x), N, C, ldx, mask, pivot, t.tpr,
                                                     partial);
    GMLM_LAUNCH_CHECK();
    return GMLM_OK;
  });
  if (rc) return rc;
  colstats_final_kernel<<<unsigned((C + 31) / 32), 32 * kFinalGroups, 0, st>>>(partial, row_blocks, C, pivot, N,
                                                                               out0, out1);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

int gmlm_colstats(const void* x, int dtype, int64_t N, int64_t C, int64_t ldx, double* colsum, double* colsq,
                  void* ws, size_t ws_bytes, void* stream) {
  return colstats_impl(x, dtype, N, C, ldx, nullptr, colsum, colsq, ws, ws_bytes, as_stream(stream));
}

int gmlm_graphnorm_fwd(const void* x, int dtype, int64_t N, int64_t C, int64_t ldx, const double* colsum,
                       const double* colsq, const float* weight, const float* bias, const float* mean_scale,
                       float eps, int fuse_gelu, void* y, int64_t ldy, float* mean_out, float* rstd_out,
                       int64_t stat_rows, void* stream) {
  if (stat_rows <= 0) stat_rows = N;
  GMLM_REQUIRE(N >= 0 && stat_rows >= 1 && stat_rows >= N && C >= 0 && ldx >= C && ldy >= C, "graphnorm_fwd: bad sizes");
  if (C == 0) return GMLM_OK;
  GMLM_REQUIRE((N == 0 || (x && y)) && colsum && colsq && weight && bias && mean_scale && mean_out && rstd_out,
               "graphnorm_fwd: null pointer");
  cudaStream_t st = as_stream(stream);
  graphnorm_prepare_kernel<<<unsigned((C + 255) / 256), 256, 0, st>>>(colsum, colsq, mean_scale, stat_rows, C, eps,
                                                                      mean_out, rstd_out);
  GMLM_LAUNCH_CHECK();
  if (N == 0) return GMLM_OK;
  const bool v = vec_ok(dtype, C, {x, y}, {ldx, ldy});
  return dispatch(dtype, v, [&]<typename T, int VEC>() -> int {
    Tile t = make_tile(N, C, VEC, resident_ctas<graphnorm_fwd_kernel<T, VEC>>());
    graphnorm_fwd_kernel<T, VEC><<<t.grid, kCta, 0, st>>>(static_cast<const T*>(x), N, C, ldx, mean_out, rstd_out,
                                                          weight, bias, mean_scale, fuse_gelu, t.tpr,
                                                          static_cast<T*>(y), ldy);
    GMLM_LAUNCH_CHECK();
    return GMLM_OK;
  });
}

int gmlm_graphnorm_bwd_stats(const void* x, const void* gy, int dtype, int64_t N, int64_t C, int64_t ldx,
                             int64_t ldg, const float* mean, const float* rstd, const float* weight,
                             const float* bias, const float* mean_scale, int fuse_gelu, double* sum_g,
                             double* sum_go, void* ws, size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(N >= 0 && C >= 0 && ldx >= C && ldg >= C, "graphnorm_bwd_stats: bad sizes");
  if (C == 0) return GMLM_OK;
  GMLM_REQUIRE(ws && ws_bytes >= partial_bytes(C), "graphnorm_bwd_stats: workspace too small");
  cudaStream_t st = as_stream(stream);
  double* partial = static_cast<double*>(ws);
  const bool v = vec_ok(dtype, C, {x, gy}, {ldx, ldg});
  int row_blocks = 1;
  int rc = dispatch(dtype, v, [&]<typename T, int VEC>() -> int {
    Tile t = make_tile(N, C, VEC, resident_ctas<graphnorm_bwd_stats_kernel<T, VEC>>());
    row_blocks = int(t.grid.y);
    graphnorm_bwd_stats_kernel<T, VEC><<<t.grid, kCta, 0, st>>>(static_cast<const T*>(x), static_cast<const T*>(gy),
                                                                N, C, ldx, ldg, mean, rstd, weight, bias, mean_scale,
                                                                fuse_gelu, t.tpr, partial);
    GMLM_LAUNCH_CHECK();
    return GMLM_OK;
  });
  if (rc) return rc;
  colstats_final_kernel<<<unsigned((C + 31) / 32), 32 * kFinalGroups, 0, st>>>(partial, row_blocks, C, nullptr, N,
                                                                               sum_g, sum_go);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

int gmlm_graphnorm_bwd_apply(const void* x, const void* gy, int dtype, int64_t N, int64_t C, int64_t ldx,
                             int64_t ldg, const float* mean, const float* rstd, const float* weight,
                             const float* bias, const float* mean_scale, int fuse_gelu, const double* sum_g,
                             const double* sum_go, void* gx, int64_t ldgx, float* g_weight, float* g_bias,
                             float* g_mean_scale, int64_t stat_rows, void* stream) {
  if (stat_rows <= 0) stat_rows = N;
  GMLM_REQUIRE(N >= 0 && stat_rows >= 1 && stat_rows >= N && C >= 0 && ldx >= C && ldg >= C,
               "graphnorm_bwd_apply: bad sizes");
  if (C == 0) return GMLM_OK;
  cudaStream_t st = as_stream(stream);
  graphnorm_bwd_params_kernel<<<unsigned((C + 255) / 256), 256, 0, st>>>(sum_g, sum_go, mean, rstd, weight,
                                                                         mean_scale, stat_rows, C, g_weight, g_bias,
                                                                         g_mean_scale);
  GMLM_LAUNCH_CHECK();
  if (gx == nullptr || N == 0) return GMLM_OK;
  GMLM_REQUIRE(ldgx >= C, "graphnorm_bwd_apply: bad ldgx");
  const bool v = vec_ok(dtype, C, {x, gy, gx}, {ldx, ldg, ldgx});
  return dispatch(dtype, v, [&]<typename T, int VEC>() -> int {
    Tile t = make_tile(N, C, VEC, resident_ctas<graphnorm_bwd_apply_kernel<T, VEC>>());
    graphnorm_bwd_apply_kernel<T, VEC><<<t.grid, kCta, 0, st>>>(
        static_cast<const T*>(x), static_cast<const T*>(gy), N, C, ldx, ldg, mean, rstd, weight, bias, mean_scale,
        fuse_gelu, sum_g, sum_go, stat_rows, t.tpr, static_cast<T*>(gx), ldgx);
    GMLM_LAUNCH_CHECK();
    return GMLM_OK;
  });
}

int gmlm_soft_mask_fwd(const void* x, int dtype, int64_t N, int64_t F, int64_t ldx, const uint8_t* mask,
                       const float* token, float beta, void* y, int64_t ldy, void* stream) {
  GMLM_REQUIRE(N >= 0 && F >= 0 && ldx >= F && ldy >= F, "soft_mask_fwd: bad sizes");
  if (N == 0 || F == 0) return GMLM_OK;
  GMLM_REQUIRE(x && y && mask && token, "soft_mask_fwd: null pointer");
  cudaStream_t st = as_stream(stream);
  const float omb = float(1.0 - double(beta));
  const bool v = vec_ok(dtype, F, {x, y}, {ldx, ldy});
  return dispatch(dtype, v, [&]<typename T, int VEC>() -> int {
    Tile t = make_tile(N, F, VEC, kMaxRowBlocks * 4);
    soft_mask_fwd_kernel<T, VEC><<<t.grid, kCta, 0, st>>>(static_cast<const T*>(x), N, F, ldx, mask, token, beta, omb,
                                                          t.tpr, static_cast<T*>(y), ldy);
    GMLM_LAUNCH_CHECK();
    return GMLM_OK;
  });
}

size_t gmlm_soft_mask_bwd_workspace_bytes(int64_t /*num_rows*/, int64_t feat) {
  return partial_bytes(feat) + size_t(feat) * sizeof(double) + 256;
}

int gmlm_soft_mask_bwd(const void* gy, int dtype, int64_t N, int64_t F, int64_t ldg, const uint8_t* mask, float beta,
                       float* g_token, void* gx, int64_t ldgx, void* ws, size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(N >= 0 && F >= 0 && ldg >= F, "soft_mask_bwd: bad sizes");
  if (F == 0) return GMLM_OK;
  GMLM_REQUIRE(ws && ws_bytes >= gmlm_soft_mask_bwd_workspace_bytes(N, F), "soft_mask_bwd: workspace too small");
  cudaStream_t st = as_stream(stream);
  if (g_token) {
    Carver cv(ws);
    double* colsum = cv.take<double>(F);
    void* part = cv.take<char>(0);
    int rc = colstats_impl(gy, dtype, N, F, ldg, mask, colsum, nullptr, part, ws_bytes - cv.used(), st);
    if (rc) return rc;
    scale_to_f32_kernel<<<unsigned((F + 255) / 256), 256, 0, st>>>(colsum, beta, F, g_token);
    GMLM_LAUNCH_CHECK();
  }
  if (gx && N > 0) {
    GMLM_REQUIRE(ldgx >= F, "soft_mask_bwd: bad ldgx");
    const float omb = float(1.0 - double(beta));
    const bool v = vec_ok(dtype, F, {gy, gx}, {ldg, ldgx});
    return dispatch(dtype, v, [&]<typename T, int VEC>() -> int {
      Tile t = make_tile(N, F, VEC, kMaxRowBlocks * 4);
      soft_mask_gx_kernel<T, VEC><<<t.grid, kCta, 0, st>>>(static_cast<const T*>(gy), N, F, ldg, mask, omb, t.tpr,
                                                           static_cast<T*>(gx), ldgx);
      GMLM_LAUNCH_CHECK();
      return GMLM_OK;
    });
  }
  return GMLM_OK;
}

}  // extern "C"
