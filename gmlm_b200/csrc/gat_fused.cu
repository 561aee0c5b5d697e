// gat_fused.cu — GAT edge-softmax aggregation (SURVEY §8a row A9, BASELINE.json configs[2]; an extension named by
// north_star with no counterpart in /root/reference — oracle: upstream GATConv restated in oracle/pyg_ref.py).
//
//   out[i,h,:] = sum_{e -> i} alpha[e,h] * z[src_e,h,:],
//   alpha[e,h] = exp(s[e,h] - max_i) / (sum_i exp(s - max_i) + 1e-16),   s[e,h] = leaky_relu(a_src[src_e,h] + a_dst[i,h])
//
// Edge features (upstream GATConv(edge_dim)): the `_eattr` entry points take a_edge [nnz, H], a per-(edge, head)
// score term in CSR order (loop entries included), read where a_src is read and added before the leaky ReLU:
// s[e,h] = leaky_relu((a_src[src_e,h] + a_edge[e,h]) + a_dst[i,h]), in the forward scan and in the backward's
// recomputed score alike.  Its gradient is d_score, which the backward edge pass writes anyway.  The term is the
// template flag E, so the instantiations without it (a_edge = NULL) carry no code for it.
//
// Forward = ONE pass over the in-edges of a destination row with an ONLINE softmax: the score is computed where
// the source row is gathered, the running maximum m, normaliser l and the fp32 accumulator are rescaled by
// exp(m_old - m_new) whenever the maximum grows, and alpha is never written (round 1: three passes over the scores
// into an [E, H] array, then a separate weighted aggregation).  Per row only (m, l) [N, H] are kept; the backward
// recomputes alpha from them.  Rows longer than `hub_thresh` are cut into chunks (the hub plan of the CSR): one
// warp per chunk produces a partial (m, l, acc), a final kernel merges the partials of a row in chunk order —
// the split-softmax identity  acc = sum_k acc_k exp(m_k - M),  l = sum_k l_k exp(m_k - M) — so a hub costs
// O(deg / chunks) per warp and the result is deterministic.
//
// Backward, edge pass (rows = destinations, the same hub plan): per edge  d_alpha = <g[i,h,:], z[src,h,:]>,
// d_e = alpha (keep * d_alpha - t[i,h])  with  t[i,h] = <g[i,h,:], out[i,h,:]>  (= sum_e alpha_e keep_e d_alpha_e,
// no extra pass), d_score = d_e * leaky_relu'(raw);  writes alpha_eff[e,h] (what the transposed aggregation of g
// needs), d_score[e,h], and da_dst[i,h] = sum_e d_score.  da_src and dz are then gathers over the transposed CSR.
//
// Attention dropout (upstream: F.dropout on alpha): keep[e,h] comes from a counter-based hash of (seed, CSR
// position, head), so forward, backward and `gmlm_gat_dropout_mask` (tests) agree without storing a mask.
//
// Lane mapping: one warp per row / chunk and head group; lane owns packs p = lane, lane+32, ... of the group's
// features (a pack never straddles heads: C % VEC == 0), at most CH packs per lane.
//
// Head groups: the heads of a row are independent in the softmax, so a row wider than one warp's CH packs is cut
// into groups of whole heads (GatParams::hg heads each), one per grid.y index, each walking the same CSR row or hub
// chunk.  A group reads and writes only its own heads; a_src, a_dst, m, l and the dropout hash keep the global head
// index and H as the stride, so the result does not depend on the cut.  Rows that fit one warp are one group
// (grid.y = 1, hg = H) and run the G = false instantiations, whose code has no group offsets at all; grouped rows run
// G = true at the widest CH of their path.
#include "common.cuh"

namespace gmlm {
namespace {

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// keep-probability test: splitmix64 of (seed, index) -> 24 random bits
__device__ __host__ __forceinline__ bool drop_keep(uint64_t seed, uint64_t idx, float p_drop) {
  uint64_t x = seed + 0x9E3779B97F4A7C15ull * (idx + 1);
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  x ^= x >> 31;
  return float(uint32_t(x >> 40)) * (1.0f / 16777216.0f) >= p_drop;
}

struct GatParams {
  const int32_t* rowptr;
  const int32_t* col;
  const void* z;
  int64_t ldz;
  const float* a_src;   // [num_src, H]
  const float* a_dst;   // [num_rows, H]
  int H, C;
  int hg;               // heads per group (grid.y = ceil(H / hg)); hg = H: the whole row in one group
  float slope, p_drop;
  uint64_t seed;
  int32_t hub_thresh;
  const float* a_edge;  // [nnz, H] in CSR order, read only by the E = true instantiations
};

template <typename T, int VEC, int CH, bool G>
struct Lane {
  int head[CH];
  bool valid[CH];
  int64_t f[CH];
  // features [h0*C, h1*C) of head group blockIdx.y (G), or all H*C features
  __device__ __forceinline__ void init(int lane, const GatParams& p) {
    int64_t f0 = 0, f1 = int64_t(p.H) * p.C;
    if constexpr (G) {
      const int h0 = int(blockIdx.y) * p.hg, h1 = min(h0 + p.hg, p.H);
      f0 = int64_t(h0) * p.C;
      f1 = int64_t(h1) * p.C;
    }
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
      f[ch] = f0 + int64_t(ch * 32 + lane) * VEC;
      valid[ch] = f[ch] < f1;
      head[ch] = valid[ch] ? int(f[ch] / p.C) : 0;
    }
  }
};

// online-softmax scan of edges [b, e) of destination row `row`
template <typename T, int VEC, int CH, bool G, bool E>
__device__ __forceinline__ void gat_scan(const GatParams& p, const Lane<T, VEC, CH, G>& ln, int64_t row, int32_t b, int32_t e,
                                         float (&m)[CH], float (&l)[CH], float (&acc)[CH][VEC]) {
  const T* __restrict__ z = static_cast<const T*>(p.z);
  float ad[CH];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    ad[ch] = ln.valid[ch] ? __ldg(p.a_dst + row * p.H + ln.head[ch]) : 0.f;
    m[ch] = -INFINITY;
    l[ch] = 0.f;
#pragma unroll
    for (int v = 0; v < VEC; ++v) acc[ch][v] = 0.f;
  }
  for (int32_t k = b; k < e; k += 2) {          // two edges in flight
    const bool two = k + 1 < e;
    const int32_t s0 = __ldg(p.col + k), s1 = two ? __ldg(p.col + k + 1) : s0;
    Pack<T, VEC> z0[CH], z1[CH];
    float as0[CH], as1[CH];
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
      if (!ln.valid[ch]) continue;
      as0[ch] = __ldg(p.a_src + int64_t(s0) * p.H + ln.head[ch]);
      if constexpr (E) as0[ch] += __ldg(p.a_edge + int64_t(k) * p.H + ln.head[ch]);
      z0[ch].load(z + int64_t(s0) * p.ldz + ln.f[ch]);
      if (two) {
        as1[ch] = __ldg(p.a_src + int64_t(s1) * p.H + ln.head[ch]);
        if constexpr (E) as1[ch] += __ldg(p.a_edge + int64_t(k + 1) * p.H + ln.head[ch]);
        z1[ch].load(z + int64_t(s1) * p.ldz + ln.f[ch]);
      }
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (u == 1 && !two) break;
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        if (!ln.valid[ch]) continue;
        const float s = lrelu((u ? as1[ch] : as0[ch]) + ad[ch], p.slope);
        const float mn = fmaxf(m[ch], s);
        const float sc = expf(m[ch] - mn);          // exp(-inf) = 0 on the first edge
        const float pe = expf(s - mn);
        l[ch] = l[ch] * sc + pe;
        const bool keep = p.p_drop <= 0.f || drop_keep(p.seed, uint64_t(k + u) * p.H + ln.head[ch], p.p_drop);
        const float w = keep ? pe : 0.f;
        float zf[VEC];
        (u ? z1[ch] : z0[ch]).unpack(zf);
#pragma unroll
        for (int v = 0; v < VEC; ++v) acc[ch][v] = fmaf(w, zf[v], acc[ch][v] * sc);
        m[ch] = mn;
      }
    }
  }
}

template <typename T, int VEC, int CH, bool G, bool E>
__global__ void __launch_bounds__(256) gat_rows_kernel(const GatParams p, int64_t num_rows, T* __restrict__ out,
                                                       int64_t ldo, float* __restrict__ m_out, float* __restrict__ l_out) {
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= num_rows) return;
  const int32_t b = __ldg(p.rowptr + r), e = __ldg(p.rowptr + r + 1);
  if (e - b > p.hub_thresh) return;                 // a hub row: chunk kernel + final kernel
  Lane<T, VEC, CH, G> ln;
  ln.init(lane, p);
  float m[CH], l[CH], acc[CH][VEC];
  gat_scan<T, VEC, CH, G, E>(p, ln, r, b, e, m, l, acc);
  const float keep_scale = p.p_drop > 0.f ? 1.0f / (1.0f - p.p_drop) : 1.0f;
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    if (!ln.valid[ch]) continue;
    const float inv = keep_scale / (l[ch] + 1e-16f);
    float o[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) o[v] = acc[ch][v] * inv;
    Pack<T, VEC> pk;
    pk.pack(o);
    pk.store(out + r * ldo + ln.f[ch]);
    if (ln.f[ch] % p.C == 0) {                      // first pack of a head: the row's softmax statistics
      m_out[r * p.H + ln.head[ch]] = m[ch];
      l_out[r * p.H + ln.head[ch]] = l[ch];
    }
  }
}

template <typename T, int VEC, int CH, bool G, bool E>
__global__ void __launch_bounds__(256) gat_chunk_kernel(const GatParams p, const int32_t* __restrict__ chunk_beg,
                                                        const int32_t* __restrict__ chunk_end,
                                                        const int32_t* __restrict__ chunk_row, int64_t n_chunks,
                                                        float* __restrict__ pm, float* __restrict__ pl,
                                                        float* __restrict__ pacc) {
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= n_chunks) return;
  Lane<T, VEC, CH, G> ln;
  ln.init(lane, p);
  float m[CH], l[CH], acc[CH][VEC];
  gat_scan<T, VEC, CH, G, E>(p, ln, __ldg(chunk_row + c), __ldg(chunk_beg + c), __ldg(chunk_end + c), m, l, acc);
  const int64_t hc = int64_t(p.H) * p.C;
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    if (!ln.valid[ch]) continue;
#pragma unroll
    for (int v = 0; v < VEC; ++v) pacc[c * hc + ln.f[ch] + v] = acc[ch][v];
    if (ln.f[ch] % p.C == 0) {
      pm[c * p.H + ln.head[ch]] = m[ch];
      pl[c * p.H + ln.head[ch]] = l[ch];
    }
  }
}

// merge the chunk partials of every hub row (chunk order => deterministic)
template <typename T>
__global__ void __launch_bounds__(256) gat_final_kernel(const int32_t* __restrict__ hub_row,
                                                        const int32_t* __restrict__ hub_chunk_ptr, int64_t n_hub, int H,
                                                        int C, float p_drop, const float* __restrict__ pm,
                                                        const float* __restrict__ pl, const float* __restrict__ pacc,
                                                        T* __restrict__ out, int64_t ldo, float* __restrict__ m_out,
                                                        float* __restrict__ l_out) {
  const int64_t hidx = blockIdx.x;
  if (hidx >= n_hub) return;
  const int32_t r = hub_row[hidx], c0 = hub_chunk_ptr[hidx], c1 = hub_chunk_ptr[hidx + 1];
  const int64_t hc = int64_t(H) * C;
  const float keep_scale = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
  for (int64_t f = threadIdx.x; f < hc; f += blockDim.x) {
    const int h = int(f / C);
    float M = -INFINITY;
    for (int32_t c = c0; c < c1; ++c) M = fmaxf(M, pm[int64_t(c) * H + h]);
    float L = 0.f, A = 0.f;
    for (int32_t c = c0; c < c1; ++c) {
      const float sc = expf(pm[int64_t(c) * H + h] - M);
      L = fmaf(pl[int64_t(c) * H + h], sc, L);
      A = fmaf(pacc[int64_t(c) * hc + f], sc, A);
    }
    out[int64_t(r) * ldo + f] = from_float<T>(A * keep_scale / (L + 1e-16f));
    if (f % C == 0) { m_out[int64_t(r) * H + h] = M; l_out[int64_t(r) * H + h] = L; }
  }
}

__global__ void chunk_rows_kernel(const int32_t* __restrict__ hub_row, const int32_t* __restrict__ hub_chunk_ptr,
                                  int64_t n_hub, int32_t* __restrict__ chunk_row) {
  const int64_t h = blockIdx.x;
  if (h >= n_hub) return;
  for (int32_t c = hub_chunk_ptr[h] + threadIdx.x; c < hub_chunk_ptr[h + 1]; c += blockDim.x) chunk_row[c] = hub_row[h];
}

// ---------------------------------------------------------------------------------- backward, edge pass
// one warp per (row | chunk): alpha_eff[k,h], d_score[k,h] for its edges, partial da_dst[., h]
template <typename T, int VEC, int CH, bool G, bool E>
__device__ __forceinline__ void gat_bwd_scan(const GatParams& p, const Lane<T, VEC, CH, G>& ln, int lane, int64_t row,
                                             int32_t b, int32_t e, const T* __restrict__ g, int64_t ldg,
                                             const float* __restrict__ m_in, const float* __restrict__ l_in,
                                             const float* __restrict__ t_in, float* __restrict__ alpha_eff,
                                             float* __restrict__ d_score, float* __restrict__ da_dst_out) {
  const T* __restrict__ z = static_cast<const T*>(p.z);
  float gf[CH][VEC];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    if (ln.valid[ch]) {
      Pack<T, VEC> pk;
      pk.load(g + row * ldg + ln.f[ch]);
      pk.unpack(gf[ch]);
    }
  }
  // lane j (< the group's head count) carries the per-head scalars of head h0 + j
  int h0 = 0, nh = p.H;
  if constexpr (G) {
    h0 = int(blockIdx.y) * p.hg;
    nh = min(p.hg, p.H - h0);
  }
  const int hh = h0 + (lane < nh ? lane : 0);
  const float ad = __ldg(p.a_dst + row * p.H + hh), mm = __ldg(m_in + row * p.H + hh);
  const float inv_l = 1.0f / (__ldg(l_in + row * p.H + hh) + 1e-16f), tt = __ldg(t_in + row * p.H + hh);
  const float keep_scale = p.p_drop > 0.f ? 1.0f / (1.0f - p.p_drop) : 1.0f;
  float dsum = 0.f;
  for (int32_t k = b; k < e; ++k) {
    const int32_t s = __ldg(p.col + k);
    float part[CH];
#pragma unroll
    for (int ch = 0; ch < CH; ++ch) {
      part[ch] = 0.f;
      if (!ln.valid[ch]) continue;
      Pack<T, VEC> pk;
      pk.load(z + int64_t(s) * p.ldz + ln.f[ch]);
      float zf[VEC];
      pk.unpack(zf);
#pragma unroll
      for (int v = 0; v < VEC; ++v) part[ch] = fmaf(gf[ch][v], zf[v], part[ch]);
    }
    float dot_mine = 0.f;                              // <g[row,h,:], z[s,h,:]> for h = h0 + lane
    for (int j = 0; j < nh; ++j) {
      float v = 0.f;
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) v += (ln.valid[ch] && ln.head[ch] == h0 + j) ? part[ch] : 0.f;
      v = warp_sum(v);
      if (lane == j) dot_mine = v;
    }
    if (lane < nh) {
      const int hd = G ? hh : lane;                    // this lane's head (global index)
      float as = __ldg(p.a_src + int64_t(s) * p.H + hd);
      if constexpr (E) as += __ldg(p.a_edge + int64_t(k) * p.H + hd);   // summed as in the forward's scan
      const float raw = as + ad;
      const float alpha = expf(lrelu(raw, p.slope) - mm) * inv_l;
      const bool keep = p.p_drop <= 0.f || drop_keep(p.seed, uint64_t(k) * p.H + hd, p.p_drop);
      const float ks = keep ? keep_scale : 0.f;
      const float de = alpha * (ks * dot_mine - tt);
      const float ds = raw > 0.f ? de : de * p.slope;
      alpha_eff[int64_t(k) * p.H + hd] = alpha * ks;
      d_score[int64_t(k) * p.H + hd] = ds;
      dsum += ds;
    }
  }
  if (lane < nh) da_dst_out[G ? hh : lane] = dsum;
}

template <typename T, int VEC, int CH, bool G, bool E>
__global__ void __launch_bounds__(256) gat_bwd_rows_kernel(const GatParams p, int64_t num_rows, const T* __restrict__ g,
                                                           int64_t ldg, const float* __restrict__ m_in,
                                                           const float* __restrict__ l_in, const float* __restrict__ t_in,
                                                           float* __restrict__ alpha_eff, float* __restrict__ d_score,
                                                           float* __restrict__ da_dst) {
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= num_rows) return;
  const int32_t b = __ldg(p.rowptr + r), e = __ldg(p.rowptr + r + 1);
  if (e - b > p.hub_thresh) return;
  Lane<T, VEC, CH, G> ln;
  ln.init(lane, p);
  gat_bwd_scan<T, VEC, CH, G, E>(p, ln, lane, r, b, e, g, ldg, m_in, l_in, t_in, alpha_eff, d_score, da_dst + r * p.H);
}

template <typename T, int VEC, int CH, bool G, bool E>
__global__ void __launch_bounds__(256) gat_bwd_chunk_kernel(const GatParams p, const int32_t* __restrict__ chunk_beg,
                                                            const int32_t* __restrict__ chunk_end,
                                                            const int32_t* __restrict__ chunk_row, int64_t n_chunks,
                                                            const T* __restrict__ g, int64_t ldg,
                                                            const float* __restrict__ m_in, const float* __restrict__ l_in,
                                                            const float* __restrict__ t_in, float* __restrict__ alpha_eff,
                                                            float* __restrict__ d_score, float* __restrict__ da_part) {
  const int64_t c = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (c >= n_chunks) return;
  Lane<T, VEC, CH, G> ln;
  ln.init(lane, p);
  gat_bwd_scan<T, VEC, CH, G, E>(p, ln, lane, __ldg(chunk_row + c), __ldg(chunk_beg + c), __ldg(chunk_end + c), g, ldg, m_in,
                           l_in, t_in, alpha_eff, d_score, da_part + c * p.H);
}

// da_dst[hub_row[h], :] = sum over the row's chunks, in chunk order
__global__ void gat_bwd_final_kernel(const int32_t* __restrict__ hub_row, const int32_t* __restrict__ hub_chunk_ptr,
                                     int64_t n_hub, int H, const float* __restrict__ da_part, float* __restrict__ da_dst) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_hub * H) return;
  const int64_t h = i / H;
  const int hd = int(i - h * H);
  float a = 0.f;
  for (int32_t c = hub_chunk_ptr[h]; c < hub_chunk_ptr[h + 1]; ++c) a += da_part[int64_t(c) * H + hd];
  da_dst[int64_t(hub_row[h]) * H + hd] = a;
}

__global__ void dropout_mask_kernel(uint64_t seed, int64_t n, float p_drop, uint8_t* __restrict__ keep) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) keep[i] = drop_keep(seed, uint64_t(i), p_drop) ? 1 : 0;
}

template <typename Fn>
int dispatch_geo(int dtype, int64_t hc, bool aligned, Fn&& fn) {
  // packs per lane: CH in {1, 2, 4, 8}; unaligned / odd widths take scalar packs
  if (dtype == GMLM_F32) {
    if (aligned) {
      const int64_t packs = hc / 4;
      if (packs <= 32) return fn.template operator()<float, 4, 1>();
      if (packs <= 64) return fn.template operator()<float, 4, 2>();
      if (packs <= 128) return fn.template operator()<float, 4, 4>();
      if (packs <= 256) return fn.template operator()<float, 4, 8>();
    } else {
      if (hc <= 32) return fn.template operator()<float, 1, 1>();
      if (hc <= 128) return fn.template operator()<float, 1, 4>();
      if (hc <= 256) return fn.template operator()<float, 1, 8>();
    }
  } else {
    if (aligned) {
      const int64_t packs = hc / 8;
      if (packs <= 32) return fn.template operator()<__nv_bfloat16, 8, 1>();
      if (packs <= 64) return fn.template operator()<__nv_bfloat16, 8, 2>();
      if (packs <= 128) return fn.template operator()<__nv_bfloat16, 8, 4>();
    } else {
      if (hc <= 32) return fn.template operator()<__nv_bfloat16, 1, 1>();
      if (hc <= 128) return fn.template operator()<__nv_bfloat16, 1, 4>();
      if (hc <= 256) return fn.template operator()<__nv_bfloat16, 1, 8>();
    }
  }
  return fail(GMLM_ERR_INVALID, "gat: heads * head_dim = %lld is wider than this kernel covers", (long long)hc);
}

// a row that fits one warp: the instantiation for its width, no group offsets (G = false); a row cut into head groups:
// the widest instantiation of its path (G = true).  E: the per-edge score term a_edge is read (a compile-time flag,
// so the instantiations without it are the code that runs when no term is passed)
template <bool E, typename Fn>
int dispatch_gat_e(int dtype, int64_t hc, bool aligned, int n_groups, Fn&& fn) {
  if (n_groups == 1)
    return dispatch_geo(dtype, hc, aligned, [&]<typename T, int VEC, int CH>() -> int {
      return fn.template operator()<T, VEC, CH, false, E>();
    });
  if (dtype == GMLM_F32)
    return aligned ? fn.template operator()<float, 4, 8, true, E>() : fn.template operator()<float, 1, 8, true, E>();
  return aligned ? fn.template operator()<__nv_bfloat16, 8, 4, true, E>()
                 : fn.template operator()<__nv_bfloat16, 1, 8, true, E>();
}

template <typename Fn>
int dispatch_gat(int dtype, int64_t hc, bool aligned, int n_groups, bool edge, Fn&& fn) {
  return edge ? dispatch_gat_e<true>(dtype, hc, aligned, n_groups, fn)
              : dispatch_gat_e<false>(dtype, hc, aligned, n_groups, fn);
}

inline bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// The head-group cut of a row: the fewest groups of whole heads whose width fits the widest instantiation of the
// path (1024 features on 16-byte packs, 256 on scalar packs), heads spread evenly over the groups.  A row that fits
// is one group of all H heads.
struct HeadGroups {
  int hg, n;
};
inline int head_groups(int heads, int head_dim, bool aligned, const char* who, HeadGroups* out) {
  const int64_t cap = aligned ? 1024 : 256;
  if (head_dim > cap)
    return fail(GMLM_ERR_INVALID, "%s: one head of head_dim = %d is wider than this kernel covers (%lld features%s)",
                who, head_dim, (long long)cap, aligned ? "" : " on the scalar path: odd or misaligned widths");
  const int per = int(cap / head_dim);               // most heads one group can take
  const int n = (heads + per - 1) / per;
  out->n = n;
  out->hg = (heads + n - 1) / n;
  return GMLM_OK;
}

}  // namespace
}  // namespace gmlm

using namespace gmlm;

extern "C" size_t gmlm_gat_workspace_bytes(int64_t n_chunks, int heads, int head_dim) {
  // chunk_row (i32) + pm, pl (f32 [chunks, H]) + pacc (f32 [chunks, H*C]); the head groups of a chunk write
  // disjoint heads / features of the same arrays, so the split needs no more
  return size_t(n_chunks) * (4 + size_t(heads) * 8 + size_t(heads) * head_dim * 4) + 1024;
}

extern "C" int gmlm_gat_fused_fwd_eattr(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z,
                                        int dtype, int64_t ldz, const float* a_src, const float* a_dst,
                                        const float* a_edge, int heads, int head_dim, float negative_slope,
                                        float p_drop, uint64_t seed, int32_t hub_thresh, int64_t n_hub,
                                        int64_t n_chunks, const int32_t* hub_row, const int32_t* hub_chunk_ptr,
                                        const int32_t* chunk_beg, const int32_t* chunk_end, void* ws, size_t ws_bytes,
                                        void* out, int64_t ldo, float* m_out, float* l_out, void* stream) {
  GMLM_REQUIRE(dtype == GMLM_F32 || dtype == GMLM_BF16, "gat_fused_fwd: dtype must be GMLM_F32 or GMLM_BF16");
  GMLM_REQUIRE(num_rows >= 0 && heads >= 1 && heads <= 32 && head_dim >= 1, "gat_fused_fwd: bad sizes (1..32 heads)");
  GMLM_REQUIRE(p_drop >= 0.f && p_drop < 1.f, "gat_fused_fwd: dropout must be in [0, 1)");
  const int64_t hc = int64_t(heads) * head_dim;
  GMLM_REQUIRE(ldz >= hc && ldo >= hc, "gat_fused_fwd: bad leading dimensions");
  if (num_rows == 0) return GMLM_OK;
  GMLM_REQUIRE(rowptr && col && z && a_src && a_dst && out && m_out && l_out, "gat_fused_fwd: null pointer");
  GMLM_REQUIRE(n_hub == 0 || (hub_row && hub_chunk_ptr && chunk_beg && chunk_end && ws &&
                              ws_bytes >= gmlm_gat_workspace_bytes(n_chunks, heads, head_dim)),
               "gat_fused_fwd: hub plan / workspace missing");
  const int v = dtype == GMLM_F32 ? 4 : 8;
  const bool aligned = head_dim % v == 0 && ldz % v == 0 && ldo % v == 0 && al16(z) && al16(out);
  HeadGroups hgp;
  if (int rc = head_groups(heads, head_dim, aligned, "gat_fused_fwd", &hgp)) return rc;
  cudaStream_t st = as_stream(stream);
  GatParams p{rowptr, col, z, ldz, a_src, a_dst, heads, head_dim, hgp.hg, negative_slope, p_drop, seed,
              n_hub > 0 ? hub_thresh : 0x7fffffff, a_edge};
  Carver cv(ws);
  int32_t* chunk_row = n_hub ? cv.take<int32_t>(n_chunks) : nullptr;
  float* pm = n_hub ? cv.take<float>(n_chunks * heads) : nullptr;
  float* pl = n_hub ? cv.take<float>(n_chunks * heads) : nullptr;
  float* pacc = n_hub ? cv.take<float>(n_chunks * hc) : nullptr;
  const dim3 grid(unsigned((num_rows * 32 + 255) / 256), unsigned(hgp.n));
  const dim3 cgrid(unsigned((n_chunks * 32 + 255) / 256), unsigned(hgp.n));
  const bool edge = a_edge != nullptr;
  int rc = dispatch_gat(dtype, hc, aligned, hgp.n, edge, [&]<typename T, int VEC, int CH, bool G, bool E>() -> int {
    gat_rows_kernel<T, VEC, CH, G, E><<<grid, 256, 0, st>>>(p, num_rows, static_cast<T*>(out), ldo, m_out, l_out);
    GMLM_LAUNCH_CHECK();
    if (n_hub) {
      chunk_rows_kernel<<<unsigned(n_hub), 128, 0, st>>>(hub_row, hub_chunk_ptr, n_hub, chunk_row);
      GMLM_LAUNCH_CHECK();
      gat_chunk_kernel<T, VEC, CH, G, E><<<cgrid, 256, 0, st>>>(p, chunk_beg, chunk_end, chunk_row, n_chunks, pm, pl, pacc);
      GMLM_LAUNCH_CHECK();
      gat_final_kernel<T><<<unsigned(n_hub), 256, 0, st>>>(hub_row, hub_chunk_ptr, n_hub, heads, head_dim, p_drop, pm, pl,
                                                           pacc, static_cast<T*>(out), ldo, m_out, l_out);
      GMLM_LAUNCH_CHECK();
    }
    return GMLM_OK;
  });
  return rc;
}

extern "C" int gmlm_gat_fused_fwd(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z, int dtype,
                                  int64_t ldz, const float* a_src, const float* a_dst, int heads, int head_dim,
                                  float negative_slope, float p_drop, uint64_t seed, int32_t hub_thresh, int64_t n_hub,
                                  int64_t n_chunks, const int32_t* hub_row, const int32_t* hub_chunk_ptr,
                                  const int32_t* chunk_beg, const int32_t* chunk_end, void* ws, size_t ws_bytes,
                                  void* out, int64_t ldo, float* m_out, float* l_out, void* stream) {
  return gmlm_gat_fused_fwd_eattr(rowptr, col, num_rows, z, dtype, ldz, a_src, a_dst, nullptr, heads, head_dim,
                                  negative_slope, p_drop, seed, hub_thresh, n_hub, n_chunks, hub_row, hub_chunk_ptr,
                                  chunk_beg, chunk_end, ws, ws_bytes, out, ldo, m_out, l_out, stream);
}

extern "C" int gmlm_gat_bwd_edges_eattr(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z,
                                        int dtype, int64_t ldz, const void* g, int64_t ldg, const float* a_src,
                                        const float* a_dst, const float* a_edge, const float* m_in, const float* l_in,
                                        const float* t_in, int heads, int head_dim, float negative_slope, float p_drop,
                                        uint64_t seed, int32_t hub_thresh, int64_t n_hub, int64_t n_chunks,
                                        const int32_t* hub_row, const int32_t* hub_chunk_ptr, const int32_t* chunk_beg,
                                        const int32_t* chunk_end, void* ws, size_t ws_bytes, float* alpha_eff,
                                        float* d_score, float* da_dst, void* stream) {
  GMLM_REQUIRE(dtype == GMLM_F32 || dtype == GMLM_BF16, "gat_bwd_edges: dtype must be GMLM_F32 or GMLM_BF16");
  GMLM_REQUIRE(num_rows >= 0 && heads >= 1 && heads <= 32 && head_dim >= 1, "gat_bwd_edges: bad sizes (1..32 heads)");
  const int64_t hc = int64_t(heads) * head_dim;
  GMLM_REQUIRE(ldz >= hc && ldg >= hc, "gat_bwd_edges: bad leading dimensions");
  if (num_rows == 0) return GMLM_OK;
  GMLM_REQUIRE(rowptr && col && z && g && a_src && a_dst && m_in && l_in && t_in && alpha_eff && d_score && da_dst,
               "gat_bwd_edges: null pointer");
  GMLM_REQUIRE(n_hub == 0 || (hub_row && hub_chunk_ptr && chunk_beg && chunk_end && ws &&
                              ws_bytes >= gmlm_gat_workspace_bytes(n_chunks, heads, head_dim)),
               "gat_bwd_edges: hub plan / workspace missing");
  const int v = dtype == GMLM_F32 ? 4 : 8;
  const bool aligned = head_dim % v == 0 && ldz % v == 0 && ldg % v == 0 && al16(z) && al16(g);
  HeadGroups hgp;
  if (int rc = head_groups(heads, head_dim, aligned, "gat_bwd_edges", &hgp)) return rc;
  cudaStream_t st = as_stream(stream);
  GatParams p{rowptr, col, z, ldz, a_src, a_dst, heads, head_dim, hgp.hg, negative_slope, p_drop, seed,
              n_hub > 0 ? hub_thresh : 0x7fffffff, a_edge};
  Carver cv(ws);
  int32_t* chunk_row = n_hub ? cv.take<int32_t>(n_chunks) : nullptr;
  float* da_part = n_hub ? cv.take<float>(n_chunks * heads) : nullptr;
  const dim3 grid(unsigned((num_rows * 32 + 255) / 256), unsigned(hgp.n));
  const dim3 cgrid(unsigned((n_chunks * 32 + 255) / 256), unsigned(hgp.n));
  const bool edge = a_edge != nullptr;
  return dispatch_gat(dtype, hc, aligned, hgp.n, edge, [&]<typename T, int VEC, int CH, bool G, bool E>() -> int {
    gat_bwd_rows_kernel<T, VEC, CH, G, E><<<grid, 256, 0, st>>>(p, num_rows, static_cast<const T*>(g), ldg, m_in, l_in, t_in,
                                                            alpha_eff, d_score, da_dst);
    GMLM_LAUNCH_CHECK();
    if (n_hub) {
      chunk_rows_kernel<<<unsigned(n_hub), 128, 0, st>>>(hub_row, hub_chunk_ptr, n_hub, chunk_row);
      GMLM_LAUNCH_CHECK();
      gat_bwd_chunk_kernel<T, VEC, CH, G, E><<<cgrid, 256, 0, st>>>(
          p, chunk_beg, chunk_end, chunk_row, n_chunks, static_cast<const T*>(g), ldg, m_in, l_in, t_in, alpha_eff,
          d_score, da_part);
      GMLM_LAUNCH_CHECK();
      gat_bwd_final_kernel<<<unsigned((n_hub * heads + 255) / 256), 256, 0, st>>>(hub_row, hub_chunk_ptr, n_hub, heads,
                                                                                  da_part, da_dst);
      GMLM_LAUNCH_CHECK();
    }
    return GMLM_OK;
  });
}

extern "C" int gmlm_gat_bwd_edges(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z, int dtype,
                                  int64_t ldz, const void* g, int64_t ldg, const float* a_src, const float* a_dst,
                                  const float* m_in, const float* l_in, const float* t_in, int heads, int head_dim,
                                  float negative_slope, float p_drop, uint64_t seed, int32_t hub_thresh, int64_t n_hub,
                                  int64_t n_chunks, const int32_t* hub_row, const int32_t* hub_chunk_ptr,
                                  const int32_t* chunk_beg, const int32_t* chunk_end, void* ws, size_t ws_bytes,
                                  float* alpha_eff, float* d_score, float* da_dst, void* stream) {
  return gmlm_gat_bwd_edges_eattr(rowptr, col, num_rows, z, dtype, ldz, g, ldg, a_src, a_dst, nullptr, m_in, l_in, t_in,
                                  heads, head_dim, negative_slope, p_drop, seed, hub_thresh, n_hub, n_chunks, hub_row,
                                  hub_chunk_ptr, chunk_beg, chunk_end, ws, ws_bytes, alpha_eff, d_score, da_dst, stream);
}

extern "C" int gmlm_gat_dropout_mask(uint64_t seed, int64_t n, float p_drop, uint8_t* keep, void* stream) {
  GMLM_REQUIRE(n >= 0 && (n == 0 || keep), "gat_dropout_mask: bad arguments");
  if (n == 0) return GMLM_OK;
  dropout_mask_kernel<<<unsigned((n + 255) / 256), 256, 0, as_stream(stream)>>>(seed, n, p_drop, keep);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}
