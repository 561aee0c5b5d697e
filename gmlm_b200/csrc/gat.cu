// gat.cu — edge scores for the two aggregation variants north_star names beside the RGCN mean
// (SURVEY §8a rows A8 and A9; extensions with no counterpart in /root/reference — their oracle is
// the restatement of upstream GCNConv / GATConv in oracle/pyg_ref.py):
//
//   gcn_edge_weights : w_e = deg[src]^-1/2 * deg[dst]^-1/2      (deg = in-degree incl. self-loops)
//   segment_sum_f32  : out[r,h] = sum_{i in row r} vals[idx[i], h]   (scatter of edge scalars as a gather)
//   gat_loop_fill    : per-edge scores in input order -> forward-CSR order, each row's loop entry = the mean of
//                      the row's other entries (upstream add_self_loops(fill_value="mean")), and its backward
//
// The GAT edge-softmax itself lives in gat_fused.cu (one-pass online softmax fused into the gather).
// One warp per row, lanes stride over the row's edges, warp-shuffle reductions in a fixed order
// (deterministic).  Scalars are fp32.
#include "common.cuh"

namespace gmlm {
namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__global__ void __launch_bounds__(256) deg_from_rowptr_rsqrt_kernel(const int32_t* __restrict__ rowptr, int64_t n,
                                                                    float* __restrict__ dis) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int32_t d = rowptr[i + 1] - rowptr[i];
  dis[i] = d > 0 ? 1.0f / sqrtf(float(d)) : 0.f;   // deg^-1/2 with inf -> 0, as upstream gcn_norm
}

// CSR keyed on dst: w[e] = dis[col[e]] * dis[row]
__global__ void __launch_bounds__(256) gcn_weights_kernel(const int32_t* __restrict__ rowptr,
                                                          const int32_t* __restrict__ col, int64_t num_rows,
                                                          const float* __restrict__ dis, float* __restrict__ w) {
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= num_rows) return;
  const int32_t b = rowptr[r], e = rowptr[r + 1];
  const float dr = dis[r];
  for (int32_t k = b + lane; k < e; k += 32) w[k] = __fmul_rn(__fmul_rn(dis[col[k]], 1.0f), dr);
}

// out[r,h] = sum_{i in row r} vals[idx[i], h]: one warp per row, lanes stride over the row's entries, fixed-order
// shuffle reduction (deterministic; a hub row costs O(deg / 32) per lane instead of O(deg) in one thread)
__global__ void __launch_bounds__(256) segment_sum_kernel(const float* __restrict__ vals,
                                                          const int64_t* __restrict__ idx,
                                                          const int32_t* __restrict__ rowptr, int64_t num_rows, int H,
                                                          float* __restrict__ out) {
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= num_rows) return;
  const int32_t b = rowptr[r], e = rowptr[r + 1];
  for (int h = 0; h < H; ++h) {
    float a = 0.f;
    for (int32_t k = b + lane; k < e; k += 32) a += vals[(idx ? idx[k] : int64_t(k)) * H + h];
    a = warp_sum(a);
    if (lane == 0) out[r * H + h] = a;
  }
}

// one warp per row r: a_edge[k,h] = alpha[csr_src[k],h] for the row's kept entries, and at the row's loop entry
// loop_csr[r] the mean of those (0 without any: the sum is 0 and the count is clamped at 1)
__global__ void __launch_bounds__(256) loop_fill_kernel(const float* __restrict__ alpha,
                                                        const int32_t* __restrict__ csr_src,
                                                        const int32_t* __restrict__ loop_csr,
                                                        const int32_t* __restrict__ rowptr, int64_t num_rows, int H,
                                                        float* __restrict__ a_edge) {
  const int64_t r = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= num_rows) return;
  const int32_t b = rowptr[r], e = rowptr[r + 1], lp = loop_csr[r];
  const float inv_cnt = 1.0f / float(max(e - b - 1, 1));
  for (int h = 0; h < H; ++h) {
    float a = 0.f;
    for (int32_t k = b + lane; k < e; k += 32) {
      if (k == lp) continue;
      const float v = alpha[int64_t(csr_src[k]) * H + h];
      a_edge[int64_t(k) * H + h] = v;
      a += v;
    }
    a = warp_sum(a);
    if (lane == 0) a_edge[int64_t(lp) * H + h] = a * inv_cnt;
  }
}

// one thread per (input edge j, head): d_alpha = g[in2csr[j]] + g[loop of dst_j] / cnt(dst_j); 0 for a dropped loop
__global__ void __launch_bounds__(256) loop_fill_bwd_kernel(const float* __restrict__ g,
                                                            const int32_t* __restrict__ in2csr,
                                                            const int32_t* __restrict__ in_dst,
                                                            const int32_t* __restrict__ loop_csr,
                                                            const int32_t* __restrict__ rowptr, int64_t num_edges,
                                                            int H, float* __restrict__ d_alpha) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= num_edges * H) return;
  const int64_t j = i / H;
  const int h = int(i - j * H);
  const int32_t c = in2csr[j];
  float d = 0.f;
  if (c >= 0) {
    const int32_t r = in_dst[j];
    const float inv_cnt = 1.0f / float(max(rowptr[r + 1] - rowptr[r] - 1, 1));
    d = g[int64_t(c) * H + h] + g[int64_t(loop_csr[r]) * H + h] * inv_cnt;
  }
  d_alpha[i] = d;
}

}  // namespace
}  // namespace gmlm

using namespace gmlm;

extern "C" int gmlm_gcn_edge_weights(const int32_t* rowptr, const int32_t* col, int64_t num_rows, float* dis_ws,
                                     float* w, void* stream) {
  GMLM_REQUIRE(num_rows >= 0, "gcn_edge_weights: bad sizes");
  if (num_rows == 0) return GMLM_OK;
  GMLM_REQUIRE(rowptr && col && dis_ws && w, "gcn_edge_weights: null pointer");
  cudaStream_t st = as_stream(stream);
  deg_from_rowptr_rsqrt_kernel<<<unsigned((num_rows + 255) / 256), 256, 0, st>>>(rowptr, num_rows, dis_ws);
  GMLM_LAUNCH_CHECK();
  gcn_weights_kernel<<<unsigned((num_rows * 32 + 255) / 256), 256, 0, st>>>(rowptr, col, num_rows, dis_ws, w);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

extern "C" int gmlm_segment_sum_f32(const float* vals, const int64_t* idx, const int32_t* rowptr, int64_t num_rows,
                                    int heads, float* out, void* stream) {
  GMLM_REQUIRE(num_rows >= 0 && heads >= 1, "segment_sum: bad sizes");
  if (num_rows == 0) return GMLM_OK;
  GMLM_REQUIRE(vals && rowptr && out, "segment_sum: null pointer");
  segment_sum_kernel<<<unsigned((num_rows * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(vals, idx, rowptr, num_rows,
                                                                                           heads, out);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

extern "C" int gmlm_gat_loop_fill(const float* alpha, const int32_t* csr_src, const int32_t* loop_csr,
                                  const int32_t* rowptr, int64_t num_rows, int heads, float* a_edge, void* stream) {
  GMLM_REQUIRE(num_rows >= 0 && heads >= 1, "gat_loop_fill: bad sizes");
  if (num_rows == 0) return GMLM_OK;
  GMLM_REQUIRE(csr_src && loop_csr && rowptr && a_edge, "gat_loop_fill: null pointer");
  loop_fill_kernel<<<unsigned((num_rows * 32 + 255) / 256), 256, 0, as_stream(stream)>>>(alpha, csr_src, loop_csr,
                                                                                        rowptr, num_rows, heads, a_edge);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

extern "C" int gmlm_gat_loop_fill_bwd(const float* g, const int32_t* in2csr, const int32_t* in_dst,
                                      const int32_t* loop_csr, const int32_t* rowptr, int64_t num_edges, int heads,
                                      float* d_alpha, void* stream) {
  GMLM_REQUIRE(num_edges >= 0 && heads >= 1, "gat_loop_fill_bwd: bad sizes");
  if (num_edges == 0) return GMLM_OK;
  GMLM_REQUIRE(g && in2csr && in_dst && loop_csr && rowptr && d_alpha, "gat_loop_fill_bwd: null pointer");
  loop_fill_bwd_kernel<<<unsigned((num_edges * heads + 255) / 256), 256, 0, as_stream(stream)>>>(
      g, in2csr, in_dst, loop_csr, rowptr, num_edges, heads, d_alpha);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}
