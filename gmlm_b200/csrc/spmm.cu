// spmm.cu — the message-passing aggregation kernels (SURVEY §8a rows A5 and A14).
//
//   out[r, :] = reduce_{e in [rowptr[r], rowptr[r+1])} w[e] * x[col[e], :]
//
// Forward (RGCN mean, [PyG] RGCNConv.propagate, called main.py:272,285,298,308): rows are
// (dst,rel) segments, col = source node, reduce = mean.  Backward (autograd of the same):
// rows are source nodes of the transposed CSR, col = forward segment, w = 1/|segment|.
//
// Design (B200; roofline = E*F*b gather + 4E index + N*F*b write, HBM/L2-bound):
//   * A group of LPR lanes walks a contiguous run of CSR rows; each lane owns CH 16-byte packs
//     of the feature row, so one gathered row is LPR coalesced 128-bit loads.  Groups smaller
//     than a warp (LPR = 8/16) serve narrow feature rows without idle lanes.
//   * Work is balanced by COST, not by row count: the group plan (gmlm_group_plan) cuts the row
//     sequence where  r + rowptr[r]  crosses multiples of a quantum, so every group moves about
//     the same number of row-sized units (one per gathered edge, one per written row) whatever
//     the degree distribution — on the power-law graphs 79 % of the (dst,rel) rows are empty
//     and two thirds of the edges sit in rows longer than 256.
//   * rows kernel ("flat walk"): the group streams the *concatenated* edge list of up to LPR
//     rows.  Indices are fetched LPR at a time with one coalesced streaming load and broadcast
//     by shuffle, U feature-row loads are issued back-to-back before any is consumed
//     (memory-level parallelism independent of row length), and the fp32 accumulator is
//     flushed whenever the edge cursor crosses a row end (a segmented reduction in CSR order).
//     Empty rows are written as zeros without touching the accumulator.
//   * chunk kernel (hub path): rows longer than `hub_thresh` are cut into fixed chunks of
//     hub_thresh edges, one group per chunk, fp32 partials, then an in-order final sum.
//   * Determinism: fp32 accumulation strictly in CSR order (stable-sorted = original edge
//     order), fixed chunking, no atomics: bit-identical run to run.
#include <cuda.h>

#include <algorithm>

#include "common.cuh"

namespace gmlm {

int row_gather_map(void* out_map, const void* base, int64_t rows, int64_t cols, int64_t ld, int dtype);  // gemm_tcgen05.cu
int tuning_spmm_variant();
int tuning_spmm_unroll();
int tuning_spmm_overlap();

namespace {

struct RowsParams {
  const void* x;
  int64_t ldx;
  int64_t feat;
  const int32_t* rowptr;   // [num_rows+1]
  const int32_t* col;
  const float* w;          // [nnz, w_stride]; head h (= grid.y slab) reads column h when w_stride > 1
  int64_t w_stride;
  int64_t slab_stride;     // features between consecutive slabs (0 = LPR*VEC*CH)
  int64_t slab_width;      // valid features inside a slab (0 = slab_stride)
  int64_t num_rows;
  const int32_t* grp_row;  // [n_groups+1] cost-balanced row cuts, or nullptr = uniform LPR rows
  int64_t n_groups;
  int mean;                // 1: divide by row length
  int single;              // 1: never merge rows into a flat run (debug / A-B variant 0)
  int32_t hub_thresh;      // rows longer than this are left to the chunk kernel
  void* out;               // T [num_rows, feat]
  int64_t ldo;
};

struct ChunkParams {
  const void* x;
  int64_t ldx;
  int64_t feat;
  const int32_t* chunk_beg;
  const int32_t* chunk_end;
  const int32_t* col;
  const float* w;
  int64_t w_stride;
  int64_t slab_stride;
  int64_t slab_width;
  int64_t n_chunks;
  float* out;              // float [n_chunks, feat]
};

// address of gathered row c: base + c * row_bytes with a 32x32->64 multiply-add (one IMAD.WIDE.U32).
// The naive `xf + int64_t(c) * ldx` costs nine integer instructions per edge (sign extension + a
// full 64x64 multiply), a quarter of the per-edge instruction count of these issue-bound kernels.
template <typename T>
__device__ __forceinline__ const T* row_ptr(const T* base, int c, uint32_t row_bytes) {
  return reinterpret_cast<const T*>(reinterpret_cast<const char*>(base) + uint64_t(uint32_t(c)) * row_bytes);
}

template <typename T, int VEC, int CH>
__device__ __forceinline__ void add_pack(const Pack<T, VEC> (&v)[CH], const bool (&fvalid)[CH], float wgt,
                                         bool weighted, float (&acc)[CH][VEC]) {
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    if (fvalid[ch]) {
      float f[VEC];
      v[ch].unpack(f);
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[ch][k] = weighted ? fmaf(wgt, f[k], acc[ch][k]) : acc[ch][k] + f[k];
    }
  }
}

// ------------------------------------------------------------------------------ rows kernel
template <typename T, int VEC, int CH, int LPR, int U, int MINB, bool WEIGHTED>
__global__ void __launch_bounds__(256, MINB) rows_kernel(const RowsParams p) {
  constexpr int GROUPS = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int gl = lane % LPR;
  const int g = lane / LPR;
  const unsigned gmask = (LPR == 32) ? 0xffffffffu : (((1u << LPR) - 1u) << (g * LPR));
  const int64_t group_id = (int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * GROUPS + g;
  if (group_id >= p.n_groups) return;  // the whole group leaves together

  int64_t r_lo, r_hi;
  if (p.grp_row != nullptr) {
    r_lo = __ldg(p.grp_row + group_id);
    r_hi = __ldg(p.grp_row + group_id + 1);
  } else {
    r_lo = group_id * LPR;
    r_hi = min(r_lo + LPR, p.num_rows);
  }

  const int64_t slab_stride = p.slab_stride ? p.slab_stride : int64_t(LPR) * VEC * CH;
  const int64_t slab_width = p.slab_width ? p.slab_width : slab_stride;
  const int64_t f0 = int64_t(blockIdx.y) * slab_stride + gl * VEC;
  bool fvalid[CH];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
    fvalid[ch] = (gl * VEC + ch * LPR * VEC < slab_width) && (f0 + ch * LPR * VEC < p.feat);
  const T* __restrict__ xf = static_cast<const T*>(p.x) + f0;
  const uint32_t row_bytes = uint32_t(p.ldx) * uint32_t(sizeof(T));
  const float* __restrict__ wp = WEIGHTED ? p.w + (p.w_stride > 1 ? int64_t(blockIdx.y) : 0) : nullptr;
  const int64_t wst = p.w_stride;

  float acc[CH][VEC];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[ch][k] = 0.f;

  for (int64_t r0 = r_lo; r0 < r_hi; r0 += LPR) {
    const int nr = int(min(int64_t(LPR), r_hi - r0));
    // lane gl holds the extent of row r0+gl (an empty extent beyond nr)
    const int64_t rr = r0 + min(gl, nr - 1);
    int my_beg = __ldg(p.rowptr + rr);
    const int my_end = __ldg(p.rowptr + rr + 1);
    if (gl >= nr) my_beg = my_end;
    const unsigned hub_bits = __ballot_sync(gmask, (my_end - my_beg) > p.hub_thresh) >> (g * LPR);
    T* __restrict__ outf = static_cast<T*>(p.out) + r0 * p.ldo + f0;

    int i = 0;
    while (i < nr) {
      if ((hub_bits >> i) & 1u) { ++i; continue; }  // written by the hub path
      // maximal run [i, i+run) of non-hub rows -> one flat walk over their concatenated edges
      const unsigned rest = hub_bits >> i;
      int run = rest ? (__ffs(rest) - 1) : (nr - i);
      run = min(run, nr - i);
      if (p.single) run = 1;
      const int last = i + run;
      const int e0 = __shfl_sync(gmask, my_beg, i, LPR);
      const int e1 = __shfl_sync(gmask, my_end, last - 1, LPR);
      int cur = i;
      int cur_beg = e0;
      int cur_end = __shfl_sync(gmask, my_end, i, LPR);
      for (int base = e0; base < e1; base += LPR) {
        const int idx = base + gl;
        const int my_col = idx < e1 ? ld_stream(p.col + idx) : 0;
        float my_w = 0.f;
        if (WEIGHTED) my_w = idx < e1 ? ld_stream(wp + int64_t(idx) * wst) : 0.f;
        const int nb = min(LPR, e1 - base);
        for (int j0 = 0; j0 < nb; j0 += U) {
          Pack<T, VEC> v[U][CH];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int c = __shfl_sync(gmask, my_col, j0 + u, LPR);
            if (j0 + u < nb) {
              const T* rowp = row_ptr(xf, c, row_bytes);
#pragma unroll
              for (int ch = 0; ch < CH; ++ch)
                if (fvalid[ch]) v[u][ch].load(rowp + ch * LPR * VEC);
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            float wgt = 1.f;
            if (WEIGHTED) wgt = __shfl_sync(gmask, my_w, j0 + u, LPR);
            if (j0 + u < nb) {
              const int ee = base + j0 + u;
              while (ee >= cur_end) {  // crossed one (or several empty) row ends: flush in order
                T* dst = outf + int64_t(cur) * p.ldo;
                if (cur_end == cur_beg) {
#pragma unroll
                  for (int ch = 0; ch < CH; ++ch)
                    if (fvalid[ch]) { Pack<T, VEC> z; z.zero(); z.store(dst + ch * LPR * VEC); }
                } else {
                  const float scale = (p.mean && cur_end - cur_beg > 1) ? 1.0f / float(cur_end - cur_beg) : 1.0f;
#pragma unroll
                  for (int ch = 0; ch < CH; ++ch) {
                    if (fvalid[ch]) {
#pragma unroll
                      for (int k = 0; k < VEC; ++k) acc[ch][k] *= scale;
                      Pack<T, VEC> o;
                      o.pack(acc[ch]);
                      o.store(dst + ch * LPR * VEC);
                    }
#pragma unroll
                    for (int k = 0; k < VEC; ++k) acc[ch][k] = 0.f;
                  }
                }
                cur_beg = cur_end;
                ++cur;
                cur_end = __shfl_sync(gmask, my_end, cur, LPR);
              }
              add_pack<T, VEC, CH>(v[u], fvalid, wgt, WEIGHTED, acc);
            }
          }
        }
      }
      while (cur < last) {  // last row with edges, then trailing empty rows
        T* dst = outf + int64_t(cur) * p.ldo;
        if (cur_end == cur_beg) {
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
            if (fvalid[ch]) { Pack<T, VEC> z; z.zero(); z.store(dst + ch * LPR * VEC); }
        } else {
          const float scale = (p.mean && cur_end - cur_beg > 1) ? 1.0f / float(cur_end - cur_beg) : 1.0f;
#pragma unroll
          for (int ch = 0; ch < CH; ++ch) {
            if (fvalid[ch]) {
#pragma unroll
              for (int k = 0; k < VEC; ++k) acc[ch][k] *= scale;
              Pack<T, VEC> o;
              o.pack(acc[ch]);
              o.store(dst + ch * LPR * VEC);
            }
#pragma unroll
            for (int k = 0; k < VEC; ++k) acc[ch][k] = 0.f;
          }
        }
        cur_beg = cur_end;
        ++cur;
        if (cur < last) cur_end = __shfl_sync(gmask, my_end, cur, LPR);
      }
      i = last;
    }
  }
}

// ------------------------------------------------------------------------------ rows kernel, narrow rows
// Rows of at most 16 packs (F <= 64 / 128 bf16): 8- or 16-lane groups, two or four groups per warp.  The general
// kernel above walks its rows in batches of LPR: with 8-lane groups and 79 % empty (dst,rel) rows one batch is
// eight rows, two of them with edges, and the per-batch bookkeeping (row extents, ballots, run detection, one
// flush per row) is paid per ~12 units of work; the groups of a warp also leave their inner loops at different
// trip counts.  ncu (C4, F = 64): 727 M warp instructions for 21 M units, 13.4 of 32 lanes active per
// instruction, DRAM 13 % busy (profiles/r2b_narrow_rows.md).  Four row loads per batch at 4 CTAs per SM (64
// registers) beat eight at 3 (bwd F = 64: 1.21 vs 1.77 ms) and two at 5 (1.29 ms).  Here a group
//   1. zero-fills ALL its rows with one coalesced 16-byte store per lane and row (warp-uniform loop),
//   2. walks its edges [rowptr[r_lo], rowptr[r_hi]) in batches of U with the batch loop uniform over the warp,
//      column indices / weights read with group-uniform (broadcast) loads one batch ahead, U row loads in flight,
//   3. on a row end scales / packs / stores the accumulator over the zeros and finds the next NON-EMPTY row with one
//      cooperative look-ahead (LPR row ends per load + ballot): empty rows cost nothing in the edge walk.
// Same per-row summation order as the general kernel (CSR order, fp32): bit-identical results.
template <typename T, int VEC, int LPR, int U, int MINB, bool WEIGHTED>
__global__ void __launch_bounds__(256, MINB) rows_narrow_kernel(const RowsParams p) {
  constexpr int GROUPS = 32 / LPR;
  constexpr unsigned kLprMask = LPR == 32 ? 0xffffffffu : ((1u << (LPR & 31)) - 1u);
  const int lane = threadIdx.x & 31;
  const int gl = lane % LPR;
  const int g = lane / LPR;
  const unsigned gmask = kLprMask << (g * LPR);
  // (Re-cutting the rows of a warp's groups at equal EDGE counts -- the plan balances rows + edges -- measured 8 %
  // slower: the groups of a warp are balanced well enough, the binary searches cost more than they save.)
  const int64_t group_id = (int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * GROUPS + g;
  int64_t r_lo = 0, r_hi = 0;                       // a group past the plan keeps running with no rows (warp-wide votes)
  if (group_id < p.n_groups) {
    if (p.grp_row != nullptr) {
      r_lo = __ldg(p.grp_row + group_id);
      r_hi = __ldg(p.grp_row + group_id + 1);
    } else {
      r_lo = group_id * LPR;
      r_hi = min(r_lo + LPR, p.num_rows);
    }
  }
  const bool fvalid = gl * VEC < p.feat;
  const T* __restrict__ xf = static_cast<const T*>(p.x) + gl * VEC;
  T* __restrict__ outf = static_cast<T*>(p.out) + gl * VEC;
  const uint32_t row_bytes = uint32_t(p.ldx) * uint32_t(sizeof(T));

  // ---- 1. zeros
  const int n_rows = int(r_hi - r_lo);
  int t1 = n_rows;
#pragma unroll
  for (int d = LPR; d < 32; d <<= 1) t1 = max(t1, __shfl_xor_sync(0xffffffffu, t1, d));
  for (int i = 0; i < t1; ++i) {
    if (i < n_rows && fvalid) {
      Pack<T, VEC> z;
      z.zero();
      z.store(outf + (r_lo + i) * p.ldo);
    }
  }

  // ---- 2. edges
  int e = 0, e_end = 0;
  if (n_rows > 0) {
    e = __ldg(p.rowptr + r_lo);
    e_end = __ldg(p.rowptr + r_hi);
  }
  int64_t cur = r_lo - 1;                            // current row; its extent [cur_beg, cur_end)
  int cur_beg = e, cur_end = e;
  bool hub = false;
  float acc[VEC];
#pragma unroll
  for (int k = 0; k < VEC; ++k) acc[k] = 0.f;

  // edge `at` starts the next non-empty row after `cur` (every row in between is empty): find it with a cooperative
  // look-ahead (LPR row ends per load + ballot).  (A register window of row ends with the next window prefetched
  // measured no faster: the row-end load is not what the walk waits for.)
  auto advance = [&](int at) {
    if (at >= e_end) {
      cur = r_hi;
      cur_beg = cur_end = e_end;
      hub = false;
      return;
    }
    int64_t base = cur + 1;
    while (true) {
      const int64_t r = base + gl;
      const int v = r < r_hi ? __ldg(p.rowptr + r + 1) : 0x7fffffff;
      const unsigned bits = (__ballot_sync(gmask, v > at) >> (g * LPR)) & kLprMask;
      if (bits) {
        const int j = __ffs(bits) - 1;
        cur = base + j;
        cur_end = __shfl_sync(gmask, v, j, LPR);
        break;
      }
      base += LPR;
    }
    cur_beg = at;
    hub = (cur_end - cur_beg) > p.hub_thresh;        // hub rows belong to the chunk path: walked over, not gathered
  };
  auto flush = [&]() {
    if (!hub && fvalid) {
      const float scale = (p.mean && cur_end - cur_beg > 1) ? 1.0f / float(cur_end - cur_beg) : 1.0f;
#pragma unroll
      for (int k = 0; k < VEC; ++k) acc[k] *= scale;
      Pack<T, VEC> o;
      o.pack(acc);
      o.store(outf + cur * p.ldo);
    }
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
  };

  advance(e);
  // column indices / weights: group-uniform (broadcast) loads, one batch ahead.  (One coalesced load per batch and
  // group + shuffle broadcast -- the general kernel's scheme -- measured 30 % slower here: the shuffles sit in the
  // dependency chain of every row load.)
  int c_next[U];
  float w_next[U];
  int pre_at = -1;                                   // edge the prefetched indices start at
  while (__any_sync(0xffffffffu, e < e_end)) {
    while (hub && e < e_end) {                       // skip a hub row's edges
      e = cur_end;
      advance(e);
    }
    if (pre_at != e) {                               // first batch, or the cursor jumped over a hub row
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int ee = e + u;
        c_next[u] = ee < e_end ? ld_stream(p.col + ee) : 0;
        if (WEIGHTED) w_next[u] = ee < e_end ? ld_stream(p.w + ee) : 0.f;
      }
    }
    Pack<T, VEC> v[U];
    float wv[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      wv[u] = WEIGHTED ? w_next[u] : 1.f;
      if (e + u < e_end && fvalid) v[u].load(row_ptr(xf, c_next[u], row_bytes));
    }
    pre_at = e + U;                                  // the next batch's indices, under the row loads
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int ee = pre_at + u;
      c_next[u] = ee < e_end ? ld_stream(p.col + ee) : 0;
      if (WEIGHTED) w_next[u] = ee < e_end ? ld_stream(p.w + ee) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int ee = e + u;
      if (ee < e_end) {
        if (ee >= cur_end) {                         // the previous row is complete
          flush();
          advance(ee);
        }
        if (!hub && fvalid) {
          float f[VEC];
          v[u].unpack(f);
#pragma unroll
          for (int k = 0; k < VEC; ++k) acc[k] = WEIGHTED ? fmaf(wv[u], f[k], acc[k]) : acc[k] + f[k];
        }
      }
    }
    if (e < e_end) e += U;
  }
  if (cur < r_hi && cur_end > cur_beg) flush();      // the last row with edges
}

// ------------------------------------------------------------------------------ chunk kernel
// one group per hub chunk: out[c, :] = sum_{e in chunk c} w[e] * x[col[e], :]  (fp32 partial)
template <typename T, int VEC, int CH, int LPR, int U, int MINB, bool WEIGHTED>
__global__ void __launch_bounds__(256, MINB) chunk_kernel(const ChunkParams p) {
  constexpr int GROUPS = 32 / LPR;
  const int lane = threadIdx.x & 31;
  const int gl = lane % LPR;
  const int g = lane / LPR;
  const unsigned gmask = (LPR == 32) ? 0xffffffffu : (((1u << LPR) - 1u) << (g * LPR));
  const int64_t c_id = (int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5)) * GROUPS + g;
  if (c_id >= p.n_chunks) return;
  const int64_t slab_stride = p.slab_stride ? p.slab_stride : int64_t(LPR) * VEC * CH;
  const int64_t slab_width = p.slab_width ? p.slab_width : slab_stride;
  const int64_t f0 = int64_t(blockIdx.y) * slab_stride + gl * VEC;
  bool fvalid[CH];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
    fvalid[ch] = (gl * VEC + ch * LPR * VEC < slab_width) && (f0 + ch * LPR * VEC < p.feat);
  const T* __restrict__ xf = static_cast<const T*>(p.x) + f0;
  const uint32_t row_bytes = uint32_t(p.ldx) * uint32_t(sizeof(T));
  const float* __restrict__ wp = WEIGHTED ? p.w + (p.w_stride > 1 ? int64_t(blockIdx.y) : 0) : nullptr;
  const int64_t wst = p.w_stride;
  const int beg = __ldg(p.chunk_beg + c_id);
  const int end = __ldg(p.chunk_end + c_id);

  float acc[CH][VEC];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[ch][k] = 0.f;

  int base = beg;
  // full index batches: no per-edge predicates
  for (; base + LPR <= end; base += LPR) {
    const int my_col = ld_stream(p.col + base + gl);
    float my_w = 0.f;
    if (WEIGHTED) my_w = ld_stream(wp + int64_t(base + gl) * wst);
#pragma unroll
    for (int j0 = 0; j0 < LPR; j0 += U) {
      Pack<T, VEC> v[U][CH];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = __shfl_sync(gmask, my_col, j0 + u, LPR);
        const T* rowp = row_ptr(xf, c, row_bytes);
#pragma unroll
        for (int ch = 0; ch < CH; ++ch)
          if (fvalid[ch]) v[u][ch].load(rowp + ch * LPR * VEC);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float wgt = 1.f;
        if (WEIGHTED) wgt = __shfl_sync(gmask, my_w, j0 + u, LPR);
        add_pack<T, VEC, CH>(v[u], fvalid, wgt, WEIGHTED, acc);
      }
    }
  }
  if (base < end) {  // ragged tail
    const int idx = base + gl;
    const int my_col = idx < end ? ld_stream(p.col + idx) : 0;
    float my_w = 0.f;
    if (WEIGHTED) my_w = idx < end ? ld_stream(wp + int64_t(idx) * wst) : 0.f;
    const int nb = end - base;
    for (int j0 = 0; j0 < nb; j0 += U) {
      Pack<T, VEC> v[U][CH];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const int c = __shfl_sync(gmask, my_col, j0 + u, LPR);
        if (j0 + u < nb) {
          const T* rowp = row_ptr(xf, c, row_bytes);
#pragma unroll
          for (int ch = 0; ch < CH; ++ch)
            if (fvalid[ch]) v[u][ch].load(rowp + ch * LPR * VEC);
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
        float wgt = 1.f;
        if (WEIGHTED) wgt = __shfl_sync(gmask, my_w, j0 + u, LPR);
        if (j0 + u < nb) add_pack<T, VEC, CH>(v[u], fvalid, wgt, WEIGHTED, acc);
      }
    }
  }
  float* __restrict__ dst = p.out + c_id * p.feat + f0;
#pragma unroll
  for (int ch = 0; ch < CH; ++ch) {
    if (fvalid[ch]) {
      if constexpr (VEC == 8) {
        reinterpret_cast<float4*>(dst + ch * LPR * VEC)[0] = make_float4(acc[ch][0], acc[ch][1], acc[ch][2], acc[ch][3]);
        reinterpret_cast<float4*>(dst + ch * LPR * VEC)[1] = make_float4(acc[ch][4], acc[ch][5], acc[ch][6], acc[ch][7]);
      } else if constexpr (VEC == 4) {
        reinterpret_cast<float4*>(dst + ch * LPR * VEC)[0] = make_float4(acc[ch][0], acc[ch][1], acc[ch][2], acc[ch][3]);
      } else {
#pragma unroll
        for (int k = 0; k < VEC; ++k) dst[ch * LPR * VEC + k] = acc[ch][k];
      }
    }
  }
}


// NOTE (round 2, measured): a cp.async (LDGSTS) variant of these kernels -- every lane owning a private
// 32-slot FIFO in shared memory so that 186 KB of gathered rows per SM are in flight instead of 64 KB -- is
// bit-exact but 3.4x SLOWER on B200 (C5: 112.7 ms/step against 33.4; profiles/r2_spmm_cp_async_fifo_ab.jsonl):
// LDGSTS.128 issues at ~24 cycles per 512-byte row per SM (~21 B/clk/SM), a third of what LDG.128 sustains.
// The kernels above are bound by the bytes one SM's load path keeps outstanding (long-scoreboard stalls, DRAM
// 53-61 % busy); the copy path that is NOT bounded that way is the bulk-copy engine, whose per-row issue cost
// (one UBLKCP per row from uniform registers, ~75 cycles) is measured in profiles/r2_row_gather_tma_vs_ldg.log.
// The FIFO kernels are in the history (commit "Experiment: cp.async ... FIFO variants").


// ================================================================== bulk-copy (TMA) hub-chunk kernel
// The chunk kernel above keeps U = 4 row loads per warp in registers; what bounds it is the bytes one SM's load
// path keeps outstanding (ncu: 15.8 warps stalled on the long scoreboard per issued instruction, DRAM 53 % busy).
// Here the rows of a chunk are staged by the bulk-copy engine instead: every warp owns a ring of SLOTS batches of
// TB rows in shared memory; lane l issues `cp.async.bulk.shared.global` for row l of a batch against the batch's
// mbarrier, the whole warp then reads its 16-byte packs back with LDS and accumulates in CSR order (bit-identical
// to the register kernel).  Bytes in flight are bounded by shared memory (NW warps x (SLOTS-1) batches x TB rows),
// not by the load queues: the path measured at 95 % of the copy peak for a plain row gather
// (profiles/r2_row_gather_tma_vs_ldg.log).  Rows must be exactly CH x 512 bytes (F = 256 bf16 / 128 fp32: CH = 1).
constexpr int kTmaRows = 16;     // rows per batch

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

// PERSISTENT: one CTA per SM, every warp streams the batches of its chunks (chunk c -> warp c mod #warps) back to
// back, the issue cursor running SLOTS-1 batches ahead of the consume cursor ACROSS chunk boundaries, so the ring
// never drains (one chunk per warp and CTA left start-up and tail bubbles with one resident CTA per SM).
template <typename T, int VEC, int CH, int NW, int SLOTS, bool WEIGHTED>
__global__ void __launch_bounds__(NW * 32, 1) chunk_tma_kernel(const __grid_constant__ CUtensorMap xmap,
                                                               const ChunkParams p) {
  extern __shared__ __align__(128) uint8_t tma_ring[];
  constexpr uint32_t ROW_BYTES = 512u * CH;
  constexpr uint32_t SLOT_BYTES = kTmaRows * ROW_BYTES;
  constexpr int D = SLOTS - 1;                     // batches in flight
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  uint8_t* ring = tma_ring + size_t(warp) * SLOTS * SLOT_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tma_ring + size_t(NW) * SLOTS * SLOT_BYTES) + warp * SLOTS;
  if (lane == 0) {
    for (int s = 0; s < SLOTS; ++s) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bars + s)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  const int64_t first = int64_t(blockIdx.x) * NW + warp, stride = int64_t(gridDim.x) * NW;

  struct Cursor {            // a position in this warp's batch stream
    int64_t c;               // chunk id
    int b, nb, beg, end;     // batch inside the chunk, #batches, edge range
  };
  auto open_chunk = [&](Cursor& k, int64_t c) {
    k.c = c;
    k.b = 0;
    if (c < p.n_chunks) {
      k.beg = __ldg(p.chunk_beg + c);
      k.end = __ldg(p.chunk_end + c);
      k.nb = (k.end - k.beg + kTmaRows - 1) / kTmaRows;
    } else {
      k.beg = k.end = k.nb = 0;
    }
  };
  auto advance = [&](Cursor& k) {
    if (++k.b >= k.nb) open_chunk(k, k.c + stride);
  };
  auto load_col = [&](const Cursor& k) -> int {
    const int idx = k.beg + k.b * kTmaRows + lane;
    return (k.c < p.n_chunks && lane < kTmaRows && idx < k.end) ? ld_stream(p.col + idx) : 0;
  };
  // `tile::gather4`: ONE bulk-tensor op fetches four arbitrary rows (2 KB): the per-op cost of the copy engine
  // (about one op per 18 cycles per SM whatever its size) capped single-row bulk copies at the LDG rate
  auto issue = [&](const Cursor& k, uint32_t g, int my_col) {
    if (k.c >= p.n_chunks) return;
    const int s = int(g % SLOTS);
    const int n = min(kTmaRows, k.end - (k.beg + k.b * kTmaRows));
    const uint32_t bar = smem_u32(bars + s);
    const int n_ops = (n + 3) >> 2;
    if (lane == 0)
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(uint32_t(n_ops) * 4u * ROW_BYTES)
                   : "memory");
    __syncwarp();
    const int q = (lane & 3) * 4;                     // op `lane` takes rows 4*lane .. 4*lane+3 of the batch
    const int r0 = __shfl_sync(0xffffffffu, my_col, q), r1 = __shfl_sync(0xffffffffu, my_col, q + 1);
    const int r2 = __shfl_sync(0xffffffffu, my_col, q + 2), r3 = __shfl_sync(0xffffffffu, my_col, q + 3);
    if (lane < n_ops) {                               // rows past the chunk end hold index 0: fetched, never read
      asm volatile(
          "cp.async.bulk.tensor.2d.shared::cluster.global.tile::gather4.mbarrier::complete_tx::bytes"
          " [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(smem_u32(ring + size_t(s) * SLOT_BYTES + size_t(lane) * 4 * ROW_BYTES)),
          "l"(reinterpret_cast<uint64_t>(&xmap)), "r"(bar), "r"(0), "r"(r0), "r"(r1), "r"(r2), "r"(r3)
          : "memory");
    }
  };

  Cursor ic, cc;                                    // issue / consume cursors
  open_chunk(ic, first);
  open_chunk(cc, first);
  uint32_t gi = 0, gc = 0;                          // batches issued / consumed so far (ring positions)
  int col_cur = load_col(ic);
  for (int d = 0; d < D; ++d) {                     // prime the ring
    Cursor nx = ic;
    advance(nx);
    const int col_nx = load_col(nx);
    issue(ic, gi, col_cur);
    if (ic.c < p.n_chunks) ++gi;
    ic = nx;
    col_cur = col_nx;
  }
  float acc[CH][VEC];
#pragma unroll
  for (int ch = 0; ch < CH; ++ch)
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[ch][k] = 0.f;

  while (cc.c < p.n_chunks) {
    const int s = int(gc % SLOTS);
    const uint32_t bar = smem_u32(bars + s);
    const uint32_t parity = (gc / SLOTS) & 1u;
    float my_w = 0.f;
    if (WEIGHTED) {
      const int idx = cc.beg + cc.b * kTmaRows + lane;
      my_w = (lane < kTmaRows && idx < cc.end) ? ld_stream(p.w + idx) : 0.f;
    }
    uint32_t spins = 0;
    while (true) {
      uint32_t ok;
      asm volatile(
          "{\n\t.reg .pred q;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 q, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, q;\n\t}"
          : "=r"(ok)
          : "r"(bar), "r"(parity)
          : "memory");
      if (ok) break;
      if (++spins > (1u << 26)) __trap();
    }
    const int n = min(kTmaRows, cc.end - (cc.beg + cc.b * kTmaRows));
    const uint32_t base = smem_u32(ring + size_t(s) * SLOT_BYTES) + uint32_t(lane) * 16u;
#pragma unroll 4
    for (int r = 0; r < n; ++r) {
      float wgt = 1.f;
      if (WEIGHTED) wgt = __shfl_sync(0xffffffffu, my_w, r);
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        uint32_t a0, a1, a2, a3;
        asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(a3)
                     : "r"(base + uint32_t(r) * ROW_BYTES + uint32_t(ch) * 512u)
                     : "memory");
        Pack<T, VEC> v;
        uint4 u = make_uint4(a0, a1, a2, a3);
        v.v = *reinterpret_cast<decltype(v.v)*>(&u);
        float f[VEC];
        v.unpack(f);
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[ch][k] = WEIGHTED ? fmaf(wgt, f[k], acc[ch][k]) : acc[ch][k] + f[k];
      }
    }
    __syncwarp();                                  // every lane has read the slot: it may be refilled
    ++gc;
    {                                              // refill: the batch D ahead in the stream
      Cursor nx = ic;
      advance(nx);
      const int col_nx = load_col(nx);
      issue(ic, gi, col_cur);
      if (ic.c < p.n_chunks) ++gi;
      ic = nx;
      col_cur = col_nx;
    }
    if (cc.b + 1 >= cc.nb) {                       // chunk complete: its fp32 partial sum
      float* __restrict__ dst = p.out + cc.c * p.feat + lane * VEC;
#pragma unroll
      for (int ch = 0; ch < CH; ++ch) {
        if constexpr (VEC == 8) {
          reinterpret_cast<float4*>(dst + ch * 32 * VEC)[0] = make_float4(acc[ch][0], acc[ch][1], acc[ch][2], acc[ch][3]);
          reinterpret_cast<float4*>(dst + ch * 32 * VEC)[1] = make_float4(acc[ch][4], acc[ch][5], acc[ch][6], acc[ch][7]);
        } else {
          reinterpret_cast<float4*>(dst + ch * 32 * VEC)[0] = make_float4(acc[ch][0], acc[ch][1], acc[ch][2], acc[ch][3]);
        }
#pragma unroll
        for (int k = 0; k < VEC; ++k) acc[ch][k] = 0.f;
      }
    }
    advance(cc);
  }
}

// final in-order reduction of the hub partials: `tpr` threads per hub row, each thread owns the
// features f = t, t+tpr, ...; chunk partials are loaded 8 at a time (independent loads) and added
// in chunk order (fixed order => deterministic).
template <typename T>
__global__ void __launch_bounds__(256) hub_final_kernel(const float* __restrict__ ws, int64_t feat,
                                                        const int32_t* __restrict__ rowptr,
                                                        const int32_t* __restrict__ hub_row,
                                                        const int32_t* __restrict__ hub_chunk_ptr, int64_t n_hub,
                                                        int tpr, int mean, T* __restrict__ out, int64_t ldo) {
  const int rows_per_cta = blockDim.x / tpr;
  const int64_t h = int64_t(blockIdx.x) * rows_per_cta + threadIdx.x / tpr;
  const int t = threadIdx.x % tpr;
  if (h >= n_hub) return;
  const int32_t r = __ldg(hub_row + h);
  const int32_t c0 = __ldg(hub_chunk_ptr + h), c1 = __ldg(hub_chunk_ptr + h + 1);
  const int len = __ldg(rowptr + r + 1) - __ldg(rowptr + r);
  const float scale = (mean && len > 1) ? 1.0f / float(len) : 1.0f;
  for (int64_t f = t; f < feat; f += tpr) {
    float a = 0.f;
    int32_t c = c0;
    for (; c + 8 <= c1; c += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldcs(ws + int64_t(c + u) * feat + f);
#pragma unroll
      for (int u = 0; u < 8; ++u) a += v[u];
    }
    for (; c < c1; ++c) a += __ldcs(ws + int64_t(c) * feat + f);
    out[int64_t(r) * ldo + f] = from_float<T>(a * scale);
  }
}

// cost-balanced cuts: grp_row[g] = first row r with r + rowptr[r] >= g * quantum
__global__ void group_plan_kernel(const int32_t* __restrict__ rowptr, int64_t num_rows, int64_t quantum,
                                  int64_t n_groups, int32_t* __restrict__ grp_row) {
  const int64_t g = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (g > n_groups) return;
  if (g == n_groups) { grp_row[g] = int32_t(num_rows); return; }
  const int64_t target = g * quantum;
  int64_t lo = 0, hi = num_rows;  // answer in [0, num_rows]
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (mid + int64_t(rowptr[mid]) >= target) hi = mid; else lo = mid + 1;
  }
  grp_row[g] = int32_t(lo);
}

// ------------------------------------------------------------------------------ dispatch
struct Job {
  RowsParams rows;
  ChunkParams chunks;
  bool weighted;
  bool do_rows;
  bool do_chunks;
  int unroll;  // 0 = default
  cudaStream_t chunk_stream = nullptr;   // where the chunk kernel goes (the caller's stream unless the hub path is forked)
  bool forked = false;
};

// fork / join resources of the overlapped hub path: per host thread and device (events are reused across calls)
struct SideStream {
  cudaStream_t stream = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
};
SideStream* side_stream() {
  static thread_local SideStream s[kMaxDevices];
  SideStream& r = s[current_device()];
  if (!r.stream) {
    if (cudaStreamCreateWithFlags(&r.stream, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&r.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&r.join, cudaEventDisableTiming) != cudaSuccess)
      return nullptr;
  }
  return &r;
}

template <typename T, int VEC, int CH, int NW, int SLOTS>
int launch_chunk_tma(Job& job, cudaStream_t st) {
  ChunkParams& q = job.chunks;
  CUtensorMap xmap;
  // the C ABI does not carry the number of source rows: the map is bounded by INT32_MAX rows (col is int32), which
  // only widens the coordinate range the engine accepts -- rows that no col entry names are never touched
  if (int rc = row_gather_map(&xmap, q.x, 0x7fffffff, q.feat, q.ldx, sizeof(T) == 4 ? GMLM_F32 : GMLM_BF16)) return rc;
  constexpr size_t smem = size_t(NW) * SLOTS * kTmaRows * 512 * CH + size_t(NW) * SLOTS * 8;
  static_assert(smem <= 227 * 1024, "ring exceeds the shared memory of one SM");
  static bool configured[kMaxDevices][2] = {};
  const int dev = current_device();
  if (q.n_chunks == 0) return GMLM_OK;
  const int64_t gx = std::min<int64_t>((q.n_chunks + NW - 1) / NW, num_sms());     // persistent: one CTA per SM
  if (job.weighted) {
    auto k = chunk_tma_kernel<T, VEC, CH, NW, SLOTS, true>;
    if (!configured[dev][0]) {
      GMLM_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
      configured[dev][0] = true;
    }
    k<<<unsigned(gx), NW * 32, smem, st>>>(xmap, q);
  } else {
    auto k = chunk_tma_kernel<T, VEC, CH, NW, SLOTS, false>;
    if (!configured[dev][1]) {
      GMLM_CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
      configured[dev][1] = true;
    }
    k<<<unsigned(gx), NW * 32, smem, st>>>(xmap, q);
  }
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

template <typename T, int VEC, int CH, int LPR, int U, int MINB>
int launch_geo(Job& job, cudaStream_t st) {
  constexpr int GROUPS = 32 / LPR;
  const int64_t groups_per_cta = int64_t(256 / 32) * GROUPS;
  const int64_t slab = int64_t(LPR) * VEC * CH;
  if (job.do_rows) {
    RowsParams& p = job.rows;
    if (p.grp_row == nullptr) p.n_groups = (p.num_rows + LPR - 1) / LPR;
    const int64_t gx = (p.n_groups + groups_per_cta - 1) / groups_per_cta;
    const int64_t sstride = p.slab_stride ? p.slab_stride : slab;
    const int64_t gy = (p.feat + sstride - 1) / sstride;
    GMLM_REQUIRE(gx <= 0x7fffffffLL && gy <= 65535, "spmm: grid too large");
    if (gx > 0) {
      dim3 grid((unsigned)gx, (unsigned)gy);
      if (job.weighted) rows_kernel<T, VEC, CH, LPR, U, MINB, true><<<grid, 256, 0, st>>>(p);
      else rows_kernel<T, VEC, CH, LPR, U, MINB, false><<<grid, 256, 0, st>>>(p);
      GMLM_LAUNCH_CHECK();
    }
  }
  if (job.do_chunks) {
    ChunkParams& q = job.chunks;
    const int64_t gx = (q.n_chunks + groups_per_cta - 1) / groups_per_cta;
    const int64_t sstride = q.slab_stride ? q.slab_stride : slab;
    const int64_t gy = (q.feat + sstride - 1) / sstride;
    GMLM_REQUIRE(gx <= 0x7fffffffLL && gy <= 65535, "spmm: grid too large");
    if (gx > 0) {
      dim3 grid((unsigned)gx, (unsigned)gy);
      cudaStream_t cs = job.chunk_stream ? job.chunk_stream : st;
      if (job.weighted) chunk_kernel<T, VEC, CH, LPR, U, MINB, true><<<grid, 256, 0, cs>>>(q);
      else chunk_kernel<T, VEC, CH, LPR, U, MINB, false><<<grid, 256, 0, cs>>>(q);
      GMLM_LAUNCH_CHECK();
    }
  }
  return GMLM_OK;
}

// narrow rows: rows_narrow_kernel for the rows, the general chunk kernel for the hub chunks
template <typename T, int VEC, int LPR, int U, int MINB>
int launch_narrow(Job& job, cudaStream_t st) {
  constexpr int GROUPS = 32 / LPR;
  const int64_t groups_per_cta = int64_t(256 / 32) * GROUPS;
  RowsParams& p = job.rows;
  if (p.grp_row == nullptr) p.n_groups = (p.num_rows + LPR - 1) / LPR;
  const int64_t gx = (p.n_groups + groups_per_cta - 1) / groups_per_cta;
  GMLM_REQUIRE(gx <= 0x7fffffffLL, "spmm: grid too large");
  if (gx > 0) {
    if (job.weighted) rows_narrow_kernel<T, VEC, LPR, U, MINB, true><<<unsigned(gx), 256, 0, st>>>(p);
    else rows_narrow_kernel<T, VEC, LPR, U, MINB, false><<<unsigned(gx), 256, 0, st>>>(p);
    GMLM_LAUNCH_CHECK();
  }
  if (!job.do_chunks) return GMLM_OK;
  Job chunks_only = job;
  chunks_only.do_rows = false;
  return launch_geo<T, VEC, 1, LPR, U, MINB>(chunks_only, st);     // same stream (see gmlm_spmm_csr: never forked)
}

template <typename T, int VEC>
int launch_vec(Job& job, cudaStream_t st) {
  const int64_t width = job.rows.slab_width ? job.rows.slab_width : job.rows.feat;
  const int64_t nvec = (width + VEC - 1) / VEC;
  if (job.rows.slab_width) GMLM_REQUIRE(nvec <= 256, "spmm: per-head width above 256 packs is not supported");
  // one head slab per warp up to 256 packs: the GAT input gradient of heads wider than 128 packs (520 fp32 features on
  // 16-byte packs, 130 on scalar packs); every other width keeps the instantiations below
  if (job.rows.slab_width && nvec > 128) return launch_geo<T, VEC, 8, 32, 1, 1>(job, st);
  // narrow rows without head slabs: the warp-uniform edge walk (spmm_variant 2 keeps the general kernel for A/B)
  const bool narrow = job.do_rows && job.rows.slab_stride == 0 && job.rows.w_stride <= 1 && !job.rows.single &&
                      tuning_spmm_variant() != 2;
  if (nvec <= 8) return narrow ? launch_narrow<T, VEC, 8, 4, 4>(job, st) : launch_geo<T, VEC, 1, 8, 8, 3>(job, st);
  if (nvec <= 16) return narrow ? launch_narrow<T, VEC, 16, 4, 4>(job, st) : launch_geo<T, VEC, 1, 16, 8, 3>(job, st);
  if (nvec <= 32) {
    if constexpr (VEC * sizeof(T) == 16) {
      // rows of exactly 512 bytes (F = 256 bf16 / 128 fp32), no head slabs: the hub chunks can take the
      // bulk-copy kernel (spmm_variant 3 / 4: 8 warps x 3 slots / 12 warps x 2 slots per SM)
      const int var = tuning_spmm_variant();
      if (var >= 3 && job.do_chunks && nvec == 32 && job.chunks.slab_stride == 0 && job.chunks.w_stride <= 1 &&
          job.chunks.ldx * int64_t(sizeof(T)) % 16 == 0) {
        Job rows_only = job;
        rows_only.do_chunks = false;
        int rc = launch_geo<T, VEC, 1, 32, 4, 4>(rows_only, st);
        if (rc) return rc;
        return var == 3 ? launch_chunk_tma<T, VEC, 1, 8, 3>(job, st) : launch_chunk_tma<T, VEC, 1, 12, 2>(job, st);
      }
    }
    // (the edge-walk kernel instantiated for 32-lane rows measured slower than the general kernel: C4 F = 256 pair
    // 3.07 + 2.74 ms against 2.99 + 2.50 ms, C5 forward 32.9 against 17.7 ms -- with one group per warp there is no
    // divergence to remove, and zero-filling 40 M rows up front is a second pass over the output)
    // measured on B200 (C4, bf16 F=256): U=4 at 4 CTAs/SM beats U=8 at 3 CTAs/SM by 12 %
    if (job.unroll == 8) return launch_geo<T, VEC, 1, 32, 8, 3>(job, st);
    return launch_geo<T, VEC, 1, 32, 4, 4>(job, st);
  }
  if (nvec <= 64) return launch_geo<T, VEC, 2, 32, 4, 3>(job, st);
  if (nvec <= 96) return launch_geo<T, VEC, 3, 32, 2, 3>(job, st);
  return launch_geo<T, VEC, 4, 32, 2, 2>(job, st);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

}  // namespace
}  // namespace gmlm

using namespace gmlm;

extern "C" int64_t gmlm_group_plan_size(int64_t num_rows, int64_t nnz, int64_t quantum) {
  if (quantum < 1) quantum = 1;
  return (num_rows + nnz + quantum - 1) / quantum;
}

extern "C" int gmlm_group_plan(const int32_t* rowptr, int64_t num_rows, int64_t nnz, int64_t quantum,
                               int32_t* grp_row, void* stream) {
  GMLM_REQUIRE(quantum >= 1 && num_rows >= 0 && nnz >= 0, "group_plan: bad sizes");
  GMLM_REQUIRE(rowptr && grp_row, "group_plan: null pointer");
  const int64_t n_groups = gmlm_group_plan_size(num_rows, nnz, quantum);
  const int64_t threads = n_groups + 1;
  group_plan_kernel<<<unsigned((threads + 255) / 256), 256, 0, as_stream(stream)>>>(rowptr, num_rows, quantum,
                                                                                    n_groups, grp_row);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

extern "C" int gmlm_spmm_csr(const void* x, int dtype, int64_t feat, int64_t ldx, const int32_t* rowptr,
                             const int32_t* col, const float* w, int32_t w_heads, int64_t num_rows, int mode,
                             const int32_t* grp_row, int64_t n_groups, int32_t hub_thresh, int64_t n_hub,
                             int64_t n_chunks, const int32_t* hub_row, const int32_t* hub_chunk_ptr,
                             const int32_t* chunk_beg, const int32_t* chunk_end, float* hub_ws, void* out,
                             int64_t ldo, void* stream) {
  GMLM_REQUIRE(dtype == GMLM_F32 || dtype == GMLM_BF16, "spmm: dtype must be GMLM_F32 or GMLM_BF16");
  GMLM_REQUIRE(mode == GMLM_AGG_SUM || mode == GMLM_AGG_MEAN || mode == GMLM_AGG_WEIGHTED, "spmm: bad mode");
  GMLM_REQUIRE(feat >= 0 && num_rows >= 0 && ldx >= feat && ldo >= feat, "spmm: bad sizes");
  GMLM_REQUIRE(ldx * (dtype == GMLM_F32 ? 4 : 2) < (int64_t(1) << 32), "spmm: a gathered row must be shorter than 4 GiB");
  GMLM_REQUIRE(mode != GMLM_AGG_WEIGHTED || w != nullptr, "spmm: weighted mode needs w");
  GMLM_REQUIRE(w_heads >= 1 && (w_heads == 1 || (mode == GMLM_AGG_WEIGHTED && feat % w_heads == 0)),
               "spmm: w_heads must divide feat (and needs weighted mode)");
  GMLM_REQUIRE(n_hub >= 0 && n_chunks >= n_hub, "spmm: bad hub plan");
  GMLM_REQUIRE(grp_row == nullptr || n_groups >= 0, "spmm: bad group plan");
  if (num_rows == 0 || feat == 0) return GMLM_OK;
  GMLM_REQUIRE(x && rowptr && out, "spmm: null pointer");
  GMLM_REQUIRE(n_hub == 0 || (hub_row && hub_chunk_ptr && chunk_beg && chunk_end && hub_ws && hub_thresh >= 1),
               "spmm: hub plan arrays missing");
  cudaStream_t st = as_stream(stream);
  const int esz = dtype == GMLM_F32 ? 4 : 2;
  const int fullvec = 16 / esz;
  const int64_t head_width = w_heads > 1 ? feat / w_heads : 0;
  const bool aligned = aligned16(x) && aligned16(out) && aligned16(hub_ws) && feat % fullvec == 0 &&
                       ldx % fullvec == 0 && ldo % fullvec == 0 && head_width % fullvec == 0;

  Job job;
  job.weighted = mode == GMLM_AGG_WEIGHTED;
  job.do_rows = true;
  job.do_chunks = n_hub > 0;
  job.unroll = tuning_spmm_unroll();
  RowsParams& p = job.rows;
  p.x = x; p.ldx = ldx; p.feat = feat;
  p.rowptr = rowptr; p.col = col; p.w = w; p.num_rows = num_rows;
  p.w_stride = w_heads; p.slab_stride = head_width; p.slab_width = head_width;
  p.grp_row = grp_row; p.n_groups = n_groups;
  p.mean = mode == GMLM_AGG_MEAN;
  p.single = tuning_spmm_variant() == 0;
  p.hub_thresh = n_hub > 0 ? hub_thresh : 0x7fffffff;
  p.out = out; p.ldo = ldo;
  ChunkParams& q = job.chunks;
  q.x = x; q.ldx = ldx; q.feat = feat;
  q.chunk_beg = chunk_beg; q.chunk_end = chunk_end; q.col = col; q.w = w;
  q.w_stride = w_heads; q.slab_stride = head_width; q.slab_width = head_width;
  q.n_chunks = n_chunks; q.out = hub_ws;

  // (Also measured and not kept: `prefetch.global.L2` of the rows the NEXT index batch gathers, issued by each lane while
  // the current batch is in flight -- bytes in flight towards L2 without registers: C5 forward 17.7 -> 18.8 ms in the
  // rows kernel alone, 32 ms with the chunk kernel prefetching too: the extra instructions and the L2 churn cost more
  // than the earlier arrival buys.)
  // Overlapped hub path (tuning "spmm_overlap", default off): the chunk + final kernels work on rows the rows kernel
  // skips, so they can be forked onto a side stream.  Measured: C5 32.45 -> 32.34 ms/step, C4 5.46 -> 5.33 -- the rows
  // kernel fills every SM, the side stream only gets its tail, and both kernels already sit at the same ~70 % of DRAM
  // peak (the LDG row-gather ceiling of profiles/r2_row_gather_tma_vs_ldg.log), so there is no idle resource to fill.
  // Not for the narrow-row kernel (it zero-fills every row first, the hub rows included).
  SideStream* side = nullptr;
  {
    const int64_t nvec_rows = (feat + fullvec - 1) / fullvec;
    const bool narrow_path = aligned ? (nvec_rows <= 16 && head_width == 0 && w_heads <= 1) : (feat <= 16 && w_heads <= 1);
    if (tuning_spmm_overlap() && n_hub > 0 && !narrow_path) side = side_stream();
  }
  if (side) {
    GMLM_CUDA_TRY(cudaEventRecord(side->fork, st));
    GMLM_CUDA_TRY(cudaStreamWaitEvent(side->stream, side->fork, 0));
    job.chunk_stream = side->stream;
    job.forked = true;
  }
  int rc;
  if (dtype == GMLM_F32) rc = aligned ? launch_vec<float, 4>(job, st) : launch_vec<float, 1>(job, st);
  else rc = aligned ? launch_vec<__nv_bfloat16, 8>(job, st) : launch_vec<__nv_bfloat16, 1>(job, st);
  if (rc) return rc;
  if (n_hub == 0) return GMLM_OK;
  cudaStream_t st_rows = st;
  if (side) st = side->stream;                       // the final kernel follows the chunk kernel

  int tpr = 256;
  if (feat <= 128) tpr = int((feat + 31) / 32) * 32;
  if (tpr == 96) tpr = 128;
  const int rows_per_cta = 256 / tpr;
  const unsigned blocks = unsigned((n_hub + rows_per_cta - 1) / rows_per_cta);
  if (dtype == GMLM_F32)
    hub_final_kernel<float><<<blocks, 256, 0, st>>>(hub_ws, feat, rowptr, hub_row, hub_chunk_ptr, n_hub, tpr, p.mean,
                                                    static_cast<float*>(out), ldo);
  else
    hub_final_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(hub_ws, feat, rowptr, hub_row, hub_chunk_ptr, n_hub, tpr,
                                                            p.mean, static_cast<__nv_bfloat16*>(out), ldo);
  GMLM_LAUNCH_CHECK();
  if (side) {                                        // join: the caller's stream continues after both branches
    GMLM_CUDA_TRY(cudaEventRecord(side->join, side->stream));
    GMLM_CUDA_TRY(cudaStreamWaitEvent(st_rows, side->join, 0));
  }
  return GMLM_OK;
}
