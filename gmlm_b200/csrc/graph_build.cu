// graph_build.cu — one-off graph preprocessing on the GPU (SURVEY §8a rows A1-A3, A14):
// degree histogram, degree-bucket edge typing, the (dst,rel)-keyed CSR, its transpose for the
// backward gather, and the hub plan that keeps power-law rows balanced and deterministic.
//
// All integer work: results are bit-exact against oracle/csr_ref.py and oracle/pyg_ref.py.
// The stable radix sort / exclusive scan / ordered selection are this library's own (primitives.cuh; round 1 used
// CUB).  This is HBM-bound byte shuffling: coalesced 64-bit index reads, int32 outputs, grid sized in multiples of
// the SM count.
#include <algorithm>

#include "common.cuh"
#include "primitives.cuh"

namespace gmlm {

char* err_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}

static int g_spmm_variant = 1;   // 0 = one row per walk, 1 = flat walk over runs of rows (default)
static int g_spmm_unroll = 0;
static int g_spmm_overlap = 0;   // 1 = the hub chunks (chunk + final kernels) run on a side stream beside the rows kernel
int tuning_spmm_overlap() { return g_spmm_overlap; }
int tuning_spmm_variant() { return g_spmm_variant; }
int tuning_spmm_unroll() { return g_spmm_unroll; }
static int g_halo_pull_ctas = 0;
int tuning_halo_pull_ctas() { return g_halo_pull_ctas; }
static int g_halo_pull_threads = 0;
int tuning_halo_pull_threads() { return g_halo_pull_threads; }

namespace {

constexpr int kThreads = 256;

inline int grid_for(int64_t n, int per_thread = 1) {
  int64_t blocks = (n + int64_t(kThreads) * per_thread - 1) / (int64_t(kThreads) * per_thread);
  int64_t cap = int64_t(num_sms()) * 32;  // grid-stride beyond this
  if (blocks < 1) blocks = 1;
  return int(blocks < cap ? blocks : cap);
}

// Index-out-of-range flag: one int PER CALL, carved from the caller's workspace (or stream-allocated), so
// concurrent builds on different streams / threads / devices cannot see each other's errors.  Kernels
// take the pointer; nullptr = do not record.
__device__ __forceinline__ void flag_error(int* flag) {
  if (flag) *flag = 1;
}

int read_flag(const int* d_flag, cudaStream_t st, int* out) {
  int h = 0;
  GMLM_CUDA_TRY(cudaMemcpyAsync(&h, d_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
  GMLM_CUDA_TRY(cudaStreamSynchronize(st));
  *out = h;
  return GMLM_OK;
}

// ------------------------------------------------------------------------ A1
__global__ void degree_kernel(const int64_t* __restrict__ index, const uint8_t* __restrict__ keep, int64_t E, int64_t N,
                              int32_t* __restrict__ deg, int* __restrict__ err) {
  for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < E; e += int64_t(gridDim.x) * blockDim.x) {
    if (keep && !keep[e]) continue;               // edge dropout (main.py:832-837) fused into the histogram
    int64_t i = index[e];
    if (i >= 0 && i < N) atomicAdd(deg + i, 1);   // integer atomics: order-independent result
    else flag_error(err);
  }
}

__global__ void i32_to_f32_kernel(const int32_t* __restrict__ in, float* __restrict__ out, int64_t n) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    out[i] = float(in[i]);
}

// ------------------------------------------------------------------------ A2
struct Bounds { int32_t b[8]; int n; };

__global__ void edge_type_kernel(const int64_t* __restrict__ src, int64_t E, const int32_t* __restrict__ deg,
                                 int64_t N, Bounds bounds, int64_t* __restrict__ out, int* __restrict__ err) {
  for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < E; e += int64_t(gridDim.x) * blockDim.x) {
    int64_t s = src[e];
    int t = 0;
    if (s >= 0 && s < N) {
      int32_t d = deg[s];
#pragma unroll
      for (int k = 0; k < 8; ++k) t += (k < bounds.n && d > bounds.b[k]) ? 1 : 0;
    } else {
      flag_error(err);
    }
    out[e] = t;
  }
}

__global__ void rel_hist_kernel(const int64_t* __restrict__ et, const uint8_t* __restrict__ keep, int64_t E, int R,
                                unsigned long long* __restrict__ counts) {
  // values outside [0, R) are simply not counted: the caller compares the total with E
  __shared__ unsigned int sh[64];
  for (int i = threadIdx.x; i < 64; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < E; e += int64_t(gridDim.x) * blockDim.x) {
    if (keep && !keep[e]) continue;
    int64_t t = et[e];
    if (t >= 0 && t < R) atomicAdd(&sh[t], 1u);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < R; i += blockDim.x)
    if (sh[i]) atomicAdd(counts + i, (unsigned long long)sh[i]);
}

// ---------------------------------------------------------------- content key of an index tensor
// out[0] = sum_i x_i * (2i+1),  out[1] = sum_i (x_i ^ (x_i >> 17)) * (i * 0x9E3779B97F4A7C15 + 1)   (mod 2^64).
// Position-weighted, so permutations change it; integer atomics, so the result does not depend on the order of
// the additions.  Used to recognise a graph whose edge tensors were re-created with the same contents (the
// reference builds a fresh edge_type tensor on every call, main.py:255) without rebuilding its CSR.
__global__ void checksum_kernel(const uint64_t* __restrict__ x, int64_t n, unsigned long long* __restrict__ out) {
  unsigned long long a = 0, b = 0;
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const unsigned long long v = x[i];
    a += v * (2ull * (unsigned long long)i + 1ull);
    b += (v ^ (v >> 17)) * ((unsigned long long)i * 0x9E3779B97F4A7C15ull + 1ull);
  }
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  if ((threadIdx.x & 31) == 0) { atomicAdd(out, a); atomicAdd(out + 1, b); }
}

// ------------------------------------------------------------------------ A3
struct SlotMap { int32_t slot[64]; };

// A dropped edge (keep[e] == 0: the reference's `augment_graph` edge dropout, main.py:832-837) gets the sentinel
// key N*S: it is not counted, sorts behind every kept edge, and rowptr[N*S] ends up as the number of kept edges.
__global__ void make_keys_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst,
                                 const int64_t* __restrict__ et, const uint8_t* __restrict__ keep, int64_t E, int64_t N,
                                 int64_t Nsrc, int R, SlotMap sm, int S,
                                 uint32_t* __restrict__ keys, int32_t* __restrict__ vals,
                                 int32_t* __restrict__ seg_of_edge, int32_t* __restrict__ counts,
                                 int* __restrict__ err) {
  for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < E; e += int64_t(gridDim.x) * blockDim.x) {
    if (keep && !keep[e]) {
      keys[e] = uint32_t(N * S);
      vals[e] = int32_t(e);
      if (seg_of_edge) seg_of_edge[e] = int32_t(N * S);
      continue;
    }
    int64_t s = src[e], d = dst[e];
    int64_t t = et ? et[e] : 0;
    bool ok = s >= 0 && s < Nsrc && d >= 0 && d < N && t >= 0 && t < R;
    int slot = ok ? sm.slot[t] : 0;
    ok = ok && slot >= 0;
    uint32_t key = 0;
    if (ok) {
      key = uint32_t(d * S + slot);
      atomicAdd(counts + key, 1);
    } else {
      flag_error(err);
    }
    keys[e] = key;
    vals[e] = int32_t(e);
    if (seg_of_edge) seg_of_edge[e] = int32_t(key);
  }
}

__global__ void gather_col_kernel(const int64_t* __restrict__ src, const int32_t* __restrict__ perm, int64_t E,
                                  int32_t* __restrict__ col) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < E; i += int64_t(gridDim.x) * blockDim.x)
    col[i] = int32_t(src[perm[i]]);
}

// ----------------------------------------------------------------------- A14
__global__ void make_keys_t_kernel(const int64_t* __restrict__ row_of_edge, const uint8_t* __restrict__ keep, int64_t E,
                                   int64_t num_rows, uint32_t* __restrict__ keys, int32_t* __restrict__ vals,
                                   int32_t* __restrict__ counts, int* __restrict__ err) {
  for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < E; e += int64_t(gridDim.x) * blockDim.x) {
    if (keep && !keep[e]) { keys[e] = uint32_t(num_rows); vals[e] = int32_t(e); continue; }   // dropped: sentinel key
    int64_t r = row_of_edge[e];
    uint32_t key = 0;
    if (r >= 0 && r < num_rows) {
      key = uint32_t(r);
      atomicAdd(counts + key, 1);
    } else {
      flag_error(err);
    }
    keys[e] = key;
    vals[e] = int32_t(e);
  }
}

__global__ void gather_payload_t_kernel(const int32_t* __restrict__ payload, const float* __restrict__ edge_w,
                                        const int32_t* __restrict__ fwd_rowptr, const int32_t* __restrict__ perm_t,
                                        const uint8_t* __restrict__ keep, int64_t E, int32_t* __restrict__ payload_t,
                                        float* __restrict__ w_t) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < E; i += int64_t(gridDim.x) * blockDim.x) {
    int32_t e = perm_t[i];
    if (keep && !keep[e]) { payload_t[i] = 0; if (w_t) w_t[i] = 0.f; continue; }   // dropped edges: the unused tail
    int32_t p = payload[e];
    payload_t[i] = p;
    if (fwd_rowptr) {
      int32_t c = fwd_rowptr[p + 1] - fwd_rowptr[p];
      w_t[i] = 1.0f / float(c);   // IEEE division: equals numpy float32(1)/float32(c)
    } else if (edge_w) {
      w_t[i] = edge_w[e];
    }
  }
}

// --------------------------------------------------- transform-first plan (dst-keyed view of the fwd CSR)
// For  out[i] = sum_s mean_{e in seg(i,s)} Z[src_e, s]  +  Z[i, S]   (Z = x @ [W_0 | .. | W_{S-1} | root], slab s of
// row j being row j*(S+1)+s of Z viewed as [N*(S+1), Fo]) the (dst,rel) CSR is re-read as a dst-keyed CSR whose
// rows are whole destination nodes: the edges of segments i*S .. i*S+S-1 in order, then one self "edge" for the
// root slab.  col = gathered Z row, w = 1/|segment| (1 for the root slab), dst = destination of every entry (the
// payload of the transposed plan).  One thread per entry; the segment of an edge is found by binary search.
__global__ void dst_plan_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col, int64_t N, int S,
                                int64_t E, int32_t* __restrict__ rowptr_d, int32_t* __restrict__ col_d,
                                float* __restrict__ w_d, int32_t* __restrict__ dst_d) {
  const int64_t total = E + N;
  const int64_t rows = N * S;
  for (int64_t t = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; t < total + N + 1;
       t += int64_t(gridDim.x) * blockDim.x) {
    if (t >= total) {                       // the N+1 row pointers
      const int64_t i = t - total;
      rowptr_d[i] = int32_t((i < N ? int64_t(rowptr[i * S]) : E) + i);
      continue;
    }
    if (t < E) {                            // an original edge (position t of the fwd CSR)
      int64_t lo = 0, hi = rows;            // last segment s with rowptr[s] <= t
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (int64_t(rowptr[mid]) <= t) lo = mid; else hi = mid;
      }
      const int64_t seg = lo, i = seg / S, slot = seg - i * S;
      const int32_t len = rowptr[seg + 1] - rowptr[seg];
      const int64_t pos = t + i;            // i self entries precede this row
      col_d[pos] = int32_t(int64_t(col[t]) * (S + 1) + slot);
      w_d[pos] = 1.0f / float(len);
      dst_d[pos] = int32_t(i);
    } else {                                // the self entry of destination i (last in its row)
      const int64_t i = t - E;
      const int64_t pos = int64_t(rowptr[(i + 1) * S]) + i;
      col_d[pos] = int32_t(i * (S + 1) + S);
      w_d[pos] = 1.0f;
      dst_d[pos] = int32_t(i);
    }
  }
}

// ------------------------------------------------------------------ hub plan
__global__ void hub_count_kernel(const int32_t* __restrict__ rowptr, int64_t num_rows, int32_t thresh,
                                 unsigned long long* __restrict__ counts) {
  unsigned long long hubs = 0, chunks = 0;
  for (int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; r < num_rows; r += int64_t(gridDim.x) * blockDim.x) {
    int32_t len = rowptr[r + 1] - rowptr[r];
    if (len > thresh) { hubs += 1; chunks += (len + thresh - 1) / thresh; }
  }
  // warp reduce then one atomic per warp (integers: deterministic result)
  for (int o = 16; o > 0; o >>= 1) {
    hubs += __shfl_xor_sync(0xffffffffu, hubs, o);
    chunks += __shfl_xor_sync(0xffffffffu, chunks, o);
  }
  if ((threadIdx.x & 31) == 0 && hubs) { atomicAdd(counts, hubs); atomicAdd(counts + 1, chunks); }
}

__global__ void hub_nchunks_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ hub_row,
                                   int64_t n_hub, int32_t thresh, int32_t* __restrict__ nch /* [n_hub+1] */) {
  int64_t h = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (h < n_hub) {
    int32_t r = hub_row[h];
    nch[h] = (rowptr[r + 1] - rowptr[r] + thresh - 1) / thresh;
  } else if (h == n_hub) {
    nch[h] = 0;
  }
}

__global__ void hub_fill_chunks_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ hub_row,
                                       const int32_t* __restrict__ hub_chunk_ptr, int64_t n_hub, int32_t thresh,
                                       int32_t* __restrict__ chunk_beg, int32_t* __restrict__ chunk_end) {
  // one warp per hub row; lanes stride over its chunks
  int64_t h = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (h >= n_hub) return;
  int32_t r = hub_row[h];
  int32_t b = rowptr[r], e = rowptr[r + 1];
  int32_t c0 = hub_chunk_ptr[h], c1 = hub_chunk_ptr[h + 1];
  for (int32_t c = c0 + lane; c < c1; c += 32) {
    int32_t cb = b + (c - c0) * thresh;
    int32_t ce = cb + thresh < e ? cb + thresh : e;
    chunk_beg[c] = cb;
    chunk_end[c] = ce;
  }
}

// ------------------------------------------------------------------ use rank of gathered rows
// count[c] = edges of the CSR that gather row c (integer atomics: order-independent)
__global__ void col_count_kernel(const int32_t* __restrict__ col, int64_t nnz, int64_t num_cols,
                                 int32_t* __restrict__ count, int* __restrict__ err) {
  for (int64_t e = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; e < nnz; e += int64_t(gridDim.x) * blockDim.x) {
    const int32_t c = col[e];
    if (c >= 0 && c < num_cols) atomicAdd(count + c, 1);
    else flag_error(err);
  }
}

// In place: count -> sort key nnz - count (the stable ascending sort then orders by count desc, id asc); vals = id.
__global__ void col_rank_keys_kernel(uint32_t* __restrict__ keys, int64_t nnz, int64_t num_cols,
                                     int32_t* __restrict__ vals) {
  for (int64_t c = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; c < num_cols; c += int64_t(gridDim.x) * blockDim.x) {
    keys[c] = uint32_t(nnz - int64_t(keys[c]));
    vals[c] = int32_t(c);
  }
}

__global__ void col_rank_scatter_kernel(const int32_t* __restrict__ order, int64_t num_cols, int32_t* __restrict__ rank) {
  for (int64_t r = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; r < num_cols; r += int64_t(gridDim.x) * blockDim.x)
    rank[order[r]] = int32_t(r);
}

// ------------------------------------------------------------------ band-ordered hub plan
// The band key of a gathered row: its use rank when a rank is given, else the row id itself.
__device__ __forceinline__ int32_t band_key(const int32_t* __restrict__ rank, int32_t c) { return rank ? rank[c] : c; }

// The hub edges listed row by row (hub_off[h] = first position of hub row h): key = band key of the gathered row,
// value = position.
__global__ void hub_band_keys_kernel(const int32_t* __restrict__ rowptr, const int32_t* __restrict__ col,
                                     const int32_t* __restrict__ rank, const int32_t* __restrict__ hub_row,
                                     const int32_t* __restrict__ hub_off, int64_t n_hub, uint32_t* __restrict__ keys,
                                     int32_t* __restrict__ vals) {
  const int64_t h = (blockIdx.x * int64_t(blockDim.x) + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (h >= n_hub) return;
  const int32_t e0 = rowptr[hub_row[h]], o0 = hub_off[h], n = hub_off[h + 1] - o0;
  for (int32_t j = lane; j < n; j += 32) {
    keys[o0 + j] = uint32_t(band_key(rank, col[e0 + j]));
    vals[o0 + j] = o0 + j;
  }
}

// key = hub row of list position vals[k] (last h with hub_off[h] <= vals[k])
__global__ void hub_band_rowkey_kernel(const int32_t* __restrict__ vals, int64_t n, const int32_t* __restrict__ hub_off,
                                       int64_t n_hub, uint32_t* __restrict__ keys) {
  for (int64_t k = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x) {
    const int32_t i = vals[k];
    int64_t lo = 0, hi = n_hub;
    while (hi - lo > 1) {
      const int64_t mid = (lo + hi) >> 1;
      if (hub_off[mid] <= i) lo = mid; else hi = mid;
    }
    keys[k] = uint32_t(lo);
  }
}

__global__ void hub_band_gather_kernel(const uint32_t* __restrict__ row_key, const int32_t* __restrict__ vals, int64_t n,
                                       const int32_t* __restrict__ rowptr, const int32_t* __restrict__ hub_row,
                                       const int32_t* __restrict__ hub_off, const int32_t* __restrict__ col,
                                       const float* __restrict__ w, int32_t* __restrict__ hub_col,
                                       float* __restrict__ hub_w) {
  for (int64_t k = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; k < n; k += int64_t(gridDim.x) * blockDim.x) {
    const int32_t h = int32_t(row_key[k]);
    const int32_t e = rowptr[hub_row[h]] + (vals[k] - hub_off[h]);
    hub_col[k] = col[e];
    if (hub_w) hub_w[k] = w[e];
  }
}

// Chunk starts of one hub row, whose edges [a, b) of hub_col are sorted by band key.  A band boundary (the key
// crosses a multiple of 2^shift) is kept as a cut when the pieces on both sides hold at least `min_run` edges; every
// piece between kept cuts is then cut into chunks of `thresh` edges.  emit(k, start) receives the k-th chunk start.
template <typename F>
__device__ int32_t hub_band_walk(const int32_t* __restrict__ hub_col, const int32_t* __restrict__ rank, int32_t a,
                                 int32_t b, int shift, int32_t thresh, int32_t min_run, F emit) {
  int32_t k = 0, last = a, s = a;
  while (s < b) {
    const int64_t next = (int64_t(band_key(rank, hub_col[s]) >> shift) + 1) << shift;   // first key of the next band
    int32_t lo = s, hi = b;                                              // first p in (s, b] with key(p) >= next
    while (lo < hi) {
      const int32_t mid = lo + ((hi - lo) >> 1);
      if (int64_t(band_key(rank, hub_col[mid])) >= next) hi = mid; else lo = mid + 1;
    }
    const int32_t p = lo;
    if (p < b && (p - last < min_run || b - p < min_run)) { s = p; continue; }
    for (int32_t q = last; q < p; q += thresh) emit(k++, q);
    last = s = p;
  }
  return k;
}

__global__ void hub_band_count_kernel(const int32_t* __restrict__ hub_col, const int32_t* __restrict__ rank,
                                      const int32_t* __restrict__ hub_off, int64_t n_hub, int shift, int32_t thresh,
                                      int32_t min_run, int32_t* __restrict__ nch /* [n_hub+1] */) {
  const int64_t h = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (h < n_hub)
    nch[h] = hub_band_walk(hub_col, rank, hub_off[h], hub_off[h + 1], shift, thresh, min_run, [](int32_t, int32_t) {});
  else if (h == n_hub) nch[h] = 0;
}

__global__ void hub_band_fill_kernel(const int32_t* __restrict__ hub_col, const int32_t* __restrict__ rank,
                                     const int32_t* __restrict__ hub_off, const int32_t* __restrict__ band_chunk_ptr,
                                     int64_t n_hub, int shift, int32_t thresh, int32_t min_run, int32_t* __restrict__ cut,
                                     uint32_t* __restrict__ keys, int32_t* __restrict__ vals) {
  const int64_t h = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  if (h == n_hub) cut[band_chunk_ptr[n_hub]] = hub_off[n_hub];        // the end of the last chunk
  if (h >= n_hub) return;
  const int32_t c0 = band_chunk_ptr[h];
  hub_band_walk(hub_col, rank, hub_off[h], hub_off[h + 1], shift, thresh, min_run, [&](int32_t k, int32_t q) {
    cut[c0 + k] = q;
    keys[c0 + k] = uint32_t(band_key(rank, hub_col[q]) >> shift);     // band of the chunk's first edge
    vals[c0 + k] = c0 + k;
  });
}

int bits_for(uint64_t n_keys) {  // number of key bits needed to represent values < n_keys
  int b = 1;
  while ((uint64_t(1) << b) < n_keys && b < 32) ++b;
  return b;
}

size_t sort_temp_bytes(int64_t E) { return prim::sort_temp_bytes(E); }
size_t scan_temp_bytes(int64_t n) { return prim::scan_temp_bytes(n); }
size_t select_temp_bytes(int64_t n) { return prim::select_temp_bytes(n); }

}  // namespace
}  // namespace gmlm

using namespace gmlm;

extern "C" {

int gmlm_abi_version(void) { return 1; }

const char* gmlm_last_error(void) { return err_buf(); }

int gmlm_set_tuning(const char* key, int value) {
  int old = -1;
  if (!strcmp(key, "spmm_variant")) { old = g_spmm_variant; g_spmm_variant = value; }
  else if (!strcmp(key, "spmm_unroll")) { old = g_spmm_unroll; g_spmm_unroll = value; }
  else if (!strcmp(key, "spmm_overlap")) { old = g_spmm_overlap; g_spmm_overlap = value; }
  else if (!strcmp(key, "halo_pull_ctas")) { old = g_halo_pull_ctas; g_halo_pull_ctas = value; }
  else if (!strcmp(key, "halo_pull_threads")) { old = g_halo_pull_threads; g_halo_pull_threads = value; }
  return old;
}

int gmlm_degree_i32(const int64_t* index, int64_t E, int64_t N, int32_t* deg, int check, void* stream) {
  return gmlm_degree_i32_masked(index, nullptr, E, N, deg, check, stream);
}

int gmlm_degree_i32_masked(const int64_t* index, const uint8_t* keep, int64_t E, int64_t N, int32_t* deg, int check,
                           void* stream) {
  GMLM_REQUIRE(E >= 0 && N >= 0, "degree: negative size");
  GMLM_REQUIRE(E == 0 || index != nullptr, "degree: null index");
  cudaStream_t st = as_stream(stream);
  if (N == 0) return GMLM_OK;
  int* d_flag = nullptr;
  if (check) {   // per-call flag from the stream-ordered allocator (this entry point has no workspace argument)
    GMLM_CUDA_TRY(cudaMallocAsync(reinterpret_cast<void**>(&d_flag), sizeof(int), st));
    GMLM_CUDA_TRY(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
  }
  GMLM_CUDA_TRY(cudaMemsetAsync(deg, 0, size_t(N) * sizeof(int32_t), st));
  if (E > 0) {
    degree_kernel<<<grid_for(E, 4), kThreads, 0, st>>>(index, keep, E, N, deg, d_flag);
    GMLM_LAUNCH_CHECK();
  }
  if (check) {
    int flag = 0;
    int rc = read_flag(d_flag, st, &flag);
    cudaFreeAsync(d_flag, st);
    if (rc) return rc;
    if (flag) return fail(GMLM_ERR_INDEX, "degree: index out of range [0,%lld)", (long long)N);
  }
  return GMLM_OK;
}

int gmlm_degree_f32(const int64_t* index, int64_t E, int64_t N, float* deg, int32_t* ws, int check, void* stream) {
  GMLM_REQUIRE(N == 0 || (deg && ws), "degree_f32: null output");
  int rc = gmlm_degree_i32(index, E, N, ws, check, stream);
  if (rc) return rc;
  if (N > 0) {
    i32_to_f32_kernel<<<grid_for(N, 4), kThreads, 0, as_stream(stream)>>>(ws, deg, N);
    GMLM_LAUNCH_CHECK();
  }
  return GMLM_OK;
}

int gmlm_edge_type_bucket(const int64_t* src, int64_t E, const int32_t* deg, int64_t N, const int32_t* bounds_host,
                          int num_bounds, int64_t* edge_type, void* stream) {
  GMLM_REQUIRE(num_bounds >= 0 && num_bounds <= 8, "edge_type_bucket: at most 8 bounds");
  GMLM_REQUIRE(E == 0 || (src && deg && edge_type), "edge_type_bucket: null pointer");
  Bounds b;
  b.n = num_bounds;
  for (int k = 0; k < 8; ++k) b.b[k] = k < num_bounds ? bounds_host[k] : 0;
  for (int k = 1; k < num_bounds; ++k) GMLM_REQUIRE(b.b[k] >= b.b[k - 1], "edge_type_bucket: bounds must ascend");
  if (E == 0) return GMLM_OK;
  edge_type_kernel<<<grid_for(E, 4), kThreads, 0, as_stream(stream)>>>(src, E, deg, N, b, edge_type, nullptr);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

int gmlm_checksum_i64(const int64_t* x, int64_t n, uint64_t* out2, void* stream) {
  GMLM_REQUIRE(n >= 0 && out2 != nullptr && (n == 0 || x != nullptr), "checksum: bad arguments");
  cudaStream_t st = as_stream(stream);
  GMLM_CUDA_TRY(cudaMemsetAsync(out2, 0, 2 * sizeof(uint64_t), st));
  if (n > 0) {
    checksum_kernel<<<grid_for(n, 8), kThreads, 0, st>>>(reinterpret_cast<const uint64_t*>(x), n,
                                                         reinterpret_cast<unsigned long long*>(out2));
    GMLM_LAUNCH_CHECK();
  }
  return GMLM_OK;
}

int gmlm_relation_histogram(const int64_t* edge_type, const uint8_t* keep, int64_t E, int R, int64_t* counts,
                            void* stream) {
  GMLM_REQUIRE(R >= 1 && R <= 64, "relation_histogram: 1..64 relations supported");
  cudaStream_t st = as_stream(stream);
  GMLM_CUDA_TRY(cudaMemsetAsync(counts, 0, size_t(R) * sizeof(int64_t), st));
  if (E > 0) {
    rel_hist_kernel<<<grid_for(E, 8), kThreads, 0, st>>>(edge_type, keep, E, R,
                                                         reinterpret_cast<unsigned long long*>(counts));
    GMLM_LAUNCH_CHECK();
  }
  return GMLM_OK;
}

size_t gmlm_csr_workspace_bytes(int64_t E, int64_t num_rows) {
  if (E < 1) E = 1;
  size_t t = sort_temp_bytes(E);
  size_t s = scan_temp_bytes(num_rows + 1);
  size_t sel = select_temp_bytes(num_rows);
  size_t prim_bytes = t > s ? t : s;
  if (sel > prim_bytes) prim_bytes = sel;
  // keys_in, keys_out (u32), vals_in (i32) + hub scratch (2 x u64) + the per-call error flag + alignment slack
  return prim_bytes + 3 * (size_t(E) * 4 + 256) + 4096;
}

int gmlm_csr_build(const int64_t* src, const int64_t* dst, const int64_t* edge_type, const uint8_t* keep, int64_t E,
                   int64_t N, int64_t Nsrc, int R, const int32_t* slot_of_rel_host, int S, int32_t* rowptr, int32_t* col,
                   int32_t* perm, int32_t* seg_of_edge, int64_t* nnz_host, void* ws, size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(E >= 0 && N >= 0 && Nsrc >= 0 && R >= 1 && R <= 64 && S >= 1 && S <= R, "csr_build: bad sizes");
  GMLM_REQUIRE(Nsrc < (int64_t(1) << 31) - 1, "csr_build: num_src must fit int32");
  GMLM_REQUIRE(E < (int64_t(1) << 31) - 1, "csr_build: more than 2^31-2 edges needs a 64-bit CSR");
  const int64_t rows = N * S;
  GMLM_REQUIRE(rows < (int64_t(1) << 31) - 1, "csr_build: num_nodes*num_slots must fit int32");
  GMLM_REQUIRE(rowptr != nullptr, "csr_build: null rowptr");
  GMLM_REQUIRE(ws_bytes >= gmlm_csr_workspace_bytes(E, rows), "csr_build: workspace too small");
  cudaStream_t st = as_stream(stream);
  SlotMap sm;
  for (int r = 0; r < 64; ++r) sm.slot[r] = -1;
  if (edge_type == nullptr) {
    sm.slot[0] = 0;
  } else {
    for (int r = 0; r < R; ++r) {
      int32_t s = slot_of_rel_host ? slot_of_rel_host[r] : r;
      GMLM_REQUIRE(s >= -1 && s < S, "csr_build: slot_of_rel out of range");
      sm.slot[r] = s;
    }
  }
  GMLM_CUDA_TRY(cudaMemsetAsync(rowptr, 0, size_t(rows + 1) * sizeof(int32_t), st));
  if (nnz_host) *nnz_host = 0;
  if (E == 0) return GMLM_OK;
  GMLM_REQUIRE(src && dst && col && perm, "csr_build: null pointer");

  Carver cv(ws);
  uint32_t* keys_in = cv.take<uint32_t>(E);
  uint32_t* keys_out = cv.take<uint32_t>(E);
  int32_t* vals_in = cv.take<int32_t>(E);
  int* d_flag = cv.take<int>(1);
  void* prim_ws = cv.take<char>(0);
  size_t prim_bytes = ws_bytes - cv.used();

  GMLM_CUDA_TRY(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
  make_keys_kernel<<<grid_for(E, 2), kThreads, 0, st>>>(src, dst, edge_type, keep, E, N, Nsrc, edge_type ? R : 1, sm, S,
                                                        keys_in, vals_in, seg_of_edge, rowptr, d_flag);
  GMLM_LAUNCH_CHECK();
  // counts -> exclusive prefix (in place); entry [rows] is 0 on input so rowptr[rows] = E
  if (int rc = prim::exclusive_scan_i32(rowptr, rowptr, rows + 1, prim_ws, prim_bytes, st)) return rc;
  // the LSD radix sort is stable: equal (dst,slot) keys keep the original edge order
  if (int rc = prim::radix_sort_pairs(keys_in, vals_in, keys_out, perm, E, bits_for(uint64_t(rows) + (keep ? 1 : 0)),
                                      prim_ws, prim_bytes, st))
    return rc;
  gather_col_kernel<<<grid_for(E, 2), kThreads, 0, st>>>(src, perm, E, col);
  GMLM_LAUNCH_CHECK();
  int flag = 0;
  int32_t kept = int32_t(E);
  if (nnz_host) GMLM_CUDA_TRY(cudaMemcpyAsync(&kept, rowptr + rows, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  int rc = read_flag(d_flag, st, &flag);       // synchronises the stream: `kept` has arrived too
  if (rc) return rc;
  if (nnz_host) *nnz_host = kept;
  if (flag) return fail(GMLM_ERR_INDEX, "csr_build: dst outside [0,%lld), src outside [0,%lld) or relation outside [0,%d)",
                        (long long)N, (long long)Nsrc, R);
  return GMLM_OK;
}

int gmlm_csr_transpose(const int64_t* row_of_edge, const int32_t* payload, const float* edge_w,
                       const int32_t* fwd_rowptr, const uint8_t* keep, int64_t E, int64_t num_rows, int32_t* rowptr_t,
                       int32_t* payload_t, float* w_t, int32_t* perm_t, void* ws, size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(E >= 0 && num_rows >= 0, "csr_transpose: bad sizes");
  GMLM_REQUIRE(E < (int64_t(1) << 31) - 1 && num_rows < (int64_t(1) << 31) - 1, "csr_transpose: int32 limits");
  GMLM_REQUIRE(ws_bytes >= gmlm_csr_workspace_bytes(E, num_rows), "csr_transpose: workspace too small");
  cudaStream_t st = as_stream(stream);
  GMLM_CUDA_TRY(cudaMemsetAsync(rowptr_t, 0, size_t(num_rows + 1) * sizeof(int32_t), st));
  if (E == 0) return GMLM_OK;
  GMLM_REQUIRE(row_of_edge && payload && payload_t && perm_t, "csr_transpose: null pointer");
  GMLM_REQUIRE(!(fwd_rowptr || edge_w) || w_t, "csr_transpose: w_t required");

  Carver cv(ws);
  uint32_t* keys_in = cv.take<uint32_t>(E);
  uint32_t* keys_out = cv.take<uint32_t>(E);
  int32_t* vals_in = cv.take<int32_t>(E);
  int* d_flag = cv.take<int>(1);
  void* prim_ws = cv.take<char>(0);
  size_t prim_bytes = ws_bytes - cv.used();

  GMLM_CUDA_TRY(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
  make_keys_t_kernel<<<grid_for(E, 2), kThreads, 0, st>>>(row_of_edge, keep, E, num_rows, keys_in, vals_in, rowptr_t,
                                                          d_flag);
  GMLM_LAUNCH_CHECK();
  if (int rc = prim::exclusive_scan_i32(rowptr_t, rowptr_t, num_rows + 1, prim_ws, prim_bytes, st)) return rc;
  if (int rc = prim::radix_sort_pairs(keys_in, vals_in, keys_out, perm_t, E,
                                      bits_for(uint64_t(num_rows) + (keep ? 1 : 0)), prim_ws, prim_bytes, st))
    return rc;
  gather_payload_t_kernel<<<grid_for(E, 2), kThreads, 0, st>>>(payload, edge_w, fwd_rowptr, perm_t, keep, E, payload_t,
                                                               w_t);
  GMLM_LAUNCH_CHECK();
  int flag = 0;
  int rc = read_flag(d_flag, st, &flag);
  if (rc) return rc;
  if (flag) return fail(GMLM_ERR_INDEX, "csr_transpose: row id outside [0,%lld)", (long long)num_rows);
  return GMLM_OK;
}

int gmlm_dst_plan(const int32_t* rowptr, const int32_t* col, int64_t N, int S, int64_t E, int64_t Nsrc,
                  int32_t* rowptr_d, int32_t* col_d, float* w_d, int32_t* dst_d, void* stream) {
  GMLM_REQUIRE(N >= 0 && S >= 1 && E >= 0 && Nsrc >= N, "dst_plan: bad sizes");
  GMLM_REQUIRE(E + N < (int64_t(1) << 31) - 1 && Nsrc * (S + 1) < (int64_t(1) << 31) - 1, "dst_plan: int32 limits");
  GMLM_REQUIRE(rowptr && rowptr_d && (E + N == 0 || (col_d && w_d && dst_d)) && (E == 0 || col), "dst_plan: null pointer");
  const int64_t threads = E + 2 * N + 1;
  dst_plan_kernel<<<grid_for(threads, 2), kThreads, 0, as_stream(stream)>>>(rowptr, col, N, S, E, rowptr_d, col_d, w_d,
                                                                           dst_d);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

int gmlm_hub_count(const int32_t* rowptr, int64_t num_rows, int32_t thresh, int64_t* counts_host, void* ws,
                   size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(thresh >= 1, "hub_count: thresh must be >= 1");
  GMLM_REQUIRE(ws_bytes >= 16, "hub_count: workspace too small");
  cudaStream_t st = as_stream(stream);
  counts_host[0] = counts_host[1] = 0;
  if (num_rows == 0) return GMLM_OK;
  unsigned long long* d = static_cast<unsigned long long*>(ws);
  GMLM_CUDA_TRY(cudaMemsetAsync(d, 0, 16, st));
  hub_count_kernel<<<grid_for(num_rows, 4), kThreads, 0, st>>>(rowptr, num_rows, thresh, d);
  GMLM_LAUNCH_CHECK();
  unsigned long long h[2];
  GMLM_CUDA_TRY(cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, st));
  GMLM_CUDA_TRY(cudaStreamSynchronize(st));
  counts_host[0] = int64_t(h[0]);
  counts_host[1] = int64_t(h[1]);
  return GMLM_OK;
}

int gmlm_hub_fill(const int32_t* rowptr, int64_t num_rows, int32_t thresh, int64_t n_hub, int64_t n_chunks,
                  int32_t* hub_row, int32_t* hub_chunk_ptr, int32_t* chunk_beg, int32_t* chunk_end, void* ws,
                  size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(thresh >= 1 && n_hub >= 0 && n_chunks >= 0, "hub_fill: bad sizes");
  if (n_hub == 0) return GMLM_OK;
  GMLM_REQUIRE(hub_row && hub_chunk_ptr && chunk_beg && chunk_end, "hub_fill: null pointer");
  cudaStream_t st = as_stream(stream);
  Carver cv(ws);
  int32_t* d_num = cv.take<int32_t>(1);
  void* prim_ws = cv.take<char>(0);
  GMLM_REQUIRE(ws_bytes > cv.used(), "hub_fill: workspace too small");
  size_t prim_bytes = ws_bytes - cv.used();
  // ascending list of hub rows (the selection keeps input order)
  (void)d_num;
  if (int rc = prim::select_rows(rowptr, num_rows, thresh, hub_row, n_hub, prim_ws, prim_bytes, st)) return rc;
  hub_nchunks_kernel<<<int((n_hub + 1 + kThreads - 1) / kThreads), kThreads, 0, st>>>(rowptr, hub_row, n_hub, thresh,
                                                                                   hub_chunk_ptr);
  GMLM_LAUNCH_CHECK();
  if (int rc = prim::exclusive_scan_i32(hub_chunk_ptr, hub_chunk_ptr, n_hub + 1, prim_ws, prim_bytes, st)) return rc;
  int64_t threads = n_hub * 32;
  hub_fill_chunks_kernel<<<int((threads + kThreads - 1) / kThreads), kThreads, 0, st>>>(
      rowptr, hub_row, hub_chunk_ptr, n_hub, thresh, chunk_beg, chunk_end);
  GMLM_LAUNCH_CHECK();
  return GMLM_OK;
}

size_t gmlm_col_rank_workspace_bytes(int64_t num_cols) {
  if (num_cols < 1) num_cols = 1;
  // keys, sorted keys (u32), ids, order (i32) + the per-call error flag + alignment slack
  return sort_temp_bytes(num_cols) + 4 * (size_t(num_cols) * 4 + 256) + 4096;
}

int gmlm_col_rank(const int32_t* col, int64_t nnz, int64_t num_cols, int32_t* rank, void* ws, size_t ws_bytes,
                  void* stream) {
  GMLM_REQUIRE(nnz >= 0 && num_cols >= 0 && nnz < (int64_t(1) << 31) - 1 && num_cols < (int64_t(1) << 31) - 1,
               "col_rank: bad sizes");
  GMLM_REQUIRE(ws_bytes >= gmlm_col_rank_workspace_bytes(num_cols), "col_rank: workspace too small");
  if (num_cols == 0) return GMLM_OK;
  GMLM_REQUIRE(rank && (nnz == 0 || col), "col_rank: null pointer");
  cudaStream_t st = as_stream(stream);
  Carver cv(ws);
  uint32_t* keys_a = cv.take<uint32_t>(num_cols);
  uint32_t* keys_b = cv.take<uint32_t>(num_cols);
  int32_t* vals_a = cv.take<int32_t>(num_cols);
  int32_t* order = cv.take<int32_t>(num_cols);
  int* d_flag = cv.take<int>(1);
  void* prim_ws = cv.take<char>(0);
  const size_t prim_bytes = ws_bytes - cv.used();
  GMLM_CUDA_TRY(cudaMemsetAsync(d_flag, 0, sizeof(int), st));
  GMLM_CUDA_TRY(cudaMemsetAsync(keys_a, 0, size_t(num_cols) * sizeof(uint32_t), st));
  if (nnz > 0) {
    col_count_kernel<<<grid_for(nnz, 4), kThreads, 0, st>>>(col, nnz, num_cols, reinterpret_cast<int32_t*>(keys_a),
                                                            d_flag);
    GMLM_LAUNCH_CHECK();
  }
  col_rank_keys_kernel<<<grid_for(num_cols, 2), kThreads, 0, st>>>(keys_a, nnz, num_cols, vals_a);
  GMLM_LAUNCH_CHECK();
  // stable: rows of equal use keep ascending id order
  if (int rc = prim::radix_sort_pairs(keys_a, vals_a, keys_b, order, num_cols, bits_for(uint64_t(nnz) + 1), prim_ws,
                                      prim_bytes, st))
    return rc;
  col_rank_scatter_kernel<<<grid_for(num_cols, 2), kThreads, 0, st>>>(order, num_cols, rank);
  GMLM_LAUNCH_CHECK();
  int flag = 0;
  if (int rc = read_flag(d_flag, st, &flag)) return rc;
  if (flag) return fail(GMLM_ERR_INDEX, "col_rank: col outside [0,%lld)", (long long)num_cols);
  return GMLM_OK;
}

size_t gmlm_hub_band_workspace_bytes(int64_t n_hub_edges) {
  if (n_hub_edges < 1) n_hub_edges = 1;
  const size_t prim_bytes = std::max(sort_temp_bytes(n_hub_edges), scan_temp_bytes(n_hub_edges + 1));
  return prim_bytes + 4 * (size_t(n_hub_edges) * 4 + 256) + 4096;
}

int gmlm_hub_band_sort(const int32_t* rowptr, const int32_t* col, const float* w, const int32_t* rank, int64_t n_hub,
                       const int32_t* hub_row, const int32_t* hub_off, int64_t n_hub_edges, int band_shift,
                       int32_t thresh, int32_t min_run,
                       int32_t* hub_col, float* hub_w, int32_t* band_chunk_ptr, int64_t* n_band_host, void* ws,
                       size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(n_hub >= 0 && n_hub_edges >= 0 && n_hub_edges < (int64_t(1) << 31) - 1, "hub_band_sort: bad sizes");
  GMLM_REQUIRE(band_shift >= 1 && band_shift <= 30 && thresh >= 1 && min_run >= 1, "hub_band_sort: bad band parameters");
  GMLM_REQUIRE(ws_bytes >= gmlm_hub_band_workspace_bytes(n_hub_edges), "hub_band_sort: workspace too small");
  *n_band_host = 0;
  if (n_hub == 0) return GMLM_OK;
  GMLM_REQUIRE(rowptr && col && hub_row && hub_off && hub_col && band_chunk_ptr && (hub_w == nullptr || w != nullptr),
               "hub_band_sort: null pointer");
  cudaStream_t st = as_stream(stream);
  Carver cv(ws);
  uint32_t* keys_a = cv.take<uint32_t>(n_hub_edges);
  uint32_t* keys_b = cv.take<uint32_t>(n_hub_edges);
  int32_t* vals_a = cv.take<int32_t>(n_hub_edges);
  int32_t* vals_b = cv.take<int32_t>(n_hub_edges);
  void* prim_ws = cv.take<char>(0);
  const size_t prim_bytes = ws_bytes - cv.used();
  // stable by band key, then stable by hub row: each row's edges in key order, ties in CSR order
  hub_band_keys_kernel<<<int((n_hub * 32 + kThreads - 1) / kThreads), kThreads, 0, st>>>(rowptr, col, rank, hub_row,
                                                                                       hub_off, n_hub, keys_a, vals_a);
  GMLM_LAUNCH_CHECK();
  if (int rc = prim::radix_sort_pairs(keys_a, vals_a, keys_b, vals_b, n_hub_edges, 31, prim_ws, prim_bytes, st)) return rc;
  hub_band_rowkey_kernel<<<grid_for(n_hub_edges, 2), kThreads, 0, st>>>(vals_b, n_hub_edges, hub_off, n_hub, keys_b);
  GMLM_LAUNCH_CHECK();
  if (int rc = prim::radix_sort_pairs(keys_b, vals_b, keys_a, vals_a, n_hub_edges, bits_for(uint64_t(n_hub)), prim_ws,
                                      prim_bytes, st))
    return rc;
  hub_band_gather_kernel<<<grid_for(n_hub_edges, 2), kThreads, 0, st>>>(keys_a, vals_a, n_hub_edges, rowptr, hub_row,
                                                                        hub_off, col, w, hub_col, hub_w);
  GMLM_LAUNCH_CHECK();
  hub_band_count_kernel<<<int((n_hub + 1 + kThreads - 1) / kThreads), kThreads, 0, st>>>(
      hub_col, rank, hub_off, n_hub, band_shift, thresh, min_run, band_chunk_ptr);
  GMLM_LAUNCH_CHECK();
  if (int rc = prim::exclusive_scan_i32(band_chunk_ptr, band_chunk_ptr, n_hub + 1, prim_ws, prim_bytes, st)) return rc;
  int32_t n_band = 0;
  GMLM_CUDA_TRY(cudaMemcpyAsync(&n_band, band_chunk_ptr + n_hub, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
  GMLM_CUDA_TRY(cudaStreamSynchronize(st));
  *n_band_host = n_band;
  return GMLM_OK;
}

int gmlm_hub_band_order(const int32_t* hub_col, const int32_t* rank, const int32_t* hub_off, int64_t n_hub,
                        int64_t n_hub_edges, int64_t n_band, int band_shift, int32_t thresh, int32_t min_run,
                        int32_t* band_plan, void* ws, size_t ws_bytes, void* stream) {
  GMLM_REQUIRE(n_hub >= 0 && n_band >= n_hub && n_band <= n_hub_edges, "hub_band_order: bad sizes");
  GMLM_REQUIRE(band_shift >= 1 && band_shift <= 30 && thresh >= 1 && min_run >= 1, "hub_band_order: bad band parameters");
  GMLM_REQUIRE(ws_bytes >= gmlm_hub_band_workspace_bytes(n_hub_edges), "hub_band_order: workspace too small");
  if (n_hub == 0) return GMLM_OK;
  GMLM_REQUIRE(hub_col && hub_off && band_plan, "hub_band_order: null pointer");
  cudaStream_t st = as_stream(stream);
  const int32_t* band_chunk_ptr = band_plan;
  int32_t* cut = band_plan + n_hub + 1;
  int32_t* order = cut + n_band + 1;
  Carver cv(ws);
  uint32_t* keys_a = cv.take<uint32_t>(n_band);
  uint32_t* keys_b = cv.take<uint32_t>(n_band);
  int32_t* vals_a = cv.take<int32_t>(n_band);
  void* prim_ws = cv.take<char>(0);
  const size_t prim_bytes = ws_bytes - cv.used();
  hub_band_fill_kernel<<<int((n_hub + 1 + kThreads - 1) / kThreads), kThreads, 0, st>>>(
      hub_col, rank, hub_off, band_chunk_ptr, n_hub, band_shift, thresh, min_run, cut, keys_a, vals_a);
  GMLM_LAUNCH_CHECK();
  // stable by band: chunks of one band keep their row order
  if (int rc = prim::radix_sort_pairs(keys_a, vals_a, keys_b, order, n_band, bits_for((uint64_t(0x7fffffff) >> band_shift) + 1),
                                      prim_ws, prim_bytes, st))
    return rc;
  return GMLM_OK;
}

}  // extern "C"
