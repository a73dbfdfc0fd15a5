// Radius submap selection of the offline loader on the GPU (SURVEY.md 8f rank 1).
//
// Reference: src/sps/datasets/blt_dataset.py:222-226,258-271 --
//     kd_tree_scan.query_ball_tree(kd_tree_target, VOXEL_SIZE)  ->  np.concatenate(per-scan-point lists)
// i.e. for every scan point, in scan order, the indices of ALL map points within Euclidean distance <= r
// (float64, scipy cKDTree), duplicates kept across scan points; the submap rows are map[idx] with their original
// coordinates.  The kd-trees are replaced by a uniform grid of edge r over the (static) map, held in the library's
// open-addressing hash: a ball of radius r around p only meets the 27 cells around cell(p).
//   build (once per map):  cell key per map point -> hash insert -> per-cell counts -> exclusive scan -> indices
//                          grouped by cell, ascending inside a cell
//   query (per scan):      pass 1 counts the hits of every scan point, a single-block scan turns counts into
//                          offsets, pass 2 writes them: per scan point the hits come cell by cell (dz, dy, dx
//                          ascending), ascending map index inside a cell.  scipy's order inside one point's list is
//                          its tree traversal order (unspecified); the multiset per scan point is identical.
// Distances are evaluated in fp64 on the fp32 coordinates, like scipy after its float64 conversion.
#include "partials.cuh"
#include "scan.cuh"

struct sps_ballmap {
  sps::Slot* table = nullptr;   // cell key -> val = slot index + 1 (= index into cell_start)
  uint32_t cap = 0;
  int32_t* cell_start = nullptr;   // [cap + 1] exclusive scan of the per-slot point counts
  int32_t* sorted_idx = nullptr;   // [n] map point indices grouped by cell
  const float* xyz = nullptr;      // the caller's map points (must stay alive)
  int32_t* scalars = nullptr;      // [2] status
  int64_t n = 0;
  double radius = 0.0;
};

namespace sps {

constexpr int kBallBlock = 1024;

__device__ __forceinline__ bool cell_of(const float* __restrict__ p, double inv_r, int& cx, int& cy, int& cz) {
  const double fx = floor((double)p[0] * inv_r), fy = floor((double)p[1] * inv_r), fz = floor((double)p[2] * inv_r);
  const bool ok = fx >= -(double)kXBias + 1 && fx < (double)kXBias - 1 && fy >= -(double)kXBias + 1 &&
                  fy < (double)kXBias - 1 && fz >= -(double)kZBias + 1 && fz < (double)kZBias - 1;
  cx = (int)fx; cy = (int)fy; cz = (int)fz;
  return ok;   // also false for NaN
}

__global__ void k_ball_clear(Slot* tab, uint32_t cap) {
  const int4 empty = make_int4(-1, -1, 0, 0);
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += gridDim.x * blockDim.x)
    reinterpret_cast<int4*>(tab)[i] = empty;
}

// hash slot of every map point's cell (the slot index doubles as the cell's index in cell_start), per-cell counts
__global__ void k_ball_insert(const float* __restrict__ xyz, int n, double inv_r, Slot* tab, uint32_t mask,
                              int32_t* __restrict__ cell_of_pt, int32_t* __restrict__ cell_count, int32_t* scalars) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int cx, cy, cz;
    if (!cell_of(xyz + (int64_t)i * 3, inv_r, cx, cy, cz)) {
      atomicOr(scalars + 2, kStatusRange);
      cell_of_pt[i] = -1;
      continue;
    }
    const unsigned long long key = pack_key(0, cx, cy, cz, 0);
    uint32_t s = hash_key(key) & mask;
    while (true) {
      const unsigned long long prev = atomicCAS(&tab[s].key, kEmptyKey, key);
      if (prev == kEmptyKey) { tab[s].val = (int)s + 1; break; }   // read by the query kernels only
      if (prev == key) break;
      s = (s + 1) & mask;
    }
    cell_of_pt[i] = (int)s;
    atomicAdd(cell_count + s, 1);
  }
}

// single-block exclusive scan: out[i] = sum_{j<i} in[j], out[n] = total
__global__ void __launch_bounds__(kBallBlock) k_ball_scan(const int32_t* __restrict__ in, const int32_t* __restrict__ n_ptr,
                                                          int n_host, int32_t* __restrict__ out, int32_t* total_out) {
  __shared__ int warp_sums[kBallBlock / 32];
  __shared__ int carry;
  const int n = n_ptr ? *n_ptr : n_host;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < n; base += kBallBlock) {
    const int j = base + tid;
    const int v = j < n ? in[j] : 0;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += u;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      const int w = warp_sums[lane];
      int wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int u = __shfl_up_sync(0xffffffffu, wi, d);
        if (lane >= d) wi += u;
      }
      warp_sums[lane] = wi - w;
    }
    __syncthreads();
    const int ex = inc - v + warp_sums[wid] + carry;
    if (j < n) out[j] = ex;
    __syncthreads();
    if (tid == kBallBlock - 1) carry = ex + v;
    __syncthreads();
  }
  if (tid == 0) {
    out[n] = carry;
    if (total_out) *total_out = carry;
  }
}

__global__ void k_ball_fill(const int32_t* __restrict__ cell_of_pt, int n, const int32_t* __restrict__ cell_start,
                            int32_t* __restrict__ cursor, int32_t* __restrict__ sorted_idx) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int c = cell_of_pt[i];
    if (c < 0) continue;
    sorted_idx[cell_start[c] + atomicAdd(cursor + c, 1)] = i;
  }
}

// ascending map index inside every cell (cells hold a handful of points): insertion sort, one thread per cell
__global__ void k_ball_sort_cells(const int32_t* __restrict__ cell_start, int nc, int32_t* __restrict__ sorted_idx) {
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < nc; c += gridDim.x * blockDim.x) {
    const int b = cell_start[c], e = cell_start[c + 1];
    for (int i = b + 1; i < e; ++i) {
      const int v = sorted_idx[i];
      int j = i - 1;
      while (j >= b && sorted_idx[j] > v) { sorted_idx[j + 1] = sorted_idx[j]; --j; }
      sorted_idx[j + 1] = v;
    }
  }
}

// The map side of a query: the hash of occupied cells, the per-cell index lists and the radius.
struct BallGrid {
  const Slot* tab; uint32_t mask; const int32_t* cell_start; const int32_t* sorted_idx; const float* xyz;
  double inv_r, r2;
};

// Every map point within the radius of p, cell by cell (dz, dy, dx ascending), ascending map index inside a cell:
// hit(m, q) per hit (q = map point m's xyz).  Returns the number of hits; points outside the grid's range have none.
template <class Hit>
__device__ __forceinline__ int ball_probe(const float* __restrict__ p, const BallGrid& g, Hit&& hit) {
  int cx, cy, cz;
  int hits = 0;
  if (cell_of(p, g.inv_r, cx, cy, cz)) {
    const double px = p[0], py = p[1], pz = p[2];
    for (int dz = -1; dz <= 1; ++dz)
      for (int dy = -1; dy <= 1; ++dy)
        for (int dx = -1; dx <= 1; ++dx) {
          const int c = table_find(g.tab, g.mask, pack_key(0, cx + dx, cy + dy, cz + dz, 0));
          if (c <= 0) continue;                    // val = hash slot + 1
          const int b = __ldg(g.cell_start + c - 1), e = __ldg(g.cell_start + c);
          for (int j = b; j < e; ++j) {
            const int m = __ldg(g.sorted_idx + j);
            const float* q = g.xyz + (int64_t)m * 3;
            const double ex = (double)__ldg(q) - px, ey = (double)__ldg(q + 1) - py, ez = (double)__ldg(q + 2) - pz;
            if (ex * ex + ey * ey + ez * ez <= g.r2) {
              hit(m, q);
              ++hits;
            }
          }
        }
  }
  return hits;
}

// WRITE = false: counts[i] = hits of scan point i; WRITE = true: out[offsets[i] ...] = their map indices
template <bool WRITE>
__global__ void k_ball_query(const float* __restrict__ scan, int64_t ld, int n_scan, BallGrid g,
                             int32_t* __restrict__ counts, const int32_t* __restrict__ offsets,
                             int32_t* __restrict__ out, int64_t out_cap) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_scan; i += gridDim.x * blockDim.x) {
    int64_t w = WRITE ? offsets[i] : 0;
    const int hits = ball_probe(scan + (int64_t)i * ld, g, [&](int m, const float*) {
      if (WRITE) { if (w < out_cap) out[w] = m; ++w; }
    });
    if (!WRITE) counts[i] = hits;
  }
}

// ---- batched query: B scans concatenated -> collated rows [b, x, y, z, t, label] ----
// blt_dataset.py:173-182 (collate) over 209-243 (one item per scan): for b = 0..B-1 the n_b scan rows (t = 1, their
// label), then scan b's submap rows map[idx] (t = 0, label 1), idx as sps_submap_ball_query returns it for that scan.
// With H = the exclusive prefix of the per-point hit counts over the whole batch, scan b's rows start at
// off[b] + H[off[b]] and scan point i's hits at off[b+1] + H[i] (BatchOffsets, batch_of, hit_prefix: scan.cuh).

// pass 1: hits of every scan point of the batch, fused with the grid-wide exclusive scan of the counts (scan.cuh)
__global__ void __launch_bounds__(kScanBlock)
k_radius_batch_count(const float* __restrict__ scan, int64_t ld, int n, BallGrid g, int32_t* __restrict__ rank,
                     int32_t* block_sums, uint32_t* ticket, int32_t* total) {
  const int nb = max(1, (n + kScanBlock - 1) / kScanBlock);
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  const int hits = i < n ? ball_probe(scan + (int64_t)i * ld, g, [](int, const float*) {}) : 0;
  scan_flags(hits, i, n, nb, rank, block_sums, ticket, total);
}

__device__ __forceinline__ void write_row(float* __restrict__ rows, int64_t r, float b, float x, float y, float z, float t,
                                          float label) {
  float* o = rows + r * 6;
  o[0] = b; o[1] = x; o[2] = y; o[3] = z; o[4] = t; o[5] = label;
}

// pass 2: the rows in collate order (none at or past `cap`), the per-scan row offsets and the true row count.
// n_fwd / status (optional, fused call): the row count the forward runs on (0 when the rows did not fit) and the
// context's sticky status word, which gets kStatusCapacity then.
__global__ void __launch_bounds__(256, 4)   // (without the minimum ptxas settles on 32 registers and spills)
k_radius_batch_write(const float* __restrict__ scan, int64_t ld, int n, const __grid_constant__ BatchOffsets bo, BallGrid g,
                     const int32_t* __restrict__ rank, const int32_t* __restrict__ block_sums,
                     const int32_t* __restrict__ total_ptr, float* __restrict__ rows, int64_t cap,
                     int32_t* __restrict__ row_off, int32_t* __restrict__ n_rows, int32_t* __restrict__ n_fwd,
                     int32_t* status) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  const int total = *total_ptr;
  if (blockIdx.x == 0) {
    for (int b = threadIdx.x; b <= bo.batch; b += blockDim.x)
      row_off[b] = s_off[b] + hit_prefix(rank, block_sums, n, total, s_off[b]);
    if (threadIdx.x == 0) {
      const int64_t nr = (int64_t)n + total;
      *n_rows = (int32_t)nr;
      if (n_fwd) *n_fwd = nr <= cap ? (int32_t)nr : 0;
      if (status && nr > cap) atomicOr(status, kStatusCapacity);
    }
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int b = batch_of(s_off, bo.batch, i);
    const float* p = scan + (int64_t)i * ld;
    const float fb = (float)b;
    const int64_t r = (int64_t)i + hit_prefix(rank, block_sums, n, total, s_off[b]);
    if (r < cap) write_row(rows, r, fb, p[0], p[1], p[2], 1.0f, p[3]);
    int64_t w = (int64_t)s_off[b + 1] + hit_prefix(rank, block_sums, n, total, i);
    ball_probe(p, g, [&](int, const float* q) {
      if (w < cap) write_row(rows, w, fb, __ldg(q), __ldg(q + 1), __ldg(q + 2), 0.0f, 1.0f);
      ++w;
    });
  }
}

// per-scan metric partials of the fused call: k_radius_partials (partials.cuh)

static inline int grid_of(int64_t work, int block) {
  int64_t g = (work + block - 1) / block;
  if (g < 1) g = 1;
  if (g > 148 * 16) g = 148 * 16;
  return (int)g;
}

struct BallCarve {
  int32_t* scalars; Slot* table; uint32_t cap; int32_t* cell_of_pt; int32_t* cell_count; int32_t* cell_start;
  int32_t* sorted_idx; size_t bytes;
};
static BallCarve carve_ball(void* base, int64_t n) {
  BallCarve c;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t b) { off = (off + 255) & ~size_t(255); char* r = p ? p + off : nullptr; off += b; return r; };
  c.scalars = (int32_t*)take(64 * 4);
  c.cap = table_capacity(n);
  c.table = (Slot*)take((size_t)c.cap * sizeof(Slot));
  c.cell_of_pt = (int32_t*)take((size_t)n * 4);
  c.cell_count = (int32_t*)take((size_t)(c.cap + 1) * 4);   // per hash slot; reused as the fill cursor
  c.cell_start = (int32_t*)take((size_t)(c.cap + 2) * 4);
  c.sorted_idx = (int32_t*)take((size_t)n * 4);
  c.bytes = (off + 255) & ~size_t(255);
  return c;
}

}  // namespace sps

using namespace sps;

extern "C" size_t sps_ballmap_bytes(int64_t n_map) { return carve_ball(nullptr, n_map < 1 ? 1 : n_map).bytes; }

extern "C" int sps_ballmap_build(sps_ballmap** out, void* d_storage, size_t bytes, const float* d_map_xyz, int64_t n,
                                 double radius, void* stream_) {
  if (!out || !d_storage || ((uintptr_t)d_storage & 255) || (!d_map_xyz && n > 0) || n < 0 || !(radius > 0.0) ||
      n > 0x7fffffff)
    return SPS_ERR_BAD_ARG;
  const int64_t nn = n > 0 ? n : 1;
  BallCarve c = carve_ball(d_storage, nn);
  if (c.bytes > bytes) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream_;
  SPS_CUDA_CHECK(cudaMemsetAsync(c.scalars, 0, 64 * 4, st));
  SPS_CUDA_CHECK(cudaMemsetAsync(c.cell_count, 0, (size_t)(c.cap + 1) * 4, st));
  k_ball_clear<<<grid_of(c.cap, 256), 256, 0, st>>>(c.table, c.cap);
  k_ball_insert<<<grid_of(nn, 256), 256, 0, st>>>(d_map_xyz, (int)n, 1.0 / radius, c.table, c.cap - 1, c.cell_of_pt,
                                                   c.cell_count, c.scalars);
  k_ball_scan<<<1, kBallBlock, 0, st>>>(c.cell_count, nullptr, (int)c.cap, c.cell_start, nullptr);
  SPS_CUDA_CHECK(cudaMemsetAsync(c.cell_count, 0, (size_t)(c.cap + 1) * 4, st));
  k_ball_fill<<<grid_of(nn, 256), 256, 0, st>>>(c.cell_of_pt, (int)n, c.cell_start, c.cell_count, c.sorted_idx);
  k_ball_sort_cells<<<grid_of(c.cap, 256), 256, 0, st>>>(c.cell_start, (int)c.cap, c.sorted_idx);
  SPS_CUDA_CHECK(cudaGetLastError());
  int32_t status = 0;
  SPS_CUDA_CHECK(cudaMemcpyAsync(&status, c.scalars + 2, 4, cudaMemcpyDeviceToHost, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  if (status & kStatusRange) return SPS_ERR_COORD_RANGE;
  sps_ballmap* m = new sps_ballmap();
  m->table = c.table; m->cap = c.cap; m->cell_start = c.cell_start; m->sorted_idx = c.sorted_idx; m->xyz = d_map_xyz;
  m->scalars = c.scalars; m->n = n; m->radius = radius;
  *out = m;
  return SPS_OK;
}

extern "C" int sps_ballmap_destroy(sps_ballmap* m) {
  delete m;
  return SPS_OK;
}

extern "C" size_t sps_ball_query_scratch_bytes(int64_t n_scan) {
  if (n_scan < 1) n_scan = 1;
  return (((size_t)(n_scan + 2) * 4 + 255) & ~size_t(255)) * 2;
}

static BallGrid grid_of_map(const sps_ballmap* bm) {
  return BallGrid{bm->table, bm->cap - 1, bm->cell_start, bm->sorted_idx, bm->xyz, 1.0 / bm->radius, bm->radius * bm->radius};
}

extern "C" int sps_submap_ball_query(const sps_ballmap* bm, const float* d_scan_xyz, int64_t n_scan, int32_t* d_offsets,
                                     int32_t* d_out_idx, int64_t out_capacity, int32_t* d_total, void* d_scratch,
                                     size_t scratch_bytes, void* stream_) {
  if (!bm || (!d_scan_xyz && n_scan > 0) || n_scan < 0 || n_scan > 0x7ffffffe || !d_out_idx || out_capacity < 0 ||
      !d_total || !d_scratch || ((uintptr_t)d_scratch & 255))
    return SPS_ERR_BAD_ARG;
  if (scratch_bytes < sps_ball_query_scratch_bytes(n_scan)) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream_;
  const size_t half = sps_ball_query_scratch_bytes(n_scan) / 2;
  int32_t* counts = (int32_t*)d_scratch;
  int32_t* offsets = d_offsets ? d_offsets : (int32_t*)((char*)d_scratch + half);
  const BallGrid g = grid_of_map(bm);
  const int grid = grid_of(n_scan > 0 ? n_scan : 1, 128);
  k_ball_query<false><<<grid, 128, 0, st>>>(d_scan_xyz, 3, (int)n_scan, g, counts, nullptr, nullptr, 0);
  k_ball_scan<<<1, kBallBlock, 0, st>>>(counts, nullptr, (int)n_scan, offsets, d_total);
  k_ball_query<true><<<grid, 128, 0, st>>>(d_scan_xyz, 3, (int)n_scan, g, nullptr, offsets, d_out_idx, out_capacity);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

namespace sps {

// scratch of the batched query: scalars (scan ticket, hit total, forward row count) | hit ranks [n] | chunk sums
struct BatchCarve {
  uint32_t* ticket; int32_t* total; int32_t* n_fwd; int32_t* rank; int32_t* block_sums; size_t bytes;
};
static BatchCarve carve_batch(void* base, int64_t n) {
  BatchCarve c;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t b) { off = (off + 255) & ~size_t(255); char* r = p ? p + off : nullptr; off += b; return r; };
  int32_t* scalars = (int32_t*)take(64 * 4);
  c.ticket = (uint32_t*)scalars; c.total = scalars + 1; c.n_fwd = scalars + 2;
  c.rank = (int32_t*)take((size_t)n * 4);
  c.block_sums = (int32_t*)take((size_t)(n / kScanBlock + 2) * 4);
  c.bytes = (off + 255) & ~size_t(255);
  return c;
}

// arguments shared by sps_radius_batch and sps_predict_radius_batch; fills `bo` and n_total
static int check_batch_args(const sps_ballmap* bm, const float* d_scans, int64_t ld, const int64_t* h_offsets, int batch,
                            const float* d_rows, int64_t row_capacity, const int32_t* d_row_offsets,
                            const int32_t* d_n_rows, const void* d_scratch, size_t scratch_bytes, BatchOffsets& bo,
                            int64_t& n_total) {
  if (!bm || !h_offsets || !d_rows || !d_row_offsets || !d_n_rows || !d_scratch || ((uintptr_t)d_scratch & 255) ||
      ld < 4 || batch < 1 || batch > kMaxBatch || row_capacity < 0 || h_offsets[0] != 0)
    return SPS_ERR_BAD_ARG;
  for (int b = 0; b < batch; ++b)
    if (h_offsets[b + 1] < h_offsets[b]) return SPS_ERR_BAD_ARG;
  n_total = h_offsets[batch];
  if (n_total > 0x7ffffffe || (!d_scans && n_total > 0)) return SPS_ERR_BAD_ARG;
  if (scratch_bytes < carve_batch(nullptr, n_total > 0 ? n_total : 1).bytes) return SPS_ERR_CAPACITY;
  bo.batch = batch;
  for (int b = 0; b <= batch; ++b) bo.off[b] = (int32_t)h_offsets[b];
  return SPS_OK;
}

static int radius_batch_launch(const sps_ballmap* bm, const float* d_scans, int64_t ld, const BatchOffsets& bo, int n,
                               float* d_rows, int64_t row_capacity, int32_t* d_row_offsets, int32_t* d_n_rows,
                               const BatchCarve& c, int32_t* status, cudaStream_t st) {
  const BallGrid g = grid_of_map(bm);
  SPS_CUDA_CHECK(cudaMemsetAsync(c.ticket, 0, 64 * 4, st));
  k_radius_batch_count<<<cdiv(n > 0 ? n : 1, kScanBlock), kScanBlock, 0, st>>>(d_scans, ld, n, g, c.rank, c.block_sums,
                                                                                c.ticket, c.total);
  k_radius_batch_write<<<grid_of(n > 0 ? n : 1, 256), 256, 0, st>>>(d_scans, ld, n, bo, g, c.rank, c.block_sums, c.total,
                                                                   d_rows, row_capacity, d_row_offsets, d_n_rows,
                                                                   c.n_fwd, status);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

int forward_impl(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n_upper, const int32_t* d_n,
                 int64_t ld_points, float voxel_size, float* d_scores, int64_t n_scores, cudaStream_t st);

}  // namespace sps

extern "C" size_t sps_radius_batch_scratch_bytes(int64_t n_scan_total, int batch) {
  (void)batch;   // the per-scan offsets travel as kernel arguments
  return carve_batch(nullptr, n_scan_total > 0 ? n_scan_total : 1).bytes;
}

extern "C" int sps_radius_batch(const sps_ballmap* bm, const float* d_scans, int64_t ld, const int64_t* h_offsets, int batch,
                                float* d_rows, int64_t row_capacity, int32_t* d_row_offsets, int32_t* d_n_rows,
                                void* d_scratch, size_t scratch_bytes, void* stream) {
  BatchOffsets bo;
  int64_t n = 0;
  int rc = check_batch_args(bm, d_scans, ld, h_offsets, batch, d_rows, row_capacity, d_row_offsets, d_n_rows, d_scratch,
                            scratch_bytes, bo, n);
  if (rc != SPS_OK) return rc;
  return radius_batch_launch(bm, d_scans, ld, bo, (int)n, d_rows, row_capacity, d_row_offsets, d_n_rows,
                             carve_batch(d_scratch, n > 0 ? n : 1), nullptr, (cudaStream_t)stream);
}

extern "C" int sps_predict_radius_batch(sps_ctx* ctx, const sps_net* net, const sps_ballmap* bm, const float* d_scans,
                                        int64_t ld, const int64_t* h_offsets, int batch, float* d_rows,
                                        int64_t row_capacity, int32_t* d_row_offsets, int32_t* d_n_rows, void* d_scratch,
                                        size_t scratch_bytes, float voxel_size, float eps, float* d_scan_scores,
                                        int64_t* d_counts, double* d_sums, void* stream) {
  if (!ctx || !net || !d_scan_scores || !d_counts || !d_sums || !(voxel_size > 0.f)) return SPS_ERR_BAD_ARG;
  BatchOffsets bo;
  int64_t n = 0;
  int rc = check_batch_args(bm, d_scans, ld, h_offsets, batch, d_rows, row_capacity, d_row_offsets, d_n_rows, d_scratch,
                            scratch_bytes, bo, n);
  if (rc != SPS_OK) return rc;
  if (row_capacity > ctx->max_points) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream;
  const BatchCarve c = carve_batch(d_scratch, n > 0 ? n : 1);
  rc = radius_batch_launch(bm, d_scans, ld, bo, (int)n, d_rows, row_capacity, d_row_offsets, d_n_rows, c, ctx->status, st);
  if (rc != SPS_OK) return rc;
  // SPSModel.forward on the rows (models.py:20-30): the launches are sized by the capacity, the row count stays on the
  // device (0 when the rows did not fit); scores of every row land in the context's score buffer
  rc = forward_impl(ctx, net, d_rows, row_capacity, c.n_fwd, 6, voxel_size, ctx->scores, row_capacity, st);
  if (rc != SPS_OK) return rc;
  SPS_CUDA_CHECK(cudaMemsetAsync(d_counts, 0, (size_t)batch * 4 * sizeof(int64_t), st));
  SPS_CUDA_CHECK(cudaMemsetAsync(d_sums, 0, (size_t)batch * 5 * sizeof(double), st));
  if (n > 0) {
    const int per_block = 256 * kPartialsSpan;   // points per block: 8 warps x kPartialsSpan x 32
    k_radius_partials<<<cdiv(n, per_block), 256, 0, st>>>(d_scans, ld, (int)n, bo, c.rank, c.block_sums, c.total, d_n_rows,
                                                         c.n_fwd, ctx->scores, eps, d_scan_scores,
                                                         reinterpret_cast<unsigned long long*>(d_counts), d_sums);
    SPS_CUDA_CHECK(cudaGetLastError());
  }
  return SPS_OK;
}
