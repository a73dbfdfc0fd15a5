// Coordinate hashing: voxelisation (a1/a2), strided coordinate maps (a4) and kernel maps.
//
// One primitive does all the set work: unique_by_hash() = open-addressing insert of 64-bit
// voxel keys + "first occurrence" ranking (atomicMin of the input index per slot, then a
// block scan with a last-block-done carry) so that the voxel order is deterministic and equal
// to ME's CPU insert order.  Level 0 hashes the quantised points, level L+1 hashes the
// level-L keys with the low spatial bits masked off (floor to the tensor stride).
// All sizes below level 0 live on the device; launches are sized by the host upper bound and
// surplus blocks exit on the device count, so a whole forward needs no host synchronisation.
#include <limits.h>
#include <utility>
#include "ctx.h"
#include "partials.cuh"
#include "profile.h"
#include "rosio.cuh"
#include "scan.cuh"

namespace sps {

constexpr uint32_t kInvalidSlot = 0xFFFFFFFFu;

__global__ void k_set_i32(int32_t* p, int32_t v) { *p = v; }

constexpr int kRankChunks = 4;    // chunks of kScanBlock rows a block of k_first_rank scans
constexpr int kSliceBatch = 16;   // kernel-map entries a thread of k_tile_masks_perm reads before it stores them
constexpr int kInsertBatch = 4;   // rows a thread of the level-0 insert kernel keeps in flight

// First kernel of a level: empties the open-addressing table for `n` keys and, for a strided level, presets the
// child table of the level being built to "absent" for every column a coarse row can take (coarse count <= fine count).
// n comes from the device (`n_ptr`) or, at level 0, from the host (`n_host` >= 0, also published to `n_dev`).
__global__ void k_level_begin(Slot* __restrict__ tab, const int32_t* __restrict__ n_ptr, int32_t n_host, int32_t* n_dev,
                              int32_t* __restrict__ child, int64_t ld, int32_t* tplanes = nullptr, int32_t* cls = nullptr) {
  const int n = n_host >= 0 ? n_host : *n_ptr;
  if (n_dev && blockIdx.x == 0 && threadIdx.x == 0) *n_dev = n;
  if (tplanes && blockIdx.x == 0 && threadIdx.x == 0) *tplanes = 0;
  if (cls && blockIdx.x == 0 && threadIdx.x < 16) cls[threadIdx.x] = 0;     // child-class counters of the fine level
  const uint32_t cap = table_capacity(n);
  const int4 empty = make_int4(-1, -1, -1, INT_MAX);
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += stride) reinterpret_cast<int4*>(tab)[i] = empty;
  if (child) {   // (no division per element: this loop was 79 % issue-bound with idx / n)
    for (uint32_t c = blockIdx.x * blockDim.x + threadIdx.x; c < (uint32_t)n; c += stride) {
#pragma unroll
      for (int r = 0; r < 8; ++r) child[r * ld + c] = -1;
    }
  }
}

// a1 + a2: fp32 IEEE division by the voxel size (src/sps/models/models.py:21), floor
// (ME TensorField.sparse()), key packing, hash insert.
__global__ void k_insert_points(const float* __restrict__ pts, int64_t ld, const int32_t* __restrict__ n_ptr,
                                float vs, Slot* tab, uint32_t* __restrict__ slot_of, int32_t* status, int32_t* tplanes) {
  const int n = *n_ptr;
  const uint32_t mask = table_capacity(n) - 1;
  uint32_t seen = 0;   // time planes this thread met (bit t)
  // kInsertBatch rows per thread at a time: their home slots are read back to back, so the L2 / DRAM round trips of the
  // random accesses overlap (ncu: 53 of 57 stall cycles per issue were long-scoreboard waits with one row at a time), and
  // the atomics are only issued when they can change something: 57 % of the rows find their voxel already in the table
  const int stride = gridDim.x * blockDim.x;
  for (int i0 = blockIdx.x * blockDim.x + threadIdx.x; i0 < n; i0 += kInsertBatch * stride) {
    unsigned long long key[kInsertBatch];
    uint32_t sl[kInsertBatch];
    int4 raw[kInsertBatch];
    bool ok[kInsertBatch];
#pragma unroll
    for (int u = 0; u < kInsertBatch; ++u) {
      const int i = i0 + u * stride;
      ok[u] = false;
      if (i >= n) continue;
      const float* p = pts + (int64_t)i * ld;
      const float fb = floorf(__fdiv_rn(p[0], 1.0f));
      const float fx = floorf(__fdiv_rn(p[1], vs));
      const float fy = floorf(__fdiv_rn(p[2], vs));
      const float fz = floorf(__fdiv_rn(p[3], vs));
      const float ft = floorf(__fdiv_rn(p[4], 1.0f));
      ok[u] = fb >= 0.f && fb < 255.f && fx >= -(float)kXBias && fx < (float)kXBias &&
              fy >= -(float)kXBias && fy < (float)kXBias && fz >= -(float)kZBias &&
              fz < (float)kZBias && ft >= 0.f && ft < 16.f;
      if (!ok[u]) {  // also catches NaN
        atomicOr(status, kStatusRange);
        slot_of[i] = kInvalidSlot;
        continue;
      }
      key[u] = pack_key((int)fb, (int)fx, (int)fy, (int)fz, (int)ft);
      sl[u] = hash_key(key[u]) & mask;
      raw[u] = __ldcg(reinterpret_cast<const int4*>(tab + sl[u]));
      seen |= 1u << (int)ft;
    }
#pragma unroll
    for (int u = 0; u < kInsertBatch; ++u)
      if (ok[u]) slot_of[i0 + u * stride] = table_insert_first(tab, mask, key[u], i0 + u * stride, sl[u], raw[u]);
  }
  // which time planes hold voxels at all (SPS: t in {0, 1}): the kernel-map pass does not probe the others
  seen = __reduce_or_sync(0xffffffffu, seen);
  if ((threadIdx.x & 31) == 0 && seen) atomicOr(tplanes, (int)seen);
}

// a4: ME stride map -- floor the spatial coordinates to the new tensor stride 2^log2m.
__global__ void k_insert_coarse(const unsigned long long* __restrict__ fine, const int32_t* __restrict__ n_ptr,
                                int log2m, Slot* tab, uint32_t* __restrict__ slot_of) {
  const int n = *n_ptr;
  const uint32_t mask = table_capacity(n) - 1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = table_insert(tab, mask, coarsen_key(fine[i], log2m));
    atomicMin(&tab[s].first, i);
    slot_of[i] = s;
  }
}

// flag = "this input is the first occurrence of its voxel" (optionally: "... and the voxel is
// also present in `filter`", the map/scan intersection of util.prune).
__global__ void __launch_bounds__(kScanBlock)
k_first_rank(Slot* tab, const uint32_t* __restrict__ slot_of, const int32_t* __restrict__ n_ptr,
             int32_t* __restrict__ rank, int32_t* block_sums, uint32_t* ticket, int32_t* count_out,
             const Slot* __restrict__ filter, uint32_t filter_mask, int32_t* first_count) {
  const int n = *n_ptr;
  const int nb = max(1, (n + kScanBlock - 1) / kScanBlock);          // chunks of kScanBlock inputs
  const int nblocks = (nb + kRankChunks - 1) / kRankChunks;          // blocks that take part (kRankChunks chunks each)
  if ((int)blockIdx.x >= nblocks) return;
  // A block scans kRankChunks consecutive chunks: the random slot reads behind all its flags are issued first (the kernel
  // waits on exactly those), and the grid takes a quarter of the tickets (one same-address atomic per block).
  int flag[kRankChunks];
  uint32_t s[kRankChunks];
#pragma unroll
  for (int r = 0; r < kRankChunks; ++r) {
    const int i = (blockIdx.x * kRankChunks + r) * kScanBlock + threadIdx.x;
    s[r] = i < n ? slot_of[i] : kInvalidSlot;
  }
#pragma unroll
  for (int r = 0; r < kRankChunks; ++r) {
    const int i = (blockIdx.x * kRankChunks + r) * kScanBlock + threadIdx.x;
    flag[r] = (s[r] != kInvalidSlot) && (tab[s[r]].first == i);
  }
#pragma unroll
  for (int r = 0; r < kRankChunks; ++r) {
    const int chunk = blockIdx.x * kRankChunks + r;
    if (chunk >= nb) break;                                           // block-uniform
    const int i = chunk * kScanBlock + threadIdx.x;
    if (filter) {
      const unsigned ballot = __ballot_sync(0xffffffffu, flag[r]);
      if (first_count && (threadIdx.x & 31) == 0 && ballot) atomicAdd(first_count, __popc(ballot));
      if (flag[r]) flag[r] = table_find(filter, filter_mask, tab[s[r]].key) >= 0;
    }
    const int excl = scan_chunk(flag[r], i, n, chunk, rank, block_sums);
    // the first occurrence leaves its chunk-local rank in the slot: whoever maps an input to its voxel row later
    // reads ONE 16-byte slot (key, local rank, first index) instead of chasing slot -> first -> rank[first]
    if (flag[r] && !filter) tab[s[r]].val = excl;
  }
  scan_finish(nb, nblocks, block_sums, ticket, count_out);
}

// Level 0: inverse mapping point -> voxel row; the first occurrence publishes the voxel.
__global__ void k_assign_points(Slot* tab, const uint32_t* __restrict__ slot_of, const int32_t* __restrict__ n_ptr,
                                const int32_t* __restrict__ rank, const int32_t* __restrict__ block_sums,
                                unsigned long long* __restrict__ ukeys, int32_t* __restrict__ inv) {
  const int n = *n_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = slot_of[i];
    if (s == kInvalidSlot) { inv[i] = -1; continue; }
    const int4 raw = *reinterpret_cast<const int4*>(tab + s);   // key | block-local rank | first input
    const int f = raw.w;
    const int id = raw.z + block_sums[f / kScanBlock];
    inv[i] = id;
    if (f == i) ukeys[id] = ((unsigned long long)(unsigned)raw.y << 32) | (unsigned)raw.x;
  }
}

// Level L+1: parent row and 2x2x2x1 offset index of every fine voxel (the stride-2 kernel map
// and, swapped, the transposed-conv map: minkunet.py:64-70,107-113), plus the child table.
__global__ void k_assign_coarse(Slot* tab, const uint32_t* __restrict__ slot_of, const int32_t* __restrict__ n_ptr,
                                const int32_t* __restrict__ rank, const int32_t* __restrict__ block_sums,
                                const unsigned long long* __restrict__ fine, int log2s,
                                unsigned long long* __restrict__ ukeys, int32_t* __restrict__ parent,
                                int32_t* __restrict__ child, int64_t ld, int32_t* __restrict__ cls) {
  __shared__ int s_cls[8];
  if (threadIdx.x < 8) s_cls[threadIdx.x] = 0;
  __syncthreads();
  const int n = *n_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = slot_of[i];
    const int4 raw = *reinterpret_cast<const int4*>(tab + s);   // key | block-local rank | first input
    const int f = raw.w;
    const int id = raw.z + block_sums[f / kScanBlock];
    const int k = child_index(fine[i], log2s);
    atomicAdd(&s_cls[k], 1);                                    // rows per child class (order of the transposed conv)
    parent[i] = id * 8 + k;
    child[(int64_t)k * ld + id] = i;
    // (the transposed convolution reads `parent` itself: SPS_CONV_MAP_PARENT -- no dense [8][ld] up-map is written)
    if (f == i) ukeys[id] = ((unsigned long long)(unsigned)raw.y << 32) | (unsigned)raw.x;
  }
  __syncthreads();
  if (threadIdx.x < 8 && s_cls[threadIdx.x]) atomicAdd(cls + threadIdx.x, s_cls[threadIdx.x]);
}

// Processing order of the transposed convolutions (minkunet.py:107-147): a fine row has exactly ONE input row (its parent)
// and one of eight weight matrices (its child class k), so in physical order every 128-row tile walks all eight offsets
// with one slot in eight filled.  Grouped by class a tile walks one offset (two where a class ends).  The order inside a
// class is whatever the atomics give: every output row is computed on its own, so results do not depend on it.
struct UpOrderArgs {
  const int32_t* parent[SPS_NUM_LEVELS];
  int32_t* perm[SPS_NUM_LEVELS];
  uint32_t* masks[SPS_NUM_LEVELS];
  const int32_t* counts;
  int32_t* cls;           // [4][16]: class counts, cursors
};
__global__ void __launch_bounds__(256)
k_up_order(const UpOrderArgs A) {
  const int L = blockIdx.y;
  const int n = A.counts[L];
  int32_t* cls = A.cls + 16 * L;
  __shared__ int s_base[9], s_cnt[8], s_cur[8];
  if (threadIdx.x == 0) {
    int run = 0;
    for (int k = 0; k < 8; ++k) { s_base[k] = run; run += cls[k]; }
    s_base[8] = run;
  }
  if (threadIdx.x < 8) s_cnt[threadIdx.x] = 0;
  __syncthreads();
  // each block owns one contiguous chunk of rows: count its classes, take its eight ranges with ONE global atomic per
  // class (a cursor per row, even warp-aggregated, serialises on eight addresses), then scatter
  const int lane = threadIdx.x & 31;
  const int chunk = ((n + (int)gridDim.x - 1) / (int)gridDim.x + 31) & ~31;
  const int r0 = blockIdx.x * chunk, r1 = min(n, r0 + chunk);
  const int32_t* __restrict__ parent = A.parent[L];
  for (int i = r0 + threadIdx.x; i < r1; i += blockDim.x) atomicAdd(&s_cnt[__ldg(parent + i) & 7], 1);
  __syncthreads();
  if (threadIdx.x < 8) s_cur[threadIdx.x] = s_base[threadIdx.x] + (s_cnt[threadIdx.x] ? atomicAdd(cls + 8 + threadIdx.x, s_cnt[threadIdx.x]) : 0);
  __syncthreads();
  for (int i0 = r0 + (threadIdx.x & ~31); i0 < r1; i0 += blockDim.x) {
    const int i = i0 + lane;
    const int k = i < r1 ? (__ldg(parent + i) & 7) : 8 + lane;          // dead lanes match nobody
    const unsigned peers = __match_any_sync(0xffffffffu, k);
    const int leader = __ffs(peers) - 1;
    int pos = 0;
    if (lane == leader && i < r1) pos = atomicAdd(&s_cur[k], __popc(peers));
    pos = __shfl_sync(0xffffffffu, pos, leader);
    if (i < r1) A.perm[L][pos + __popc(peers & ((1u << lane) - 1u))] = i;
  }
  // tile masks in this order: the classes whose row range meets the tile
  const int ntiles = (n + 127) / 128;
  for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < ntiles; t += gridDim.x * blockDim.x) {
    uint32_t m = 0;
    for (int k = 0; k < 8; ++k)
      if (s_base[k] < 128 * (t + 1) && s_base[k + 1] > 128 * t) m |= 1u << k;
    reinterpret_cast<uint4*>(A.masks[L])[t] = make_uint4(m, 0u, 0u, 0u);
  }
}


// ---- block tables: 4x4x4-cell blocks of a level's lattice -> 64 voxel rows each ----------------------
// The kernel-map probes of one voxel fall into at most 8 such blocks per time plane, and
// neighbouring voxels share them, so a probe costs a (mostly L1/L2-resident) 4-byte read inside a
// 256-byte block instead of one random 32-byte sector of a per-voxel hash table.
// The tables of ALL levels are built by the same three launches (blockIdx.y = level): the coarse levels hold a few
// thousand voxels each and were pure launch latency as separate kernels.
// Levels 0..2 build no block hash of their own: the 4x4x4 blocks of level L are the voxels of level L + 2, and the stride
// chain's hash of those voxels answers "block key -> block row".  That hash was built from, and sized for, the rows of
// level L + 1.
__host__ __device__ constexpr bool blocks_are_voxels(int L) { return L + 2 < SPS_NUM_LEVELS; }
// the level whose row count sized the block hash of level L
__host__ __device__ constexpr int btab_sized_for(int L) { return blocks_are_voxels(L) ? L + 1 : L; }
struct LevelTabs {
  const unsigned long long* keys[SPS_NUM_LEVELS];
  const int32_t* counts;                 // [SPS_NUM_LEVELS] device voxel counts
  Slot* btab[SPS_NUM_LEVELS];            // block key -> block id (own hash), or the voxel hash of level L + 2 (blocks_are_voxels)
  const int32_t* parent[SPS_NUM_LEVELS]; // fine row -> parent * 8 + k (levels 0..3)
  int32_t* cells[SPS_NUM_LEVELS];        // [blocks][64] voxel rows
  unsigned long long* occ[SPS_NUM_LEVELS];   // [blocks] 64-bit occupancy words
  int32_t* nblocks;                      // [SPS_NUM_LEVELS] block counters
  const int32_t* tplanes;                // bit t: some voxel of the input lies in time plane t
};

// Clears the block tables and zeroes the small scratch arrays the map-building pass accumulates into: the
// physical-order tile masks (atomicOr targets) and the shape sort's digit histograms, tile tickets and look-back words.
struct ScratchZero {
  uint32_t* tmask3[SPS_NUM_LEVELS];   // nullptr: level keeps no physical-order tile masks
  uint32_t* sort_hist;                // [4][256] + 4 tile tickets (1028 words), or nullptr: no shape sort this forward
  uint32_t* sort_status;              // [tiles][4][256]
};
// keys of the shape sort: the voxels of all levels (a rolled loop: unrolled, it costs the sort passes 12 registers)
__device__ __forceinline__ int sort_total(const int32_t* counts) {
  int t = 0;
#pragma unroll 1
  for (int j = 0; j < SPS_NUM_LEVELS; ++j) t += counts[j];
  return t;
}
__global__ void k_blocks_begin(const LevelTabs T, const ScratchZero z) {
  const int L = blockIdx.y;
  const int n = T.counts[L];
  const uint32_t stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  if (blocks_are_voxels(L)) {
    // the blocks are the voxels of level L + 2 and their hash was built by the stride chain: its slots still hold the
    // scan's block-local ranks, so every voxel writes its ROW into its slot (one probe each) -- from here on the table maps
    // a block key to the block id.  Only the occupancy words start from zero: every reader of the cells goes through them.
    const int nb = T.counts[L + 2];
    const uint32_t mask = table_capacity(T.counts[btab_sized_for(L)]) - 1;
    const unsigned long long* __restrict__ bkeys = T.keys[L + 2];
    Slot* tab = T.btab[L];
    for (uint32_t i = t0; i < (uint32_t)nb; i += stride) {
      T.occ[L][i] = 0ull;
      const unsigned long long key = bkeys[i];
      uint32_t s = hash_key(key) & mask;
      while (tab[s].key != key) s = (s + 1) & mask;
      tab[s].val = (int)i;
    }
    if (t0 == 0) T.nblocks[L] = nb;
  } else {
    const uint32_t cap = table_capacity(n);
    const int4 empty = make_int4(-1, -1, -1, INT_MAX);
    for (uint32_t i = t0; i < cap; i += stride) reinterpret_cast<int4*>(T.btab[L])[i] = empty;
    if (t0 == 0) T.nblocks[L] = 0;
  }
  if (z.tmask3[L]) {
    const uint32_t w = 4u * (uint32_t)(n / 128 + 1);
    for (uint32_t i = t0; i < w; i += stride) z.tmask3[L][i] = 0u;
  }
  if (L == 0 && z.sort_hist) {
    for (uint32_t i = t0; i < 1028u; i += stride) z.sort_hist[i] = 0u;
    const int64_t w = (int64_t)((sort_total(T.counts) + 1023) / 1024) * 1024;
    for (int64_t i = t0; i < w; i += stride) z.sort_status[i] = 0u;
  }
}

__device__ __forceinline__ int cell_local(unsigned long long key, int L) {
  return ((int)(key >> (kXShift + L)) & 3) + 4 * ((int)(key >> (kYShift + L)) & 3) + 16 * ((int)(key >> (kZShift + L)) & 3);
}

__global__ void __launch_bounds__(256)
k_block_insert(const LevelTabs T) {
  // Block ids come from ONE counter per level.  ncu's source view put 75 % of the stall samples of the first version on
  // the result of that same-address atomicAdd (the compiler's warp aggregation still leaves ~10^5 of them at level 0), so
  // the winners of a whole CTA are ranked in shared memory first and one thread takes the CTA's id range with a single
  // global atomic.  The winner of a block also presets the block's 64 cells and its occupancy word.
  __shared__ int s_cnt, s_base;
  const int L = blockIdx.y;
  if (blocks_are_voxels(L)) return;      // blocks = voxels of level L + 2: nothing to insert
  const int n = T.counts[L];
  const uint32_t mask = table_capacity(n) - 1;
  Slot* tab = T.btab[L];
  const unsigned long long* keys = T.keys[L];
  if (threadIdx.x == 0) s_cnt = 0;
  __syncthreads();
  for (int base = blockIdx.x * blockDim.x; base < n; base += gridDim.x * blockDim.x) {   // CTA-uniform trip count
    const int i = base + threadIdx.x;
    uint32_t s = 0;
    int local = -1;
    if (i < n) {
      const unsigned long long bkey = coarsen_key(keys[i], L + 2);
      s = hash_key(bkey) & mask;
      while (true) {
        const unsigned long long prev = atomicCAS(&tab[s].key, kEmptyKey, bkey);
        if (prev == kEmptyKey) { local = atomicAdd(&s_cnt, 1); break; }
        if (prev == bkey) break;
        s = (s + 1) & mask;
      }
    }
    __syncthreads();
    if (threadIdx.x == 0) { s_base = s_cnt ? atomicAdd(T.nblocks + L, s_cnt) : 0; s_cnt = 0; }
    __syncthreads();
    if (local >= 0) {
      const int id = s_base + local;
      tab[s].val = id;
      int4* c4 = reinterpret_cast<int4*>(T.cells[L] + (int64_t)id * 64);
      const int4 v = make_int4(-1, -1, -1, -1);
#pragma unroll
      for (int j = 0; j < 16; ++j) c4[j] = v;
      T.occ[L][id] = 0ull;
    }
  }
}

__global__ void k_cells_fill(const LevelTabs T) {
  const int L = blockIdx.y;
  const int n = T.counts[L];
  const uint32_t mask = table_capacity(n) - 1;
  const unsigned long long* keys = T.keys[L];
  const bool by_parent = blocks_are_voxels(L);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned long long key = keys[i];
    // block id = the voxel's grandparent row (two reads of the parent arrays), or a lookup in the level's block hash
    const int id = by_parent ? (__ldg(T.parent[L + 1] + (__ldg(T.parent[L] + i) >> 3)) >> 3)
                             : table_find(T.btab[L], mask, coarsen_key(key, L + 2));
    const int l = cell_local(key, L);
    T.cells[L][(int64_t)id * 64 + l] = i;
    atomicOr(T.occ[L] + id, 1ull << l);     // 64-bit occupancy word per block: presence tests without the index read
  }
}

// Kernel map of the 5x5x5x1 kernel on level 0 through the block table: thread o resolves the 125 spatial neighbours of
// voxel o in its own time plane; k = (dx+2) + 5 ((dy+2) + 5 (dz+2)) (ME order), nbr[k][o] coalesced over o.
__global__ void __launch_bounds__(256)
k_kernel_map_blk5(const unsigned long long* __restrict__ keys, const int32_t* __restrict__ n_ptr,
                  const Slot* __restrict__ tab, const int32_t* __restrict__ cap_n, const int32_t* __restrict__ cells,
                  const unsigned long long* __restrict__ occ, int32_t* __restrict__ nbr, int64_t ld) {
  const int n = *n_ptr;
  if (n == 0) return;
  const uint32_t mask = table_capacity(*cap_n) - 1;
  const int xlim = 1 << kXBits, zlim = 1 << kZBits;
  const int lane = threadIdx.x & 31;
  // warp-aligned rows (dead lanes past n ride along): ptxas spills 16 bytes for a plain grid-stride loop over o
  for (int o0 = (blockIdx.x * blockDim.x + threadIdx.x) & ~31; o0 < n; o0 += gridDim.x * blockDim.x) {
    const int o = o0 + lane;
    const bool live = o < n;
    const unsigned long long key = live ? keys[o] : 0ull;
    int32_t* out = nbr + o;
    const int cx = (int)((key >> kXShift) & ((1u << kXBits) - 1));
    const int cy = (int)((key >> kYShift) & ((1u << kYBits) - 1));
    const int cz = (int)((key >> kZShift) & ((1u << kZBits) - 1));
    const unsigned long long bt = key & ((0xFFull << kBShift) | ((1ull << kTBits) - 1));
    unsigned long long cached_key = kEmptyKey, cached_occ = 0ull;
    const int32_t* cached = nullptr;
#pragma unroll 1
    for (int dz = -2; dz <= 2; ++dz) {
      const int nz = cz + dz;
      const bool zok = (unsigned)nz < (unsigned)zlim;
#pragma unroll
      for (int dy = -2; dy <= 2; ++dy) {   // (dy, dx) unrolled: up to 25 independent probes in flight per thread
        const int ny = cy + dy;
        const bool yok = zok && (unsigned)ny < (unsigned)xlim;
        const unsigned long long byz = bt | ((unsigned long long)(unsigned)((ny >> 2) << 2) << kYShift) |
                                       ((unsigned long long)(unsigned)((nz >> 2) << 2) << kZShift);
        const int lyz = 4 * (ny & 3) + 16 * (nz & 3);
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
          const int nx = cx + dx;
          int res = -1;
          if (yok && (unsigned)nx < (unsigned)xlim) {
            const unsigned long long bkey = byz | ((unsigned long long)(unsigned)((nx >> 2) << 2) << kXShift);
            if (bkey != cached_key) {
              cached_key = bkey;
              const int id = table_find(tab, mask, bkey);
              cached = cells + (int64_t)(id >= 0 ? id : 0) * 64;
              cached_occ = id >= 0 ? __ldg(occ + id) : 0ull;
            }
            const int l = lyz + (nx & 3);
            if ((cached_occ >> l) & 1ull) res = __ldg(cached + l);
          }
          if (live) out[(int64_t)((dx + 2) + 5 * ((dy + 2) + 5 * (dz + 2))) * ld] = res;
        }
      }
    }
  }
}

// The 3x3x3 case, restructured around the probes: a voxel's 27 spatial neighbours live in its own 4x4x4 block
// and, per axis, in at most ONE adjacent block (when the voxel sits on that face), i.e. in 1, 2, 4 or 8 blocks
// (3.4 on average).  Each thread first resolves those blocks (independent hash probes, all in flight), parks
// block id + occupancy word in shared memory, then answers the 27 lookups with a bit test and, for present
// neighbours only, one 4-byte read.  (Probing like the 5x5x5 kernel above, again whenever the block changes along x, took
// ~13 probes per thread; this was the dominant kernel after the convolutions were sped up.)
struct KmapOut {
  int32_t* nbr[SPS_NUM_LEVELS];           // [81][ld] per level
  uint32_t* tile_masks[SPS_NUM_LEVELS];   // physical-order tile masks, or nullptr (shape-sorted level of the fused forward)
  uint32_t* vmask[SPS_NUM_LEVELS];        // [ld][4] per-voxel 27-bit presence words of the three time planes (+ pad): one 16-byte line
  int64_t ld;
  int dense;                              // absent entries (-1) are stored too
  // shape sort fused in (nullptr: no sort this forward): the voxel's sort key, its row number and the digit histograms of
  // the four radix passes leave this kernel, so the presence words are not read back by a separate key pass
  uint32_t* sort_keys; int32_t* sort_vals; uint32_t* sort_hist;
};
// All levels in one launch: blockIdx.z = level; a thread walks the three time planes of the kernel.
// (capping this kernel at 32 registers to fit more blocks beside another lane's convolution CTA made it 1.5x slower
// and the step 18 % slower: profiles/r2_experiments.md)
__device__ __forceinline__ uint32_t shape_bits(uint32_t pat);
__global__ void __launch_bounds__(256, 6)
k_kernel_map_blk3(const LevelTabs T, const KmapOut O) {
  constexpr int KT = 3;   // time planes of the kernel
  __shared__ int sId[8][256];
  __shared__ unsigned long long sOcc[8][256];
  const int L = blockIdx.z;
  const int n = T.counts[L];
  if (n == 0) return;
  const unsigned long long* __restrict__ keys = T.keys[L];
  const Slot* __restrict__ tab = T.btab[L];
  const int32_t* __restrict__ cells = T.cells[L];
  const unsigned long long* __restrict__ occ = T.occ[L];
  int32_t* __restrict__ nbr = O.nbr[L];
  uint32_t* __restrict__ tile_masks = O.tile_masks[L];
  uint32_t* __restrict__ vmask = O.vmask[L];
  const int64_t ld = O.ld;
  const int dense = O.dense;
  const uint32_t mask = table_capacity(T.counts[btab_sized_for(L)]) - 1;
  const int xlim = 1 << (kXBits - L), zlim = 1 << (kZBits - L);
  const int tid = threadIdx.x, lane = tid & 31;
  const uint32_t planes = (uint32_t)*T.tplanes;
  const bool sorting = O.sort_keys != nullptr;
  __shared__ uint32_t s_hist[4][256];
  int sort_off = 0;
  if (sorting) {
    for (int i = tid; i < 1024; i += blockDim.x) (&s_hist[0][0])[i] = 0u;
    for (int q = 0; q < L; ++q) sort_off += T.counts[q];
    __syncthreads();
  }
  for (int o0 = (blockIdx.x * blockDim.x + tid) & ~31; o0 < n; o0 += gridDim.x * blockDim.x) {
    const int o = o0 + lane;
    const bool live = o < n;
    const unsigned long long key = live ? keys[o] : 0ull;
    uint32_t por = 0u, pm0 = 0u, pm1 = 0u, pm2 = 0u;   // presence words of the planes and their OR
#pragma unroll 1
    for (int it = 0; it < KT; ++it) {             // time plane of the kernel: t + (it - KT/2)
    const int t2 = (int)(key & ((1u << kTBits) - 1)) + it - KT / 2;
    const bool pok = live && (unsigned)t2 < (1u << kTBits) && ((planes >> t2) & 1u);   // empty time planes are not probed
    int32_t* out = nbr + (int64_t)it * 27 * ld + o;
    if (!__any_sync(0xffffffffu, pok)) {
      // no row of this warp has the time plane (rows of one scan / one submap are contiguous, so a third of the warps end
      // here: the map rows have no t - 1 plane, the scan rows no t + 1 plane): nothing to probe, nothing present
      if (live) {
        if (dense) {
#pragma unroll
          for (int k3 = 0; k3 < 27; ++k3) out[(int64_t)k3 * ld] = -1;
        }
      }
      continue;
    }
    const int cx = (int)((key >> kXShift) & ((1u << kXBits) - 1)) >> L;
    const int cy = (int)((key >> kYShift) & ((1u << kYBits) - 1)) >> L;
    const int cz = (int)((key >> kZShift) & ((1u << kZBits) - 1)) >> L;
    const unsigned long long bt = (key & (0xFFull << kBShift)) | (unsigned long long)(unsigned)(pok ? t2 : 0);
    // which face of its block the voxel touches per axis: -1 / +1, or 0 (interior along that axis)
    const int sx = (cx & 3) == 0 ? -1 : ((cx & 3) == 3 ? 1 : 0);
    const int sy = (cy & 3) == 0 ? -1 : ((cy & 3) == 3 ? 1 : 0);
    const int sz = (cz & 3) == 0 ? -1 : ((cz & 3) == 3 ? 1 : 0);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int jx = j & 1, jy = (j >> 1) & 1, jz = j >> 2;
      const int bx = cx + (jx ? sx : 0), by = cy + (jy ? sy : 0), bz = cz + (jz ? sz : 0);   // a cell of block j
      const bool need = pok && (!jx || sx) && (!jy || sy) && (!jz || sz) && (unsigned)bx < (unsigned)xlim &&
                        (unsigned)by < (unsigned)xlim && (unsigned)bz < (unsigned)zlim;
      int id = -1;
      unsigned long long oc = 0ull;
      if (need) {
        const unsigned long long bkey = bt | ((unsigned long long)(unsigned)((bx >> 2) << (L + 2)) << kXShift) |
                                        ((unsigned long long)(unsigned)((by >> 2) << (L + 2)) << kYShift) |
                                        ((unsigned long long)(unsigned)((bz >> 2) << (L + 2)) << kZShift);
        id = table_find(tab, mask, bkey);
        if (id >= 0) oc = __ldg(occ + id);
      }
      sId[j][tid] = id;
      sOcc[j][tid] = oc;
    }
    uint32_t* tm = tile_masks ? tile_masks + 4 * (o0 >> 7) : nullptr;
    // Presence first, from the occupancy words alone: per (dz, dy) row the three x-neighbours are three adjacent bits of a
    // 6-bit line = [last cell of the -x block | the four cells of the own block's x-row | first cell of the +x block].
    uint32_t present = 0;   // bit k3: neighbour k3 of this time plane exists
    const int lx = cx & 3;
#pragma unroll
    for (int dz = -1; dz <= 1; ++dz) {
      const int jz = (sz != 0 && dz == sz) ? 4 : 0;
#pragma unroll
      for (int dy = -1; dy <= 1; ++dy) {
        const int jyz = jz + ((sy != 0 && dy == sy) ? 2 : 0);
        const int lyz = 4 * ((cy + dy) & 3) + 16 * ((cz + dz) & 3);
        const uint32_t rowA = (uint32_t)(sOcc[jyz][tid] >> lyz) & 15u;
        const uint32_t rowB = (uint32_t)(sOcc[jyz + 1][tid] >> lyz) & 15u;    // the x-adjacent block (all zero when sx == 0)
        const uint32_t line = (sx < 0 ? (rowB >> 3) : 0u) | (rowA << 1) | (sx > 0 ? ((rowB & 1u) << 5) : 0u);
        present |= ((line >> lx) & 7u) << (3 * ((dy + 1) + 3 * (dz + 1)));
      }
    }
    // dense = 0: only present entries are stored (87 % of the table is -1); allowed when every reader of this level's
    // table goes through the presence words `vmask` (the tile slices of a shape-sorted level)
    if (dense && live) {
#pragma unroll
      for (int k3 = 0; k3 < 27; ++k3) out[(int64_t)k3 * ld] = -1;
    }
    // then one index read and one store per PRESENT neighbour (5-12 of the 27)
    uint32_t todo = live ? present : 0u;
    while (todo) {
      const int k3 = __ffs(todo) - 1;
      todo &= todo - 1;
      const int dz = k3 / 9 - 1, dy = (k3 / 3) % 3 - 1, dx = k3 % 3 - 1;
      const int jj = ((sz != 0 && dz == sz) ? 4 : 0) + ((sy != 0 && dy == sy) ? 2 : 0) + ((sx != 0 && dx == sx) ? 1 : 0);
      const int l = ((cx + dx) & 3) + 4 * ((cy + dy) & 3) + 16 * ((cz + dz) & 3);
      out[(int64_t)k3 * ld] = __ldg(cells + (int64_t)sId[jj][tid] * 64 + l);
    }
    if (tm) {   // physical-order tile masks: the offsets any row of the warp has
      const uint32_t any = __reduce_or_sync(0xffffffffu, present);
      if (lane == 0 && any) {
        const int lo = it * 27, w0 = lo >> 5, sh = lo & 31;
        atomicOr(tm + w0, any << sh);
        if (sh + 27 > 32) atomicOr(tm + w0 + 1, any >> (32 - sh));
      }
    }
    por |= present;
    if (it == 0) pm0 = present;
    else if (it == 1) pm1 = present;
    else pm2 = present;
    }   // planes
    const uint32_t has_lo = pm0 ? 1u : 0u, has_hi = pm2 ? 1u : 0u;    // lowest / highest plane non-empty
    if (vmask && live) reinterpret_cast<uint4*>(vmask)[o] = make_uint4(pm0, pm1, pm2, 0u);
    if (sorting && live) {
      // sort key of the voxel: the Gray-code RANK of [has t+1][has t-1][27 spatial bits, OR over the planes] -- neighbouring
      // keys then differ in one offset instead of arbitrarily many in the low bits, so a tile that straddles two shapes walks
      // one offset more, not their whole difference (offsets walked per tile -3..4 %, tools/tile_stats.py)
      uint32_t g = shape_bits(por) | (has_lo << 27) | (has_hi << 28);
      g ^= g >> 1; g ^= g >> 2; g ^= g >> 4; g ^= g >> 8; g ^= g >> 16;
      const uint32_t skey = g | ((uint32_t)L << 29);
      O.sort_keys[sort_off + o] = skey;
      O.sort_vals[sort_off + o] = o;
#pragma unroll
      for (int p = 0; p < 4; ++p) atomicAdd(&s_hist[p][(skey >> (8 * p)) & 255u], 1u);
    }
  }
  if (sorting) {
    __syncthreads();
    for (int i = tid; i < 1024; i += blockDim.x) {
      const uint32_t c = (&s_hist[0][0])[i];
      if (c) atomicAdd(O.sort_hist + i, c);
    }
  }
}

// ---- pattern-sorted processing order for the 3x3x3x3 convolutions ---------------------------------
// Only 22-36 % of the (row, offset) slots of an output-stationary 128-row tile hold a neighbour, and a tile
// must walk every offset that ANY of its rows uses.  Rows with the same neighbourhood shape use the same
// offsets, so the convolutions walk the voxels in an order sorted by a 29-bit shape key
//   [has dt=+1 neighbours][has dt=-1 neighbours][27-bit spatial presence, OR over the time planes]
// (measured on the bench scan: offsets walked per tile 46-50 -> 26-28).  The physical voxel order is
// untouched: `perm` is only the order in which the conv kernels visit rows.
//
// All sorted levels are sorted TOGETHER: the level index sits above the shape key (31-bit keys), so one stable LSD
// radix sort (4 passes of 8 bits) orders every level at once and its last pass scatters straight into the per-level
// `perm` arrays.  Each pass is ONE kernel ("onesweep"): the digit histograms of all four passes are taken while the
// keys are produced, and a tile learns the number of equal digits in the tiles before it by decoupled look-back over
// per-tile status words (aggregate / inclusive-prefix flags in the top two bits).  Round 1 ran 13 launches per level.
struct SortArgs {
  int32_t* perm[SPS_NUM_LEVELS];
  const int32_t* counts;
  int32_t* status;      // sticky status word of the context (a look-back that never completes is reported, not waited for)
};
constexpr int kSortThreads = 256, kSortItems = 8, kSortTile = kSortThreads * kSortItems;
constexpr uint32_t kOsAggregate = 1u << 30, kOsPrefix = 2u << 30, kOsValue = (1u << 30) - 1u;

// Bit order of the spatial part of the key: a tile of 128 consecutive sorted rows shares the HIGH bits of the key and
// mixes the low ones, and it must walk every offset any of its rows has.  So the offsets that most voxels have anyway
// (centre, then the 6 face neighbours) sit in the low bits -- they are walked regardless -- and the rare ones (12 edge,
// then 8 corner neighbours: 9-15 % of the voxels of a LiDAR surface) in the high bits, where a tile either has them or
// not.  Measured offline on the bench scan (tools/tile_stats.py): offsets walked per tile 22.3 / 22.6 / 23.8 / 23.1 at
// levels 0-3 with the natural bit order (bit = offset index) -> 20.3 / 20.9 / 21.2 / 22.2.
__device__ __forceinline__ uint32_t shape_bits(uint32_t pat) {
  // offset index k3 = (dx+1) + 3 (dy+1) + 9 (dz+1), listed by |dx| + |dy| + |dz| (ties: |dz|)
  constexpr int order[27] = {13,                                     // centre
                             12, 14, 10, 16, 4, 22,                  // faces: x, y, z
                             9, 11, 15, 17, 3, 5, 21, 23, 1, 7, 19, 25,   // edges: xy, xz, yz
                             0, 2, 6, 8, 18, 20, 24, 26};            // corners
  uint32_t key = 0;
#pragma unroll
  for (int pos = 0; pos < 27; ++pos) key |= ((pat >> order[pos]) & 1u) << pos;
  return key;
}

// One radix pass over the concatenated levels.  LAST: the sorted row numbers go to the per-level perm arrays.
// 256 threads x 8 keys per tile (2048 keys, element order = round-major; 48 registers, 34 KB of shared memory): the per-tile
// work -- prefix over the slot counters, look-back over the predecessors' status words -- is amortised over twice the keys
// of the first version (4 keys per thread: 49 us per pass, now 37 us; 10 keys per thread measured the same as 8).
template <bool LAST>
__global__ void __launch_bounds__(kSortThreads)
k_onesweep_pass(const SortArgs A, const uint32_t* __restrict__ keys, const int32_t* __restrict__ vals, int shift,
                const uint32_t* __restrict__ hist, uint32_t* status, uint32_t* ticket, int pass,
                uint32_t* __restrict__ keys_out, int32_t* __restrict__ vals_out) {
  constexpr int kWarps = kSortThreads / 32, kSlots = kSortItems * kWarps;   // (round, warp) slots in element order
  __shared__ uint16_t wcount[kSlots][256];      // per-slot digit counts, then exclusive offsets across slots
  __shared__ int s_tile;
  __shared__ int s_base[256];                   // global position of this tile's first element per digit
  __shared__ int s_scan[kWarps];
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const int n = sort_total(A.counts);
  const int ntiles = (n + kSortTile - 1) / kSortTile;
  // the grid is sized by the host bound (rows x levels): the surplus blocks leave before touching anything, the first
  // ntiles blocks take one ticket each
  if ((int)blockIdx.x >= ntiles) return;
  if (tid == 0) s_tile = (int)atomicAdd(ticket, 1u);   // tiles are handed out in launch order: a tile's predecessors run
  for (int j = tid; j < kSlots * 128; j += kSortThreads) reinterpret_cast<uint32_t*>(&wcount[0][0])[j] = 0u;
  __syncthreads();
  const int tile = s_tile;
  uint32_t key[kSortItems];
  int val[kSortItems], rank[kSortItems];
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const int i = tile * kSortTile + r * kSortThreads + tid;
    const bool live = i < n;
    key[r] = live ? keys[i] : 0xFFFFFFFFu;
    val[r] = live ? vals[i] : -1;
  }
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    const bool live = val[r] >= 0;
    const unsigned digit = live ? ((key[r] >> shift) & 255u) : (256u + lane);   // dead lanes match nobody
    const unsigned peers = __match_any_sync(0xffffffffu, digit);
    rank[r] = __popc(peers & ((1u << lane) - 1u));
    if (live && rank[r] == 0) wcount[r * kWarps + w][digit] = (uint16_t)__popc(peers);
  }
  __syncthreads();
  {
    int run = 0;   // exclusive prefix over the slots of this tile for digit `tid`
#pragma unroll 8
    for (int sl = 0; sl < kSlots; ++sl) {
      const int c = wcount[sl][tid];
      wcount[sl][tid] = (uint16_t)run;
      run += c;
    }
    // decoupled look-back: digits of the tiles before this one
    uint32_t* st = status + ((size_t)tile * 4 + pass) * 256 + tid;
    int excl = 0;
    if (tile == 0) {
      atomicExch(st, kOsPrefix | (uint32_t)run);
    } else {
      atomicExch(st, kOsAggregate | (uint32_t)run);
      int t = tile - 1;
      unsigned spins = 0;
      while (true) {
        const uint32_t v = *reinterpret_cast<volatile uint32_t*>(status + ((size_t)t * 4 + pass) * 256 + tid);
        if ((v >> 30) == 0u) {                         // predecessor has not published yet (it is running: ticket order)
          if (++spins > (1u << 22)) { atomicOr(A.status, kStatusCapacity); break; }   // never hang: report instead
          __nanosleep(40);
          continue;
        }
        excl += (int)(v & kOsValue);
        if ((v >> 30) == 2u) break;
        --t;
      }
      atomicExch(st, kOsPrefix | (uint32_t)(excl + run));
    }
    // exclusive scan of the global digit histogram (256 values) = start of every digit's run
    const int hv = (int)hist[tid];
    int inc = hv;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int u = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += u;
    }
    if (lane == 31) s_scan[w] = inc;
    s_base[tid] = inc - hv + excl;
  }
  __syncthreads();
  {
    int add = 0;
    for (int ww = 0; ww < w; ++ww) add += s_scan[ww];
    s_base[tid] += add;
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < kSortItems; ++r) {
    if (val[r] < 0) continue;
    const unsigned digit = (key[r] >> shift) & 255u;
    const int pos = s_base[digit] + wcount[r * kWarps + w][digit] + rank[r];
    if (LAST) {
      const int j = (int)(key[r] >> 29);
      int off = 0;   // (a predicated sum: with a loop to j the kernel takes 64 registers instead of 48)
#pragma unroll
      for (int q = 0; q < SPS_NUM_LEVELS - 1; ++q) if (q < j) off += A.counts[q];
      A.perm[j][pos - off] = val[r];
    } else {
      keys_out[pos] = key[r];
      vals_out[pos] = val[r];
    }
  }
}

// present-offset masks of the 128-row tiles taken in `perm` order, and the tiles' slices of the kernel map gathered once
// for all the convolutions of the level: slices[tile][e][r] = input row of sorted row r under the tile's e-th present
// offset, entry e = #present = the tile's own rows.  All levels in one launch (blockIdx.y).
struct SliceArgs {
  const uint32_t* vmask[SPS_NUM_LEVELS];
  const int32_t* perm[SPS_NUM_LEVELS];
  uint32_t* masks[SPS_NUM_LEVELS];
  const int32_t* nbr[SPS_NUM_LEVELS];
  int32_t* slices[SPS_NUM_LEVELS];
  const int32_t* counts;
  int64_t ld;
};
__global__ void __launch_bounds__(128)
k_tile_masks_perm(const SliceArgs A) {
  const int L = blockIdx.y;
  const int n = A.counts[L];
  const int ntiles = (n + 127) / 128;
  const uint32_t* __restrict__ vmask = A.vmask[L];
  const int32_t* __restrict__ perm = A.perm[L];
  uint32_t* __restrict__ masks = A.masks[L];
  const int32_t* __restrict__ nbr = A.nbr[L];
  int32_t* __restrict__ slices = A.slices[L];
  const int64_t ld = A.ld;
  __shared__ uint32_t m[4][3];
  __shared__ uint8_t klist[96];
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int r = tile * 128 + threadIdx.x;
    uint32_t w0 = 0, w1 = 0, w2 = 0;
    int v = -1;
    if (r < n) {
      v = perm[r];
      const uint4 vm4 = __ldg(reinterpret_cast<const uint4*>(vmask) + v);          // 27 bits per time plane, one 16-byte read
      const uint32_t m0 = vm4.x, m1 = vm4.y, m2 = vm4.z;
      w0 = m0 | (m1 << 27);
      w1 = (m1 >> 5) | (m2 << 22);
      w2 = m2 >> 10;
    }
    const uint32_t t0 = __reduce_or_sync(0xffffffffu, w0);
    const uint32_t t1 = __reduce_or_sync(0xffffffffu, w1);
    const uint32_t t2 = __reduce_or_sync(0xffffffffu, w2);
    if ((threadIdx.x & 31) == 0) { m[threadIdx.x >> 5][0] = t0; m[threadIdx.x >> 5][1] = t1; m[threadIdx.x >> 5][2] = t2; }
    __syncthreads();
    const uint32_t tm[3] = {m[0][0] | m[1][0] | m[2][0] | m[3][0], m[0][1] | m[1][1] | m[2][1] | m[3][1],
                            m[0][2] | m[1][2] | m[2][2] | m[3][2]};
    if (threadIdx.x < 3) masks[4 * tile + threadIdx.x] = tm[threadIdx.x];
    if (threadIdx.x == 3) masks[4 * tile + 3] = 0;
    const int nact = __popc(tm[0]) + __popc(tm[1]) + __popc(tm[2]);
    if (threadIdx.x < 96) {
      const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
      if ((tm[w] >> l) & 1u) {
        const int before = (w > 0 ? __popc(tm[0]) : 0) + (w > 1 ? __popc(tm[1]) : 0) + __popc(tm[w] & ((1u << l) - 1u));
        klist[before] = (uint8_t)threadIdx.x;
      }
    }
    __syncthreads();
    int32_t* dst = slices + (int64_t)tile * (SPS_TILE_SLICE_ENTRIES * 128) + threadIdx.x;
    const uint32_t mine[3] = {w0, w1, w2};
    // kSliceBatch entries at a time: the loads of a batch are issued before the first store (the pass waits on these random
    // 4-byte reads; unroll depth = reads in flight per thread)
    for (int e0 = 0; e0 < nact; e0 += kSliceBatch) {
      int val[kSliceBatch];
#pragma unroll
      for (int u = 0; u < kSliceBatch; ++u) {
        const int e = e0 + u;
        const int k = e < nact ? klist[e] : 0;
        val[u] = -1;
        if (e < nact && ((mine[k >> 5] >> (k & 31)) & 1u)) val[u] = __ldg(nbr + (int64_t)k * ld + v);
      }
#pragma unroll
      for (int u = 0; u < kSliceBatch; ++u)
        if (e0 + u < nact) dst[(e0 + u) * 128] = val[u];
    }
    dst[nact * 128] = v;
    __syncthreads();
  }
}

// conv0 when every voxel carries the SAME input feature c (SPSModel.forward: the mean of the constant
// 0.5 point features, models.py:22-25): out[o] = relu(c * sum_{k present} W[k][:] + shift).  Only the
// PRESENCE of the 125 neighbours matters, and that is one bit of the 64-bit occupancy word of a 4x4x4
// block: 8 block probes per voxel, no index reads at all; the weight sum goes through per-row tables.
__global__ void __launch_bounds__(256, 4)
k_conv0_const(const unsigned long long* __restrict__ keys, const int32_t* __restrict__ n_ptr,
              const Slot* __restrict__ tab, const int32_t* __restrict__ cap_n,
              const unsigned long long* __restrict__ occ, float cfeat,
              const float* __restrict__ w, const float* __restrict__ shift, int round_out, float* __restrict__ out,
              int64_t out_ld) {
  // row tables: T[row = (dz, dy)][5-bit x pattern][8] = sum of W[k][:] over the pattern's present dx.  A voxel then
  // needs 25 table rows (skipping empty ones) instead of 125 predicated weight adds.
  __shared__ __align__(16) float w_t[25 * 32 * 8];
  for (int e = threadIdx.x; e < 25 * 32; e += blockDim.x) {
    const int row = e >> 5, pat = e & 31;
    float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int dx = 0; dx < 5; ++dx)
      if ((pat >> dx) & 1)
        for (int c = 0; c < 8; ++c) a[c] += __ldg(w + (row * 5 + dx) * 8 + c);
    for (int c = 0; c < 8; ++c) w_t[e * 8 + c] = a[c];
  }
  __syncthreads();
  const int n = *n_ptr;
  if (n == 0) return;
  const uint32_t mask = table_capacity(*cap_n) - 1;
  const int blim = 1 << (kXBits - 2), zblim = 1 << (kZBits - 2);
  for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < n; o += gridDim.x * blockDim.x) {
    const unsigned long long key = keys[o];
    const int cx = (int)((key >> kXShift) & ((1u << kXBits) - 1));
    const int cy = (int)((key >> kYShift) & ((1u << kYBits) - 1));
    const int cz = (int)((key >> kZShift) & ((1u << kZBits) - 1));
    const unsigned long long bt = key & ((0xFFull << kBShift) | ((1ull << kTBits) - 1));
    // the window [c-2, c+2] touches at most two blocks per axis: b0 and b0 + 1.  Pass 1 (block-relative,
    // divergent but ALU-only): collect the presence bits of the 125 neighbours into a 128-bit vector,
    // bit k = kernel offset index.  Pass 2 (warp-uniform over k): weights are shared-memory broadcasts.
    const int bx0 = (cx - 2) >> 2, by0 = (cy - 2) >> 2, bz0 = (cz - 2) >> 2;
    unsigned long long o8[8];     // occupancy words of the 2 x 2 x 2 blocks the window meets (0: no such block)
#pragma unroll
    for (int jb = 0; jb < 8; ++jb) {
      const int bx = bx0 + (jb & 1), by = by0 + ((jb >> 1) & 1), bz = bz0 + (jb >> 2);
      o8[jb] = 0ull;
      if (max(cx - 2, bx * 4) > min(cx + 2, bx * 4 + 3) || max(cy - 2, by * 4) > min(cy + 2, by * 4 + 3) ||
          max(cz - 2, bz * 4) > min(cz + 2, bz * 4 + 3))
        continue;
      if ((unsigned)bx >= (unsigned)blim || (unsigned)by >= (unsigned)blim || (unsigned)bz >= (unsigned)zblim) continue;
      const unsigned long long bkey = bt | ((unsigned long long)(unsigned)(bx << 2) << kXShift) |
                                      ((unsigned long long)(unsigned)(by << 2) << kYShift) |
                                      ((unsigned long long)(unsigned)(bz << 2) << kZShift);
      const int id = table_find(tab, mask, bkey);
      if (id >= 0) o8[jb] = __ldg(occ + id);
    }
    // Per (dz, dy) row of the window the five x-neighbours are five adjacent bits of an 8-bit line: the x-rows of the two
    // blocks side by side.  Rows in ascending kernel-offset order (the order of the weight sums is part of the result).
    const int offx = (cx - 2) - bx0 * 4;        // 0..3: where the window starts in the line
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
#pragma unroll
    for (int dz = -2; dz <= 2; ++dz) {
      const int nz = cz + dz;
      const bool jz = ((nz >> 2) - bz0) != 0;
      const unsigned long long a00 = jz ? o8[4] : o8[0], a01 = jz ? o8[5] : o8[1], a10 = jz ? o8[6] : o8[2], a11 = jz ? o8[7] : o8[3];
#pragma unroll
      for (int dy = -2; dy <= 2; ++dy) {
        const int ny = cy + dy;
        const bool jy = ((ny >> 2) - by0) != 0;
        const unsigned long long A = jy ? a10 : a00, B = jy ? a11 : a01;
        const int lyz = 4 * (ny & 3) + 16 * (nz & 3);
        const uint32_t line = ((uint32_t)(A >> lyz) & 15u) | (((uint32_t)(B >> lyz) & 15u) << 4);
        const uint32_t pat = (line >> offx) & 31u;
        const int row = (dy + 2) + 5 * (dz + 2);
        if (pat) {
          const float4 w0 = *reinterpret_cast<const float4*>(w_t + (row * 32 + pat) * 8);
          const float4 w1 = *reinterpret_cast<const float4*>(w_t + (row * 32 + pat) * 8 + 4);
          acc[0] += w0.x; acc[1] += w0.y; acc[2] += w0.z; acc[3] += w0.w;
          acc[4] += w1.x; acc[5] += w1.y; acc[6] += w1.z; acc[7] += w1.w;
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = fmaxf(fmaf(cfeat, acc[c], __ldg(shift + c)), 0.f);
    store_row8(out, out_ld, o, acc, round_out);
  }
}

// conv0p1s1 (5x5x5x1, Cin = 1 -> 8; minkunet.py:55-62,162-164) fused with its kernel-map probes:
// out[o] = relu( sum_k feat[nbr5(k, o)] * W[k][:] + shift ), the 125 neighbours resolved through the
// block table on the fly, so the 125 x V index table is neither written nor read back.
__global__ void __launch_bounds__(256)
k_conv0_blk(const unsigned long long* __restrict__ keys, const int32_t* __restrict__ n_ptr,
            const Slot* __restrict__ tab, const int32_t* __restrict__ cap_n,
            const int32_t* __restrict__ cells, const unsigned long long* __restrict__ occ, const float* __restrict__ feat,
            const float* __restrict__ w, const float* __restrict__ shift, int round_out, float* __restrict__ out,
            int64_t out_ld) {
  __shared__ float w_s[125 * 8];
  for (int i = threadIdx.x; i < 125 * 8; i += blockDim.x) w_s[i] = __ldg(w + i);
  __syncthreads();
  const int n = *n_ptr;
  if (n == 0) return;
  const uint32_t mask = table_capacity(*cap_n) - 1;
  const int xlim = 1 << kXBits, zlim = 1 << kZBits;
  for (int o = blockIdx.x * blockDim.x + threadIdx.x; o < n; o += gridDim.x * blockDim.x) {
    const unsigned long long key = keys[o];
    const int cx = (int)((key >> kXShift) & ((1u << kXBits) - 1));
    const int cy = (int)((key >> kYShift) & ((1u << kYBits) - 1));
    const int cz = (int)((key >> kZShift) & ((1u << kZBits) - 1));
    const unsigned long long bt = key & ((0xFFull << kBShift) | ((1ull << kTBits) - 1));
    unsigned long long cached_key = kEmptyKey, cached_occ = 0ull;
    const int32_t* cached = nullptr;
    float acc[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = 0.f;
#pragma unroll 1
    for (int dz = -2; dz <= 2; ++dz) {
      const int nz = cz + dz;
      const bool zok = (unsigned)nz < (unsigned)zlim;
#pragma unroll 1
      for (int dy = -2; dy <= 2; ++dy) {
        const int ny = cy + dy;
        const bool yok = zok && (unsigned)ny < (unsigned)xlim;
        const unsigned long long byz = bt | ((unsigned long long)(unsigned)((ny >> 2) << 2) << kYShift) |
                                       ((unsigned long long)(unsigned)((nz >> 2) << 2) << kZShift);
        const int lyz = 4 * (ny & 3) + 16 * (nz & 3);
        const float* wk = w_s + ((dy + 2) * 5 + (dz + 2) * 25) * 8;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
          const int nx = cx + dx;
          if (!(yok && (unsigned)nx < (unsigned)xlim)) continue;
          const unsigned long long bkey = byz | ((unsigned long long)(unsigned)((nx >> 2) << 2) << kXShift);
          if (bkey != cached_key) {
            cached_key = bkey;
            const int id = table_find(tab, mask, bkey);
            cached = id >= 0 ? cells + (int64_t)id * 64 : nullptr;
            cached_occ = id >= 0 ? __ldg(occ + id) : 0ull;
          }
          const int l = lyz + (nx & 3);
          if (!((cached_occ >> l) & 1ull)) continue;     // the cells of a block are only defined where its occupancy bit is set
          const int idx = __ldg(cached + l);
          const float x = __ldg(feat + idx);
          const float4 w0 = *reinterpret_cast<const float4*>(wk + (dx + 2) * 8);
          const float4 w1 = *reinterpret_cast<const float4*>(wk + (dx + 2) * 8 + 4);
          acc[0] = fmaf(x, w0.x, acc[0]); acc[1] = fmaf(x, w0.y, acc[1]);
          acc[2] = fmaf(x, w0.z, acc[2]); acc[3] = fmaf(x, w0.w, acc[3]);
          acc[4] = fmaf(x, w1.x, acc[4]); acc[5] = fmaf(x, w1.y, acc[5]);
          acc[6] = fmaf(x, w1.z, acc[6]); acc[7] = fmaf(x, w1.w, acc[7]);
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 8; ++c) acc[c] = fmaxf(acc[c] + __ldg(shift + c), 0.f);
    store_row8(out, out_ld, o, acc, round_out);
  }
}


__global__ void k_unpack(const unsigned long long* __restrict__ keys, const int32_t* __restrict__ n_ptr,
                         int32_t* __restrict__ out) {
  const int n = *n_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    int b, x, y, z, t;
    unpack_key(keys[i], b, x, y, z, t);
    int32_t* o = out + (int64_t)i * 5;
    o[0] = b; o[1] = x; o[2] = y; o[3] = z; o[4] = t;
  }
}

static inline int grid_for(int64_t work, int block, int cap = 148 * 32) {
  int64_t g = (work + block - 1) / block;
  if (g < 1) g = 1;
  if (g > cap) g = cap;
  return (int)g;
}

}  // namespace sps

using namespace sps;

namespace sps {

// n_upper sizes the launches; the true row count is n_upper, or *d_n when d_n is given.
int voxelize_impl(sps_ctx* ctx, const float* d_points, int64_t n, const int32_t* d_n, int64_t ld_points,
                  float voxel_size, cudaStream_t st) {
  if (!ctx || (!d_points && n > 0) || n < 0 || ld_points < 5 || !(voxel_size > 0.f)) return SPS_ERR_BAD_ARG;
  if (n > ctx->max_points) return SPS_ERR_CAPACITY;
  ctx->n = n;
  ctx->have_l0 = ctx->have_maps = false;
  // n travels as a kernel-visible scalar so that every level shares one code path
  const int nblk = cdiv(n > 0 ? n : 1, kScanBlock);
  k_level_begin<<<grid_for(table_capacity(n), 256), 256, 0, st>>>(ctx->table, d_n, d_n ? -1 : (int32_t)n, ctx->n_dev, nullptr, 0,
                                                                  ctx->tplanes);
  prof_mark(ctx, "vox.clear", st);
  k_insert_points<<<grid_for(cdiv(n, kInsertBatch), 256, 148 * 8), 256, 0, st>>>(d_points, ld_points, ctx->n_dev, voxel_size, ctx->table,
                                                     ctx->slot_of, ctx->status, ctx->tplanes);
  prof_mark(ctx, "vox.insert", st);
  k_first_rank<<<cdiv(nblk, kRankChunks), kScanBlock, 0, st>>>(ctx->table, ctx->slot_of, ctx->n_dev, ctx->rank, ctx->block_sums,
                                            ctx->ticket, ctx->counts + 0, nullptr, 0, nullptr);
  prof_mark(ctx, "vox.rank", st);
  k_assign_points<<<grid_for(n, 256), 256, 0, st>>>(ctx->table, ctx->slot_of, ctx->n_dev, ctx->rank,
                                                     ctx->block_sums, ctx->keys[0], ctx->inv);
  prof_mark(ctx, "vox.assign", st);
  SPS_CUDA_CHECK(cudaGetLastError());
  ctx->have_l0 = true;
  return SPS_OK;
}
}  // namespace sps

extern "C" int sps_voxelize(sps_ctx* ctx, const float* d_points, int64_t n, int64_t ld_points, float voxel_size,
                            void* stream_) {
  return voxelize_impl(ctx, d_points, n, nullptr, ld_points, voxel_size, (cudaStream_t)stream_);
}

namespace sps {
int build_maps_impl(sps_ctx* ctx, const Conv0Fused* c0, cudaStream_t st);
// exact-fp32 mode gathers from the dense maps (generic CUDA-core kernels)
static inline bool needs_dense_maps(const sps_ctx* ctx) { return ctx->backend == SPS_BACKEND_FP32; }

constexpr int64_t kMinRowsForSort = 400000;   // small inputs (single scans) are launch-bound: the sort does not pay

static inline bool sort_active(const sps_ctx* ctx) {
  return ctx->pattern_sort == 2 || (ctx->pattern_sort == 1 && ctx->n >= kMinRowsForSort);
}

// perm[L] = voxel rows of level L sorted by neighbourhood-shape key, ptmask[L] = tile masks in that order, tslice[L] = the
// kernel map gathered per sorted tile -- for all levels at once (level 4 adds 2 % to the keys): 4 + 1 launches.
static int pattern_order(sps_ctx* ctx, cudaStream_t st) {
  if (!sort_active(ctx)) return SPS_OK;
  const int64_t n = ctx->n > 0 ? ctx->n : 1;
  SortArgs A;
  for (int L = 0; L < SPS_NUM_LEVELS; ++L) A.perm[L] = ctx->perm[L];
  A.counts = ctx->counts; A.status = ctx->status;
  uint32_t* hist = ctx->sort_hist;
  // (keys, row numbers and digit histograms were left behind by the 3x3x3x3 kernel-map pass)
  const int tiles_max = cdiv(n * SPS_NUM_LEVELS, kSortTile);
  for (int pass = 0; pass < 4; ++pass) {
    const uint32_t* ki = ctx->sort_keys[pass & 1];
    const int32_t* vi = ctx->sort_vals[pass & 1];
    uint32_t* ko = ctx->sort_keys[(pass & 1) ^ 1];
    int32_t* vo = ctx->sort_vals[(pass & 1) ^ 1];
    if (pass < 3)
      k_onesweep_pass<false><<<tiles_max, kSortThreads, 0, st>>>(A, ki, vi, 8 * pass, hist + 256 * pass, ctx->sort_status, hist + 1024 + pass,
                                                              pass, ko, vo);
    else
      k_onesweep_pass<true><<<tiles_max, kSortThreads, 0, st>>>(A, ki, vi, 8 * pass, hist + 256 * pass, ctx->sort_status, hist + 1024 + pass,
                                                             pass, nullptr, nullptr);
  }
  prof_mark(ctx, "sort", st);
  SliceArgs S;
  for (int L = 0; L < SPS_NUM_LEVELS; ++L) {
    S.vmask[L] = ctx->vmask[L]; S.perm[L] = ctx->perm[L]; S.masks[L] = ctx->ptmask[L]; S.nbr[L] = ctx->nbr3[L];
    S.slices[L] = ctx->tslice[L];
  }
  S.counts = ctx->counts; S.ld = ctx->ld;
  k_tile_masks_perm<<<dim3(grid_for(n / 128 + 1, 1, 148 * 8), SPS_NUM_LEVELS), 128, 0, st>>>(S);
  prof_mark(ctx, "slices", st);
  SPS_CUDA_CHECK(cudaGetLastError());
  ctx->forward_launches += 5;
  return SPS_OK;
}
}
extern "C" int sps_build_maps(sps_ctx* ctx, void* stream_) {
  return build_maps_impl(ctx, nullptr, (cudaStream_t)stream_);
}

// c0 != nullptr: the fused forward -- conv0 runs here, straight off the level-0 block table, and the
// 5x5x5x1 index table is not materialised.
int sps::build_maps_impl(sps_ctx* ctx, const Conv0Fused* c0, cudaStream_t st) {
  if (!ctx) return SPS_ERR_BAD_ARG;
  if (!ctx->have_l0) return SPS_ERR_STATE;
  const int64_t n = ctx->n > 0 ? ctx->n : 1;  // host upper bound of every level's voxel count
  const int nblk = cdiv(n, kScanBlock);
  // ---- 1. strided coordinate sets, levels 1..4 (each level hashes the keys of the one below: a sequential chain) ----
  for (int L = 1; L < SPS_NUM_LEVELS; ++L) {
    const int32_t* n_fine = ctx->counts + (L - 1);
    // The voxels of level L are the 4x4x4-cell blocks of level L - 2: levels 2..4 build their hash where the block table
    // of that level lives, so that it answers "block key -> block row" later without a second hash build
    // (k_block_insert was 100 us per forward); k_blocks_begin writes the rows into the slots.
    Slot* tab = L >= 2 ? ctx->btab[L - 2] : ctx->table;
    int32_t* sums = ctx->block_sums;
    k_level_begin<<<grid_for(table_capacity(n), 256), 256, 0, st>>>(tab, n_fine, -1, nullptr, ctx->child[L], ctx->ld, nullptr,
                                                                    ctx->up_cls + 16 * (L - 1));
    k_insert_coarse<<<grid_for(n, 256), 256, 0, st>>>(ctx->keys[L - 1], n_fine, L, tab, ctx->slot_of);
    k_first_rank<<<cdiv(nblk, kRankChunks), kScanBlock, 0, st>>>(tab, ctx->slot_of, n_fine, ctx->rank, sums,
                                              ctx->ticket, ctx->counts + L, nullptr, 0, nullptr);
    k_assign_coarse<<<grid_for(n, 256), 256, 0, st>>>(tab, ctx->slot_of, n_fine, ctx->rank, sums,
                                                       ctx->keys[L - 1], L - 1, ctx->keys[L], ctx->parent[L - 1],
                                                       ctx->child[L], ctx->ld, ctx->up_cls + 16 * (L - 1));
    static const char* nm_s[5] = {"", "stride.L1", "stride.L2", "stride.L3", "stride.L4"};
    prof_mark(ctx, nm_s[L], st);
  }
  {   // class order of the fine rows of levels 0..3 for the transposed convolutions (one launch)
    UpOrderArgs U;
    for (int L = 0; L < SPS_NUM_LEVELS; ++L) { U.parent[L] = ctx->parent[L]; U.perm[L] = ctx->perm_up[L]; U.masks[L] = ctx->tmask_up[L]; }
    U.counts = ctx->counts; U.cls = ctx->up_cls;
    k_up_order<<<dim3(grid_for(n, 256, 148 * 4), SPS_NUM_LEVELS - 1), 256, 0, st>>>(U);
    prof_mark(ctx, "up_order", st);
  }
  // ---- 2. block tables of all five levels (three launches) ----
  // fused forward with the shape sort: the convolutions read the tile slices and the sorted tile masks, the slices read
  // only present entries -> neither the -1 entries nor the physical-order tile masks are produced
  const bool sorting = sort_active(ctx);
  const bool sparse = c0 != nullptr && !needs_dense_maps(ctx) && sorting;
  LevelTabs T;
  ScratchZero Z;
  KmapOut O;
  for (int L = 0; L < SPS_NUM_LEVELS; ++L) {
    T.keys[L] = ctx->keys[L]; T.btab[L] = ctx->btab[L]; T.cells[L] = ctx->bcells[L]; T.occ[L] = ctx->bocc[L];
    T.parent[L] = ctx->parent[L];
    Z.tmask3[L] = sparse ? nullptr : ctx->tmask3[L];
    O.nbr[L] = ctx->nbr3[L]; O.tile_masks[L] = Z.tmask3[L]; O.vmask[L] = ctx->vmask[L];
  }
  T.counts = ctx->counts; T.nblocks = ctx->nblocks; T.tplanes = ctx->tplanes;
  Z.sort_hist = sorting ? ctx->sort_hist : nullptr; Z.sort_status = ctx->sort_status;
  O.ld = ctx->ld;
  O.dense = sparse ? 0 : 1;
  O.sort_keys = sorting ? ctx->sort_keys[0] : nullptr; O.sort_vals = ctx->sort_vals[0]; O.sort_hist = ctx->sort_hist;
  const int gx = grid_for(n, 256, 148 * 6);   // one wave of the kernel-map pass (6 blocks of 256 threads per SM at 40 registers)
  k_blocks_begin<<<dim3(grid_for(table_capacity(n), 256, 148 * 8), SPS_NUM_LEVELS), 256, 0, st>>>(T, Z);
  k_block_insert<<<dim3(gx, SPS_NUM_LEVELS), 256, 0, st>>>(T);
  k_cells_fill<<<dim3(gx, SPS_NUM_LEVELS), 256, 0, st>>>(T);
  prof_mark(ctx, "blocks", st);
  // ---- 3. conv0 off the level-0 block table (fused forward), or the 5x5x5x1 table (layer-level API) ----
  if (c0) {
    if (c0->feat)   // per-voxel features: gather them through the block table
      k_conv0_blk<<<grid_for(n, 256), 256, 0, st>>>(ctx->keys[0], ctx->counts + 0, ctx->btab[0], ctx->counts + btab_sized_for(0), ctx->bcells[0], ctx->bocc[0], c0->feat,
                                                     c0->w, c0->shift, c0->round_out, c0->out, c0->out_ld);
    else            // one constant feature (SPSModel.forward): presence bits only
      k_conv0_const<<<grid_for(n, 256), 256, 0, st>>>(ctx->keys[0], ctx->counts + 0, ctx->btab[0], ctx->counts + btab_sized_for(0), ctx->bocc[0], c0->cfeat,
                                                       c0->w, c0->shift, c0->round_out, c0->out, c0->out_ld);
    prof_mark(ctx, "conv0+kmap5", st);
  } else {
    k_kernel_map_blk5<<<grid_for(n, 256), 256, 0, st>>>(ctx->keys[0], ctx->counts + 0, ctx->btab[0], ctx->counts + btab_sized_for(0), ctx->bcells[0],
                                                         ctx->bocc[0], ctx->nbr5, ctx->ld);
    prof_mark(ctx, "kmap5.L0", st);
  }
  ctx->have_nbr5 = c0 == nullptr;
  // ---- 4. 3x3x3x3 kernel maps of all five levels (one launch: level x time plane) ----
  k_kernel_map_blk3<<<dim3(gx, 1, SPS_NUM_LEVELS), 256, 0, st>>>(T, O);
  prof_mark(ctx, "kmap3", st);
  SPS_CUDA_CHECK(cudaGetLastError());
  ctx->forward_launches += 16 + 1 + 3 + 1 + 1;
  // ---- 5. shape sort + per-tile slices ----
  { const int rc = pattern_order(ctx, st); if (rc != SPS_OK) return rc; }
  ctx->have_maps = true;
  ctx->dense_maps = !sparse;
  ctx->have_perm = sorting;
  return SPS_OK;
}

extern "C" int sps_unpack_coords(sps_ctx* ctx, int level, int32_t* d_out, void* stream_) {
  if (!ctx || !d_out || level < 0 || level >= SPS_NUM_LEVELS) return SPS_ERR_BAD_ARG;
  if (!ctx->have_l0 || (level > 0 && !ctx->have_maps)) return SPS_ERR_STATE;
  const int64_t n = ctx->n > 0 ? ctx->n : 1;
  k_unpack<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream_>>>(ctx->keys[level], ctx->counts + level, d_out);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

// =====================================================================================
// Submap selection: replicated base-map voxel hash + crops (a12/a13, SURVEY.md §8a)
// =====================================================================================
struct sps_map {
  sps::Slot* table = nullptr;
  uint32_t cap = 0;
  int64_t n = 0;
  float ds = 0.f;
  int32_t* scalars = nullptr;  // [0] = n (device copy), [1] = status
};

namespace sps {

struct Scratch {  // carve of a sps_map_bytes(n) buffer
  int32_t* scalars;   // 64 ints: [0]=n_dev; second 128-byte line (atomics): [32]=ticket [40]=status
  Slot* table;
  uint32_t cap;
  uint32_t* slot_of;
  int32_t* rank;
  int32_t* block_sums;
  size_t bytes;
};
static Scratch carve_scratch(void* base, int64_t n) {
  Scratch s;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t b) { off = (off + 255) & ~size_t(255); char* r = p ? p + off : nullptr; off += b; return r; };
  s.scalars = (int32_t*)take(64 * 4);
  s.cap = table_capacity(n);
  s.table = (Slot*)take((size_t)s.cap * sizeof(Slot));
  s.slot_of = (uint32_t*)take((size_t)n * 4);
  s.rank = (int32_t*)take((size_t)n * 4);
  s.block_sums = (int32_t*)take((size_t)(n / kScanBlock + 2) * 4);
  s.bytes = (off + 255) & ~size_t(255);
  return s;
}

// util.to_coords_features (src/sps/datasets/util.py:72-75): fp32 division by ds, then
// `.int()` = truncation toward zero; the time field is 0 in this 3-D lattice, the batch field is 0 except in the
// scratch table of a batched prune (which keeps the scans of a batch apart).
__device__ inline bool trunc_key(const float* __restrict__ p, float ds, unsigned long long& key, int b = 0) {
  const float qx = truncf(__fdiv_rn(p[0], ds)), qy = truncf(__fdiv_rn(p[1], ds)), qz = truncf(__fdiv_rn(p[2], ds));
  const bool ok = qx >= -(float)kXBias && qx < (float)kXBias && qy >= -(float)kXBias && qy < (float)kXBias &&
                  qz >= -(float)kZBias && qz < (float)kZBias;
  if (!ok) return false;
  key = pack_key(b, (int)qx, (int)qy, (int)qz, 0);
  return true;
}

// point i (xyz at p, scan b) into the crop table, `first` lowered to i; out-of-range points get no slot
__device__ __forceinline__ void insert_xyz(const float* __restrict__ p, int i, int b, float ds, Slot* tab, uint32_t mask,
                                           uint32_t* __restrict__ slot_of, int32_t* status) {
  unsigned long long key;
  if (!trunc_key(p, ds, key, b)) {
    atomicOr(status, kStatusRange);
    if (slot_of) slot_of[i] = kInvalidSlot;
    return;
  }
  const uint32_t s = table_insert(tab, mask, key);
  atomicMin(&tab[s].first, i);
  tab[s].val = 0;
  if (slot_of) slot_of[i] = s;
}

__global__ void k_insert_xyz(const float* __restrict__ xyz, const int32_t* __restrict__ n_ptr, float ds, Slot* tab,
                             uint32_t* __restrict__ slot_of, int32_t* status) {
  const int n = *n_ptr;
  const uint32_t mask = table_capacity(n) - 1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    insert_xyz(xyz + (int64_t)i * 3, i, 0, ds, tab, mask, slot_of, status);
}

// util.prune tail (util.py:101-112): a kept voxel -> `coordinates * ds` in fp32
__device__ __forceinline__ void write_corner(unsigned long long key, float ds, float* __restrict__ o) {
  int b, x, y, z, t;
  unpack_key(key, b, x, y, z, t);
  o[0] = __fmul_rn((float)x, ds);
  o[1] = __fmul_rn((float)y, ds);
  o[2] = __fmul_rn((float)z, ds);
}

__global__ void k_write_submap(const Slot* __restrict__ tab, const uint32_t* __restrict__ slot_of,
                               const int32_t* __restrict__ n_ptr, const int32_t* __restrict__ rank,
                               const int32_t* __restrict__ block_sums, const Slot* __restrict__ filter,
                               uint32_t filter_mask, float ds, float* __restrict__ out) {
  const int n = *n_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t s = slot_of[i];
    if (s == kInvalidSlot || tab[s].first != i) continue;
    const unsigned long long key = tab[s].key;
    if (table_find(filter, filter_mask, key) < 0) continue;
    const int id = rank[i] + block_sums[i / kScanBlock];
    write_corner(key, ds, out + (int64_t)id * 3);
  }
}

// ---- batched prune: B scans concatenated -> util.infer's rows per scan, collated ----
// Scan b's rows are its n_b scan rows [b, x, y, z, 1], then its submap rows [b, corner, 0] (sps_submap_crop_voxel of
// scan b alone, same order).  The scratch table keys voxels by (b, trunc xyz), so scans never share a voxel and the
// first occurrence of a voxel is its first point in scan b; the map is probed with b cleared.  With K = the exclusive
// prefix of the "kept" flags (first occurrence and in the map) over the whole batch, scan b's rows start at
// off[b] + K(off[b]) and the kept voxel of point i sits at off[b+1] + K(i).
constexpr unsigned long long kKeyNoBatch = (1ull << kBShift) - 1;

__global__ void k_prune_batch_insert(const float* __restrict__ scan, int64_t ld, int n, const __grid_constant__ BatchOffsets bo,
                                     float ds, Slot* tab, uint32_t* __restrict__ slot_of, int32_t* status) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  const uint32_t mask = table_capacity(n) - 1;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    insert_xyz(scan + (int64_t)i * ld, i, batch_of(s_off, bo.batch, i), ds, tab, mask, slot_of, status);
}

// kept flags -> grid-wide exclusive scan (scan.cuh); counts[2b+1] += unique scan voxels of scan b (counts zeroed before)
__global__ void __launch_bounds__(kScanBlock)
k_prune_batch_rank(const Slot* __restrict__ tab, const uint32_t* __restrict__ slot_of, int n,
                   const __grid_constant__ BatchOffsets bo, const Slot* __restrict__ filter, uint32_t filter_mask,
                   int32_t* __restrict__ rank, int32_t* block_sums, uint32_t* ticket, int32_t* total, int32_t* counts) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  const int nb = max(1, (n + kScanBlock - 1) / kScanBlock);
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  int b = kMaxBatch + 1, first = 0;            // past-the-end lanes: a scan of their own
  unsigned long long key = 0;
  if (i < n) {
    b = batch_of(s_off, bo.batch, i);
    const uint32_t s = slot_of[i];
    if (s != kInvalidSlot) {
      const int4 raw = *reinterpret_cast<const int4*>(tab + s);   // key | val | first input
      first = raw.w == i;
      key = ((unsigned long long)(unsigned)raw.y << 32) | (unsigned)raw.x;
    }
  }
  // the lanes of one scan add their first occurrences with one atomic
  const unsigned peers = __match_any_sync(0xffffffffu, b);
  const unsigned firsts = __ballot_sync(0xffffffffu, first) & peers;
  if (i < n && (threadIdx.x & 31) == __ffs(peers) - 1 && firsts) atomicAdd(counts + 2 * b + 1, __popc(firsts));
  const int kept = first && table_find(filter, filter_mask, key & kKeyNoBatch) >= 0;
  scan_flags(kept, i, n, nb, rank, block_sums, ticket, total);
}

__device__ __forceinline__ void write_row5(float* __restrict__ rows, int64_t r, float b, float x, float y, float z, float t) {
  float* o = rows + r * 5;
  o[0] = b; o[1] = x; o[2] = y; o[3] = z; o[4] = t;
}

// every row at its collate position, the per-scan row offsets, the row count and counts[2b] = submap voxels of scan b
__global__ void __launch_bounds__(256)
k_prune_batch_write(const float* __restrict__ scan, int64_t ld, int n, const __grid_constant__ BatchOffsets bo,
                    const Slot* __restrict__ tab, const uint32_t* __restrict__ slot_of, const int32_t* __restrict__ rank,
                    const int32_t* __restrict__ block_sums, const int32_t* __restrict__ total_ptr, float ds,
                    float* __restrict__ rows, int32_t* __restrict__ row_off, int32_t* __restrict__ n_rows,
                    int32_t* __restrict__ counts) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  const int total = *total_ptr;
  if (blockIdx.x == 0) {
    for (int b = threadIdx.x; b <= bo.batch; b += blockDim.x) {
      const int k0 = hit_prefix(rank, block_sums, n, total, s_off[b]);
      row_off[b] = s_off[b] + k0;
      if (b < bo.batch) counts[2 * b] = hit_prefix(rank, block_sums, n, total, s_off[b + 1]) - k0;
    }
    if (threadIdx.x == 0) *n_rows = n + total;
  }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int b = batch_of(s_off, bo.batch, i);
    const float* p = scan + (int64_t)i * ld;
    const float fb = (float)b;
    write_row5(rows, (int64_t)i + hit_prefix(rank, block_sums, n, total, s_off[b]), fb, p[0], p[1], p[2], 1.0f);
    const int k = hit_prefix(rank, block_sums, n, total, i);
    if (hit_prefix(rank, block_sums, n, total, i + 1) == k) continue;    // not a kept voxel
    float c[3];
    write_corner(tab[slot_of[i]].key, ds, c);
    write_row5(rows, (int64_t)s_off[b + 1] + k, fb, c[0], c[1], c[2], 0.0f);
  }
}

// fused call: the scan rows' scores in input order
__global__ void __launch_bounds__(256)
k_prune_batch_scores(int n, const __grid_constant__ BatchOffsets bo, const int32_t* __restrict__ rank,
                     const int32_t* __restrict__ block_sums, const int32_t* __restrict__ total_ptr,
                     const float* __restrict__ scores, float* __restrict__ scan_scores) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  const int total = *total_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int b = batch_of(s_off, bo.batch, i);
    scan_scores[i] = scores[(int64_t)i + hit_prefix(rank, block_sums, n, total, s_off[b])];
  }
}

// mapmos_node.py:63-68: sqrt(sum((p - c)^2)) <= r in float64 (fp32 map promoted by the fp64 centre)
__global__ void __launch_bounds__(kScanBlock)
k_radius_rank(const float* __restrict__ xyz, const int32_t* __restrict__ n_ptr, double cx, double cy, double cz,
              double radius, int32_t* __restrict__ rank, int32_t* block_sums, uint32_t* ticket, int32_t* count_out) {
  const int n = *n_ptr;
  const int nb = max(1, (n + kScanBlock - 1) / kScanBlock);
  if ((int)blockIdx.x >= nb) return;
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  int flag = 0;
  if (i < n) {
    const double dx = __dsub_rn((double)xyz[(int64_t)i * 3 + 0], cx), dy = __dsub_rn((double)xyz[(int64_t)i * 3 + 1], cy),
                 dz = __dsub_rn((double)xyz[(int64_t)i * 3 + 2], cz);
    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    flag = __dsqrt_rn(d2) <= radius;
  }
  scan_flags(flag, i, n, nb, rank, block_sums, ticket, count_out);
}
__global__ void k_radius_write(const float* __restrict__ xyz, const int32_t* __restrict__ n_ptr, double cx, double cy,
                               double cz, double radius, const int32_t* __restrict__ rank,
                               const int32_t* __restrict__ block_sums, int32_t* __restrict__ out_idx) {
  const int n = *n_ptr;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const double dx = __dsub_rn((double)xyz[(int64_t)i * 3 + 0], cx), dy = __dsub_rn((double)xyz[(int64_t)i * 3 + 1], cy),
                 dz = __dsub_rn((double)xyz[(int64_t)i * 3 + 2], cz);
    const double d2 = __dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz));
    if (__dsqrt_rn(d2) <= radius) out_idx[rank[i] + block_sums[i / kScanBlock]] = i;
  }
}

// util.add_timestamp + vstack/hstack (util.py:156-174): [b, x,y,z, t], scan rows (t=1) then submap rows (t=0)
__global__ void k_assemble(const float* __restrict__ scan, int64_t n_scan, const float* __restrict__ sub,
                           const int32_t* __restrict__ n_sub_ptr, float b, float* __restrict__ out,
                           int32_t* __restrict__ n_total) {
  const int64_t n_sub = *n_sub_ptr;
  const int64_t n = n_scan + n_sub;
  if (n_total && blockIdx.x == 0 && threadIdx.x == 0) *n_total = (int32_t)n;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float* p = i < n_scan ? scan + i * 3 : sub + (i - n_scan) * 3;
    float* o = out + i * 5;
    o[0] = b; o[1] = p[0]; o[2] = p[1]; o[3] = p[2]; o[4] = i < n_scan ? 1.0f : 0.0f;
  }
}

}  // namespace sps

extern "C" size_t sps_map_bytes(int64_t max_points) {
  if (max_points < 1) max_points = 1;
  return carve_scratch(nullptr, max_points).bytes;
}

extern "C" int sps_map_build(sps_map** out, void* d_storage, size_t bytes, const float* d_map_xyz, int64_t n, float ds,
                             void* stream_) {
  if (!out || !d_storage || ((uintptr_t)d_storage & 255) || (!d_map_xyz && n > 0) || n < 0 || !(ds > 0.f))
    return SPS_ERR_BAD_ARG;
  Scratch s = carve_scratch(d_storage, n > 0 ? n : 1);
  if (s.bytes > bytes) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream_;
  SPS_CUDA_CHECK(cudaMemsetAsync(s.scalars, 0, 64 * 4, st));
  k_level_begin<<<grid_for(s.cap, 256), 256, 0, st>>>(s.table, nullptr, (int32_t)n, s.scalars + 0, nullptr, 0);
  k_insert_xyz<<<grid_for(n, 256), 256, 0, st>>>(d_map_xyz, s.scalars + 0, ds, s.table, nullptr, s.scalars + 40);
  SPS_CUDA_CHECK(cudaGetLastError());
  int32_t status = 0;
  SPS_CUDA_CHECK(cudaMemcpyAsync(&status, s.scalars + 40, 4, cudaMemcpyDeviceToHost, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  if (status & kStatusRange) return SPS_ERR_COORD_RANGE;
  sps_map* m = new sps_map();
  m->table = s.table; m->cap = s.cap; m->n = n; m->ds = ds; m->scalars = s.scalars;
  *out = m;
  return SPS_OK;
}

extern "C" int sps_map_destroy(sps_map* m) {
  delete m;
  return SPS_OK;
}

extern "C" int sps_submap_crop_voxel(const sps_map* map, const float* d_scan_xyz, int64_t n_scan, void* d_scratch,
                                     size_t scratch_bytes, float* d_out_xyz, int32_t* d_counts, void* stream_) {
  if (!map || (!d_scan_xyz && n_scan > 0) || n_scan < 0 || !d_scratch || ((uintptr_t)d_scratch & 255) ||
      !d_out_xyz || !d_counts)
    return SPS_ERR_BAD_ARG;
  const int64_t n = n_scan > 0 ? n_scan : 1;
  Scratch s = carve_scratch(d_scratch, n);
  if (s.bytes > scratch_bytes) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream_;
  SPS_CUDA_CHECK(cudaMemsetAsync(s.scalars, 0, 64 * 4, st));
  SPS_CUDA_CHECK(cudaMemsetAsync(d_counts, 0, 2 * 4, st));
  k_level_begin<<<grid_for(s.cap, 256), 256, 0, st>>>(s.table, nullptr, (int32_t)n_scan, s.scalars + 0, nullptr, 0);
  k_insert_xyz<<<grid_for(n, 256), 256, 0, st>>>(d_scan_xyz, s.scalars + 0, map->ds, s.table, s.slot_of,
                                                  s.scalars + 40);
  k_first_rank<<<cdiv(cdiv(n, kScanBlock), kRankChunks), kScanBlock, 0, st>>>(s.table, s.slot_of, s.scalars + 0, s.rank, s.block_sums,
                                                           (uint32_t*)(s.scalars + 32), d_counts + 0, map->table,
                                                           map->cap - 1, d_counts + 1);
  k_write_submap<<<grid_for(n, 256), 256, 0, st>>>(s.table, s.slot_of, s.scalars + 0, s.rank, s.block_sums,
                                                    map->table, map->cap - 1, map->ds, d_out_xyz);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" int sps_submap_crop_radius(const float* d_map_xyz, int64_t n, const double center[3], double radius,
                                      int32_t* d_out_idx, int32_t* d_count, void* d_scratch, size_t scratch_bytes,
                                      void* stream_) {
  if ((!d_map_xyz && n > 0) || n < 0 || !center || !d_out_idx || !d_count || !d_scratch ||
      ((uintptr_t)d_scratch & 255))
    return SPS_ERR_BAD_ARG;
  const int64_t nn = n > 0 ? n : 1;
  Scratch s = carve_scratch(d_scratch, nn);
  if (s.bytes > scratch_bytes) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream_;
  SPS_CUDA_CHECK(cudaMemsetAsync(s.scalars, 0, 64 * 4, st));
  k_set_i32<<<1, 1, 0, st>>>(s.scalars + 0, (int32_t)n);
  k_radius_rank<<<cdiv(nn, kScanBlock), kScanBlock, 0, st>>>(d_map_xyz, s.scalars + 0, center[0], center[1], center[2],
                                                             radius, s.rank, s.block_sums, (uint32_t*)(s.scalars + 32),
                                                             d_count);
  k_radius_write<<<grid_for(nn, 256), 256, 0, st>>>(d_map_xyz, s.scalars + 0, center[0], center[1], center[2], radius,
                                                    s.rank, s.block_sums, d_out_idx);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" int sps_assemble(const float* d_scan_xyz, int64_t n_scan, const float* d_sub_xyz, const int32_t* d_n_sub,
                            int64_t n_sub_max, float batch_index, float* d_out, void* stream_) {
  if ((!d_scan_xyz && n_scan > 0) || n_scan < 0 || n_sub_max < 0 || !d_n_sub || !d_out) return SPS_ERR_BAD_ARG;
  const int64_t n = n_scan + n_sub_max;
  if (n == 0) return SPS_OK;
  k_assemble<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream_>>>(d_scan_xyz, n_scan, d_sub_xyz, d_n_sub, batch_index,
                                                                  d_out, nullptr);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

namespace sps {
int forward_impl(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n_upper, const int32_t* d_n,
                 int64_t ld_points, float voxel_size, float* d_scores, int64_t n_scores, cudaStream_t st);
}

extern "C" size_t sps_infer_scan_scratch_bytes(int64_t n_scan) {
  if (n_scan < 1) n_scan = 1;
  // crop scratch + submap xyz [n_scan,3] + assembled rows [2*n_scan,5] + total-row scalar
  return sps_map_bytes(n_scan) + (((size_t)n_scan * 3 * 4 + 255) & ~size_t(255)) +
         (((size_t)n_scan * 2 * 5 * 4 + 255) & ~size_t(255)) + 256;
}

extern "C" int sps_infer_scan(sps_ctx* ctx, const sps_net* net, const sps_map* map, const float* d_scan_xyz,
                              int64_t n_scan, float voxel_size, float* d_scores, void* d_scratch, size_t scratch_bytes,
                              int32_t* d_counts, void* stream_) {
  if (!ctx || !net || !map || !d_scan_xyz || n_scan < 1 || !d_scores || !d_scratch || !d_counts ||
      ((uintptr_t)d_scratch & 255))
    return SPS_ERR_BAD_ARG;
  if (scratch_bytes < sps_infer_scan_scratch_bytes(n_scan)) return SPS_ERR_CAPACITY;
  if (2 * n_scan > ctx->max_points) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream_;
  char* p = (char*)d_scratch;
  const size_t crop_bytes = sps_map_bytes(n_scan);
  float* sub = (float*)(p + crop_bytes);
  float* rows = (float*)(p + crop_bytes + (((size_t)n_scan * 3 * 4 + 255) & ~size_t(255)));
  int32_t* n_total = (int32_t*)((char*)rows + (((size_t)n_scan * 2 * 5 * 4 + 255) & ~size_t(255)));
  int rc = sps_submap_crop_voxel(map, d_scan_xyz, n_scan, d_scratch, crop_bytes, sub, d_counts, stream_);
  if (rc != SPS_OK) return rc;
  k_assemble<<<grid_for(2 * n_scan, 256), 256, 0, st>>>(d_scan_xyz, n_scan, sub, d_counts + 0, 0.0f, rows, n_total);
  SPS_CUDA_CHECK(cudaGetLastError());
  return forward_impl(ctx, net, rows, 2 * n_scan, n_total, 5, voxel_size, d_scores, n_scan, st);
}

// ---- a batch of deployment scans: sps_submap_crop_voxel + util.infer's assembly per scan, collated ----
namespace sps {

// arguments shared by sps_prune_batch and sps_infer_prune_batch; fills `bo` and n_total
static int check_prune_args(const sps_map* map, const float* d_scans, int64_t ld, const int64_t* h_offsets, int batch,
                            const float* d_rows, const int32_t* d_row_offsets, const int32_t* d_n_rows,
                            const int32_t* d_counts, const void* d_scratch, size_t scratch_bytes, BatchOffsets& bo,
                            int64_t& n_total) {
  if (!map || !h_offsets || !d_rows || !d_row_offsets || !d_n_rows || !d_counts || !d_scratch ||
      ((uintptr_t)d_scratch & 255) || ld < 3 || batch < 1 || batch > kMaxBatch || h_offsets[0] != 0)
    return SPS_ERR_BAD_ARG;
  for (int b = 0; b < batch; ++b)
    if (h_offsets[b + 1] < h_offsets[b]) return SPS_ERR_BAD_ARG;
  n_total = h_offsets[batch];
  if (n_total > 0x3fffffff || (!d_scans && n_total > 0)) return SPS_ERR_BAD_ARG;   // rows (<= 2 n_total) index as int32
  if (scratch_bytes < carve_scratch(nullptr, n_total > 0 ? n_total : 1).bytes) return SPS_ERR_CAPACITY;
  bo.batch = batch;
  for (int b = 0; b <= batch; ++b) bo.off[b] = (int32_t)h_offsets[b];
  return SPS_OK;
}

// insert -> rank -> write on the scratch carve `s`; its kept-flag ranks, chunk sums and kept total (scalars[1]) stay
// valid for the score pass of the fused call
static int prune_batch_launch(const sps_map* map, const float* d_scans, int64_t ld, const BatchOffsets& bo, int n,
                              float* d_rows, int32_t* d_row_offsets, int32_t* d_n_rows, int32_t* d_counts,
                              const Scratch& s, cudaStream_t st) {
  const int nn = n > 0 ? n : 1;
  SPS_CUDA_CHECK(cudaMemsetAsync(s.scalars, 0, 64 * 4, st));
  SPS_CUDA_CHECK(cudaMemsetAsync(d_counts, 0, (size_t)bo.batch * 2 * 4, st));
  k_level_begin<<<grid_for(s.cap, 256), 256, 0, st>>>(s.table, nullptr, n, nullptr, nullptr, 0);
  k_prune_batch_insert<<<grid_for(nn, 256), 256, 0, st>>>(d_scans, ld, n, bo, map->ds, s.table, s.slot_of, s.scalars + 40);
  k_prune_batch_rank<<<cdiv(nn, kScanBlock), kScanBlock, 0, st>>>(s.table, s.slot_of, n, bo, map->table, map->cap - 1,
                                                                  s.rank, s.block_sums, (uint32_t*)(s.scalars + 32),
                                                                  s.scalars + 1, d_counts);
  k_prune_batch_write<<<grid_for(nn, 256), 256, 0, st>>>(d_scans, ld, n, bo, s.table, s.slot_of, s.rank, s.block_sums,
                                                         s.scalars + 1, map->ds, d_rows, d_row_offsets, d_n_rows, d_counts);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

}  // namespace sps

extern "C" size_t sps_prune_batch_scratch_bytes(int64_t n_scan_total, int batch) {
  (void)batch;   // the per-scan offsets travel as kernel arguments
  return carve_scratch(nullptr, n_scan_total > 0 ? n_scan_total : 1).bytes;
}

extern "C" int sps_prune_batch(const sps_map* map, const float* d_scans, int64_t ld, const int64_t* h_offsets, int batch,
                               float* d_rows, int32_t* d_row_offsets, int32_t* d_n_rows, int32_t* d_counts,
                               void* d_scratch, size_t scratch_bytes, void* stream) {
  BatchOffsets bo;
  int64_t n = 0;
  const int rc = check_prune_args(map, d_scans, ld, h_offsets, batch, d_rows, d_row_offsets, d_n_rows, d_counts, d_scratch,
                                  scratch_bytes, bo, n);
  if (rc != SPS_OK) return rc;
  return prune_batch_launch(map, d_scans, ld, bo, (int)n, d_rows, d_row_offsets, d_n_rows, d_counts,
                            carve_scratch(d_scratch, n > 0 ? n : 1), (cudaStream_t)stream);
}

extern "C" int sps_infer_prune_batch(sps_ctx* ctx, const sps_net* net, const sps_map* map, const float* d_scans, int64_t ld,
                                     const int64_t* h_offsets, int batch, float* d_rows, int32_t* d_row_offsets,
                                     int32_t* d_n_rows, int32_t* d_counts, void* d_scratch, size_t scratch_bytes,
                                     float voxel_size, float* d_scan_scores, void* stream) {
  if (!ctx || !net || !d_scan_scores || !(voxel_size > 0.f)) return SPS_ERR_BAD_ARG;
  BatchOffsets bo;
  int64_t n = 0;
  int rc = check_prune_args(map, d_scans, ld, h_offsets, batch, d_rows, d_row_offsets, d_n_rows, d_counts, d_scratch,
                            scratch_bytes, bo, n);
  if (rc != SPS_OK) return rc;
  if (2 * n > ctx->max_points) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream;
  const Scratch s = carve_scratch(d_scratch, n > 0 ? n : 1);
  rc = prune_batch_launch(map, d_scans, ld, bo, (int)n, d_rows, d_row_offsets, d_n_rows, d_counts, s, st);
  if (rc != SPS_OK) return rc;
  // SPSModel.forward on the rows (models.py:20-30): the launches are sized by 2 n, the row count stays on the device;
  // scores of every row land in the context's score buffer
  rc = forward_impl(ctx, net, d_rows, 2 * n, d_n_rows, 5, voxel_size, ctx->scores, 2 * n, st);
  if (rc != SPS_OK || n == 0) return rc;
  k_prune_batch_scores<<<grid_for(n, 256), 256, 0, st>>>((int)n, bo, s.rank, s.block_sums, s.scalars + 1, ctx->scores,
                                                        d_scan_scores);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

// ---- a batch of sensor-frame deployment scans: the ROS node's callback (sps_node.py:88-176) per scan, collated ----
// Per scan: the pose transform into the map frame (util.transform_point_cloud), util.prune + util.infer (the launches of
// sps_infer_prune_batch on the transformed scans), the node's metrics against column 3 and the published rows (score
// <= eps, sensor frame).  The partials are k_radius_partials (partials.cuh) on the prune layout, the published rows one
// compaction of the whole batch (k_filter_rank / k_filter_write, rosio.cuh): the scans are concatenated in order, so it
// is the per-scan compactions laid end to end.
namespace sps {

// point i -> the map frame with its scan's pose (transform_point, rosio.cuh); a run of threads reads the same 128 bytes
__global__ void __launch_bounds__(256)
k_transform_batch(const float* __restrict__ scan, int64_t ld, int n, const __grid_constant__ BatchOffsets bo,
                  const double* __restrict__ poses, float* __restrict__ xyz) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    transform_point(scan, ld, i, poses + 16 * batch_of(s_off, bo.batch, i), xyz);
}

// kept_off[b] = published rows of the scans before b: the filter's exclusive prefix at b's first point
__global__ void k_kept_offsets(int n, const __grid_constant__ BatchOffsets bo, const int32_t* __restrict__ rank,
                               const int32_t* __restrict__ block_sums, const int32_t* __restrict__ total_ptr,
                               int32_t* __restrict__ kept_off) {
  const int total = *total_ptr;
  for (int b = threadIdx.x; b <= bo.batch; b += blockDim.x) kept_off[b] = hit_prefix(rank, block_sums, n, total, bo.off[b]);
}

// scratch of the filter call: map-frame xyz [n, 3] | the prune carve | the filter's ranks, chunk sums, ticket line
// (ticket, kept total)
struct FilterCarve {
  float* xyz; Scratch prune; int32_t* rank; int32_t* block_sums; uint32_t* ticket; int32_t* total; size_t bytes;
};
static FilterCarve carve_filter(void* base, int64_t n) {
  FilterCarve c;
  char* p = (char*)base;
  size_t off = 0;
  auto take = [&](size_t b) { off = (off + 255) & ~size_t(255); char* r = p ? p + off : nullptr; off += b; return r; };
  c.xyz = (float*)take((size_t)n * 3 * 4);
  c.prune = carve_scratch(take(carve_scratch(nullptr, n).bytes), n);
  c.rank = (int32_t*)take((size_t)n * 4);
  c.block_sums = (int32_t*)take((size_t)(n / kScanBlock + 2) * 4);
  c.ticket = (uint32_t*)take(256);
  c.total = (int32_t*)(c.ticket + 1);
  c.bytes = (off + 255) & ~size_t(255);
  return c;
}

}  // namespace sps

extern "C" size_t sps_filter_scans_batch_scratch_bytes(int64_t n_scan_total, int batch) {
  (void)batch;   // the per-scan offsets travel as kernel arguments
  return carve_filter(nullptr, n_scan_total > 0 ? n_scan_total : 1).bytes;
}

extern "C" int sps_filter_scans_batch(sps_ctx* ctx, const sps_net* net, const sps_map* map, const float* d_scans, int64_t ld,
                                      const int64_t* h_offsets, int batch, const double* d_poses, float eps,
                                      float voxel_size, float* d_rows, int32_t* d_row_offsets, int32_t* d_n_rows,
                                      int32_t* d_counts, float* d_scan_scores, int64_t* d_metric_counts,
                                      double* d_metric_sums, float* d_kept, int32_t* d_kept_offsets, void* d_scratch,
                                      size_t scratch_bytes, void* stream) {
  if (!ctx || !net || !d_scan_scores || !d_poses || !d_metric_counts || !d_metric_sums || !d_kept || !d_kept_offsets ||
      ((uintptr_t)d_kept & 15) || ld < 4 || eps != eps || !(voxel_size > 0.f))
    return SPS_ERR_BAD_ARG;
  BatchOffsets bo;
  int64_t n = 0;
  int rc = check_prune_args(map, d_scans, ld, h_offsets, batch, d_rows, d_row_offsets, d_n_rows, d_counts, d_scratch,
                            scratch_bytes, bo, n);
  if (rc != SPS_OK) return rc;
  const FilterCarve c = carve_filter(d_scratch, n > 0 ? n : 1);
  if (scratch_bytes < c.bytes || 2 * n > ctx->max_points) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream;
  if (n > 0) {
    k_transform_batch<<<grid_for(n, 256), 256, 0, st>>>(d_scans, ld, (int)n, bo, d_poses, c.xyz);
    SPS_CUDA_CHECK(cudaGetLastError());
  }
  // sps_infer_prune_batch on the map-frame scans: the rows, then the forward on them (scores in the context's buffer)
  rc = prune_batch_launch(map, c.xyz, 3, bo, (int)n, d_rows, d_row_offsets, d_n_rows, d_counts, c.prune, st);
  if (rc != SPS_OK) return rc;
  rc = forward_impl(ctx, net, d_rows, 2 * n, d_n_rows, 5, voxel_size, ctx->scores, 2 * n, st);
  if (rc != SPS_OK) return rc;
  SPS_CUDA_CHECK(cudaMemsetAsync(d_metric_counts, 0, (size_t)batch * 4 * sizeof(int64_t), st));
  SPS_CUDA_CHECK(cudaMemsetAsync(d_metric_sums, 0, (size_t)batch * 5 * sizeof(double), st));
  if (n == 0) {
    SPS_CUDA_CHECK(cudaMemsetAsync(d_kept_offsets, 0, (size_t)(batch + 1) * 4, st));
    return SPS_OK;
  }
  // scan point i's row is i + K(off[b]) (the prune's kept-flag prefix); every row is scored (n_rows == n_fwd); the
  // labels are column 3 of the sensor-frame input
  const int per_block = 256 * kPartialsSpan;
  k_radius_partials<<<cdiv(n, per_block), 256, 0, st>>>(d_scans, ld, (int)n, bo, c.prune.rank, c.prune.block_sums,
                                                       c.prune.scalars + 1, d_n_rows, d_n_rows, ctx->scores, eps,
                                                       d_scan_scores, reinterpret_cast<unsigned long long*>(d_metric_counts),
                                                       d_metric_sums);
  // the published rows: sps_pointcloud2_pack over the whole batch, plus where each scan's rows start
  SPS_CUDA_CHECK(cudaMemsetAsync(c.ticket, 0, 256, st));
  k_filter_rank<<<cdiv(n, kScanBlock), kScanBlock, 0, st>>>(d_scan_scores, (int)n, eps, c.rank, c.block_sums, c.ticket,
                                                            c.total);
  k_filter_write<<<grid_for(n, 256, 148 * 16), 256, 0, st>>>(d_scans, ld, n, d_scan_scores, eps, c.rank, c.block_sums, d_kept);
  k_kept_offsets<<<1, 256, 0, st>>>((int)n, bo, c.rank, c.block_sums, c.total, d_kept_offsets);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}
