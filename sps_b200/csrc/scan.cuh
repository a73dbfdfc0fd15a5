// Grid-wide exclusive scan of one flag per input in a single launch (block scan + last-block-done carry), and the
// helpers of the batched calls that place every scan of a batch by such a scan.
#pragma once
#include "ctx.h"

namespace sps {

// Exclusive scan of one 0/1 flag per input over the whole grid: block scan (rank[i] = rank inside its chunk of kScanBlock
// inputs), per-chunk sums, and the last block to finish turns the sums into exclusive chunk offsets and publishes the
// total.  Global rank of i = rank[i] + block_sums[i / kScanBlock].
//
// scan_chunk: one chunk (every thread of the block calls it; a block may scan several chunks one after the other, which
// lets it issue the loads behind all its flags first and divides the number of tickets).  scan_finish: once per block after
// its last chunk, with nblocks = blocks that take part and nb = chunks in total.
__device__ __forceinline__ int scan_chunk(int flag, int i, int n, int chunk, int32_t* __restrict__ rank, int32_t* block_sums) {
  __shared__ int warp_sums[kScanBlock / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  int incl = flag;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    int v = __shfl_up_sync(0xffffffffu, incl, d);
    if (lane >= d) incl += v;
  }
  __syncthreads();                       // the previous chunk's readers of warp_sums are done
  if (lane == 31) warp_sums[wid] = incl;
  __syncthreads();
  if (wid == 0) {
    int w = lane < kScanBlock / 32 ? warp_sums[lane] : 0;
    int wi = w;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int v = __shfl_up_sync(0xffffffffu, wi, d);
      if (lane >= d) wi += v;
    }
    if (lane < kScanBlock / 32) warp_sums[lane] = wi - w;  // exclusive
  }
  __syncthreads();
  const int excl = incl - flag + warp_sums[wid];
  if (i < n) rank[i] = excl;
  if (tid == kScanBlock - 1) block_sums[chunk] = excl + flag;
  return excl;
}

__device__ __forceinline__ void scan_finish(int nb, int nblocks, int32_t* block_sums, uint32_t* ticket, int32_t* count_out) {
  __shared__ int warp_sums[kScanBlock / 32];
  __shared__ bool is_last;
  __shared__ int carry;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  if (tid == kScanBlock - 1) {           // the thread that wrote this block's chunk sums
    __threadfence();
    is_last = (atomicAdd(ticket, 1u) == (uint32_t)(nblocks - 1));
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // serial-over-chunks exclusive scan of block_sums[0..nb) by this block
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int base = 0; base < nb; base += kScanBlock) {
    const int j = base + tid;
    const int v = (j < nb) ? ((volatile int32_t*)block_sums)[j] : 0;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, inc, d);
      if (lane >= d) inc += u;
    }
    if (lane == 31) warp_sums[wid] = inc;
    __syncthreads();
    if (wid == 0) {
      int w = lane < kScanBlock / 32 ? warp_sums[lane] : 0;
      int wi = w;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        int u = __shfl_up_sync(0xffffffffu, wi, d);
        if (lane >= d) wi += u;
      }
      if (lane < kScanBlock / 32) warp_sums[lane] = wi - w;
    }
    __syncthreads();
    const int ex = inc - v + warp_sums[wid] + carry;
    if (j < nb) block_sums[j] = ex;
    __syncthreads();
    if (tid == kScanBlock - 1) carry = ex + v;
    __syncthreads();
  }
  if (tid == 0) {
    *count_out = carry;
    *ticket = 0;  // ready for the next scan on this stream
  }
}

// one chunk per block (blockIdx.x = chunk): must be called by every thread of every block with blockIdx.x < nb
__device__ __forceinline__ int scan_flags(int flag, int i, int n, int nb, int32_t* __restrict__ rank, int32_t* block_sums,
                                 uint32_t* ticket, int32_t* count_out) {
  const int excl = scan_chunk(flag, i, n, blockIdx.x, rank, block_sums);
  scan_finish(nb, nb, block_sums, ticket, count_out);
  return excl;
}

// ---- batches of B scans concatenated: scan b = inputs off[b] .. off[b+1] ----
constexpr int kMaxBatch = 255;     // the batch index is the voxel key's 8-bit b field (255 is reserved)
struct BatchOffsets { int32_t off[kMaxBatch + 1]; int batch; };   // by value: no copy, no host synchronisation

__device__ __forceinline__ void load_offsets(const BatchOffsets& bo, int32_t* s_off) {
  for (int j = threadIdx.x; j <= bo.batch; j += blockDim.x) s_off[j] = bo.off[j];
  __syncthreads();
}
// scan of point i: the last b with off[b] <= i (empty scans never own a point)
__device__ __forceinline__ int batch_of(const int32_t* s_off, int batch, int i) {
  int lo = 0, hi = batch;
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (s_off[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}
// global exclusive prefix of the scanned flags (or counts) at input j (j == n: the total)
__device__ __forceinline__ int hit_prefix(const int32_t* __restrict__ rank, const int32_t* __restrict__ block_sums, int n,
                                          int total, int j) {
  return j < n ? rank[j] + block_sums[j / kScanBlock] : total;
}


}  // namespace sps
