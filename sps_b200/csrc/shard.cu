// Reassembly of per-rank result blocks in sequence order (parallel.ShardedScans).  After a gather, rank r's rows sit in
// block r of a [world][cap][width] buffer; batch k of a sequence ran on rank k mod world and wrote its rows at a
// host-known start of that rank's block, but how many rows it wrote (the published rows of a replay call) may be known
// on the device only.  One launch per kSegChunk segments scans the device lengths and copies every segment to its place
// in sequence order, with no host synchronisation.
#include "ctx.h"
#include "scan.cuh"

namespace sps {

constexpr int kSegChunk = 1024;    // segments per launch: their table travels as a kernel argument (12 KB)
struct SegmentChunk {
  int64_t src[kSegChunk];          // first source row of the segment: rank * cap + start
  int32_t room[kSegChunk];         // the most rows the segment may hold
  int first, count;                // segments first .. first + count - 1
};

// Every block scans the chunk's lengths (clamped to 0 .. room) into shared memory, kScanBlock at a time, on top of the
// rows of the segments before the chunk (out_off[first], written by the previous chunk's launch); block 0 publishes the
// offsets.  Then each thread copies whole output rows, upr units of V each (float4 where rows and pointers allow):
// output row -> segment by binary search in shared memory -> source row.
template <typename V>
__global__ void __launch_bounds__(kScanBlock)
k_gather_segments(const V* __restrict__ src, int upr, const __grid_constant__ SegmentChunk sc,
                  const int32_t* __restrict__ len, V* __restrict__ out, int32_t* __restrict__ out_off) {
  __shared__ int32_t s_off[kSegChunk + 1];
  __shared__ int32_t s_sum;
  const int carry = sc.first ? out_off[sc.first] : 0;
  int run = 0;
  for (int base = 0; base < sc.count; base += kScanBlock) {
    const int s = base + threadIdx.x;
    int l = 0;
    if (s < sc.count) {
      l = len[sc.first + s];
      l = l < 0 ? 0 : (l > sc.room[s] ? sc.room[s] : l);
    }
    // n = 0: no per-input store, only the exclusive prefix inside this chunk and the chunk's sum (into s_sum)
    const int excl = scan_chunk(l, 0, 0, 0, nullptr, &s_sum);
    if (s < sc.count) s_off[s] = carry + run + excl;
    __syncthreads();
    run += s_sum;        // read before the next scan_chunk's first barrier; its last thread writes s_sum after two more
  }
  if (threadIdx.x == 0) s_off[sc.count] = carry + run;
  __syncthreads();
  if (blockIdx.x == 0)
    for (int s = threadIdx.x; s <= sc.count; s += blockDim.x) out_off[sc.first + s] = s_off[s];
  const int end = s_off[sc.count];
  for (int row = s_off[0] + blockIdx.x * blockDim.x + threadIdx.x; row < end; row += gridDim.x * blockDim.x) {
    const int s = batch_of(s_off, sc.count, row);
    const V* from = src + (sc.src[s] + (row - s_off[s])) * upr;
    V* to = out + (int64_t)row * upr;
    for (int c = 0; c < upr; ++c) to[c] = from[c];
  }
}

}  // namespace sps

using namespace sps;

extern "C" int sps_gather_segments(const float* d_src, int world, int64_t cap, int width, int n_seg,
                                   const int32_t* h_seg_rank, const int64_t* h_seg_start, const int64_t* h_seg_rows,
                                   const int32_t* d_seg_len, float* d_out, int64_t out_capacity, int32_t* d_out_offsets,
                                   void* stream) {
  if (world < 1 || cap < 0 || width < 1 || n_seg < 0 || out_capacity < 0 || !d_out_offsets ||
      ((uintptr_t)d_out_offsets & 3) || ((uintptr_t)d_src & 3) || ((uintptr_t)d_out & 3) || ((uintptr_t)d_seg_len & 3))
    return SPS_ERR_BAD_ARG;
  if (cap > (INT64_MAX / 16) / world / width) return SPS_ERR_BAD_ARG;
  if (n_seg > 0 && (!h_seg_rank || !h_seg_start || !h_seg_rows || !d_seg_len)) return SPS_ERR_BAD_ARG;
  int64_t rows = 0;                  // upper bound of the output: every segment full
  for (int s = 0; s < n_seg; ++s) {
    if (h_seg_rank[s] < 0 || h_seg_rank[s] >= world || h_seg_start[s] < 0 || h_seg_rows[s] < 0 ||
        h_seg_rows[s] > cap - h_seg_start[s])
      return SPS_ERR_BAD_ARG;
    rows += h_seg_rows[s];
    if (rows > INT32_MAX) return SPS_ERR_BAD_ARG;          // the offsets are int32
  }
  if (rows > 0 && !d_src) return SPS_ERR_BAD_ARG;
  if (out_capacity < rows) return SPS_ERR_CAPACITY;
  if (rows > 0 && !d_out) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = width % 4 == 0 && !((uintptr_t)d_src & 15) && !((uintptr_t)d_out & 15);
  const int upr = vec ? width / 4 : width;
  SegmentChunk sc;
  for (int first = 0; first == 0 || first < n_seg; first += kSegChunk) {
    sc.first = first;
    sc.count = n_seg - first < kSegChunk ? n_seg - first : kSegChunk;
    int64_t bound = 0;
    for (int s = 0; s < sc.count; ++s) {
      sc.src[s] = h_seg_rank[first + s] * cap + h_seg_start[first + s];
      sc.room[s] = (int32_t)h_seg_rows[first + s];
      bound += h_seg_rows[first + s];
    }
    int64_t g = (bound + kScanBlock - 1) / kScanBlock;
    g = g < 1 ? 1 : (g > 148 * 8 ? 148 * 8 : g);
    if (vec)
      k_gather_segments<float4><<<(int)g, kScanBlock, 0, st>>>(reinterpret_cast<const float4*>(d_src), upr, sc, d_seg_len,
                                                               reinterpret_cast<float4*>(d_out), d_out_offsets);
    else
      k_gather_segments<float><<<(int)g, kScanBlock, 0, st>>>(d_src, upr, sc, d_seg_len, d_out, d_out_offsets);
    SPS_CUDA_CHECK(cudaGetLastError());
  }
  return SPS_OK;
}
