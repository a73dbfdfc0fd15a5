// Per-scan metric partials of a batch of scored scans, shared by the batched calls of ballquery.cu and maps.cu.  The
// kernel is static, so every translation unit that includes this header gets its own copy.
#pragma once
#include "ctx.h"
#include "scan.cuh"

namespace sps {

// ---- per-scan metric partials of the fused call (k_confusion's arithmetic, api.cu) ----
// One pass over the scan points: each reads its score at its row position, writes it compacted, and adds to the
// partials of its scan.  A warp walks kPartialsSpan x 32 consecutive points and keeps per-lane partials while all its
// lanes are in one scan; at a scan boundary it flushes them and adds that iteration with a segmented warp reduction.
constexpr int kPartialsSpan = 16;

struct Partials {
  unsigned long long c[4];
  double s[5];
};
__device__ __forceinline__ void partials_add(Partials& a, float sc, float lb, float eps) {
  const int p = sc < eps ? 0 : 1, gt = lb < eps ? 0 : 1;
  const int k = (gt == 1 && p == 1) ? 0 : (gt == 0 && p == 0) ? 1 : (gt == 0 && p == 1) ? 2 : 3;
#pragma unroll
  for (int j = 0; j < 4; ++j) a.c[j] += j == k;        // (no dynamic index: the partials stay in registers)
  const double e = (double)sc - (double)lb;
  a.s[0] += 1.0; a.s[1] += e * e; a.s[2] += lb; a.s[3] += (double)lb * lb; a.s[4] += sc;
}
__device__ __forceinline__ void partials_atomic(const Partials& a, int b, unsigned long long* counts, double* sums) {
#pragma unroll
  for (int j = 0; j < 4; ++j) if (a.c[j]) atomicAdd(counts + b * 4 + j, a.c[j]);
#pragma unroll
  for (int j = 0; j < 5; ++j) if (a.s[j] != 0.0) atomicAdd(sums + b * 5 + j, a.s[j]);
}
// sum over the lanes holding the same b (b non-decreasing along the lanes): the first lane of each run gets its total
__device__ __forceinline__ void partials_segmented_sum(Partials& a, int b) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int bo = __shfl_down_sync(0xffffffffu, b, d);
    const bool take = lane + d < 32 && bo == b;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const unsigned long long v = __shfl_down_sync(0xffffffffu, a.c[j], d);
      if (take) a.c[j] += v;
    }
#pragma unroll
    for (int j = 0; j < 5; ++j) {
      const double v = __shfl_down_sync(0xffffffffu, a.s[j], d);
      if (take) a.s[j] += v;
    }
  }
}

static __global__ void __launch_bounds__(256)
k_radius_partials(const float* __restrict__ scan, int64_t ld, int n, const __grid_constant__ BatchOffsets bo, const int32_t* __restrict__ rank,
                  const int32_t* __restrict__ block_sums, const int32_t* __restrict__ total_ptr,
                  const int32_t* __restrict__ n_rows, const int32_t* __restrict__ n_fwd, const float* __restrict__ scores,
                  float eps, float* __restrict__ scan_scores, unsigned long long* counts, double* sums) {
  __shared__ int32_t s_off[kMaxBatch + 1];
  load_offsets(bo, s_off);
  const int total = *total_ptr;
  const bool scored = *n_fwd == *n_rows;       // else the rows did not fit and the forward ran on none of them
  const int lane = threadIdx.x & 31;
  const int64_t w0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x - lane) * kPartialsSpan;
  Partials acc = {};
  int wb = -1;                                 // scan of the per-lane partials in `acc` (warp-uniform)
  for (int it = 0; it < kPartialsSpan; ++it) {
    const int64_t base = w0 + it * 32;
    if (base >= n) break;
    const int i = (int)base + lane;
    const bool in = i < n;
    const int b = in ? batch_of(s_off, bo.batch, i) : kMaxBatch + 1;   // past-the-end lanes: a run of their own
    float sc = nanf(""), lb = 0.f;
    if (in) {
      lb = scan[(int64_t)i * ld + 3];
      if (scored) sc = scores[(int64_t)i + hit_prefix(rank, block_sums, n, total, s_off[b])];
      scan_scores[i] = sc;
    }
    if (!scored) continue;
    if (__all_sync(0xffffffffu, b == wb || !in)) {
      if (in) partials_add(acc, sc, lb, eps);
      continue;
    }
    if (wb >= 0) {                             // flush the running partials of scan wb
      partials_segmented_sum(acc, wb);
      if (lane == 0) partials_atomic(acc, wb, counts, sums);
    }
    Partials one = {};
    if (in) partials_add(one, sc, lb, eps);
    partials_segmented_sum(one, b);
    const int bprev = __shfl_up_sync(0xffffffffu, b, 1);
    if (in && (lane == 0 || bprev != b)) partials_atomic(one, b, counts, sums);
    acc = Partials{};
    wb = __shfl_sync(0xffffffffu, b, 31);
  }
  if (wb >= 0 && wb <= kMaxBatch) {
    partials_segmented_sum(acc, wb);
    if (lane == 0) partials_atomic(acc, wb, counts, sums);
  }
}

}  // namespace sps
