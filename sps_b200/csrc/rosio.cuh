// Per-point arithmetic of the ROS deployment path shared by the single-scan entry points (rosio.cu) and the batched
// filter call (maps.cu): the sensor -> map frame transform and the threshold filter of the published cloud.  The kernels
// are static, so every translation unit that includes this header gets its own copy.
#pragma once
#include "ctx.h"
#include "scan.cuh"

namespace sps {

// util.transform_point_cloud: homogeneous coordinates in float64 (the fp32 cloud is promoted by the float64 matrix),
// np.dot(h, T.T), division by the homogeneous coordinate, then torch.tensor(..., dtype=float32) (sps_node.py:106).
// Point i of xyz (row stride ld) -> out[i * 3 .. i * 3 + 3); T: the row-major 4x4 matrix.
struct Mat4 { double m[16]; };
__device__ __forceinline__ void transform_point(const float* __restrict__ xyz, int64_t ld, int64_t i, const double* T,
                                                float* __restrict__ out) {
  const double x = xyz[i * ld + 0], y = xyz[i * ld + 1], z = xyz[i * ld + 2];
  double r[4];
#pragma unroll
  for (int j = 0; j < 4; ++j)   // row j of T against (x, y, z, 1): the fused multiply-add chain of numpy's dgemm on an
    // FMA machine (OpenBLAS / MKL on x86-64: x*T0, then fma(y,T1,.), fma(z,T2,.), fma(1,T3,.)) -- verified against
    // np.dot with exact rational arithmetic, 9000 of 9000 float64 values identical (tests/test_rosio.py)
    r[j] = __dadd_rn(__fma_rn(z, T[4 * j + 2], __fma_rn(y, T[4 * j + 1], __dmul_rn(x, T[4 * j + 0]))), T[4 * j + 3]);
  out[i * 3 + 0] = (float)__ddiv_rn(r[0], r[3]);
  out[i * 3 + 1] = (float)__ddiv_rn(r[1], r[3]);
  out[i * 3 + 2] = (float)__ddiv_rn(r[2], r[3]);
}

// sps_node.py:148: keep the scan rows whose score is <= epsilon (NaN scores are dropped, as the comparison is false)
static __global__ void __launch_bounds__(kScanBlock)
k_filter_rank(const float* __restrict__ scores, int n, float eps, int32_t* __restrict__ rank, int32_t* block_sums, uint32_t* ticket,
              int32_t* count_out) {
  const int nb = max(1, (n + kScanBlock - 1) / kScanBlock);
  if ((int)blockIdx.x >= nb) return;
  const int i = blockIdx.x * kScanBlock + threadIdx.x;
  scan_flags(i < n && scores[i] <= eps, i, n, nb, rank, block_sums, ticket, count_out);
}
static __global__ void k_filter_write(const float* __restrict__ scan, int64_t ld, int64_t n, const float* __restrict__ scores, float eps,
                                      const int32_t* __restrict__ rank, const int32_t* __restrict__ block_sums, float* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    if (!(scores[i] <= eps)) continue;
    const int64_t o = rank[i] + block_sums[i / kScanBlock];
    const float* r = scan + i * ld;
    *reinterpret_cast<float4*>(out + o * 4) = make_float4(r[0], r[1], r[2], r[3]);    // point_step 16: x, y, z, intensity
  }
}

}  // namespace sps
