// Per-scan host work of the ROS deployment path moved to the device (SURVEY.md §8f rank 3):
//   * PointCloud2 payload -> fp32 [n, fields]          util.to_numpy            (src/sps/datasets/util.py:146-153)
//   * sensor frame -> map frame, SE(3) in float64      util.transform_point_cloud (util.py:187-194; sps_node.py:103-107)
//   * threshold filter + PointCloud2 payload           sps_node.py:148-149 + util.to_rosmsg (util.py:117-143)
// All three are byte / elementwise work bound by HBM; the scan (57 600 x 16 bytes) is a few hundred KB, so the point of
// these kernels is to keep the streamed path free of host round trips, not bandwidth.
#include "ctx.h"
#include "rosio.cuh"

namespace sps {

// sensor_msgs/PointField datatypes
enum { kPfInt8 = 1, kPfUint8 = 2, kPfInt16 = 3, kPfUint16 = 4, kPfInt32 = 5, kPfUint32 = 6, kPfFloat32 = 7, kPfFloat64 = 8 };
constexpr int kMaxFields = 16;

struct FieldTable {
  int32_t offset[kMaxFields];
  int32_t datatype[kMaxFields];
  int nfields;
};

__device__ __forceinline__ float read_field(const uint8_t* p, int datatype, bool swap) {
  uint8_t b[8];
  const int size = datatype == kPfFloat64 ? 8 : (datatype >= kPfInt32 ? 4 : (datatype >= kPfInt16 ? 2 : 1));
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < size) b[i] = p[swap ? size - 1 - i : i];      // little-endian value bytes (fields may be unaligned)
  switch (datatype) {
    case kPfInt8: return (float)(int8_t)b[0];
    case kPfUint8: return (float)b[0];
    case kPfInt16: return (float)(int16_t)((uint16_t)b[0] | ((uint16_t)b[1] << 8));
    case kPfUint16: return (float)((uint16_t)b[0] | ((uint16_t)b[1] << 8));
    case kPfInt32: return (float)(int32_t)((uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24));
    case kPfUint32: return (float)((uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24));
    case kPfFloat32: return __uint_as_float((uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24));
    default: {
      unsigned long long u = 0;
#pragma unroll
      for (int i = 0; i < 8; ++i) u |= (unsigned long long)b[i] << (8 * i);
      return (float)__longlong_as_double((long long)u);     // numpy's float64 -> float32 assignment: round to nearest
    }
  }
}

// util.to_numpy: scan[:, i] = np.resize(pc[field_i], height * width) -- every field cast to float32, fields in message order
__global__ void k_pc2_unpack(const uint8_t* __restrict__ data, int64_t width, int64_t height, int64_t point_step, int64_t row_step,
                             const FieldTable ft, int swap, float* __restrict__ out) {
  const int64_t n = width * height;
  const int64_t total = n * ft.nfields;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = idx / ft.nfields;
    const int f = (int)(idx - p * ft.nfields);
    const int64_t row = p / width, col = p - row * width;
    out[idx] = read_field(data + row * row_step + col * point_step + ft.offset[f], ft.datatype[f], swap != 0);
  }
}

// util.transform_point_cloud on one scan (transform_point, rosio.cuh)
__global__ void k_transform_points(const float* __restrict__ xyz, int64_t ld, int64_t n, const Mat4 T, float* __restrict__ out) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    transform_point(xyz, ld, i, T.m, out);
}

// sps_node.py:148's threshold filter: k_filter_rank / k_filter_write (rosio.cuh)

}  // namespace sps

using namespace sps;

extern "C" int sps_pointcloud2_unpack(const void* d_data, int64_t width, int64_t height, int64_t point_step, int64_t row_step,
                                      int nfields, const int32_t* h_offsets, const int32_t* h_datatypes, int is_bigendian,
                                      float* d_out, void* stream) {
  if (!d_out || width < 0 || height < 0 || point_step < 1 || row_step < 0 || nfields < 1 || nfields > kMaxFields || !h_offsets ||
      !h_datatypes)
    return SPS_ERR_BAD_ARG;
  if (width * height == 0) return SPS_OK;
  if (!d_data || row_step < width * point_step) return SPS_ERR_BAD_ARG;
  FieldTable ft;
  ft.nfields = nfields;
  for (int f = 0; f < nfields; ++f) {
    const int dt = h_datatypes[f];
    if (dt < kPfInt8 || dt > kPfFloat64) return SPS_ERR_BAD_ARG;
    const int size = dt == kPfFloat64 ? 8 : (dt >= kPfInt32 ? 4 : (dt >= kPfInt16 ? 2 : 1));
    if (h_offsets[f] < 0 || h_offsets[f] + size > point_step) return SPS_ERR_BAD_ARG;
    ft.offset[f] = h_offsets[f];
    ft.datatype[f] = dt;
  }
  const int64_t total = width * height * nfields;
  int64_t g = (total + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  k_pc2_unpack<<<(int)g, 256, 0, (cudaStream_t)stream>>>(static_cast<const uint8_t*>(d_data), width, height, point_step, row_step, ft,
                                                          is_bigendian, d_out);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" int sps_transform_points(const float* d_xyz, int64_t ld, int64_t n, const double* h_matrix, float* d_out, void* stream) {
  if (n < 0 || ld < 3 || !h_matrix || (n > 0 && (!d_xyz || !d_out))) return SPS_ERR_BAD_ARG;
  if (n == 0) return SPS_OK;
  Mat4 T;
  for (int i = 0; i < 16; ++i) T.m[i] = h_matrix[i];
  int64_t g = (n + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  k_transform_points<<<(int)g, 256, 0, (cudaStream_t)stream>>>(d_xyz, ld, n, T, d_out);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" size_t sps_pointcloud2_pack_scratch_bytes(int64_t n) {
  if (n < 1) n = 1;
  // rank [n] + block sums + ticket line
  return (((size_t)n * 4 + 255) & ~size_t(255)) + ((((size_t)n / kScanBlock + 2) * 4 + 255) & ~size_t(255)) + 256;
}

extern "C" int sps_pointcloud2_pack(const float* d_scan, int64_t ld, int64_t n, const float* d_scores, float eps, float* d_out,
                                    int32_t* d_count, void* d_scratch, size_t scratch_bytes, void* stream) {
  if (n < 0 || ld < 4 || !d_count || !d_scratch || ((uintptr_t)d_scratch & 255) || (n > 0 && (!d_scan || !d_scores || !d_out)))
    return SPS_ERR_BAD_ARG;
  if (n > INT32_MAX) return SPS_ERR_CAPACITY;
  if (scratch_bytes < sps_pointcloud2_pack_scratch_bytes(n)) return SPS_ERR_CAPACITY;
  if ((uintptr_t)d_out & 15) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  char* p = static_cast<char*>(d_scratch);
  int32_t* rank = reinterpret_cast<int32_t*>(p);
  p += ((size_t)(n > 0 ? n : 1) * 4 + 255) & ~size_t(255);
  int32_t* block_sums = reinterpret_cast<int32_t*>(p);
  p += (((size_t)n / kScanBlock + 2) * 4 + 255) & ~size_t(255);
  uint32_t* ticket = reinterpret_cast<uint32_t*>(p);
  SPS_CUDA_CHECK(cudaMemsetAsync(ticket, 0, 256, st));
  SPS_CUDA_CHECK(cudaMemsetAsync(d_count, 0, 4, st));
  if (n == 0) return SPS_OK;
  const int nb = (int)((n + kScanBlock - 1) / kScanBlock);
  k_filter_rank<<<nb, kScanBlock, 0, st>>>(d_scores, (int)n, eps, rank, block_sums, ticket, d_count);
  int64_t g = (n + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  k_filter_write<<<(int)g, 256, 0, st>>>(d_scan, ld, n, d_scores, eps, rank, block_sums, d_out);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}
