// Shared device helpers: voxel key packing, open-addressing hash slots, status flags.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include "../../include/sps_b200.h"

namespace sps {

// ---- activation storage of the fused forward ----
// mode 0: fp32 as computed; 1: fp32 rounded to TF32 (nearest), so a tensor-core consumer does not truncate;
// 2: fp16 rows (`out` then points at __half, out_ld counts halves) -- same 10-bit mantissa as TF32, half the
// bytes per gathered row; saturating conversion (|x| > 65504 -> +-65504).
// mode 3: fp16 hi|lo pairs -- per 8 channels 16 halves [fp16(v) x 8 | fp16(v - hi) x 8], ~21 bits per value; the consumer
// contracts such a row as 2 x 8 fp16 channels against weights duplicated along K (exact products, fp32 accumulation).
enum { kStoreF32 = 0, kStoreTF32 = 1, kStoreF16 = 2, kStoreF16x2 = 3 };
__device__ __forceinline__ uint32_t pack_half2_sat(float a, float b) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));   // low half = a
  return r;
}
__device__ __forceinline__ void store_row8(float* out, int64_t out_ld, int64_t row, const float (&v)[8], int mode) {
  if (mode == kStoreF16x2) {
    // `out` already points at the 16-half slot of this channel group inside the (doubled) row
    __half* op = reinterpret_cast<__half*>(out) + row * out_ld;
    float lo[8];
    uint32_t hi[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      hi[j] = pack_half2_sat(v[2 * j], v[2 * j + 1]);
      const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi[j]));
      lo[2 * j] = v[2 * j] - h.x;          // exact in fp32 (unless hi saturated: then lo saturates too)
      lo[2 * j + 1] = v[2 * j + 1] - h.y;
    }
    *reinterpret_cast<uint4*>(op) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(op + 8) = make_uint4(pack_half2_sat(lo[0], lo[1]), pack_half2_sat(lo[2], lo[3]),
                                                   pack_half2_sat(lo[4], lo[5]), pack_half2_sat(lo[6], lo[7]));
  } else if (mode == kStoreF16) {
    __half* op = reinterpret_cast<__half*>(out) + row * out_ld;
    *reinterpret_cast<uint4*>(op) = make_uint4(pack_half2_sat(v[0], v[1]), pack_half2_sat(v[2], v[3]),
                                               pack_half2_sat(v[4], v[5]), pack_half2_sat(v[6], v[7]));
  } else {
    float w[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      w[c] = v[c];
      if (mode == kStoreTF32) {
        uint32_t r;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v[c]));
        w[c] = __uint_as_float(r);
      }
    }
    float* op = out + row * out_ld;
    *reinterpret_cast<float4*>(op) = make_float4(w[0], w[1], w[2], w[3]);
    *reinterpret_cast<float4*>(op + 4) = make_float4(w[4], w[5], w[6], w[7]);
  }
}

// ---- 64-bit voxel key: b:8 | x:18 | y:18 | z:16 | t:4 (biased; see include/sps_b200.h) ----
constexpr int kTBits = 4, kZBits = 16, kYBits = 18, kXBits = 18, kBBits = 8;
constexpr int kZShift = kTBits, kYShift = kZShift + kZBits, kXShift = kYShift + kYBits,
              kBShift = kXShift + kXBits;
constexpr unsigned long long kEmptyKey = 0xFFFFFFFFFFFFFFFFull;
constexpr int kXBias = SPS_X_BIAS, kZBias = SPS_Z_BIAS;

__host__ __device__ inline bool coord_in_range(int b, int x, int y, int z, int t) {
  return (unsigned)b < 255u && (unsigned)(x + kXBias) < (1u << kXBits) &&
         (unsigned)(y + kXBias) < (1u << kYBits) && (unsigned)(z + kZBias) < (1u << kZBits) &&
         (unsigned)t < (1u << kTBits);
}
__host__ __device__ inline unsigned long long pack_key(int b, int x, int y, int z, int t) {
  return ((unsigned long long)(unsigned)b << kBShift) |
         ((unsigned long long)(unsigned)(x + kXBias) << kXShift) |
         ((unsigned long long)(unsigned)(y + kXBias) << kYShift) |
         ((unsigned long long)(unsigned)(z + kZBias) << kZShift) | (unsigned long long)(unsigned)t;
}
__host__ __device__ inline void unpack_key(unsigned long long k, int& b, int& x, int& y, int& z, int& t) {
  b = (int)(k >> kBShift);
  x = (int)((k >> kXShift) & ((1u << kXBits) - 1)) - kXBias;
  y = (int)((k >> kYShift) & ((1u << kYBits) - 1)) - kXBias;
  z = (int)((k >> kZShift) & ((1u << kZBits) - 1)) - kZBias;
  t = (int)(k & ((1u << kTBits) - 1));
}
// floor(x / m) * m on every spatial field for m = 2^log2m (biases are multiples of 16).
__host__ __device__ inline unsigned long long coarsen_key(unsigned long long k, int log2m) {
  unsigned long long low = (1ull << log2m) - 1;
  unsigned long long mask = ~((low << kXShift) | (low << kYShift) | (low << kZShift));
  return k & mask;
}
// index of a fine voxel inside its 2x2x2 parent: ox + 2*oy + 4*oz (ME offset order, x fastest)
__host__ __device__ inline int child_index(unsigned long long k, int log2s) {
  int ox = (int)(k >> (kXShift + log2s)) & 1, oy = (int)(k >> (kYShift + log2s)) & 1,
      oz = (int)(k >> (kZShift + log2s)) & 1;
  return ox + 2 * oy + 4 * oz;
}

// ---- hash table ----
struct __align__(16) Slot {
  unsigned long long key;
  int val;    // voxel tables: block-local rank of the first occurrence (k_first_rank); block tables: block id
  int first;  // smallest input index that mapped here (first-occurrence order)
};

__host__ __device__ inline uint32_t hash_key(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (uint32_t)k;
}
// table capacity for n keys: smallest power of two >= max(1024, 1.5 n) -- load factor <= 0.67 if every key is distinct
// (linear probing: ~2.5 probes per miss at that load), in practice 0.2-0.45 (2.3 input rows per voxel on the bench scans).
// 2n would double the table: 134 MB instead of 67 MB for the 2.47 M-row batch, i.e. past the 126 MB L2.
__host__ __device__ inline uint32_t table_capacity(int64_t n) {
#ifdef __CUDA_ARCH__
  const unsigned long long need = ((unsigned long long)n * 3 + 1) / 2;
  return need <= 1024ull ? 1024u : 1u << (64 - __clzll((long long)(need - 1)));
#else
  uint32_t c = 1024;
  while ((int64_t)c * 2 < n * 3) c <<= 1;
  return c;
#endif
}

__device__ inline int table_find(const Slot* __restrict__ tab, uint32_t mask, unsigned long long key) {
  uint32_t s = hash_key(key) & mask;
  while (true) {
    // one 16-byte load per probe: key + val in the same sector
    const int4 raw = __ldg(reinterpret_cast<const int4*>(tab + s));
    unsigned long long k = ((unsigned long long)(unsigned)raw.y << 32) | (unsigned)raw.x;
    if (k == key) return raw.z;
    if (k == kEmptyKey) return -1;
    s = (s + 1) & mask;
  }
}

// threads per block of the grid-wide scans: small enough (512 x ~31 registers) to co-run with another lane's convolution CTAs
constexpr int kScanBlock = 512;

// returns the slot index of `key` (inserting it if absent)
__device__ inline uint32_t table_insert(Slot* tab, uint32_t mask, unsigned long long key) {
  uint32_t s = hash_key(key) & mask;
  while (true) {
    unsigned long long prev = atomicCAS(&tab[s].key, kEmptyKey, key);
    if (prev == kEmptyKey || prev == key) return s;
    s = (s + 1) & mask;
  }
}

// Insert `key` and lower the slot's `first` to `i` (first-occurrence index).  Most rows find their voxel already in the table
// (2-3 input rows per voxel, 2-8 fine voxels per coarse one): one 16-byte L2 read of the slot answers both questions, and
// the two atomics are only issued when they can change something (`first` only ever decreases, so a stale read is safe).
// `s` / `raw`: the home slot and its content as read by the caller (callers issue the reads of several rows back to back: the
// insert kernels are bound by the latency of this first random access, not by atomics or bandwidth).
__device__ inline uint32_t table_insert_first(Slot* tab, uint32_t mask, unsigned long long key, int i, uint32_t s, int4 raw) {
  while (true) {
    const unsigned long long cur = ((unsigned long long)(unsigned)raw.y << 32) | (unsigned)raw.x;
    if (cur == key) {
      if (raw.w > i) atomicMin(&tab[s].first, i);
      return s;
    }
    if (cur == kEmptyKey) {
      const unsigned long long prev = atomicCAS(&tab[s].key, kEmptyKey, key);
      if (prev == kEmptyKey || prev == key) {
        atomicMin(&tab[s].first, i);
        return s;
      }
    }
    s = (s + 1) & mask;
    raw = __ldcg(reinterpret_cast<const int4*>(tab + s));
  }
}
__device__ inline uint32_t table_insert_first(Slot* tab, uint32_t mask, unsigned long long key, int i) {
  const uint32_t s = hash_key(key) & mask;
  return table_insert_first(tab, mask, key, i, s, __ldcg(reinterpret_cast<const int4*>(tab + s)));
}

// sticky status word bits (device)
constexpr int kStatusRange = 1, kStatusCapacity = 2;

#define SPS_CUDA_CHECK(expr)                                   \
  do {                                                         \
    cudaError_t _e = (expr);                                   \
    if (_e != cudaSuccess) return sps::set_cuda_error(_e, #expr); \
  } while (0)
int set_cuda_error(cudaError_t e, const char* what);

// per-device one-time opt-in to large dynamic shared memory (the attribute is per device AND per kernel)
template <class Kernel>
inline cudaError_t ensure_dynamic_smem(Kernel kernel, size_t bytes, unsigned long long* done_mask) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  const unsigned long long bit = 1ull << (dev & 63);
  if (__atomic_load_n(done_mask, __ATOMIC_ACQUIRE) & bit) return cudaSuccess;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) __atomic_fetch_or(done_mask, bit, __ATOMIC_RELEASE);
  return e;
}

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

}  // namespace sps
