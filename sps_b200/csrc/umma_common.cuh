// Device helpers shared by the tcgen05 convolution kernels (inline PTX for mbarrier, cp.async,
// tcgen05 MMA / TMEM, UMMA descriptors).
#pragma once
#include <cstring>
#include <cuda.h>   // CUtensorMap (types only: the encoder entry point is fetched at run time, no -lcuda)
#include "common.cuh"

namespace sps {

constexpr int kTileM = 128;
constexpr int kAStageBytes = kTileM * 128;  // 16 KB
constexpr int kMaxK = 81;  // kernel volumes this kernel takes (neighbour indices are staged in smem)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// SM100 shared-memory matrix descriptor, K-major, SWIZZLE_128B: 8-row x 128-byte atoms, 1024 B
// apart (SBO); LBO unused for swizzled K-major; version 1; layout type 2.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);  // start address   bits [0,14)
  d |= (uint64_t)1 << 16;                   // LBO (ignored)   bits [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;         // SBO = 1024 B    bits [32,46)
  d |= (uint64_t)1 << 46;                   // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                   // SWIZZLE_128B
  return d;
}
// kind::tf32, fp32 accumulate, both operands K-major: c_format F32 (1<<4), a/b format TF32 (2),
// N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// kind::f16 with fp16 operands (a/b format 0), fp32 accumulate, both operands K-major
__host__ __device__ constexpr uint32_t make_idesc_f16(int n) {
  return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float* v) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr));
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

// groups (of 4 channels) reserved per kernel offset in the K-major weight matrix / the stage plan
__host__ __device__ inline int padded_groups(int cin) {
  const int g = (cin + 3) >> 2;
  return g <= 2 ? 2 : g <= 4 ? 4 : (g + 7) & ~7;
}

// the same for a row of `groups` 16-byte groups; fp16 rows may be a single group (8 channels)
__host__ __device__ inline int padded_groups_of(int groups, bool allow_one) {
  return groups <= 1 && allow_one ? 1 : groups <= 2 ? 2 : groups <= 4 ? 4 : (groups + 7) & ~7;
}

struct UmmaParams {
  const float* wt;  // [cout][ldk] K-major, TF32-rounded (layout: sps_conv_pack_kmajor); fp16 storage: __half,
                    // layout sps_conv_pack_kmajor_f16, ldk in halves
  int64_t ldk;
  int round_out;
  int flags;        // SPS_CONV_FOLD_LO | SPS_CONV_OUT_SPLIT
  int split_groups; // two-segment input rows: 16-byte groups of the FIRST segment (0 = one segment)
  int use_tma;      // the weight stages of a full-width (64-channel) K slab come through TMA: `tmap` is valid
  alignas(64) CUtensorMap tmap;   // 2-D map of the fp16 K-major weight matrix, box = 64 halves x NPAD rows, SWIZZLE_128B
};

// ---- TMA (cp.async.bulk.tensor) of one weight stage: box (64 halves, NPAD rows) at column c0 of the K-major matrix ----
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// arrive on `bar` once all cp.async issued so far by this thread have landed (no pending-count bump)
__device__ __forceinline__ void cp_async_arrive(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
}  // namespace sps
