// tcgen05 implicit-GEMM sparse convolution (the layers with >= 16 output channels of the fused forward, and
// sps_conv_fwd on its tensor-core backends):
//   out[o] = act( sum_k in[nbr[k][o]] . W[k]  (+ in2[o] . W2)  + shift (+ res[o]) )
// 128 output rows = the 128 TMEM lanes of one fp32 accumulator, two accumulators per CTA, persistent
// warp-specialised CTAs.  The gather side is built around what ncu's source view showed about the first
// generations (profiles/r1_conv_source_level.md): 8 producer warps that spent 27 % of their time staging the
// next tile's kernel-map slice, 54 % executing ~130 instructions per pipeline stage and only 8 % waiting for
// a free stage.  Here
//   * a dedicated LOADER warp builds the per-tile list of present offsets and stages the kernel-map
//     slice (and the tile's own row numbers) up to 8 tiles ahead with 16-byte cp.async copies, packed
//     into a ring by the tiles' present offsets; a producer thread fetches the indices of its four
//     rows with one 16-byte shared load;
//   * the stage ring is 4 deep: the gathered rows are re-read from L1 by neighbouring output rows,
//     and measured run time follows the L1 size the carve-out leaves (4 stages beat 2, 3 and 5-7;
//     +40 KB of unused shared memory costs +25 % on the 32/48-channel layers).  A variant that
//     streamed the slices through a 16 KB ring with synchronous L1::no_allocate loads (88 KB of
//     shared memory in total) was not faster on the wide layers and starved the narrow ones;
//   * the producers walk the stage ring with COMPILE-TIME slot numbers (the stage loop is unrolled
//     by the ring depth), so every shared address and mbarrier address is base + immediate and the
//     "copies landed" arrive is a single uniform-address instruction;
//   * the per-stage parameters of the next stage are fetched before waiting for its slot;
//   * global addresses are one IMAD.WIDE per 16-byte chunk.
//   * (tried and dropped, profiles/r2_experiments.md: a warp issuing prefetch.global.L2 for the next tile's rows made
//     every layer 3-6x slower -- the prefetches go through the same L1 data pipe the gathers saturate.)
// Warp roles (448 threads): 0-7 producers, 8 loader, 9 MMA issuer, 10-13 epilogue.
#include "umma_common.cuh"

namespace sps {

// ring depth per accumulator width.  Round 1 ran ONE CTA per SM with a 4-deep ring (4 beat 2, 3 and 5-7).  Round 2: TWO
// CTAs per SM, each with a 2-deep ring and the 42 KB index area (<= 113 KB of shared memory, <= 72 registers):
// convolution family 1.79 -> 1.61 ms per forward (3-deep rings: 1.64) -- two independent gather streams fill the L1 data
// pipe better than one deep ring, and the loader's bubble at a tile boundary hides behind the other CTA.
constexpr int kV6CtasPerSm = 2;   // resident CTAs per SM for N <= 64 (the wide accumulators of the width sweep take a whole SM)
constexpr int kV6ProducerWarps = 8;
constexpr int kV6ProducerThreads = kV6ProducerWarps * 32;
constexpr int kV6LoaderWarp = kV6ProducerWarps;
constexpr int kV6MmaWarp = kV6LoaderWarp + 1;
constexpr int kV6EpiWarp0 = kV6MmaWarp + 1;
constexpr int kV6Threads = (kV6EpiWarp0 + 4) * 32;
constexpr int kV6Entries = kMaxK + 1;                 // present offsets + the tile's own rows
constexpr int kV6EntryBytes = kTileM * 4;
// The index area (82 entries) is a ring: a tile takes nact + 1 consecutive entries (its present offsets, then its own
// rows) from a running cursor, wrapping at the end, and the producers release tiles in order.  So the area holds as
// many tiles as their PRESENT offsets allow, not K + 1 entries per tile: about three 81-offset tiles in shape-sorted
// order (~22 offsets walked per tile; a tile with all 81 takes the whole area), eight of the 2x2x2 kernels (9 entries).
// Without a second tile in flight the producers wait a full global round trip for the next slice at every tile
// boundary; tiles of the small kernels are one or two stages long, so the number of tiles in flight -- not the stage
// ring -- bounds their memory-level parallelism.
constexpr int kV6MaxTilesAhead = 8;
// ordered present-offset lists of the staged tiles: one byte per ring entry (the kernel offset whose rows it holds)
constexpr int kV6KlistBytes = (kV6Entries + 15) & ~15;

template <int NPAD>
struct V6Cfg {
  // SPS's own widths (N <= 64): 2 stages (above).  Wide accumulators of the width sweep (N = 128 / 256, 16 / 32 KB of
  // weights per stage): 4 / 3 stages -- a stage of such a layer keeps the tensor pipe busy for 256 / 512 cycles, the
  // loader's bubble at a tile boundary is noise there.  Every width has the same index ring.
  static constexpr int S = NPAD == 256 ? 3 : NPAD == 128 ? 4 : 2;
  static constexpr int kBStage = NPAD * 128;
  static constexpr int kTmemCols = 2 * NPAD < 32 ? 32 : 2 * NPAD;
  static constexpr int kIdxEntries = kV6Entries;
  static constexpr int kShift = NPAD < 64 ? 64 : NPAD;
  // A ring | B ring | row-index ring [kIdxEntries][128] | barriers | offset ring [kIdxEntries] | (start, nact) [8] |
  // shift | tmem slot
  static constexpr size_t smem = (size_t)S * (kAStageBytes + kBStage) + (size_t)kIdxEntries * kV6EntryBytes +
                                 8 * (2 * S + 2 * kV6MaxTilesAhead + 4) + kV6KlistBytes + 8 * kV6MaxTilesAhead +
                                 kShift * 4 + 16;
};
// two CTAs per SM: 228 KB of shared memory per SM, 1 KB of it reserved per CTA
static_assert(kV6CtasPerSm * (V6Cfg<64>::smem + 1024) <= 228 * 1024, "two N <= 64 CTAs no longer fit on an SM");

// 16-byte copy that writes zeros instead when `skip` is set (the ignore-src form: one predicate, no size select)
template <bool kBypassL1>
__device__ __forceinline__ void cp_async16_or_zero(uint32_t dst, const void* src, bool skip) {
  if (kBypassL1)
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %2, 0;\n"
        "cp.async.cg.shared.global [%0], [%1], 16, p;\n"
        "}\n" ::"r"(dst), "l"(src), "r"((int)skip)
        : "memory");
  else
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %2, 0;\n"
        "cp.async.ca.shared.global [%0], [%1], 16, p;\n"
        "}\n" ::"r"(dst), "l"(src), "r"((int)skip)
        : "memory");
}
// The gathers of the A operand bypass L1 (cp.async.cg): measured alone the convolution family is 2 % SLOWER that way
// (1.517 -> 1.553 ms, the 8- and 24-channel layers lose their L1 hits), but the three-lane step is 1.8 % FASTER (2.414 ->
// 2.372 ms, reproduced twice): the gathered rows no longer evict the lines the other lanes' map kernels work on.  The
// weight copies keep L1 (cp.async.ca).
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}

// T = float: fp32 rows, TF32 operands (kind::tf32); T = __half: fp16 rows and weights (kind::f16, 8 channels per
// 16-byte group, so a stage carries twice the channels).  GPC = 16-byte groups per kernel offset: 1 (fp16
// only), 2 or 4 -> 8/GPC offsets share a stage; 8 -> one offset spans GP/8 stages.
// GPC2 > 0: the input row is TWO channel segments (the halves of a concat buffer, minkunet.py:192): `split_groups`
// 16-byte groups walked as above (GPC), then GPC2 (1, 2 or 4) groups packed 8 / GPC2 offsets per stage -- 96 = 64 + 32,
// 48 = 32 + 16 and 24 = 16 + 8 channels without a single padded column (1.5 / 0.75 / 0.375 stages per offset instead
// of 2 / 1 / 0.5).
template <int NPAD, int GPC, typename T, int GPC2 = 0>
__global__ void __launch_bounds__(kV6Threads, NPAD <= 64 ? kV6CtasPerSm : 1) k_conv_umma6(const sps_conv_args a, const __grid_constant__ UmmaParams p) {
  using Cfg = V6Cfg<NPAD>;
  constexpr int EB = sizeof(T);                         // bytes per stored activation
  constexpr bool kHalf = EB == 2;
  constexpr int S = Cfg::S;
  constexpr int kBStageBytes = Cfg::kBStage;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* sA = smem;
  uint8_t* sB = smem + S * kAStageBytes;
  int32_t* sidx = reinterpret_cast<int32_t*>(sB + S * kBStageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(sidx) + Cfg::kIdxEntries * kV6EntryBytes);
  // bars: full[S], empty[S], idx_full[8], idx_empty[8], acc_full[2], acc_empty[2]
  uint8_t* klist = reinterpret_cast<uint8_t*>(bars + 2 * S + 2 * kV6MaxTilesAhead + 4);
  int2* sslice = reinterpret_cast<int2*>(klist + kV6KlistBytes);   // per tile slot: first ring entry, present offsets
  float* sshift = reinterpret_cast<float*>(sslice + kV6MaxTilesAhead);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sshift + Cfg::kShift);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t sA_u = smem_u32(sA), sB_u = smem_u32(sB), sidx_u = smem_u32(sidx);
  const uint32_t bar_full = smem_u32(bars), bar_empty = bar_full + 8 * S, bar_idxf = bar_empty + 8 * S,
                 bar_idxe = bar_idxf + 8 * kV6MaxTilesAhead, bar_accf = bar_idxe + 8 * kV6MaxTilesAhead,
                 bar_acce = bar_accf + 16;
  if (sA_u & 1023) __trap();

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbar_init(bar_full + 8 * s, kV6ProducerThreads); mbar_init(bar_empty + 8 * s, 1); }
    for (int i = 0; i < kV6MaxTilesAhead; ++i) {
      mbar_init(bar_idxf + 8 * i, 33);                 // 32 async arrivals (copies landed) + 1 for the plain stores
      mbar_init(bar_idxe + 8 * i, kV6ProducerWarps);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(bar_accf + 8 * i, 1);
      mbar_init(bar_acce + 8 * i, 128);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = tid; i < NPAD; i += kV6Threads) sshift[i] = (a.shift && i < a.cout) ? __ldg(a.shift + i) : 0.f;
  // Weight stages by TMA: a full-width K slab (64 fp16 channels of one kernel offset, all NPAD rows) is ONE 2-D box of
  // the K-major weight matrix, landed in the SWIZZLE_128B layout the MMA descriptor reads -- off the LSU path that
  // the gathers saturate.  Narrower slabs (several offsets per stage) would need one small box per offset: those
  // layers keep the cp.async weight copies.
  const bool tma_b = kHalf && GPC == 8 && p.use_tma != 0;
  if (tma_b && tid == 0) tma_prefetch_desc(&p.tmap);
  if (warp == kV6MmaWarp) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"((uint32_t)Cfg::kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int n_out = *a.n_out;
  const int ntiles = (n_out + kTileM - 1) / kTileM;
  const int K = a.K;
  const int gpk = GPC2 ? p.split_groups : ((a.cin * EB) >> 4);   // real 16-byte groups per offset (of the first segment)
  const int GP = GPC < 8 ? GPC : padded_groups_of(gpk, kHalf);  // padded groups per offset
  const int SPE = GPC < 8 ? 1 : GP >> 3;                // stages per offset (Cin >= 24)
  constexpr int EPS = GPC < 8 ? 8 / GPC : 1;            // offsets per stage (Cin <= 16)
  constexpr int EPS2 = GPC2 ? 8 / GPC2 : 1;             // second segment: offsets per stage
  const int gpk2 = a.in2 ? ((a.cin2 * EB) >> 4) : 0;
  // The fused 1x1 term: a pseudo-offset appended to the tile's list of present offsets when its row fits the slot of an
  // offset (several offsets per stage, Cin2 <= padded Cin) -- it then rides in the last, usually partial stage; otherwise
  // stages of its own.
  constexpr int kGpcDiv = GPC < 8 ? GPC : 1;
  const int n2 = (GPC < 8 && GPC2 == 0 && gpk2 > 0 && gpk2 <= 8) ? (gpk2 + kGpcDiv - 1) / kGpcDiv : 0;   // slots it takes (a wide row: several)
  const bool in2_packed = n2 > 0;
  const int st2 = in2_packed ? 0 : (gpk2 + 7) >> 3;     // stages of the fused 1x1 term
  const uint32_t* tmask = a.tile_mask;
  const int gstep = gridDim.x;
  // ring position of entry x of the tile whose entries start at `start`
  auto ring = [](int start, int x) { const int q = start + x; return q >= Cfg::kIdxEntries ? q - Cfg::kIdxEntries : q; };
  auto tile_nact = [&](int tile) {
    return __popc(__ldg(tmask + 4 * tile)) + __popc(__ldg(tmask + 4 * tile + 1)) + __popc(__ldg(tmask + 4 * tile + 2));
  };
  auto stages_a = [&](int nact) { return GPC < 8 ? (nact + n2 + EPS - 1) / EPS : nact * SPE; };
  auto stages_b = [&](int nact) { return GPC2 ? (nact + EPS2 - 1) / EPS2 : 0; };
  auto tile_stages = [&](int nact) { return stages_a(nact) + stages_b(nact) + st2; };

  if (warp < kV6ProducerWarps) {
    // =========================== PRODUCERS (256 threads) ===========================
    const int r0 = tid >> 3, cB = tid & 7;          // chunk column cB of rows 4 r0 + i (one 16-byte index load)
    uint32_t a_off[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int r = 4 * r0 + i;
      a_off[i] = (uint32_t)((r >> 3) * 1024 + (r & 7) * 128) + (((uint32_t)cB ^ (uint32_t)(r & 7)) << 4);
    }
    const uint32_t in_ld_b = (uint32_t)a.in_ld * EB, in2_ld_b = (uint32_t)a.in2_ld * EB;
    const char* in_b = reinterpret_cast<const char*>(a.in);
    const char* in2_b = reinterpret_cast<const char*>(a.in2);
    constexpr int NB = (NPAD + 31) / 32;            // weight chunks per thread per stage
    const char* wrow[NB];
    uint32_t b_off[NB];
    bool wok[NB];
#pragma unroll
    for (int i = 0; i < NB; ++i) {
      const int n = r0 + 32 * i;
      wok[i] = n < ((p.flags & SPS_CONV_FOLD_LO) ? 16 : a.cout) && n < NPAD;
      wrow[i] = reinterpret_cast<const char*>(p.wt) + (int64_t)(wok[i] ? n : 0) * p.ldk * EB;
      b_off[i] = (uint32_t)((n >> 3) * 1024 + (n & 7) * 128) + (((uint32_t)cB ^ (uint32_t)(n & 7)) << 4);
    }
    const bool b_lane = r0 < NPAD;
    constexpr int GPCc = GPC < 8 ? GPC : 1;
    const int e_off = GPC < 8 ? cB / GPCc : 0;      // small Cin: which of the stage's offsets this column belongs to
    const int cg0 = GPC < 8 ? cB % GPCc : cB;       // channel group inside the offset
    constexpr int GPC2c = GPC2 ? GPC2 : 1;
    const int e_off2 = cB / GPC2c, cg02 = cB % GPC2c;   // the same for the second segment

    // ---- cursor over the stages of this CTA's tiles ----
    int tile = blockIdx.x, it_tile = 0;
    int start = 0, nact = 0, m = 0, nst = 0;        // first ring entry, present offsets, current stage, stages of the tile
    int ns_a = 0, ns_b = 0;                         // stages of the two channel segments of the tile
    bool stage_tma = false;                         // the weights of the stage about to be issued come through TMA
    int e = 0, sub = 0;                             // large Cin: offset entry and sub-stage
    const uint32_t sx = sidx_u + (uint32_t)r0 * 16u;   // shared byte address of this thread's int4 in ring entry 0
    // parameters of the stage about to be issued
    int idx[4] = {-1, -1, -1, -1};
    const char* base = in_b;
    uint32_t ld_b = in_ld_b;
    bool okc = false, bok = false;
    uint32_t wofs = 0;

    auto lds4 = [&](uint32_t addr) {
      asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(idx[0]), "=r"(idx[1]), "=r"(idx[2]), "=r"(idx[3])
                   : "r"(addr));
    };
    // fetch the parameters of stage m of the current tile: first channel segment, second segment, fused 1x1 term
    auto fetch = [&]() {
      if (m < ns_a) {
        if (GPC < 8) {
          const int ee = m * EPS + e_off;
          const bool e_ok = ee < nact;
          const bool e_in2 = ee >= nact && ee < nact + n2;  // the slots after the last present offset: the 1x1 term
          const int pos = ring(start, e_ok ? ee : (e_in2 ? nact : 0));
          lds4(sx + (uint32_t)pos * kV6EntryBytes);
          if (e_in2) {
            const int cg = (ee - nact) * GPCc + cg0;        // group of the in2 row this column carries
            base = in2_b + cg * 16; ld_b = in2_ld_b;
            okc = cg < gpk2; bok = true;
            wofs = (uint32_t)(K * GPCc + cg) * 16u;
          } else {
            base = in_b + cg0 * 16; ld_b = in_ld_b;
            okc = e_ok && cg0 < gpk; bok = e_ok;
            wofs = (uint32_t)((int)klist[pos] * GPCc + cg0) * 16u;
          }
          stage_tma = false;
        } else {
          // entry e = kernel offset klist[e], sub-stage `sub` of its SPE stages
          const int pos = ring(start, e);
          if (sub == 0) lds4(sx + (uint32_t)pos * kV6EntryBytes);
          const int cg = cB + 8 * sub;
          base = in_b + cg * 16; ld_b = in_ld_b;
          okc = cg < gpk; bok = okc;
          wofs = (uint32_t)((int)klist[pos] * GP + cg) * 16u;
          stage_tma = tma_b;
        }
      } else if (GPC2 && m < ns_a + ns_b) {
        const int ee = (m - ns_a) * EPS2 + e_off2;
        const bool e_ok = ee < nact;
        const int pos = ring(start, e_ok ? ee : 0);
        lds4(sx + (uint32_t)pos * kV6EntryBytes);
        base = in_b + (gpk + cg02) * 16; ld_b = in_ld_b;
        okc = e_ok; bok = e_ok;
        wofs = (uint32_t)(K * GP + (int)klist[pos] * GPC2c + cg02) * 16u;
        stage_tma = false;
      } else {
        // the fused 1x1 term on the tile's own rows (entry nact)
        const int cg = cB + 8 * (m - ns_a - ns_b);
        lds4(sx + (uint32_t)ring(start, nact) * kV6EntryBytes);
        base = in2_b + cg * 16; ld_b = in2_ld_b;
        okc = cg < gpk2; bok = okc;
        wofs = (uint32_t)(K * (GP + GPC2) + cg) * 16u;
        stage_tma = tma_b;
      }
    };
    // make `tile` current (skipping tiles without stages); false when the CTA has no tile left
    auto open_tile = [&]() -> bool {
      for (;;) {
        if (tile >= ntiles) return false;
        const int slot = it_tile % kV6MaxTilesAhead;
        mbar_wait(bar_idxf + 8 * slot, (it_tile / kV6MaxTilesAhead) & 1);
        const int2 sl = sslice[slot];
        start = sl.x; nact = sl.y;
        ns_a = stages_a(nact); ns_b = stages_b(nact);
        nst = ns_a + ns_b + st2;
        m = 0; e = 0; sub = 0;
        if (nst > 0) { fetch(); return true; }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_idxe + 8 * slot);
        tile += gstep; ++it_tile;
      }
    };
    // step to the next stage; false when the CTA is out of work
    auto advance = [&]() -> bool {
      ++m;
      if (m < nst) {
        if (GPC >= 8 && m < ns_a) {
          if (++sub == SPE) { sub = 0; ++e; }
        }
        fetch();
        return true;
      }
      __syncwarp();                                   // every lane holds its indices in registers by now
      if (lane == 0) mbar_arrive(bar_idxe + 8 * (it_tile % kV6MaxTilesAhead));
      tile += gstep; ++it_tile;
      return open_tile();
    };

    bool more = open_tile();
    uint32_t phase = 0;
    while (more) {
#pragma unroll
      for (int s = 0; s < S; ++s) {
        if (more) {
          mbar_wait(bar_empty + 8 * s, phase ^ 1);    // the MMAs that read slot s have completed
          const uint32_t dstA = sA_u + (uint32_t)s * kAStageBytes;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const bool ok = okc && idx[i] >= 0;
            const uint32_t row = (uint32_t)(idx[i] < 0 ? 0 : idx[i]);
            cp_async16_or_zero<true>(dstA + a_off[i], base + (uint64_t)row * ld_b, !ok);
          }
          if (stage_tma) {
            if (tid == 0) {   // thread 0 holds column 0 of the slab: wofs = byte offset of the slab in a weight row
              mbar_expect_tx(bar_full + 8 * s, (uint32_t)kBStageBytes);
              tma_load_2d(sB_u + (uint32_t)s * kBStageBytes, &p.tmap, (int)(wofs >> 1), 0, bar_full + 8 * s);
            }
          } else if (b_lane) {
#pragma unroll
            for (int i = 0; i < NB; ++i)
              cp_async16_or_zero<false>(sB_u + (uint32_t)s * kBStageBytes + b_off[i], wrow[i] + wofs, !(bok && wok[i]));
          }
          cp_async_arrive(bar_full + 8 * s);          // fires when this thread's copies of the stage have landed
          more = advance();
        }
      }
      phase ^= 1;
    }
    cp_async_wait<0>();
  } else if (warp == kV6LoaderWarp) {
    // =========================== LOADER (one warp, up to kV6MaxTilesAhead tiles ahead) ===========================
    int it = 0;
    int head = 0, used = 0, it_free = 0;   // next free ring entry, entries held by tiles in flight, oldest tile in flight
    const bool map_vec = ((reinterpret_cast<uintptr_t>(a.map) & 15) == 0) && ((a.map_ld & 3) == 0);
    // the tile mask is the head of every tile's dependency chain: keep the NEXT tile's words in flight
    uint32_t mw[3] = {0u, 0u, 0u};
    if ((int)blockIdx.x < ntiles) {
#pragma unroll
      for (int w = 0; w < 3; ++w) mw[w] = __ldg(tmask + 4 * blockIdx.x + w);
    }
    for (int tile = blockIdx.x; tile < ntiles; tile += gstep, ++it) {
      const int slot = it % kV6MaxTilesAhead;
      const uint32_t cur[3] = {mw[0], mw[1], mw[2]};
      if (tile + gstep < ntiles) {
#pragma unroll
        for (int w = 0; w < 3; ++w) mw[w] = __ldg(tmask + 4 * (tile + gstep) + w);
      }
      const int nact = __popc(cur[0]) + __popc(cur[1]) + __popc(cur[2]);
      // wait until the tile's nact + 1 entries and its slot are free; the producers release tiles in order
      while (it - it_free == kV6MaxTilesAhead || used + nact + 1 > Cfg::kIdxEntries) {
        const int fs = it_free % kV6MaxTilesAhead;
        mbar_wait(bar_idxe + 8 * fs, (it_free / kV6MaxTilesAhead) & 1);
        used -= sslice[fs].y + 1;
        ++it_free;
      }
      const int start = head;
      head = ring(start, nact + 1);
      used += nact + 1;
      int n = 0;
#pragma unroll
      for (int w = 0; w < 3; ++w) {
        const uint32_t bits = cur[w];
        if ((bits >> lane) & 1u) klist[ring(start, n + __popc(bits & ((1u << lane) - 1u)))] = (uint8_t)(32 * w + lane);
        n += __popc(bits);
      }
      if (lane == 0) sslice[slot] = make_int2(start, nact);
      __syncwarp();
      // entries are 128 row indices in tile order; lane owns rows 4 lane .. 4 lane + 3 (one 16-byte chunk per entry)
      const uint32_t dst0 = sidx_u + (uint32_t)lane * 16u;
      auto dst = [&](int e) { return dst0 + (uint32_t)ring(start, e) * kV6EntryBytes; };
      if (a.tile_slices) {
        // the level's pass already gathered this tile's slice (entries 0..nact, the last one = own rows)
        const char* src = reinterpret_cast<const char*>(a.tile_slices + (int64_t)tile * (SPS_TILE_SLICE_ENTRIES * kTileM)) + lane * 16;
        for (int e = 0; e <= nact; ++e)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst(e)), "l"(src + (size_t)e * kV6EntryBytes)
                       : "memory");
      } else if (!a.perm && map_vec && !(p.flags & SPS_CONV_MAP_PARENT) && tile * kTileM + kTileM <= n_out) {
        // physical row order, full tile: the slice of map[k] is contiguous -> one 16-byte copy per lane and entry
        const int row0 = tile * kTileM + 4 * lane;
        asm volatile("st.shared.v4.s32 [%0], {%1, %2, %3, %4};" ::"r"(dst(nact)), "r"(row0),
                     "r"(row0 + 1), "r"(row0 + 2), "r"(row0 + 3)
                     : "memory");
        const int32_t* src = a.map + row0;
        for (int e = 0; e < nact; ++e)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst(e)), "l"(src + (int64_t)klist[ring(start, e)] * a.map_ld)
                       : "memory");
      } else {
        const int32_t* src[4];
        bool rok[4];
        int pw[4];   // SPS_CONV_MAP_PARENT: the rows' parent words (coarse row * 8 + child class)
        const bool from_parent = (p.flags & SPS_CONV_MAP_PARENT) != 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int prow = tile * kTileM + 4 * lane + i;
          rok[i] = prow < n_out;
          const int row = rok[i] ? (a.perm ? __ldg(a.perm + prow) : prow) : 0;
          src[i] = a.map + row;
          pw[i] = (from_parent && rok[i]) ? __ldg(a.map + row) : -1;
          asm volatile("st.shared.s32 [%0], %1;" ::"r"(dst(nact) + 4u * i), "r"(rok[i] ? row : -1) : "memory");
        }
        for (int e = 0; e < nact; ++e) {
          const int k = klist[ring(start, e)];
          const int64_t koff = (int64_t)k * a.map_ld;
          const uint32_t d = dst(e);
          if (from_parent) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int val = (pw[i] >= 0 && (pw[i] & 7) == k) ? (pw[i] >> 3) : -1;
              asm volatile("st.shared.s32 [%0], %1;" ::"r"(d + 4u * i), "r"(val) : "memory");
            }
            continue;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            if (rok[i]) cp_async4(d + 4u * i, src[i] + koff);
            else asm volatile("st.shared.s32 [%0], %1;" ::"r"(d + 4u * i), "r"(-1) : "memory");
          }
        }
      }
      cp_async_arrive(bar_idxf + 8 * slot);
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_idxf + 8 * slot);        // orders the plain shared stores of the whole warp
    }
    cp_async_wait<0>();
  } else if (warp == kV6MmaWarp) {
    // =========================== MMA ISSUER (one lane) ===========================
    const uint32_t idesc = kHalf ? make_idesc_f16(NPAD) : make_idesc_tf32(NPAD);
    uint32_t gs = 0;
    int n_acc = 0;
    int tile = blockIdx.x;
    int nact_next = tile < ntiles ? tile_nact(tile) : 0;
    for (; tile < ntiles; tile += gstep) {
      const int nstages = tile_stages(nact_next);
      if (tile + gstep < ntiles) nact_next = tile_nact(tile + gstep);   // in flight behind this tile's stages
      if (nstages == 0) continue;
      const int b = n_acc & 1;
      mbar_wait(bar_acce + 8 * b, ((n_acc >> 1) & 1) ^ 1);
      ++n_acc;
      tc_fence_after();
      const uint32_t tacc = tmem_base + (uint32_t)(b * NPAD);
      for (int it = 0; it < nstages; ++it, ++gs) {
        const uint32_t slot = gs % S;
        mbar_wait(bar_full + 8 * slot, (gs / S) & 1);
        fence_proxy_async();   // the stage was written through the generic proxy (cp.async); the MMA reads it through the async proxy
        tc_fence_after();
        if (lane == 0) {
          const uint64_t adesc = make_smem_desc(sA_u + slot * kAStageBytes);
          const uint64_t bdesc = make_smem_desc(sB_u + slot * kBStageBytes);
#pragma unroll
          for (int j = 0; j < 4; ++j) {   // 4 x 32 bytes of K (8 tf32 / 16 fp16) inside the 128-byte swizzle atom
            if (kHalf) umma_f16(tacc, adesc + (uint64_t)(j * 2), bdesc + (uint64_t)(j * 2), idesc, (it | j) ? 1u : 0u);
            else umma_tf32(tacc, adesc + (uint64_t)(j * 2), bdesc + (uint64_t)(j * 2), idesc, (it | j) ? 1u : 0u);
          }
          umma_commit(bar_empty + 8 * slot);
          if (it == nstages - 1) umma_commit(bar_accf + 8 * b);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== EPILOGUE (4 warps = 128 TMEM lanes) ===========================
    const int q = warp & 3;
    const int r = q * 32 + lane;
    const int cout = a.cout;
    const bool res_vec = a.res && ((reinterpret_cast<uintptr_t>(a.res) & 15) == 0) && ((a.res_ld & 3) == 0);
    int n_acc = 0;
    int tile = blockIdx.x;
    int nact_next = 0, row_next = -1;
    auto look = [&](int t) {
      nact_next = tile_nact(t);
      const int prow = t * kTileM + r;
      row_next = prow < n_out ? (a.perm ? __ldg(a.perm + prow) : prow) : -1;
    };
    if (tile < ntiles) look(tile);
    for (; tile < ntiles; tile += gstep) {
      const int nstages = tile_stages(nact_next);
      const int row = row_next;
      if (tile + gstep < ntiles) look(tile + gstep);
      const int b = n_acc & 1;
      const bool have = nstages > 0;
      if (have) {
        mbar_wait(bar_accf + 8 * b, (n_acc >> 1) & 1);
        ++n_acc;
        tc_fence_after();
      }
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(b * NPAD);
      const bool live = row >= 0;
      // 16 accumulator columns at a time: few live registers (the CTA leaves room for another lane's map kernels on
      // the same SM), and the same code serves the wide accumulators of the width sweep
#pragma unroll 4
      for (int c0 = 0; c0 < NPAD; c0 += 16) {
        float acc[16];
        __syncwarp();                       // tcgen05.ld is warp-collective: every lane is back from the stores
        if (have) {
          tmem_ld8(taddr + c0, acc);
          tmem_ld8(taddr + c0 + 8, acc + 8);
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (c0 + 16 >= NPAD) {            // last chunk read: the accumulator may be overwritten
            tc_fence_before();
            mbar_arrive(bar_acce + 8 * b);
          }
        } else {
#pragma unroll
          for (int c = 0; c < 16; ++c) acc[c] = 0.f;
        }
        if (live && c0 < cout) {
          if (NPAD == 16 && (p.flags & SPS_CONV_FOLD_LO)) {   // columns 8..15 = the row times the LOW parts of the weights
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[c] += acc[c + 8];
          }
#pragma unroll
          for (int c = 0; c < 16; c += 8) {
            const int cc = c0 + c;
            if (cc >= cout) continue;
            float rv[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (a.res) {
              if (kHalf) {
                const uint4 u = __ldg(reinterpret_cast<const uint4*>(reinterpret_cast<const __half*>(a.res) + (int64_t)row * a.res_ld + cc));
                const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
                for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(h[j]); rv[2 * j] = f.x; rv[2 * j + 1] = f.y; }
              } else {
                const float* resp = a.res + (int64_t)row * a.res_ld + cc;
                if (res_vec) {
                  const float4 r0 = __ldg(reinterpret_cast<const float4*>(resp)), r1 = __ldg(reinterpret_cast<const float4*>(resp + 4));
                  rv[0] = r0.x; rv[1] = r0.y; rv[2] = r0.z; rv[3] = r0.w; rv[4] = r1.x; rv[5] = r1.y; rv[6] = r1.z; rv[7] = r1.w;
                } else {
#pragma unroll
                  for (int j = 0; j < 8; ++j) rv[j] = __ldg(resp + j);
                }
              }
            }
            float v8[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              float v = acc[c + j] + sshift[cc + j] + rv[j];
              if (a.relu) v = fmaxf(v, 0.f);
              v8[j] = v;
            }
            if (a.head_out && cc == 0) {     // final 1x1 conv + bias on the 8 channels of the block output
              float sum = a.head_b;
#pragma unroll
              for (int j = 0; j < 8; ++j) sum = fmaf(v8[j], __ldg(a.head_w + j), sum);
              a.head_out[row] = sum;
            }
            if (a.out) {
              if (kHalf && (p.flags & SPS_CONV_OUT_SPLIT)) store_row8(a.out + cc, a.out_ld, row, v8, kStoreF16x2);   // 16 halves per 8 channels
              else store_row8(a.out + (kHalf ? cc / 2 : cc), a.out_ld, row, v8, kHalf ? kStoreF16 : (p.round_out ? kStoreTF32 : kStoreF32));
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kV6MmaWarp)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::kTmemCols)
                 : "memory");
}

// cuTensorMapEncodeTiled through the runtime's driver entry point lookup (the library does not link libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      return nullptr;
    return reinterpret_cast<EncodeTiledFn>(f);
  }();
  return fn;
}
// 2-D map of the fp16 K-major weight matrix [cout][ldk]: box = 64 halves (one 128-byte swizzle row) x npad rows
static bool make_weight_tmap(CUtensorMap* m, const void* wt, int64_t ldk, int cout, int npad) {
  EncodeTiledFn enc = encode_tiled_fn();
  if (!enc || (ldk & 7) || (reinterpret_cast<uintptr_t>(wt) & 15)) return false;
  const cuuint64_t dims[2] = {(cuuint64_t)ldk, (cuuint64_t)cout};
  const cuuint64_t strides[1] = {(cuuint64_t)ldk * 2};
  const cuuint32_t box[2] = {64, (cuuint32_t)npad};
  const cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(wt), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

template <int NPAD, int GPC, typename T, int GPC2 = 0>
static int launch_umma6(const sps_conv_args& a, const UmmaParams& p_in, cudaStream_t st) {
  UmmaParams p = p_in;
  p.split_groups = GPC2 ? a.cin_split >> 3 : 0;
  if (sizeof(T) == 2 && GPC == 8) p.use_tma = make_weight_tmap(&p.tmap, p.wt, p.ldk, (a.flags & SPS_CONV_FOLD_LO) ? 16 : a.cout, NPAD) ? 1 : 0;
  const size_t smem = V6Cfg<NPAD>::smem;
  static unsigned long long attr_done = 0;   // bit per device: the opt-in is per device and per kernel
  SPS_CUDA_CHECK(ensure_dynamic_smem(k_conv_umma6<NPAD, GPC, T, GPC2>, smem, &attr_done));
  int64_t tiles = (a.n_out_max + kTileM - 1) / kTileM;
  if (tiles < 1) tiles = 1;
  const int per_sm = NPAD <= 64 ? kV6CtasPerSm : 1;
  const int grid = (int)(tiles < 148 * per_sm ? tiles : 148 * per_sm);
  k_conv_umma6<NPAD, GPC, T, GPC2><<<grid, kV6Threads, smem, st>>>(a, p);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

template <int NPAD, typename T>
static int launch_umma6_n(const sps_conv_args& a, const UmmaParams& p, cudaStream_t st) {
  constexpr bool kHalf = sizeof(T) == 2;
  if (a.cin_split) {
    // two channel segments (fp16 rows): 64 + 32, 32 + 16 or 16 + 8 channels
    if constexpr (kHalf) {
      const int ga = a.cin_split >> 3, gb = (a.cin - a.cin_split) >> 3;
      if (ga == 8 && gb == 4) return launch_umma6<NPAD, 8, T, 4>(a, p, st);
      if (ga == 4 && gb == 2) return launch_umma6<NPAD, 4, T, 2>(a, p, st);
      if (ga == 2 && gb == 1) return launch_umma6<NPAD, 2, T, 1>(a, p, st);
    }
    return SPS_ERR_UNSUPPORTED;
  }
  const int gp = padded_groups_of((a.cin * (int)sizeof(T)) >> 4, kHalf);
  if (kHalf && gp == 1) return launch_umma6<NPAD, kHalf ? 1 : 2, T>(a, p, st);
  if (gp == 2) return launch_umma6<NPAD, 2, T>(a, p, st);
  if (gp == 4) return launch_umma6<NPAD, 4, T>(a, p, st);
  return launch_umma6<NPAD, 8, T>(a, p, st);
}

template <typename T>
static int conv_umma6_t(const sps_conv_args& a, const UmmaParams& p, cudaStream_t st) {
  switch (a.cout) {
    case 8:
    case 16: return launch_umma6_n<16, T>(a, p, st);
    case 32: return launch_umma6_n<32, T>(a, p, st);
    case 64: return launch_umma6_n<64, T>(a, p, st);
    default: break;
  }
  if (sizeof(T) != 2) return SPS_ERR_UNSUPPORTED;
  // wide layers (the PLANES x2 .. x8 sweep of BASELINE config 5), fp16 rows only
  if (a.cout == 128) return launch_umma6<128, 8, T>(a, p, st);
  if (a.cout == 256) return launch_umma6<256, 8, T>(a, p, st);
  if (a.cout == 512) {
    // two passes of 256 output channels: the accumulator pair of one pass fills the 512 TMEM columns
    for (int h = 0; h < 2; ++h) {
      sps_conv_args b = a;
      UmmaParams q = p;
      b.cout = 256;
      q.wt = reinterpret_cast<const float*>(reinterpret_cast<const __half*>(p.wt) + (int64_t)h * 256 * p.ldk);
      if (a.shift) b.shift = a.shift + 256 * h;
      if (a.out) b.out = reinterpret_cast<float*>(reinterpret_cast<__half*>(a.out) + 256 * h);
      if (a.res) b.res = reinterpret_cast<const float*>(reinterpret_cast<const __half*>(a.res) + 256 * h);
      const int rc = launch_umma6<256, 8, T>(b, q, st);
      if (rc != SPS_OK) return rc;
    }
    return SPS_OK;
  }
  return SPS_ERR_UNSUPPORTED;
}

int conv_umma(const sps_conv_args& a, cudaStream_t st) {
  UmmaParams p;
  memset(&p, 0, sizeof(p));
  p.wt = a.weight_kmajor;
  p.ldk = a.kmajor_ld;
  p.round_out = a.round_out;
  p.flags = a.flags;
  return a.io_dtype == SPS_IO_F16 ? conv_umma6_t<__half>(a, p, st) : conv_umma6_t<float>(a, p, st);
}

// fp32 rows, TF32 operands
bool conv_umma_supports(const sps_conv_args& a) {
  if (a.io_dtype != SPS_IO_F32 || a.mode != SPS_CONV_NBR || !a.map || !a.weight_kmajor || !a.tile_mask) return false;
  if (a.K < 1 || a.K > kMaxK || a.cin_split) return false;
  if ((a.flags & SPS_CONV_MAP_PARENT) && a.K != 8) return false;
  if (a.cin < 4 || (a.cin & 3) || (a.in_ld & 3)) return false;
  if (a.in2 && ((a.cin2 & 3) || (a.in2_ld & 3))) return false;
  if (!(a.cout == 8 || a.cout == 16 || a.cout == 32 || a.cout == 64)) return false;
  if (a.kmajor_ld & 3) return false;
  return true;
}

// Per-tile (128 consecutive output rows) bitmask of the kernel offsets that have at least one
// neighbour in the tile: masks[tile][4] (bits 0..K-1 over the first 3 words).
__global__ void __launch_bounds__(128)
k_tile_masks(const int32_t* __restrict__ map, int64_t ld, int K, const int32_t* __restrict__ n_ptr,
             uint32_t* __restrict__ masks) {
  const int n = *n_ptr;
  const int ntiles = (n + kTileM - 1) / kTileM;
  __shared__ uint32_t m[4];
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    if (threadIdx.x < 4) m[threadIdx.x] = 0;
    __syncthreads();
    const int row = tile * kTileM + threadIdx.x;
    for (int k = 0; k < K; ++k) {
      const bool hit = row < n && __ldg(map + (int64_t)k * ld + row) >= 0;
      if (__any_sync(0xffffffffu, hit) && (threadIdx.x & 31) == 0) atomicOr(&m[k >> 5], 1u << (k & 31));
    }
    __syncthreads();
    if (threadIdx.x < 4) masks[4 * tile + threadIdx.x] = m[threadIdx.x];
    __syncthreads();
  }
}

// fp16 storage: every layer of the network fits (channel counts are multiples of 8, rows 16-byte aligned)
bool conv_umma_f16_supports(const sps_conv_args& a) {
  if (a.io_dtype != SPS_IO_F16 || a.mode != SPS_CONV_NBR || (!a.map && !a.tile_slices) || !a.weight_kmajor || !a.tile_mask) return false;
  if (a.tile_slices && !a.perm) return false;
  if (a.K < 1 || a.K > kMaxK) return false;
  if ((a.flags & SPS_CONV_MAP_PARENT) && (a.K != 8 || !a.map || a.tile_slices)) return false;
  if (a.cin < 8 || (a.cin & 7) || (a.in_ld & 7)) return false;
  if (a.in2 && ((a.cin2 & 7) || (a.in2_ld & 7))) return false;
  if (a.res && (a.res_ld & 7)) return false;
  if (a.out && (a.out_ld & 7)) return false;
  if (!(a.cout == 8 || a.cout == 16 || a.cout == 32 || a.cout == 64 || a.cout == 128 || a.cout == 256 || a.cout == 512)) return false;
  if (a.cout > 64 && (a.cin < 64 || a.head_out)) return false;   // wide accumulators: full 64-channel K slabs only
  if (a.kmajor_ld & 7) return false;
  if ((a.flags & SPS_CONV_FOLD_LO) && a.cout != 8) return false;
  if ((a.flags & SPS_CONV_OUT_SPLIT) && a.out && (a.out_ld & 15)) return false;
  if (a.cin_split) {   // two channel segments: 64 + 32, 32 + 16, 16 + 8
    const int ga = a.cin_split >> 3, gb = (a.cin - a.cin_split) >> 3;
    if ((a.cin_split & 7) || a.cout > 64) return false;
    if (!((ga == 8 && gb == 4) || (ga == 4 && gb == 2) || (ga == 2 && gb == 1))) return false;
  }
  return true;
}

}  // namespace sps

// fp16 twin of sps_conv_pack_kmajor: ME-layout weights [K][cin][cout] (+ optional 1x1 term [cin2][cout]) ->
// K-major __half [rows][ld]; per kernel offset padded_groups_of(cin_eff/8) * 8 halves, the 1x1 term padded to 64.
// pack_flags (include/sps_b200.h): SPS_PACK_IN_SPLIT / SPS_PACK_IN2_SPLIT double the channels of `in` / `in2` (rows stored
// as hi|lo pairs: every 8-channel group of the weights appears twice along K), SPS_PACK_FOLD_LO appends the low parts
// of the weights as rows 8..15 (cout == 8).
// cin_split > 0 (sps_conv_args.cin_split): the K axis holds the first cin_split channels of every offset, THEN the remaining
// channels of every offset (unpadded: 8, 16 or 32 of them), then the 1x1 term.
extern "C" int64_t sps_conv_kmajor_ld_f16s(int K, int cin, int cin2, int pack_flags, int cin_split) {
  const int ce = (pack_flags & SPS_PACK_IN_SPLIT) ? 2 * cin : cin, c2e = (pack_flags & SPS_PACK_IN2_SPLIT) ? 2 * cin2 : cin2;
  if (cin_split > 0 && cin_split < cin)
    return (int64_t)K * (sps::padded_groups_of((cin_split + 7) >> 3, true) * 8 + (((cin - cin_split) + 7) & ~7)) + ((c2e + 63) & ~63);
  return (int64_t)K * sps::padded_groups_of((ce + 7) >> 3, true) * 8 + ((c2e + 63) & ~63);
}
extern "C" int64_t sps_conv_kmajor_ld_f16x(int K, int cin, int cin2, int pack_flags) {
  return sps_conv_kmajor_ld_f16s(K, cin, cin2, pack_flags, 0);
}
extern "C" int sps_conv_pack_kmajor_f16s(const float* w, int K, int cin, int cout, const float* w2, int cin2, int pack_flags,
                                         int cin_split, void* out_) {
  if (!w || !out_ || K < 1 || cin < 1 || cout < 1 || (w2 == nullptr) != (cin2 == 0)) return SPS_ERR_BAD_ARG;
  if (cin_split < 0 || cin_split >= cin) return SPS_ERR_BAD_ARG;
  if (cin_split && ((pack_flags & SPS_PACK_IN_SPLIT) || (cin_split & 7) || (cin & 7))) return SPS_ERR_BAD_ARG;
  const bool in_split = pack_flags & SPS_PACK_IN_SPLIT, in2_split = pack_flags & SPS_PACK_IN2_SPLIT,
             fold = pack_flags & SPS_PACK_FOLD_LO;
  if (fold && cout != 8) return SPS_ERR_BAD_ARG;
  if ((in_split && (cin & 7)) || (in2_split && (cin2 & 7))) return SPS_ERR_BAD_ARG;
  __half* out = static_cast<__half*>(out_);
  const int64_t ldk = sps_conv_kmajor_ld_f16s(K, cin, cin2, pack_flags, cin_split);
  const int ce = cin_split ? cin_split : (in_split ? 2 * cin : cin);
  const int cpad = sps::padded_groups_of((ce + 7) >> 3, true) * 8;       // first segment, per offset
  const int cb = cin_split ? cin - cin_split : 0;                         // second segment, per offset
  const int64_t k_end = (int64_t)K * (cpad + cb);                         // where the 1x1 term starts
  const int rows = fold ? 16 : cout;
  // position of input channel ci inside its (possibly doubled) block, and of its low-half twin
  auto pos = [](int ci, bool split) { return split ? (ci >> 3) * 16 + (ci & 7) : ci; };
  for (int r = 0; r < rows; ++r) {
    __half* row = out + (int64_t)r * ldk;
    for (int64_t i = 0; i < ldk; ++i) row[i] = __float2half_rn(0.f);
    const int nn = fold ? (r & 7) : r;      // output channel this row belongs to
    auto val = [&](float x) {
      const __half hi = __float2half_rn(x);
      return (fold && r >= 8) ? __float2half_rn(x - __half2float(hi)) : hi;
    };
    for (int k = 0; k < K; ++k)
      for (int ci = 0; ci < cin; ++ci) {
        const __half v = val(w[((int64_t)k * cin + ci) * cout + nn]);
        if (cin_split && ci >= cin_split) { row[(int64_t)K * cpad + (int64_t)k * cb + (ci - cin_split)] = v; continue; }
        row[(int64_t)k * cpad + pos(ci, in_split)] = v;
        if (in_split) row[(int64_t)k * cpad + pos(ci, true) + 8] = v;
      }
    for (int ci = 0; ci < cin2; ++ci) {
      const __half v = val(w2[(int64_t)ci * cout + nn]);
      row[k_end + pos(ci, in2_split)] = v;
      if (in2_split) row[k_end + pos(ci, true) + 8] = v;
    }
  }
  return SPS_OK;
}
extern "C" int sps_conv_pack_kmajor_f16x(const float* w, int K, int cin, int cout, const float* w2, int cin2, int pack_flags,
                                         void* out) {
  return sps_conv_pack_kmajor_f16s(w, K, cin, cout, w2, cin2, pack_flags, 0, out);
}
extern "C" int64_t sps_conv_kmajor_ld_f16(int K, int cin, int cin2) { return sps_conv_kmajor_ld_f16x(K, cin, cin2, 0); }
extern "C" int sps_conv_pack_kmajor_f16(const float* w, int K, int cin, int cout, const float* w2, int cin2, void* out) {
  return sps_conv_pack_kmajor_f16x(w, K, cin, cout, w2, cin2, 0, out);
}

extern "C" int sps_tma_weights_available(void) { return sps::encode_tiled_fn() != nullptr ? 1 : 0; }

extern "C" int sps_kernel_map_tile_masks(const int32_t* d_map, int64_t map_ld, int K, const int32_t* d_n_out,
                                         int64_t n_out_max, uint32_t* d_masks, void* stream) {
  if (!d_map || !d_n_out || !d_masks || K < 1 || K > sps::kMaxK || n_out_max < 0) return SPS_ERR_BAD_ARG;
  int64_t tiles = (n_out_max + sps::kTileM - 1) / sps::kTileM;
  if (tiles < 1) tiles = 1;
  const int grid = (int)(tiles < 148 * 16 ? tiles : 148 * 16);
  sps::k_tile_masks<<<grid, 128, 0, (cudaStream_t)stream>>>(d_map, map_ld, K, d_n_out, d_masks);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

// Host helper: ME-layout weights [K][cin][cout] (+ optional 1x1 term [cin2][cout]) -> K-major
// [cout][ld]: row n holds, for every kernel offset k, padded_groups(cin)*4 floats (channels of
// W[k][:, n], zero padded), then the 1x1 term padded to a multiple of 32; values rounded to
// TF32 (nearest even).
extern "C" int64_t sps_conv_kmajor_ld(int K, int cin, int cin2) {
  return (int64_t)K * sps::padded_groups(cin) * 4 + ((cin2 + 31) & ~31);
}

extern "C" int sps_conv_pack_kmajor(const float* w, int K, int cin, int cout, const float* w2, int cin2, float* out) {
  if (!w || !out || K < 1 || cin < 1 || cout < 1 || (w2 == nullptr) != (cin2 == 0)) return SPS_ERR_BAD_ARG;
  const int64_t ldk = sps_conv_kmajor_ld(K, cin, cin2);
  const int cpad = sps::padded_groups(cin) * 4;
  auto rnd = [](float x) {
    uint32_t u;
    memcpy(&u, &x, 4);
    u += 0xFFFu + ((u >> 13) & 1u);
    u &= ~0x1FFFu;
    float y;
    memcpy(&y, &u, 4);
    return y;
  };
  for (int n = 0; n < cout; ++n) {
    float* row = out + (int64_t)n * ldk;
    for (int64_t i = 0; i < ldk; ++i) row[i] = 0.f;
    for (int k = 0; k < K; ++k)
      for (int ci = 0; ci < cin; ++ci) row[(int64_t)k * cpad + ci] = rnd(w[((int64_t)k * cin + ci) * cout + n]);
    for (int ci = 0; ci < cin2; ++ci) row[(int64_t)K * cpad + ci] = rnd(w2[(int64_t)ci * cout + n]);
  }
  return SPS_OK;
}
