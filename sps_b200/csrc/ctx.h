// Host-side context: carve-up of the caller's workspace arena (no device allocation here), plus every
// piece of mutable host state of the library (arithmetic mode, processing-order mode, launch counter,
// stage timers): there are no process-wide switches, two host threads may drive two contexts freely.
#pragma once
#include <string>
#include <vector>
#include "common.cuh"


struct sps_ctx {
  int64_t max_points = 0;
  int64_t ld = 0;            // leading dimension of the [K][ld] map tables (multiple of 32)
  int64_t n = 0;             // rows of the last voxelize call
  bool have_l0 = false, have_maps = false, have_nbr5 = false;
  bool have_perm = false;    // the 3^4 convs of every level visit rows in pattern-sorted order (perm, ptmask, tslice are valid)
  bool dense_maps = true;    // false after a fused forward that stored only the present entries of the sorted tables

  // ---- settings (sps_ctx_set_conv_backend / sps_ctx_set_pattern_sort) and per-forward state ----
  int backend = SPS_BACKEND_AUTO;
  int pattern_sort = 1;      // 0 never, 1 for inputs of >= 400 000 rows, 2 always
  bool run_half = false;     // the forward being enqueued stores its activations as fp16
  int forward_launches = 0;  // kernels enqueued by the last fused forward
  // stage timers (sps_profile_enable): CUDA events recorded on the launch stream
  bool prof = false;
  std::vector<cudaEvent_t> prof_ev;
  std::vector<std::string> prof_names;
  size_t prof_used = 0;

  char* base = nullptr;
  size_t bytes = 0;

  // scalars (device)
  int32_t* counts = nullptr;   // [SPS_NUM_LEVELS] voxel counts
  int32_t* status = nullptr;   // sticky status word
  uint32_t* ticket = nullptr;  // last-block-done counters, one per unique() call
  int32_t* n_dev = nullptr;    // device copy of n (so level-0 kernels share the code path)
  int32_t* nblocks = nullptr;  // [SPS_NUM_LEVELS] blocks in each level's block table
  int32_t* tplanes = nullptr;  // bit t: the input holds voxels in time plane t (written by the voxelisation)
  // 4x4x4 block tables, one per level (all levels are built and probed by the same launches)
  sps::Slot* btab[SPS_NUM_LEVELS] = {};              // block key -> block id, capacity table_capacity(max_points)
  int32_t* bcells[SPS_NUM_LEVELS] = {};              // [max_points][64] voxel rows per block (upper bound: one block per voxel)
  unsigned long long* bocc[SPS_NUM_LEVELS] = {};     // [max_points] 64-bit occupancy word per block

  float* staging = nullptr;    // [max_points][8] host->device landing zone
  float* scores = nullptr;     // [max_points]
  sps::Slot* table = nullptr;  // open-addressing table, capacity table_capacity(max_points)
  uint32_t table_cap = 0;
  uint32_t* slot_of = nullptr; // [max_points]
  int32_t* rank = nullptr;     // [max_points]
  int32_t* block_sums = nullptr;

  unsigned long long* keys[SPS_NUM_LEVELS] = {};
  int32_t* inv = nullptr;                      // [max_points] point -> level-0 row
  int32_t* parent[SPS_NUM_LEVELS] = {};        // [L] fine row -> parent*8 + k   (L = 0..3)
  int32_t* child[SPS_NUM_LEVELS] = {};         // [L] [8][ld] children of level-L rows (L = 1..4)
  uint32_t* vmask[SPS_NUM_LEVELS] = {};        // [L] [ld][4] per-voxel 27-bit presence words of the 3x3x3 neighbours in the three time planes (+ pad)
  int32_t* perm[SPS_NUM_LEVELS] = {};          // [L] rows of level L in neighbourhood-shape order (conv processing order)
  uint32_t* ptmask[SPS_NUM_LEVELS] = {};       // [L] tile masks of nbr3 in perm order
  int32_t* tslice[SPS_NUM_LEVELS] = {};        // [L] [tiles][82][128] nbr3 gathered per tile in perm order
  // shape sort of all five levels together (5 x max_points keys): ping-pong buffers, [4][256] digit histograms of the four
  // radix passes + 4 tile tickets, look-back status words [tiles][4][256]
  uint32_t* sort_keys[2] = {};
  int32_t* sort_vals[2] = {};
  uint32_t* sort_hist = nullptr;
  uint32_t* sort_status = nullptr;
  int32_t* up_cls = nullptr;                   // [4][16] per fine level: rows per 2x2x2 child class (8) + scatter cursors (8)
  int32_t* perm_up[SPS_NUM_LEVELS] = {};       // [L] rows of level L grouped by child class: processing order of the transposed conv INTO level L
  uint32_t* tmask_up[SPS_NUM_LEVELS] = {};     // [L] tile masks of the 8-class up-map in that order (one or two classes per tile)
  uint32_t* tmask8 = nullptr;                  // [tiles][4] all-eight-offsets mask for the 2x2x2x1 maps
  int32_t* nbr3[SPS_NUM_LEVELS] = {};          // [81][ld]
  int32_t* nbr5 = nullptr;                     // [125][ld]
  uint32_t* tmask3[SPS_NUM_LEVELS] = {};       // [L] [tiles][4] present-offset masks of nbr3 per 128-row tile

  // feature buffers (row-major, upper bound max_points rows; widths in fp32 elements, so that every storage mode fits)
  enum Buf { CAT8, E1, H1, CAT7, E2, H2, CAT6, E3, H3, CAT5, E4, H4, B4, H5, B5, H6, B6, H7, B7, H8,
             FEAT0, LOGITS, NBUF };
  float* buf[NBUF] = {};

  ~sps_ctx() {
    for (cudaEvent_t e : prof_ev) cudaEventDestroy(e);
  }
};

namespace sps {
// conv0 fused into the map-building pass (level-0 block table still alive): see maps.cu
struct Conv0Fused {
  const float* feat;   // per-voxel input feature, or nullptr: every voxel carries `cfeat`
  float cfeat;
  const float* w; const float* shift; int round_out; float* out; int64_t out_ld;
};
// Row strides of the concat buffers, unpadded: padding them to a power of two (so that a gathered fp16 row never straddles a
// 128-byte line) measured neutral (block6.conv1 0.1685 ms either way).
constexpr int kCatLd[4] = {16, 24, 48, 96};   // CAT8, CAT7, CAT6, CAT5
constexpr int kBufWidth[sps_ctx::NBUF] = {16, 8, 8, kCatLd[1], 8, 16, kCatLd[2], 16, 32, kCatLd[3], 32, 64, 64, 64, 64, 32, 32,
                                          16, 16, 8, 1, 1};

// arithmetic mode of a context (see sps_ctx_set_conv_backend)
inline bool ctx_half_storage(const sps_ctx* c) { return c->backend == SPS_BACKEND_AUTO || c->backend == SPS_BACKEND_F16; }

}
