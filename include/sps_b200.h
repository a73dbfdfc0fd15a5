/*
 * sps_b200 -- C ABI of the B200-native SPS inference hot path.
 *
 * The reference (ibrahimhroob/SPS) is pure Python; the arithmetic of its hot path lives behind
 * the MinkowskiEngine (ME) Python API (a pybind11 module -- there is no C ABI upstream).  This
 * header is the boundary a maintainer binds instead (ctypes, see INTEGRATION.md).  Each entry
 * point names the reference call site(s) it replaces (paths under the reference repo root).
 *
 * Conventions
 *   - every function returns an int status (SPS_OK == 0); nothing throws across the boundary;
 *   - the CALLER owns all memory: device buffers are raw pointers with element counts, the
 *     library allocates nothing on the device (the workspace arena is handed in);
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it, no host
 *     synchronisation happens unless stated (the *_host and *_status calls);
 *   - sizes that are only known on the device (voxel counts) stay on the device; the
 *     `sps_level_view` exposes their addresses;
 *   - one sps_ctx per stream.  The library keeps NO process-wide mutable state: arithmetic mode, processing-order
 *     mode, launch counters and stage timers live in the sps_ctx, a sps_net is read-only after sps_net_finalize,
 *     sps_last_error is thread-local.  Distinct host threads may drive distinct contexts concurrently (also on
 *     distinct devices); one context must not be used from two threads at once.
 */
#ifndef SPS_B200_H
#define SPS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPS_OK 0
#define SPS_ERR_BAD_ARG 1      /* null pointer, negative count, unsupported channel width ... */
#define SPS_ERR_CAPACITY 2     /* n exceeds what the context / buffers were sized for       */
#define SPS_ERR_COORD_RANGE 3  /* a quantised coordinate does not fit the 64-bit voxel key  */
#define SPS_ERR_CUDA 4         /* a CUDA runtime call failed (see sps_last_error)           */
#define SPS_ERR_UNSUPPORTED 5
#define SPS_ERR_STATE 6        /* call order violated (e.g. forward before voxelize)        */

#define SPS_NUM_LEVELS 5       /* tensor strides 1,2,4,8,16 (minkunet.py:64-104)            */

/* Voxel key packing (device side): b:8 | x:18 | y:18 | z:16 | t:4, biased so that floor-to-
 * stride is a mask.  Valid ranges: b in [0,254], x,y in [-131072,131071], z in [-32768,32767],
 * t in [0,15].  Anything outside raises SPS_ERR_COORD_RANGE at the next status check. */
#define SPS_X_BIAS 131072
#define SPS_Z_BIAS 32768

typedef struct sps_ctx sps_ctx;   /* coordinate manager + scratch for one stream  */
typedef struct sps_net sps_net;   /* BN-folded, packed CustomMinkUNet weights      */

const char* sps_version(void);
const char* sps_last_error(void);           /* text of the last SPS_ERR_CUDA on this thread */

/* ---------------------------------------------------------------- context / workspace ---- */
/* Bytes of device workspace needed for inputs of at most `max_points` rows. */
size_t sps_workspace_bytes(int64_t max_points);
/* Replaces the per-forward ME CoordinateManager (src/sps/models/models.py:24). */
int sps_ctx_create(sps_ctx** ctx, void* d_workspace, size_t workspace_bytes, int64_t max_points);
int sps_ctx_destroy(sps_ctx* ctx);
/* Host-synchronising: waits for `stream`, returns the sticky device status word
 * (SPS_OK / SPS_ERR_COORD_RANGE / SPS_ERR_CAPACITY) and clears it. */
int sps_ctx_status(sps_ctx* ctx, void* stream);

typedef struct sps_level_view {
  const uint64_t* keys;     /* [count] packed voxel keys, first-occurrence order            */
  const int32_t* count;     /* device scalar: number of voxels at this level                */
  const int32_t* nbr3;      /* [81][ld] 3x3x3x3 kernel map at this level's tensor stride    */
  const int32_t* nbr5;      /* [125][ld] 5x5x5x1 kernel map (level 0 only, else NULL)       */
  const int32_t* parent;    /* [count] parent*8 + child-offset index into level+1 (NULL at 4)*/
  const int32_t* child;     /* [8][ld] child table of the level BELOW (NULL at level 0)     */
  int64_t ld;               /* leading dimension (in voxels) of nbr3/nbr5/child             */
  /* Processing order of the 3x3x3x3 convolutions after a fused forward that shape-sorted this level (levels 0-3 of
   * inputs >= 400 000 rows, or sps_ctx_set_pattern_sort(ctx, 2)); all NULL otherwise.  These are what
   * sps_conv_args.perm / tile_mask / tile_slices take: a caller can run its own layers on the forward's maps. */
  const int32_t* perm;          /* [count] rows in neighbourhood-shape order                                  */
  const uint32_t* tile_mask;    /* [ceil(count/128)][4] present-offset masks of the tiles in that order       */
  const int32_t* tile_slices;   /* [tiles][SPS_TILE_SLICE_ENTRIES][128] kernel map gathered per tile          */
} sps_level_view;
/* Valid after sps_voxelize (+ sps_build_maps for the maps).  After a FUSED forward (sps_forward*, sps_infer_scan) on
 * an input large enough for the shape sort (>= 400 000 rows), the 3x3x3x3 tables of levels 0-3 hold only their PRESENT
 * entries (absent ones are not rewritten to -1: every reader inside the library goes through the presence words):
 * the view then carries nbr3 == NULL for every level; call sps_build_maps to get the complete tables back
 * (sps_ctx_pair_count counts from the presence words and works in both states). */
int sps_ctx_level(sps_ctx* ctx, int level, sps_level_view* out);
const int32_t* sps_ctx_inverse_map(sps_ctx* ctx);   /* [n] point -> level-0 voxel row        */

/* ---------------------------------------------------------------- a1/a2 voxelisation ---- */
/* `torch.div(coords, [1,vs,vs,vs,1])` + ME.TensorField(...).sparse()
 * (src/sps/models/models.py:21-25): IEEE fp32 division, floor to int32, unique voxels in
 * first-occurrence order, inverse mapping.  d_points: fp32 [n,ld_points] rows (b,x,y,z,t,...). */
int sps_voxelize(sps_ctx* ctx, const float* d_points, int64_t n, int64_t ld_points,
                 float voxel_size, void* stream);
/* Strided coordinate maps (MinkowskiConvolution stride=[2,2,2,1], minkunet.py:64-104) for
 * levels 1..4 plus every kernel map the network needs: 5x5x5x1 at level 0 (minkunet.py:55-60),
 * 3x3x3x3 at levels 0..4 (BasicBlock convs), 2x2x2x1 parent/child tables. */
int sps_build_maps(sps_ctx* ctx, void* stream);
/* Unpack a level's keys into int32 [count,5] rows (b,x,y,z,t) == ME `SparseTensor.C`. */
int sps_unpack_coords(sps_ctx* ctx, int level, int32_t* d_out, void* stream);

/* ---------------------------------------------------------------- convolution ------------ */
#define SPS_CONV_NBR 0    /* stride-1 (or child-table stride-2) conv through a [K][ld] map   */
#define SPS_CONV_UP 1     /* transposed 2x2x2x1: out[child[k][c]] = in[c] @ W[k] for coarse rows c */

#define SPS_TILE_SLICE_ENTRIES 82
#define SPS_IO_F32 0
#define SPS_IO_F16 1
/* sps_conv_args.flags (tensor-core path, fp16 rows): how the fused forward keeps the level-0 tail of the network at
 * ~21 bits although every tensor-core operand is fp16 (tools/precision_study.py):
 *   SPS_CONV_FOLD_LO    cout == 8: rows 8..15 of weight_kmajor hold the LOW parts of the weights (w - fp16(w), as
 *                       fp16); the accumulator's columns 8..15 are added to columns 0..7 in the epilogue.  The
 *                       N = 16 accumulator of an 8-channel layer has those columns anyway: split weights for free.
 *   SPS_CONV_OUT_SPLIT  `out` rows are written as hi|lo pairs: per 8 channels 16 halves, [fp16(v) x 8 | fp16(v - hi) x 8]
 *                       (out_ld counts halves of that doubled row).  A consumer reads such a row as 2 x cin fp16
 *                       channels with its weights duplicated along K (sps_conv_pack_kmajor_f16x, SPS_PACK_IN_SPLIT):
 *                       sum_c (hi_c + lo_c) * w_c, exact products, fp32 accumulation. */
#define SPS_CONV_FOLD_LO 1
#define SPS_CONV_OUT_SPLIT 2
/* SPS_CONV_MAP_PARENT (tensor-core path, NBR mode, K == 8): `map` is the fine level's parent array -- parent[row] =
 * coarse_row * 8 + k (sps_ctx_level.parent) -- instead of a dense [8][map_ld] table: entry k of a row is (p & 7) == k ? p >> 3 : -1.
 * The transposed convolution (minkunet.py:107-147) needs no up-map this way. */
#define SPS_CONV_MAP_PARENT 4
typedef struct sps_conv_args {
  int mode;                 /* SPS_CONV_NBR | SPS_CONV_UP                                    */
  int K;                    /* kernel volume (125, 81, 8, 1)                                 */
  int cin, cout;
  const int32_t* map;       /* NBR: [K][map_ld] input rows (-1 = absent); K==1 && map==NULL
                               means identity (1x1 conv).  UP: [8][map_ld] child table of the
                               coarse (input) level; n_out then counts the COARSE rows        */
  int64_t map_ld;
  const int32_t* n_out;     /* device scalar: number of output rows                          */
  int64_t n_out_max;        /* host upper bound used to size the launch                      */
  const float* in;  int64_t in_ld;    /* fp32 rows; `in` already points at the channel slice */
  const float* weight;      /* [K][cin][cout] fp32 (ME `.kernel` layout), BN scale folded by
                               the caller if wanted                                          */
  const float* shift;       /* [cout] added after the contraction (folded BN shift/bias), or NULL */
  /* optional fused 1x1 term: + in2[row] @ weight2  (BasicBlock downsample, resnet.py:97-108) */
  const float* in2; int64_t in2_ld; int cin2; const float* weight2;
  /* optional identity residual: + res[row]  (BasicBlock without downsample)                */
  const float* res; int64_t res_ld;
  int relu;
  float* out; int64_t out_ld;         /* may be a channel slice of a concat buffer (ME.cat)  */
  /* optional fused head: logit[row] = dot(relu_out[row], head_w) + head_b  (final 1x1 conv,
   * minkunet.py:152-158,219); requires cout == 8; `out` may then be NULL                   */
  const float* head_w; float head_b; float* head_out;
  /* tensor-core path (optional): the same weights (and weight2) as a K-major [cout][kmajor_ld]
   * matrix, TF32-rounded, made by sps_conv_pack_kmajor; NULL -> only the CUDA-core kernel fits */
  const float* weight_kmajor; int64_t kmajor_ld;
  int round_out;            /* store outputs rounded to TF32 (nearest), so that a following
                               tensor-core layer does not truncate its operand               */
  const uint32_t* tile_mask; /* tensor-core path: [ceil(n_out/128)][4] present-offset bitmasks of
                               `map` per 128-row tile (sps_kernel_map_tile_masks); NULL -> CUDA-core */
  const int32_t* perm;      /* optional processing order: tile t covers output rows perm[128t..128t+127]
                               (tile_mask must describe the tiles in THIS order); results do not
                               depend on it.  NULL = identity                                  */
  const int32_t* tile_slices; /* optional, with perm: the kernel map already gathered per tile --
                               [tile][SPS_TILE_SLICE_ENTRIES][128] int32, entry e < popcount(mask) = input
                               rows of the tile's e-th present offset, entry popcount(mask) = the tile's own
                               rows (perm).  NULL = the kernel gathers from `map` through `perm` itself */
  int io_dtype;             /* SPS_IO_F32 (0): `in`, `in2`, `res`, `out` are fp32 rows.  SPS_IO_F16: they point
                               at fp16 rows (leading dimensions in halves, multiples of 8) and weight_kmajor is
                               the sps_conv_pack_kmajor_f16 matrix: the fused forward's storage format
                               (same 10-bit mantissa as the TF32 operands, half the bytes per gathered row)   */
  int backend;              /* SPS_BACKEND_*: which kernel family serves this call (AUTO: tensor cores where
                               the layer shape and the optional inputs allow, CUDA cores otherwise)          */
  int flags;                /* SPS_CONV_FOLD_LO | SPS_CONV_OUT_SPLIT (fp16 rows on the tensor-core path only) | SPS_CONV_MAP_PARENT */
  int cin_split;            /* 0, or the channels of the FIRST of two segments of `in` rows (a concat buffer,
                               minkunet.py:192: 64 + 32, 32 + 16 or 16 + 8 channels, fp16 rows, tensor-core path):
                               the K axis of weight_kmajor (sps_conv_pack_kmajor_f16s) then walks segment by
                               segment, so that neither carries padded columns.  Results do not depend on it */
} sps_conv_args;
/* MinkowskiConvolution / MinkowskiConvolutionTranspose (+ folded MinkowskiBatchNorm, ReLU,
 * residual) forward: minkunet.py:55-158, resnet.py:97-108, ME BasicBlock.  Served by the tcgen05
 * implicit-GEMM kernel (TF32 / fp16 operands, fp32 accumulate) or the fp32 CUDA-core kernels, see
 * sps_conv_args.backend. */
int sps_conv_fwd(const sps_conv_args* args, void* stream);

/* ---------------------------------------------------------------- network ---------------- */
int sps_net_create(sps_net** net);
int sps_net_destroy(sps_net* net);
/* Hand over one state_dict tensor (host fp32, ME layout; names without the Lightning prefix
 * `model.MinkUNet.`, cf. src/sps/datasets/util.py:33-39).  1x1 kernels may be [Cin,Cout] or
 * [1,Cin,Cout].  `*.num_batches_tracked` entries are ignored by the caller. */
int sps_net_set_tensor(sps_net* net, const char* name, const float* h_data, int64_t numel);
/* Which column of `final` ([8, Cout] kernel, [1, Cout] bias) the forward returns, and whether the sigmoid of
 * models.py:29 is applied.  Default (0, 1) = SPSModel.  MOS4DNet (c_ws/src/mos4d/scripts/mos4d.py:15,32:
 * CustomMinkUNet(1, 3, D=4), `out.features[:, 2]`, no sigmoid) = (2, 0).  Call before sps_net_finalize. */
int sps_net_set_output(sps_net* net, int channel, int apply_sigmoid);
size_t sps_net_device_bytes(void);
/* Folds every BatchNorm (eval) into the preceding kernel + a shift, packs, uploads into the
 * caller's device buffer.  Fails with SPS_ERR_BAD_ARG if a tensor of CustomMinkUNet(1,1,D=4)
 * is missing or mis-sized. */
int sps_net_finalize(sps_net* net, void* d_weights, size_t bytes, void* stream);

/* SPSModel.forward (src/sps/models/models.py:20-30) end to end on device buffers:
 * voxelize -> maps -> CustomMinkUNet (minkunet.py:161-219) -> slice + sigmoid.
 * d_scores: fp32 [n].  No host synchronisation. */
int sps_forward(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n,
                int64_t ld_points, float voxel_size, float* d_scores, void* stream);
/* As sps_forward with one input feature per point (d_feat fp32 [n]): the voxel feature is the mean of its points'
 * features (ME.TensorField(features=[N,1]).sparse(), UNWEIGHTED_AVERAGE) -- MapMOSNet.forward,
 * c_ws/src/mapmos/scripts/mapmos.py:59-83 (index-normalised features, raw logits: sps_net_set_output(net, 0, 0)). */
int sps_forward_features(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n,
                         int64_t ld_points, const float* d_feat, float voxel_size, float* d_scores,
                         void* stream);
/* Same through HOST buffers (pinned or pageable): H2D of the points into the context's staging
 * area, forward, D2H of the scores, stream synchronise, status check. This is the call
 * `util.infer` (src/sps/datasets/util.py:163-184) maps onto. */
int sps_forward_host(sps_ctx* ctx, const sps_net* net, const float* h_points, int64_t n,
                     int64_t ld_points, float voxel_size, float* h_scores, void* stream);
/* U-Net only, on the maps already built in `ctx` (for layer-wise parity tests):
 * d_feat0 fp32 [V0] input feature, d_logits fp32 [V0] output of `final`. */
int sps_unet_forward(sps_ctx* ctx, const sps_net* net, const float* d_feat0, float* d_logits,
                     void* stream);
/* SparseTensor.slice + sigmoid (models.py:28-29): scores[p] = sigmoid(logits[inv[p]]). */
int sps_devox_sigmoid(const float* d_logits, const int32_t* d_inv, int64_t n, float* d_scores,
                      void* stream);
/* Number of kernels the last fused forward of this context enqueued (bench.py's gpu_launches claim). */
int sps_ctx_launch_count(const sps_ctx* ctx);

/* ---------------------------------------------------------------- submap selection ------- */
typedef struct sps_map sps_map;  /* replicated base-map voxel hash, built once per process  */
size_t sps_map_bytes(int64_t max_map_points);
/* util.to_coords_features(map,'map',ds) + the map half of util.prune
 * (src/sps/datasets/util.py:67-82,86-89): trunc(xyz/ds) int32, de-duplicated, hashed ONCE
 * instead of per scan.  d_map_xyz: fp32 [n,3]. */
int sps_map_build(sps_map** map, void* d_storage, size_t bytes, const float* d_map_xyz,
                  int64_t n, float ds, void* stream);
int sps_map_destroy(sps_map* map);
/* util.prune (src/sps/datasets/util.py:85-114): voxels present in both the map and the scan,
 * returned as fp32 corners `coords*ds` [m,3]; d_counts[0] = m, d_counts[1] = number of unique
 * scan voxels (the function's second return value).  d_scratch: sps_map_bytes(n_scan) bytes. */
int sps_submap_crop_voxel(const sps_map* map, const float* d_scan_xyz, int64_t n_scan,
                          void* d_scratch, size_t scratch_bytes, float* d_out_xyz,
                          int32_t* d_counts, void* stream);
/* Radius crop of the raw map (c_ws/src/mapmos/scripts/mapmos_node.py:63-68): indices of map
 * points with ||p - center|| <= radius (float64, as numpy promotes) in map order; d_count[0] = how many. */
int sps_submap_crop_radius(const float* d_map_xyz, int64_t n, const double center[3], double radius,
                           int32_t* d_out_idx, int32_t* d_count, void* d_scratch,
                           size_t scratch_bytes, void* stream);
/* Assembly of the network input (util.add_timestamp + vstack/hstack, util.py:156-174):
 * rows [b, x,y,z, t] with the scan rows (t=1) first and the submap rows (t=0) after. */
int sps_assemble(const float* d_scan_xyz, int64_t n_scan, const float* d_sub_xyz,
                 const int32_t* d_n_sub, int64_t n_sub_max, float batch_index, float* d_out,
                 void* stream);

/* One scan of the ROS deployment path (c_ws/src/sps_filter/scripts/sps_node.py:111-120):
 * util.prune against the replicated map hash -> util.infer assembly -> SPSModel.forward ->
 * scores of the scan rows only (util.py:180).  No host synchronisation: the submap size stays
 * on the device.  ctx must be sized for 2*n_scan rows; d_counts as in sps_submap_crop_voxel. */
size_t sps_infer_scan_scratch_bytes(int64_t n_scan);
int sps_infer_scan(sps_ctx* ctx, const sps_net* net, const sps_map* map, const float* d_scan_xyz,
                   int64_t n_scan, float voxel_size, float* d_scores, void* d_scratch,
                   size_t scratch_bytes, int32_t* d_counts, void* stream);

/* ---------------------------------------------------------------- ROS-path scan I/O (SURVEY 8f rank 3) --- */
/* util.to_numpy (src/sps/datasets/util.py:146-153): the payload of a sensor_msgs/PointCloud2 -> fp32 [height*width,
 * nfields], every field cast to float32, fields in message order.  d_data: the message's `data` bytes on the device;
 * h_offsets / h_datatypes: PointField.offset / PointField.datatype (1 INT8 ... 7 FLOAT32, 8 FLOAT64) of each field. */
int sps_pointcloud2_unpack(const void* d_data, int64_t width, int64_t height, int64_t point_step, int64_t row_step,
                           int nfields, const int32_t* h_offsets, const int32_t* h_datatypes, int is_bigendian,
                           float* d_out, void* stream);
/* util.transform_point_cloud (util.py:187-194) as sps_node.py:103-107 uses it: fp32 points promoted to float64,
 * homogeneous product with the row-major 4x4 float64 matrix (host pointer), division by the homogeneous coordinate,
 * result rounded to fp32.  d_xyz: fp32 [n, ld>=3]; d_out: fp32 [n,3]. */
int sps_transform_points(const float* d_xyz, int64_t ld, int64_t n, const double* h_matrix, float* d_out, void* stream);
/* sps_node.py:148-149 + util.to_rosmsg (util.py:117-143): the scan rows (sensor frame x, y, z, intensity = columns
 * 0..3 of d_scan, fp32 [n, ld>=4]) whose score is <= eps, in scan order, as the PointCloud2 payload the node publishes
 * (point_step 16, fields x/y/z/intensity FLOAT32): d_out fp32 [n,4] (16-byte aligned), d_count[0] = rows kept.
 * d_scratch: sps_pointcloud2_pack_scratch_bytes(n) bytes, 256-byte aligned. */
size_t sps_pointcloud2_pack_scratch_bytes(int64_t n);
int sps_pointcloud2_pack(const float* d_scan, int64_t ld, int64_t n, const float* d_scores, float eps, float* d_out,
                         int32_t* d_count, void* d_scratch, size_t scratch_bytes, void* stream);

/* ---------------------------------------------------------------- offline-loader submap --- */
/* BLTDataset.select_closest_points (src/sps/datasets/blt_dataset.py:222-226,258-271):
 *     kd_tree_scan.query_ball_tree(kd_tree_target, VOXEL_SIZE) -> np.concatenate(lists)
 * = for every scan point, in scan order, the indices of ALL map points within Euclidean distance
 * <= radius (evaluated in fp64 like scipy), duplicates kept across scan points.  The two kd-trees
 * are replaced by a uniform grid of edge `radius` over the static map (27-cell ball query). */
typedef struct sps_ballmap sps_ballmap;
size_t sps_ballmap_bytes(int64_t n_map);
/* Built once per map (= kd_tree_target, blt_dataset.py:193).  d_map_xyz fp32 [n,3] must stay alive. */
int sps_ballmap_build(sps_ballmap** bm, void* d_storage, size_t bytes, const float* d_map_xyz,
                      int64_t n, double radius, void* stream);
int sps_ballmap_destroy(sps_ballmap* bm);
size_t sps_ball_query_scratch_bytes(int64_t n_scan);
/* d_out_idx int32 [out_capacity]: map indices, scan point by scan point; inside one scan point's
 * list: cell by cell (dz, dy, dx ascending), ascending map index inside a cell (scipy's order inside
 * a list is its tree-traversal order; the lists hold the same indices).  d_offsets (optional) int32
 * [n_scan+1]: list i = d_out_idx[d_offsets[i] .. d_offsets[i+1]).  *d_total = number of hits (the
 * caller compares it with out_capacity after its synchronisation: entries past the capacity are
 * counted but not written). */
int sps_submap_ball_query(const sps_ballmap* bm, const float* d_scan_xyz, int64_t n_scan,
                          int32_t* d_offsets, int32_t* d_out_idx, int64_t out_capacity, int32_t* d_total,
                          void* d_scratch, size_t scratch_bytes, void* stream);

/* A whole evaluation batch from its scans: BLTDataset.__getitem__ per scan (blt_dataset.py:209-243, no augmentation)
 * + collate_fn (blt_dataset.py:173-182).  d_scans fp32 [n_total, ld >= 4] = x, y, z, label of `batch` scans already in
 * the map frame, concatenated; h_offsets (HOST) int64 [batch + 1]: scan b = rows h_offsets[b] .. h_offsets[b+1], with
 * h_offsets[0] == 0, non-decreasing, n_total = h_offsets[batch]; batch in 1..255 (the batch index is the voxel key's
 * b field).  d_rows fp32 [row_capacity, 6] = (b, x, y, z, t, label) in collate order: for b = 0..batch-1 the scan
 * rows of b (t = 1, their label), then b's submap rows map[idx] (t = 0, label 1), idx exactly what
 * sps_submap_ball_query returns for that scan alone (same order, duplicates kept).  d_row_offsets int32 [batch + 1]:
 * scan b's rows start at d_row_offsets[b]; *d_n_rows = number of rows.  When that exceeds row_capacity nothing is
 * written past the capacity, and *d_n_rows and d_row_offsets still hold the true values (the caller compares after
 * its synchronisation).  d_scratch: sps_radius_batch_scratch_bytes(n_total, batch) bytes, 256-byte aligned.
 * No host synchronisation.  SPS_ERR_BAD_ARG: a null pointer, ld < 4, batch outside 1..255, offsets not starting at 0
 * or decreasing, misaligned scratch; SPS_ERR_CAPACITY: scratch too small. */
size_t sps_radius_batch_scratch_bytes(int64_t n_scan_total, int batch);
int sps_radius_batch(const sps_ballmap* bm, const float* d_scans, int64_t ld, const int64_t* h_offsets, int batch,
                     float* d_rows, int64_t row_capacity, int32_t* d_row_offsets, int32_t* d_n_rows, void* d_scratch,
                     size_t scratch_bytes, void* stream);
/* scripts/predict.py:70-83 over such a batch in one call: sps_radius_batch -> SPSModel.forward on the rows
 * (models.py:20-30; the row count stays on the device, as in sps_infer_scan) -> SPSNet.predict_step's per-scan metric
 * partials (models.py:84-104).  d_scan_scores fp32 [n_total]: the scores of the scan rows, in input order;
 * d_counts int64 [batch][4] and d_sums double [batch][5]: per scan, laid out as in sps_confusion_counts (threshold eps).
 * The rows are written to d_rows as by sps_radius_batch; the scores of all rows go to the context's own buffer.
 * row_capacity sizes the forward's launches and, like a row count, decides the shape sort of sps_ctx_set_pattern_sort
 * mode 1: pick it on the same side of 400 000 as the row count for scores bit-identical to sps_forward on the rows.
 * When the rows do not fit row_capacity, the forward runs on none of them, the scan scores are NaN, the partials zero,
 * *d_n_rows holds the true count and the context's status word reports SPS_ERR_CAPACITY at the next sps_ctx_status.
 * No host synchronisation.  Errors as sps_radius_batch, plus SPS_ERR_CAPACITY when row_capacity > the context's
 * max_points. */
int sps_predict_radius_batch(sps_ctx* ctx, const sps_net* net, const sps_ballmap* bm, const float* d_scans, int64_t ld,
                             const int64_t* h_offsets, int batch, float* d_rows, int64_t row_capacity,
                             int32_t* d_row_offsets, int32_t* d_n_rows, void* d_scratch, size_t scratch_bytes,
                             float voxel_size, float eps, float* d_scan_scores, int64_t* d_counts, double* d_sums,
                             void* stream);

/* ---------------------------------------------------------------- arithmetic / processing order ---- */
/* Which kernels serve the fused forward of a context (and, through sps_conv_args.backend, one sps_conv_fwd call):
 *   SPS_BACKEND_AUTO (0)  tcgen05 implicit GEMM on fp16 rows (fp16 operands, fp32 accumulate and epilogue); the
 *                         8-output-channel layers carry split (hi + lo) fp16 weights in the spare accumulator columns
 *                         and the level-0 tail of the network (conv0 output, convtr7p2s2, block8) stores its
 *                         activations as fp16 hi|lo pairs -- what holds the 2e-3 score bar on spread-out scores;
 *   SPS_BACKEND_FP32 (1)  fp32 CUDA-core kernels everywhere (exact fp32);
 *   SPS_BACKEND_TF32 (2)  as AUTO but fp32 rows everywhere, TF32 operands in the tensor-core layers;
 *   SPS_BACKEND_F16  (3)  = AUTO regardless of build flags. */
#define SPS_BACKEND_AUTO 0
#define SPS_BACKEND_FP32 1
#define SPS_BACKEND_TF32 2
#define SPS_BACKEND_F16 3
int sps_ctx_set_conv_backend(sps_ctx* ctx, int backend);
/* The fused forward can visit the rows of the 3x3x3x3 convolutions (levels 0-3) in an order sorted by
 * neighbourhood shape: fewer kernel offsets per 128-row tile.  mode 0: never (physical row order); 1 (default): for
 * inputs of >= 400 000 rows (smaller ones are launch-bound); 2: always.  Results do not depend on it beyond the last
 * bit of a stored fp16 activation. */
int sps_ctx_set_pattern_sort(sps_ctx* ctx, int mode);
/* fp16 twins of sps_conv_kmajor_ld / sps_conv_pack_kmajor below (out: __half [cout][ld]; per offset 1, 2, 4 or
 * 8k groups of 8 channels). */
int64_t sps_conv_kmajor_ld_f16(int K, int cin, int cin2);
int sps_conv_pack_kmajor_f16(const float* w, int K, int cin, int cout, const float* w2, int cin2, void* out);
/* The same with the two precision options of sps_conv_args.flags.  pack_flags: SPS_PACK_IN_SPLIT = `in` rows are
 * hi|lo pairs (every 8-channel group of W[k] appears twice along K; the kernel is then called with cin = 2 x cin),
 * SPS_PACK_IN2_SPLIT = the same for the fused 1x1 term, SPS_PACK_FOLD_LO = cout == 8 and rows 8..15 of the matrix hold
 * the low parts of rows 0..7 (the matrix then has 16 rows).  ld and the packed rows count the DOUBLED channels. */
#define SPS_PACK_IN_SPLIT 1
#define SPS_PACK_IN2_SPLIT 2
#define SPS_PACK_FOLD_LO 4
int64_t sps_conv_kmajor_ld_f16x(int K, int cin, int cin2, int pack_flags);
int sps_conv_pack_kmajor_f16x(const float* w, int K, int cin, int cout, const float* w2, int cin2, int pack_flags, void* out);
/* The same for two-segment input rows (sps_conv_args.cin_split; not together with SPS_PACK_IN_SPLIT): along K the first
 * cin_split channels of every offset (padded to 1, 2, 4 or 8k groups), then the remaining cin - cin_split channels of every
 * offset (unpadded), then the 1x1 term.  cin_split = 0: identical to the _f16x functions. */
int64_t sps_conv_kmajor_ld_f16s(int K, int cin, int cin2, int pack_flags, int cin_split);
int sps_conv_pack_kmajor_f16s(const float* w, int K, int cin, int cout, const float* w2, int cin2, int pack_flags, int cin_split,
                              void* out);
/* 1 when the tensor-core kernel can stage its 64-channel weight slabs through TMA (cp.async.bulk.tensor): the driver's
 * cuTensorMapEncodeTiled was found (cudaGetDriverEntryPoint) and SPS_NO_TMA_B is not set in the environment; 0: every
 * weight stage goes through cp.async (same results). */
int sps_tma_weights_available(void);
/* Per-tile present-offset bitmasks of a kernel map (K <= 81) for the tensor-core path:
 * d_masks uint32 [ceil(n_out_max/128)][4]. */
int sps_kernel_map_tile_masks(const int32_t* d_map, int64_t map_ld, int K, const int32_t* d_n_out,
                              int64_t n_out_max, uint32_t* d_masks, void* stream);
/* Host helper for the tensor-core path: ME-layout weights [K][cin][cout] (+ optional fused 1x1
 * term w2 [cin2][cout]) -> K-major [cout][ld], ld = sps_conv_kmajor_ld(K,cin,cin2), values
 * rounded to TF32 (nearest even).  `out` is a HOST buffer of cout*ld floats. */
int64_t sps_conv_kmajor_ld(int K, int cin, int cin2);
int sps_conv_pack_kmajor(const float* w, int K, int cin, int cout, const float* w2, int cin2,
                         float* out);

/* ---------------------------------------------------------------- measurement ------------ */
/* Per-stage CUDA-event timing of the fused forward of one context on its launch stream (bench.py roofline
 * figures).  sps_profile_read synchronises and returns up to `max` segments: names[i*32..] and ms[i]. */
int sps_profile_enable(sps_ctx* ctx, int on);
int sps_profile_read(sps_ctx* ctx, char* names, float* ms, int max, int* n_out);
/* Number of (in,out) pairs of a kernel map of the last forward: kind 3 (3x3x3x3), 5 (5x5x5x1,
 * level 0) or 8 (children of `level`).  Host-synchronising.  Used for algorithmic FLOP counts. */
int sps_ctx_pair_count(sps_ctx* ctx, int level, int kind, int64_t* h_out, void* stream);

/* SPSNet.predict_step metric partials (src/sps/models/models.py:84-104, util.py:285-299) of one
 * scan on the device: rows fp32 [n,ld>=6] = (b,x,y,z,t,label); only rows with t == 1 (and
 * b == batch_index when batch_index >= 0) count.  d_counts int64[4] = TP,TN,FP,FN with class 1 =
 * unstable (value >= eps); d_sums double[5] = n, sum((score-label)^2), sum(label),
 * sum(label^2), sum(score).  These are what the NCCL gather of metrics carries. */
int sps_confusion_counts(const float* d_scores, const float* d_rows, int64_t ld_rows, int64_t n,
                         float batch_index, float eps, int64_t* d_counts, double* d_sums,
                         void* stream);

/* ---------------------------------------------------------------- layer-level pieces ----- */
/* ME.TensorField(...).sparse() feature reduction (UNWEIGHTED_AVERAGE, models.py:24-25): mean of the
 * point features per level-0 voxel of the last sps_voxelize.  d_out [>= n rows, channels],
 * d_count [>= n] scratch. */
int sps_voxel_mean(sps_ctx* ctx, const float* d_feat, int64_t ld, int channels, float* d_out,
                   float* d_count, void* stream);
/* The same without the division: per-voxel SUM of the point features and the member count (d_count).  This is the
 * feature rule of ME.MinkowskiUnion (coincident coordinates add, src/sps/datasets/util.py:98-99). */
int sps_voxel_sum(sps_ctx* ctx, const float* d_feat, int64_t ld, int channels, float* d_out,
                  float* d_count, void* stream);
/* SparseTensor.slice(tensor_field) (models.py:28): out[p, :] = F[inv[p], :]. */
int sps_gather_rows(const float* d_f, int64_t ld, int channels, const int32_t* d_inv, int64_t n,
                    float* d_out, void* stream);
/* MinkowskiBatchNorm (eval: per-channel affine) / MinkowskiReLU on a feature matrix. */
int sps_affine_relu(const float* d_x, int64_t ld, int channels, int64_t n, const float* d_scale,
                    const float* d_shift, int relu, float* d_y, int64_t ldy, void* stream);

/* Small helpers so that host code needs no second CUDA binding. */
int sps_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes, void* stream);
int sps_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SPS_B200_H */
