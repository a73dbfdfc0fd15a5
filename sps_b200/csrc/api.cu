// Context management, workspace carve-up, status plumbing and small helpers of the C ABI.
#include <cstdio>
#include <cstring>
#include <vector>
#include "ctx.h"

namespace sps {

static thread_local char g_err[512] = "";

int set_cuda_error(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s: %s", what, cudaGetErrorString(e));
  return SPS_ERR_CUDA;
}

// Bump carve of the workspace; with base == nullptr it only measures.
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base((char*)b) {}
  template <class T>
  T* take(size_t count) {
    off = (off + 255) & ~size_t(255);
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += count * sizeof(T);
    return p;
  }
};

static size_t carve(sps_ctx* c, void* base, int64_t max_points) {
  Carver cv(base);
  const int64_t N = max_points;
  const int64_t ld = (N + 31) & ~int64_t(31);
  c->max_points = N;
  c->ld = ld;
  // Device scalars, one 128-byte line per role: counts[0..4] + n_dev are READ by every thread of every map kernel,
  // the words that kernels hit with atomics (scan tickets, the block-id counter, the status word) get their own lines.
  c->counts = cv.take<int32_t>(256);
  c->n_dev = c->counts + 5;
  c->ticket = reinterpret_cast<uint32_t*>(c->counts + 32);
  c->nblocks = c->counts + 64;
  c->tplanes = c->counts + 160;
  c->up_cls = c->counts + 192;
  c->status = c->counts + 96;
  c->staging = cv.take<float>((size_t)N * 8);
  c->scores = cv.take<float>(N);
  c->table_cap = table_capacity(N);
  c->table = cv.take<Slot>(c->table_cap);
  c->slot_of = cv.take<uint32_t>(N);
  c->rank = cv.take<int32_t>(N);
  c->block_sums = cv.take<int32_t>(N / kScanBlock + 2);
  c->inv = cv.take<int32_t>(N);
  for (int L = 0; L < SPS_NUM_LEVELS; ++L) {
    c->keys[L] = cv.take<unsigned long long>(N);
    c->nbr3[L] = cv.take<int32_t>((size_t)81 * ld);
    c->tmask3[L] = cv.take<uint32_t>((size_t)(ld / 128 + 1) * 4);
    c->ptmask[L] = cv.take<uint32_t>((size_t)(ld / 128 + 1) * 4);
    c->perm[L] = cv.take<int32_t>(N);
    c->tslice[L] = cv.take<int32_t>((size_t)(ld / 128 + 1) * SPS_TILE_SLICE_ENTRIES * 128);
    c->btab[L] = cv.take<Slot>(c->table_cap);
    c->bcells[L] = cv.take<int32_t>((size_t)N * 64);
    c->bocc[L] = cv.take<unsigned long long>(N);
    c->vmask[L] = cv.take<uint32_t>((size_t)4 * ld);
    c->parent[L] = (L < SPS_NUM_LEVELS - 1) ? cv.take<int32_t>(N) : nullptr;
    c->child[L] = (L > 0) ? cv.take<int32_t>((size_t)8 * ld) : nullptr;
    c->perm_up[L] = (L < SPS_NUM_LEVELS - 1) ? cv.take<int32_t>(N) : nullptr;
    c->tmask_up[L] = (L < SPS_NUM_LEVELS - 1) ? cv.take<uint32_t>((size_t)(ld / 128 + 1) * 4) : nullptr;
  }
  c->nbr5 = cv.take<int32_t>((size_t)125 * ld);
  c->tmask8 = cv.take<uint32_t>((size_t)(ld / 128 + 1) * 4);
  for (int j = 0; j < 2; ++j) {
    c->sort_keys[j] = cv.take<uint32_t>((size_t)SPS_NUM_LEVELS * N);
    c->sort_vals[j] = cv.take<int32_t>((size_t)SPS_NUM_LEVELS * N);
  }
  c->sort_hist = cv.take<uint32_t>(1028);
  c->sort_status = cv.take<uint32_t>(((size_t)SPS_NUM_LEVELS * N / 1024 + 2) * 1024);
  for (int b = 0; b < sps_ctx::NBUF; ++b) c->buf[b] = cv.take<float>((size_t)N * kBufWidth[b]);
  return (cv.off + 255) & ~size_t(255);
}

int conv_simt(const sps_conv_args& a, cudaStream_t st);
int conv_umma(const sps_conv_args& a, cudaStream_t st);
bool conv_umma_supports(const sps_conv_args& a);
bool conv_umma_f16_supports(const sps_conv_args& a);

// Kernel family of one convolution call (sps_conv_args.backend; the fused forward passes its context's mode):
// FP32 -> the fp32 CUDA-core kernels; otherwise the tcgen05 kernel whenever the call fits it (fp16 rows: always, there
// is no CUDA-core kernel for them), else the CUDA-core kernels.
int conv_dispatch(const sps_conv_args& a, cudaStream_t st) {
  if (a.io_dtype == SPS_IO_F16) return conv_umma_f16_supports(a) ? conv_umma(a, st) : SPS_ERR_UNSUPPORTED;
  if ((a.flags & ~SPS_CONV_MAP_PARENT) || a.cin_split) return SPS_ERR_UNSUPPORTED;   // split-precision options and K segments exist on fp16 rows only
  if (a.backend != SPS_BACKEND_FP32 && conv_umma_supports(a)) return conv_umma(a, st);
  if (a.flags & SPS_CONV_MAP_PARENT) return SPS_ERR_UNSUPPORTED;                      // the CUDA-core kernels want a dense table
  return conv_simt(a, st);
}

}  // namespace sps

using namespace sps;

extern "C" int sps_ctx_set_conv_backend(sps_ctx* ctx, int backend) {
  if (!ctx || backend < 0 || backend > 3) return SPS_ERR_BAD_ARG;
  ctx->backend = backend;
  return SPS_OK;
}
extern "C" int sps_ctx_set_pattern_sort(sps_ctx* ctx, int mode) {
  if (!ctx || mode < 0 || mode > 2) return SPS_ERR_BAD_ARG;
  ctx->pattern_sort = mode;
  return SPS_OK;
}
extern "C" int sps_ctx_launch_count(const sps_ctx* ctx) { return ctx ? ctx->forward_launches : 0; }
extern "C" const char* sps_version(void) { return "sps_b200 0.1 (sm_100a)"; }
extern "C" const char* sps_last_error(void) { return g_err; }

extern "C" size_t sps_workspace_bytes(int64_t max_points) {
  if (max_points < 1) max_points = 1;
  sps_ctx tmp;
  return carve(&tmp, nullptr, max_points);
}

extern "C" int sps_ctx_create(sps_ctx** out, void* d_workspace, size_t workspace_bytes, int64_t max_points) {
  if (!out || !d_workspace || max_points < 1 || max_points > (int64_t(1) << 28)) return SPS_ERR_BAD_ARG;
  if ((uintptr_t)d_workspace & 255) return SPS_ERR_BAD_ARG;
  sps_ctx* c = new sps_ctx();
  const size_t need = carve(c, d_workspace, max_points);
  if (need > workspace_bytes) { delete c; return SPS_ERR_CAPACITY; }
  c->base = (char*)d_workspace;
  c->bytes = workspace_bytes;
  cudaError_t e = cudaMemset(c->counts, 0, 256 * sizeof(int32_t));
  if (e == cudaSuccess) {  // every 128-row tile of a 2x2x2x1 map may hold all eight offsets
    std::vector<uint32_t> m((size_t)(c->ld / 128 + 1) * 4, 0u);
    for (size_t i = 0; i < m.size(); i += 4) m[i] = 0xFFu;
    e = cudaMemcpy(c->tmask8, m.data(), m.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  }
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { delete c; return set_cuda_error(e, "cudaMemset(ctx scalars)"); }
  *out = c;
  return SPS_OK;
}

extern "C" int sps_ctx_destroy(sps_ctx* ctx) {
  delete ctx;
  return SPS_OK;
}

extern "C" int sps_ctx_status(sps_ctx* ctx, void* stream) {
  if (!ctx) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int32_t word = 0;
  SPS_CUDA_CHECK(cudaMemcpyAsync(&word, ctx->status, sizeof(word), cudaMemcpyDeviceToHost, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  if (word) {
    SPS_CUDA_CHECK(cudaMemsetAsync(ctx->status, 0, sizeof(int32_t), st));
    SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  }
  if (word & kStatusRange) return SPS_ERR_COORD_RANGE;
  if (word & kStatusCapacity) return SPS_ERR_CAPACITY;
  return SPS_OK;
}

extern "C" int sps_ctx_level(sps_ctx* ctx, int level, sps_level_view* v) {
  if (!ctx || !v || level < 0 || level >= SPS_NUM_LEVELS) return SPS_ERR_BAD_ARG;
  v->keys = (const uint64_t*)ctx->keys[level];
  v->count = ctx->counts + level;
  v->nbr3 = ctx->dense_maps ? ctx->nbr3[level] : nullptr;   // sparse tables are never handed out
  v->nbr5 = level == 0 ? ctx->nbr5 : nullptr;
  v->parent = ctx->parent[level];
  v->child = ctx->child[level];
  v->ld = ctx->ld;
  const bool sorted = ctx->have_maps && ctx->have_perm;
  v->perm = sorted ? ctx->perm[level] : nullptr;
  v->tile_mask = sorted ? ctx->ptmask[level] : nullptr;
  v->tile_slices = sorted ? ctx->tslice[level] : nullptr;
  return SPS_OK;
}

extern "C" const int32_t* sps_ctx_inverse_map(sps_ctx* ctx) { return ctx ? ctx->inv : nullptr; }

extern "C" int sps_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes, void* stream) {
  if (!h_dst || !d_src) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  SPS_CUDA_CHECK(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  return SPS_OK;
}
extern "C" int sps_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes, void* stream) {
  if (!d_dst || !h_src) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  SPS_CUDA_CHECK(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  return SPS_OK;
}

// ---------------------------------------------------------------- profiling ---------------
#include "profile.h"
namespace sps {
static cudaEvent_t next_event(sps_ctx* c) {
  if (c->prof_used == c->prof_ev.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    c->prof_ev.push_back(e);
  }
  return c->prof_ev[c->prof_used++];
}
void prof_begin(sps_ctx* c, cudaStream_t st) {
  if (!c->prof) return;
  c->prof_used = 0;
  c->prof_names.clear();
  cudaEventRecord(next_event(c), st);
}
void prof_mark(sps_ctx* c, const char* name, cudaStream_t st) {
  if (!c->prof || c->prof_used == 0) return;
  cudaEventRecord(next_event(c), st);
  c->prof_names.push_back(name);
}
}  // namespace sps

extern "C" int sps_profile_enable(sps_ctx* ctx, int on) {
  if (!ctx) return SPS_ERR_BAD_ARG;
  ctx->prof = on != 0;
  ctx->prof_used = 0;
  ctx->prof_names.clear();
  return SPS_OK;
}

extern "C" int sps_profile_read(sps_ctx* ctx, char* names, float* ms, int max, int* n_out) {
  if (!ctx || !names || !ms || !n_out || max < 0) return SPS_ERR_BAD_ARG;
  int n = (int)ctx->prof_names.size();
  if (n > max) n = max;
  if (ctx->prof_used > 0) SPS_CUDA_CHECK(cudaEventSynchronize(ctx->prof_ev[ctx->prof_used - 1]));
  for (int i = 0; i < n; ++i) {
    SPS_CUDA_CHECK(cudaEventElapsedTime(&ms[i], ctx->prof_ev[i], ctx->prof_ev[i + 1]));
    snprintf(names + 32 * i, 32, "%s", ctx->prof_names[i].c_str());
  }
  *n_out = n;
  return SPS_OK;
}

namespace sps {
// pairs of a 3x3x3x3 map from the per-voxel presence words (valid also when the tables hold only present entries)
__global__ void k_count_presence(const uint32_t* __restrict__ vmask, int64_t ld, const int32_t* __restrict__ n_ptr,
                                 unsigned long long* out) {
  const int n = *n_ptr;
  unsigned long long local = 0;
  for (int64_t o = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; o < n; o += (int64_t)gridDim.x * blockDim.x) {
    const uint4 m = reinterpret_cast<const uint4*>(vmask)[o];       // [ld][4]: the three planes of a voxel side by side
    local += __popc(m.x) + __popc(m.y) + __popc(m.z);
  }
  for (int d = 16; d; d >>= 1) local += __shfl_down_sync(0xffffffffu, local, d);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(out, local);
}
__global__ void k_count_nonneg(const int32_t* __restrict__ map, int64_t ld, int K, const int32_t* __restrict__ n_ptr,
                               unsigned long long* out) {
  const int n = *n_ptr;
  const int64_t total = (int64_t)K * n;
  unsigned long long local = 0;
  for (int64_t idx = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    const int k = (int)(idx / n), o = (int)(idx - (int64_t)k * n);
    local += map[(int64_t)k * ld + o] >= 0;
  }
  for (int d = 16; d; d >>= 1) local += __shfl_down_sync(0xffffffffu, local, d);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(out, local);
}
}  // namespace sps

extern "C" int sps_ctx_pair_count(sps_ctx* ctx, int level, int kind, int64_t* h_out, void* stream) {
  if (!ctx || !h_out || level < 0 || level >= SPS_NUM_LEVELS) return SPS_ERR_BAD_ARG;
  if (!ctx->have_maps || (kind == 5 && !ctx->have_nbr5)) return SPS_ERR_STATE;
  const int32_t* map = kind == 3 ? ctx->nbr3[level] : kind == 5 ? (level == 0 ? ctx->nbr5 : nullptr)
                                                    : kind == 8 ? ctx->child[level] : nullptr;
  const int K = kind == 3 ? 81 : kind == 5 ? 125 : 8;
  if (!map) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  unsigned long long* d_out = reinterpret_cast<unsigned long long*>(ctx->counts + 128);
  SPS_CUDA_CHECK(cudaMemsetAsync(d_out, 0, 8, st));
  if (kind == 3) k_count_presence<<<148 * 8, 256, 0, st>>>(ctx->vmask[level], ctx->ld, ctx->counts + level, d_out);
  else k_count_nonneg<<<148 * 8, 256, 0, st>>>(map, ctx->ld, K, ctx->counts + level, d_out);
  SPS_CUDA_CHECK(cudaGetLastError());
  unsigned long long h = 0;
  SPS_CUDA_CHECK(cudaMemcpyAsync(&h, d_out, 8, cudaMemcpyDeviceToHost, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));
  *h_out = (int64_t)h;
  return SPS_OK;
}

// ---------------------------------------------------------------- per-scan metric partials ----
// SPSNet.predict_step (src/sps/models/models.py:84-104): over the scan rows (t == 1) of ONE scan,
// pred = score < eps ? 0 : 1, gt = label < eps ? 0 : 1 -> TP/TN/FP/FN (class 1 = unstable), plus
// the sums MSE and R2 need.  counts: int64 [4] = TP,TN,FP,FN; sums: double [5] = n, sum(err^2),
// sum(label), sum(label^2), sum(score).
namespace sps {
__global__ void k_confusion(const float* __restrict__ scores, const float* __restrict__ rows, int64_t ld, int64_t n,
                            float batch_index, float eps, unsigned long long* counts, double* sums) {
  unsigned long long c[4] = {0, 0, 0, 0};
  double s[5] = {0, 0, 0, 0, 0};
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float* r = rows + i * ld;
    if (r[4] != 1.0f || (batch_index >= 0.f && r[0] != batch_index)) continue;
    const float sc = scores[i], lb = r[5];
    const int p = sc < eps ? 0 : 1, g = lb < eps ? 0 : 1;
    c[(g == 1 && p == 1) ? 0 : (g == 0 && p == 0) ? 1 : (g == 0 && p == 1) ? 2 : 3] += 1;
    const double e = (double)sc - (double)lb;
    s[0] += 1.0; s[1] += e * e; s[2] += lb; s[3] += (double)lb * lb; s[4] += sc;
  }
  for (int j = 0; j < 4; ++j) {
    for (int d = 16; d; d >>= 1) c[j] += __shfl_down_sync(0xffffffffu, c[j], d);
    if ((threadIdx.x & 31) == 0 && c[j]) atomicAdd(counts + j, c[j]);
  }
  for (int j = 0; j < 5; ++j) {
    for (int d = 16; d; d >>= 1) s[j] += __shfl_down_sync(0xffffffffu, s[j], d);
    if ((threadIdx.x & 31) == 0 && s[j] != 0.0) atomicAdd(sums + j, s[j]);
  }
}
}  // namespace sps

extern "C" int sps_confusion_counts(const float* d_scores, const float* d_rows, int64_t ld_rows, int64_t n,
                                    float batch_index, float eps, int64_t* d_counts, double* d_sums, void* stream) {
  if (!d_scores || !d_rows || ld_rows < 6 || n < 0 || !d_counts || !d_sums) return SPS_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  SPS_CUDA_CHECK(cudaMemsetAsync(d_counts, 0, 4 * sizeof(int64_t), st));
  SPS_CUDA_CHECK(cudaMemsetAsync(d_sums, 0, 5 * sizeof(double), st));
  if (n > 0) {
    int64_t g = (n + 255) / 256;
    if (g > 148 * 8) g = 148 * 8;
    k_confusion<<<(int)g, 256, 0, st>>>(d_scores, d_rows, ld_rows, n, batch_index, eps,
                                        reinterpret_cast<unsigned long long*>(d_counts), d_sums);
    SPS_CUDA_CHECK(cudaGetLastError());
  }
  return SPS_OK;
}

// ---------------------------------------------------------------- layer-level helpers (ME-shaped API) ----
namespace sps {
// ME.TensorField.sparse() with UNWEIGHTED_AVERAGE: voxel feature = mean of its points' features
__global__ void k_voxel_accumulate(const float* __restrict__ feat, int64_t ld, int c, const int32_t* __restrict__ inv,
                                   int64_t n, float* __restrict__ sum, float* __restrict__ cnt) {
  const int64_t total = n * c;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / c;
    const int j = (int)(i - p * c);
    const int v = inv[p];
    if (v < 0) continue;
    atomicAdd(sum + (int64_t)v * c + j, feat[p * ld + j]);
    if (j == 0) atomicAdd(cnt + v, 1.0f);
  }
}
__global__ void k_voxel_divide(float* __restrict__ sum, const float* __restrict__ cnt, int c, const int32_t* __restrict__ v_ptr) {
  const int64_t total = (int64_t)(*v_ptr) * c;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x)
    sum[i] = sum[i] / cnt[i / c];
}
// SparseTensor.slice(field): out[p] = F[inv[p]]
__global__ void k_gather_rows(const float* __restrict__ f, int64_t ld, int c, const int32_t* __restrict__ inv, int64_t n,
                              float* __restrict__ out) {
  const int64_t total = n * c;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / c;
    const int j = (int)(i - p * c);
    const int v = inv[p];
    out[i] = v >= 0 ? f[(int64_t)v * ld + j] : nanf("");
  }
}
// MinkowskiBatchNorm (eval) / MinkowskiReLU: y = x * scale + shift, optional ReLU (scale/shift may be NULL)
__global__ void k_affine_relu(const float* __restrict__ x, int64_t ld, int c, int64_t n, const float* __restrict__ scale,
                              const float* __restrict__ shift, int relu, float* __restrict__ y, int64_t ldy) {
  const int64_t total = n * c;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t p = i / c;
    const int j = (int)(i - p * c);
    float v = x[p * ld + j];
    if (scale) v *= scale[j];
    if (shift) v += shift[j];
    if (relu) v = fmaxf(v, 0.f);
    y[p * ldy + j] = v;
  }
}
static inline int ew_grid(int64_t total) {
  int64_t g = (total + 255) / 256;
  return (int)(g < 1 ? 1 : g > 148 * 16 ? 148 * 16 : g);
}
}  // namespace sps

extern "C" int sps_voxel_mean(sps_ctx* ctx, const float* d_feat, int64_t ld, int channels, float* d_out, float* d_count,
                              void* stream) {
  if (!ctx || !d_feat || !d_out || !d_count || channels < 1 || ld < channels) return SPS_ERR_BAD_ARG;
  if (!ctx->have_l0) return SPS_ERR_STATE;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = ctx->n;
  SPS_CUDA_CHECK(cudaMemsetAsync(d_out, 0, (size_t)n * channels * sizeof(float), st));   // V0 <= n rows
  SPS_CUDA_CHECK(cudaMemsetAsync(d_count, 0, (size_t)n * sizeof(float), st));
  if (n > 0) {
    k_voxel_accumulate<<<ew_grid(n * channels), 256, 0, st>>>(d_feat, ld, channels, ctx->inv, n, d_out, d_count);
    k_voxel_divide<<<ew_grid(n * channels), 256, 0, st>>>(d_out, d_count, channels, ctx->counts + 0);
  }
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" int sps_voxel_sum(sps_ctx* ctx, const float* d_feat, int64_t ld, int channels, float* d_out, float* d_count,
                             void* stream) {
  if (!ctx || !d_feat || !d_out || !d_count || channels < 1 || ld < channels) return SPS_ERR_BAD_ARG;
  if (!ctx->have_l0) return SPS_ERR_STATE;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t n = ctx->n;
  SPS_CUDA_CHECK(cudaMemsetAsync(d_out, 0, (size_t)n * channels * sizeof(float), st));   // V0 <= n rows
  SPS_CUDA_CHECK(cudaMemsetAsync(d_count, 0, (size_t)n * sizeof(float), st));
  if (n > 0) k_voxel_accumulate<<<ew_grid(n * channels), 256, 0, st>>>(d_feat, ld, channels, ctx->inv, n, d_out, d_count);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" int sps_gather_rows(const float* d_f, int64_t ld, int channels, const int32_t* d_inv, int64_t n, float* d_out,
                               void* stream) {
  if (!d_f || !d_inv || !d_out || channels < 1 || n < 0) return SPS_ERR_BAD_ARG;
  if (n) k_gather_rows<<<ew_grid(n * channels), 256, 0, (cudaStream_t)stream>>>(d_f, ld, channels, d_inv, n, d_out);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}

extern "C" int sps_affine_relu(const float* d_x, int64_t ld, int channels, int64_t n, const float* d_scale,
                               const float* d_shift, int relu, float* d_y, int64_t ldy, void* stream) {
  if (!d_x || !d_y || channels < 1 || n < 0) return SPS_ERR_BAD_ARG;
  if (n) k_affine_relu<<<ew_grid(n * channels), 256, 0, (cudaStream_t)stream>>>(d_x, ld, channels, n, d_scale, d_shift, relu,
                                                                             d_y, ldy);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}
