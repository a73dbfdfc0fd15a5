// CustomMinkUNet(1,1,D=4) weights (BN folded) and the fused forward schedule.
//
// Layer graph: src/sps/models/MinkowskiEngine/minkunet.py:52-219 with
// PLANES=(8,16,32,64,64,32,16,8), INIT_DIM=8 (customminkunet.py:10-12), BasicBlock from ME
// (mirrored at c_ws/src/mapmos/scripts/minkunet.py:31-82), downsample = 1x1 conv + BN iff
// inplanes != planes (resnet.py:96-108).  Eval-mode MinkowskiBatchNorm is an affine map per
// channel and is folded into the preceding kernel (scale) and a shift vector; ME.cat is free
// because producers write straight into channel slices of the concat buffers.
#include <map>
#include <string>
#include <vector>
#include <cmath>
#include <cstring>
#include "ctx.h"
#include "profile.h"

namespace sps {
int conv_dispatch(const sps_conv_args& a, cudaStream_t st);

struct ConvW {
  float* w = nullptr;      // [K][cin][cout], BN scale folded
  float* shift = nullptr;  // [cout]
  float* w2 = nullptr;     // fused downsample [cin2][cout], BN scale folded (blocks only)
  float* wt = nullptr;     // K-major TF32 copy for the tcgen05 kernel (81-offset convs)
  int64_t ldk = 0;
  float* wth = nullptr;    // K-major fp16 copy (every conv but conv0): the fp16-storage forward
  int64_t ldkh = 0;
  int pack_flags = 0;      // SPS_PACK_*: how `wth` was packed (split inputs double the K columns, folded low parts add rows)
  int conv_flags = 0;      // SPS_CONV_*: what the fp16 forward asks of the kernel for this layer
  int cin_split = 0;       // fp16 forward: channels of the first of two input segments (sps_conv_args.cin_split), 0 = one segment
  int K = 0, cin = 0, cout = 0, cin2 = 0;
};

constexpr int kPlanes[8] = {8, 16, 32, 64, 64, 32, 16, 8};
constexpr int kInitDim = 8;
}  // namespace sps

struct sps_net {
  std::map<std::string, std::vector<float>> host;
  bool finalized = false;
  int head_channel = 0;      // column of `final` that the forward returns (out_channels > 1: MOS4DNet returns column 2)
  int apply_sigmoid = 1;     // SPSModel: sigmoid(logit); MOS4DNet: the raw logit
  sps::ConvW conv0, down[4], up[4], blk1[8], blk2[8];
  float* head_w = nullptr;
  float head_b = 0.f;
};

using namespace sps;

namespace {

struct Spec { std::string name; int K, cin, cout; };

// total floats of the packed device image
struct Packer {
  std::vector<float> image;
  size_t add(const std::vector<float>& v) {
    size_t off = image.size();
    image.insert(image.end(), v.begin(), v.end());
    while (image.size() % 64) image.push_back(0.f);  // 256-byte alignment of every tensor
    return off;
  }
};

bool get(const sps_net* net, const std::string& name, size_t numel, const std::vector<float>** out) {
  auto it = net->host.find(name);
  if (it == net->host.end() || it->second.size() != numel) return false;
  *out = &it->second;
  return true;
}

// BN eval: y = (x - mean) / sqrt(var + 1e-5) * gamma + beta  ->  scale, shift
bool bn_fold(const sps_net* net, const std::string& prefix, int C, std::vector<double>& scale,
             std::vector<double>& shift) {
  const std::vector<float>*g, *b, *m, *v;
  if (!get(net, prefix + ".bn.weight", C, &g) || !get(net, prefix + ".bn.bias", C, &b) ||
      !get(net, prefix + ".bn.running_mean", C, &m) || !get(net, prefix + ".bn.running_var", C, &v))
    return false;
  scale.resize(C); shift.resize(C);
  for (int c = 0; c < C; ++c) {
    // computed the way nn.BatchNorm1d does in fp32, then widened
    const float inv = 1.0f / std::sqrt((*v)[c] + 1e-5f);
    scale[c] = (double)(*g)[c] * inv;
    shift[c] = (double)(*b)[c] - (double)(*m)[c] * scale[c];
  }
  return true;
}

bool fold_conv(const sps_net* net, const std::string& kname, const std::string& bnname, int K, int cin, int cout,
               std::vector<float>& w, std::vector<double>& shift) {
  const std::vector<float>* k;
  if (!get(net, kname, (size_t)K * cin * cout, &k)) return false;
  std::vector<double> scale;
  if (!bn_fold(net, bnname, cout, scale, shift)) return false;
  w.resize(k->size());
  for (size_t i = 0; i < k->size(); ++i) w[i] = (float)((double)(*k)[i] * scale[i % cout]);
  return true;
}

}  // namespace

extern "C" int sps_net_create(sps_net** net) {
  if (!net) return SPS_ERR_BAD_ARG;
  *net = new sps_net();
  return SPS_OK;
}
extern "C" int sps_net_destroy(sps_net* net) {
  delete net;
  return SPS_OK;
}
extern "C" int sps_net_set_tensor(sps_net* net, const char* name, const float* h_data, int64_t numel) {
  if (!net || !name || !h_data || numel <= 0) return SPS_ERR_BAD_ARG;
  net->host[name] = std::vector<float>(h_data, h_data + numel);
  net->finalized = false;
  return SPS_OK;
}
extern "C" int sps_net_set_output(sps_net* net, int channel, int apply_sigmoid) {
  if (!net || channel < 0) return SPS_ERR_BAD_ARG;
  net->head_channel = channel;
  net->apply_sigmoid = apply_sigmoid != 0;
  net->finalized = false;
  return SPS_OK;
}
extern "C" size_t sps_net_device_bytes(void) { return 32u << 20; }  // 1.85 M parameters, ME + K-major copies, padding

extern "C" int sps_net_finalize(sps_net* net, void* d_weights, size_t bytes, void* stream) {
  if (!net || !d_weights) return SPS_ERR_BAD_ARG;
  Packer pk;
  struct Pending { ConvW* cw; size_t w, shift, w2; bool has_w2; size_t wt = 0; bool has_wt = false; size_t wth = 0; bool has_wth = false; };
  // fp16 K-major copy, stored inside the float image (two halves per float slot)
  auto add_kmajor_h = [&](Pending& p, const std::vector<float>& w, int K, int cin, int cout,
                          const std::vector<float>* w2, int cin2) {
    const int pf = p.cw->pack_flags;
    const int cs = p.cw->cin_split;
    const int64_t ldk = sps_conv_kmajor_ld_f16s(K, cin, cin2, pf, cs);
    const int rows = (pf & SPS_PACK_FOLD_LO) ? 16 : cout;
    std::vector<float> wt(((size_t)rows * ldk + 1) / 2);
    sps_conv_pack_kmajor_f16s(w.data(), K, cin, cout, w2 ? w2->data() : nullptr, cin2, pf, cs, wt.data());
    p.cw->ldkh = ldk;
    p.wth = pk.add(wt);
    p.has_wth = true;
  };
  auto add_kmajor = [&](Pending& p, const std::vector<float>& w, int K, int cin, int cout,
                        const std::vector<float>* w2, int cin2) {
    const int64_t ldk = sps_conv_kmajor_ld(K, cin, cin2);
    std::vector<float> wt((size_t)cout * ldk);
    sps_conv_pack_kmajor(w.data(), K, cin, cout, w2 ? w2->data() : nullptr, cin2, wt.data());
    p.cw->ldk = ldk;
    p.wt = pk.add(wt);
    p.has_wt = true;
  };
  std::vector<Pending> pend;
  // Precision plan of the fp16 forward (tools/precision_study.py): every 8-output-channel layer carries the low parts of
  // its weights in the spare accumulator columns (free); the level-0 concat buffer -- conv0's output (skip0) and
  // convtr7p2s2's output -- is stored as fp16 hi|lo pairs and read back as doubled channels by conv1p1s2, block8.conv1
  // and block8's downsample term.  (Also splitting block8.conv1's output would take the score error from 4e-4 to
  // 2.7e-4 at 35 us per step: not needed for the 2e-3 bar.)
  auto plan = [](ConvW& cw, int cout, bool in_split, bool in2_split, bool out_split) {
    cw.pack_flags = (cout == 8 ? SPS_PACK_FOLD_LO : 0) | (in_split ? SPS_PACK_IN_SPLIT : 0) | (in2_split ? SPS_PACK_IN2_SPLIT : 0);
    cw.conv_flags = (cout == 8 ? SPS_CONV_FOLD_LO : 0) | (out_split ? SPS_CONV_OUT_SPLIT : 0);
  };
  auto add_conv = [&](ConvW& cw, const std::string& kname, const std::string& bn, int K, int cin, int cout,
                      bool in_split = false, bool out_split = false, int cin_split = 0) {
    std::vector<float> w; std::vector<double> sh;
    if (!fold_conv(net, kname, bn, K, cin, cout, w, sh)) return false;
    std::vector<float> shf(sh.begin(), sh.end());
    cw.K = K; cw.cin = cin; cw.cout = cout; cw.cin2 = 0; cw.cin_split = cin_split;
    plan(cw, cout, in_split, false, out_split);
    Pending p{&cw, pk.add(w), pk.add(shf), 0, false};
    if (K == 81 || (K == 8 && cin >= 16 && cin % 4 == 0)) add_kmajor(p, w, K, cin, cout, nullptr, 0);  // 8-channel 2x2x2 layers stay on the CUDA-core kernel (measured faster)
    if (K == 81 || K == 8) add_kmajor_h(p, w, K, cin, cout, nullptr, 0);
    pend.push_back(p);
    return true;
  };
  auto add_block = [&](int b, const std::string& name, int cin, int cout, bool tail = false) {
    // tail = block8: its input (the level-0 concat buffer) holds hi|lo rows.  block5 reads a concat buffer of 64 + 32
    // channels: two K segments (1.5 stages per offset instead of 2; measured 135 -> 121 us).  The 32 + 16 and 16 + 8
    // buffers of block6 / block7 stay one padded segment: splitting them fetches every row twice and the gather is bound
    // by rows, not bytes (block7.conv1 119 -> 132 us with the split).
    const int seg = (!tail && cin > cout && cout == 64) ? cout : 0;
    if (!add_conv(net->blk1[b], name + ".0.conv1.kernel", name + ".0.norm1", 81, cin, cout, tail, false, seg)) return false;
    std::vector<float> w; std::vector<double> sh;
    if (!fold_conv(net, name + ".0.conv2.kernel", name + ".0.norm2", 81, cout, cout, w, sh)) return false;
    ConvW& cw = net->blk2[b];
    cw.K = 81; cw.cin = cout; cw.cout = cout; cw.cin2 = 0;
    plan(cw, cout, false, tail && cin != cout, false);
    Pending p{&cw, pk.add(w), 0, 0, false};
    if (cin != cout) {
      std::vector<float> w2; std::vector<double> sh2;
      if (!fold_conv(net, name + ".0.downsample.0.kernel", name + ".0.downsample.1", 1, cin, cout, w2, sh2))
        return false;
      for (int c = 0; c < cout; ++c) sh[c] += sh2[c];
      cw.cin2 = cin;
      p.w2 = pk.add(w2);
      p.has_w2 = true;
      add_kmajor(p, w, 81, cout, cout, &w2, cin);
      add_kmajor_h(p, w, 81, cout, cout, &w2, cin);
    } else {
      add_kmajor(p, w, 81, cout, cout, nullptr, 0);
      add_kmajor_h(p, w, 81, cout, cout, nullptr, 0);
    }
    std::vector<float> shf(sh.begin(), sh.end());
    p.shift = pk.add(shf);
    pend.push_back(p);
    return true;
  };
  const int I = kInitDim;
  const int* P = kPlanes;
  bool ok = add_conv(net->conv0, "conv0p1s1.kernel", "bn0", 125, 1, I);
  const char* enc_c[4] = {"conv1p1s2", "conv2p2s2", "conv3p4s2", "conv4p8s2"};
  const char* enc_b[4] = {"bn1", "bn2", "bn3", "bn4"};
  const char* dec_c[4] = {"convtr4p16s2", "convtr5p8s2", "convtr6p4s2", "convtr7p2s2"};
  const char* dec_b[4] = {"bntr4", "bntr5", "bntr6", "bntr7"};
  int inpl = I;
  for (int i = 0; i < 4 && ok; ++i) {
    ok = ok && add_conv(net->down[i], std::string(enc_c[i]) + ".kernel", enc_b[i], 8, inpl, inpl, /*in_split=*/i == 0);   // conv1p1s2 reads skip0
    ok = ok && add_block(i, "block" + std::to_string(i + 1), inpl, P[i]);
    inpl = P[i];
  }
  const int skip[4] = {P[2], P[1], P[0], I};
  for (int i = 0; i < 4 && ok; ++i) {
    ok = ok && add_conv(net->up[i], std::string(dec_c[i]) + ".kernel", dec_b[i], 8, inpl, P[4 + i], false, /*out_split=*/i == 3);
    ok = ok && add_block(4 + i, "block" + std::to_string(5 + i), P[4 + i] + skip[i], P[4 + i], /*tail=*/i == 3);
    inpl = P[4 + i];
  }
  const std::vector<float>*fw, *fb;
  // final: [8, Cout] kernel + [1, Cout] bias (minkunet.py:152-158); the forward returns ONE column of it
  // (SPSModel: Cout = 1; MOS4DNet, c_ws/src/mos4d/scripts/mos4d.py:15,32: Cout = 3, `out.features[:, 2]`)
  auto itb = net->host.find("final.bias");
  const int cout_final = itb == net->host.end() ? 0 : (int)itb->second.size();
  ok = ok && cout_final >= 1 && net->head_channel < cout_final &&
       get(net, "final.kernel", (size_t)P[7] * cout_final, &fw) && get(net, "final.bias", cout_final, &fb);
  if (!ok) return SPS_ERR_BAD_ARG;
  std::vector<float> head(P[7]);
  for (int c = 0; c < P[7]; ++c) head[c] = (*fw)[(size_t)c * cout_final + net->head_channel];
  const size_t head_off = pk.add(head);
  net->head_b = (*fb)[net->head_channel];
  if (pk.image.size() * sizeof(float) > bytes) return SPS_ERR_CAPACITY;
  float* base = (float*)d_weights;
  cudaStream_t st = (cudaStream_t)stream;
  SPS_CUDA_CHECK(cudaMemcpyAsync(base, pk.image.data(), pk.image.size() * sizeof(float), cudaMemcpyHostToDevice, st));
  SPS_CUDA_CHECK(cudaStreamSynchronize(st));  // pk.image dies with this frame
  for (auto& p : pend) {
    p.cw->w = base + p.w;
    p.cw->shift = base + p.shift;
    p.cw->w2 = p.has_w2 ? base + p.w2 : nullptr;
    p.cw->wt = p.has_wt ? base + p.wt : nullptr;
    p.cw->wth = p.has_wth ? base + p.wth : nullptr;
  }
  net->head_w = base + head_off;
  net->finalized = true;
  return SPS_OK;
}

namespace sps {

// SparseTensor.slice(tensor_field) + sigmoid (src/sps/models/models.py:28-29); n_ptr (optional): the device row count,
// rows at or past it are left untouched
__global__ void k_devox_sigmoid(const float* __restrict__ logits, const int32_t* __restrict__ inv, int64_t n,
                                float* __restrict__ scores, int apply_sigmoid, const int32_t* __restrict__ n_ptr) {
  if (n_ptr && *n_ptr < n) n = *n_ptr;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int v = __ldg(inv + i);
    float s = nanf("");
    if (v >= 0) {
      s = __ldg(logits + v);
      if (apply_sigmoid) s = 1.0f / (1.0f + expf(-s));
    }
    scores[i] = s;
  }
}

// A feature matrix (or a channel slice of one): pointer, leading dimension in elements of ITS dtype, dtype.
struct Act {
  float* p = nullptr;
  int64_t ld = 0;
  bool f16 = false;
  Act() {}
  Act(float* p_, int64_t ld_, bool f16_) : p(p_), ld(ld_), f16(f16_) {}
  Act at(int ch) const { return Act(f16 ? reinterpret_cast<float*>(reinterpret_cast<__half*>(p) + ch) : p + ch, ld, f16); }
};

struct ConvIo {
  const uint32_t* tmask; const int32_t* perm; const int32_t* slices;   // processing order (see sps_conv_args)
  int mode; const int32_t* map;
  int flags = 0;                                                        // SPS_CONV_MAP_PARENT
};

// One layer of the fused forward.  FP32 mode: generic fp32 CUDA-core kernels; TF32 mode: fp32 rows, the tcgen05 kernel
// with TF32 operands where the layer fits it; AUTO / F16: fp16 rows through the tcgen05 kernel, with the layer's
// precision plan (folded low weight parts, hi|lo rows: sps_net_finalize).
static int run_conv(sps_ctx* c, const ConvIo& io, const char* name, const ConvW& w, const int32_t* n_out, int64_t n_out_max,
                    Act in, Act in2, Act res, Act out, cudaStream_t st, const float* head_w = nullptr,
                    float head_b = 0.f, float* head_out = nullptr) {
  sps_conv_args a;
  memset(&a, 0, sizeof(a));
  const bool half = c->run_half;
  a.mode = io.mode; a.K = w.K; a.cin = w.cin; a.cout = w.cout;
  a.map = io.map; a.map_ld = c->ld; a.n_out = n_out; a.n_out_max = n_out_max;
  a.in = in.p; a.in_ld = in.ld; a.weight = w.w; a.shift = w.shift;
  if (in2.p) { a.in2 = in2.p; a.in2_ld = in2.ld; a.cin2 = w.cin2; a.weight2 = w.w2; }
  a.res = res.p; a.res_ld = res.ld; a.relu = 1; a.out = out.p; a.out_ld = out.ld;
  a.head_w = head_w; a.head_b = head_b; a.head_out = head_out;
  if (half) {
    if ((w.pack_flags & SPS_PACK_IN_SPLIT)) a.cin = 2 * w.cin;        // hi|lo rows read as doubled channels
    if (in2.p && (w.pack_flags & SPS_PACK_IN2_SPLIT)) a.cin2 = 2 * w.cin2;
    a.flags = w.conv_flags;
    a.cin_split = w.cin_split;
    a.io_dtype = SPS_IO_F16;
    a.weight_kmajor = w.wth; a.kmajor_ld = w.ldkh;
  } else {
    a.io_dtype = SPS_IO_F32;
    a.weight_kmajor = w.wt; a.kmajor_ld = w.ldk;
  }
  a.tile_mask = io.tmask; a.perm = io.perm; a.tile_slices = io.perm ? io.slices : nullptr;
  a.flags |= io.flags;
  a.round_out = c->backend != SPS_BACKEND_FP32;   // pure fp32 mode keeps full-precision activations
  a.backend = c->backend;
  ++c->forward_launches;
  const int rc = conv_dispatch(a, st);
  prof_mark(c, name, st);
  return rc;
}

// processing order of the 3x3x3x3 convs at level L: rows in neighbourhood-shape order when the maps were sorted,
// otherwise physical order; both kinds of tile masks exist.
static ConvIo io3(const sps_ctx* c, int L) {
  const bool pm = c->have_perm;
  return ConvIo{pm ? c->ptmask[L] : c->tmask3[L], pm ? c->perm[L] : nullptr, pm ? c->tslice[L] : nullptr, SPS_CONV_NBR, c->nbr3[L]};
}

int unet_forward(sps_ctx* c, const sps_net* net, const float* feat0, float* logits, cudaStream_t st,
                 bool conv0_done = false) {
  const int64_t nmax = c->n > 0 ? c->n : 1;
  float** B = c->buf;
  using C = sps_ctx;
  const bool exact = c->backend == SPS_BACKEND_FP32;
  // fp16 rows need conv0's output in the hi|lo format, which only the fused forward's conv0 kernels write
  const bool hm = ctx_half_storage(c) && conv0_done;
  c->run_half = hm;
  // Storage plan.  fp16 forward: plain fp16 rows, except the level-0 concat buffer [convtr7p2s2 out | skip0], whose rows
  // are fp16 hi|lo pairs (16 halves per 8 channels): their rounding dominated the score error of plain fp16 storage
  // (tools/precision_study.py).  Other modes: fp32 rows.
  const int x2 = hm ? 2 : 1;
  const Act cat8(B[C::CAT8], kCatLd[0] * x2, hm), h8(B[C::H8], 8, hm);
  const Act cat[4] = {cat8, Act(B[C::CAT7], kCatLd[1], hm), Act(B[C::CAT6], kCatLd[2], hm), Act(B[C::CAT5], kCatLd[3], hm)};
  // skip tensors live in the tail channel slice of the concat buffers (ME.cat(out, skip), minkunet.py:192)
  const Act skip[4] = {cat[0].at(8 * x2), cat[1].at(16), cat[2].at(32), cat[3].at(64)};
  const Act E[4] = {Act(B[C::E1], 8, hm), Act(B[C::E2], 8, hm), Act(B[C::E3], 16, hm), Act(B[C::E4], 32, hm)};
  const Act H[4] = {Act(B[C::H1], 8, hm), Act(B[C::H2], 16, hm), Act(B[C::H3], 32, hm), Act(B[C::H4], 64, hm)};
  const Act b4(B[C::B4], 64, hm);
  const Act Hd[4] = {Act(B[C::H5], 64, hm), Act(B[C::H6], 32, hm), Act(B[C::H7], 16, hm), h8};
  const Act Bd[3] = {Act(B[C::B5], 64, hm), Act(B[C::B6], 32, hm), Act(B[C::B7], 16, hm)};
  const Act none;
  static const char* nm_down[4] = {"conv1p1s2", "conv2p2s2", "conv3p4s2", "conv4p8s2"};
  static const char* nm_up[4] = {"convtr4p16s2", "convtr5p8s2", "convtr6p4s2", "convtr7p2s2"};
  static const char* nm_c1[8] = {"block1.conv1", "block2.conv1", "block3.conv1", "block4.conv1",
                                 "block5.conv1", "block6.conv1", "block7.conv1", "block8.conv1"};
  static const char* nm_c2[8] = {"block1.conv2", "block2.conv2", "block3.conv2", "block4.conv2",
                                 "block5.conv2", "block6.conv2", "block7.conv2", "block8.conv2+final"};
  int rc;
#define RUN(...) do { rc = run_conv(c, __VA_ARGS__); if (rc != SPS_OK) return rc; } while (0)
  // conv0p1s1 + bn0 + relu  (minkunet.py:162-164); the fused forward computed it while the level-0 block table was alive
  if (!conv0_done) {
    if (!c->have_nbr5) return SPS_ERR_STATE;
    const Act f0(const_cast<float*>(feat0), 1, false);
    RUN(ConvIo{nullptr, nullptr, nullptr, SPS_CONV_NBR, c->nbr5}, "conv0", net->conv0, c->counts + 0, nmax, f0, none, none, skip[0], st);
  }
  // encoder (minkunet.py:166-185)
  for (int i = 0; i < 4; ++i) {
    const int L = i + 1;
    RUN(ConvIo{c->tmask8, nullptr, nullptr, SPS_CONV_NBR, c->child[L]}, nm_down[i], net->down[i], c->counts + L, nmax, skip[i], none,
        none, E[i], st);
    const ConvW& c1 = net->blk1[i];
    const ConvW& c2 = net->blk2[i];
    RUN(io3(c, L), nm_c1[i], c1, c->counts + L, nmax, E[i], none, none, H[i], st);
    const Act out = (L < 4) ? skip[L] : b4;
    if (c2.cin2) RUN(io3(c, L), nm_c2[i], c2, c->counts + L, nmax, H[i], E[i], none, out, st);
    else RUN(io3(c, L), nm_c2[i], c2, c->counts + L, nmax, H[i], none, E[i], out, st);
  }
  // decoder (minkunet.py:188-217)
  Act dec_in = b4;
  for (int i = 0; i < 4; ++i) {
    const int L = 3 - i;  // output level
    if (exact) {   // exact-fp32 mode: scatter over the child table (no atomics, each row once)
      RUN(ConvIo{nullptr, nullptr, nullptr, SPS_CONV_UP, c->child[L + 1]}, nm_up[i], net->up[i], c->counts + L + 1, nmax, dec_in, none,
          none, cat[L], st);
    } else {       // the same transposed conv as an 8-offset gather map of the fine rows
      // rows visited by child class (perm_up): a tile walks one of the eight offsets instead of all of them
      RUN(ConvIo{c->tmask_up[L], c->perm_up[L], nullptr, SPS_CONV_NBR, c->parent[L], SPS_CONV_MAP_PARENT}, nm_up[i], net->up[i], c->counts + L, nmax, dec_in, none, none,
          cat[L], st);
    }
    const ConvW& c1 = net->blk1[4 + i];
    const ConvW& c2 = net->blk2[4 + i];
    RUN(io3(c, L), nm_c1[4 + i], c1, c->counts + L, nmax, cat[L], none, none, Hd[i], st);
    if (i < 3) {
      RUN(io3(c, L), nm_c2[4 + i], c2, c->counts + L, nmax, Hd[i], cat[L], none, Bd[i], st);
      dec_in = Bd[i];
    } else {
      // block8.conv2 + norm2 + downsample + relu, with `final` (8->1, bias; minkunet.py:219) fused
      RUN(io3(c, L), nm_c2[4 + i], c2, c->counts + L, nmax, Hd[i], cat[L], none, none, st, net->head_w, net->head_b, logits);
    }
  }
#undef RUN
  return SPS_OK;
}

}  // namespace sps

extern "C" int sps_unet_forward(sps_ctx* ctx, const sps_net* net, const float* d_feat0, float* d_logits,
                                void* stream) {
  if (!ctx || !net || !d_feat0 || !d_logits) return SPS_ERR_BAD_ARG;
  if (!net->finalized || !ctx->have_maps) return SPS_ERR_STATE;
  return unet_forward(ctx, net, d_feat0, d_logits, (cudaStream_t)stream);
}

static int devox(const float* d_logits, const int32_t* d_inv, int64_t n, float* d_scores, int apply_sigmoid, void* stream,
                 const int32_t* d_n = nullptr) {
  if (!d_logits || !d_inv || !d_scores || n < 0) return SPS_ERR_BAD_ARG;
  if (n == 0) return SPS_OK;
  int64_t g = (n + 255) / 256;
  if (g > 148 * 16) g = 148 * 16;
  k_devox_sigmoid<<<(int)g, 256, 0, (cudaStream_t)stream>>>(d_logits, d_inv, n, d_scores, apply_sigmoid, d_n);
  SPS_CUDA_CHECK(cudaGetLastError());
  return SPS_OK;
}
extern "C" int sps_devox_sigmoid(const float* d_logits, const int32_t* d_inv, int64_t n, float* d_scores,
                                 void* stream) {
  return devox(d_logits, d_inv, n, d_scores, 1, stream);
}

namespace sps {
int voxelize_impl(sps_ctx* ctx, const float* d_points, int64_t n, const int32_t* d_n, int64_t ld_points,
                  float voxel_size, cudaStream_t st);
int build_maps_impl(sps_ctx* ctx, const Conv0Fused* c0, cudaStream_t st);

static int forward_feat_impl(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n, const int32_t* d_n,
                             int64_t ld_points, const float* d_feat, float voxel_size, float* d_scores, int64_t n_scores,
                             cudaStream_t st);
int forward_impl(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n, const int32_t* d_n,
                 int64_t ld_points, float voxel_size, float* d_scores, int64_t n_scores, cudaStream_t st) {
  return forward_feat_impl(ctx, net, d_points, n, d_n, ld_points, nullptr, voxel_size, d_scores, n_scores, st);
}
// d_feat == nullptr: SPSModel.forward (every point carries 0.5); else one input feature per point, averaged per voxel
// (ME.TensorField(...).sparse(), UNWEIGHTED_AVERAGE): MapMOSNet.forward, c_ws/src/mapmos/scripts/mapmos.py:59-83
static int forward_feat_impl(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n, const int32_t* d_n,
                             int64_t ld_points, const float* d_feat, float voxel_size, float* d_scores, int64_t n_scores,
                             cudaStream_t st) {
  if (!ctx || !net || n < 0) return SPS_ERR_BAD_ARG;
  if (!net->finalized) return SPS_ERR_STATE;
  ctx->forward_launches = 0;
  if (n == 0) {  // empty input: nothing to score (an empty TensorField in the reference)
    ctx->n = 0;
    ctx->have_l0 = ctx->have_maps = false;
    return SPS_OK;
  }
  if (!d_scores || !d_points) return SPS_ERR_BAD_ARG;
  prof_begin(ctx, st);
  int rc = voxelize_impl(ctx, d_points, n, d_n, ld_points, voxel_size, st);
  if (rc != SPS_OK) return rc;
  // TensorField.sparse(): voxel feature = mean of the constant 0.5 point features = 0.5
  // (src/sps/models/models.py:22-25)
  // conv0's output = skip0, channels 8..15 of the level-0 concat buffer: fp16 hi|lo pairs in the fp16 forward (halves
  // 16..31 of 32-half rows), fp32 otherwise (TF32-rounded when a TF32 tensor-core layer reads it)
  const bool hm = ctx_half_storage(ctx);
  float* c0_out = ctx->buf[sps_ctx::CAT8] + 8;      // 8 floats = 16 halves into the row, either way
  const float* vfeat = nullptr;
  if (d_feat) {   // voxel feature = mean of its points' features; the logits buffer is free until the last layer
    rc = sps_voxel_mean(ctx, d_feat, 1, 1, ctx->buf[sps_ctx::FEAT0], ctx->buf[sps_ctx::LOGITS], st);
    if (rc != SPS_OK) return rc;
    vfeat = ctx->buf[sps_ctx::FEAT0];
  }
  Conv0Fused c0{vfeat, 0.5f, net->conv0.w, net->conv0.shift, hm ? kStoreF16x2 : (ctx->backend != SPS_BACKEND_FP32 ? kStoreTF32 : kStoreF32),
                c0_out, hm ? 2 * kCatLd[0] : kCatLd[0]};
  rc = build_maps_impl(ctx, &c0, st);
  if (rc != SPS_OK) return rc;
  rc = unet_forward(ctx, net, ctx->buf[sps_ctx::FEAT0], ctx->buf[sps_ctx::LOGITS], st, /*conv0_done=*/true);
  if (rc != SPS_OK) return rc;
  rc = devox(ctx->buf[sps_ctx::LOGITS], ctx->inv, n_scores, d_scores, net->apply_sigmoid, st, d_n);
  if (rc != SPS_OK) return rc;
  prof_mark(ctx, "devox_sigmoid", st);
  ctx->forward_launches += 4 + 1;   // voxelise (4) and the devoxelisation; build_maps_impl / run_conv count their own
  return SPS_OK;
}
}  // namespace sps

extern "C" int sps_forward(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n, int64_t ld_points,
                           float voxel_size, float* d_scores, void* stream) {
  return forward_impl(ctx, net, d_points, n, nullptr, ld_points, voxel_size, d_scores, n, (cudaStream_t)stream);
}

extern "C" int sps_forward_features(sps_ctx* ctx, const sps_net* net, const float* d_points, int64_t n, int64_t ld_points,
                                    const float* d_feat, float voxel_size, float* d_scores, void* stream) {
  if (!d_feat && n > 0) return SPS_ERR_BAD_ARG;
  return forward_feat_impl(ctx, net, d_points, n, nullptr, ld_points, d_feat, voxel_size, d_scores, n, (cudaStream_t)stream);
}

extern "C" int sps_forward_host(sps_ctx* ctx, const sps_net* net, const float* h_points, int64_t n,
                                int64_t ld_points, float voxel_size, float* h_scores, void* stream) {
  if (!ctx || !net || n < 0 || (n > 0 && (!h_points || !h_scores)) || ld_points < 5 || ld_points > 8)
    return SPS_ERR_BAD_ARG;
  if (n > ctx->max_points) return SPS_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream;
  if (n > 0)
    SPS_CUDA_CHECK(cudaMemcpyAsync(ctx->staging, h_points, (size_t)n * ld_points * sizeof(float),
                                   cudaMemcpyHostToDevice, st));
  int rc = sps_forward(ctx, net, ctx->staging, n, ld_points, voxel_size, ctx->scores, stream);
  if (rc != SPS_OK) return rc;
  if (n > 0)
    SPS_CUDA_CHECK(cudaMemcpyAsync(h_scores, ctx->scores, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
  return sps_ctx_status(ctx, stream);
}
