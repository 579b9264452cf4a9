// ResNet-50/101 + GeM + FC + L2 descriptor network on one GPU: weight packing and the launch schedule.
//
// Reference: dirtorch/nets/backbones/resnet.py:46-87 (Bottleneck), :102-168 (ResNet.__init__/forward),
//            dirtorch/nets/rmac_resnet.py:12-69 (head), dirtorch/nets/layers/pooling.py:38-54 (GeM).
// Data layout in HBM: activations NHWC fp16; conv weights [Cout][KH][KW][Cin] fp16 (K-major rows, the B operand
// of the implicit GEMM); BatchNorm folded to per-channel fp32 (scale, shift) applied in the conv epilogue together
// with the residual add and ReLU; head weights fp32.  A batch is processed in chunks of `chunk` images so that
// the activations of consecutive layers stay L2-resident.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "conv.h"

using namespace dirb;

namespace {

struct HostTensor {
  std::vector<float> data;
  std::vector<int64_t> shape;
};

struct ConvLayer {
  std::string conv, bn;          // state-dict prefixes
  int Cin, Cout, K, stride, pad;
  int CinPad, Kpad;              // packed layout
  __half* w = nullptr;
  float* scale = nullptr;
  float* shift = nullptr;
};

struct Block {
  ConvLayer c1, c2, c3, down;
  bool has_down = false;
  // block 0 of a layer: conv3 + projection shortcut as ONE GEMM over K = [conv2 output | block input]:
  // wcat[o] = [scale3[o] * W3[o][:], scale_d[o] * Wd[o][:]] (fp16), shift = shift3 + shift_d, scale = 1.
  __half* wcat = nullptr;
  float* cat_shift = nullptr;
  float* ones = nullptr;
};

}  // namespace

// Per-launch CUDA-event timing of one forward (option "profile"): class 0 = tcgen05 conv, 1 = stem conv (mma.sync),
// 2 = layout/maxpool, 3 = head.  Events sit on the launch stream, so they time exactly the kernels between them.
struct Profiler {
  struct Rec { cudaEvent_t a, b; int cls; double flops, bytes; std::string tag; };
  std::vector<Rec> recs;
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  cudaEvent_t get() {
    if (used == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[used++];
  }
  void reset() { recs.clear(); used = 0; }
  ~Profiler() { for (auto e : pool) cudaEventDestroy(e); }
};

struct dirb200_net {
  int device = 0;
  std::string arch;
  std::vector<int> nblocks;
  // options
  int pooling = 0, norm_features = 0, without_fc = 0, out_dim = 2048, chunk = 0, conv_impl = 0;
  float gem_p = 3.0f, gem_eps = 1e-6f;
  float center_bias = 0.0f;       // rmac_resnet.py:52-56
  // host state dict
  std::map<std::string, HostTensor> sd;
  bool finalized = false;
  // device weights
  ConvLayer stem;
  __half* stem_w2 = nullptr;      // [64][256] space-to-depth tap layout for the tcgen05 stem
  std::vector<Block> blocks;      // flattened over layer1..4
  std::vector<int> layer_end;     // index (exclusive) of the last block of each layer
  float* fc_w = nullptr;
  float* fc_b = nullptr;
  unsigned int* head_bar = nullptr;   // grid-barrier words of the fused head kernel (zero once, self-resetting)
  std::vector<void*> owned;
  // workspace
  void* ws = nullptr;
  size_t ws_bytes = 0;
  // staging for forward_host
  float* h2d = nullptr;
  size_t h2d_bytes = 0;
  float* d_desc = nullptr;
  size_t d_desc_bytes = 0;
  cudaStream_t own_stream = nullptr;
  // debug taps of the last chunk (copies, only when the "debug_taps" option is set)
  struct Tap { __half* ptr; size_t cap; int n, h, w, c; };
  std::map<std::string, Tap> taps;
  int debug_taps = 0;
  int64_t last_launches = 0;
  double last_flops = 0;
  int profile = 0;
  Profiler prof;
  float mean_std[6] = {0.485f, 0.456f, 0.406f, 0.229f, 0.224f, 0.225f};   // preprocess of resnet.py:110-111
  int fuse_ds = 1;                // fuse the projection shortcut into conv3 of block 0 (tcgen05 path only)
  int c23_variant = 1;            // 1 = CTA pairs (cta_group::2), 0 = one CTA per tile
  int fuse_c23 = 0;               // conv2 + conv3 (+ residual) of the identity blocks as one kernel (conv_c23.cuh):
                                  // 0 off, 1 where every SM gets several tiles, 2 wherever the kernel supports the shape
  // trunk / head variants (rmac_resnet.py:74-88, rmac_resnet_fpn.py:92-110)
  bool basic = false;             // BasicBlock trunk (resnet18): two 3x3 convolutions per block, expansion 1
  int expansion = 4;
  int stage_ch[5] = {64, 256, 512, 1024, 2048};   // channels of the output of stage 0..4
  int fpn = 0;                    // FPN head: GeM of layer3 (after the lateral merge in mode 1) and of layer4, concatenated
  int fpn_mode = 1;               // rmac_resnet_fpn.py:27-30,55-62: 1 = lateral 1x1 + upsample-add + 3x3 smoothing, 0 = none
  float gem_p4 = 3.0f;            // adpoolc4.p (layer3 map); gem_p holds adpoolx5.p (layer4 map) for FPN heads
  ConvLayer fpn_lat, fpn_smooth;  // conv1x5 (1x1, C4 -> C3), conv3c4 (3x3, C3 -> C3): no BN, ReLU after each
  int feat_in() const { return fpn ? stage_ch[3] + stage_ch[4] : stage_ch[4]; }     // fc.in_features
  int desc_dim() const { return without_fc ? feat_in() : out_dim; }
  int sub[5] = {0, 0, 0, 0, 0};   // images per sub-chunk of stage 0..4 (0 = auto)
  int stage_sched = 0;            // 0 = every stage over the whole chunk (fastest measured), 1 = per-stage sub-chunks
  // pipelined host entry point
  cudaStream_t copy_stream = nullptr;
  std::vector<cudaEvent_t> pipe_events;
  int host_chunk = 16;
};

struct ProfScope {
  dirb200_net* n; cudaStream_t st; bool on;
  ProfScope(dirb200_net* n_, cudaStream_t st_, int cls, double flops, double bytes, const std::string& tag = std::string())
      : n(n_), st(st_), on(n_->profile != 0) {
    if (on) {
      Profiler::Rec r{n->prof.get(), n->prof.get(), cls, flops, bytes, tag};
      cudaEventRecord(r.a, st);
      n->prof.recs.push_back(r);
    }
  }
  ~ProfScope() { if (on) cudaEventRecord(n->prof.recs.back().b, st); }
};

static int dev_alloc(dirb200_net* n, void** p, size_t bytes) {
  DIRB_CUDA(cudaMalloc(p, bytes));
  n->owned.push_back(*p);
  return 0;
}

// keep a copy of an intermediate activation (the rotating buffers are overwritten by later layers)
static int record_tap(dirb200_net* n, const std::string& name, const __half* src, int nb, int h, int w, int c,
                      cudaStream_t stream) {
  if (!n->debug_taps) return 0;
  const size_t bytes = static_cast<size_t>(nb) * h * w * c * 2;
  auto& t = n->taps[name];
  if (t.cap < bytes) {
    if (t.ptr) DIRB_CUDA(cudaFree(t.ptr));
    t.ptr = nullptr;
    DIRB_CUDA(cudaMalloc(reinterpret_cast<void**>(&t.ptr), bytes));
    t.cap = bytes;
  }
  t.n = nb; t.h = h; t.w = w; t.c = c;
  DIRB_CUDA(cudaMemcpyAsync(t.ptr, src, bytes, cudaMemcpyDeviceToDevice, stream));
  return 0;
}

static int get_tensor(dirb200_net* n, const std::string& name, const HostTensor** out, size_t expect) {
  auto it = n->sd.find(name);
  DIRB_REQUIRE(it != n->sd.end(), DIRB200_EKEY, "missing state-dict tensor '%s'", name.c_str());
  DIRB_REQUIRE(it->second.data.size() == expect, DIRB200_EINVAL, "tensor '%s' has %zu elements, expected %zu",
               name.c_str(), it->second.data.size(), expect);
  *out = &it->second;
  return 0;
}

// OIHW fp32 -> [Cout][KH][KW][CinPad] fp16 rows padded to Kpad; BN -> (scale, shift).
static int pack_conv(dirb200_net* n, ConvLayer& L) {
  const HostTensor *w, *g, *b, *m, *v;
  const size_t kk = static_cast<size_t>(L.K) * L.K;
  DIRB_TRY(get_tensor(n, L.conv + ".weight", &w, static_cast<size_t>(L.Cout) * L.Cin * kk));
  DIRB_TRY(get_tensor(n, L.bn + ".weight", &g, L.Cout));
  DIRB_TRY(get_tensor(n, L.bn + ".bias", &b, L.Cout));
  DIRB_TRY(get_tensor(n, L.bn + ".running_mean", &m, L.Cout));
  DIRB_TRY(get_tensor(n, L.bn + ".running_var", &v, L.Cout));
  L.CinPad = (L.Cin % 8 == 0) ? L.Cin : ((L.Cin + 7) / 8 * 8);
  const int Ktot = L.K * L.K * L.CinPad;
  L.Kpad = (Ktot + 31) / 32 * 32;
  std::vector<__half> hw(static_cast<size_t>(L.Cout) * L.Kpad, __float2half(0.f));
  for (int o = 0; o < L.Cout; ++o)
    for (int c = 0; c < L.Cin; ++c)
      for (int kh = 0; kh < L.K; ++kh)
        for (int kw = 0; kw < L.K; ++kw)
          hw[static_cast<size_t>(o) * L.Kpad + (static_cast<size_t>(kh) * L.K + kw) * L.CinPad + c] =
              __float2half_rn(w->data[((static_cast<size_t>(o) * L.Cin + c) * L.K + kh) * L.K + kw]);
  std::vector<float> sc(L.Cout), sh(L.Cout);
  for (int o = 0; o < L.Cout; ++o) {
    // BatchNorm2d eval: y = (x - mean) / sqrt(var + 1e-5) * gamma + beta   (eps: torch default, resnet.py:57)
    const float s = g->data[o] / sqrtf(v->data[o] + 1e-5f);
    sc[o] = s;
    sh[o] = b->data[o] - m->data[o] * s;
  }
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&L.w), hw.size() * sizeof(__half)));
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&L.scale), L.Cout * sizeof(float)));
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&L.shift), L.Cout * sizeof(float)));
  DIRB_CUDA(cudaMemcpy(L.w, hw.data(), hw.size() * sizeof(__half), cudaMemcpyHostToDevice));
  DIRB_CUDA(cudaMemcpy(L.scale, sc.data(), L.Cout * sizeof(float), cudaMemcpyHostToDevice));
  DIRB_CUDA(cudaMemcpy(L.shift, sh.data(), L.Cout * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

// Convolution without BatchNorm (FPN lateral / smoothing convs): scale = 1, shift = 0.
static int pack_conv_plain(dirb200_net* n, ConvLayer& L) {
  const HostTensor* w;
  const size_t kk = static_cast<size_t>(L.K) * L.K;
  DIRB_TRY(get_tensor(n, L.conv + ".weight", &w, static_cast<size_t>(L.Cout) * L.Cin * kk));
  L.CinPad = L.Cin;
  const int Ktot = L.K * L.K * L.CinPad;
  L.Kpad = (Ktot + 31) / 32 * 32;
  std::vector<__half> hw(static_cast<size_t>(L.Cout) * L.Kpad, __float2half(0.f));
  for (int o = 0; o < L.Cout; ++o)
    for (int c = 0; c < L.Cin; ++c)
      for (int kh = 0; kh < L.K; ++kh)
        for (int kw = 0; kw < L.K; ++kw)
          hw[static_cast<size_t>(o) * L.Kpad + (static_cast<size_t>(kh) * L.K + kw) * L.CinPad + c] =
              __float2half_rn(w->data[((static_cast<size_t>(o) * L.Cin + c) * L.K + kh) * L.K + kw]);
  std::vector<float> sc(L.Cout, 1.0f), sh(L.Cout, 0.0f);
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&L.w), hw.size() * sizeof(__half)));
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&L.scale), L.Cout * sizeof(float)));
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&L.shift), L.Cout * sizeof(float)));
  DIRB_CUDA(cudaMemcpy(L.w, hw.data(), hw.size() * sizeof(__half), cudaMemcpyHostToDevice));
  DIRB_CUDA(cudaMemcpy(L.scale, sc.data(), L.Cout * sizeof(float), cudaMemcpyHostToDevice));
  DIRB_CUDA(cudaMemcpy(L.shift, sh.data(), L.Cout * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

static ConvLayer make_layer(const std::string& conv, const std::string& bn, int cin, int cout, int k, int stride,
                            int pad) {
  ConvLayer L;
  L.conv = conv; L.bn = bn; L.Cin = cin; L.Cout = cout; L.K = k; L.stride = stride; L.pad = pad;
  L.CinPad = cin; L.Kpad = 0;
  return L;
}

static int run_conv(dirb200_net* n, const ConvLayer& L, const __half* in, int B, int H, int W, const __half* res,
                    int relu, __half* out, cudaStream_t stream, int force_mma = 0) {
  ConvShape s{B, H, W, L.CinPad, L.Cout, L.K, L.K, L.stride, L.pad};
  const double flops = 2.0 * B * s.Ho() * s.Wo() * static_cast<double>(L.Cout) * L.K * L.K * L.Cin;
  // algorithmic bytes: input + output (+ residual) activations once, weights once
  const double bytes = 2.0 * (static_cast<double>(B) * H * W * L.CinPad + static_cast<double>(B) * s.Ho() * s.Wo() * L.Cout * (res ? 2 : 1) +
                              static_cast<double>(L.Cout) * L.K * L.K * L.CinPad);
  n->last_flops += flops;
  const bool mma = force_mma || n->conv_impl == 1 || L.CinPad % 64 != 0;
  std::string tag;
  if (n->profile) {
    char buf[96];
    snprintf(buf, sizeof(buf), "%dx%d%s %d->%d%s @%dx%d", L.K, L.K, L.stride == 2 ? "/s2" : "", L.Cin, L.Cout, res ? " +res" : "", s.Ho(), s.Wo());
    tag = buf;
  }
  ProfScope ps(n, stream, mma ? 1 : 0, flops, bytes, tag);
  if (mma)
    return conv_mma(s, in, L.w, L.Kpad, L.scale, L.shift, res, relu, out, stream);
  if (n->conv_impl == 2) return conv_tc_np(s, in, L.w, L.scale, L.shift, res, relu, out, stream);
  return conv_tc(s, in, L.w, L.scale, L.shift, res, relu, out, stream);
}

extern "C" {

int dirb200_net_create(const char* arch, int device, dirb200_net** out) {
  DIRB_REQUIRE(arch && out, DIRB200_EINVAL, "null argument");
  DIRB_TRY(dirb200_device_check(device));
  auto* n = new dirb200_net();
  n->device = device;
  n->arch = arch;
  // "<trunk>_rmac" (rmac_resnet.py:74-88), "<trunk>_fpn_rmac" / "resnet101_fpn0_rmac" (rmac_resnet_fpn.py:92-110)
  std::string trunk = n->arch;
  const char* suffixes[3] = {"_fpn0_rmac", "_fpn_rmac", "_rmac"};
  int which = -1;
  for (int i = 0; i < 3 && which < 0; ++i) {
    const std::string suf(suffixes[i]);
    if (trunk.size() > suf.size() && trunk.compare(trunk.size() - suf.size(), suf.size(), suf) == 0) {
      trunk = trunk.substr(0, trunk.size() - suf.size());
      which = i;
    }
  }
  n->fpn = (which == 0 || which == 1) ? 1 : 0;
  n->fpn_mode = (which == 0) ? 0 : 1;
  if (trunk == "resnet18") { n->nblocks = {2, 2, 2, 2}; n->basic = true; }        // rmac_resnet.py:76
  else if (trunk == "resnet50") n->nblocks = {3, 4, 6, 3};                         // rmac_resnet.py:80
  else if (trunk == "resnet101") n->nblocks = {3, 4, 23, 3};                       // rmac_resnet.py:84
  else if (trunk == "resnet152") n->nblocks = {3, 8, 36, 3};                       // rmac_resnet.py:88
  const bool known = which >= 0 && !n->nblocks.empty() && !(which == 0 && trunk != "resnet101");
  if (!known) {
    delete n;
    DIRB_REQUIRE(false, DIRB200_ENOTSUP,
                 "unknown model architecture '%s' (supported: resnet{18,50,101,152}_rmac, resnet{18,50,101,152}_fpn_rmac, "
                 "resnet101_fpn0_rmac)", arch);
  }
  n->expansion = n->basic ? 1 : 4;
  for (int s = 1; s < 5; ++s) n->stage_ch[s] = (64 << (s - 1)) * n->expansion;
  *out = n;
  return 0;
}

static bool is_global_option(const std::string& k) {
  return k == "halo" || k == "pdl" || k == "res_variant" || k == "head_fused" || k == "l2_prefetch" || k == "epi_mode" || k == "epi_warps";
}

int dirb200_set_global_option(const char* key, double value) {
  DIRB_REQUIRE(key, DIRB200_EINVAL, "null argument");
  const std::string k(key);
  if (k == "halo") set_conv_halo(value != 0);
  else if (k == "pdl") g_use_pdl = value != 0;
  else if (k == "res_variant") set_res_variant(static_cast<int>(value));
  else if (k == "head_fused") set_head_fused(static_cast<int>(value));
  else if (k == "l2_prefetch") set_l2_prefetch(static_cast<int>(value));
  else if (k == "epi_mode") set_epi_mode(static_cast<int>(value));
  else if (k == "epi_warps") set_epi_warps(static_cast<int>(value));
  else DIRB_REQUIRE(false, DIRB200_EKEY, "unknown global option '%s'", key);
  return 0;
}

int dirb200_get_global_option(const char* key, double* value) {
  DIRB_REQUIRE(key && value, DIRB200_EINVAL, "null argument");
  const std::string k(key);
  if (k == "halo") *value = get_conv_halo();
  else if (k == "pdl") *value = g_use_pdl;
  else if (k == "res_variant") *value = get_res_variant();
  else if (k == "head_fused") *value = get_head_fused();
  else if (k == "l2_prefetch") *value = get_l2_prefetch();
  else if (k == "epi_mode") *value = get_epi_mode();
  else if (k == "epi_warps") *value = get_epi_warps();
  else DIRB_REQUIRE(false, DIRB200_EKEY, "unknown global option '%s'", key);
  return 0;
}

int dirb200_net_set_option(dirb200_net* n, const char* key, double value) {
  DIRB_REQUIRE(n && key, DIRB200_EINVAL, "null argument");
  const std::string k(key);
  // options that decide which tensors dirb200_net_finalize reads / packs cannot change afterwards
  const bool structural = (k == "pooling" || k == "without_fc" || k == "out_dim" || k == "fpn_mode");
  DIRB_REQUIRE(!(structural && n->finalized), DIRB200_ESTATE, "option '%s' must be set before dirb200_net_finalize", key);
  if (k == "pooling") n->pooling = static_cast<int>(value);
  else if (k == "norm_features") n->norm_features = value != 0;
  else if (k == "without_fc") n->without_fc = value != 0;
  else if (k == "out_dim") n->out_dim = static_cast<int>(value);
  else if (k == "fpn_mode") {
    DIRB_REQUIRE(n->fpn && (value == 0 || value == 1), DIRB200_EINVAL, "fpn_mode is 0 or 1 and only applies to *_fpn_rmac networks");
    n->fpn_mode = static_cast<int>(value);
  }
  else if (k == "chunk") n->chunk = static_cast<int>(value);
  else if (k == "conv_impl") n->conv_impl = static_cast<int>(value);
  else if (k == "gem_eps") n->gem_eps = static_cast<float>(value);
  else if (k == "center_bias") n->center_bias = static_cast<float>(value);
  else if (k == "debug_taps") n->debug_taps = value != 0;
  else if (k == "profile") {             // 1 = time every launch of the NEXT forward; 2 = accumulate over forwards
    n->profile = static_cast<int>(value);
    n->prof.reset();
  }
  else if (k == "fuse_ds") n->fuse_ds = value != 0;
  else if (k == "fuse_c23") n->fuse_c23 = static_cast<int>(value);
  else if (k == "c23_variant") n->c23_variant = static_cast<int>(value);
  else if (is_global_option(k)) return dirb200_set_global_option(key, value);   // process-wide kernel selectors
  else if (k.size() == 5 && k.compare(0, 4, "mean") == 0 && k[4] >= '0' && k[4] <= '2') n->mean_std[k[4] - '0'] = static_cast<float>(value);
  else if (k.size() == 4 && k.compare(0, 3, "std") == 0 && k[3] >= '0' && k[3] <= '2') n->mean_std[3 + k[3] - '0'] = static_cast<float>(value);
  else if (k == "stage_sched") n->stage_sched = static_cast<int>(value);
  else if (k.size() == 4 && k.compare(0, 3, "sub") == 0 && k[3] >= '0' && k[3] <= '4') n->sub[k[3] - '0'] = static_cast<int>(value);
  else if (k == "host_chunk") n->host_chunk = std::max(1, static_cast<int>(value));
  else DIRB_REQUIRE(false, DIRB200_EKEY, "unknown net option '%s'", key);
  return 0;
}

int dirb200_net_set_tensor(dirb200_net* n, const char* name, const float* host_data, const int64_t* shape, int ndim) {
  DIRB_REQUIRE(n && name && (host_data || ndim == 0) && ndim >= 0 && ndim <= 4, DIRB200_EINVAL, "bad tensor argument");
  DIRB_REQUIRE(!n->finalized, DIRB200_ESTATE, "network already finalized");
  std::string key(name);
  if (key.rfind("module.", 0) == 0) key = key.substr(7);  // DataParallel prefix, common.py:128-133
  const char* nbt = "num_batches_tracked";
  if (key.size() >= strlen(nbt) && key.compare(key.size() - strlen(nbt), strlen(nbt), nbt) == 0) return 0;
  HostTensor t;
  size_t numel = 1;
  for (int i = 0; i < ndim; ++i) {
    t.shape.push_back(shape[i]);
    numel *= static_cast<size_t>(shape[i]);
  }
  t.data.assign(host_data, host_data + numel);
  n->sd[key] = std::move(t);
  return 0;
}

int dirb200_net_finalize(dirb200_net* n) {
  DIRB_REQUIRE(n, DIRB200_EINVAL, "null");
  DIRB_REQUIRE(!n->finalized, DIRB200_ESTATE, "network already finalized");
  DIRB_CUDA(cudaSetDevice(n->device));
  n->stem = make_layer("conv1", "bn1", 3, 64, 7, 2, 3);          // resnet.py:115-117
  DIRB_TRY(pack_conv(n, n->stem));
  {
    const HostTensor* w;
    DIRB_TRY(get_tensor(n, "conv1.weight", &w, 64 * 3 * 7 * 7));
    std::vector<__half> w2(64 * 256);
    pack_stem_w2(w->data.data(), w2.data());
    DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&n->stem_w2), w2.size() * sizeof(__half)));
    DIRB_CUDA(cudaMemcpy(n->stem_w2, w2.data(), w2.size() * sizeof(__half), cudaMemcpyHostToDevice));
  }
  int inplanes = 64;
  const int planes_per_layer[4] = {64, 128, 256, 512};           // resnet.py:120-123
  for (int li = 0; li < 4; ++li) {
    const int planes = planes_per_layer[li];
    for (int b = 0; b < n->nblocks[li]; ++b) {
      const std::string p = "layer" + std::to_string(li + 1) + "." + std::to_string(b) + ".";
      const int stride = (li > 0 && b == 0) ? 2 : 1;
      Block blk;
      const int cout = planes * n->expansion;
      if (n->basic) {                                                              // resnet.py:15-44
        blk.c1 = make_layer(p + "conv1", p + "bn1", inplanes, planes, 3, stride, 1);
        blk.c2 = make_layer(p + "conv2", p + "bn2", planes, planes, 3, 1, 1);
        blk.has_down = (b == 0) && (stride != 1 || inplanes != cout);              // resnet.py:136-141
        DIRB_TRY(pack_conv(n, blk.c1));
        DIRB_TRY(pack_conv(n, blk.c2));
        if (blk.has_down) {
          blk.down = make_layer(p + "downsample.0", p + "downsample.1", inplanes, cout, 1, stride, 0);
          DIRB_TRY(pack_conv(n, blk.down));
        }
        n->blocks.push_back(blk);
        inplanes = cout;
        continue;
      }
      blk.c1 = make_layer(p + "conv1", p + "bn1", inplanes, planes, 1, 1, 0);
      blk.c2 = make_layer(p + "conv2", p + "bn2", planes, planes, 3, stride, 1);     // stride on conv2, resnet.py:58
      blk.c3 = make_layer(p + "conv3", p + "bn3", planes, planes * 4, 1, 1, 0);
      blk.has_down = (b == 0);                                                     // resnet.py:136-141
      DIRB_TRY(pack_conv(n, blk.c1));
      DIRB_TRY(pack_conv(n, blk.c2));
      DIRB_TRY(pack_conv(n, blk.c3));
      if (blk.has_down) {
        blk.down = make_layer(p + "downsample.0", p + "downsample.1", inplanes, planes * 4, 1, stride, 0);
        DIRB_TRY(pack_conv(n, blk.down));
        // K-concatenated, BN-scaled weights for the fused conv3 + shortcut
        const HostTensor *w3, *wd;
        const int kcat = planes + inplanes;
        DIRB_TRY(get_tensor(n, p + "conv3.weight", &w3, static_cast<size_t>(cout) * planes));
        DIRB_TRY(get_tensor(n, p + "downsample.0.weight", &wd, static_cast<size_t>(cout) * inplanes));
        std::vector<float> s3(cout), sh3(cout), sd(cout), shd(cout);
        DIRB_CUDA(cudaMemcpy(s3.data(), blk.c3.scale, cout * 4, cudaMemcpyDeviceToHost));
        DIRB_CUDA(cudaMemcpy(sh3.data(), blk.c3.shift, cout * 4, cudaMemcpyDeviceToHost));
        DIRB_CUDA(cudaMemcpy(sd.data(), blk.down.scale, cout * 4, cudaMemcpyDeviceToHost));
        DIRB_CUDA(cudaMemcpy(shd.data(), blk.down.shift, cout * 4, cudaMemcpyDeviceToHost));
        std::vector<__half> wc(static_cast<size_t>(cout) * kcat);
        std::vector<float> shc(cout), one(cout, 1.0f);
        for (int o = 0; o < cout; ++o) {
          for (int c = 0; c < planes; ++c) wc[static_cast<size_t>(o) * kcat + c] = __float2half_rn(s3[o] * w3->data[static_cast<size_t>(o) * planes + c]);
          for (int c = 0; c < inplanes; ++c) wc[static_cast<size_t>(o) * kcat + planes + c] = __float2half_rn(sd[o] * wd->data[static_cast<size_t>(o) * inplanes + c]);
          shc[o] = sh3[o] + shd[o];
        }
        DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&blk.wcat), wc.size() * sizeof(__half)));
        DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&blk.cat_shift), cout * 4));
        DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&blk.ones), cout * 4));
        DIRB_CUDA(cudaMemcpy(blk.wcat, wc.data(), wc.size() * sizeof(__half), cudaMemcpyHostToDevice));
        DIRB_CUDA(cudaMemcpy(blk.cat_shift, shc.data(), cout * 4, cudaMemcpyHostToDevice));
        DIRB_CUDA(cudaMemcpy(blk.ones, one.data(), cout * 4, cudaMemcpyHostToDevice));
      }
      n->blocks.push_back(blk);
      inplanes = planes * 4;
    }
    n->layer_end.push_back(static_cast<int>(n->blocks.size()));
  }
  if (n->fpn) {
    // rmac_resnet_fpn.py:36-43: only the 'gem' branch creates the two pooling layers forward() uses
    DIRB_REQUIRE(n->pooling == 0, DIRB200_ENOTSUP, "FPN heads support pooling='gem' only (rmac_resnet_fpn.py:36-43,76-77)");
    const HostTensor *p5, *p4;
    DIRB_TRY(get_tensor(n, "adpoolx5.p", &p5, 1));
    DIRB_TRY(get_tensor(n, "adpoolc4.p", &p4, 1));
    n->gem_p = p5->data[0];
    n->gem_p4 = p4->data[0];
    DIRB_REQUIRE(n->gem_p > 0 && n->gem_p4 > 0, DIRB200_EINVAL, "GeM p must be positive");
    if (n->fpn_mode == 1) {                                                       // rmac_resnet_fpn.py:27-30
      n->fpn_lat = make_layer("conv1x5", "", n->stage_ch[4], n->stage_ch[3], 1, 1, 0);
      n->fpn_smooth = make_layer("conv3c4", "", n->stage_ch[3], n->stage_ch[3], 3, 1, 1);
      DIRB_TRY(pack_conv_plain(n, n->fpn_lat));
      DIRB_TRY(pack_conv_plain(n, n->fpn_smooth));
    }
  } else if (n->pooling == 0) {
    const HostTensor* p;
    DIRB_TRY(get_tensor(n, "adpool.p", &p, 1));                  // pooling.py:54
    n->gem_p = p->data[0];
    DIRB_REQUIRE(n->gem_p > 0, DIRB200_EINVAL, "GeM p must be positive");
  }
  if (!n->without_fc) {
    const HostTensor *w, *b;
    DIRB_TRY(get_tensor(n, "fc.weight", &w, static_cast<size_t>(n->out_dim) * n->feat_in()));   // rmac_resnet.py:34, rmac_resnet_fpn.py:46
    DIRB_TRY(get_tensor(n, "fc.bias", &b, n->out_dim));
    DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&n->fc_w), w->data.size() * 4));
    DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&n->fc_b), b->data.size() * 4));
    DIRB_CUDA(cudaMemcpy(n->fc_w, w->data.data(), w->data.size() * 4, cudaMemcpyHostToDevice));
    DIRB_CUDA(cudaMemcpy(n->fc_b, b->data.data(), b->data.size() * 4, cudaMemcpyHostToDevice));
  }
  DIRB_TRY(dev_alloc(n, reinterpret_cast<void**>(&n->head_bar), 128));
  DIRB_CUDA(cudaMemset(n->head_bar, 0, 128));
  n->sd.clear();
  n->finalized = true;
  return 0;
}

static int auto_chunk(int B, int H, int W) {
  // Large chunks keep every launch at many tiles per SM (the persistent kernels lose ~1/waves to the tail);
  // bound the activation workspace to ~24 GB of the 180 GB HBM.
  const double per_img = 2.0 * (static_cast<double>(H) * W * 8 + (H / 2.0) * (W / 2.0) * 64 + 5.0 * (H / 4.0) * (W / 4.0) * 256);
  int c = static_cast<int>(24e9 / per_img);
  if (c < 1) c = 1;
  if (c > 64) c = 64;
  if (c > B) c = B;
  return c;
}

namespace {
// Stage schedule.  The network is cut into 5 stages: 0 = stem + maxpool, 1..4 = layer1..layer4 (+ head after 4).
// A stage runs over the chunk in sub-chunks of sub[s] images: the tensors passed between the blocks of a stage are
// then small enough to stay in the 126 MB L2, while the stage outputs of the whole chunk live in HBM buffers.
struct Workspace {
  __half* stem_ws;        // s2d / nhwc8 staging of one stem sub-chunk
  __half* stem_out;       // stem conv output of one sub-chunk (before the maxpool)
  __half* stage_out[4];   // outputs of stage 0..3 for the whole chunk
  __half* scratch[4];     // rotating tensors inside a stage
  float* head_ws;
  int H1, W1;             // stem conv output size
  int h[5], w[5];         // spatial size of the output of stage 0..4
  int sub[5];
};
}  // namespace

static int setup_workspace(dirb200_net* n, int chunk, int H, int W, Workspace* w) {
  w->H1 = (H + 6 - 7) / 2 + 1; w->W1 = (W + 6 - 7) / 2 + 1;                 // stem conv
  w->h[0] = (w->H1 + 2 - 3) / 2 + 1; w->w[0] = (w->W1 + 2 - 3) / 2 + 1;     // maxpool
  w->h[1] = w->h[0]; w->w[1] = w->w[0];                                     // layer1: stride 1
  for (int s = 2; s < 5; ++s) { w->h[s] = (w->h[s - 1] + 2 - 3) / 2 + 1; w->w[s] = (w->w[s - 1] + 2 - 3) / 2 + 1; }
  // sub-chunk sizes: option "subN", else auto = enough images for ~2 tiles per SM in the stage's smallest GEMM,
  // but not more than keeps one stage tensor around 32 MB
  for (int s = 0; s < 5; ++s) {
    int v = n->sub[s];
    if (v <= 0) {
      if (n->stage_sched == 0) {
        v = chunk;                              // flat schedule: every stage over the whole chunk
      } else {
        // enough images for ~2 waves of 128-pixel tiles in the stage's narrowest GEMM
        const double px = static_cast<double>(w->h[s]) * w->w[s];
        v = std::max(1, static_cast<int>(ceil(2.0 * 148.0 * 128.0 / px)));
        if (s == 0) v = std::max(v, 2);
      }
    }
    w->sub[s] = std::max(1, std::min(v, chunk));
  }
  size_t off = 0;
  auto carve = [&](size_t bytes) { size_t o = off; off += (bytes + 1023) / 1024 * 1024; return o; };
  const size_t o_sws = carve(std::max(static_cast<size_t>(w->sub[0]) * H * W * 8 * 2, stem_workspace_bytes(w->sub[0], H, W)));
  const size_t o_stem = carve(static_cast<size_t>(w->sub[0]) * w->H1 * w->W1 * 64 * 2);
  size_t o_stage[4], o_scr[4];
  for (int s = 0; s < 4; ++s) o_stage[s] = carve(static_cast<size_t>(chunk) * w->h[s] * w->w[s] * n->stage_ch[s] * 2);
  size_t scr = 0;   // largest tensor inside any stage = the stage's sub-chunk at the stage's INPUT resolution x output channels / or input
  for (int s = 1; s < 5; ++s) {
    const size_t in_px = static_cast<size_t>(w->h[s - 1]) * w->w[s - 1];
    scr = std::max(scr, static_cast<size_t>(w->sub[s]) * in_px * (n->stage_ch[s] / 4) * 2);          // conv1 output at input resolution
    scr = std::max(scr, static_cast<size_t>(w->sub[s]) * w->h[s] * w->w[s] * n->stage_ch[s] * 2);    // block output
  }
  if (n->fpn)   // the merged / smoothed layer3 map of a stage-4 sub-chunk lives in a scratch tensor
    scr = std::max(scr, static_cast<size_t>(w->sub[4]) * w->h[3] * w->w[3] * n->stage_ch[3] * 2);
  for (int i = 0; i < 4; ++i) o_scr[i] = carve(scr);
  size_t head_floats = head_workspace_floats(w->sub[4], w->h[4] * w->w[4], n->stage_ch[4], n->out_dim);
  if (n->fpn) {
    const size_t partial = std::max(head_partial_floats(w->sub[4], w->h[3] * w->w[3], n->stage_ch[3]),
                                    head_partial_floats(w->sub[4], w->h[4] * w->w[4], n->stage_ch[4]));
    head_floats = partial + static_cast<size_t>(w->sub[4]) * (n->feat_in() + std::max(n->out_dim, n->feat_in()));
  }
  const size_t o_head = carve(head_floats * 4);
  if (off > n->ws_bytes) {
    if (n->ws) DIRB_CUDA(cudaFree(n->ws));
    n->ws = nullptr;
    DIRB_CUDA(cudaMalloc(&n->ws, off));
    n->ws_bytes = off;
  }
  uint8_t* ws = static_cast<uint8_t*>(n->ws);
  w->stem_ws = reinterpret_cast<__half*>(ws + o_sws);
  w->stem_out = reinterpret_cast<__half*>(ws + o_stem);
  for (int s = 0; s < 4; ++s) w->stage_out[s] = reinterpret_cast<__half*>(ws + o_stage[s]);
  for (int i = 0; i < 4; ++i) w->scratch[i] = reinterpret_cast<__half*>(ws + o_scr[i]);
  w->head_ws = reinterpret_cast<float*>(ws + o_head);
  return 0;
}

// One pass of the network over `cb` images (NCHW fp32 on the device) -> cb descriptors.
static int run_chunk(dirb200_net* n, const Workspace& w, const float* imgs_dev, int cb, int H, int W, float* desc_dev,
                     __half* desc16_dev, cudaStream_t stream, const uint8_t* imgs_u8 = nullptr) {
  const int D = n->desc_dim();
  // ---------------------------------------------------------------- stage 0: stem + maxpool
  for (int b0 = 0; b0 < cb; b0 += w.sub[0]) {
    const int sb = std::min(w.sub[0], cb - b0);
    const float* img = imgs_dev ? imgs_dev + static_cast<size_t>(b0) * 3 * H * W : nullptr;
    const uint8_t* img8 = imgs_u8 ? imgs_u8 + static_cast<size_t>(b0) * 3 * H * W : nullptr;
    if (n->conv_impl == 1) {
      DIRB_REQUIRE(img8 == nullptr, DIRB200_ENOTSUP, "uint8 input needs the tcgen05 stem (conv_impl 0)");
      {
        ProfScope ps(n, stream, 2, 0, static_cast<double>(sb) * H * W * (12 + 16));
        DIRB_TRY(nchw_to_nhwc8(img, sb, H, W, w.stem_ws, stream));
      }
      DIRB_TRY(run_conv(n, n->stem, w.stem_ws, sb, H, W, nullptr, 1, w.stem_out, stream, /*force_mma=*/1));
    } else {
      const double flops = 2.0 * sb * w.H1 * w.W1 * 64.0 * 147.0;
      n->last_flops += flops;
      ProfScope ps(n, stream, 1, flops, static_cast<double>(sb) * (12.0 * H * W + 2.0 * stem_workspace_bytes(1, H, W) + 128.0 * w.H1 * w.W1), "stem s2d + 7x7/s2 3->64");
      DIRB_TRY(stem_tc(img, sb, H, W, n->stem_w2, n->stem.scale, n->stem.shift, w.stem_ws, w.stem_out, stream, img8,
                       n->mean_std));
    }
    ProfScope ps(n, stream, 2, 0, 2.0 * sb * 64 * (static_cast<double>(w.H1) * w.W1 + static_cast<double>(w.h[0]) * w.w[0]), "maxpool 3x3/s2");
    DIRB_TRY(maxpool_3x3s2(w.stem_out, sb, w.H1, w.W1, 64,
                           w.stage_out[0] + static_cast<size_t>(b0) * w.h[0] * w.w[0] * 64, stream));
  }
  DIRB_TRY(record_tap(n, "stem", w.stage_out[0], cb, w.h[0], w.w[0], 64, stream));
  // ---------------------------------------------------------------- stages 1..4: layer1..layer4 (+ head)
  int first = 0;
  for (int s = 1; s < 5; ++s) {
    const int last = n->layer_end[s - 1];       // blocks [first, last)
    const int hi = w.h[s - 1], wi = w.w[s - 1], ho = w.h[s], wo = w.w[s];
    const __half* stage_in = w.stage_out[s - 1];
    for (int b0 = 0; b0 < cb; b0 += w.sub[s]) {
      const int sb = std::min(w.sub[s], cb - b0);
      const __half* x = stage_in + static_cast<size_t>(b0) * hi * wi * n->stage_ch[s - 1];
      int h = hi, wd = wi;
      for (int bi = first; bi < last; ++bi) {
        const Block& blk = n->blocks[bi];
        const int j = bi - first;
        __half* t1 = w.scratch[0];
        __half* t2 = w.scratch[1];
        __half* rs = w.scratch[2];
        __half* y = (j % 2 == 0) ? w.scratch[3] : w.scratch[2];
        if (bi == last - 1 && s < 4) y = w.stage_out[s] + static_cast<size_t>(b0) * ho * wo * n->stage_ch[s];
        if (n->basic) {
          // BasicBlock, resnet.py:27-44: 3x3(stride) + BN + ReLU -> 3x3 + BN -> + (projected) x -> ReLU
          const int st = blk.c1.stride;
          const int h2 = (h + 2 - 3) / st + 1, w2 = (wd + 2 - 3) / st + 1;
          DIRB_TRY(run_conv(n, blk.c1, x, sb, h, wd, nullptr, 1, t1, stream));
          const __half* res = x;
          if (blk.has_down) {
            DIRB_TRY(run_conv(n, blk.down, x, sb, h, wd, nullptr, 0, rs, stream));
            res = rs;
          }
          DIRB_TRY(run_conv(n, blk.c2, t1, sb, h2, w2, res, 1, y, stream));
          x = y;
          h = h2;
          wd = w2;
          continue;
        }
        const int st = blk.c2.stride;
        const int h2 = (h + 2 - 3) / st + 1, w2 = (wd + 2 - 3) / st + 1;
        DIRB_TRY(run_conv(n, blk.c1, x, sb, h, wd, nullptr, 1, t1, stream));
        if (!blk.has_down && n->fuse_c23 && n->conv_impl == 0 && st == 1 &&
            (n->fuse_c23 == 2 ? conv_c23_supported(h, wd, blk.c2.Cin) : conv_c23_profitable(sb, h, wd, blk.c2.Cin))) {
          // identity block: conv2 -> conv3 (+ x) in one kernel, the conv2 output stays in shared memory
          const int Cm = blk.c2.Cin;
          const double flops = 2.0 * sb * h * wd * (9.0 * Cm * Cm + 4.0 * Cm * Cm);
          const double bytes = 2.0 * (static_cast<double>(sb) * h * wd * (Cm + 8.0 * Cm) + 13.0 * Cm * Cm);   // t1 + residual + output, weights
          n->last_flops += flops;
          char tg[96];
          snprintf(tg, sizeof(tg), "3x3 %d->%d + 1x1 ->%d +res fused @%dx%d", Cm, Cm, 4 * Cm, h, wd);
          ProfScope ps(n, stream, 0, flops, bytes, tg);
          DIRB_TRY(conv_c23(sb, h, wd, Cm, t1, blk.c2.w, blk.c2.scale, blk.c2.shift, blk.c3.w, blk.c3.scale, blk.c3.shift, x, y,
                            stream, n->c23_variant));
          x = y;
          continue;
        }
        DIRB_TRY(run_conv(n, blk.c2, t1, sb, h, wd, nullptr, 1, t2, stream));
        const __half* res = x;
        if (blk.has_down && n->fuse_ds && n->conv_impl == 0 && blk.c3.Cout % 256 == 0) {
          const double flops = 2.0 * sb * h2 * w2 * static_cast<double>(blk.c3.Cout) * (blk.c3.Cin + blk.down.Cin);
          const double bytes = 2.0 * (static_cast<double>(sb) * h2 * w2 * (blk.c3.Cin + blk.c3.Cout) +
                                      static_cast<double>(sb) * h * wd * blk.down.Cin +
                                      static_cast<double>(blk.c3.Cout) * (blk.c3.Cin + blk.down.Cin));
          n->last_flops += flops;
          char tbuf_[96];
          snprintf(tbuf_, sizeof(tbuf_), "1x1 [%d|%d%s]->%d fused-shortcut @%dx%d", blk.c3.Cin, blk.down.Cin, st == 2 ? "/s2" : "", blk.c3.Cout, h2, w2);
          ProfScope ps(n, stream, 0, flops, bytes, tbuf_);
          DIRB_TRY(conv_fused_ds(sb, h2, w2, blk.c3.Cin, t2, h, wd, blk.down.Cin, st, x, blk.wcat, blk.c3.Cout, blk.ones,
                                 blk.cat_shift, y, stream));
          x = y;
          h = h2;
          wd = w2;
          continue;
        }
        if (blk.has_down) {
          DIRB_TRY(run_conv(n, blk.down, x, sb, h, wd, nullptr, 0, rs, stream));
          res = rs;
        }
        DIRB_TRY(run_conv(n, blk.c3, t2, sb, h2, w2, res, 1, y, stream));
        x = y;
        h = h2;
        wd = w2;
      }
      if (s == 4) {
        const int C4 = n->stage_ch[4];
        if (b0 + sb >= cb) DIRB_TRY(record_tap(n, "layer4", x, sb, ho, wo, C4, stream));
        if (n->fpn) {
          // ---- FPN head, rmac_resnet_fpn.py:52-90
          const int C3 = n->stage_ch[3], h3 = w.h[3], w3 = w.w[3], Ct = C3 + C4;
          const __half* x4 = w.stage_out[3] + static_cast<size_t>(b0) * h3 * w3 * C3;
          if (n->fpn_mode == 1) {
            // relu(conv1x5(upsample(x5))) == upsample(relu(conv1x5(x5))): the 1x1 convolution runs on the small map.
            // x (layer4 output) sits in scratch[2] or [3]; scratch[0] / [1] are free after the last block.
            __half* tbuf = w.scratch[0];
            __half* x4p = w.scratch[1];
            DIRB_TRY(run_conv(n, n->fpn_lat, x, sb, ho, wo, nullptr, 1, tbuf, stream));
            {
              ProfScope ps(n, stream, 2, 0, 2.0 * sb * (2.0 * h3 * w3 + static_cast<double>(ho) * wo) * C3);
              DIRB_TRY(upsample_add(x4, tbuf, x4p, sb, h3, w3, ho, wo, C3, stream));
            }
            DIRB_TRY(run_conv(n, n->fpn_smooth, x4p, sb, h3, w3, nullptr, 1, tbuf, stream));
            x4 = tbuf;
            if (b0 + sb >= cb) DIRB_TRY(record_tap(n, "fpn_c4", x4, sb, h3, w3, C3, stream));
          }
          ProfScope ps(n, stream, 3, n->without_fc ? 0.0 : 2.0 * sb * static_cast<double>(Ct) * n->out_dim,
                       2.0 * sb * (static_cast<double>(ho) * wo * C4 + static_cast<double>(h3) * w3 * C3));
          const size_t partial_floats = std::max(head_partial_floats(w.sub[4], h3 * w3, C3), head_partial_floats(w.sub[4], ho * wo, C4));
          float* partial = w.head_ws;
          float* g = partial + partial_floats;
          float* yv = g + static_cast<size_t>(w.sub[4]) * Ct;
          DIRB_TRY(head_pool(x4, sb, h3 * w3, C3, 0, n->gem_p4, n->gem_eps, 0, partial, g, Ct, 0, stream));    // torch.cat((x4, x5), 1)
          DIRB_TRY(head_pool(x, sb, ho * wo, C4, 0, n->gem_p, n->gem_eps, 0, partial, g, Ct, C3, stream));
          if (n->norm_features) DIRB_TRY(l2_normalize(g, sb, Ct, 1e-12f, g, nullptr, stream));
          DIRB_TRY(head_fc_l2(g, sb, Ct, n->without_fc ? nullptr : n->fc_w, n->without_fc ? nullptr : n->fc_b, D, yv,
                              desc_dev + static_cast<size_t>(b0) * D,
                              desc16_dev ? desc16_dev + static_cast<size_t>(b0) * D : nullptr, stream));
          if (!n->without_fc) n->last_flops += 2.0 * sb * static_cast<double>(Ct) * n->out_dim;
          continue;
        }
        ProfScope ps(n, stream, 3, n->without_fc ? 0.0 : 2.0 * sb * static_cast<double>(C4) * n->out_dim, 2.0 * sb * ho * wo * static_cast<double>(C4), "head pool+fc+l2");
        if (n->center_bias > 0.0f)   // x is a scratch buffer whose only remaining reader is the pooling below
          DIRB_TRY(center_bias(const_cast<__half*>(x), sb, ho, wo, C4, n->center_bias, stream));
        DIRB_TRY(head_pool_fc_l2(x, sb, ho * wo, C4, n->pooling, n->gem_p, n->gem_eps, n->norm_features,
                                 n->without_fc ? nullptr : n->fc_w, n->without_fc ? nullptr : n->fc_b, D, w.head_ws,
                                 desc_dev + static_cast<size_t>(b0) * D,
                                 desc16_dev ? desc16_dev + static_cast<size_t>(b0) * D : nullptr, stream, n->head_bar));
        if (!n->without_fc) n->last_flops += 2.0 * sb * static_cast<double>(C4) * n->out_dim;
      }
    }
    if (s < 4) DIRB_TRY(record_tap(n, "layer" + std::to_string(s), w.stage_out[s], cb, ho, wo, n->stage_ch[s], stream));
    first = last;
  }
  return 0;
}

static int check_forward_args(dirb200_net* n, int B, int H, int W) {
  DIRB_REQUIRE(n->finalized, DIRB200_ESTATE, "dirb200_net_finalize has not been called");
  DIRB_REQUIRE(B >= 1 && H >= 32 && W >= 32, DIRB200_ENOTSUP, "need B >= 1 and H, W >= 32 (got %d, %d, %d)", B, H, W);
  return 0;
}

int dirb200_net_forward(dirb200_net* n, const float* imgs_dev, int B, int H, int W, float* desc_dev, void* desc16_dev,
                        void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(n && imgs_dev && desc_dev, DIRB200_EINVAL, "null argument");
  DIRB_TRY(check_forward_args(n, B, H, W));
  DIRB_CUDA(cudaSetDevice(n->device));
  const int64_t launches0 = launches_total();
  n->last_flops = 0;
  if (n->profile != 2) n->prof.reset();
  const int chunk = n->chunk > 0 ? std::min(n->chunk, B) : auto_chunk(B, H, W);
  const int D = n->desc_dim();
  Workspace w;
  DIRB_TRY(setup_workspace(n, chunk, H, W, &w));
  for (int b0 = 0; b0 < B; b0 += chunk) {
    const int cb = std::min(chunk, B - b0);
    DIRB_TRY(run_chunk(n, w, imgs_dev + static_cast<size_t>(b0) * 3 * H * W, cb, H, W,
                       desc_dev + static_cast<size_t>(b0) * D,
                       desc16_dev ? static_cast<__half*>(desc16_dev) + static_cast<size_t>(b0) * D : nullptr, stream));
  }
  n->last_launches = launches_total() - launches0;
  return 0;
}

// Host buffers in, host descriptors out.  The batch is cut into chunks of `host_chunk` images; the H2D copy of
// chunk i+1 (copy stream) overlaps the network pass over chunk i (compute stream), two device input buffers.
static int forward_host_impl(dirb200_net* n, const void* imgs_host, int is_u8, int B, int H, int W, float* desc_host);

int dirb200_net_forward_host(dirb200_net* n, const float* imgs_host, int B, int H, int W, float* desc_host) {
  return forward_host_impl(n, imgs_host, 0, B, H, W, desc_host);
}

int dirb200_net_forward_host_u8(dirb200_net* n, const uint8_t* imgs_host, int B, int H, int W, float* desc_host) {
  return forward_host_impl(n, imgs_host, 1, B, H, W, desc_host);
}

int dirb200_net_forward_u8(dirb200_net* n, const uint8_t* imgs_dev, int B, int H, int W, float* desc_dev, void* desc16_dev,
                           void* stream_) {
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DIRB_REQUIRE(n && imgs_dev && desc_dev, DIRB200_EINVAL, "null argument");
  DIRB_TRY(check_forward_args(n, B, H, W));
  DIRB_CUDA(cudaSetDevice(n->device));
  const int64_t launches0 = launches_total();
  n->last_flops = 0;
  if (n->profile != 2) n->prof.reset();
  const int chunk = n->chunk > 0 ? std::min(n->chunk, B) : auto_chunk(B, H, W);
  const int D = n->desc_dim();
  Workspace w;
  DIRB_TRY(setup_workspace(n, chunk, H, W, &w));
  for (int b0 = 0; b0 < B; b0 += chunk) {
    const int cb = std::min(chunk, B - b0);
    DIRB_TRY(run_chunk(n, w, nullptr, cb, H, W, desc_dev + static_cast<size_t>(b0) * D,
                       desc16_dev ? static_cast<__half*>(desc16_dev) + static_cast<size_t>(b0) * D : nullptr, stream,
                       imgs_dev + static_cast<size_t>(b0) * 3 * H * W));
  }
  n->last_launches = launches_total() - launches0;
  return 0;
}

static int forward_host_impl(dirb200_net* n, const void* imgs_host_, int is_u8, int B, int H, int W, float* desc_host) {
  const uint8_t* imgs_host = static_cast<const uint8_t*>(imgs_host_);
  DIRB_REQUIRE(n && imgs_host && desc_host, DIRB200_EINVAL, "null argument");
  DIRB_TRY(check_forward_args(n, B, H, W));
  DIRB_CUDA(cudaSetDevice(n->device));
  if (!n->own_stream) DIRB_CUDA(cudaStreamCreateWithFlags(&n->own_stream, cudaStreamNonBlocking));
  if (!n->copy_stream) DIRB_CUDA(cudaStreamCreateWithFlags(&n->copy_stream, cudaStreamNonBlocking));
  // Chunk schedule: small chunks first so that compute starts after a short copy, then doubling sizes (large chunks
  // run the network more efficiently): host_chunk/2, host_chunk/2, host_chunk, 2*host_chunk, ... (option "chunk"
  // forces a uniform size).
  std::vector<int> sizes;
  {
    int left = B;
    if (n->chunk > 0) {
      while (left > 0) { sizes.push_back(std::min(left, n->chunk)); left -= sizes.back(); }
    } else {
      int c = std::max(1, n->host_chunk / 2);
      int reps = 2;
      while (left > 0) {
        const int v = std::min(left, c);
        sizes.push_back(v);
        left -= v;
        if (--reps == 0) { c = std::min(c * 2, 2 * n->host_chunk); reps = 1; }
      }
    }
  }
  const int nchunks = static_cast<int>(sizes.size());
  const int chunk = *std::max_element(sizes.begin(), sizes.end());
  const size_t img_bytes = static_cast<size_t>(3) * H * W * (is_u8 ? 1 : 4);
  const size_t in_bytes = 2 * static_cast<size_t>(chunk) * img_bytes;
  const int D = n->desc_dim();
  const size_t out_bytes = static_cast<size_t>(B) * D * 4;
  if (in_bytes > n->h2d_bytes) {
    if (n->h2d) DIRB_CUDA(cudaFree(n->h2d));
    n->h2d = nullptr;
    DIRB_CUDA(cudaMalloc(reinterpret_cast<void**>(&n->h2d), in_bytes));
    n->h2d_bytes = in_bytes;
  }
  if (out_bytes > n->d_desc_bytes) {
    if (n->d_desc) DIRB_CUDA(cudaFree(n->d_desc));
    n->d_desc = nullptr;
    DIRB_CUDA(cudaMalloc(reinterpret_cast<void**>(&n->d_desc), out_bytes));
    n->d_desc_bytes = out_bytes;
  }
  while (n->pipe_events.size() < static_cast<size_t>(2 * nchunks)) {
    cudaEvent_t e;
    DIRB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    n->pipe_events.push_back(e);
  }
  const int64_t launches0 = launches_total();
  n->last_flops = 0;
  if (n->profile != 2) n->prof.reset();
  Workspace w;
  DIRB_TRY(setup_workspace(n, chunk, H, W, &w));
  int b0 = 0;
  for (int c = 0; c < nchunks; ++c) {
    const int cb = sizes[c];
    uint8_t* dst = reinterpret_cast<uint8_t*>(n->h2d) + static_cast<size_t>(c & 1) * chunk * img_bytes;
    cudaEvent_t copied = n->pipe_events[2 * c], done = n->pipe_events[2 * c + 1];
    if (c >= 2) DIRB_CUDA(cudaStreamWaitEvent(n->copy_stream, n->pipe_events[2 * (c - 2) + 1], 0));   // buffer free
    DIRB_CUDA(cudaMemcpyAsync(dst, imgs_host + static_cast<size_t>(b0) * img_bytes, static_cast<size_t>(cb) * img_bytes,
                              cudaMemcpyHostToDevice, n->copy_stream));
    DIRB_CUDA(cudaEventRecord(copied, n->copy_stream));
    DIRB_CUDA(cudaStreamWaitEvent(n->own_stream, copied, 0));
    DIRB_TRY(run_chunk(n, w, is_u8 ? nullptr : reinterpret_cast<const float*>(dst), cb, H, W,
                       n->d_desc + static_cast<size_t>(b0) * D, nullptr, n->own_stream, is_u8 ? dst : nullptr));
    DIRB_CUDA(cudaEventRecord(done, n->own_stream));
    b0 += cb;
  }
  DIRB_CUDA(cudaMemcpyAsync(desc_host, n->d_desc, out_bytes, cudaMemcpyDeviceToHost, n->own_stream));
  DIRB_CUDA(cudaStreamSynchronize(n->own_stream));
  n->last_launches = launches_total() - launches0;
  return 0;
}

// Aggregated per-class timing of the last forward run with option "profile": out[4][4] = {launches, ms, flops, bytes}
// for class 0 tcgen05 convs, 1 stem conv, 2 layout + maxpool, 3 head.  Synchronises the device.
int dirb200_net_profile(dirb200_net* n, double* out16) {
  DIRB_REQUIRE(n && out16, DIRB200_EINVAL, "null argument");
  DIRB_CUDA(cudaDeviceSynchronize());
  for (int i = 0; i < 16; ++i) out16[i] = 0;
  for (auto& r : n->prof.recs) {
    float ms = 0;
    DIRB_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    double* o = out16 + 4 * r.cls;
    o[0] += 1; o[1] += ms; o[2] += r.flops; o[3] += r.bytes;
  }
  return 0;
}

// Per launch-type timing of the profiled forward(s) as JSON text: [{"tag","cls","launches","ms","flops","bytes"}, ...]
// in first-launch order.  Returns the number of bytes needed (incl. the terminator) through *needed when buf is too
// small or NULL.  Synchronises the device.
int dirb200_net_profile_table(dirb200_net* n, char* buf, size_t cap, size_t* needed) {
  DIRB_REQUIRE(n, DIRB200_EINVAL, "null argument");
  DIRB_CUDA(cudaDeviceSynchronize());
  struct Row { std::string tag; int cls; double launches, ms, flops, bytes; };
  std::vector<Row> rows;
  std::map<std::string, size_t> at;
  for (auto& r : n->prof.recs) {
    float ms = 0;
    DIRB_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    auto it = at.find(r.tag);
    if (it == at.end()) {
      at[r.tag] = rows.size();
      rows.push_back(Row{r.tag, r.cls, 0, 0, 0, 0});
      it = at.find(r.tag);
    }
    Row& row = rows[it->second];
    row.launches += 1; row.ms += ms; row.flops += r.flops; row.bytes += r.bytes;
  }
  std::string out = "[";
  for (size_t i = 0; i < rows.size(); ++i) {
    char line[320];
    snprintf(line, sizeof(line), "%s{\"tag\": \"%s\", \"cls\": %d, \"launches\": %.0f, \"ms\": %.6f, \"flops\": %.6e, \"bytes\": %.6e}",
             i ? ", " : "", rows[i].tag.c_str(), rows[i].cls, rows[i].launches, rows[i].ms, rows[i].flops, rows[i].bytes);
    out += line;
  }
  out += "]";
  if (needed) *needed = out.size() + 1;
  if (buf && cap >= out.size() + 1) memcpy(buf, out.c_str(), out.size() + 1);
  return 0;
}

int dirb200_net_debug_stage(dirb200_net* n, const char* what, void* dst_dev, size_t capacity, int dims[4],
                            void* stream_) {
  DIRB_REQUIRE(n && what && dims, DIRB200_EINVAL, "null argument");
  auto it = n->taps.find(what);
  DIRB_REQUIRE(it != n->taps.end() && it->second.ptr, DIRB200_EKEY,
               "no stage '%s' recorded (set option debug_taps=1 and run a forward first)", what);
  const auto& t = it->second;
  const size_t bytes = static_cast<size_t>(t.n) * t.h * t.w * t.c * 2;
  dims[0] = t.n; dims[1] = t.h; dims[2] = t.w; dims[3] = t.c;     // also when the buffer is too small: size query
  if (!dst_dev) return 0;
  DIRB_REQUIRE(bytes <= capacity, DIRB200_EINVAL, "stage '%s' needs %zu bytes", what, bytes);
  DIRB_CUDA(cudaMemcpyAsync(dst_dev, t.ptr, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream_)));
  return 0;
}

int dirb200_net_last_launches(dirb200_net* n, int64_t* launches, double* flops) {
  DIRB_REQUIRE(n, DIRB200_EINVAL, "null");
  if (launches) *launches = n->last_launches;
  if (flops) *flops = n->last_flops;
  return 0;
}

int dirb200_net_destroy(dirb200_net* n) {
  if (!n) return 0;
  cudaSetDevice(n->device);
  for (void* p : n->owned) cudaFree(p);
  for (auto& kv : n->taps) if (kv.second.ptr) cudaFree(kv.second.ptr);
  if (n->ws) cudaFree(n->ws);
  if (n->h2d) cudaFree(n->h2d);
  if (n->d_desc) cudaFree(n->d_desc);
  if (n->own_stream) cudaStreamDestroy(n->own_stream);
  if (n->copy_stream) cudaStreamDestroy(n->copy_stream);
  for (auto e : n->pipe_events) cudaEventDestroy(e);
  delete n;
  return 0;
}

}  // extern "C"
