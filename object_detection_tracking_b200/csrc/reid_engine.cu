// OSNet-x1.0 ReID embedding engine (torchreid FeatureExtractor replacement) and the distance-matrix
// GEMM, behind the C ABI.  One b2_reid = one device = one fixed crop batch; the pass is a fixed launch
// sequence replayed as a CUDA graph.
//
// Reference graph: torchreid/models/osnet.py OSNet.forward (:413-438) with osnet_x1_0 (:522-534):
//   conv1 7x7/2 + BN + ReLU -> maxpool 3/2 -> [OSBlock x2 + Conv1x1 + AvgPool2] x2 -> OSBlock x2 -> conv5 1x1
//   -> global avg-pool -> fc(512) + BatchNorm1d + ReLU  (eval mode returns this 512-d vector)
// Input contract (torchreid/feature_extractor.py:190-196,209-252): RGB uint8 crops already resized to
// 256x128 (the PIL resize stays on the host), ToTensor + Normalize happen in the stem pack kernel.
//
// Second model (b2_reid_create_model(..., model = 1)): torchreid's resnet101 (torchreid/models/resnet.py:441-455 ->
// ResNet(Bottleneck, [3, 4, 23, 3], last_stride=2, fc_dims=None), forward :342-366), the vehicle extractor of
// single_video_reid.py:410-415 with image_size (128, 256):  conv1 7x7/2 + BN + ReLU -> maxpool 3/2 pad 1 ->
// layer1..4 of Bottleneck blocks (1x1 -> 3x3 carrying the stride -> 1x1, BN folded, ReLU / residual in the epilogue,
// 1x1 strided downsample on the first block of a layer) -> global avg-pool = the 2048-d feature (eval mode).
// Every conv runs on conv_tc_kernel (tcgen05); max-pool / global-average kernels are shared with OSNet.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <memory>
#include <string>
#include <vector>

#include "../../include/b200det.h"
#include "common.h"
#include "kernels.h"

using namespace b2;

namespace {

struct RPlanes {
  __half* hi = nullptr;
  __half* lo = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  size_t elems() const { return static_cast<size_t>(B) * H * W * C; }
};

struct RConv {
  std::string wname;      // torch parameter name of the conv weight (OIHW)
  std::string bnname;     // BatchNorm prefix ("" = none)
  std::string biasname;   // Linear bias ("" = none)
  ConvDesc d;
  ConvWeights w;
  ConvIO io;
  ConvPlan* plan = nullptr;
  int cin_real = 0, cout_real = 0, kind = 0;   // kind 0 = 1x1/dense, 1 = stem (packed 7x7), 2 = RxS conv (torch OIHW)
};

struct RDw {
  std::string wname, bnname;
  RPlanes in, out;
  float* w = nullptr;      // [9][C]
  float* bias = nullptr;   // [C]
  int creal = 0;
};

struct RGate {
  std::string prefix;      // "...gate"
  RPlanes s[4], out;
  float *pooled = nullptr, *gates = nullptr, *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr;
  int creal = 0, cr = 0;
};

struct RStep {
  int kind;   // 0 conv, 1 pack, 2 maxpool, 3 dw, 4 gate, 5 avgpool, 6 final gap
  int idx;
  RPlanes a, b;
};

}  // namespace

struct b2_reid {
  int device = 0, num_sms = 148, B = 0;
  int model = 0;                     // 0 osnet_x1_0, 1 resnet101
  int in_h = 256, in_w = 128;        // crop size (h, w) the extractor resizes to
  int feat_dim = 512;
  bool split = true;
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  std::vector<std::unique_ptr<RConv>> convs;
  std::vector<std::unique_ptr<RDw>> dws;
  std::vector<std::unique_ptr<RGate>> gates;
  std::vector<RStep> steps;
  std::map<std::string, RPlanes> named;     // stage-addressable activations (parity tests)
  uint8_t* crops = nullptr;
  RPlanes stem_u, gap_planes;
  float* gap_f32 = nullptr;
  float* feats = nullptr;      // [Bpad][512]
  cudaGraphExec_t graph = nullptr;
  bool loaded = false;

  template <typename T>
  T* alloc(size_t n) {
    void* p = nullptr;
    if (cudaMalloc(&p, n * sizeof(T) + 256) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, n * sizeof(T) + 256);
    allocs.push_back(p);
    return static_cast<T*>(p);
  }
  RPlanes planes(int b, int h, int w, int c) {
    RPlanes p;
    p.B = b; p.H = h; p.W = w; p.C = c;
    p.hi = alloc<__half>(p.elems());
    p.lo = split ? alloc<__half>(p.elems()) : nullptr;
    return p;
  }
};

namespace {

int pad64(int c) { return (c + 63) / 64 * 64; }

// 1x1 conv (or dense) in -> out, optional BN / bias / ReLU / residual
RConv* add_pw(b2_reid* c, const std::string& wname, const std::string& bn, const std::string& bias, const RPlanes& in,
              int cin_real, const RPlanes& out, int cout_real, bool relu, const RPlanes* res, float* out_f32 = nullptr,
              int ldc32 = 0) {
  std::unique_ptr<RConv> L(new RConv());
  L->wname = wname; L->bnname = bn; L->biasname = bias;
  L->cin_real = cin_real; L->cout_real = cout_real;
  ConvDesc& d = L->d;
  d.B = in.B; d.in_H = in.H; d.in_W = in.W; d.Cin = in.C; d.in_pitch_H = in.H; d.in_pitch_W = in.W; d.in_ld = in.C;
  d.Cout = cout_real; d.relu = relu ? 1 : 0;
  if (out_f32) { d.out_H = in.H; d.out_W = in.W; d.ldc = ldc32; }
  else { d.out_H = out.H; d.out_W = out.W; d.ldc = out.C; }
  if (res) { d.res_H = res->H; d.res_W = res->W; d.ldr = res->C; }
  L->w.Cout_pad = (cout_real + 15) / 16 * 16;
  L->w.K = in.C;
  L->w.w_hi = c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K);
  L->w.w_lo = c->split ? c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K) : nullptr;
  L->w.bias = c->alloc<float>(L->w.Cout_pad);
  L->io.in_hi = in.hi; L->io.in_lo = in.lo; L->io.out_hi = out.hi; L->io.out_lo = out.lo; L->io.out_f32 = out_f32;
  if (res) { L->io.res_hi = res->hi; L->io.res_lo = res->lo; }
  RConv* raw = L.get();
  c->steps.push_back({0, static_cast<int>(c->convs.size()), RPlanes(), RPlanes()});
  c->convs.push_back(std::move(L));
  return raw;
}

RPlanes add_light(b2_reid* c, const std::string& pre, const RPlanes& in, int creal) {
  // LightConv3x3 (osnet.py:128-156): 1x1 linear (no BN) -> depthwise 3x3 -> BN -> ReLU
  RPlanes t = c->planes(in.B, in.H, in.W, in.C);
  add_pw(c, pre + ".conv1.weight", "", "", in, creal, t, creal, false, nullptr);
  std::unique_ptr<RDw> D(new RDw());
  D->wname = pre + ".conv2.weight"; D->bnname = pre + ".bn";
  D->in = t; D->out = c->planes(in.B, in.H, in.W, in.C);
  D->w = c->alloc<float>(9 * in.C); D->bias = c->alloc<float>(in.C);
  D->creal = creal;
  RPlanes out = D->out;
  c->steps.push_back({3, static_cast<int>(c->dws.size()), RPlanes(), RPlanes()});
  c->dws.push_back(std::move(D));
  return out;
}

RPlanes add_osblock(b2_reid* c, const std::string& pre, const RPlanes& x, int cin, int cout) {
  // OSBlock (osnet.py:223-276)
  const int mid = cout / 4, midp = pad64(mid);
  RPlanes x1 = c->planes(x.B, x.H, x.W, midp);
  add_pw(c, pre + ".conv1.conv.weight", pre + ".conv1.bn", "", x, cin, x1, mid, true, nullptr);
  RPlanes s[4];
  const char* names[4] = {".conv2a", ".conv2b", ".conv2c", ".conv2d"};
  for (int k = 0; k < 4; ++k) {
    RPlanes t = x1;
    if (k == 0) t = add_light(c, pre + names[k], t, mid);
    else
      for (int j = 0; j <= k; ++j) t = add_light(c, pre + names[k] + "." + std::to_string(j), t, mid);
    s[k] = t;
  }
  std::unique_ptr<RGate> G(new RGate());
  G->prefix = pre + ".gate";
  for (int k = 0; k < 4; ++k) G->s[k] = s[k];
  G->out = c->planes(x.B, x.H, x.W, midp);
  G->creal = mid; G->cr = mid / 16;
  G->pooled = c->alloc<float>(static_cast<size_t>(x.B) * 4 * midp);
  G->gates = c->alloc<float>(static_cast<size_t>(x.B) * 4 * midp);
  G->w1 = c->alloc<float>(static_cast<size_t>(G->cr) * mid); G->b1 = c->alloc<float>(G->cr);
  G->w2 = c->alloc<float>(static_cast<size_t>(mid) * G->cr); G->b2 = c->alloc<float>(mid);
  RPlanes x2 = G->out;
  c->named[pre + ".x1"] = x1;
  for (int k = 0; k < 4; ++k) c->named[pre + ".s" + std::to_string(k)] = s[k];
  c->named[pre + ".x2"] = x2;
  c->steps.push_back({4, static_cast<int>(c->gates.size()), RPlanes(), RPlanes()});
  c->gates.push_back(std::move(G));
  RPlanes identity = x;
  if (cin != cout) {
    identity = c->planes(x.B, x.H, x.W, cout);
    add_pw(c, pre + ".downsample.conv.weight", pre + ".downsample.bn", "", x, cin, identity, cout, false, nullptr);
  }
  RPlanes out = c->planes(x.B, x.H, x.W, cout);
  add_pw(c, pre + ".conv3.conv.weight", pre + ".conv3.bn", "", x2, mid, out, cout, true, &identity);   // relu(x3 + identity)
  return out;
}

int build(b2_reid* c) {
  const int B = c->B, H = 256, W = 128;
  c->crops = c->alloc<uint8_t>(static_cast<size_t>(B) * H * W * 3);
  // conv1 7x7/2 pad 3 (osnet.py:307) through the packed-operand trick of stem.cu
  const int h1 = (H + 6 - 7) / 2 + 1, w1 = (W + 6 - 7) / 2 + 1;
  c->stem_u = c->planes(B, h1 + 3, w1, 64);
  c->steps.push_back({1, 0, RPlanes(), RPlanes()});
  RPlanes c1 = c->planes(B, h1, w1, 64);
  {
    RConv* L = add_pw(c, "conv1.conv.weight", "conv1.bn", "", c->stem_u, 64, c1, 64, true, nullptr);
    L->kind = 1;
    L->d.R = 4; L->d.S = 1; L->w.K = 4 * 64;
    L->d.in_H = h1 + 3; L->d.out_H = h1;
    // reallocate the packed weight for K = 256
    L->w.w_hi = c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K);
    L->w.w_lo = c->split ? c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K) : nullptr;
  }
  RPlanes p1 = c->planes(B, h1 / 2, w1 / 2, 64);       // maxpool 3/2 pad 1 (:308)
  c->steps.push_back({2, 0, c1, p1});
  c->named["stem_u"] = c->stem_u;
  c->named["conv1"] = c1;
  c->named["maxpool"] = p1;
  RPlanes x = p1;
  const int chans[4] = {64, 256, 384, 512};
  for (int stage = 0; stage < 3; ++stage) {
    const std::string sn = "conv" + std::to_string(stage + 2);
    x = add_osblock(c, sn + ".0", x, chans[stage], chans[stage + 1]);
    c->named[sn + ".0"] = x;
    x = add_osblock(c, sn + ".1", x, chans[stage + 1], chans[stage + 1]);
    c->named[sn + ".1"] = x;
    if (stage < 2) {   // transition: Conv1x1 + AvgPool2d(2) (:375-381)
      RPlanes t = c->planes(B, x.H, x.W, x.C);
      add_pw(c, sn + ".2.0.conv.weight", sn + ".2.0.bn", "", x, x.C, t, x.C, true, nullptr);
      RPlanes q = c->planes(B, x.H / 2, x.W / 2, x.C);
      c->steps.push_back({5, 0, t, q});
      c->named[sn + ".t"] = t;
      x = q;
      c->named[sn] = x;
    }
  }
  RPlanes x5 = c->planes(B, x.H, x.W, 512);
  add_pw(c, "conv5.conv.weight", "conv5.bn", "", x, 512, x5, 512, true, nullptr);
  c->named["conv5"] = x5;
  // global average pool -> fc + BN1d + ReLU (:428-431, fc built by _construct_fc_layer :386-405)
  const int Bp = (B + 127) / 128 * 128;
  c->gap_f32 = c->alloc<float>(static_cast<size_t>(Bp) * 512);
  c->gap_planes = c->planes(1, 1, Bp, 512);
  c->steps.push_back({6, 0, x5, RPlanes()});
  c->feats = c->alloc<float>(static_cast<size_t>(Bp) * 512);
  RPlanes gp = c->gap_planes; gp.W = B;
  add_pw(c, "fc.0.weight", "fc.1", "fc.0.bias", gp, 512, RPlanes(), 512, true, nullptr, c->feats, 512);
  for (auto& L : c->convs) {
    L->plan = conv_tc_plan_create(L->d, L->w, L->io, c->split, c->num_sms);
    if (!L->plan) {
      set_error("reid plan for " + L->wname + ": " + last_error());
      return -1;
    }
  }
  return 0;
}

// General RxS conv (torch Conv2d, symmetric padding) + BN (+ReLU) (+residual) on conv_tc_kernel.
RConv* add_conv(b2_reid* c, const std::string& wname, const std::string& bn, const RPlanes& in, const RPlanes& out, int k,
                int stride, int pad, bool relu, const RPlanes* res) {
  RConv* L = add_pw(c, wname, bn, "", in, in.C, out, out.C, relu, res);
  if (k != 1 || stride != 1) {
    L->kind = 2;
    L->d.R = k; L->d.S = k; L->d.stride = stride;
    L->d.pad_t = L->d.pad_l = pad;
    // stride 2 on even extents: the last window ends one row / column before torch's bottom / right padding, so
    // (pad, pad - 1) is the same convolution -- and exactly the geometry the detector's strided layers use
    // (nn.py:487-492 3x3 with pads (1,0); :555-560 1x1 with the last row / column dropped).
    L->d.pad_b = L->d.pad_r = stride == 2 ? pad - 1 : pad;
    L->w.K = k * k * in.C;
    L->w.w_hi = c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K);
    L->w.w_lo = c->split ? c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K) : nullptr;
  }
  return L;
}

// torchreid resnet101 (resnet.py:157-366): see the header comment.
int build_resnet101(b2_reid* c) {
  const int B = c->B, H = c->in_h, W = c->in_w;
  c->crops = c->alloc<uint8_t>(static_cast<size_t>(B) * H * W * 3);
  const int h1 = (H + 6 - 7) / 2 + 1, w1 = (W + 6 - 7) / 2 + 1;       // conv1 7x7/2 pad 3 (:211-213)
  c->stem_u = c->planes(B, h1 + 3, w1, 64);
  c->steps.push_back({1, 0, RPlanes(), RPlanes()});
  RPlanes c1 = c->planes(B, h1, w1, 64);
  {
    RConv* L = add_pw(c, "conv1.weight", "bn1", "", c->stem_u, 64, c1, 64, true, nullptr);
    L->kind = 1;
    L->d.R = 4; L->d.S = 1; L->w.K = 4 * 64;
    L->d.in_H = h1 + 3; L->d.out_H = h1;
    L->w.w_hi = c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K);
    L->w.w_lo = c->split ? c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K) : nullptr;
  }
  RPlanes x = c->planes(B, h1 / 2, w1 / 2, 64);                       // maxpool 3/2 pad 1 (:216)
  c->steps.push_back({2, 0, c1, x});
  c->named["conv1"] = c1;
  c->named["maxpool"] = x;
  const int blocks[4] = {3, 4, 23, 3}, planes[4] = {64, 128, 256, 512};
  for (int li = 0; li < 4; ++li) {
    const std::string ln = "layer" + std::to_string(li + 1);
    for (int bi = 0; bi < blocks[li]; ++bi) {
      const std::string pre = ln + "." + std::to_string(bi);
      const int stride = (bi == 0 && li > 0) ? 2 : 1;                 // _make_layer :246-290 (last_stride = 2)
      const int width = planes[li], cout = width * 4;
      if (stride == 2 && ((x.H | x.W) & 1)) {
        set_error("resnet101 reid: odd feature-map extent before a stride-2 layer");
        return -1;
      }
      const int ho = x.H / stride, wo = x.W / stride;
      RPlanes t1 = c->planes(B, x.H, x.W, width);
      add_conv(c, pre + ".conv1.weight", pre + ".bn1", x, t1, 1, 1, 0, true, nullptr);
      RPlanes t2 = c->planes(B, ho, wo, width);
      add_conv(c, pre + ".conv2.weight", pre + ".bn2", t1, t2, 3, stride, 1, true, nullptr);   // stride on the 3x3 (:126)
      RPlanes identity = x;
      if (bi == 0) {                                                   // downsample: conv1x1(stride) + BN (:262-268)
        identity = c->planes(B, ho, wo, cout);
        add_conv(c, pre + ".downsample.0.weight", pre + ".downsample.1", x, identity, 1, stride, 0, false, nullptr);
      }
      RPlanes out = c->planes(B, ho, wo, cout);
      add_conv(c, pre + ".conv3.weight", pre + ".bn3", t2, out, 1, 1, 0, true, &identity);       // relu(bn3 + identity)
      x = out;
      c->named[pre] = x;
    }
    c->named[ln] = x;
  }
  const int Bp = (B + 127) / 128 * 128;
  c->feats = c->alloc<float>(static_cast<size_t>(Bp) * c->feat_dim);
  c->steps.push_back({7, 0, x, RPlanes()});                            // global_avgpool -> v (:355-359)
  for (auto& L : c->convs) {
    L->plan = conv_tc_plan_create(L->d, L->w, L->io, c->split, c->num_sms);
    if (!L->plan) {
      set_error("reid plan for " + L->wname + ": " + last_error());
      return -1;
    }
  }
  return 0;
}

int run_step(b2_reid* c, const RStep& s) {
  cudaStream_t st = c->stream;
  switch (s.kind) {
    case 0: return conv_tc_launch(c->convs[s.idx]->plan, st);
    case 1: return stem_pack_launch(c->crops, 1, c->B, c->in_h, c->in_w, c->stem_u.hi, c->stem_u.lo, c->stem_u.H, c->stem_u.W, 1, st);
    case 2: return maxpool_launch(s.a.hi, s.a.lo, s.a.B, s.a.H, s.a.W, s.a.C, s.b.hi, s.b.lo, s.b.H, s.b.W, st);
    case 3: {
      RDw* d = c->dws[s.idx].get();
      return dwconv3x3_launch(d->in.hi, d->in.lo, d->in.B, d->in.H, d->in.W, d->in.C, d->w, d->bias, d->out.hi, d->out.lo, st);
    }
    case 4: {
      RGate* g = c->gates[s.idx].get();
      const int C = g->out.C, HW = g->out.H * g->out.W, B = g->out.B;
      for (int k = 0; k < 4; ++k)
        if (gap_launch(g->s[k].hi, g->s[k].lo, B, HW, C, g->pooled + static_cast<size_t>(k) * C, 4 * C, st)) return -1;
      if (gate_mlp_launch(g->pooled, B * 4, C, g->creal, g->cr, g->w1, g->b1, g->w2, g->b2, g->gates, st)) return -1;
      const __half* hi[4] = {g->s[0].hi, g->s[1].hi, g->s[2].hi, g->s[3].hi};
      const __half* lo[4] = {g->s[0].lo, g->s[1].lo, g->s[2].lo, g->s[3].lo};
      return gated_sum4_launch(hi, lo, g->gates, B, HW, C, g->out.hi, g->out.lo, st);
    }
    case 5: return avgpool2_launch(s.a.hi, s.a.lo, s.a.B, s.a.H, s.a.W, s.a.C, s.b.hi, s.b.lo, st);
    case 6:
      if (gap_launch(s.a.hi, s.a.lo, s.a.B, s.a.H * s.a.W, s.a.C, c->gap_f32, s.a.C, st)) return -1;
      return f32_to_planes(c->gap_f32, c->gap_planes.hi, c->gap_planes.lo, static_cast<size_t>(s.a.B) * s.a.C, st);
    case 7: return gap_launch(s.a.hi, s.a.lo, s.a.B, s.a.H * s.a.W, s.a.C, c->feats, s.a.C, st);
  }
  return -1;
}

struct WS {
  std::map<std::string, std::pair<const float*, int64_t>> m;
  const float* get(const std::string& n, int64_t expect) const {
    auto it = m.find(n);
    if (it == m.end()) { set_error("missing weight: " + n); return nullptr; }
    if (it->second.second != expect) {
      set_error("weight " + n + ": expected " + std::to_string(expect) + " values, got " + std::to_string(it->second.second));
      return nullptr;
    }
    return it->second.first;
  }
};

int bn_fold(const WS& ws, const std::string& bn, int C, std::vector<double>& scale, std::vector<double>& shift) {
  scale.assign(C, 1.0);
  shift.assign(C, 0.0);
  if (bn.empty()) return 0;
  const float* g = ws.get(bn + ".weight", C);
  const float* b = ws.get(bn + ".bias", C);
  const float* m = ws.get(bn + ".running_mean", C);
  const float* v = ws.get(bn + ".running_var", C);
  if (!g || !b || !m || !v) return -1;
  for (int i = 0; i < C; ++i) {
    scale[i] = static_cast<double>(g[i]) / sqrt(static_cast<double>(v[i]) + 1e-5);   // torch BatchNorm eps
    shift[i] = static_cast<double>(b[i]) - static_cast<double>(m[i]) * scale[i];
  }
  return 0;
}

int upload(b2_reid* c, RConv* L, const std::vector<float>& packed, const std::vector<float>& bias) {
  float* tmp = nullptr;
  B2_CUDA(cudaMalloc(&tmp, packed.size() * 4));
  // same stream as the conversion kernel: a pageable cudaMemcpy on the legacy stream may return before its DMA
  // lands, and the context stream is non-blocking (not ordered after the legacy stream)
  B2_CUDA(cudaMemcpyAsync(tmp, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice, c->stream));
  if (f32_to_planes(tmp, L->w.w_hi, L->w.w_lo, packed.size(), c->stream)) return -1;
  B2_CUDA(cudaMemcpyAsync(L->w.bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_CUDA(cudaFree(tmp));
  return 0;
}

}  // namespace

extern "C" {

int b2_reid_create(b2_reid** out, int device, int batch, int precision) {
  return b2_reid_create_model(out, device, batch, precision, 0);
}

int b2_reid_create_model(b2_reid** out, int device, int batch, int precision, int model) {
  B2_CHECK(out && batch >= 1, "b2_reid_create: bad argument");
  *out = nullptr;
  B2_CHECK(model == 0 || model == 1, "b2_reid_create_model: model must be 0 (osnet_x1_0) or 1 (resnet101)");
  B2_CUDA(cudaSetDevice(device));
  std::unique_ptr<b2_reid> c(new b2_reid());
  c->device = device; c->B = batch; c->split = precision == 1;
  c->model = model;
  if (model == 1) { c->in_h = 128; c->in_w = 256; c->feat_dim = 2048; }   // single_video_reid.py:410-415
  cudaDeviceProp prop;
  B2_CUDA(cudaGetDeviceProperties(&prop, device));
  B2_CHECK(prop.major == 10, "b2_reid_create: this library is built for sm_100a (B200) only");
  c->num_sms = prop.multiProcessorCount;
  B2_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  if ((model == 1 ? build_resnet101(c.get()) : build(c.get()))) { b2_reid_destroy(c.release()); return -1; }
  B2_CUDA(cudaDeviceSynchronize());
  *out = c.release();
  return 0;
}

void b2_reid_destroy(b2_reid* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (c->graph) cudaGraphExecDestroy(c->graph);
  for (auto& L : c->convs) if (L->plan) conv_tc_plan_destroy(L->plan);
  for (void* p : c->allocs) cudaFree(p);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

// state_dict of torchreid's osnet_x1_0 (names as model.state_dict(): "conv2.0.conv2b.1.conv1.weight", ...)
int b2_reid_load_weights(b2_reid* c, const char* const* names, const float* const* data, const int64_t* numel, int n) {
  B2_CHECK(c && names && data && numel, "b2_reid_load_weights: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  WS ws;
  for (int i = 0; i < n; ++i) ws.m[names[i]] = std::make_pair(data[i], numel[i]);
  for (auto& L : c->convs) {
    const int K = L->w.K, Cp = L->w.Cout_pad, co = L->cout_real, ci = L->cin_real;
    std::vector<float> packed(static_cast<size_t>(Cp) * K, 0.f), bias(Cp, 0.f);
    std::vector<double> scale, shift;
    if (bn_fold(ws, L->bnname, co, scale, shift)) return -1;
    if (L->kind == 1) {
      // torch OIHW [64,3,7,7] -> packed stem operand order (stem.cu): k = r*64 + s*12 + ry*6 + sx*3 + c
      const float* w = ws.get(L->wname, 64 * 3 * 49);
      if (!w) return -1;
      for (int o = 0; o < 64; ++o)
        for (int r = 0; r < 4; ++r)
          for (int ch = 0; ch < 48; ++ch) {
            const int s4 = ch / 12, r12 = ch % 12, ry = r12 / 6, sx = (r12 % 6) / 3, cc = r12 % 3;
            const int rr = 2 * r + ry, ss = 2 * s4 + sx;
            if (rr >= 7 || ss >= 7) continue;
            packed[static_cast<size_t>(o) * K + r * 64 + ch] = static_cast<float>(w[((o * 3 + cc) * 7 + rr) * 7 + ss] * scale[o]);
          }
    } else if (L->kind == 2) {
      // torch OIHW [co][ci][R][S] -> K-major [o][r][s][ci]
      const int R = L->d.R, S = L->d.S;
      const float* w = ws.get(L->wname, static_cast<int64_t>(co) * ci * R * S);
      if (!w) return -1;
      for (int o = 0; o < co; ++o)
        for (int i = 0; i < ci; ++i)
          for (int r = 0; r < R; ++r)
            for (int q = 0; q < S; ++q)
              packed[static_cast<size_t>(o) * K + (static_cast<size_t>(r) * S + q) * ci + i] =
                  static_cast<float>(w[((static_cast<size_t>(o) * ci + i) * R + r) * S + q] * scale[o]);
    } else {
      const float* w = ws.get(L->wname, static_cast<int64_t>(co) * ci);   // [O][I] (1x1 OIHW or Linear)
      if (!w) return -1;
      for (int o = 0; o < co; ++o)
        for (int i = 0; i < ci; ++i) packed[static_cast<size_t>(o) * K + i] = static_cast<float>(w[static_cast<size_t>(o) * ci + i] * scale[o]);
    }
    if (!L->biasname.empty()) {
      const float* b = ws.get(L->biasname, co);
      if (!b) return -1;
      for (int o = 0; o < co; ++o) shift[o] += static_cast<double>(b[o]) * scale[o];   // BN(Wx + b)
    }
    for (int o = 0; o < co; ++o) bias[o] = static_cast<float>(shift[o]);
    if (upload(c, L.get(), packed, bias)) return -1;
  }
  for (auto& D : c->dws) {
    const int C = D->in.C, cr = D->creal;
    const float* w = ws.get(D->wname, static_cast<int64_t>(cr) * 9);   // [C,1,3,3]
    std::vector<double> scale, shift;
    if (!w || bn_fold(ws, D->bnname, cr, scale, shift)) return -1;
    std::vector<float> pw(9 * C, 0.f), pb(C, 0.f);
    for (int ch = 0; ch < cr; ++ch) {
      for (int t = 0; t < 9; ++t) pw[t * C + ch] = static_cast<float>(w[ch * 9 + t] * scale[ch]);
      pb[ch] = static_cast<float>(shift[ch]);
    }
    B2_CUDA(cudaMemcpyAsync(D->w, pw.data(), pw.size() * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(D->bias, pb.data(), pb.size() * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  for (auto& G : c->gates) {
    const int m = G->creal, r = G->cr;
    const float* w1 = ws.get(G->prefix + ".fc1.weight", static_cast<int64_t>(r) * m);
    const float* b1 = ws.get(G->prefix + ".fc1.bias", r);
    const float* w2 = ws.get(G->prefix + ".fc2.weight", static_cast<int64_t>(m) * r);
    const float* b2 = ws.get(G->prefix + ".fc2.bias", m);
    if (!w1 || !b1 || !w2 || !b2) return -1;
    B2_CUDA(cudaMemcpyAsync(G->w1, w1, sizeof(float) * r * m, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(G->b1, b1, sizeof(float) * r, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(G->w2, w2, sizeof(float) * m * r, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(G->b2, b2, sizeof(float) * m, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  c->loaded = true;
  return 0;
}

static int reid_enqueue(b2_reid* c) {
  for (const auto& s : c->steps)
    if (run_step(c, s)) return -1;
  return 0;
}

// crops: host [B,256,128,3] uint8 RGB (already resized); feats: host [B,512] float32
// crops: host RGB uint8; the features go to `feats` (host, or device memory of the context's GPU when to_device)
static int reid_embed_impl(b2_reid* c, const uint8_t* crops_host, int n, float* feats, bool to_device) {
  B2_CHECK(c && crops_host && feats, "b2_reid_embed: null argument");
  B2_CHECK(n >= 1 && n <= c->B, "b2_reid_embed: batch larger than the context was created for");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->loaded, "b2_reid_embed: weights not loaded");
  const size_t per = static_cast<size_t>(c->in_h) * c->in_w * 3;
  const cudaMemcpyKind out_kind = to_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (n < c->B) B2_CUDA(cudaMemsetAsync(c->crops + n * per, 0, (c->B - n) * per, c->stream));
  B2_CUDA(cudaMemcpyAsync(c->crops, crops_host, n * per, cudaMemcpyHostToDevice, c->stream));
  if (!c->graph) {
    if (reid_enqueue(c)) return -1;                 // eager warm-up before the capture
    B2_CUDA(cudaStreamSynchronize(c->stream));
    cudaGraph_t g = nullptr;
    B2_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    const int rc = reid_enqueue(c);
    cudaError_t e = cudaStreamEndCapture(c->stream, &g);
    if (rc) return -1;
    B2_CUDA(e);
    B2_CUDA(cudaGraphInstantiate(&c->graph, g, 0));
    B2_CUDA(cudaGraphDestroy(g));
  }
  B2_CUDA(cudaGraphLaunch(c->graph, c->stream));
  B2_CUDA(cudaMemcpyAsync(feats, c->feats, sizeof(float) * n * c->feat_dim, out_kind, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int b2_reid_embed(b2_reid* c, const uint8_t* crops_host, int n, float* feats_host) {
  return reid_embed_impl(c, crops_host, n, feats_host, false);
}

// The features stay in HBM: `feats_dev` is device memory of the context's GPU (e.g. this camera's slice of the gallery
// buffer that the NCCL all-gather / the peer-memory pair cost of config 5 reads), so a gallery never crosses PCIe.
int b2_reid_embed_dev(b2_reid* c, const uint8_t* crops_host, int n, float* feats_dev) {
  return reid_embed_impl(c, crops_host, n, feats_dev, true);
}

int b2_reid_feat_dim(b2_reid* c) { return c ? c->feat_dim : -1; }

// Stage-addressable activation of the last pass as fp32 NHWC (names: "conv1", "maxpool", "conv2.0", "conv2.0.x1",
// "conv2.0.s0".."s3", "conv2.0.x2", "conv2.1", "conv2", ..., "conv5").
int b2_reid_get_activation(b2_reid* c, const char* name, float* dst, int64_t capacity, int64_t shape[4]) {
  B2_CHECK(c && name && dst && shape, "b2_reid_get_activation: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  auto it = c->named.find(name);
  B2_CHECK(it != c->named.end(), std::string("unknown activation: ") + name);
  const RPlanes& p = it->second;
  shape[0] = p.B; shape[1] = p.H; shape[2] = p.W; shape[3] = p.C;
  const int64_t n = static_cast<int64_t>(p.elems());
  B2_CHECK(capacity >= n * 4, "b2_reid_get_activation: buffer too small");
  float* tmp = nullptr;
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_CUDA(cudaMalloc(&tmp, n * 4));
  if (planes_to_f32(p.hi, p.lo, tmp, n, c->stream)) return -1;
  B2_CUDA(cudaMemcpyAsync(dst, tmp, n * 4, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_CUDA(cudaFree(tmp));
  return 0;
}

int b2_reid_num_launches(b2_reid* c) {
  if (!c) return -1;
  int n = 0;
  for (const auto& s : c->steps) n += s.kind == 4 ? 6 : (s.kind == 6 ? 2 : 1);   // gate = 4 GAP + MLP + sum
  return n;
}

}  // extern "C"
