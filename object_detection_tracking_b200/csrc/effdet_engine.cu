// EfficientDet feature network (BiFPN), class/box nets and post-processing behind the C ABI.
// One b2_effdet = one device = one fixed network input size; the pass is a fixed launch sequence replayed as a
// CUDA graph.  Batch is 1 like the reference wrapper (efficientdet_wrapper.py:304-363 runs one frame per call).
//
// Reference graph: efficientdet_arch.py build_feature_network (:440-505) / build_bifpn_layer (:594-682) /
// resample_feature_map (:105-200) / class_net (:227-282) / box_net (:285-340), then
// efficientdet_wrapper.py add_metric_fn_inputs (:367-474), anchors.py _generate_detections_tf (:399-487) and the
// wrapper's own-level ROIAlign box feature (:265-301).
//
// Every separable conv = depthwise 3x3 kernel (effdet.cu) + pointwise GEMM on the tcgen05 conv kernel with bias,
// folded BatchNorm (eps 1e-3) and swish in the epilogue.  The class/box nets share conv weights across levels but
// not BatchNorm statistics, so each level gets its own folded copy of the pointwise weights.
#include <math.h>
#include <stdio.h>
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

struct EPlanes {
  __half* hi = nullptr;
  __half* lo = nullptr;
  int H = 0, W = 0, C = 0, creal = 0;
  size_t elems() const { return static_cast<size_t>(H) * W * C; }
};

struct EConv {
  std::string wname;      // TF variable of the kernel ([1,1,Cin,Cout] HWIO)
  std::string biasname;
  std::string bnname;     // "" = none
  ConvDesc d;
  ConvWeights w;
  ConvIO io;
  ConvPlan* plan = nullptr;
  int cin_real = 0, cout_real = 0;
  float* w_master = nullptr;   // fp32 copy of the packed weights (projection convs re-scaled by the SE gate per frame)
};

struct EDw {
  std::string wname;      // [3,3,C,1]
  EPlanes in, out;
  float* w = nullptr;     // [9][Cpad]
};

struct ECombine {
  BifpnCombineParams p;
  std::string wnames[3];  // fast-attention scalars
};

// backbone: depthwise KxK + BN + swish
struct EDwBn {
  std::string wname, bnname;
  DwConvParams p;
  float* w = nullptr;
  float* bias = nullptr;
  int creal = 0;
};

// backbone: squeeze-excite whose gate is folded into the projection conv's weights every frame
struct ESe {
  std::string pre;          // ".../blocks_i/se"
  EPlanes x;
  int creal = 0, nr = 0;
  float *partial = nullptr, *r_part = nullptr, *gate = nullptr, *w1 = nullptr, *b1 = nullptr, *w2 = nullptr, *b2 = nullptr;
  float* w_master = nullptr;   // BN-folded projection weights [Cout_pad][K] fp32
  EConv* proj = nullptr;
};

struct EStep { int kind, idx; };   // 0 conv, 1 depthwise, 2 combine, 3 backbone depthwise, 4 squeeze-excite, 5 stem im2col

struct F32Out { float* p = nullptr; int H = 0, W = 0, ld = 0, creal = 0; };

int pad64(int c) { return (c + 63) / 64 * 64; }
int pad16(int c) { return (c + 15) / 16 * 16; }

}  // namespace

struct b2_effdet {
  b2_effdet_config cfg;
  int device = 0, num_sms = 148;
  bool split = true;
  int F = 0, Fp = 0, nlev = 0, na = 0;
  int fh[8] = {0}, fw[8] = {0};               // feature size per level (index = level)
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  std::vector<std::unique_ptr<EConv>> convs;
  std::vector<std::unique_ptr<EDw>> dws;
  std::vector<std::unique_ptr<ECombine>> combines;
  std::map<std::string, float*> dw_shared;    // depthwise kernels shared across levels
  std::vector<std::unique_ptr<EDwBn>> dwbns;
  std::vector<std::unique_ptr<ESe>> ses;
  std::vector<EStep> steps;          // feature network + heads
  std::vector<EStep> bb_steps;       // backbone (only when cfg.backbone >= 0)
  std::string bb_name;
  float* image = nullptr;            // [H][W][3] fp32, pre-processed network input
  uint8_t* frame = nullptr;          // device copy of the caller's BGR frame
  size_t frame_cap = 0;
  EPlanes stem_cols;
  cudaGraphExec_t graph_full = nullptr;
  std::map<std::string, EPlanes> named;
  std::map<std::string, F32Out> named_f32;
  EPlanes backbone[3];
  EPlanes fpn_out[5];
  F32Out cls_out[5], box_out[5];
  EffdetPostParams post;
  LevelRoiFeatParams roi;
  float* scale_dev = nullptr;
  float4* out_boxes = nullptr;
  float* out_scores = nullptr;
  int *out_classes = nullptr, *out_levels = nullptr, *out_count = nullptr;
  float* out_feat = nullptr;
  cudaGraphExec_t graph = nullptr;
  bool loaded = false;
  bool building_backbone = false;

  template <typename T>
  T* alloc(size_t n) {
    void* p = nullptr;
    if (cudaMalloc(&p, n * sizeof(T) + 256) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, n * sizeof(T) + 256);
    allocs.push_back(p);
    return static_cast<T*>(p);
  }
  EPlanes planes(int h, int w, int c, int creal) {
    EPlanes p;
    p.H = h; p.W = w; p.C = c; p.creal = creal;
    p.hi = alloc<__half>(p.elems());
    p.lo = split ? alloc<__half>(p.elems()) : nullptr;
    return p;
  }
};

namespace {

// pointwise conv in -> out (planes) or -> fp32 [H*W][ldc32]; act: 0 none, 2 swish
EConv* add_pw(b2_effdet* c, const std::string& wname, const std::string& biasname, const std::string& bn, const EPlanes& in,
              const EPlanes& out, int cout_real, int act, float* out_f32 = nullptr, int ldc32 = 0) {
  std::unique_ptr<EConv> L(new EConv());
  L->wname = wname; L->biasname = biasname; L->bnname = bn;
  L->cin_real = in.creal; L->cout_real = cout_real;
  ConvDesc& d = L->d;
  d.B = 1; d.in_H = in.H; d.in_W = in.W; d.Cin = in.C; d.in_pitch_H = in.H; d.in_pitch_W = in.W; d.in_ld = in.C;
  d.Cout = cout_real; d.relu = act;
  // chunked re-accumulation (conv_tc ACC) on every layer with more than one K-block.  Round 1 switched it off up to
  // K = 512 for speed; at D7 depth (EfficientNet-b6: 45 blocks, then 8 BiFPN cells and 5-deep heads at 1536^2) the
  // truncation bias of up to 32 tensor-core accumulation steps per layer then compounds to 3e-5 relative on c5 -- six
  // times the rounding noise of a float32 evaluation -- and boxes leave the 1e-3 px bar.
  d.acc_kb = 0;   // the kernel's default chunk (one K-block)
  d.out_H = in.H; d.out_W = in.W; d.ldc = out_f32 ? ldc32 : out.C;
  L->w.Cout_pad = pad16(cout_real);
  L->w.K = in.C;
  L->w.w_hi = c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K);
  L->w.w_lo = c->split ? c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K) : nullptr;
  L->w.bias = c->alloc<float>(L->w.Cout_pad);
  L->io.in_hi = in.hi; L->io.in_lo = in.lo; L->io.out_hi = out.hi; L->io.out_lo = out.lo; L->io.out_f32 = out_f32;
  EConv* raw = L.get();
  (c->building_backbone ? c->bb_steps : c->steps).push_back({0, static_cast<int>(c->convs.size())});
  c->convs.push_back(std::move(L));
  return raw;
}

void add_dw(b2_effdet* c, const std::string& wname, const EPlanes& in, const EPlanes& out) {
  std::unique_ptr<EDw> D(new EDw());
  D->wname = wname; D->in = in; D->out = out;
  auto it = c->dw_shared.find(wname);
  if (it == c->dw_shared.end()) {
    D->w = c->alloc<float>(9 * static_cast<size_t>(in.C));
    c->dw_shared[wname] = D->w;
  } else {
    D->w = it->second;
  }
  c->steps.push_back({1, static_cast<int>(c->dws.size())});
  c->dws.push_back(std::move(D));
}

int set_input(BifpnInput& bi, const EPlanes& src, int th, int tw) {
  bi.hi = src.hi; bi.lo = src.lo; bi.H = src.H; bi.W = src.W; bi.pad_t = bi.pad_l = 0; bi.weight = 1.f;
  if (src.H == th && src.W == tw) {
    bi.mode = 0;
  } else if (src.H > th && src.W > tw) {
    B2_CHECK((src.H - 1) / th + 1 == 2 && (src.W - 1) / tw + 1 == 2, "effdet: only stride-2 downsampling between levels");
    const int ph = (th - 1) * 2 + 3 - src.H, pw = (tw - 1) * 2 + 3 - src.W;
    bi.mode = 1;
    bi.pad_t = (ph > 0 ? ph : 0) / 2;
    bi.pad_l = (pw > 0 ? pw : 0) / 2;
  } else {
    B2_CHECK(src.H * 2 == th && src.W * 2 == tw, "effdet: only exact 2x nearest upsampling between levels");
    bi.mode = 2;
  }
  return 0;
}

// resample_feature_map's optional 1x1 conv + BN (at the source resolution), arch.py:131-146
EPlanes maybe_1x1(b2_effdet* c, const EPlanes& src, const std::string& name) {
  if (src.creal == c->F) return src;
  EPlanes t = c->planes(src.H, src.W, c->Fp, c->F);
  add_pw(c, name + "/conv2d/kernel", name + "/conv2d/bias", name + "/bn", src, t, c->F, 0);
  return t;
}

int add_pool(b2_effdet* c, const EPlanes& src, const EPlanes& dst) {
  std::unique_ptr<ECombine> K(new ECombine());
  memset(&K->p, 0, sizeof(K->p));
  if (set_input(K->p.in[0], src, dst.H, dst.W)) return -1;
  K->p.n_in = 1; K->p.B = 1; K->p.Ho = dst.H; K->p.Wo = dst.W; K->p.C = dst.C;
  K->p.weighted = 0; K->p.denom = 1.f; K->p.swish = 0;
  K->p.out_hi = dst.hi; K->p.out_lo = dst.lo;
  c->steps.push_back({2, static_cast<int>(c->combines.size())});
  c->combines.push_back(std::move(K));
  return 0;
}


struct BlockSpec { int kernel, stride, expand, cin, cout; };

int round_filters(double filters, double width) {
  filters *= width;
  int nf = static_cast<int>(filters + 4.0) / 8 * 8;      // efficientnet_model.py:137-151, divisor 8
  if (nf < 8) nf = 8;
  if (nf < 0.9 * filters) nf += 8;
  return nf;
}

void same_pad(int n, int k, int s, int* out, int* before) {
  *out = (n + s - 1) / s;
  const int total = (*out - 1) * s + k - n;
  *before = (total > 0 ? total : 0) / 2;
}

// EfficientNet-b{0..7} trunk up to reduction_5 (efficientnet_model.py:504-704); endpoints land in c->backbone[0..2]
int build_backbone(b2_effdet* c) {
  static const double kWidth[8] = {1.0, 1.0, 1.1, 1.2, 1.4, 1.6, 1.8, 2.0};
  static const double kDepth[8] = {1.0, 1.1, 1.2, 1.4, 1.8, 2.2, 2.6, 3.1};
  static const int kStage[7][6] = {{1, 3, 1, 1, 32, 16}, {2, 3, 2, 6, 16, 24}, {2, 5, 2, 6, 24, 40}, {3, 3, 2, 6, 40, 80},
                                   {3, 5, 1, 6, 80, 112}, {4, 5, 2, 6, 112, 192}, {1, 3, 1, 6, 192, 320}};
  const b2_effdet_config& g = c->cfg;
  B2_CHECK(g.backbone >= 0 && g.backbone <= 7, "effdet: backbone must be efficientnet-b0..b7");
  const double width = kWidth[g.backbone], depth = kDepth[g.backbone];
  c->bb_name = "efficientnet-b" + std::to_string(g.backbone);
  std::vector<BlockSpec> blocks;
  for (const auto& st : kStage) {
    const int rep = static_cast<int>(ceil(depth * st[0])), ci = round_filters(st[4], width), co = round_filters(st[5], width);
    blocks.push_back({st[1], st[2], st[3], ci, co});
    for (int r = 1; r < rep; ++r) blocks.push_back({st[1], 1, st[3], co, co});
  }
  c->building_backbone = true;
  const int H = g.image_h, W = g.image_w;
  c->image = c->alloc<float>(static_cast<size_t>(H) * W * 3);
  // stem: 3x3/2 SAME as a 1x1 conv over im2col-packed pixels (27 live of 64 operand channels)
  int h = 0, w = 0, pt = 0, pl = 0;
  same_pad(H, 3, 2, &h, &pt);
  same_pad(W, 3, 2, &w, &pl);
  c->stem_cols = c->planes(h, w, 64, 27);
  c->bb_steps.push_back({5, pt * 65536 + pl});
  const int stem_c = round_filters(32, width);
  EPlanes x = c->planes(h, w, pad64(stem_c), stem_c);
  add_pw(c, c->bb_name + "/stem/conv2d/kernel", "", c->bb_name + "/stem/tpu_batch_normalization", c->stem_cols, x, stem_c, 2);
  c->named["stem"] = x;
  int reduction = 0;   // reduction_k closes when the next block strides or at the last block (Model.call :644-668)
  for (size_t i = 0; i < blocks.size(); ++i) {
    const BlockSpec& b = blocks[i];
    const std::string pre = c->bb_name + "/blocks_" + std::to_string(i);
    B2_CHECK(x.creal == b.cin, "effdet backbone: channel bookkeeping mismatch");
    const int mid = b.cin * b.expand;
    EPlanes e = x;
    std::string proj = "conv2d";
    if (b.expand != 1) {
      e = c->planes(x.H, x.W, pad64(mid), mid);
      add_pw(c, pre + "/conv2d/kernel", "", pre + "/tpu_batch_normalization", x, e, mid, 2);
      proj = "conv2d_1";
    }
    std::unique_ptr<EDwBn> D(new EDwBn());
    int ho = 0, wo = 0, dpt = 0, dpl = 0;
    same_pad(e.H, b.kernel, b.stride, &ho, &dpt);
    same_pad(e.W, b.kernel, b.stride, &wo, &dpl);
    EPlanes d = c->planes(ho, wo, e.C, mid);
    D->wname = pre + "/depthwise_conv2d/depthwise_kernel"; D->bnname = pre + "/tpu_batch_normalization_1"; D->creal = mid;
    D->w = c->alloc<float>(static_cast<size_t>(b.kernel) * b.kernel * e.C);
    D->bias = c->alloc<float>(e.C);
    D->p = DwConvParams{e.hi, e.lo, e.H, e.W, e.C, b.kernel, b.stride, dpt, dpl, ho, wo, D->w, D->bias, d.hi, d.lo};
    c->bb_steps.push_back({3, static_cast<int>(c->dwbns.size())});
    c->dwbns.push_back(std::move(D));
    // squeeze-excite (se_ratio 0.25 of the block's input filters)
    std::unique_ptr<ESe> S(new ESe());
    S->pre = pre + "/se"; S->x = d; S->creal = mid; S->nr = b.cin / 4 > 1 ? b.cin / 4 : 1;
    S->partial = c->alloc<float>(static_cast<size_t>(se_chunks(ho * wo)) * d.C);
    S->gate = c->alloc<float>(d.C);
    S->r_part = c->alloc<float>(static_cast<size_t>(se_fc1_parts()) * se_max_nr());
    S->w1 = c->alloc<float>(static_cast<size_t>(mid) * S->nr); S->b1 = c->alloc<float>(S->nr);
    S->w2 = c->alloc<float>(static_cast<size_t>(S->nr) * mid); S->b2 = c->alloc<float>(mid);
    ESe* se = S.get();
    c->bb_steps.push_back({4, static_cast<int>(c->ses.size())});
    c->ses.push_back(std::move(S));
    // projection (+ identity skip when the block keeps shape, efficientnet_model.py:381-390)
    EPlanes y = c->planes(ho, wo, pad64(b.cout), b.cout);
    EConv* P = add_pw(c, pre + "/" + proj + "/kernel", "", pre + "/tpu_batch_normalization_2", d, y, b.cout, 0);
    if (b.stride == 1 && b.cin == b.cout) {
      P->d.res_H = x.H; P->d.res_W = x.W; P->d.ldr = x.C;
      P->io.res_hi = x.hi; P->io.res_lo = x.lo;
    }
    se->proj = P;
    se->w_master = c->alloc<float>(static_cast<size_t>(P->w.Cout_pad) * P->w.K);
    P->w_master = se->w_master;
    x = y;
    c->named["block_" + std::to_string(i)] = x;
    if (i + 1 == blocks.size() || blocks[i + 1].stride > 1) {
      const int lvl = ++reduction;
      if (lvl >= 3 && lvl <= 5) {
        B2_CHECK(x.creal == g.backbone_channels[lvl - 3], "effdet: backbone_channels do not match the backbone's endpoints");
        B2_CHECK(x.H == c->fh[lvl] && x.W == c->fw[lvl], "effdet: backbone endpoint size mismatch");
        c->backbone[lvl - 3] = x;
      }
    }
  }
  c->building_backbone = false;
  return 0;
}

int build(b2_effdet* c) {
  const b2_effdet_config& g = c->cfg;
  B2_CHECK(g.min_level == 3 && g.max_level == 7, "effdet: levels 3..7 only (the reference's configuration)");
  B2_CHECK(g.image_h % 128 == 0 && g.image_w % 128 == 0, "effdet: network input size must be divisible by 128");
  c->F = g.fpn_num_filters; c->Fp = pad64(c->F); c->nlev = 5;
  c->na = g.num_scales * g.num_aspects;
  B2_CHECK(c->na >= 1 && c->na <= 9, "effdet: at most 9 anchors per cell");
  {
    int h = g.image_h, w = g.image_w;
    for (int l = 1; l <= 7; ++l) {
      h = (h - 1) / 2 + 1; w = (w - 1) / 2 + 1;
      c->fh[l] = h; c->fw[l] = w;
    }
  }
  std::vector<EPlanes> feats;
  if (g.backbone >= 0 && build_backbone(c)) return -1;
  for (int i = 0; i < 3; ++i) {
    const int cr = g.backbone_channels[i];
    if (g.backbone < 0) c->backbone[i] = c->planes(c->fh[3 + i], c->fw[3 + i], pad64(cr), cr);
    feats.push_back(c->backbone[i]);
    c->named["c" + std::to_string(3 + i)] = c->backbone[i];
  }
  // P6, P7 (arch.py:464-480): resample_p6 = [conv1x1 + BN] + max-pool, resample_p7 = max-pool
  for (int level = 6; level <= 7; ++level) {
    EPlanes src = maybe_1x1(c, feats.back(), "resample_p" + std::to_string(level));
    EPlanes dst = c->planes(c->fh[level], c->fw[level], c->Fp, c->F);
    if (add_pool(c, src, dst)) return -1;
    feats.push_back(dst);
    c->named["p" + std::to_string(level) + "_in"] = dst;
  }
  static const int node_level[8] = {6, 5, 4, 3, 4, 5, 6, 7};
  static const int node_in[8][3] = {{3, 4, -1}, {2, 5, -1}, {1, 6, -1}, {0, 7, -1}, {1, 7, 8}, {2, 6, 9}, {3, 5, 10}, {4, 11, -1}};
  for (int rep = 0; rep < g.fpn_cell_repeats; ++rep) {
    for (int i = 0; i < 8; ++i) {
      const int lvl = node_level[i], th = c->fh[lvl], tw = c->fw[lvl];
      const std::string pre = "fpn_cells/cell_" + std::to_string(rep) + "/fnode" + std::to_string(i);
      const int nfeats = static_cast<int>(feats.size());
      std::unique_ptr<ECombine> K(new ECombine());
      memset(&K->p, 0, sizeof(K->p));
      int n = 0;
      for (int idx = 0; idx < 3 && node_in[i][idx] >= 0; ++idx, ++n) {
        const int o = node_in[i][idx];
        EPlanes src = maybe_1x1(c, feats[o], pre + "/resample_" + std::to_string(idx) + "_" + std::to_string(o) + "_" +
                                                 std::to_string(nfeats));
        if (set_input(K->p.in[idx], src, th, tw)) return -1;
        K->wnames[idx] = pre + "/WSM" + (idx == 0 ? std::string() : "_" + std::to_string(idx));
      }
      EPlanes comb = c->planes(th, tw, c->Fp, c->F);
      K->p.n_in = n; K->p.B = 1; K->p.Ho = th; K->p.Wo = tw; K->p.C = c->Fp;
      K->p.weighted = g.fpn_weight_method == 1; K->p.denom = 1.f; K->p.swish = 1;
      K->p.out_hi = comb.hi; K->p.out_lo = comb.lo;
      c->steps.push_back({2, static_cast<int>(c->combines.size())});
      c->combines.push_back(std::move(K));
      const std::string op = pre + "/op_after_combine" + std::to_string(nfeats);
      EPlanes t = c->planes(th, tw, c->Fp, c->F);
      add_dw(c, op + "/conv/depthwise_kernel", comb, t);
      EPlanes node = c->planes(th, tw, c->Fp, c->F);
      add_pw(c, op + "/conv/pointwise_kernel", op + "/conv/bias", op + "/bn", t, node, c->F, 0);
      feats.push_back(node);
    }
    // the cell's outputs: the last node of every level (arch.py:495-503)
    std::vector<EPlanes> next(5);
    for (int l = 3; l <= 7; ++l)
      for (int i = 7; i >= 0; --i)
        if (node_level[i] == l) { next[l - 3] = feats[feats.size() - 8 + i]; break; }
    feats = next;
  }
  for (int l = 0; l < 5; ++l) {
    c->fpn_out[l] = feats[l];
    c->named["fpn" + std::to_string(l + 3)] = feats[l];
  }
  // class / box nets (arch.py:227-340)
  const int ncls = c->na * g.num_classes, nbox = c->na * 4;
  for (int l = 0; l < 5; ++l) {
    const int level = l + 3, h = c->fh[level], w = c->fw[level];
    for (int kind = 0; kind < 2; ++kind) {
      const std::string kn = kind == 0 ? "class" : "box";
      EPlanes x = c->fpn_out[l];
      EPlanes ping = c->planes(h, w, c->Fp, c->F), pong = c->planes(h, w, c->Fp, c->F), t = c->planes(h, w, c->Fp, c->F);
      for (int i = 0; i < g.box_class_repeats; ++i) {
        const std::string nm = kn + "_net/" + kn + "-" + std::to_string(i);
        add_dw(c, nm + "/depthwise_kernel", x, t);
        EPlanes y = (i & 1) ? pong : ping;
        add_pw(c, nm + "/pointwise_kernel", nm + "/bias", nm + "-bn-" + std::to_string(level), t, y, c->F, 2);
        x = y;
      }
      const std::string nm = kn + "_net/" + kn + "-predict";
      add_dw(c, nm + "/depthwise_kernel", x, t);
      F32Out o;
      o.creal = kind == 0 ? ncls : nbox;
      o.ld = pad16(o.creal); o.H = h; o.W = w;
      o.p = c->alloc<float>(static_cast<size_t>(h) * w * o.ld);
      add_pw(c, nm + "/pointwise_kernel", nm + "/bias", "", t, EPlanes(), o.creal, 0, o.p, o.ld);
      (kind == 0 ? c->cls_out[l] : c->box_out[l]) = o;
      c->named_f32[(kind == 0 ? "cls" : "box") + std::to_string(level)] = o;
    }
  }
  // post-processing state
  EffdetPostParams& p = c->post;
  memset(&p, 0, sizeof(p));
  unsigned long long off = 0;
  for (int l = 0; l < 5; ++l) {
    const int level = l + 3;
    p.logits[l] = c->cls_out[l].p; p.boxes[l] = c->box_out[l].p;
    p.ld[l] = c->cls_out[l].ld; p.ldb[l] = c->box_out[l].ld; p.w[l] = c->fw[level];
    p.level_off[l] = off;
    off += static_cast<unsigned long long>(c->fh[level]) * c->fw[level] * ncls;
    // anchors.py:216-257: stride = image / feature size; octave scale 2^(o / num_scales); aspect (x, y) multipliers
    p.stride_y[l] = static_cast<double>(g.image_h) / c->fh[level];
    p.stride_x[l] = static_cast<double>(g.image_w) / c->fw[level];
    int a = 0;
    for (int o = 0; o < g.num_scales; ++o)
      for (int r = 0; r < g.num_aspects; ++r, ++a) {
        const double oct = pow(2.0, o / static_cast<double>(g.num_scales));
        const double sx = static_cast<double>(g.anchor_scale) * p.stride_x[l] * oct;
        const double sy = static_cast<double>(g.anchor_scale) * p.stride_y[l] * oct;
        p.half_x[l][a] = sx * static_cast<double>(g.aspect_ratios[r][0]) / 2.0;
        p.half_y[l][a] = sy * static_cast<double>(g.aspect_ratios[r][1]) / 2.0;
      }
  }
  p.level_off[5] = off; p.total = off;
  p.n_levels = 5; p.anchors = c->na; p.num_classes = g.num_classes; p.min_level = 3;
  p.k = g.max_detection_topk; p.max_out = g.result_per_im;
  B2_CHECK(p.k >= 1 && p.k <= 8192, "effdet: max_detection_topk must be in [1, 8192]");
  p.score_thresh = g.result_score_thres; p.nms_thr = g.nms_iou_threshold;
  p.hist = c->alloc<unsigned int>(256);
  p.state = c->alloc<uint32_t>(8);
  p.cand = c->alloc<unsigned long long>(p.k);
  p.ties = c->alloc<unsigned long long>(p.k);
  p.tie_cnt = c->alloc<unsigned int>(effdet_topk_blocks());
  p.tie_off = c->alloc<unsigned int>(effdet_topk_blocks());
  p.cand_box = c->alloc<float4>(p.k);
  p.cand_score = c->alloc<float>(p.k);
  p.cand_cls = c->alloc<int>(p.k);
  p.cand_lvl = c->alloc<int>(p.k);
  p.mask = c->alloc<unsigned long long>(static_cast<size_t>(p.k) * ((p.k + 63) / 64));
  c->out_boxes = c->alloc<float4>(p.max_out);
  c->out_scores = c->alloc<float>(p.max_out);
  c->out_classes = c->alloc<int>(p.max_out);
  c->out_levels = c->alloc<int>(p.max_out);
  c->out_count = c->alloc<int>(1);
  c->out_feat = c->alloc<float>(static_cast<size_t>(p.max_out) * c->F);
  c->scale_dev = c->alloc<float>(1);
  p.out_boxes = c->out_boxes; p.out_scores = c->out_scores; p.out_classes = c->out_classes;
  p.out_levels = c->out_levels; p.out_count = c->out_count;
  LevelRoiFeatParams& r = c->roi;
  memset(&r, 0, sizeof(r));
  for (int l = 0; l < 5; ++l) {
    r.feat_hi[l] = c->fpn_out[l].hi; r.feat_lo[l] = c->fpn_out[l].lo;
    r.H[l] = c->fpn_out[l].H; r.W[l] = c->fpn_out[l].W;
    r.inv_stride[l] = 1.0f / static_cast<float>(1 << (l + 3));
  }
  r.C = c->Fp; r.Creal = c->F; r.min_level = 3; r.max_out = p.max_out;
  r.boxes = c->out_boxes; r.levels = c->out_levels; r.count = c->out_count; r.out = c->out_feat;
  for (auto& L : c->convs) {
    L->plan = conv_tc_plan_create(L->d, L->w, L->io, c->split, c->num_sms);
    if (!L->plan) {
      set_error("effdet plan for " + L->wname + ": " + last_error());
      return -1;
    }
  }
  return 0;
}

int run_step(b2_effdet* c, const EStep& s) {
  cudaStream_t st = c->stream;
  switch (s.kind) {
    case 0: return conv_tc_launch(c->convs[s.idx]->plan, st);
    case 1: {
      const EDw* d = c->dws[s.idx].get();
      return dw3x3_plain_launch(d->in.hi, d->in.lo, 1, d->in.H, d->in.W, d->in.C, d->w, d->out.hi, d->out.lo, st);
    }
    case 2: return bifpn_combine_launch(c->combines[s.idx]->p, st);
    case 3: return dwconv_bn_swish_launch(c->dwbns[s.idx]->p, st);
    case 4: {
      const ESe* e = c->ses[s.idx].get();
      return se_gate_launch(e->x.hi, e->x.lo, e->x.H * e->x.W, e->x.C, e->creal, e->nr, e->partial, e->r_part, e->w1, e->b1,
                            e->w2, e->b2, e->gate, e->w_master, e->proj->w.Cout_pad, e->proj->w.w_hi, e->proj->w.w_lo, st);
    }
    case 5:
      return stem_im2col_launch(c->image, c->cfg.image_h, c->cfg.image_w, c->stem_cols.H, c->stem_cols.W, s.idx / 65536,
                                s.idx % 65536, c->stem_cols.hi, c->stem_cols.lo, st);
  }
  return -1;
}

int enqueue(b2_effdet* c, bool with_backbone) {
  cudaStream_t st = c->stream;
  if (with_backbone)
    for (const EStep& s : c->bb_steps)
      if (run_step(c, s)) return -1;
  for (const EStep& s : c->steps)
    if (run_step(c, s)) return -1;
  if (effdet_post_launch(c->post, c->scale_dev, st)) return -1;
  return level_roi_feat_launch(c->roi, st);
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


int launch_and_fetch(b2_effdet* c, bool full, float image_scale, float* boxes, float* scores, int* classes, int* levels,
                     float* box_feat, int* count) {
  B2_CUDA(cudaMemcpyAsync(c->scale_dev, &image_scale, 4, cudaMemcpyHostToDevice, c->stream));
  cudaGraphExec_t& graph = full ? c->graph_full : c->graph;
  if (!graph) {
    if (enqueue(c, full)) return -1;           // eager warm-up before the capture
    B2_CUDA(cudaStreamSynchronize(c->stream));
    cudaGraph_t g = nullptr;
    B2_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
    const int rc = enqueue(c, full);
    cudaError_t e = cudaStreamEndCapture(c->stream, &g);
    if (rc) return -1;
    B2_CUDA(e);
    B2_CUDA(cudaGraphInstantiate(&graph, g, 0));
    B2_CUDA(cudaGraphDestroy(g));
  }
  B2_CUDA(cudaGraphLaunch(graph, c->stream));
  const int m = c->post.max_out;
  B2_CUDA(cudaMemcpyAsync(boxes, c->out_boxes, sizeof(float) * 4 * m, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaMemcpyAsync(scores, c->out_scores, sizeof(float) * m, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaMemcpyAsync(classes, c->out_classes, sizeof(int) * m, cudaMemcpyDeviceToHost, c->stream));
  if (levels) B2_CUDA(cudaMemcpyAsync(levels, c->out_levels, sizeof(int) * m, cudaMemcpyDeviceToHost, c->stream));
  if (box_feat) B2_CUDA(cudaMemcpyAsync(box_feat, c->out_feat, sizeof(float) * m * c->F, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaMemcpyAsync(count, c->out_count, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

}  // namespace

extern "C" {

int b2_effdet_create(b2_effdet** out, const b2_effdet_config* cfg, int device) {
  B2_CHECK(out && cfg, "b2_effdet_create: null argument");
  *out = nullptr;
  B2_CUDA(cudaSetDevice(device));
  if (conv_tc_init()) return -1;
  std::unique_ptr<b2_effdet> c(new b2_effdet());
  c->cfg = *cfg; c->device = device; c->split = cfg->precision == 1;
  cudaDeviceProp prop;
  B2_CUDA(cudaGetDeviceProperties(&prop, device));
  B2_CHECK(prop.major == 10, "b2_effdet_create: this library is built for sm_100a (B200) only");
  c->num_sms = prop.multiProcessorCount;
  B2_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  if (build(c.get())) { b2_effdet_destroy(c.release()); return -1; }
  B2_CUDA(cudaDeviceSynchronize());
  *out = c.release();
  return 0;
}

void b2_effdet_destroy(b2_effdet* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (c->graph) cudaGraphExecDestroy(c->graph);
  if (c->graph_full) cudaGraphExecDestroy(c->graph_full);
  for (auto& L : c->convs) if (L->plan) conv_tc_plan_destroy(L->plan);
  for (void* p : c->allocs) cudaFree(p);
  if (c->frame) cudaFree(c->frame);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

// TF checkpoint variables of the feature network and heads (names as in efficientdet_arch.py, kernels HWIO)
int b2_effdet_load_weights(b2_effdet* c, const char* const* names, const float* const* data, const int64_t* numel, int n) {
  B2_CHECK(c && names && data && numel, "b2_effdet_load_weights: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  WS ws;
  for (int i = 0; i < n; ++i) ws.m[names[i]] = std::make_pair(data[i], numel[i]);
  for (auto& L : c->convs) {
    const int K = L->w.K, Cp = L->w.Cout_pad, co = L->cout_real, ci = L->cin_real;
    const float* w = ws.get(L->wname, static_cast<int64_t>(ci) * co);
    const float* b = L->biasname.empty() ? nullptr : ws.get(L->biasname, co);   // backbone convs have no bias
    if (!w || (!b && !L->biasname.empty())) return -1;
    std::vector<double> scale(co, 1.0), shift(co, 0.0);
    if (!L->bnname.empty()) {
      const float* ga = ws.get(L->bnname + "/gamma", co);
      const float* be = ws.get(L->bnname + "/beta", co);
      const float* mm = ws.get(L->bnname + "/moving_mean", co);
      const float* mv = ws.get(L->bnname + "/moving_variance", co);
      if (!ga || !be || !mm || !mv) return -1;
      for (int o = 0; o < co; ++o) {
        scale[o] = static_cast<double>(ga[o]) / sqrt(static_cast<double>(mv[o]) + 1e-3);   // utils.py:252-303 eps
        shift[o] = static_cast<double>(be[o]) - static_cast<double>(mm[o]) * scale[o];
      }
    }
    std::vector<float> packed(static_cast<size_t>(Cp) * K, 0.f), bias(Cp, 0.f);
    for (int o = 0; o < co; ++o) {
      for (int i = 0; i < ci; ++i) packed[static_cast<size_t>(o) * K + i] = static_cast<float>(w[static_cast<size_t>(i) * co + o] * scale[o]);
      bias[o] = static_cast<float>((b ? static_cast<double>(b[o]) : 0.0) * scale[o] + shift[o]);
    }
    float* tmp = nullptr;
    B2_CUDA(cudaMalloc(&tmp, packed.size() * 4));
    B2_CUDA(cudaMemcpyAsync(tmp, packed.data(), packed.size() * 4, cudaMemcpyHostToDevice, c->stream));
    if (f32_to_planes(tmp, L->w.w_hi, L->w.w_lo, packed.size(), c->stream)) return -1;
    if (L->w_master) B2_CUDA(cudaMemcpyAsync(L->w_master, tmp, packed.size() * 4, cudaMemcpyDeviceToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(L->w.bias, bias.data(), bias.size() * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    B2_CUDA(cudaFree(tmp));
  }
  for (auto& kv : c->dw_shared) {
    const int C = c->Fp, cr = c->F;
    const float* w = ws.get(kv.first, static_cast<int64_t>(9) * cr);   // [3,3,C,1]
    if (!w) return -1;
    std::vector<float> pw(9 * static_cast<size_t>(C), 0.f);
    for (int t = 0; t < 9; ++t)
      for (int ch = 0; ch < cr; ++ch) pw[static_cast<size_t>(t) * C + ch] = w[t * cr + ch];
    B2_CUDA(cudaMemcpyAsync(kv.second, pw.data(), pw.size() * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  for (auto& D : c->dwbns) {
    const int C = D->p.C, cr = D->creal, kk = D->p.K * D->p.K;
    const float* w = ws.get(D->wname, static_cast<int64_t>(kk) * cr);   // [K,K,C,1]
    const float* ga = ws.get(D->bnname + "/gamma", cr);
    const float* be = ws.get(D->bnname + "/beta", cr);
    const float* mm = ws.get(D->bnname + "/moving_mean", cr);
    const float* mv = ws.get(D->bnname + "/moving_variance", cr);
    if (!w || !ga || !be || !mm || !mv) return -1;
    std::vector<float> pw(static_cast<size_t>(kk) * C, 0.f), pb(C, 0.f);
    for (int ch = 0; ch < cr; ++ch) {
      const double sc = static_cast<double>(ga[ch]) / sqrt(static_cast<double>(mv[ch]) + 1e-3);
      for (int t = 0; t < kk; ++t) pw[static_cast<size_t>(t) * C + ch] = static_cast<float>(w[t * cr + ch] * sc);
      pb[ch] = static_cast<float>(static_cast<double>(be[ch]) - static_cast<double>(mm[ch]) * sc);
    }
    B2_CUDA(cudaMemcpyAsync(D->w, pw.data(), pw.size() * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(D->bias, pb.data(), pb.size() * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  for (auto& S : c->ses) {
    const int m = S->creal, r = S->nr;
    const float* w1 = ws.get(S->pre + "/conv2d/kernel", static_cast<int64_t>(m) * r);
    const float* b1 = ws.get(S->pre + "/conv2d/bias", r);
    const float* w2 = ws.get(S->pre + "/conv2d_1/kernel", static_cast<int64_t>(r) * m);
    const float* b2 = ws.get(S->pre + "/conv2d_1/bias", m);
    if (!w1 || !b1 || !w2 || !b2) return -1;
    B2_CUDA(cudaMemcpyAsync(S->w1, w1, sizeof(float) * m * r, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(S->b1, b1, sizeof(float) * r, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(S->w2, w2, sizeof(float) * r * m, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(S->b2, b2, sizeof(float) * m, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  if (c->cfg.fpn_weight_method == 1) {
    for (auto& K : c->combines) {
      if (!K->p.weighted) continue;
      double tot = 0.0;
      float tot32 = 0.f;
      for (int i = 0; i < K->p.n_in; ++i) {
        const float* w = ws.get(K->wnames[i], 1);
        if (!w) return -1;
        const float r = w[0] > 0.f ? w[0] : 0.f;          // tf.nn.relu
        K->p.in[i].weight = r;
        tot32 = i == 0 ? r : tot32 + r;                    // tf.add_n in float32
        tot += r;
      }
      (void)tot;
      K->p.denom = tot32 + 0.0001f;
    }
  }
  c->loaded = true;
  if (c->graph) { cudaGraphExecDestroy(c->graph); c->graph = nullptr; }
  if (c->graph_full) { cudaGraphExecDestroy(c->graph_full); c->graph_full = nullptr; }
  return 0;
}

// Backbone features C3, C4, C5 as host NHWC fp32 ([h,w,c] with the real channel counts) -> detections.
// boxes [max][4] x1 y1 x2 y2 in original-frame pixels (network coords * image_scale), classes 1-based, levels 3..7,
// box_feat [max][fpn_num_filters].  Returns the number of detections in *count (rows beyond it are zero).
int b2_effdet_run_features(b2_effdet* c, const float* c3, const float* c4, const float* c5, float image_scale,
                           float* boxes, float* scores, int* classes, int* levels, float* box_feat, int* count) {
  B2_CHECK(c && c3 && c4 && c5 && boxes && scores && classes && count, "b2_effdet_run_features: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->loaded, "b2_effdet_run_features: weights not loaded");
  const float* src[3] = {c3, c4, c5};
  for (int i = 0; i < 3; ++i) {
    const EPlanes& p = c->backbone[i];
    std::vector<float> padded(p.elems(), 0.f);
    const size_t px = static_cast<size_t>(p.H) * p.W;
    for (size_t q = 0; q < px; ++q) memcpy(&padded[q * p.C], src[i] + q * p.creal, sizeof(float) * p.creal);
    float* tmp = nullptr;
    B2_CUDA(cudaMalloc(&tmp, padded.size() * 4));
    B2_CUDA(cudaMemcpyAsync(tmp, padded.data(), padded.size() * 4, cudaMemcpyHostToDevice, c->stream));
    if (f32_to_planes(tmp, p.hi, p.lo, padded.size(), c->stream)) return -1;
    B2_CUDA(cudaStreamSynchronize(c->stream));
    B2_CUDA(cudaFree(tmp));
  }
  return launch_and_fetch(c, false, image_scale, boxes, scores, classes, levels, box_feat, count);
}

// Full per-frame path of the reference wrapper (EfficientDet.build_preprocess + build_model): host BGR uint8 frame
// [h,w,3] -> pre-process (RGB, /255, mean/std, bilinear resize to fit, zero-pad) -> backbone -> BiFPN -> heads ->
// detections scaled back to the frame.  *image_scale_out = image_scale_to_original.
int b2_effdet_detect(b2_effdet* c, const uint8_t* frame_bgr, int h, int w, float* boxes, float* scores, int* classes,
                     int* levels, float* box_feat, int* count, float* image_scale_out) {
  B2_CHECK(c && frame_bgr && boxes && scores && classes && count, "b2_effdet_detect: null argument");
  B2_CHECK(h >= 1 && w >= 1, "b2_effdet_detect: empty frame");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->loaded, "b2_effdet_detect: weights not loaded");
  B2_CHECK(c->cfg.backbone >= 0, "b2_effdet_detect: the context was created without a backbone (use b2_effdet_run_features)");
  const size_t bytes = static_cast<size_t>(h) * w * 3;
  if (bytes > c->frame_cap) {
    if (c->frame) B2_CUDA(cudaFree(c->frame));
    c->frame = nullptr; c->frame_cap = 0;
    B2_CUDA(cudaMalloc(&c->frame, bytes));
    c->frame_cap = bytes;
  }
  // set_scale_factors_to_output_size (dataloader.py:101-113), float32 like the TF graph
  const float sy = static_cast<float>(c->cfg.image_h) / static_cast<float>(h);
  const float sx = static_cast<float>(c->cfg.image_w) / static_cast<float>(w);
  const float scale = sx < sy ? sx : sy;
  int sh = static_cast<int>(static_cast<float>(h) * scale), sw = static_cast<int>(static_cast<float>(w) * scale);
  if (sh > c->cfg.image_h) sh = c->cfg.image_h;
  if (sw > c->cfg.image_w) sw = c->cfg.image_w;
  const float image_scale = 1.0f / scale;
  if (image_scale_out) *image_scale_out = image_scale;
  B2_CUDA(cudaMemcpyAsync(c->frame, frame_bgr, bytes, cudaMemcpyHostToDevice, c->stream));
  if (effnet_preprocess_launch(c->frame, h, w, sh, sw, c->image, c->cfg.image_h, c->cfg.image_w, c->stream)) return -1;
  return launch_and_fetch(c, true, image_scale, boxes, scores, classes, levels, box_feat, count);
}

// Stage-addressable tensors of the last pass as fp32 NHWC: "fpn3".."fpn7" (BiFPN outputs, channel-padded),
// "cls3".."cls7" / "box3".."box7" (head outputs, row stride = shape[3] >= real columns).
int b2_effdet_get_stage(b2_effdet* c, const char* name, float* dst, int64_t capacity, int64_t shape[4]) {
  B2_CHECK(c && name && dst && shape, "b2_effdet_get_stage: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  auto f = c->named_f32.find(name);
  if (f != c->named_f32.end()) {
    const F32Out& o = f->second;
    shape[0] = 1; shape[1] = o.H; shape[2] = o.W; shape[3] = o.ld;
    const int64_t n = static_cast<int64_t>(o.H) * o.W * o.ld;
    B2_CHECK(capacity >= n * 4, "b2_effdet_get_stage: buffer too small");
    B2_CUDA(cudaMemcpyAsync(dst, o.p, n * 4, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  }
  if (std::string(name) == "image" && c->image) {
    shape[0] = 1; shape[1] = c->cfg.image_h; shape[2] = c->cfg.image_w; shape[3] = 3;
    const int64_t n = static_cast<int64_t>(c->cfg.image_h) * c->cfg.image_w * 3;
    B2_CHECK(capacity >= n * 4, "b2_effdet_get_stage: buffer too small");
    B2_CUDA(cudaMemcpyAsync(dst, c->image, n * 4, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  }
  auto it = c->named.find(name);
  B2_CHECK(it != c->named.end(), std::string("unknown stage: ") + name);
  const EPlanes& p = it->second;
  shape[0] = 1; shape[1] = p.H; shape[2] = p.W; shape[3] = p.C;
  const int64_t n = static_cast<int64_t>(p.elems());
  B2_CHECK(capacity >= n * 4, "b2_effdet_get_stage: buffer too small");
  float* tmp = nullptr;
  B2_CUDA(cudaMalloc(&tmp, n * 4));
  if (planes_to_f32(p.hi, p.lo, tmp, n, c->stream)) return -1;
  B2_CUDA(cudaMemcpyAsync(dst, tmp, n * 4, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_CUDA(cudaFree(tmp));
  return 0;
}

// Per-step CUDA-event timing of the whole pass (backbone when present, feature network, heads, post-processing, box
// feature), eager launches on the context stream.  ms_out[i] = mean over `reps` of step i; *n_out = number of steps.
int b2_effdet_profile_steps(b2_effdet* c, int reps, float* ms_out, int cap, int* n_out) {
  B2_CHECK(c && ms_out && n_out && reps >= 1, "b2_effdet_profile_steps: bad argument");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->loaded, "b2_effdet_profile_steps: weights not loaded");
  std::vector<EStep> all(c->bb_steps);
  all.insert(all.end(), c->steps.begin(), c->steps.end());
  const int n = static_cast<int>(all.size()) + 2;
  B2_CHECK(cap >= n, "b2_effdet_profile_steps: buffer too small");
  std::vector<cudaEvent_t> ev(2 * n);
  for (auto& e : ev) B2_CUDA(cudaEventCreate(&e));
  std::vector<double> acc(n, 0.0);
  for (int r = 0; r < reps; ++r) {
    for (int i = 0; i < n; ++i) {
      B2_CUDA(cudaEventRecord(ev[2 * i], c->stream));
      int rc = 0;
      if (i < n - 2) rc = run_step(c, all[i]);
      else if (i == n - 2) rc = effdet_post_launch(c->post, c->scale_dev, c->stream);
      else rc = level_roi_feat_launch(c->roi, c->stream);
      if (rc) return -1;
      B2_CUDA(cudaEventRecord(ev[2 * i + 1], c->stream));
    }
    B2_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < n; ++i) {
      float ms = 0.f;
      B2_CUDA(cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]));
      acc[i] += ms;
    }
  }
  for (int i = 0; i < n; ++i) ms_out[i] = static_cast<float>(acc[i] / reps);
  for (auto& e : ev) cudaEventDestroy(e);
  *n_out = n;
  return 0;
}

// Step `idx` of b2_effdet_profile_steps: kind (0 pointwise conv on the tensor cores, 1 head/BiFPN depthwise, 2 BiFPN
// combine / max-pool, 3 backbone depthwise, 4 squeeze-excite, 5 stem im2col, 6 post-processing, 7 box feature), a
// name, algorithmic FLOPs and HBM bytes (operands once, at the stored precision).
int b2_effdet_step_info(b2_effdet* c, int idx, char* name, int name_cap, double* flops, double* bytes, int* kind) {
  B2_CHECK(c && name && flops && bytes && kind, "b2_effdet_step_info: null argument");
  std::vector<EStep> all(c->bb_steps);
  all.insert(all.end(), c->steps.begin(), c->steps.end());
  const int n = static_cast<int>(all.size()) + 2;
  B2_CHECK(idx >= 0 && idx < n, "b2_effdet_step_info: index out of range");
  const double esz = c->split ? 4.0 : 2.0;
  std::string nm;
  *flops = 0; *bytes = 0;
  if (idx == n - 2) { *kind = 6; nm = "post"; *bytes = static_cast<double>(c->post.total) * 4.0 * 6.0; }
  else if (idx == n - 1) { *kind = 7; nm = "box_feat"; }
  else {
    const EStep& s = all[idx];
    *kind = s.kind;
    if (s.kind == 0) {
      const EConv* L = c->convs[s.idx].get();
      const ConvDesc& d = L->d;
      const double M = static_cast<double>(d.in_H) * d.in_W;
      *flops = 2.0 * M * L->cin_real * L->cout_real;
      *bytes = M * d.Cin * esz + static_cast<double>(L->w.K) * L->w.Cout_pad * esz +
               M * (L->io.out_f32 ? L->w.Cout_pad * 4.0 : d.ldc * esz) + (L->io.res_hi ? M * d.ldr * esz : 0.0);
      nm = L->wname + " [" + std::to_string(d.in_H) + "x" + std::to_string(d.in_W) + "x" + std::to_string(L->cin_real) + "->" +
           std::to_string(L->cout_real) + "]";
    } else if (s.kind == 1) {
      const EDw* D = c->dws[s.idx].get();
      *bytes = 2.0 * static_cast<double>(D->in.elems()) * esz;
      *flops = 18.0 * static_cast<double>(D->in.H) * D->in.W * D->in.creal;
      nm = D->wname;
    } else if (s.kind == 2) {
      const BifpnCombineParams& p = c->combines[s.idx]->p;
      double in = 0;
      for (int i = 0; i < p.n_in; ++i) in += static_cast<double>(p.in[i].H) * p.in[i].W * p.C;
      *bytes = (in + static_cast<double>(p.Ho) * p.Wo * p.C) * esz;
      nm = "combine x" + std::to_string(p.n_in) + " [" + std::to_string(p.Ho) + "x" + std::to_string(p.Wo) + "]";
    } else if (s.kind == 3) {
      const EDwBn* D = c->dwbns[s.idx].get();
      *bytes = (static_cast<double>(D->p.H) * D->p.W + static_cast<double>(D->p.Ho) * D->p.Wo) * D->p.C * esz;
      *flops = 2.0 * D->p.K * D->p.K * static_cast<double>(D->p.Ho) * D->p.Wo * D->creal;
      nm = D->wname + " [" + std::to_string(D->p.H) + "x" + std::to_string(D->p.W) + "x" + std::to_string(D->creal) + " k" +
           std::to_string(D->p.K) + "/" + std::to_string(D->p.stride) + "]";
    } else if (s.kind == 4) {
      const ESe* e = c->ses[s.idx].get();
      *bytes = static_cast<double>(e->x.elems()) * esz + 2.0 * e->proj->w.Cout_pad * e->proj->w.K * 4.0;
      nm = e->pre;
    } else {
      *bytes = static_cast<double>(c->cfg.image_h) * c->cfg.image_w * 3 * 4 + static_cast<double>(c->stem_cols.elems()) * esz;
      nm = "stem_im2col";
    }
  }
  snprintf(name, name_cap, "%s", nm.c_str());
  return 0;
}

int b2_effdet_num_launches(b2_effdet* c) {
  if (!c) return -1;
  int bb = 0;
  for (const EStep& s : c->bb_steps) bb += s.kind == 4 ? 3 : 1;
  if (bb) bb += 1;   // pre-processing
  return bb + static_cast<int>(c->steps.size()) + 15;   // + seed, 4 x (hist, pick), collect, tie scan, tie write, prepare, mask, scan, roi feature
}

}  // extern "C"
