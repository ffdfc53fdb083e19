// libb200det engine: context, weight folding/packing, the static per-frame launch plan, C ABI.
//
// The plan is built once per (batch, H, W): every activation buffer, every TMA tensor map and every
// kernel parameter block is fixed, so one frame is a fixed sequence of ~150 launches that is captured
// into a CUDA graph and replayed.  Graph structure follows Mask_RCNN_FPN.build_forward
// (models.py:488-973); citations at each phase.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200det.h"
#include "common.h"
#include "kernels.h"

namespace b2 {

static thread_local std::string g_err;
void set_error(const std::string& msg) { g_err = msg; }
const char* last_error() { return g_err.c_str(); }

namespace {

__global__ void subsample2_kernel(const __half* __restrict__ in_hi, const __half* __restrict__ in_lo, int B, int H,
                                  int W, int C, __half* __restrict__ out_hi, __half* __restrict__ out_lo, int Ho,
                                  int Wo) {
  const int cvec = C / 8;
  const size_t total = static_cast<size_t>(B) * Ho * Wo * cvec;
  for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int cv = static_cast<int>(idx % cvec);
    const size_t pix = idx / cvec;
    const int b = static_cast<int>(pix / (static_cast<size_t>(Ho) * Wo));
    const int rem = static_cast<int>(pix % (static_cast<size_t>(Ho) * Wo));
    const int p = rem / Wo, q = rem % Wo;
    const size_t src = ((static_cast<size_t>(b) * H + 2 * p) * W + 2 * q) * C + cv * 8;
    *reinterpret_cast<uint4*>(out_hi + pix * C + cv * 8) = *reinterpret_cast<const uint4*>(in_hi + src);
    if (out_lo) *reinterpret_cast<uint4*>(out_lo + pix * C + cv * 8) = *reinterpret_cast<const uint4*>(in_lo + src);
  }
}

// mean over the 7x7 bins of fpn_box_feat (deep_sort/utils.py:27-28 does this on the host)
__global__ void pool_feat_kernel(const float* __restrict__ feat, int rows, int C, float* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * C) return;
  const float* f = feat + static_cast<size_t>(idx) * 49;
  float s = 0.f;
  for (int i = 0; i < 49; ++i) s += f[i];
  out[idx] = s / 49.f;
}

// The TMOT driver's other embedding aggregations of fpn_box_feat (obj_detect_tracking_multi_queuer_tmot.py:511-525):
// mode 2 "max" = amax over the 7x7 bins -> [rows][C]; mode 3 "spatial" = mean over the channels -> [rows][49].
__global__ void agg_feat_kernel(const float* __restrict__ feat, int rows, int C, int mode, float* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (mode == 2) {
    if (idx >= rows * C) return;
    const float* f = feat + static_cast<size_t>(idx) * 49;
    float m = f[0];
    for (int i = 1; i < 49; ++i) m = fmaxf(m, f[i]);
    out[idx] = m;
  } else {
    if (idx >= rows * 49) return;
    const int r = idx / 49, bin = idx - r * 49;
    const float* f = feat + static_cast<size_t>(r) * C * 49 + bin;
    float s = 0.f;
    for (int ch = 0; ch < C; ++ch) s += f[static_cast<size_t>(ch) * 49];
    out[idx] = s / static_cast<float>(C);
  }
}

// Mask head output (models.py:950-958): per final detection the logits of its own class, sigmoid, and the un-shuffle of
// the 2x2 transposed-conv taps.  logits rows are ((roi * 196 + y * 14 + x) * 4 + dy * 2 + dx); out [B*R][28][28].
__global__ void mask_select_kernel(const float* __restrict__ logits, int ld, const int* __restrict__ labels,
                                   const int* __restrict__ count, int B, int R, float* __restrict__ out) {
  const size_t total = static_cast<size_t>(B) * R * 784;
  for (size_t idx = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; idx < total;
       idx += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const int px = static_cast<int>(idx % 784);
    const size_t roi = idx / 784;
    const int b = static_cast<int>(roi / R), j = static_cast<int>(roi % R);
    float v = 0.f;
    if (j < count[b]) {
      const int Y = px / 28, X = px % 28;
      const size_t row = (roi * 196 + static_cast<size_t>(Y >> 1) * 14 + (X >> 1)) * 4 + (Y & 1) * 2 + (X & 1);
      const float z = logits[row * ld + (labels[roi] - 1)];
      v = 1.f / (1.f + expf(-z));
    }
    out[idx] = v;
  }
}

struct Planes {
  __half* hi = nullptr;
  __half* lo = nullptr;
  int B = 0, H = 0, W = 0, C = 0;
  size_t elems() const { return static_cast<size_t>(B) * H * W * C; }
};

struct Layer {
  std::string name;        // reference variable scope, e.g. "group1/block0/conv2"
  ConvDesc d;
  ConvWeights w;
  ConvIO io;
  ConvPlan* plan = nullptr;
  std::vector<ConvPlan*> part_plan;              // the same layer over each 1/nsplit of the batch (multi-stream passes)
  bool has_bn = false, has_bias = false;
  int kind = 0;            // 0 conv HWIO, 1 fc6 (NCHW-flatten permute), 2 dense, 3 rpn class+box, 4 head outputs,
                           // 5 stem, 6 mask-head transposed conv 2x2/2 (as a 1x1 conv onto 4 taps x C outputs)
};

struct StageRef {
  int kind;                // 0 planes, 1 f32, 2 i32
  Planes pl;
  void* ptr = nullptr;
  int64_t shape[4] = {1, 1, 1, 1};
};

enum { NPHASE = 8 };

}  // namespace
}  // namespace b2

using namespace b2;

struct b2_ctx {
  b2_config cfg;
  int device = 0, num_sms = 148;
  bool split = false;
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  std::vector<std::unique_ptr<Layer>> layers;
  std::vector<Layer*> phase_layers[NPHASE];   // conv layers per phase, in launch order (phases with only convs)
  std::map<std::string, StageRef> stages;
  // geometry
  int c1h = 0, c1w = 0, ch[4], cw[4], ph[5], pw[5], pfh[5], pfw[5];
  // buffers
  void* img = nullptr;
  size_t img_bytes = 0;
  uint8_t* raw_frames = nullptr;   // b2_detect_host_resize: source-resolution uint8 frames
  size_t raw_bytes = 0;
  // pipelined ingest (b2_submit_host / b2_wait): two staging buffers fed by a copy stream
  cudaStream_t copy_stream = nullptr, down_stream = nullptr;
  void* stage_in[2] = {nullptr, nullptr};
  uint8_t* stage_out[2] = {nullptr, nullptr};     // boxes | probs | labels | count | feat, device copies per slot
  cudaEvent_t pass_done[2] = {nullptr, nullptr};
  cudaEvent_t h2d_done[2] = {nullptr, nullptr}, staged_free[2] = {nullptr, nullptr}, out_done[2] = {nullptr, nullptr};
  bool slot_busy[2] = {false, false};
  // range monitor: conv_tc_kernel ORs the device word when an fp16-plane output exceeds +-65504 (or is NaN); the word is
  // read back with every host-facing result (h_range: [0], [1] = submit slots, [2] = synchronous calls)
  unsigned int* range_flag = nullptr;
  unsigned int* h_range = nullptr;
  Planes stem_u, c1, pool, cfeat[4], lat[4], pfeat[5], rpn_h[5];
  float* rpn_out[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
  RpnParams rpn;
  RoiAlignParams roi1, roi2, roi3;
  HeadPostParams post;
  Planes roi_feat, fc6, fc7;
  float* head_logits = nullptr;
  float* box_feat = nullptr;
  float* box_feat_pooled = nullptr;
  float* given_boxes = nullptr;    // b2_box_features: [R][4] boxes + count of the current chunk
  int* given_count = nullptr;
  float* given_feat = nullptr;     // [R][C][7][7] and pooled [R][C]
  float* given_pooled = nullptr;
  float* box_feat_agg = nullptr;   // feat_mode 2 / 3 scratch ([B*R][C] or [B*R][49]), allocated on first use
  // mask head (cfg.add_mask): ROIAlign 14 of the final boxes -> 4 x conv3x3 -> deconv -> conv1x1 -> sigmoid of own class
  Planes mask_a, mask_b, mask_up;
  float* mask_logits = nullptr;
  int mask_ld = 0;
  float* final_masks = nullptr;    // [B][R][28][28]
  // launch bookkeeping
  struct Step {
    int phase;
    int kind;   // 0 conv layer, 1 stem, 2 maxpool, 3 subsample p6, 4 proposals, 5 roialign1, 6 post, 7 roialign2,
                // 8 roialign 14x14 of the final boxes (mask head), 9 mask select + sigmoid
    Layer* layer;
  };
  std::vector<Step> steps;
  cudaGraphExec_t graph = nullptr;
  // dual-stream pass: the backbone / FPN / RPN-head phases run as two half-batches on two streams, so that the tail of
  // one layer's persistent kernel (tiles % SMs != 0, no SM busy in the last round) overlaps the other half's kernels
  int nsplit = 1;                                  // batch parts (= streams) of the forked phases: 1 or 2
  cudaStream_t side_stream = nullptr;
  cudaEvent_t fork_ev = nullptr, join_ev = nullptr;
  bool weights_loaded = false;
  cudaEvent_t ev[NPHASE + 1];
  float phase_ms[NPHASE];
  int launches = 0;

  template <typename T>
  T* alloc(size_t n, bool zero = true) {
    void* p = nullptr;
    if (cudaMalloc(&p, n * sizeof(T) + 256) != cudaSuccess) return nullptr;
    if (zero) cudaMemset(p, 0, n * sizeof(T) + 256);
    allocs.push_back(p);
    return static_cast<T*>(p);
  }
  bool alloc_planes(Planes& p, int B, int H, int W, int C) {
    p.B = B; p.H = H; p.W = W; p.C = C;
    p.hi = alloc<__half>(p.elems());
    p.lo = split ? alloc<__half>(p.elems()) : nullptr;
    return p.hi != nullptr && (!split || p.lo != nullptr);
  }
};

namespace {

void reg_planes(b2_ctx* c, const std::string& name, const Planes& p) {
  StageRef s;
  s.kind = 0;
  s.pl = p;
  s.shape[0] = p.B; s.shape[1] = p.H; s.shape[2] = p.W; s.shape[3] = p.C;
  c->stages[name] = s;
}
void reg_raw(b2_ctx* c, const std::string& name, void* ptr, int kind, int64_t a, int64_t b, int64_t cc, int64_t d) {
  StageRef s;
  s.kind = kind;
  s.ptr = ptr;
  s.shape[0] = a; s.shape[1] = b; s.shape[2] = cc; s.shape[3] = d;
  c->stages[name] = s;
}

// Adds one conv layer reading `in` (view in_H x in_W of the buffer) and writing `out`.
Layer* add_conv(b2_ctx* c, int phase, const std::string& name, const Planes& in, int view_h, int view_w, int R,
                int stride, int dil, int pt, int pb, int pl, int pr, int Cout, bool bn, bool bias, bool relu,
                const Planes& out, int off_h, int off_w, const Planes* res, int res_shift, float* out_f32 = nullptr,
                int ldc_f32 = 0, int kind = 0, int S = 0) {
  std::unique_ptr<Layer> L(new Layer());
  L->name = name;
  L->has_bn = bn;
  L->has_bias = bias;
  L->kind = kind;
  ConvDesc& d = L->d;
  d.B = in.B; d.in_H = view_h; d.in_W = view_w; d.Cin = in.C;
  d.in_pitch_H = in.H; d.in_pitch_W = in.W; d.in_ld = in.C;
  d.R = R; d.S = S > 0 ? S : R; d.stride = stride; d.dil = dil;
  d.pad_t = pt; d.pad_b = pb; d.pad_l = pl; d.pad_r = pr;
  d.Cout = Cout;
  d.relu = relu ? 1 : 0;
  d.acc_kb = c->cfg.accum_chunk;
  d.off_h = off_h; d.off_w = off_w;
  if (out_f32) {
    d.out_H = d.Ho(); d.out_W = d.Wo(); d.ldc = ldc_f32;
  } else {
    d.out_H = out.H; d.out_W = out.W; d.ldc = out.C;
  }
  if (res) {
    d.res_H = res->H; d.res_W = res->W; d.ldr = res->C; d.res_shift = res_shift;
  }
  L->w.Cout_pad = (Cout + 15) / 16 * 16;
  L->w.K = d.R * d.S * in.C;
  L->w.w_hi = c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K);
  L->w.w_lo = c->split ? c->alloc<__half>(static_cast<size_t>(L->w.Cout_pad) * L->w.K) : nullptr;
  L->w.bias = c->alloc<float>(L->w.Cout_pad);
  L->io.in_hi = in.hi; L->io.in_lo = in.lo;
  L->io.out_hi = out.hi; L->io.out_lo = out.lo; L->io.out_f32 = out_f32;
  if (res) { L->io.res_hi = res->hi; L->io.res_lo = res->lo; }
  L->io.range_flag = c->range_flag;
  Layer* raw = L.get();
  c->layers.push_back(std::move(L));
  c->steps.push_back({phase, 0, raw});
  return raw;
}

int log2i(int v) { int r = 0; while ((1 << r) < v) ++r; return r; }

// generate_anchors.py:42-109 restated for one (stride, size): the 3 ratio anchors of a cell.
void cell_anchors(float stride, float size, const float* ratios, float out[3][4]) {
  const double base = stride;
  const double w0 = base, h0 = base, xc = 0.5 * (w0 - 1), yc = 0.5 * (h0 - 1);
  const double area = w0 * h0;
  const double scale = size / stride;
  for (int i = 0; i < 3; ++i) {
    const double ws = nearbyint(sqrt(area / ratios[i]));
    const double hs = nearbyint(ws * ratios[i]);
    // _mkanchors then _scale_enum (single scale)
    const double x1 = xc - 0.5 * (ws - 1), x2 = xc + 0.5 * (ws - 1);
    const double y1 = yc - 0.5 * (hs - 1), y2 = yc + 0.5 * (hs - 1);
    const double w = x2 - x1 + 1, h = y2 - y1 + 1;
    const double cx = x1 + 0.5 * (w - 1), cy = y1 + 0.5 * (h - 1);
    const double W = w * scale, H = h * scale;
    out[i][0] = static_cast<float>(cx - 0.5 * (W - 1));
    out[i][1] = static_cast<float>(cy - 0.5 * (H - 1));
    out[i][2] = static_cast<float>(cx + 0.5 * (W - 1));
    out[i][3] = static_cast<float>(cy + 0.5 * (H - 1));
  }
}

int build_plan(b2_ctx* c) {
  const b2_config& cfg = c->cfg;
  const int B = cfg.batch, H = cfg.height, W = cfg.width;
  B2_CHECK(B >= 1 && H >= 32 && W >= 32, "b2_create: bad frame geometry");
  B2_CHECK(cfg.fpn_num_channel == 256, "b2_create: fpn_num_channel must be 256");
  B2_CHECK(cfg.rpn_topk >= 1 && cfg.rpn_topk <= 1024, "b2_create: rpn_topk must be in [1,1024]");
  // ---- geometry (nn.py:843-944, tf_pad_reverse=True) ----
  const int PH = (H + 31) / 32 * 32, PW = (W + 31) / 32 * 32;
  c->c1h = (PH + 5 - 7) / 2 + 1;
  c->c1w = (PW + 5 - 7) / 2 + 1;
  int h = (c->c1h + 1 - 3) / 2 + 1, w = (c->c1w + 1 - 3) / 2 + 1;
  for (int g = 0; g < 4; ++g) {
    if (g > 0) { h = (h + 1 - 3) / 2 + 1; w = (w + 1 - 3) / 2 + 1; }
    c->ch[g] = h; c->cw[g] = w;
  }
  for (int i = 0; i < 4; ++i) { c->pfh[i] = c->ch[i]; c->pfw[i] = c->cw[i]; }
  c->pfh[4] = (c->ch[3] - 1) / 2 + 1;
  c->pfw[4] = (c->cw[3] - 1) / 2 + 1;
  for (int i = 0; i < 5; ++i) {
    c->ph[i] = c->pfh[i]; c->pw[i] = c->pfw[i];
    if (i < 3) {   // models.py:382-390 crop p2..p4 to ceil(H/stride)
      const int s = static_cast<int>(cfg.anchor_strides[i]);
      c->ph[i] = std::min(c->pfh[i], (H + s - 1) / s);
      c->pw[i] = std::min(c->pfw[i], (W + s - 1) / s);
    }
  }
  for (int i = 0; i < 3; ++i)
    B2_CHECK(c->ch[i] == 2 * c->ch[i + 1] && c->cw[i] == 2 * c->cw[i + 1], "b2_create: FPN levels must nest 2x");

  // ---- input + stem + pool (phase 0) ----
  c->img_bytes = static_cast<size_t>(B) * H * W * 3 * (cfg.input_dtype == 1 ? 1 : 4);
  c->img = c->alloc<uint8_t>(c->img_bytes);
  c->range_flag = c->alloc<unsigned int>(1);
  B2_CHECK(c->range_flag != nullptr, "out of device memory (range flag)");
  B2_CUDA(cudaMallocHost(&c->h_range, 3 * sizeof(unsigned int)));
  c->h_range[0] = c->h_range[1] = c->h_range[2] = 0;
  // compact stem operand [B][c1h + 3][c1w + 3][16]; conv0 reads 64-channel pixels out of it with a pixel stride of 16 (stem.cu)
  B2_CHECK(c->alloc_planes(c->stem_u, B, c->c1h + 3, c->c1w + 3, 16), "alloc stem operand");
  B2_CHECK(c->alloc_planes(c->c1, B, c->c1h, c->c1w, 64), "alloc c1");
  B2_CHECK(c->alloc_planes(c->pool, B, c->ch[0], c->cw[0], 64), "alloc pool");
  c->steps.push_back({0, 1, nullptr});
  // conv0 as a 4x1 VALID conv over the packed operand (see stem.cu), BN + ReLU in the epilogue
  {
    Planes view = c->stem_u;
    view.C = 64;                       // one GEMM pixel = 4 consecutive operand pixels
    Layer* L0 = add_conv(c, 0, "conv0", view, c->c1h + 3, c->c1w, 4, 1, 1, 0, 0, 0, 0, 64, true, false, true, c->c1, 0, 0,
                         nullptr, 0, nullptr, 0, 5, 1);
    L0->d.in_ld = 16;
  }
  c->steps.push_back({0, 2, nullptr});
  reg_planes(c, "c1", c->c1);
  reg_planes(c, "pool", c->pool);

  // ---- ResNet groups (nn.py:459-588) ----
  Planes cur = c->pool;
  for (int g = 0; g < 4; ++g) {
    const int feat = 64 << g, count = cfg.resnet_blocks[g];
    const int gh = c->ch[g], gw = c->cw[g];
    Planes pingpong[2];
    B2_CHECK(c->alloc_planes(pingpong[0], B, gh, gw, feat * 4), "alloc group out");
    B2_CHECK(c->alloc_planes(pingpong[1], B, gh, gw, feat * 4), "alloc group out");
    Planes t1_first, t1, t2, t2_first, sc;
    B2_CHECK(c->alloc_planes(t1_first, B, cur.H, cur.W, feat), "alloc t1");
    B2_CHECK(c->alloc_planes(t1, B, gh, gw, feat), "alloc t1");
    B2_CHECK(c->alloc_planes(t2, B, gh, gw, feat), "alloc t2");
    B2_CHECK(c->alloc_planes(t2_first, B, gh, gw, feat), "alloc t2");
    B2_CHECK(c->alloc_planes(sc, B, gh, gw, feat * 4), "alloc shortcut");
    for (int i = 0; i < count; ++i) {
      const std::string p = "group" + std::to_string(g) + "/block" + std::to_string(i);
      const int stride = (g > 0 && i == 0) ? 2 : 1;
      const bool in_last3 = i >= count - 3;
      const int dil = (g == 3 && cfg.use_dilations && in_last3) ? 2 : 1;
      const Planes& x = cur;
      const Planes& a1 = (i == 0) ? t1_first : t1;
      add_conv(c, 0, p + "/conv1", x, x.H, x.W, 1, 1, 1, 0, 0, 0, 0, feat, true, false, true, a1, 0, 0, nullptr, 0);
      const Planes* a2 = &t2;
      if (stride == 2) {
        // pad [1,0] + 3x3 stride-2 VALID (nn.py:487-492); with dilation the output is padded [1,0] again
        // (nn.py:493-497): written at offset (1,1) of a buffer whose first row/col stay zero.
        a2 = &t2_first;
        const int off = dil != 1 ? 1 : 0;
        add_conv(c, 0, p + "/conv2", a1, a1.H, a1.W, 3, 2, dil, 1, 0, 1, 0, feat, true, false, true, *a2, off, off,
                 nullptr, 0);
      } else {
        add_conv(c, 0, p + "/conv2", a1, a1.H, a1.W, 3, 1, dil, dil, dil, dil, dil, feat, true, false, true, *a2, 0,
                 0, nullptr, 0);
      }
      const Planes* resid = &x;
      if (x.C != feat * 4) {
        // resnet_shortcut (nn.py:551-566): stride 2 => drop last row/col, 1x1 stride-2 VALID
        if (stride == 2)
          add_conv(c, 0, p + "/convshortcut", x, x.H, x.W, 1, 2, 1, 0, -1, 0, -1, feat * 4, true, false, false, sc, 0,
                   0, nullptr, 0);
        else
          add_conv(c, 0, p + "/convshortcut", x, x.H, x.W, 1, 1, 1, 0, 0, 0, 0, feat * 4, true, false, false, sc, 0,
                   0, nullptr, 0);
        resid = &sc;
      }
      const Planes& out = pingpong[i & 1];
      add_conv(c, 0, p + "/conv3", *a2, a2->H, a2->W, 1, 1, 1, 0, 0, 0, 0, feat * 4, true, false, true, out, 0, 0,
               resid, 0);
      cur = out;
    }
    c->cfeat[g] = cur;
    reg_planes(c, "c" + std::to_string(g + 2), cur);
  }

  // ---- FPN (nn.py:947-1014), phase 1 ----
  const int nc = cfg.fpn_num_channel;
  for (int i = 3; i >= 0; --i) {
    B2_CHECK(c->alloc_planes(c->lat[i], B, c->ch[i], c->cw[i], nc), "alloc lateral");
    const std::string nm = "fpn/lateral_1x1_c" + std::to_string(i + 2);
    add_conv(c, 1, nm, c->cfeat[i], c->ch[i], c->cw[i], 1, 1, 1, 0, 0, 0, 0, nc, false, true, false, c->lat[i], 0, 0,
             i < 3 ? &c->lat[i + 1] : nullptr, 1);
  }
  for (int i = 0; i < 4; ++i) {
    B2_CHECK(c->alloc_planes(c->pfeat[i], B, c->pfh[i], c->pfw[i], nc), "alloc p");
    const std::string nm = "fpn/posthoc_3x3_p" + std::to_string(i + 2);
    add_conv(c, 1, nm, c->lat[i], c->ch[i], c->cw[i], 3, 1, 1, 1, 1, 1, 1, nc, false, true, false, c->pfeat[i], 0, 0,
             nullptr, 0);
    reg_planes(c, "p" + std::to_string(i + 2), c->pfeat[i]);
  }
  B2_CHECK(c->alloc_planes(c->pfeat[4], B, c->pfh[4], c->pfw[4], nc), "alloc p6");
  c->steps.push_back({1, 3, nullptr});
  reg_planes(c, "p6", c->pfeat[4]);

  // ---- RPN head (models.py:979-1009), phase 2; class+box 1x1 fused into one N=15 GEMM ----
  for (int i = 0; i < 5; ++i) {
    B2_CHECK(c->alloc_planes(c->rpn_h[i], B, c->ph[i], c->pw[i], nc), "alloc rpn hidden");
    Layer* L0 = add_conv(c, 2, "rpn/conv0", c->pfeat[i], c->ph[i], c->pw[i], 3, 1, 1, 1, 1, 1, 1, nc, false, true,
                         true, c->rpn_h[i], 0, 0, nullptr, 0);
    (void)L0;
    c->rpn_out[i] = c->alloc<float>(static_cast<size_t>(B) * c->ph[i] * c->pw[i] * 16 + 16 * 128);
    add_conv(c, 2, "rpn/classbox", c->rpn_h[i], c->ph[i], c->pw[i], 1, 1, 1, 0, 0, 0, 0, 15, false, true, false,
             Planes(), 0, 0, nullptr, 0, c->rpn_out[i], 16, 3);
    reg_raw(c, "rpn_l" + std::to_string(i), c->rpn_out[i], 1, B, c->ph[i], c->pw[i], 16);
  }

  // ---- proposals (phase 3) ----
  RpnParams& rp = c->rpn;
  memset(&rp, 0, sizeof(rp));
  const int K = cfg.rpn_topk;
  for (int i = 0; i < 5; ++i) {
    rp.logits[i] = c->rpn_out[i];
    rp.h[i] = c->ph[i];
    rp.w[i] = c->pw[i];
    rp.stride[i] = cfg.anchor_strides[i];
    cell_anchors(cfg.anchor_strides[i], cfg.anchor_sizes[i], cfg.anchor_ratios, rp.cell[i]);
  }
  rp.B = B; rp.topk = K;
  rp.img_h = static_cast<float>(H); rp.img_w = static_cast<float>(W);
  rp.decode_clip = logf(cfg.max_size / 16.0f);
  {
    const double dc = log(static_cast<double>(cfg.max_size) / 16.0);   // np.log in float64, cast at use
    rp.decode_clip = static_cast<float>(dc);
  }
  rp.min_size = cfg.rpn_min_size;
  rp.multi = cfg.multi_semantics;
  rp.nms_thr = cfg.rpn_nms_thres;
  rp.lvl_boxes = c->alloc<float>(static_cast<size_t>(B) * 5 * K * 4);
  rp.lvl_scores = c->alloc<float>(static_cast<size_t>(B) * 5 * K);
  rp.lvl_count = c->alloc<int>(B * 5);
  rp.prop_boxes = c->alloc<float>(static_cast<size_t>(B) * K * 4);
  rp.prop_scores = c->alloc<float>(static_cast<size_t>(B) * K);
  rp.prop_count = c->alloc<int>(B);
  c->steps.push_back({3, 4, nullptr});
  reg_raw(c, "lvl_boxes", rp.lvl_boxes, 1, B, 5, K, 4);
  reg_raw(c, "lvl_scores", rp.lvl_scores, 1, B, 5, K, 1);
  reg_raw(c, "lvl_count", rp.lvl_count, 2, B, 5, 1, 1);
  reg_raw(c, "proposal_boxes", rp.prop_boxes, 1, B, K, 4, 1);
  reg_raw(c, "proposal_scores", rp.prop_scores, 1, B, K, 1, 1);
  reg_raw(c, "proposal_count", rp.prop_count, 2, B, 1, 1, 1);

  // ---- ROIAlign of the proposals (phase 4) ----
  const int M = B * K;
  const int Mpad = (M + 127) / 128 * 128;
  B2_CHECK(c->alloc_planes(c->roi_feat, 1, 1, Mpad, 49 * nc), "alloc roi feat");
  RoiAlignParams& r1 = c->roi1;
  memset(&r1, 0, sizeof(r1));
  for (int i = 0; i < 4; ++i) {
    r1.feat_hi[i] = c->pfeat[i].hi;
    r1.feat_lo[i] = c->pfeat[i].lo;
    r1.H[i] = c->ph[i]; r1.W[i] = c->pw[i];
    r1.pitch_H[i] = c->pfh[i]; r1.pitch_W[i] = c->pfw[i];
    r1.inv_stride[i] = 1.0f / cfg.anchor_strides[i];
  }
  r1.C = nc; r1.B = B; r1.rois_per_image = K;
  r1.boxes = rp.prop_boxes; r1.count = rp.prop_count;
  r1.out_hi = c->roi_feat.hi; r1.out_lo = c->roi_feat.lo; r1.out_nchw = nullptr;
  c->steps.push_back({4, 5, nullptr});
  reg_planes(c, "roi_feat", c->roi_feat);

  // ---- box head (models.py:1030-1108), phase 5: fc6, fc7, class+box outputs fused (N = 5*num_class) ----
  const int dim = cfg.fc_head_dim;
  B2_CHECK(dim % 64 == 0, "b2_create: fc_head_dim must be a multiple of 64");
  B2_CHECK(c->alloc_planes(c->fc6, 1, 1, Mpad, dim), "alloc fc6");
  B2_CHECK(c->alloc_planes(c->fc7, 1, 1, Mpad, dim), "alloc fc7");
  const int nout = cfg.num_class + (cfg.class_agnostic ? 4 : cfg.num_class * 4);
  const int ldo = (nout + 15) / 16 * 16;
  c->head_logits = c->alloc<float>(static_cast<size_t>(Mpad) * ldo);
  Planes rf = c->roi_feat; rf.W = M;
  Planes f6 = c->fc6; f6.W = M;
  Planes f7 = c->fc7; f7.W = M;
  add_conv(c, 5, "fastrcnn/fc6", rf, 1, M, 1, 1, 1, 0, 0, 0, 0, dim, false, true, true, f6, 0, 0, nullptr, 0, nullptr,
           0, 1);
  add_conv(c, 5, "fastrcnn/fc7", f6, 1, M, 1, 1, 1, 0, 0, 0, 0, dim, false, true, true, f7, 0, 0, nullptr, 0, nullptr,
           0, 2);
  add_conv(c, 5, "fastrcnn/outputs", f7, 1, M, 1, 1, 1, 0, 0, 0, 0, nout, false, true, false, Planes(), 0, 0, nullptr,
           0, c->head_logits, ldo, 4);
  reg_planes(c, "fc6", f6);
  reg_planes(c, "fc7", f7);
  reg_raw(c, "head_logits", c->head_logits, 1, B, K, ldo, 1);

  // ---- post-processing (phase 6) ----
  HeadPostParams& hp = c->post;
  memset(&hp, 0, sizeof(hp));
  const int nc1 = cfg.num_class - 1, R = cfg.result_per_im;
  hp.logits = c->head_logits; hp.ld = ldo; hp.num_class = cfg.num_class; hp.B = B; hp.rois_per_image = K;
  hp.class_agnostic = cfg.class_agnostic;
  hp.rois = rp.prop_boxes; hp.roi_count = rp.prop_count;
  for (int i = 0; i < 4; ++i) hp.reg_w[i] = cfg.bbox_reg_weights[i];
  hp.decode_clip = static_cast<float>(log(1333.0 / 16.0));   // decode_bbox_target default (nn.py:1518)
  hp.img_h = static_cast<float>(H); hp.img_w = static_cast<float>(W);
  // batch graph: combined_non_max_suppression is called without a score threshold (models.py:2959-2965)
  hp.score_thresh = cfg.multi_semantics ? -INFINITY : cfg.result_score_thres;
  hp.nms_thr = cfg.fastrcnn_nms_iou_thres;
  hp.max_per_class = R; hp.max_total = R;
  hp.probs = c->alloc<float>(static_cast<size_t>(M) * cfg.num_class);
  hp.dec_boxes = c->alloc<float>(static_cast<size_t>(M) * nc1 * 4);
  hp.cls_keep = c->alloc<int>(static_cast<size_t>(B) * nc1 * R);
  hp.cls_count = c->alloc<int>(B * nc1);
  hp.final_boxes = c->alloc<float>(static_cast<size_t>(B) * R * 4);
  hp.final_probs = c->alloc<float>(static_cast<size_t>(B) * R);
  hp.final_labels = c->alloc<int>(static_cast<size_t>(B) * R);
  hp.final_count = c->alloc<int>(B);
  c->steps.push_back({6, 6, nullptr});
  reg_raw(c, "probs", hp.probs, 1, B, K, cfg.num_class, 1);
  reg_raw(c, "dec_boxes", hp.dec_boxes, 1, B, K, nc1, 4);
  reg_raw(c, "final_boxes", hp.final_boxes, 1, B, R, 4, 1);
  reg_raw(c, "final_probs", hp.final_probs, 1, B, R, 1, 1);
  reg_raw(c, "final_labels", hp.final_labels, 2, B, R, 1, 1);
  reg_raw(c, "final_count", hp.final_count, 2, B, 1, 1, 1);

  // ---- fpn_box_feat: ROIAlign of the final boxes (models.py:972-973), phase 7 ----
  c->box_feat = c->alloc<float>(static_cast<size_t>(B) * R * nc * 49);
  c->box_feat_pooled = c->alloc<float>(static_cast<size_t>(B) * R * nc);
  RoiAlignParams& r2 = c->roi2;
  r2 = r1;
  r2.rois_per_image = R;
  r2.boxes = hp.final_boxes; r2.count = hp.final_count;
  r2.out_hi = nullptr; r2.out_lo = nullptr; r2.out_nchw = c->box_feat;
  c->steps.push_back({7, 7, nullptr});
  reg_raw(c, "fpn_box_feat", c->box_feat, 1, static_cast<int64_t>(B) * R, nc, 7, 7);

  // ---- mask head (models.py:934-961, 1173-1199), phase 7, only with cfg.add_mask ----
  if (cfg.add_mask) {
    B2_CHECK(cfg.num_class >= 2, "b2_create: add_mask needs at least one foreground class");
    const int MR = B * R, md = 256;                  // mrcnn_head_dim (obj_detect_tracking.py:324)
    B2_CHECK(c->alloc_planes(c->mask_a, MR, 14, 14, md), "alloc mask head a");
    B2_CHECK(c->alloc_planes(c->mask_b, MR, 14, 14, md), "alloc mask head b");
    B2_CHECK(c->alloc_planes(c->mask_up, MR, 14, 14, 4 * md), "alloc mask head deconv");
    RoiAlignParams& r3 = c->roi3;
    r3 = r1;
    r3.rois_per_image = R;
    r3.boxes = hp.final_boxes; r3.count = hp.final_count;
    r3.out_hi = c->mask_a.hi; r3.out_lo = c->mask_a.lo; r3.out_nchw = nullptr; r3.out_res = 14;
    c->steps.push_back({7, 8, nullptr});
    const Planes* pp[2] = {&c->mask_a, &c->mask_b};
    for (int k = 0; k < 4; ++k)                      // conv2d 3x3 SAME + bias + ReLU
      add_conv(c, 7, "maskrcnn/fcn" + std::to_string(k), *pp[k & 1], 14, 14, 3, 1, 1, 1, 1, 1, 1, md, false, true, true,
               *pp[(k + 1) & 1], 0, 0, nullptr, 0);
    // Conv2DTranspose 2x2 stride 2: no overlap between taps, so it is a 1x1 conv onto (tap, channel) outputs
    add_conv(c, 7, "maskrcnn/deconv", c->mask_a, 14, 14, 1, 1, 1, 0, 0, 0, 0, 4 * md, false, true, true, c->mask_up, 0, 0,
             nullptr, 0, nullptr, 0, 6);
    // the 1x1 class conv commutes with the pixel shuffle: apply it to the (pixel, tap) rows directly
    const int rows = MR * 196 * 4, rows_pad = (rows + 127) / 128 * 128;
    c->mask_ld = (cfg.num_class - 1 + 15) / 16 * 16;
    c->mask_logits = c->alloc<float>(static_cast<size_t>(rows_pad) * c->mask_ld);
    Planes up_rows = c->mask_up;
    up_rows.B = 1; up_rows.H = 1; up_rows.W = rows; up_rows.C = md;
    add_conv(c, 7, "maskrcnn/conv", up_rows, 1, rows, 1, 1, 1, 0, 0, 0, 0, cfg.num_class - 1, false, true, false, Planes(),
             0, 0, nullptr, 0, c->mask_logits, c->mask_ld);
    c->final_masks = c->alloc<float>(static_cast<size_t>(MR) * 784);
    c->steps.push_back({7, 9, nullptr});
    reg_planes(c, "mask_roi_feat", c->mask_a);       // valid right after step 8 only (ping-pong buffer)
    reg_raw(c, "mask_logits", c->mask_logits, 1, MR, 196 * 4, c->mask_ld, 1);
    reg_raw(c, "final_masks", c->final_masks, 1, B, R, 28, 28);
  }

  // ---- tensor-core plans ----
  if (cfg.conv_impl == 0) {
    for (auto& L : c->layers) {
      L->plan = conv_tc_plan_create(L->d, L->w, L->io, c->split, c->num_sms);
      if (!L->plan) {
        set_error(std::string("plan for ") + L->name + ": " + last_error());
        return -1;
      }
    }
    // Images are independent through phases 0-2 (stem, ResNet, FPN, RPN head): a second set of plans covers each
    // half of the batch by itself (same tiles per image, so the results are bit-identical to the full-batch plan).
    c->nsplit = B % 2 == 0 ? 2 : 1;
    if (c->nsplit == 2) {
      for (const auto& s : c->steps) {
        if (s.kind != 0 || s.phase > 2) continue;
        Layer* L = s.layer;
        L->part_plan.assign(c->nsplit, nullptr);
        for (int h = 0; h < c->nsplit; ++h) {
          ConvDesc d = L->d;
          ConvIO io = L->io;
          d.B = B / c->nsplit;
          const size_t in_off = static_cast<size_t>(h) * d.B * d.in_pitch_H * d.in_pitch_W * (d.in_ld > 0 ? d.in_ld : d.Cin);
          const size_t out_off = static_cast<size_t>(h) * d.B * d.out_H * d.out_W * d.ldc;
          const size_t res_off = static_cast<size_t>(h) * d.B * d.res_H * d.res_W * d.ldr;
          io.in_hi += in_off;
          if (io.in_lo) io.in_lo += in_off;
          if (io.out_hi) io.out_hi += out_off;
          if (io.out_lo) io.out_lo += out_off;
          if (io.out_f32) io.out_f32 += out_off;
          if (io.res_hi) io.res_hi += res_off;
          if (io.res_lo) io.res_lo += res_off;
          L->part_plan[h] = conv_tc_plan_create(d, L->w, io, c->split, c->num_sms);
          if (!L->part_plan[h]) {
            set_error(std::string("half-batch plan for ") + L->name + ": " + last_error());
            return -1;
          }
        }
      }
    }
  }
  return 0;
}

int run_step(b2_ctx* c, const b2_ctx::Step& s) {
  const b2_config& cfg = c->cfg;
  cudaStream_t st = c->stream;
  switch (s.kind) {
    case 0:
      if (cfg.conv_impl == 0) return conv_tc_launch(s.layer->plan, st);
      return conv_simt_launch(s.layer->d, s.layer->w, s.layer->io, c->split, st);
    case 1:
      return stem_pack16_launch(c->img, cfg.input_dtype == 1, cfg.batch, cfg.height, cfg.width, c->stem_u.hi,
                                c->stem_u.lo, c->stem_u.H, c->stem_u.W, st);
    case 2:
      return maxpool_launch(c->c1.hi, c->c1.lo, cfg.batch, c->c1h, c->c1w, 64, c->pool.hi, c->pool.lo, c->ch[0],
                            c->cw[0], st);
    case 3: {
      const Planes& p5 = c->pfeat[3];
      const Planes& p6 = c->pfeat[4];
      const size_t total = static_cast<size_t>(p6.B) * p6.H * p6.W * (p6.C / 8);
      subsample2_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(p5.hi, p5.lo, p5.B, p5.H, p5.W,
                                                                                     p5.C, p6.hi, p6.lo, p6.H, p6.W);
      B2_CUDA(cudaGetLastError());
      return 0;
    }
    case 4:
      return rpn_proposals_launch(c->rpn, st);
    case 5:
      return roialign_launch(c->roi1, st);
    case 6:
      return head_post_launch(c->post, st);
    case 7: {
      if (roialign_launch(c->roi2, st)) return -1;
      const int rows = cfg.batch * cfg.result_per_im;
      pool_feat_kernel<<<(rows * cfg.fpn_num_channel + 255) / 256, 256, 0, st>>>(c->box_feat, rows,
                                                                                 cfg.fpn_num_channel,
                                                                                 c->box_feat_pooled);
      B2_CUDA(cudaGetLastError());
      return 0;
    }
    case 8:
      return roialign_launch(c->roi3, st);
    case 9: {
      const size_t total = static_cast<size_t>(cfg.batch) * cfg.result_per_im * 784;
      mask_select_kernel<<<static_cast<unsigned>(std::min<size_t>((total + 255) / 256, 148 * 32)), 256, 0, st>>>(
          c->mask_logits, c->mask_ld, c->post.final_labels, c->post.final_count, cfg.batch, cfg.result_per_im,
          c->final_masks);
      B2_CUDA(cudaGetLastError());
      return 0;
    }
  }
  return -1;
}

// One step of phases 0-2 over part `h` (of nsplit) of the batch, on stream `st`.
int run_step_half(b2_ctx* c, const b2_ctx::Step& s, int h, cudaStream_t st) {
  const b2_config& cfg = c->cfg;
  const int hb = cfg.batch / c->nsplit;
  auto off = [&](const Planes& p) { return static_cast<size_t>(h) * hb * p.H * p.W * p.C; };
  auto lo = [&](const Planes& p) { return p.lo ? p.lo + off(p) : nullptr; };
  switch (s.kind) {
    case 0:
      return conv_tc_launch(s.layer->part_plan[h], st);
    case 1:
      return stem_pack16_launch(static_cast<const uint8_t*>(c->img) + static_cast<size_t>(h) * (c->img_bytes / c->nsplit),
                                cfg.input_dtype == 1, hb, cfg.height, cfg.width, c->stem_u.hi + off(c->stem_u),
                                lo(c->stem_u), c->stem_u.H, c->stem_u.W, st);
    case 2:
      return maxpool_launch(c->c1.hi + off(c->c1), lo(c->c1), hb, c->c1h, c->c1w, 64, c->pool.hi + off(c->pool),
                            lo(c->pool), c->ch[0], c->cw[0], st);
    case 3: {
      const Planes& p5 = c->pfeat[3];
      const Planes& p6 = c->pfeat[4];
      const size_t total = static_cast<size_t>(hb) * p6.H * p6.W * (p6.C / 8);
      subsample2_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, st>>>(
          p5.hi + off(p5), lo(p5), hb, p5.H, p5.W, p5.C, p6.hi + off(p6), lo(p6), p6.H, p6.W);
      B2_CUDA(cudaGetLastError());
      return 0;
    }
  }
  return -1;
}

int step_launches(const b2_ctx::Step& s) {
  switch (s.kind) {
    case 4: return 2;
    case 6: return 3;
    case 7: return 2;
    default: return 1;
  }
}

// The whole pass with phases 0-2 forked over two streams (also valid inside a stream capture: the second stream joins
// the capture through the fork event and rejoins before the proposals).
int enqueue_dual(b2_ctx* c) {
  B2_CUDA(cudaEventRecord(c->fork_ev, c->stream));
  B2_CUDA(cudaStreamWaitEvent(c->side_stream, c->fork_ev, 0));
  for (const auto& s : c->steps) {
    if (s.phase > 2) continue;
    if (run_step_half(c, s, 0, c->stream) || run_step_half(c, s, 1, c->side_stream)) return -1;
  }
  B2_CUDA(cudaEventRecord(c->join_ev, c->side_stream));
  B2_CUDA(cudaStreamWaitEvent(c->stream, c->join_ev, 0));
  for (const auto& s : c->steps)
    if (s.phase > 2 && run_step(c, s)) return -1;
  return 0;
}

int enqueue(b2_ctx* c, int mask, bool with_events) {
  if (c->nsplit == 2 && !with_events && mask == B2_PHASE_ALL) return enqueue_dual(c);
  if (with_events) B2_CUDA(cudaEventRecord(c->ev[0], c->stream));
  int last = -1;
  for (const auto& s : c->steps) {
    if (!(mask & (1 << s.phase))) continue;
    if (with_events && last >= 0 && s.phase != last) B2_CUDA(cudaEventRecord(c->ev[last + 1], c->stream));
    if (run_step(c, s)) return -1;
    last = s.phase;
  }
  if (with_events && last >= 0) B2_CUDA(cudaEventRecord(c->ev[last + 1], c->stream));
  return 0;
}

// ---- weight loading -------------------------------------------------------------------------
struct WeightSet {
  std::map<std::string, std::pair<const float*, int64_t>> m;
  const float* get(const std::string& n, int64_t expect) const {
    auto it = m.find(n);
    if (it == m.end()) { set_error("missing weight: " + n); return nullptr; }
    if (it->second.second != expect) {
      set_error("weight " + n + ": expected " + std::to_string(expect) + " values, got " +
                std::to_string(it->second.second));
      return nullptr;
    }
    return it->second.first;
  }
  bool has(const std::string& n) const { return m.count(n) != 0; }
};

// BatchNorm inference folded into a per-output-channel scale/shift (nn.py:1771-1774, eps 1e-5)
int bn_fold(const WeightSet& ws, const std::string& scope, int C, std::vector<double>& scale,
            std::vector<double>& shift) {
  const float* g = ws.get(scope + "/bn/gamma", C);
  const float* b = ws.get(scope + "/bn/beta", C);
  const float* m = ws.get(scope + "/bn/mean/EMA", C);
  const float* v = ws.get(scope + "/bn/variance/EMA", C);
  if (!g || !b || !m || !v) return -1;
  scale.resize(C);
  shift.resize(C);
  for (int i = 0; i < C; ++i) {
    const double inv = static_cast<double>(g[i]) / sqrt(static_cast<double>(v[i]) + 1e-5);
    scale[i] = inv;
    shift[i] = static_cast<double>(b[i]) - static_cast<double>(m[i]) * inv;
  }
  return 0;
}

int upload_layer(b2_ctx* c, Layer* L, const std::vector<float>& packed, const std::vector<float>& bias) {
  const size_t n = packed.size();
  // the (hi, lo) operand planes are fp16: a folded weight beyond +-65504 (or a non-finite one) would become inf here and
  // NaN inside the MMA (inf * 0) -- refuse it at load time; activations are watched by the kernel's range monitor
  for (size_t i = 0; i < n; ++i)
    if (!(fabsf(packed[i]) <= 65504.f)) {
      set_error("weight of layer '" + L->name + "' outside the fp16-plane range (|w| > 65504 after BatchNorm folding, or not "
                "finite): this checkpoint is not representable in the (hi, lo) fp16 operand format");
      return -1;
    }
  for (size_t i = 0; i < bias.size(); ++i)
    if (!std::isfinite(bias[i])) {
      set_error("bias / folded BatchNorm shift of layer '" + L->name + "' is not finite");
      return -1;
    }
  float* tmp = nullptr;
  B2_CUDA(cudaMalloc(&tmp, n * sizeof(float)));
  B2_CUDA(cudaMemcpyAsync(tmp, packed.data(), n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  if (f32_to_planes(tmp, L->w.w_hi, L->w.w_lo, n, c->stream)) return -1;
  B2_CUDA(cudaMemcpyAsync(L->w.bias, bias.data(), bias.size() * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_CUDA(cudaFree(tmp));
  return 0;
}

int load_layer(b2_ctx* c, Layer* L, const WeightSet& ws) {
  const int Cin = L->d.Cin, R = L->d.R, S = L->d.S, Cout = L->d.Cout, K = L->w.K, Cp = L->w.Cout_pad;
  std::vector<float> packed(static_cast<size_t>(Cp) * K, 0.f), bias(Cp, 0.f);
  std::vector<double> scale(Cout, 1.0), shift(Cout, 0.0);
  if (L->kind == 0) {
    const float* w = ws.get(L->name + "/W", static_cast<int64_t>(R) * S * Cin * Cout);   // HWIO
    if (!w) return -1;
    if (L->has_bn && bn_fold(ws, L->name, Cout, scale, shift)) return -1;
    if (L->has_bias) {
      const float* b = ws.get(L->name + "/b", Cout);
      if (!b) return -1;
      for (int o = 0; o < Cout; ++o) shift[o] = b[o];
    }
    for (int t = 0; t < R * S; ++t)
      for (int ci = 0; ci < Cin; ++ci) {
        const float* src = w + (static_cast<size_t>(t) * Cin + ci) * Cout;
        for (int o = 0; o < Cout; ++o)
          packed[static_cast<size_t>(o) * K + static_cast<size_t>(t) * Cin + ci] = static_cast<float>(src[o] * scale[o]);
      }
  } else if (L->kind == 6) {
    // tf.layers.Conv2DTranspose kernel [kh=2, kw=2, out, in] (nn.py:402-412): output row (dy*2+dx)*out + o of the 1x1 conv
    const int co = Cout / 4;
    const float* w = ws.get(L->name + "/W", static_cast<int64_t>(4) * co * Cin);
    const float* b = ws.get(L->name + "/b", co);
    if (!w || !b) return -1;
    for (int t = 0; t < 4; ++t)
      for (int o = 0; o < co; ++o) {
        const float* src = w + (static_cast<size_t>(t) * co + o) * Cin;
        for (int ci = 0; ci < Cin; ++ci) packed[static_cast<size_t>(t * co + o) * K + ci] = src[ci];
        shift[t * co + o] = b[o];
      }
  } else if (L->kind == 5) {
    // stem: reference HWIO [7,7,3,64] re-indexed for the packed operand (stem.cu):
    // W'[o][r][s*16 + ry*6 + sx*3 + c] = W[2r+ry][2s+sx][c][o]   (12 real + 4 zero channels per width tap s)
    const float* w = ws.get(L->name + "/W", 7 * 7 * 3 * 64);
    if (!w || bn_fold(ws, L->name, Cout, scale, shift)) return -1;
    for (int r = 0; r < 4; ++r)
      for (int ch = 0; ch < 64; ++ch) {
        const int s4 = ch / 16, r12 = ch % 16, ry = r12 / 6, sx = (r12 % 6) / 3, cc = r12 % 3;
        const int rr = 2 * r + ry, ss = 2 * s4 + sx;
        if (r12 >= 12 || rr >= 7 || ss >= 7) continue;
        const float* src = w + (static_cast<size_t>(rr * 7 + ss) * 3 + cc) * 64;
        for (int o = 0; o < Cout; ++o)
          packed[static_cast<size_t>(o) * K + static_cast<size_t>(r) * Cin + ch] = static_cast<float>(src[o] * scale[o]);
      }
  } else if (L->kind == 1) {
    // fc6: reference flattens NCHW (index c*49 + y*7 + x, models.py:1056 + nn.py:738-740);
    // our ROI features are [y][x][c], so permute the rows of W [in, out].
    const int C = c->cfg.fpn_num_channel;
    const float* w = ws.get(L->name + "/W", static_cast<int64_t>(Cin) * Cout);
    const float* b = ws.get(L->name + "/b", Cout);
    if (!w || !b) return -1;
    for (int ch = 0; ch < C; ++ch)
      for (int s = 0; s < 49; ++s) {
        const float* src = w + (static_cast<size_t>(ch) * 49 + s) * Cout;
        const size_t k = static_cast<size_t>(s) * C + ch;
        for (int o = 0; o < Cout; ++o) packed[static_cast<size_t>(o) * K + k] = src[o];
      }
    for (int o = 0; o < Cout; ++o) shift[o] = b[o];
  } else if (L->kind == 2) {
    const float* w = ws.get(L->name + "/W", static_cast<int64_t>(Cin) * Cout);
    const float* b = ws.get(L->name + "/b", Cout);
    if (!w || !b) return -1;
    for (int k = 0; k < Cin; ++k)
      for (int o = 0; o < Cout; ++o) packed[static_cast<size_t>(o) * K + k] = w[static_cast<size_t>(k) * Cout + o];
    for (int o = 0; o < Cout; ++o) shift[o] = b[o];
  } else if (L->kind == 3 || L->kind == 4) {
    // two reference layers fused along N: rpn/{class,box} or fastrcnn/outputs/{class,box}
    const std::string base = L->kind == 3 ? "rpn" : "fastrcnn/outputs";
    const int n0 = L->kind == 3 ? 3 : c->cfg.num_class;
    const int n1 = Cout - n0;
    const float* w0 = ws.get(base + "/class/W", static_cast<int64_t>(Cin) * n0);
    const float* b0 = ws.get(base + "/class/b", n0);
    const float* w1 = ws.get(base + "/box/W", static_cast<int64_t>(Cin) * n1);
    const float* b1 = ws.get(base + "/box/b", n1);
    if (!w0 || !b0 || !w1 || !b1) return -1;
    for (int k = 0; k < Cin; ++k) {
      for (int o = 0; o < n0; ++o) packed[static_cast<size_t>(o) * K + k] = w0[static_cast<size_t>(k) * n0 + o];
      for (int o = 0; o < n1; ++o) packed[static_cast<size_t>(n0 + o) * K + k] = w1[static_cast<size_t>(k) * n1 + o];
    }
    for (int o = 0; o < n0; ++o) shift[o] = b0[o];
    for (int o = 0; o < n1; ++o) shift[n0 + o] = b1[o];
  }
  for (int o = 0; o < Cout; ++o) bias[o] = static_cast<float>(shift[o]);
  return upload_layer(c, L, packed, bias);
}

}  // namespace

// =================================================================================================
extern "C" {

const char* b2_last_error(void) { return b2::last_error(); }
int b2_version(void) { return 1; }

int b2_create(b2_ctx** out, int device, const b2_config* cfg) {
  B2_CHECK(out && cfg, "b2_create: null argument");
  *out = nullptr;
  B2_CUDA(cudaSetDevice(device));
  std::unique_ptr<b2_ctx> c(new b2_ctx());
  c->cfg = *cfg;
  c->device = device;
  c->split = cfg->precision == 1;
  cudaDeviceProp prop;
  B2_CUDA(cudaGetDeviceProperties(&prop, device));
  B2_CHECK(prop.major == 10, "b2_create: this library is built for sm_100a (B200) only");
  c->num_sms = prop.multiProcessorCount;
  B2_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  for (int i = 0; i <= NPHASE; ++i) B2_CUDA(cudaEventCreate(&c->ev[i]));
  memset(c->phase_ms, 0, sizeof(c->phase_ms));
  if (build_plan(c.get())) {
    b2_destroy(c.release());
    return -1;
  }
  if (c->nsplit == 2) {
    B2_CUDA(cudaEventCreateWithFlags(&c->fork_ev, cudaEventDisableTiming));
    B2_CUDA(cudaStreamCreateWithFlags(&c->side_stream, cudaStreamNonBlocking));
    B2_CUDA(cudaEventCreateWithFlags(&c->join_ev, cudaEventDisableTiming));
  }
  c->launches = 0;
  for (const auto& s : c->steps) c->launches += step_launches(s) * (s.phase <= 2 ? c->nsplit : 1);
  B2_CUDA(cudaDeviceSynchronize());
  *out = c.release();
  return 0;
}

void b2_destroy(b2_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaDeviceSynchronize();
  if (c->graph) cudaGraphExecDestroy(c->graph);
  for (auto& L : c->layers) {
    if (L->plan) conv_tc_plan_destroy(L->plan);
    for (ConvPlan* pp : L->part_plan)
      if (pp) conv_tc_plan_destroy(pp);
  }
  if (c->fork_ev) cudaEventDestroy(c->fork_ev);
  if (c->join_ev) cudaEventDestroy(c->join_ev);
  if (c->side_stream) cudaStreamDestroy(c->side_stream);
  if (c->raw_frames) cudaFree(c->raw_frames);
  if (c->h_range) cudaFreeHost(c->h_range);
  for (void* p : c->allocs) cudaFree(p);
  for (int i = 0; i <= NPHASE; ++i)
    if (c->ev[i]) cudaEventDestroy(c->ev[i]);
  for (int i = 0; i < 2; ++i) {
    if (c->h2d_done[i]) cudaEventDestroy(c->h2d_done[i]);
    if (c->staged_free[i]) cudaEventDestroy(c->staged_free[i]);
    if (c->out_done[i]) cudaEventDestroy(c->out_done[i]);
    if (c->pass_done[i]) cudaEventDestroy(c->pass_done[i]);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->down_stream) cudaStreamDestroy(c->down_stream);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

int b2_load_weights(b2_ctx* c, const char* const* names, const float* const* data, const int64_t* numel, int n) {
  B2_CHECK(c && names && data && numel, "b2_load_weights: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  WeightSet ws;
  for (int i = 0; i < n; ++i) ws.m[names[i]] = std::make_pair(data[i], numel[i]);
  // shared RPN weights: packed once, every level's layer gets its own copy of the (small) operand
  for (auto& L : c->layers)
    if (load_layer(c, L.get(), ws)) return -1;
  c->weights_loaded = true;
  return 0;
}

static int range_failed(b2_ctx* c, int idx);

int b2_run_phases(b2_ctx* c, int mask) {
  B2_CHECK(c, "b2_run_phases: null ctx");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_run_phases: weights not loaded");
  if (enqueue(c, mask, true)) return -1;
  B2_CUDA(cudaMemcpyAsync(&c->h_range[2], c->range_flag, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  if (range_failed(c, 2)) return -1;
  int last = -1;
  for (int ph = 0; ph < NPHASE; ++ph) {
    c->phase_ms[ph] = 0.f;
    if (!(mask & (1 << ph))) continue;
    bool any = false;
    for (const auto& s : c->steps) any = any || s.phase == ph;
    if (!any) continue;
    cudaEventElapsedTime(&c->phase_ms[ph], c->ev[last < 0 ? 0 : last + 1], c->ev[ph + 1]);
    last = ph;
  }
  return 0;
}

int b2_phase_times(b2_ctx* c, float ms[8]) {
  B2_CHECK(c && ms, "b2_phase_times: null argument");
  for (int i = 0; i < NPHASE; ++i) ms[i] = c->phase_ms[i];
  return 0;
}

int b2_kernel_launches(b2_ctx* c) { return c ? c->launches : -1; }

// Per-step device timing (CUDA events around every launch group, eager mode), averaged over `reps`.
int b2_profile_steps(b2_ctx* c, int reps, float* ms_out, int cap, int* n_out) {
  B2_CHECK(c && ms_out && n_out, "b2_profile_steps: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_profile_steps: weights not loaded");
  const int n = static_cast<int>(c->steps.size());
  B2_CHECK(cap >= n, "b2_profile_steps: buffer too small");
  std::vector<cudaEvent_t> ev(2 * n);
  for (auto& e : ev) B2_CUDA(cudaEventCreate(&e));
  std::vector<double> acc(n, 0.0);
  for (int r = 0; r < reps; ++r) {
    for (int i = 0; i < n; ++i) {
      B2_CUDA(cudaEventRecord(ev[2 * i], c->stream));
      if (run_step(c, c->steps[i])) return -1;
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

// Describes step `idx`: name, kind (0 = tensor-core conv/dense), algorithmic FLOPs and HBM bytes
// (each operand read once, output written once, at the stored precision).
int b2_step_info(b2_ctx* c, int idx, char* name, int name_cap, double* flops, double* bytes, int* kind) {
  B2_CHECK(c && name && flops && bytes && kind, "b2_step_info: null argument");
  B2_CHECK(idx >= 0 && idx < static_cast<int>(c->steps.size()), "b2_step_info: index out of range");
  const b2_ctx::Step& s = c->steps[idx];
  static const char* kKindNames[] = {"conv", "stem_pack", "maxpool", "p6_subsample", "rpn_proposals", "roialign_proposals",
                                     "head_post", "roialign_final", "roialign_mask", "mask_select"};
  std::string nm = s.kind == 0 ? s.layer->name : kKindNames[s.kind];
  *kind = s.kind;
  *flops = 0;
  *bytes = 0;
  const double esz = c->split ? 4.0 : 2.0;
  if (s.kind == 0) {
    const ConvDesc& d = s.layer->d;
    const double M = static_cast<double>(d.B) * d.Ho() * d.Wo();
    const double K = static_cast<double>(d.R) * d.S * d.Cin;
    *flops = 2.0 * M * K * d.Cout;
    const double in_px = static_cast<double>(d.B) * d.in_H * d.in_W;
    *bytes = in_px * (d.in_ld > 0 && d.in_ld < d.Cin ? d.in_ld : d.Cin) * esz + K * d.Cout * esz + M * d.Cout * (s.layer->io.out_f32 ? 4.0 : esz) +
             (s.layer->io.res_hi ? M * d.Cout * esz / (d.res_shift ? 4.0 : 1.0) : 0.0);
    nm += " [" + std::to_string(d.in_H) + "x" + std::to_string(d.in_W) + "x" + std::to_string(d.Cin) + " " +
          std::to_string(d.R) + "x" + std::to_string(d.S) + "/" + std::to_string(d.stride) + " d" +
          std::to_string(d.dil) + " ->" + std::to_string(d.Cout) + "]";
  } else if (s.kind == 1) {
    *bytes = static_cast<double>(c->img_bytes) + static_cast<double>(c->stem_u.elems()) * esz;
  } else if (s.kind == 2) {
    *bytes = (static_cast<double>(c->c1.elems()) + c->pool.elems()) * esz;
  }
  snprintf(name, name_cap, "%s", nm.c_str());
  return 0;
}
int b2_num_steps(b2_ctx* c) { return c ? static_cast<int>(c->steps.size()) : -1; }

static int ensure_graph(b2_ctx* c) {
  if (c->graph || !c->cfg.use_cuda_graph) return 0;
  cudaGraph_t g = nullptr;
  // one eager pass first: lazy one-time attribute setup must not happen inside the capture
  if (enqueue(c, B2_PHASE_ALL, false)) return -1;
  B2_CUDA(cudaStreamSynchronize(c->stream));
  B2_CUDA(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
  const int rc = enqueue(c, B2_PHASE_ALL, false);
  cudaError_t e = cudaStreamEndCapture(c->stream, &g);
  if (rc) return -1;
  B2_CUDA(e);
  B2_CUDA(cudaGraphInstantiate(&c->graph, g, 0));
  B2_CUDA(cudaGraphDestroy(g));
  return 0;
}

static int run_all(b2_ctx* c) {
  if (c->cfg.use_cuda_graph) {
    if (ensure_graph(c)) return -1;
    B2_CUDA(cudaGraphLaunch(c->graph, c->stream));
    return 0;
  }
  return enqueue(c, B2_PHASE_ALL, false);
}

// The pass left the representable range of the fp16 activation planes somewhere (the kernel flags |x| > 65504 or NaN at the
// store): the results of this call are not trustworthy.  The flag is cleared so that the next pass is judged on its own.
static int range_failed(b2_ctx* c, int idx) {
  if (c->h_range[idx] == 0) return 0;
  c->h_range[idx] = 0;
  cudaMemsetAsync(c->range_flag, 0, sizeof(unsigned int), c->stream);
  set_error("activation outside the fp16-plane range (|x| > 65504 or NaN) in a convolution output: the weights / input are "
            "not conditioned for the (hi, lo) fp16 representation (DESIGN.md section 3)");
  return -1;
}

static int copy_outputs(b2_ctx* c, float* boxes, float* probs, int32_t* labels, int32_t* valid, float* box_feat,
                        int feat_mode, cudaMemcpyKind kind) {
  const int B = c->cfg.batch, R = c->cfg.result_per_im, C = c->cfg.fpn_num_channel;
  cudaStream_t st = c->stream;
  if (boxes) B2_CUDA(cudaMemcpyAsync(boxes, c->post.final_boxes, sizeof(float) * B * R * 4, kind, st));
  if (probs) B2_CUDA(cudaMemcpyAsync(probs, c->post.final_probs, sizeof(float) * B * R, kind, st));
  if (labels) B2_CUDA(cudaMemcpyAsync(labels, c->post.final_labels, sizeof(int32_t) * B * R, kind, st));
  if (valid) B2_CUDA(cudaMemcpyAsync(valid, c->post.final_count, sizeof(int32_t) * B, kind, st));
  if (box_feat) {
    B2_CHECK(feat_mode >= 0 && feat_mode <= 3, "feat_mode must be 0 (full), 1 (mean), 2 (max) or 3 (spatial)");
    if (feat_mode == 1) {
      B2_CUDA(cudaMemcpyAsync(box_feat, c->box_feat_pooled, sizeof(float) * B * R * C, kind, st));
    } else if (feat_mode >= 2) {
      const int rows = B * R, n = feat_mode == 2 ? rows * C : rows * 49;
      if (!c->box_feat_agg) {
        c->box_feat_agg = c->alloc<float>(static_cast<size_t>(rows) * (C > 49 ? C : 49), /*zero=*/false);   // fully overwritten
        B2_CHECK(c->box_feat_agg != nullptr, "out of device memory (feature aggregation scratch)");
      }
      agg_feat_kernel<<<(n + 255) / 256, 256, 0, st>>>(c->box_feat, rows, C, feat_mode, c->box_feat_agg);
      B2_CUDA(cudaGetLastError());
      B2_CUDA(cudaMemcpyAsync(box_feat, c->box_feat_agg, sizeof(float) * n, kind, st));
    } else {
      B2_CUDA(cudaMemcpyAsync(box_feat, c->box_feat, sizeof(float) * B * R * C * 49, kind, st));
    }
  }
  return 0;
}

int b2_detect(b2_ctx* c, const void* frames_dev, float* boxes, float* probs, int32_t* labels, int32_t* valid,
              float* box_feat, int feat_mode, int sync) {
  B2_CHECK(c, "b2_detect: null ctx");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_detect: weights not loaded");
  if (frames_dev && frames_dev != c->img)
    B2_CUDA(cudaMemcpyAsync(c->img, frames_dev, c->img_bytes, cudaMemcpyDeviceToDevice, c->stream));
  if (run_all(c)) return -1;
  if (copy_outputs(c, boxes, probs, labels, valid, box_feat, feat_mode, cudaMemcpyDeviceToDevice)) return -1;
  if (sync) {
    B2_CUDA(cudaMemcpyAsync(&c->h_range[2], c->range_flag, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    return range_failed(c, 2);
  }
  return 0;
}

int b2_detect_host(b2_ctx* c, const void* frames_host, float* boxes, float* probs, int32_t* labels, int32_t* valid,
                   float* box_feat, int feat_mode) {
  B2_CHECK(c && frames_host, "b2_detect_host: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_detect_host: weights not loaded");
  B2_CUDA(cudaMemcpyAsync(c->img, frames_host, c->img_bytes, cudaMemcpyHostToDevice, c->stream));
  if (run_all(c)) return -1;
  if (copy_outputs(c, boxes, probs, labels, valid, box_feat, feat_mode, cudaMemcpyDeviceToHost)) return -1;
  B2_CUDA(cudaMemcpyAsync(&c->h_range[2], c->range_flag, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return range_failed(c, 2);
}

// Frame ingest with the resize on the device (SURVEY 8f rank 1; reference host path: frame.astype("float32") ->
// resizeImage (cv2.resize INTER_LINEAR, nn.py:1540-1545) -> feed, obj_detect_tracking.py:597-608): the uint8 source frames
// cross PCIe (4x fewer bytes than the resized float32 frames the reference feeds, no host resize), resize_u8_to_f32_kernel
// writes the float32 network input.  The caller computes the target size with get_new_hw (nn.py:1548-1560) and creates the
// context for it with input_dtype = 0.
int b2_detect_host_resize(b2_ctx* c, const uint8_t* frames_u8, int src_h, int src_w, float* boxes, float* probs,
                          int32_t* labels, int32_t* valid, float* box_feat, int feat_mode) {
  B2_CHECK(c && frames_u8, "b2_detect_host_resize: null argument");
  B2_CHECK(src_h > 0 && src_w > 0, "b2_detect_host_resize: bad source size");
  B2_CHECK(c->cfg.input_dtype == 0, "b2_detect_host_resize: the context must be created with input_dtype = 0 (float32 frames)");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_detect_host_resize: weights not loaded");
  const size_t need = static_cast<size_t>(c->cfg.batch) * src_h * src_w * 3;
  if (need > c->raw_bytes) {
    B2_CUDA(cudaStreamSynchronize(c->stream));
    if (c->raw_frames) B2_CUDA(cudaFree(c->raw_frames));
    c->raw_frames = nullptr;
    c->raw_bytes = 0;
    B2_CUDA(cudaMalloc(&c->raw_frames, need));
    c->raw_bytes = need;
  }
  B2_CUDA(cudaMemcpyAsync(c->raw_frames, frames_u8, need, cudaMemcpyHostToDevice, c->stream));
  if (resize_u8_launch(c->raw_frames, c->cfg.batch, src_h, src_w, static_cast<float*>(c->img), c->cfg.height, c->cfg.width,
                       c->stream)) return -1;
  if (run_all(c)) return -1;
  if (copy_outputs(c, boxes, probs, labels, valid, box_feat, feat_mode, cudaMemcpyDeviceToHost)) return -1;
  B2_CUDA(cudaMemcpyAsync(&c->h_range[2], c->range_flag, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return range_failed(c, 2);
}

// The resize alone (parity tests): host uint8 [n, src_h, src_w, 3] -> host float32 [n, dst_h, dst_w, 3].
int b2_resize_frames(int device, const uint8_t* frames_u8, int n, int src_h, int src_w, int dst_h, int dst_w,
                     float* out_host) {
  B2_CHECK(frames_u8 && out_host && n > 0 && src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0, "b2_resize_frames: bad argument");
  B2_CUDA(cudaSetDevice(device));
  uint8_t* d_src = nullptr;
  float* d_dst = nullptr;
  const size_t nb_src = static_cast<size_t>(n) * src_h * src_w * 3, nb_dst = static_cast<size_t>(n) * dst_h * dst_w * 3 * sizeof(float);
  B2_CUDA(cudaMalloc(&d_src, nb_src));
  cudaError_t e = cudaMalloc(&d_dst, nb_dst);
  if (e == cudaSuccess) e = cudaMemcpy(d_src, frames_u8, nb_src, cudaMemcpyHostToDevice);
  int rc = 0;
  if (e == cudaSuccess) rc = resize_u8_launch(d_src, n, src_h, src_w, d_dst, dst_h, dst_w, nullptr);
  if (e == cudaSuccess && !rc) e = cudaMemcpy(out_host, d_dst, nb_dst, cudaMemcpyDeviceToHost);
  cudaFree(d_src);
  cudaFree(d_dst);
  if (rc) return -1;
  B2_CUDA(e);
  return 0;
}

// Pipelined ingest for streaming drivers (the reference's queue-fed loop, obj_detect_tracking_multi_queuer.py:386-480):
// b2_submit_host enqueues  H2D(frames -> staging[slot]) on a copy stream, then on the compute stream
// staging[slot] -> image, the pass, and the D2H of the results into the caller's (pinned) buffers, and returns without
// waiting; b2_wait(slot) blocks until that slot's results have landed.  With two slots the upload of batch i+1 overlaps
// the pass of batch i.  Host buffers must stay valid (and should be page-locked) until b2_wait returns.
// src_h == 0: frames_host are network-input frames (b2_submit_host).  src_h > 0: uint8 source frames [B, src_h, src_w, 3]
// that the resize kernel turns into the float32 network input on the compute stream (b2_submit_host_resize).
static int submit_impl(b2_ctx* c, const void* frames_host, int src_h, int src_w, float* boxes, float* probs, int32_t* labels,
                       int32_t* valid, float* box_feat, int feat_mode, int slot) {
  B2_CHECK(c && frames_host, "b2_submit_host: null argument");
  B2_CHECK(slot == 0 || slot == 1, "b2_submit_host: slot must be 0 or 1");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_submit_host: weights not loaded");
  B2_CHECK(!c->slot_busy[slot], "b2_submit_host: slot still in flight (call b2_wait first)");
  const int B = c->cfg.batch, R = c->cfg.result_per_im, C = c->cfg.fpn_num_channel;
  const size_t nb_boxes = sizeof(float) * B * R * 4, nb_probs = sizeof(float) * B * R, nb_labels = sizeof(int32_t) * B * R;
  const size_t nb_valid = (sizeof(int32_t) * B + 255) / 256 * 256, nb_feat = sizeof(float) * B * R * C * 49;
  if (!c->copy_stream) {
    B2_CUDA(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    B2_CUDA(cudaStreamCreateWithFlags(&c->down_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      B2_CUDA(cudaMalloc(&c->stage_in[i], c->img_bytes));
      c->allocs.push_back(c->stage_in[i]);
      B2_CUDA(cudaMalloc(&c->stage_out[i], nb_boxes + nb_probs + nb_labels + nb_valid + nb_feat));
      c->allocs.push_back(c->stage_out[i]);
      B2_CUDA(cudaEventCreateWithFlags(&c->h2d_done[i], cudaEventDisableTiming));
      B2_CUDA(cudaEventCreateWithFlags(&c->staged_free[i], cudaEventDisableTiming));
      B2_CUDA(cudaEventCreateWithFlags(&c->out_done[i], cudaEventDisableTiming));
      B2_CUDA(cudaEventCreateWithFlags(&c->pass_done[i], cudaEventDisableTiming));
      B2_CUDA(cudaEventRecord(c->staged_free[i], c->stream));
    }
    if (c->cfg.use_cuda_graph && ensure_graph(c)) return -1;   // capture before anything is in flight
  }
  const size_t in_bytes = src_h > 0 ? static_cast<size_t>(B) * src_h * src_w * 3 : c->img_bytes;
  B2_CUDA(cudaStreamWaitEvent(c->copy_stream, c->staged_free[slot], 0));      // the previous use of this staging buffer
  B2_CUDA(cudaMemcpyAsync(c->stage_in[slot], frames_host, in_bytes, cudaMemcpyHostToDevice, c->copy_stream));
  B2_CUDA(cudaEventRecord(c->h2d_done[slot], c->copy_stream));
  B2_CUDA(cudaStreamWaitEvent(c->stream, c->h2d_done[slot], 0));
  if (src_h > 0) {
    if (resize_u8_launch(static_cast<const uint8_t*>(c->stage_in[slot]), B, src_h, src_w, static_cast<float*>(c->img),
                         c->cfg.height, c->cfg.width, c->stream)) return -1;
  } else {
    B2_CUDA(cudaMemcpyAsync(c->img, c->stage_in[slot], c->img_bytes, cudaMemcpyDeviceToDevice, c->stream));
  }
  B2_CUDA(cudaEventRecord(c->staged_free[slot], c->stream));
  if (run_all(c)) return -1;
  // results -> this slot's device staging (a few tens of microseconds), then off the compute stream: the download runs
  // on its own stream while the next pass is already executing
  uint8_t* so = c->stage_out[slot];
  uint8_t* d_boxes = so;
  uint8_t* d_probs = d_boxes + nb_boxes;
  uint8_t* d_labels = d_probs + nb_probs;
  uint8_t* d_valid = d_labels + nb_labels;
  uint8_t* d_feat = d_valid + nb_valid;
  const size_t feat_bytes = feat_mode == 1 || feat_mode == 2 ? sizeof(float) * B * R * C
                            : feat_mode == 3 ? sizeof(float) * B * R * 49 : nb_feat;
  if (copy_outputs(c, boxes ? reinterpret_cast<float*>(d_boxes) : nullptr, probs ? reinterpret_cast<float*>(d_probs) : nullptr,
                   labels ? reinterpret_cast<int32_t*>(d_labels) : nullptr, valid ? reinterpret_cast<int32_t*>(d_valid) : nullptr,
                   box_feat ? reinterpret_cast<float*>(d_feat) : nullptr, feat_mode, cudaMemcpyDeviceToDevice)) return -1;
  B2_CUDA(cudaMemcpyAsync(&c->h_range[slot], c->range_flag, sizeof(unsigned int), cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaEventRecord(c->pass_done[slot], c->stream));
  cudaStream_t ds = c->down_stream;
  B2_CUDA(cudaStreamWaitEvent(ds, c->pass_done[slot], 0));
  if (boxes) B2_CUDA(cudaMemcpyAsync(boxes, d_boxes, nb_boxes, cudaMemcpyDeviceToHost, ds));
  if (probs) B2_CUDA(cudaMemcpyAsync(probs, d_probs, nb_probs, cudaMemcpyDeviceToHost, ds));
  if (labels) B2_CUDA(cudaMemcpyAsync(labels, d_labels, nb_labels, cudaMemcpyDeviceToHost, ds));
  if (valid) B2_CUDA(cudaMemcpyAsync(valid, d_valid, sizeof(int32_t) * B, cudaMemcpyDeviceToHost, ds));
  if (box_feat) B2_CUDA(cudaMemcpyAsync(box_feat, d_feat, feat_bytes, cudaMemcpyDeviceToHost, ds));
  B2_CUDA(cudaEventRecord(c->out_done[slot], ds));
  c->slot_busy[slot] = true;
  return 0;
}

int b2_submit_host(b2_ctx* c, const void* frames_host, float* boxes, float* probs, int32_t* labels, int32_t* valid,
                   float* box_feat, int feat_mode, int slot) {
  return submit_impl(c, frames_host, 0, 0, boxes, probs, labels, valid, box_feat, feat_mode, slot);
}

// The streaming form of b2_detect_host_resize: uint8 source frames in (they must fit the staging buffer, i.e. at most four
// source pixels per network-input pixel), resized on the device, pipelined like b2_submit_host.
int b2_submit_host_resize(b2_ctx* c, const uint8_t* frames_u8, int src_h, int src_w, float* boxes, float* probs,
                          int32_t* labels, int32_t* valid, float* box_feat, int feat_mode, int slot) {
  B2_CHECK(c && src_h > 0 && src_w > 0, "b2_submit_host_resize: bad argument");
  B2_CHECK(c->cfg.input_dtype == 0, "b2_submit_host_resize: the context must be created with input_dtype = 0 (float32 frames)");
  B2_CHECK(static_cast<size_t>(c->cfg.batch) * src_h * src_w * 3 <= c->img_bytes,
           "b2_submit_host_resize: source frames larger than the staging buffer (more than 4 source pixels per input pixel)");
  return submit_impl(c, frames_u8, src_h, src_w, boxes, probs, labels, valid, box_feat, feat_mode, slot);
}

int b2_wait(b2_ctx* c, int slot) {
  B2_CHECK(c && (slot == 0 || slot == 1), "b2_wait: bad argument");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->slot_busy[slot], "b2_wait: nothing was submitted on this slot");
  B2_CUDA(cudaEventSynchronize(c->out_done[slot]));
  c->slot_busy[slot] = false;
  return range_failed(c, slot);
}

// RCNN_FPN_givenbox (models.py:1816-1967; get_model_feat :121-131): features of GIVEN boxes on one frame -- backbone + FPN,
// ROIAlign 7x7 of the boxes on the uncropped p2..p5 (that graph skips slice_feature_and_anchors) and the mean over the
// 7x7 bins (final_box_features [n, 256]).  The context must have batch 1; boxes are processed result_per_im at a time.
int b2_box_features(b2_ctx* c, const void* frame_host, const float* boxes_host, int n, float* feat_host) {
  B2_CHECK(c && frame_host && (n == 0 || (boxes_host && feat_host)), "b2_box_features: null argument");
  B2_CHECK(c->cfg.batch == 1, "b2_box_features: the context must be created with batch 1 (the given-box graph takes one image)");
  B2_CHECK(n >= 0, "b2_box_features: negative box count");
  B2_CUDA(cudaSetDevice(c->device));
  B2_CHECK(c->weights_loaded, "b2_box_features: weights not loaded");
  const int R = c->cfg.result_per_im, C = c->cfg.fpn_num_channel;
  if (!c->given_boxes) {
    c->given_boxes = c->alloc<float>(static_cast<size_t>(R) * 4);
    c->given_count = c->alloc<int>(1);
    c->given_feat = c->alloc<float>(static_cast<size_t>(R) * C * 49);
    c->given_pooled = c->alloc<float>(static_cast<size_t>(R) * C);
    B2_CHECK(c->given_boxes && c->given_count && c->given_feat && c->given_pooled, "out of device memory (given-box buffers)");
    B2_CUDA(cudaDeviceSynchronize());   // the zero fills of alloc() run on the legacy stream
  }
  B2_CUDA(cudaMemcpyAsync(c->img, frame_host, c->img_bytes, cudaMemcpyHostToDevice, c->stream));
  if (enqueue(c, B2_PHASE_BACKBONE | B2_PHASE_FPN, false)) return -1;
  RoiAlignParams rg = c->roi2;
  for (int i = 0; i < 4; ++i) { rg.H[i] = c->pfh[i]; rg.W[i] = c->pfw[i]; }   // uncropped levels
  rg.B = 1; rg.rois_per_image = R;
  rg.boxes = c->given_boxes; rg.count = c->given_count;
  rg.out_hi = nullptr; rg.out_lo = nullptr; rg.out_nchw = c->given_feat; rg.out_res = 7;
  for (int off = 0; off < n; off += R) {
    const int m = n - off < R ? n - off : R;
    B2_CUDA(cudaMemcpyAsync(c->given_boxes, boxes_host + static_cast<size_t>(off) * 4, sizeof(float) * m * 4,
                            cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaMemcpyAsync(c->given_count, &m, sizeof(int), cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));   // `m` lives on this stack frame
    if (roialign_launch(rg, c->stream)) return -1;
    pool_feat_kernel<<<(m * C + 255) / 256, 256, 0, c->stream>>>(c->given_feat, m, C, c->given_pooled);
    B2_CUDA(cudaGetLastError());
    B2_CUDA(cudaMemcpyAsync(feat_host + static_cast<size_t>(off) * C, c->given_pooled, sizeof(float) * m * C,
                            cudaMemcpyDeviceToHost, c->stream));
  }
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

// final_masks of the last pass (models.py:958-961): [batch][result_per_im][28][28] float32, rows beyond valid[b] are 0.
int b2_get_masks(b2_ctx* c, float* masks_host, int64_t capacity_bytes) {
  B2_CHECK(c && masks_host, "b2_get_masks: null argument");
  B2_CHECK(c->cfg.add_mask && c->final_masks, "b2_get_masks: the context was created without add_mask");
  B2_CUDA(cudaSetDevice(c->device));
  const int64_t bytes = static_cast<int64_t>(c->cfg.batch) * c->cfg.result_per_im * 784 * 4;
  B2_CHECK(capacity_bytes >= bytes, "b2_get_masks: buffer too small");
  B2_CUDA(cudaMemcpyAsync(masks_host, c->final_masks, bytes, cudaMemcpyDeviceToHost, c->stream));
  B2_CUDA(cudaStreamSynchronize(c->stream));
  return 0;
}

int b2_stage_shape(b2_ctx* c, const char* name, int64_t shape[4], int32_t* dtype) {
  B2_CHECK(c && name && shape, "b2_stage_shape: null argument");
  auto it = c->stages.find(name);
  B2_CHECK(it != c->stages.end(), std::string("unknown stage: ") + name);
  for (int i = 0; i < 4; ++i) shape[i] = it->second.shape[i];
  if (dtype) *dtype = it->second.kind == 2 ? 1 : 0;
  return 0;
}

int b2_get_stage(b2_ctx* c, const char* name, void* dst, int64_t capacity) {
  B2_CHECK(c && name && dst, "b2_get_stage: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  auto it = c->stages.find(name);
  B2_CHECK(it != c->stages.end(), std::string("unknown stage: ") + name);
  const StageRef& s = it->second;
  const int64_t n = s.shape[0] * s.shape[1] * s.shape[2] * s.shape[3];
  B2_CHECK(capacity >= n * 4, "b2_get_stage: buffer too small");
  B2_CUDA(cudaStreamSynchronize(c->stream));
  if (s.kind == 0) {
    float* tmp = nullptr;
    B2_CUDA(cudaMalloc(&tmp, n * 4));
    if (planes_to_f32(s.pl.hi, s.pl.lo, tmp, n, c->stream)) return -1;
    B2_CUDA(cudaMemcpyAsync(dst, tmp, n * 4, cudaMemcpyDeviceToHost, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    B2_CUDA(cudaFree(tmp));
  } else {
    B2_CUDA(cudaMemcpy(dst, s.ptr, n * 4, cudaMemcpyDeviceToHost));
  }
  return 0;
}

int b2_set_stage(b2_ctx* c, const char* name, const void* src, int64_t bytes) {
  B2_CHECK(c && name && src, "b2_set_stage: null argument");
  B2_CUDA(cudaSetDevice(c->device));
  if (strcmp(name, "image") == 0) {
    B2_CHECK(bytes == static_cast<int64_t>(c->img_bytes), "b2_set_stage(image): size mismatch");
    B2_CUDA(cudaMemcpyAsync(c->img, src, bytes, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
    return 0;
  }
  auto it = c->stages.find(name);
  B2_CHECK(it != c->stages.end(), std::string("unknown stage: ") + name);
  const StageRef& s = it->second;
  const int64_t n = s.shape[0] * s.shape[1] * s.shape[2] * s.shape[3];
  B2_CHECK(bytes == n * 4, "b2_set_stage: size mismatch");
  B2_CUDA(cudaStreamSynchronize(c->stream));
  if (s.kind == 0) {
    float* tmp = nullptr;
    B2_CUDA(cudaMalloc(&tmp, n * 4));
    B2_CUDA(cudaMemcpyAsync(tmp, src, n * 4, cudaMemcpyHostToDevice, c->stream));   // same stream as the kernel
    if (f32_to_planes(tmp, s.pl.hi, s.pl.lo, n, c->stream)) return -1;
    B2_CUDA(cudaStreamSynchronize(c->stream));
    B2_CUDA(cudaFree(tmp));
  } else {
    B2_CUDA(cudaMemcpyAsync(s.ptr, src, n * 4, cudaMemcpyHostToDevice, c->stream));
    B2_CUDA(cudaStreamSynchronize(c->stream));
  }
  return 0;
}

// ---- workspace for the small per-frame GEMM calls ------------------------------------------------------------------
// b2_cosine_cost / b2_distance_matrix are called once per frame (per cascade level) by the trackers.  They run out of ONE
// grow-only workspace per device with the GEMM plans cached per padded shape: a call is three uploads, four launches and
// one download on a private stream (round 1 allocated ~12 device buffers, encoded the tensor maps and freed everything
// again on every call: 48 ms per JDE frame against 1.7 ms for numpy, profiles/r2_widen_timing_before_ws.jsonl).  Operands
// are padded to the plan's shape with whatever the buffers hold (finite leftovers of earlier calls): padded rows / columns
// only produce outputs nobody reads.
struct DistWs {
  int device = -1;
  cudaStream_t stream = nullptr;
  size_t cap_a = 0, cap_b = 0, cap_rows = 0, cap_cols = 0, cap_dp = 0;
  float *d_a = nullptr, *d_b = nullptr, *d_dots = nullptr, *d_out = nullptr, *d_bias = nullptr, *d_na2 = nullptr, *d_nb2 = nullptr;
  int* d_off = nullptr;
  __half *a_hi = nullptr, *a_lo = nullptr, *b_hi = nullptr, *b_lo = nullptr;
  std::map<std::vector<int>, ConvPlan*> plans;   // key: Sp, Np, Dp, split
  int num_sms = 148;
  DistWs() = default;
  DistWs(const DistWs&) = delete;
  DistWs& operator=(const DistWs&) = delete;
  void release() {
    for (auto& kv : plans) conv_tc_plan_destroy(kv.second);
    plans.clear();
    void* ptrs[] = {d_a, d_b, d_dots, d_out, d_bias, d_na2, d_nb2, d_off, a_hi, a_lo, b_hi, b_lo};
    for (void* q : ptrs) if (q) cudaFree(q);
    d_a = d_b = d_dots = d_out = d_bias = d_na2 = d_nb2 = nullptr;
    d_off = nullptr;
    a_hi = a_lo = b_hi = b_lo = nullptr;
    cap_a = cap_b = cap_rows = cap_cols = cap_dp = 0;
  }
};
static std::map<int, DistWs> g_dist_ws;   // lives as long as the process (no CUDA calls at exit)
static std::map<int, int> g_num_sms;
static std::mutex g_dist_ws_mutex;   // one call at a time per process (the trackers are single-threaded per stream)

// Makes `w` (on `device`) hold S x D / N x D raw rows, Sp x Dp / Np x Dp operand planes, Sp x Np products, `aux` ints.
static int dist_ws_reserve(DistWs& w, int device, int S, int N, int D, int Sp, int Np, int Dp, int aux) {
  if (w.device < 0) {
    w.device = device;
    auto it = g_num_sms.find(device);
    if (it == g_num_sms.end()) {
      int n = 0;
      B2_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
      it = g_num_sms.emplace(device, n).first;
    }
    w.num_sms = it->second;
    B2_CUDA(cudaStreamCreateWithFlags(&w.stream, cudaStreamNonBlocking));
  }
  const size_t need_a = static_cast<size_t>(S) * D, need_b = static_cast<size_t>(N) * D;
  if (need_a > w.cap_a || need_b > w.cap_b || static_cast<size_t>(Sp) > w.cap_rows || static_cast<size_t>(Np) > w.cap_cols ||
      static_cast<size_t>(Dp) > w.cap_dp || static_cast<size_t>(aux) > w.cap_rows + w.cap_cols) {
    B2_CUDA(cudaStreamSynchronize(w.stream));
    const size_t o_a = w.cap_a, o_b = w.cap_b, o_r = w.cap_rows, o_c = w.cap_cols, o_d = w.cap_dp;
    w.release();                                          // the plans hold the old addresses
    auto grow = [](size_t cap, size_t need, size_t floor_) {   // only the dimension that overflowed grows (x2 head room)
      return need > cap ? std::max(need * 2, floor_) : std::max(cap, floor_);
    };
    w.cap_a = grow(o_a, need_a, 1);
    w.cap_b = grow(o_b, need_b, 1);
    w.cap_rows = grow(o_r, static_cast<size_t>(Sp), 256);
    w.cap_cols = grow(o_c, static_cast<size_t>(Np), 256);
    if (static_cast<size_t>(aux) > w.cap_rows + w.cap_cols) w.cap_rows = static_cast<size_t>(aux);
    w.cap_dp = std::max(o_d, static_cast<size_t>(Dp));
    B2_CUDA(cudaMalloc(&w.d_a, w.cap_a * 4));
    B2_CUDA(cudaMalloc(&w.d_b, w.cap_b * 4));
    B2_CUDA(cudaMalloc(&w.d_dots, w.cap_rows * w.cap_cols * 4));
    B2_CUDA(cudaMalloc(&w.d_out, w.cap_rows * w.cap_cols * 4));
    B2_CUDA(cudaMalloc(&w.d_bias, w.cap_cols * 4));
    B2_CUDA(cudaMalloc(&w.d_na2, w.cap_rows * 4));
    B2_CUDA(cudaMalloc(&w.d_nb2, w.cap_cols * 4));
    B2_CUDA(cudaMalloc(&w.d_off, (w.cap_rows + w.cap_cols + 1) * 4));
    B2_CUDA(cudaMalloc(&w.a_hi, w.cap_rows * w.cap_dp * 2));
    B2_CUDA(cudaMalloc(&w.a_lo, w.cap_rows * w.cap_dp * 2));
    B2_CUDA(cudaMalloc(&w.b_hi, w.cap_cols * w.cap_dp * 2));
    B2_CUDA(cudaMalloc(&w.b_lo, w.cap_cols * w.cap_dp * 2));
    B2_CUDA(cudaMemsetAsync(w.d_bias, 0, w.cap_cols * 4, w.stream));
    B2_CUDA(cudaMemsetAsync(w.a_hi, 0, w.cap_rows * w.cap_dp * 2, w.stream));
    B2_CUDA(cudaMemsetAsync(w.a_lo, 0, w.cap_rows * w.cap_dp * 2, w.stream));
    B2_CUDA(cudaMemsetAsync(w.b_hi, 0, w.cap_cols * w.cap_dp * 2, w.stream));
    B2_CUDA(cudaMemsetAsync(w.b_lo, 0, w.cap_cols * w.cap_dp * 2, w.stream));
    B2_CUDA(cudaStreamSynchronize(w.stream));
  }
  return 0;
}

// the [Sp rows] x [Np columns] GEMM over K = Dp on the workspace operand planes (row stride Dp)
static int dist_ws_gemm(DistWs& w, int Sp, int Np, int Dp, bool split) {
  const std::vector<int> key = {Sp, Np, Dp, split ? 1 : 0};
  auto it = w.plans.find(key);
  if (it == w.plans.end()) {
    ConvDesc d;
    d.B = 1; d.in_H = 1; d.in_W = Sp; d.Cin = Dp; d.in_pitch_H = 1; d.in_pitch_W = Sp; d.in_ld = Dp;
    d.Cout = Np; d.out_H = 1; d.out_W = Sp; d.ldc = Np;
    ConvWeights cw;
    cw.w_hi = w.b_hi; cw.w_lo = split ? w.b_lo : nullptr; cw.bias = w.d_bias; cw.Cout_pad = Np; cw.K = Dp;
    ConvIO io;
    io.in_hi = w.a_hi; io.in_lo = split ? w.a_lo : nullptr; io.out_f32 = w.d_dots;
    ConvPlan* plan = conv_tc_plan_create(d, cw, io, split, w.num_sms);
    B2_CHECK(plan != nullptr, std::string("distance workspace plan: ") + last_error());
    it = w.plans.emplace(key, plan).first;
  }
  return conv_tc_launch(it->second, w.stream);
}

static int cosine_cost_run(DistWs& w, int device, const float* gallery, const int32_t* seg_offsets, int T, const float* dets,
                           int N, int D, bool split, float* cost) {
  const int S = seg_offsets[T];
  const int Dp = (D + 63) / 64 * 64, Np = (N + 15) / 16 * 16, Sp = (S + 127) / 128 * 128;
  if (dist_ws_reserve(w, device, S, N, D, Sp, Np, Dp, T + 1)) return -1;
  cudaStream_t st = w.stream;
  B2_CUDA(cudaMemcpyAsync(w.d_a, gallery, sizeof(float) * S * D, cudaMemcpyHostToDevice, st));
  B2_CUDA(cudaMemcpyAsync(w.d_b, dets, sizeof(float) * N * D, cudaMemcpyHostToDevice, st));
  B2_CUDA(cudaMemcpyAsync(w.d_off, seg_offsets, sizeof(int) * (T + 1), cudaMemcpyHostToDevice, st));
  if (cosine_normalize_rows(w.d_a, S, D, w.a_hi, w.a_lo, Dp, st) || cosine_normalize_rows(w.d_b, N, D, w.b_hi, w.b_lo, Dp, st))
    return -1;
  if (dist_ws_gemm(w, Sp, Np, Dp, split)) return -1;
  if (cosine_segmin(w.d_dots, Np, w.d_off, T, N, w.d_out, st)) return -1;
  B2_CUDA(cudaMemcpyAsync(cost, w.d_out, sizeof(float) * T * N, cudaMemcpyDeviceToHost, st));
  B2_CUDA(cudaStreamSynchronize(st));
  return 0;
}

static int distance_matrix_run(DistWs& w, int device, const float* a, int na, const float* b, int nb, int D, int metric,
                               bool split, float* out) {
  const int Dp = (D + 63) / 64 * 64, Np = (nb + 15) / 16 * 16, Sp = (na + 127) / 128 * 128;
  if (dist_ws_reserve(w, device, na, nb, D, Sp, Np, Dp, 0)) return -1;
  cudaStream_t st = w.stream;
  B2_CUDA(cudaMemcpyAsync(w.d_a, a, sizeof(float) * na * D, cudaMemcpyHostToDevice, st));
  B2_CUDA(cudaMemcpyAsync(w.d_b, b, sizeof(float) * nb * D, cudaMemcpyHostToDevice, st));
  if (metric == 0) {
    if (cosine_normalize_rows(w.d_a, na, D, w.a_hi, w.a_lo, Dp, st) || cosine_normalize_rows(w.d_b, nb, D, w.b_hi, w.b_lo, Dp, st))
      return -1;
  } else {
    if (rows_to_planes(w.d_a, na, D, w.a_hi, w.a_lo, Dp, w.d_na2, st) || rows_to_planes(w.d_b, nb, D, w.b_hi, w.b_lo, Dp, w.d_nb2, st))
      return -1;
  }
  if (dist_ws_gemm(w, Sp, Np, Dp, split)) return -1;
  if (distance_finish(w.d_dots, Np, na, nb, metric, w.d_na2, w.d_nb2, w.d_out, st)) return -1;
  B2_CUDA(cudaMemcpyAsync(out, w.d_out, sizeof(float) * na * nb, cudaMemcpyDeviceToHost, st));
  B2_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ---- DeepSORT appearance cost ---------------------------------------------------------------
int b2_cosine_cost(int device, const float* gallery, const int32_t* seg_offsets, int T, const float* dets, int N,
                   int D, int precision, float* cost) {
  B2_CHECK(gallery && seg_offsets && dets && cost, "b2_cosine_cost: null argument");
  if (T <= 0 || N <= 0) return 0;
  B2_CHECK(D > 0 && seg_offsets[0] == 0, "b2_cosine_cost: seg_offsets must start at 0");
  for (int t = 0; t < T; ++t)
    B2_CHECK(seg_offsets[t + 1] >= seg_offsets[t], "b2_cosine_cost: seg_offsets must be non-decreasing");
  B2_CHECK(seg_offsets[T] > 0, "b2_cosine_cost: empty gallery");
  B2_CUDA(cudaSetDevice(device));
  const bool split = precision == 1;
  std::lock_guard<std::mutex> lock(g_dist_ws_mutex);
  return cosine_cost_run(g_dist_ws[device], device, gallery, seg_offsets, T, dets, N, D, split, cost);
}

// ---- distance matrix (torchreid/distance.py:6-80) ------------------------------------------------
int b2_distance_matrix(int device, const float* a, int na, const float* b, int nb, int D, int metric, int precision,
                       float* out) {
  B2_CHECK(a && b && out, "b2_distance_matrix: null argument");
  B2_CHECK(metric == 0 || metric == 1, "b2_distance_matrix: metric must be 0 (cosine) or 1 (squared euclidean)");
  if (na <= 0 || nb <= 0) return 0;
  B2_CHECK(D > 0, "b2_distance_matrix: D must be positive");
  B2_CUDA(cudaSetDevice(device));
  const bool split = precision == 1;
  std::lock_guard<std::mutex> lock(g_dist_ws_mutex);
  return distance_matrix_run(g_dist_ws[device], device, a, na, b, nb, D, metric, split, out);
}

// ---- single conv op for kernel parity tests ---------------------------------------------------
long long b2_conv_pair_launches(void) { return b2::conv_tc_pair_launches(); }

int b2_op_conv2d(int device, const float* x, const float* w, const float* bias, const float* res, int B, int H, int W,
                 int Cin, int R, int S, int Cout, int stride, int dil, int pad_t, int pad_b, int pad_l, int pad_r,
                 int relu, int res_shift, int impl, int split, int a_mode, int epi_mode, float* out) {
  B2_CHECK(x && w && out, "b2_op_conv2d: null argument");
  B2_CUDA(cudaSetDevice(device));
  ConvDesc d;
  d.B = B; d.in_H = H; d.in_W = W; d.Cin = Cin; d.in_pitch_H = H; d.in_pitch_W = W; d.in_ld = Cin;
  d.R = R; d.S = S; d.stride = stride; d.dil = dil;
  d.pad_t = pad_t; d.pad_b = pad_b; d.pad_l = pad_l; d.pad_r = pad_r;
  d.Cout = Cout; d.relu = relu; d.force_a_mode = a_mode; d.force_epi_mode = epi_mode;
  const int Ho = d.Ho(), Wo = d.Wo();
  B2_CHECK(Ho > 0 && Wo > 0, "b2_op_conv2d: empty output");
  const int Cp = (Cout + 15) / 16 * 16;
  d.out_H = Ho; d.out_W = Wo; d.ldc = Cp;
  const int rH = res_shift ? (Ho + 1) / 2 : Ho, rW = res_shift ? (Wo + 1) / 2 : Wo;
  d.res_H = rH; d.res_W = rW; d.ldr = Cp; d.res_shift = res_shift;
  const size_t nx = static_cast<size_t>(B) * H * W * Cin, K = static_cast<size_t>(R) * S * Cin;
  const size_t nw = static_cast<size_t>(Cp) * K, no = static_cast<size_t>(B) * Ho * Wo * Cp;
  const size_t nr = static_cast<size_t>(B) * rH * rW * Cp;
  // pack HWIO -> [Cout_pad][R*S*Cin]
  std::vector<float> pw(nw, 0.f), pb(Cp, 0.f);
  for (size_t k = 0; k < K; ++k)
    for (int o = 0; o < Cout; ++o) pw[static_cast<size_t>(o) * K + k] = w[k * Cout + o];
  if (bias) for (int o = 0; o < Cout; ++o) pb[o] = bias[o];
  std::vector<float> pr;
  if (res) {
    pr.assign(nr, 0.f);
    for (size_t p = 0; p < static_cast<size_t>(B) * rH * rW; ++p)
      for (int o = 0; o < Cout; ++o) pr[p * Cp + o] = res[p * Cout + o];
  }
  float *dx = nullptr, *dw = nullptr, *dr = nullptr, *dof = nullptr;
  ConvWeights cw; ConvIO io;
  __half *xh, *xl, *oh, *ol, *rh = nullptr, *rl = nullptr;
  B2_CUDA(cudaMalloc(&dx, nx * 4));
  B2_CUDA(cudaMalloc(&dw, nw * 4));
  B2_CUDA(cudaMalloc(&dof, no * 4));
  B2_CUDA(cudaMalloc(&xh, nx * 2 + 256)); B2_CUDA(cudaMalloc(&xl, nx * 2 + 256));
  B2_CUDA(cudaMalloc(&cw.w_hi, nw * 2 + 256)); B2_CUDA(cudaMalloc(&cw.w_lo, nw * 2 + 256));
  B2_CUDA(cudaMalloc(&oh, no * 2 + 256)); B2_CUDA(cudaMalloc(&ol, no * 2 + 256));
  B2_CUDA(cudaMalloc(&cw.bias, Cp * 4));
  B2_CUDA(cudaMemset(oh, 0, no * 2)); B2_CUDA(cudaMemset(ol, 0, no * 2));
  B2_CUDA(cudaMemcpy(dx, x, nx * 4, cudaMemcpyHostToDevice));
  B2_CUDA(cudaMemcpy(dw, pw.data(), nw * 4, cudaMemcpyHostToDevice));
  B2_CUDA(cudaMemcpy(cw.bias, pb.data(), Cp * 4, cudaMemcpyHostToDevice));
  cudaStream_t st = nullptr;
  if (f32_to_planes(dx, xh, xl, nx, st) || f32_to_planes(dw, cw.w_hi, cw.w_lo, nw, st)) return -1;
  if (res) {
    B2_CUDA(cudaMalloc(&dr, nr * 4));
    B2_CUDA(cudaMalloc(&rh, nr * 2 + 256)); B2_CUDA(cudaMalloc(&rl, nr * 2 + 256));
    B2_CUDA(cudaMemcpy(dr, pr.data(), nr * 4, cudaMemcpyHostToDevice));
    if (f32_to_planes(dr, rh, rl, nr, st)) return -1;
  }
  cw.Cout_pad = Cp; cw.K = static_cast<int>(K);
  if (!split) { /* keep lo planes allocated but unused */ }
  io.in_hi = xh; io.in_lo = split ? xl : nullptr;
  io.out_hi = oh; io.out_lo = split ? ol : nullptr;
  io.res_hi = rh; io.res_lo = split ? rl : nullptr;
  ConvWeights cw_use = cw;
  if (!split) cw_use.w_lo = nullptr;
  int rc = 0;
  if (impl == 0) {
    cudaDeviceProp prop;
    B2_CUDA(cudaGetDeviceProperties(&prop, device));
    ConvPlan* plan = conv_tc_plan_create(d, cw_use, io, split != 0, prop.multiProcessorCount);
    B2_CHECK(plan != nullptr, std::string("b2_op_conv2d: ") + last_error());
    rc = conv_tc_launch(plan, st);
    cudaError_t e = cudaDeviceSynchronize();
    conv_tc_plan_destroy(plan);
    if (!rc) B2_CUDA(e);
  } else {
    rc = conv_simt_launch(d, cw_use, io, split != 0, st);
    if (!rc) B2_CUDA(cudaDeviceSynchronize());
  }
  if (rc) return -1;
  if (planes_to_f32(oh, split ? ol : nullptr, dof, no, st)) return -1;
  std::vector<float> ho(no);
  B2_CUDA(cudaMemcpy(ho.data(), dof, no * 4, cudaMemcpyDeviceToHost));
  for (size_t p = 0; p < static_cast<size_t>(B) * Ho * Wo; ++p)
    for (int o = 0; o < Cout; ++o) out[p * Cout + o] = ho[p * Cp + o];
  cudaFree(dx); cudaFree(dw); cudaFree(dof); cudaFree(xh); cudaFree(xl); cudaFree(cw.w_hi); cudaFree(cw.w_lo);
  cudaFree(oh); cudaFree(ol); cudaFree(cw.bias);
  if (res) { cudaFree(dr); cudaFree(rh); cudaFree(rl); }
  return 0;
}

}  // extern "C"
