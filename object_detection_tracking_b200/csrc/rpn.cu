// RPN proposal generation: per (image, FPN level) one thread-block cluster does
//   radix-select top-k on the objectness logits (slices over the cluster's CTAs, decisions over distributed shared
//   memory) -> ordered compaction into the leader CTA -> bitonic sort
//   -> analytic anchors + box decode + clip + min-size filter -> bitmask NMS (ballot-free, smem)
// and a second kernel merges the 5 levels into the final top-k proposals.  No host sync anywhere.
//
// Reference ops replaced: get_all_anchors (utils.py:606-658, anchors recomputed analytically),
// decode_bbox_target (nn.py:1518-1538), generate_rpn_proposals (nn.py:1353-1400: tf.nn.top_k,
// clip_boxes, tf.image.non_max_suppression), generate_fpn_proposals (models.py:402-436).
#include <cooperative_groups.h>
#include <stdlib.h>

#include <algorithm>

#include "common.h"
#include "devutil.cuh"
#include "kernels.h"

namespace b2 {
namespace cg = cooperative_groups;
namespace {

__device__ __forceinline__ float level_score(const RpnParams& p, int l, int b, int i) {
  const int m = i / 3, a = i - m * 3;
  return __ldg(p.logits[l] + (static_cast<size_t>(b) * p.h[l] * p.w[l] + m) * 16 + a);
}

// One thread-block CLUSTER of kRpnCluster CTAs per (image, level): the level's anchors are split into contiguous slices,
// every CTA histograms / counts / compacts its slice, and the per-pass decisions are taken by rank 0 over distributed
// shared memory (histograms of the other CTAs are read in place; the selected keys are written straight into rank 0's
// key array).  Rank 0 then sorts, decodes and runs the NMS alone.  With one CTA per (image, level) the p2 level (172 800
// anchors at 720x1280) kept 40 blocks busy for 415 us of the 16 ms step (ncu, round 1).
constexpr int kRpnCluster = 8;

__global__ void __launch_bounds__(1024, 1) rpn_level_kernel(const __grid_constant__ RpnParams p, int KP) {
  extern __shared__ __align__(16) uint8_t sm[];
  cg::cluster_group cluster = cg::this_cluster();
  const int cs = static_cast<int>(cluster.num_blocks());
  const int rank = static_cast<int>(cluster.block_rank());
  const int l = blockIdx.x / cs, b = blockIdx.y;
  const int n = p.h[l] * p.w[l] * 3;
  const int K = min(p.topk, n);
  uint64_t* keys = reinterpret_cast<uint64_t*>(sm);                 // [KP]
  float4* boxes = reinterpret_cast<float4*>(keys + KP);             // [KP]
  float* scores = reinterpret_cast<float*>(boxes + KP);             // [KP]
  int* keep = reinterpret_cast<int*>(scores + KP);                  // [KP]
  uint32_t* mask = reinterpret_cast<uint32_t*>(keep + KP);          // [K * ceil(K/32)]
  __shared__ int hist[256];
  __shared__ int s_gt[32], s_eq[32];
  __shared__ uint32_t s_prefix, s_pmask;
  __shared__ int s_need, s_cnt;
  __shared__ int s_tot[2];          // this CTA's number of keys > kth / == kth
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // this CTA's slice [s_beg, s_end): contiguous, a multiple of 32 * 32 long so that the warp segments below stay aligned
  const int per = (((n + cs - 1) / cs) + 1023) & ~1023;
  const int s_beg = min(n, rank * per), s_end = min(n, s_beg + per);
  uint64_t* keys0 = cluster.map_shared_rank(keys, 0);
  const uint32_t* prefix0 = cluster.map_shared_rank(&s_prefix, 0);
  const uint32_t* pmask0 = cluster.map_shared_rank(&s_pmask, 0);
  const int* need0 = cluster.map_shared_rank(&s_need, 0);

  // ---- 1. radix select: key of the K-th largest score ----
  if (tid == 0) {
    s_prefix = 0;
    s_pmask = 0;
    s_need = K;
  }
  uint32_t prefix = 0, pmask = 0;
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    for (int i = tid; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = s_beg + tid; i < s_end; i += blockDim.x) {
      const uint32_t key = float_key(level_score(p, l, b, i));
      if ((key & pmask) == prefix) atomicAdd(&hist[(key >> shift) & 255], 1);
    }
    cluster.sync();                                   // every CTA's histogram of this pass is complete
    if (rank == 0) {
      if (tid < 256) {
        int sum = hist[tid];
        for (int r = 1; r < cs; ++r) sum += cluster.map_shared_rank(hist, r)[tid];
        hist[tid] = sum;
      }
      __syncthreads();
      if (tid == 0) {
        int need = s_need, cum = 0, bsel = 0;
        for (int bb = 255; bb >= 0; --bb) {
          if (cum + hist[bb] >= need) {
            bsel = bb;
            break;
          }
          cum += hist[bb];
        }
        s_need = need - cum;
        s_prefix = prefix | (static_cast<uint32_t>(bsel) << shift);
        s_pmask = pmask | (255u << shift);
      }
    }
    cluster.sync();                                   // decision published; the histograms may be cleared again
    prefix = *prefix0;
    pmask = *pmask0;
  }
  const uint32_t kth = prefix;
  const int need_eq = *need0;           // how many elements equal to kth are taken (lowest indices first)
  const int count_gt = K - need_eq;

  // ---- 2. ordered compaction (index order) of {key > kth} U first need_eq of {key == kth} into rank 0's keys ----
  const int seg = per >> 5;             // per-warp contiguous segment of the slice, a multiple of 32
  const int beg = s_beg + warp * seg, end = min(s_end, beg + seg);
  int cgt = 0, ceq = 0;
  for (int i0 = beg; i0 < end; i0 += 32) {
    const int i = i0 + lane;
    uint32_t key = 0;
    const bool in = i < end;
    if (in) key = float_key(level_score(p, l, b, i));
    cgt += __popc(__ballot_sync(0xffffffffu, in && key > kth));
    ceq += __popc(__ballot_sync(0xffffffffu, in && key == kth));
  }
  if (lane == 0) {
    s_gt[warp] = cgt;
    s_eq[warp] = ceq;
  }
  __syncthreads();
  if (tid == 0) {
    int a = 0, e = 0;
    for (int w = 0; w < 32; ++w) {
      const int ta = s_gt[w], te = s_eq[w];
      s_gt[w] = a;
      s_eq[w] = e;
      a += ta;
      e += te;
    }
    s_tot[0] = a;
    s_tot[1] = e;
  }
  if (rank == 0)
    for (int i = K + tid; i < KP; i += blockDim.x) keys[i] = ~0ull;
  cluster.sync();                                     // totals of every CTA visible
  int gbase = s_gt[warp], ebase = s_eq[warp];
  for (int r = 0; r < rank; ++r) {                    // slices are in index order: ranks below come first
    const int* t = cluster.map_shared_rank(s_tot, r);
    gbase += t[0];
    ebase += t[1];
  }
  const uint32_t lt = (1u << lane) - 1;
  for (int i0 = beg; i0 < end; i0 += 32) {
    const int i = i0 + lane;
    uint32_t key = 0;
    float sc = 0.f;
    const bool in = i < end;
    if (in) {
      sc = level_score(p, l, b, i);
      key = float_key(sc);
    }
    const uint32_t mg = __ballot_sync(0xffffffffu, in && key > kth);
    const uint32_t me = __ballot_sync(0xffffffffu, in && key == kth);
    if (in && key > kth) keys0[gbase + __popc(mg & lt)] = desc_key(sc, i);
    if (in && key == kth) {
      const int r = ebase + __popc(me & lt);
      if (r < need_eq) keys0[count_gt + r] = desc_key(sc, i);
    }
    gbase += __popc(mg);
    ebase += __popc(me);
  }
  cluster.sync();                                     // rank 0 owns all selected keys; nobody touches remote memory after this
  if (rank != 0) return;
  // ---- 3. sort candidates: score descending, index ascending ----
  block_bitonic_sort(keys, KP);

  // ---- 4. decode + clip + min-size filter, order-preserving compaction ----
  bool valid = false;
  float4 bx = make_float4(0, 0, 0, 0);
  float sc = 0.f;
  if (tid < K) {
    const int i = static_cast<int>(keys[tid] & 0xffffffffu);
    const int m = i / 3, a = i - m * 3;
    const int y = m / p.w[l], x = m - y * p.w[l];
    const float* row = p.logits[l] + (static_cast<size_t>(b) * p.h[l] * p.w[l] + m) * 16;
    sc = __ldg(row + a);
    const float tx = __ldg(row + 3 + a * 4), ty = __ldg(row + 4 + a * 4);
    const float tw = __ldg(row + 5 + a * 4), th = __ldg(row + 6 + a * 4);
    // anchor = cell anchor + shift, then +1 on x2,y2 (utils.py:633-657); all exact small integers in fp32
    const float sx = static_cast<float>(x) * p.stride[l], sy = static_cast<float>(y) * p.stride[l];
    const float ax1 = p.cell[l][a][0] + sx, ay1 = p.cell[l][a][1] + sy;
    const float ax2 = p.cell[l][a][2] + sx + 1.f, ay2 = p.cell[l][a][3] + sy + 1.f;
    const float wa = __fsub_rn(ax2, ax1), ha = __fsub_rn(ay2, ay1);
    const float xa = __fmul_rn(__fadd_rn(ax2, ax1), 0.5f), ya = __fmul_rn(__fadd_rn(ay2, ay1), 0.5f);
    const float wb = __fmul_rn(expf(fminf(tw, p.decode_clip)), wa);
    const float hb = __fmul_rn(expf(fminf(th, p.decode_clip)), ha);
    const float xb = __fadd_rn(__fmul_rn(tx, wa), xa), yb = __fadd_rn(__fmul_rn(ty, ha), ya);
    float x1 = __fsub_rn(xb, __fmul_rn(wb, 0.5f)), y1 = __fsub_rn(yb, __fmul_rn(hb, 0.5f));
    float x2 = __fadd_rn(xb, __fmul_rn(wb, 0.5f)), y2 = __fadd_rn(yb, __fmul_rn(hb, 0.5f));
    x1 = fminf(fmaxf(x1, 0.f), p.img_w);
    y1 = fminf(fmaxf(y1, 0.f), p.img_h);
    x2 = fminf(fmaxf(x2, 0.f), p.img_w);
    y2 = fminf(fmaxf(y2, 0.f), p.img_h);
    bx = make_float4(x1, y1, x2, y2);
    // single-image graph drops w/h <= rpn_min_size (nn.py:1375-1380); the batch graph does not (nn.py:1441-1455)
    valid = p.multi ? true : ((__fsub_rn(x2, x1) > p.min_size) && (__fsub_rn(y2, y1) > p.min_size));
  }
  __syncthreads();   // keys fully consumed before boxes/scores are written (separate arrays, but keep order clear)
  const uint32_t vb = __ballot_sync(0xffffffffu, valid);
  if (lane == 0) s_gt[warp] = __popc(vb);
  __syncthreads();
  if (tid == 0) {
    int a = 0;
    for (int w = 0; w < 32; ++w) {
      const int t = s_gt[w];
      s_gt[w] = a;
      a += t;
    }
    s_cnt = a;
  }
  __syncthreads();
  const int nv = s_cnt;
  if (valid) {
    const int pos = s_gt[warp] + __popc(vb & lt);
    boxes[pos] = bx;
    scores[pos] = sc;
  }
  __syncthreads();

  // ---- 5. NMS (IoU > thr suppresses), keep at most topk ----
  const int kept = block_nms_sorted(boxes, nv, p.nms_thr, p.topk, mask, keep, &s_cnt);

  float4* ob = reinterpret_cast<float4*>(p.lvl_boxes) + (static_cast<size_t>(b) * 5 + l) * p.topk;
  float* os = p.lvl_scores + (static_cast<size_t>(b) * 5 + l) * p.topk;
  for (int j = tid; j < kept; j += blockDim.x) {
    ob[j] = boxes[keep[j]];
    os[j] = scores[keep[j]];
  }
  if (tid == 0) p.lvl_count[b * 5 + l] = kept;
}

// Merge: concat the 5 levels (level order, selection order inside a level), take top-k by score
// (ties -> lower concat position), canonical order = score descending.  models.py:425-434.
// Batch graph (models.py:2490-2520): the levels are zero-padded to topk each (box 0, score 0) before the
// top-k -- so padding outranks negative logits -- and zero-area boxes are dropped afterwards.
__global__ void __launch_bounds__(1024, 1) rpn_merge_kernel(const __grid_constant__ RpnParams p, int KP2) {
  extern __shared__ __align__(16) uint8_t sm[];
  uint64_t* keys = reinterpret_cast<uint64_t*>(sm);   // [KP2]
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __shared__ int cnt[5];
  __shared__ int wsum[32];
  __shared__ int s_total;
  if (tid < 5) cnt[tid] = p.lvl_count[b * 5 + tid];
  for (int i = tid; i < KP2; i += blockDim.x) keys[i] = ~0ull;
  __syncthreads();
  int total = 0;
  for (int l = 0; l < 5; ++l) {
    const float* s = p.lvl_scores + (static_cast<size_t>(b) * 5 + l) * p.topk;
    const int n = p.multi ? p.topk : cnt[l];
    for (int j = tid; j < n; j += blockDim.x)
      keys[l * p.topk + j] = desc_key(j < cnt[l] ? s[j] : 0.f, static_cast<uint32_t>(l * p.topk + j));
    total += n;
  }
  block_bitonic_sort(keys, KP2);
  const int K = min(total, p.topk);
  // gather the selected entries (one per thread), then order-preserving compaction of the non-degenerate ones
  float4 bx = make_float4(0, 0, 0, 0);
  float sc = 0.f;
  bool keep = false;
  if (tid < K) {
    const int pos = static_cast<int>(keys[tid] & 0xffffffffu);
    const int l = pos / p.topk, j = pos - l * p.topk;
    if (j < cnt[l]) {
      const size_t src = (static_cast<size_t>(b) * 5 + l) * p.topk + j;
      bx = reinterpret_cast<const float4*>(p.lvl_boxes)[src];
      sc = p.lvl_scores[src];
    }
    keep = p.multi ? (__fmul_rn(__fsub_rn(bx.w, bx.y), __fsub_rn(bx.z, bx.x)) > 0.f) : true;
  }
  const uint32_t vb = __ballot_sync(0xffffffffu, keep);
  if (lane == 0) wsum[warp] = __popc(vb);
  __syncthreads();
  if (tid == 0) {
    int a = 0;
    for (int w = 0; w < 32; ++w) {
      const int t = wsum[w];
      wsum[w] = a;
      a += t;
    }
    s_total = a;
  }
  __syncthreads();
  float4* ob = reinterpret_cast<float4*>(p.prop_boxes) + static_cast<size_t>(b) * p.topk;
  float* os = p.prop_scores + static_cast<size_t>(b) * p.topk;
  if (keep) {
    const int o = wsum[warp] + __popc(vb & ((1u << lane) - 1));
    ob[o] = bx;
    os[o] = sc;
  }
  for (int j = s_total + tid; j < p.topk; j += blockDim.x) {
    ob[j] = make_float4(0, 0, 0, 0);
    os[j] = 0.f;
  }
  if (tid == 0) p.prop_count[b] = s_total;
}

int next_pow2(int v) {
  int p = 1;
  while (p < v) p <<= 1;
  return p;
}

}  // namespace

int rpn_proposals_launch(const RpnParams& p, cudaStream_t s) {
  B2_CHECK(p.topk >= 1 && p.topk <= 1024, "rpn: post-NMS top-k must be in [1, 1024]");
  const int KP = next_pow2(p.topk);
  const int words = (p.topk + 31) / 32;
  const size_t smem1 = static_cast<size_t>(KP) * (8 + 16 + 4 + 4) + static_cast<size_t>(p.topk) * words * 4;
  const int KP2 = next_pow2(5 * p.topk);
  const size_t smem2 = static_cast<size_t>(KP2) * 8;
  static bool attr_set = false;
  if (!attr_set) {
    B2_CUDA(cudaFuncSetAttribute(rpn_level_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    B2_CUDA(cudaFuncSetAttribute(rpn_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    attr_set = true;
  }
  B2_CHECK(smem1 <= 200 * 1024 && smem2 <= 200 * 1024, "rpn: top-k too large for shared memory");
  {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(5 * kRpnCluster, p.B);
    cfg.blockDim = dim3(1024);
    cfg.dynamicSmemBytes = smem1;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = kRpnCluster;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    B2_CUDA(cudaLaunchKernelEx(&cfg, rpn_level_kernel, p, KP));
  }
  rpn_merge_kernel<<<p.B, 1024, smem2, s>>>(p, KP2);
  B2_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace b2
