// Implicit-GEMM convolution on the 5th-gen tensor cores (tcgen05 + TMEM), operands staged by TMA.
//
//   D[M = B*Ho*Wo pixels, N = Cout] = A[M, K = R*S*Cin] * W[N, K]^T   (+bias, +residual, ReLU)
//
// * A is never materialised: each K-block (one filter tap x 64 input channels) of a 128-pixel tile
//   is fetched straight from the NHWC activation tensor by ONE TMA im2col load
//   (cp.async.bulk.tensor.4d...im2col): padding, stride, dilation and the wrap of a pixel run across
//   image rows / batch images are all resolved by the tensor map (zero fill outside the image).
// * W is pre-packed [Cout][R][S][Cin] (K-major); a 2D tiled TMA load brings block_n x 64 per K-block.
// * Both land in shared memory in the 128-byte-swizzled K-major layout tcgen05.mma consumes directly.
// * One elected thread issues tcgen05.mma (M=128, N=block_n, K=16); accumulators live in TMEM
//   (double buffered: the epilogue of tile i overlaps the main loop of tile i+1).
// * Warp roles (256 threads): warp0 = TMA producer, warp1 = MMA issuer, warp2 = TMEM allocator,
//   warps4-7 = epilogue (TMEM -> registers -> bias/residual/ReLU -> HBM).
// * Persistent: grid = min(#tiles, #SMs), static round-robin tile schedule.
// * SPLIT precision: every operand is an fp16 pair (hi, lo') with x = hi + lo'/2048.  Three MMAs per
//   K-step -- acc0 += Ahi*Bhi ; acc1 += Ahi*Blo' + Alo'*Bhi -- and D = acc0 + acc1/2048 recover
//   ~fp32 products on the fp16 tensor pipe (needed for the 1e-3 box parity of the north star).
//
// Reference ops replaced: nn.conv2d (nn.py:337-381) + BatchNorm inference (nn.py:1771-1774, folded into
// weights/bias) + ReLU (nn.py:606-613) + residual add (nn.py:519-521) + FPN upsample-add
// (nn.py:989-996) + dense (nn.py:730-774).
#include <stdlib.h>

#include <vector>

#include "common.h"
#include "ptx.cuh"

namespace b2 {

namespace {

constexpr int kBlockM = 128;
constexpr int kBlockK = 64;                 // fp16 elements = one 128-byte swizzle row
constexpr int kABytes = kBlockM * kBlockK * 2;   // 16 KB
constexpr int kUmmaK = 16;
constexpr int kEpiHalves = 2;               // column halves of a tile handled by separate epilogue warp quartets
constexpr int kEpiWarps = 4 * kEpiHalves;   // warps 4..: TMEM lane quarter = warp & 3, column half = (warp - 4) >> 2
constexpr int kThreads = 128 + kEpiWarps * 32;
constexpr int kTmemCols = 512;
constexpr int kMaxStages = 8;
constexpr int kSmemBudget = 224 * 1024;     // pipeline stages + epilogue staging (alignment slack and barriers on top)

struct ConvTcParams {
  int M, Ho, Wo, HoWo;
  int stride, dil, lower_h, lower_w;
  int S, cin_blocks, num_kb;
  int block_n, num_n_blocks, num_tiles;
  int a_mode;   // 0 = A is a plain [M][Cin] matrix (2D tiled TMA), 1 = im2col TMA
  uint32_t idesc;
  uint32_t b_bytes, stage_bytes;
  int num_stages;
  __half* out_hi;
  __half* out_lo;
  float* out_f32;
  int ldc, out_H, out_W, off_h, off_w;
  const float* bias;
  const __half* res_hi;
  const __half* res_lo;
  int ldr, res_H, res_W, res_shift;
  int relu;
  int acc_kb;        // ACC: K-blocks per tensor-core accumulation chunk
  int acc_ring;      // ACC: chunk accumulators in the TMEM ring (2 for 128-column tiles, 6 for 64-column tiles)
  int acc_stride;    // ACC: TMEM columns per accumulator (ring at 0.., the two correction accumulators after it)
  float acc_delta;   // ACC: relative compensation of the tensor-core accumulator's truncation (kAccDelta)
  unsigned int* range_flag;   // ORed with 1 when a plane output exceeds the fp16 range (nullptr = not monitored)
  int epi_mode;      // 0 = direct global loads/stores per thread, 1 = TMA-staged (residual in, result out)
  int epi_grp;       // staged: 16-column chunks per fence / barrier / store group (1 or 2)
  int epi_slots;     // staged: group slots in each column half's staging ring (2, or 3 when a residual is prefetched)
  int epi_wide;      // staged, epi_grp == 2: a group is one [128 rows][32 fp16] box per plane (64-byte swizzle, one TMA op)
  uint32_t epi_chunk_bytes;   // staged: bytes of one chunk buffer (4 KB hi plane, + 4 KB lo plane in split precision)
  uint32_t epi_off;  // byte offset of the epilogue staging buffers inside the tile area
  int num_pair_tiles;   // PAIR: tiles of 256 rows (two m-blocks, one per CTA of the pair) x block_n columns
};

constexpr int kEpiSlotsMax = 3;
constexpr int kEpiPlaneBytes = kBlockM * 16 * 2;   // 128 rows x 16 fp16 = 4 KB per plane

__device__ __forceinline__ uint32_t pack_half2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

// 16 consecutive output channels of one pixel (v = accumulator value): bias, residual, activation, store
// (fp16 hi/lo planes or fp32) straight to global memory.
template <bool SPLIT, bool SWISH>
__device__ __forceinline__ void epilogue_chunk16(const ConvTcParams& p, float (&v)[16], size_t opix, size_t rpix, int n,
                                                 float& amax) {
  const float4* b4 = reinterpret_cast<const float4*>(p.bias + n);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float4 b = __ldg(b4 + j);
    v[4 * j + 0] += b.x;
    v[4 * j + 1] += b.y;
    v[4 * j + 2] += b.z;
    v[4 * j + 3] += b.w;
  }
  if (p.res_hi != nullptr) {
    const uint4* r4 = reinterpret_cast<const uint4*>(p.res_hi + rpix * p.ldr + n);
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      uint4 r = __ldg(r4 + j);
      const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float2 f = __half22float2(h[t]);
        v[8 * j + 2 * t] += f.x;
        v[8 * j + 2 * t + 1] += f.y;
      }
    }
    if (SPLIT && p.res_lo != nullptr) {
      const uint4* l4 = reinterpret_cast<const uint4*>(p.res_lo + rpix * p.ldr + n);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        uint4 r = __ldg(l4 + j);
        const __half2* h = reinterpret_cast<const __half2*>(&r);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          float2 f = __half22float2(h[t]);
          v[8 * j + 2 * t] = fmaf(f.x, kLoInv, v[8 * j + 2 * t]);
          v[8 * j + 2 * t + 1] = fmaf(f.y, kLoInv, v[8 * j + 2 * t + 1]);
        }
      }
    }
  }
  if (p.relu == 1) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.0f);
  } else if (SWISH && p.relu == 2) {   // swish: x * sigmoid(x) -- only in the SWISH instantiations (EfficientDet): the
    // accurate expf + division are ~30 instructions per element, 2000 per kernel once inlined into every chunk copy
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = __fmul_rn(v[j], 1.f / (1.f + expf(-v[j])));   // x * sigmoid(x) as the other kernels compute it
  }
  if (p.out_f32 != nullptr) {
    float4* o = reinterpret_cast<float4*>(p.out_f32 + opix * p.ldc + n);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    return;
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) amax = fmaxf(amax, fabsf(v[j]));
  uint32_t hi[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) hi[j] = pack_half2(v[2 * j], v[2 * j + 1]);
  uint4* oh = reinterpret_cast<uint4*>(p.out_hi + opix * p.ldc + n);
  oh[0] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  oh[1] = make_uint4(hi[4], hi[5], hi[6], hi[7]);
  if (SPLIT && p.out_lo != nullptr) {
    uint32_t lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float2 h = __half22float2(*reinterpret_cast<__half2*>(&hi[j]));
      lo[j] = pack_half2((v[2 * j] - h.x) * kLoScale, (v[2 * j + 1] - h.y) * kLoScale);
    }
    uint4* ol = reinterpret_cast<uint4*>(p.out_lo + opix * p.ldc + n);
    ol[0] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    ol[1] = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
}

// Same math on a chunk whose residual sits in (and whose result goes back to) a swizzled shared-memory staging box:
// hi0 / hi1 (lo0 / lo1 for the lo plane) point at this thread's two 16-byte cells (channels 0-7 and 8-15 of the chunk).
template <bool SPLIT, bool SWISH>
__device__ __forceinline__ void epilogue_chunk16_smem(const ConvTcParams& p, float (&v)[16], uint4* hi0, uint4* hi1,
                                                      uint4* lo0, uint4* lo1, int n, bool has_res, bool has_res_lo,
                                                      float& amax) {
  const float4* b4 = reinterpret_cast<const float4*>(p.bias + n);
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float4 b = __ldg(b4 + j);
    v[4 * j + 0] += b.x;
    v[4 * j + 1] += b.y;
    v[4 * j + 2] += b.z;
    v[4 * j + 3] += b.w;
  }
  if (has_res) {
    uint4 r[2] = {*hi0, *hi1};
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const __half2* h = reinterpret_cast<const __half2*>(&r[j]);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        float2 f = __half22float2(h[t]);
        v[8 * j + 2 * t] += f.x;
        v[8 * j + 2 * t + 1] += f.y;
      }
    }
    if (SPLIT && has_res_lo) {
      uint4 l[2] = {*lo0, *lo1};
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const __half2* h = reinterpret_cast<const __half2*>(&l[j]);
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          float2 f = __half22float2(h[t]);
          v[8 * j + 2 * t] = fmaf(f.x, kLoInv, v[8 * j + 2 * t]);
          v[8 * j + 2 * t + 1] = fmaf(f.y, kLoInv, v[8 * j + 2 * t + 1]);
        }
      }
    }
  }
  if (p.relu == 1) {
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.0f);
  } else if (SWISH && p.relu == 2) {   // swish: x * sigmoid(x) -- only in the SWISH instantiations (EfficientDet): the
    // accurate expf + division are ~30 instructions per element, 2000 per kernel once inlined into every chunk copy
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = __fmul_rn(v[j], 1.f / (1.f + expf(-v[j])));   // x * sigmoid(x) as the other kernels compute it
  }
#pragma unroll
  for (int j = 0; j < 16; ++j) amax = fmaxf(amax, fabsf(v[j]));
  uint32_t hi[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) hi[j] = pack_half2(v[2 * j], v[2 * j + 1]);
  *hi0 = make_uint4(hi[0], hi[1], hi[2], hi[3]);
  *hi1 = make_uint4(hi[4], hi[5], hi[6], hi[7]);
  if (SPLIT) {
    uint32_t lo[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float2 h = __half22float2(*reinterpret_cast<__half2*>(&hi[j]));
      lo[j] = pack_half2((v[2 * j] - h.x) * kLoScale, (v[2 * j + 1] - h.y) * kLoScale);
    }
    *lo0 = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    *lo1 = make_uint4(lo[4], lo[5], lo[6], lo[7]);
  }
}

// ACC (split precision only): the tensor core adds into its fp32 accumulator with truncation (round
// toward zero), a bias that grows with the number of accumulation steps (K/16) and compounds through 100+
// layers.  With ACC the hi*hi accumulator is restarted every kAccChunkKb K-blocks in alternating TMEM
// buffers and the epilogue warps sum the chunk results in registers with round-to-nearest fp32 adds
// (overlapped with the MMAs of the next chunk), which brings the result to CUDA-core fp32 accuracy.
constexpr int kAccChunkKb = 1;   // default: restart every K-block (64 K-elements = 4 truncating accumulations)
// The (three) truncating adds that remain inside a chunk of four tcgen05.mma shrink every chunk sum toward zero by a small
// relative amount, i.e. the whole conv output by the same factor (sum_q t_q (1 - eta) = (1 - eta) sum_q t_q).  Measured on
// the 720x1280 R101 pass against the float64 evaluation of the same graph: the magnitudes of c2..c5 come out 1.8e-7 ...
// 9.2e-7 too small (the float32 CPU port: +5e-8 ... +1e-9), and that bias IS the error: max |c5 - exact| = 9.5e-7 relative.
// fmaf(v, kAccDelta, v) (one FFMA per output) gives the loss back: for delta in [2^-24, 1.5 * 2^-24) = [5.96e-8, 8.94e-8)
// the product is between half an ulp and one and a half ulps of v for every mantissa, so the result is v moved away from
// zero by exactly one ulp (0.72 * 2^-23 = 8.6e-8 relative on average); smaller values act on part of the mantissa range,
// values below 2.98e-8 are no-ops.  With it the magnitude bias of c2..c5 is +3e-8 ... +7e-8, c5 is 5.0e-7 ... 6.1e-7 from
// the exact values (the float32 port: 5.0e-7 ... 5.8e-7) and the final boxes move from 6.1e-4 to 3.1e-4 ... 3.7e-4 px
// from the exact ones (the float32 port: 2.4e-4 ... 4.9e-4).  Sweeps: profiles/r2_acc_delta_sweep.txt.
constexpr float kAccDelta = 6.8e-8f;
constexpr float kAccDelta2 = 1.7e-7f;   // chunks of two K-blocks (seven truncating adds): bias -1.6e-6 at c5 without it
constexpr int kAccRingMax = 6;
constexpr int kAccMaxChunks = 8 / kEpiHalves; // ACC tiles are at most 128 columns wide -> chunks of 16 per column half

// mbarrier wait of the PAIR kernel.  Build variant -DB2_PAIR_DIAG (bring-up of the two-CTA barrier protocol without a
// local GPU): a wait that lasts longer than ~0.5 s records who waited for what (role << 28 | CTA rank << 27 | tile << 8 |
// K-block) in g_pair_diag and every wait of the grid (and of later launches) returns at once, so a protocol error ends as a
// report on the host (conv_tc_launch) instead of a hung box.
#ifdef B2_PAIR_DIAG
__device__ unsigned int g_pair_diag[2];
#endif
template <bool PAIR>
__device__ __forceinline__ void mbar_wait_r(uint64_t* bar, uint32_t parity, uint32_t role, uint32_t crank, int tile, int kb) {
#ifdef B2_PAIR_DIAG
  if (PAIR) {
    if (*reinterpret_cast<volatile unsigned int*>(&g_pair_diag[0]) != 0u) return;
    const long long t0 = clock64();
    for (uint32_t spin = 0;; ++spin) {
      if (mbar_try_wait(bar, parity)) return;
      if ((spin & 1023u) == 1023u) {
        if (*reinterpret_cast<volatile unsigned int*>(&g_pair_diag[0]) != 0u) return;
        if (clock64() - t0 > 1000000000LL) {
          atomicCAS(&g_pair_diag[0], 0u, (role << 28) | (crank << 27) | ((static_cast<uint32_t>(tile) & 0x7FFFFu) << 8) |
                                             (static_cast<uint32_t>(kb) & 0xFFu));
          return;
        }
      }
    }
  }
#endif
  mbar_wait(bar, parity);
}

// ACC drain: fold this thread's share (my_n chunks of 16 columns of its row) of one chunk accumulator into the
// running sums with round-to-nearest adds.  All tcgen05.ld are in flight before the single wait; the accumulator is
// handed back to the MMA issuer as soon as the values sit in registers, before the adds.
// PAIR: the accumulator belongs to the pair's MMA issuer, which runs in the even CTA and waits on ITS barrier for the
// epilogue warps of both CTAs.
template <bool FMA_LO, bool PAIR>
__device__ __forceinline__ void acc_fold(float (&sums)[kAccMaxChunks * 16], uint32_t tsrc, int my_n, uint64_t* release_bar,
                                         int lane) {
  auto release = [&]() {
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (PAIR) mbar_arrive_cluster(mapa_u32(smem_u32(release_bar), 0));
      else mbar_arrive(release_bar);
    }
  };
  auto add = [&](int u, const uint32_t (&t)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i)
      sums[u * 16 + i] = FMA_LO ? fmaf(__uint_as_float(t[i]), kLoInv, sums[u * 16 + i])
                                : __fadd_rn(sums[u * 16 + i], __uint_as_float(t[i]));
  };
  if (my_n == 0) release();
#pragma unroll
  for (int u0 = 0; u0 < kAccMaxChunks; u0 += 2) {
    if (u0 < my_n) {
      uint32_t t0[16], t1[16];
      tmem_ld_32x32b_x16(tsrc + u0 * 16, t0);
      if (u0 + 1 < my_n) tmem_ld_32x32b_x16(tsrc + (u0 + 1) * 16, t1);
      tmem_ld_wait();
      if (u0 + 2 >= my_n) release();   // last batch: the accumulator now sits in registers
      add(u0, t0);
      if (u0 + 1 < my_n) add(u0 + 1, t1);
    }
  }
}

// PAIR (split + ACC only): the grid is launched in clusters of two CTAs that share 256-row tiles through
// tcgen05.mma.cta_group::2 -- CTA r of a pair loads the A rows of m-block 2*mp + r and HALF of the tile's B rows, the even
// CTA's MMA warp issues for both, each CTA finds its own 128 x block_n accumulators in its own TMEM, so everything after
// the MMA (chunk drains, output stage) is the single-CTA code.  Barrier plumbing of the pair: all operand loads count on
// the leader's full barrier (it expects both CTAs' bytes); tcgen05.commit multicasts every completion (stage free, chunk
// ready, tile ready) to the same barrier in both CTAs; the "accumulator drained" barriers live in the leader and collect
// the epilogue warps of both CTAs.
template <bool SPLIT, bool ACC, bool SWISH, bool PAIR = false>
__global__ void __launch_bounds__(kThreads, 1)
conv_tc_kernel(const __grid_constant__ CUtensorMap tmA_hi, const __grid_constant__ CUtensorMap tmA_lo,
               const __grid_constant__ CUtensorMap tmB_hi, const __grid_constant__ CUtensorMap tmB_lo,
               const __grid_constant__ CUtensorMap tmO_hi, const __grid_constant__ CUtensorMap tmO_lo,
               const __grid_constant__ CUtensorMap tmR_hi, const __grid_constant__ CUtensorMap tmR_lo,
               const __grid_constant__ ConvTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 128B swizzle atoms need 1024-byte aligned tiles
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* tiles = smem;
  const uint32_t slot_bytes = static_cast<uint32_t>(p.epi_grp) * p.epi_chunk_bytes;
  const uint32_t ring_bytes = static_cast<uint32_t>(p.epi_slots) * slot_bytes;   // per column half
  uint64_t* bars = reinterpret_cast<uint64_t*>(tiles + p.epi_off + kEpiHalves * ring_bytes);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tmem_full = bars + 2 * kMaxStages;
  uint64_t* tmem_empty = bars + 2 * kMaxStages + 2;
  uint64_t* res_full = bars + 2 * kMaxStages + 4;                       // [2 halves][kEpiSlotsMax]
  uint64_t* c_full = bars + 2 * kMaxStages + 4 + 2 * kEpiSlotsMax;      // [kAccRingMax] ACC chunk accumulator ready
  uint64_t* c_empty = c_full + kAccRingMax;                             // [kAccRingMax] ACC chunk accumulator drained
  uint64_t* grp_ready = c_empty + kAccRingMax;                          // [2 halves][kEpiSlotsMax] staged group written by its four warps
  uint64_t* slot_free = grp_ready + kEpiHalves * kEpiSlotsMax;          // [2 halves][kEpiSlotsMax] store of the slot has read it (no-residual layers)
  uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(slot_free + kEpiHalves * kEpiSlotsMax);
  uint8_t* epi = tiles + p.epi_off;

  // broadcast from lane 0 so that the compiler treats the warp index (and everything derived from it) as warp-uniform
  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA_hi);
    tma_prefetch_desc(&tmB_hi);
    if (SPLIT) {
      tma_prefetch_desc(&tmA_lo);
      tma_prefetch_desc(&tmB_lo);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < p.num_stages; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], PAIR ? 2 * kEpiWarps : kEpiWarps);   // one arrive per epilogue warp (of both CTAs)
    }
    for (int i = 0; i < 2 * kEpiSlotsMax; ++i) mbar_init(&res_full[i], 1);
    for (int i = 0; i < kAccRingMax; ++i) {
      mbar_init(&c_full[i], 1);
      mbar_init(&c_empty[i], PAIR ? 2 * kEpiWarps : kEpiWarps);
    }
    for (int i = 0; i < kEpiHalves * kEpiSlotsMax; ++i) {
      mbar_init(&grp_ready[i], 4);     // one arrive per epilogue warp of the half
      mbar_init(&slot_free[i], 1);
    }
    fence_mbar_init();
    fence_proxy_async();
  }
  if (warp == 2) {
    if (PAIR) {
      tmem_alloc_pair(tmem_holder, kTmemCols);
      tmem_relinquish_pair();
    } else {
      tmem_alloc(tmem_holder, kTmemCols);
      tmem_relinquish();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync();   // the peer's barriers are initialised before anything of this CTA signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_holder;
  if (tmem_base != 0) __trap();   // the MMA issuer addresses TMEM from column 0 / lane 0 (whole-TMEM allocation)
  // tile schedule: static round robin over CTAs (over CTA pairs in PAIR mode: pair tile = (m-block pair, n-block))
  const uint32_t crank = PAIR ? cluster_ctarank() : 0u;
  const int tile_first = PAIR ? static_cast<int>(blockIdx.x >> 1) : static_cast<int>(blockIdx.x);
  const int tile_step = PAIR ? static_cast<int>(gridDim.x >> 1) : static_cast<int>(gridDim.x);
  const int tile_count = PAIR ? p.num_pair_tiles : p.num_tiles;

  const uint32_t a_lo_off = kABytes;
  const uint32_t b_hi_off = SPLIT ? 2 * kABytes : kABytes;
  const uint32_t b_lo_off = b_hi_off + p.b_bytes;
  // accumulator stage s: acc0 at column s*256, acc1 (split) at s*256 + 128
  const uint32_t acc_stage_cols = 256;

  // ACC: the epilogue warps hold 64 running sums per thread on top of the output-stage state; take registers from the
  // (tiny) producer / MMA warpgroup.  The CTA is launched with 384 x 168 = 64512 registers; 128 x 56 + 256 x 224 = 64512
  // (the increase must fit in what the decrease freed, or setmaxnreg.inc never returns).
  if (warp < 4) {
   if (ACC) setmaxnreg_dec<56>();
   if (warp == 0) {
    // ===================== TMA producer =====================
    // converged warp, one elected lane issues (uniform-register operands, see the MMA issuer)
    {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = tile_first; tile < tile_count; tile += tile_step) {
        const int m_row = tile / p.num_n_blocks;
        const int n_blk = tile - m_row * p.num_n_blocks;
        const int m_blk = PAIR ? 2 * m_row + static_cast<int>(crank) : m_row;   // an odd m-block count leaves the last
        const int m0 = m_blk * kBlockM;                                           // pair a block past M: TMA zero-fills it
        // PAIR: this CTA loads block_n/2 of the tile's B rows (the MMA reads the other half from the peer)
        const int n0 = n_blk * p.block_n + (PAIR ? static_cast<int>(crank) * (p.block_n >> 1) : 0);
        int img = 0, ch = 0, cw = 0;
        if (p.a_mode == 1) {
          img = m0 / p.HoWo;
          const int rem = m0 - img * p.HoWo;
          const int pp = rem / p.Wo;
          const int qq = rem - pp * p.Wo;
          ch = p.lower_h + pp * p.stride;
          cw = p.lower_w + qq * p.stride;
        }
        int tap = 0, cb = 0;   // K-block = (filter tap, 64-channel block)
        for (int kb = 0; kb < p.num_kb; ++kb) {
          mbar_wait_r<PAIR>(&empty_bar[stage], phase ^ 1, 1, crank, tile, kb);
          uint8_t* st = tiles + static_cast<size_t>(stage) * p.stage_bytes;
          if (PAIR) {
            // both CTAs' loads count on the LEADER's full barrier, which expects the bytes of both
            const uint32_t fb = mapa_u32(smem_u32(&full_bar[stage]), 0);
            if (elect_one()) {
              if (crank == 0) mbar_expect_tx(&full_bar[stage], 2 * p.stage_bytes);
              if (p.a_mode == 1) {
                const int r = tap / p.S;
                const int s = tap - r * p.S;
                const uint16_t ow = static_cast<uint16_t>(s * p.dil);
                const uint16_t oh = static_cast<uint16_t>(r * p.dil);
                tma_load_im2col_4d_pair(st, &tmA_hi, fb, cb * kBlockK, cw, ch, img, ow, oh);
                tma_load_im2col_4d_pair(st + a_lo_off, &tmA_lo, fb, cb * kBlockK, cw, ch, img, ow, oh);
              } else {
                tma_load_2d_pair(st, &tmA_hi, fb, cb * kBlockK, m0);
                tma_load_2d_pair(st + a_lo_off, &tmA_lo, fb, cb * kBlockK, m0);
              }
              tma_load_2d_pair(st + b_hi_off, &tmB_hi, fb, kb * kBlockK, n0);
              tma_load_2d_pair(st + b_lo_off, &tmB_lo, fb, kb * kBlockK, n0);
            }
          } else if (elect_one()) {
            mbar_expect_tx(&full_bar[stage], p.stage_bytes);
            if (p.a_mode == 1) {
              const int r = tap / p.S;
              const int s = tap - r * p.S;
              const uint16_t ow = static_cast<uint16_t>(s * p.dil);
              const uint16_t oh = static_cast<uint16_t>(r * p.dil);
              tma_load_im2col_4d(st, &tmA_hi, &full_bar[stage], cb * kBlockK, cw, ch, img, ow, oh);
              if (SPLIT) tma_load_im2col_4d(st + a_lo_off, &tmA_lo, &full_bar[stage], cb * kBlockK, cw, ch, img, ow, oh);
            } else {
              tma_load_2d(st, &tmA_hi, &full_bar[stage], cb * kBlockK, m0);
              if (SPLIT) tma_load_2d(st + a_lo_off, &tmA_lo, &full_bar[stage], cb * kBlockK, m0);
            }
            tma_load_2d(st + b_hi_off, &tmB_hi, &full_bar[stage], kb * kBlockK, n0);
            if (SPLIT) tma_load_2d(st + b_lo_off, &tmB_lo, &full_bar[stage], kb * kBlockK, n0);
          }
          __syncwarp();
          if (++cb == p.cin_blocks) {
            cb = 0;
            ++tap;
          }
          if (++stage == p.num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (PAIR: the even CTA's, for both; the odd CTA's warp 1 idles) =====================
    // The whole warp runs the loop converged and one elected lane issues: every MMA operand (descriptors, TMEM
    // address, instruction descriptor) is then computed by warp-uniform code and lives in uniform registers.  (Run by
    // lane 0 alone, each tcgen05.mma was wrapped in an elect / broadcast / compare waterfall -- 276 instructions per
    // K-block, which bounded the MMA-bound layers: ncu showed this warp never waiting, only issuing.)
    if (!PAIR || crank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int as = 0;
      uint32_t aphase = 0;
      int cbuf = 0;          // ACC: chunk accumulator ring cursor + phase bit (flips when the ring wraps)
      uint32_t cphase = 0;
      const uint32_t tiles_u32 = smem_u32(tiles);
      // shared-memory matrix descriptor (K-major, 128-byte swizzle): low word = start address >> 4 (14 bits) | LBO 1 << 16,
      // high word = SBO 1024 >> 4 | descriptor version 1 << 14 | SWIZZLE_128B 2 << 29; offsets inside the stage and the
      // K advance (32 bytes per UMMA_K) add to the address field without carry (all of shared memory is < 2^18 bytes)
      constexpr uint64_t kDescHi = static_cast<uint64_t>((1024u >> 4) | (1u << 14) | (2u << 29)) << 32;
      // this CTA owns the whole TMEM of its SM (512 columns, one CTA per SM): the allocation starts at column 0, lane 0
      // (checked after the allocation), so the accumulator addresses are plain constants here
      for (int tile = tile_first; tile < tile_count; tile += tile_step) {
        mbar_wait_r<PAIR>(&tmem_empty[as], aphase ^ 1, 4, crank, tile, 0);
        tc_fence_after();
        // plain: acc0 at as*256, acc1 at as*256+128.  ACC: acc0 chunk buffers at 0 / 128, acc1 at 256 + as*128.
        uint32_t acc0 = as * acc_stage_cols;
        const uint32_t acc1 = ACC ? (p.acc_ring + as) * p.acc_stride : acc0 + 128;
        int kq = 0;
        for (int kb = 0; kb < p.num_kb; ++kb) {
          if (ACC && kq == 0) {
            mbar_wait_r<PAIR>(&c_empty[cbuf], cphase ^ 1, 3, crank, tile, kb);
            tc_fence_after();
            acc0 = cbuf * p.acc_stride;
          }
          mbar_wait_r<PAIR>(&full_bar[stage], phase, 2, crank, tile, kb);
          tc_fence_after();
          const uint32_t st = tiles_u32 + static_cast<uint32_t>(stage) * p.stage_bytes;
          const uint32_t d_a_hi = ((st >> 4) & 0x3FFFu) | 0x10000u;
          const uint32_t d_a_lo = d_a_hi + (a_lo_off >> 4);
          const uint32_t d_b_hi = d_a_hi + (b_hi_off >> 4);
          const uint32_t d_b_lo = d_a_hi + (b_lo_off >> 4);
          const bool chunk_end = ACC && (kq + 1 == p.acc_kb || kb == p.num_kb - 1);
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < kBlockK / kUmmaK; ++k) {
              const uint32_t ko = k * (kUmmaK * 2 >> 4);   // 32 bytes along K inside the 128B swizzle row, in 16-byte units
              const uint64_t a_hi = kDescHi | (d_a_hi + ko);
              const uint64_t b_hi = kDescHi | (d_b_hi + ko);
              const uint32_t first = (kb > 0 || k > 0) ? 1u : 0u;
              if (PAIR) {
                const uint64_t a_lo = kDescHi | (d_a_lo + ko);
                const uint64_t b_lo = kDescHi | (d_b_lo + ko);
                umma_f16_pair(acc0, a_hi, b_hi, p.idesc, (kq > 0 || k > 0) ? 1u : 0u);
                umma_f16_pair(acc1, a_hi, b_lo, p.idesc, first);
                umma_f16_pair(acc1, a_lo, b_hi, p.idesc, 1u);
              } else {
                umma_f16(acc0, a_hi, b_hi, p.idesc, ACC ? ((kq > 0 || k > 0) ? 1u : 0u) : first);
                if (SPLIT) {
                  const uint64_t a_lo = kDescHi | (d_a_lo + ko);
                  const uint64_t b_lo = kDescHi | (d_b_lo + ko);
                  umma_f16(acc1, a_hi, b_lo, p.idesc, first);
                  umma_f16(acc1, a_lo, b_hi, p.idesc, 1u);
                }
              }
            }
            if (PAIR) {   // every completion goes to the same barrier in both CTAs
              umma_commit_pair(&empty_bar[stage]);
              if (chunk_end) umma_commit_pair(&c_full[cbuf]);
              if (kb == p.num_kb - 1) umma_commit_pair(&tmem_full[as]);
            } else {
              umma_commit(&empty_bar[stage]);   // frees the smem slot once these MMAs have read it
              if (chunk_end) umma_commit(&c_full[cbuf]);   // chunk accumulator complete -> epilogue sums it
              if (kb == p.num_kb - 1) umma_commit(&tmem_full[as]);        // accumulator complete -> epilogue
            }
          }
          __syncwarp();
          if (ACC) {
            if (chunk_end) {
              if (++cbuf == p.acc_ring) {
                cbuf = 0;
                cphase ^= 1;
              }
              kq = 0;
            } else {
              ++kq;
            }
          }
          if (++stage == p.num_stages) {
            stage = 0;
            phase ^= 1;
          }
        }
        if (++as == 2) {
          as = 0;
          aphase ^= 1;
        }
      }
    }
   } else if (p.epi_mode == 1) {
    // ===================== output TMA warps (warp 2: column half 0, warp 3: column half 1) =====================
    // Staged output: the four epilogue warps of a half only compute -- they take a staging slot when its residual has
    // landed (or, without a residual, when the slot's previous store has read it), write the finished group into it and
    // arrive on grp_ready.  This warp does everything asynchronous for the half: it waits for the group, issues the TMA
    // store, and keeps the residual prefetch nslots-1 groups ahead (also across tile boundaries).  Until round 2 the first
    // epilogue warp of the half did this on top of its share of the math, behind a 128-thread named barrier per group: ncu's
    // stall sampling showed `barrier` as the top stall of the epilogue warps in the K <= 256 residual layers.
    const int hf = warp - 2;
    const int nch = p.block_n >> 4;
    const int h0 = (nch + 1) >> 1;
    const int c_beg = hf ? h0 : 0;
    const int my_n = hf ? nch - h0 : h0;
    const bool has_res = p.res_hi != nullptr;
    const bool res_lo = SPLIT && p.res_lo != nullptr;
    const int grp = p.epi_grp;
    const int nslots = p.epi_slots;
    uint8_t* ring = tiles + p.epi_off + hf * ring_bytes;
    uint64_t* rfull = res_full + hf * kEpiSlotsMax;
    uint64_t* gready = grp_ready + hf * kEpiSlotsMax;
    uint64_t* sfree = slot_free + hf * kEpiSlotsMax;
    int la_tile = tile_first, la_c = 0, la_slot = 0;   // look-ahead cursor of the residual prefetch
    auto issue_res_group = [&]() {
      if (la_tile >= tile_count) return;
      const int m_row = la_tile / p.num_n_blocks;
      const int n_blk = la_tile - m_row * p.num_n_blocks;
      const int m_blk = PAIR ? 2 * m_row + static_cast<int>(crank) : m_row;
      const int gn = (my_n - la_c) < grp ? (my_n - la_c) : grp;
      const int col = n_blk * p.block_n + (c_beg + la_c) * 16;
      uint8_t* b = ring + la_slot * slot_bytes;
      uint64_t* bar = &rfull[la_slot];
      if (elect_one()) {
        mbar_expect_tx(bar, gn * kEpiPlaneBytes * (res_lo ? 2 : 1));
        if (p.epi_wide) {   // one 32-column box per plane (groups are always full in wide mode)
          tma_load_2d(b, &tmR_hi, bar, col, m_blk * kBlockM);
          if (res_lo) tma_load_2d(b + 2 * kEpiPlaneBytes, &tmR_lo, bar, col, m_blk * kBlockM);
        } else {
          for (int u = 0; u < gn; ++u) {
            tma_load_2d(b + u * p.epi_chunk_bytes, &tmR_hi, bar, col + u * 16, m_blk * kBlockM);
            if (res_lo) tma_load_2d(b + u * p.epi_chunk_bytes + kEpiPlaneBytes, &tmR_lo, bar, col + u * 16, m_blk * kBlockM);
          }
        }
      }
      __syncwarp();
      la_c += gn;
      if (la_c >= my_n) {
        la_c = 0;
        la_tile += tile_step;
      }
      if (++la_slot == nslots) la_slot = 0;
    };
    if (my_n > 0) {
      if (has_res)
        for (int i = 0; i < nslots - 1; ++i) issue_res_group();
      int slot = 0, prev_slot = -1;
      uint32_t gph = 0;        // phase bits of gready[]
      for (int tile = tile_first; tile < tile_count; tile += tile_step) {
        const int m_row = tile / p.num_n_blocks;
        const int n_blk = tile - m_row * p.num_n_blocks;
        const int m_blk = PAIR ? 2 * m_row + static_cast<int>(crank) : m_row;
        const int n0 = n_blk * p.block_n;
        for (int c = 0; c < my_n; c += grp) {
          const int gn = (my_n - c) < grp ? (my_n - c) : grp;
          const int nb = n0 + (c_beg + c) * 16;
          uint8_t* sb = ring + slot * slot_bytes;
          mbar_wait_r<PAIR>(&gready[slot], (gph >> slot) & 1u, 9, crank, tile, c);
          gph ^= 1u << slot;
          if (elect_one()) {
            // every earlier store must be done reading its slot before the look-ahead load below refills the slot of
            // the previous group (residual ring) or before that slot is handed back to the epilogue warps (two slots)
            bulk_wait_read<0>();
            if (p.epi_wide) {
              tma_store_2d(&tmO_hi, sb, nb, m_blk * kBlockM);
              if (SPLIT && p.out_lo != nullptr) tma_store_2d(&tmO_lo, sb + 2 * kEpiPlaneBytes, nb, m_blk * kBlockM);
            } else {
              for (int t = 0; t < gn; ++t) {
                tma_store_2d(&tmO_hi, sb + t * p.epi_chunk_bytes, nb + t * 16, m_blk * kBlockM);
                if (SPLIT && p.out_lo != nullptr)
                  tma_store_2d(&tmO_lo, sb + t * p.epi_chunk_bytes + kEpiPlaneBytes, nb + t * 16, m_blk * kBlockM);
              }
            }
            bulk_commit();
            if (!has_res && prev_slot >= 0) mbar_arrive(&sfree[prev_slot]);   // its store was among those waited for above
          }
          __syncwarp();
          if (has_res) issue_res_group();
          prev_slot = slot;
          if (++slot == nslots) slot = 0;
        }
      }
      if (elect_one()) bulk_wait_all();   // the output must be globally written before the CTA retires
      __syncwarp();
    }
   }
  } else if (warp < 4 + kEpiWarps) {
    if (ACC) setmaxnreg_inc<224>();
    // ===================== epilogue =====================
    // Eight warps: warp w reads TMEM lanes 32*(w&3).. (its row quarter of the tile) and owns the column half
    // hf = (w-4)>>2 of the tile: chunks [c_beg, c_end) of 16 columns.  The two halves run independently (own staging
    // ring, own named barrier, own elected TMA thread); together they halve the time per tile of the epilogue, which
    // bounds the short-K layers and -- in ACC mode, where the same warps must keep draining chunk accumulators --
    // stalls the MMA issuer for as long as a tile's output stage takes.
    const int ew = warp & 3;
    const int hf = (warp - 4) >> 2;
    const int row = ew * 32 + lane;
    const int nch = p.block_n >> 4;
    const int h0 = (nch + 1) >> 1;
    const int c_beg = hf ? h0 : 0;
    const int my_n = hf ? nch - h0 : h0;
    const uint32_t lane_off = static_cast<uint32_t>(ew * 32) << 16;
    int as = 0;
    uint32_t aphase = 0;
    int ecbuf = 0;       // ACC: chunk accumulator ring cursor + phase bit (mirror the MMA issuer's)
    uint32_t ecphase = 0;

    // ---- staged output state (epi_mode 1): residual chunks arrive in swizzled smem buffers (TMA loads issued
    // epi_slots-1 groups ahead, also across tile boundaries), results overwrite them in place and leave by TMA store.
    const bool staged = p.epi_mode == 1;
    const bool has_res = p.res_hi != nullptr;
    const bool res_lo = SPLIT && p.res_lo != nullptr;
    // the TMA stores and the residual prefetch of this half are issued by its output TMA warp (warp 2 + hf, see above)
    const int grp = p.epi_grp;
    const int nslots = p.epi_slots;
    uint8_t* ring = epi + hf * ring_bytes;
    uint64_t* rfull = res_full + hf * kEpiSlotsMax;
    uint64_t* gready = grp_ready + hf * kEpiSlotsMax;
    uint64_t* sfree = slot_free + hf * kEpiSlotsMax;
    int slot = 0;
    uint32_t rph = 0;        // phase bits of rfull[] (residual landed) / of sfree[] (previous store has read the slot)

    for (int tile = tile_first; tile < tile_count; tile += tile_step) {
      const int m_row = tile / p.num_n_blocks;
      const int n_blk = tile - m_row * p.num_n_blocks;
      const int m_blk = PAIR ? 2 * m_row + static_cast<int>(crank) : m_row;
      const int n0 = n_blk * p.block_n;
      // direct mode: this thread's output / residual pixel
      size_t opix = 0, rpix = 0;
      bool valid = true;
      if (!staged) {
        const int m = m_blk * kBlockM + row;
        valid = m < p.M;
        if (valid) {
          const int img = m / p.HoWo;
          const int rem = m - img * p.HoWo;
          const int pp = rem / p.Wo + p.off_h;
          const int qq = rem - (rem / p.Wo) * p.Wo + p.off_w;
          opix = (static_cast<size_t>(img) * p.out_H + pp) * p.out_W + qq;
          rpix = (static_cast<size_t>(img) * p.res_H + (pp >> p.res_shift)) * p.res_W + (qq >> p.res_shift);
        }
      }
      float amax = 0.f;   // largest |output| this thread writes in this tile (range monitor)
      // one finished chunk (relative index c in this half): bias / residual / activation, then out
      auto chunk_out = [&](int c, float (&v)[16]) {
        const int n = n0 + (c_beg + c) * 16;
        if (!staged) {
          if (valid) epilogue_chunk16<SPLIT, SWISH>(p, v, opix, rpix, n, amax);
          return;
        }
        const int u = grp == 2 ? (c & 1) : 0;      // position inside the group
        uint8_t* sb = ring + slot * slot_bytes;
        if (u == 0) {   // first chunk of a group: take the slot
          if (has_res) mbar_wait_r<PAIR>(&rfull[slot], (rph >> slot) & 1u, 7, crank, tile, c);   // its residual has landed
          else mbar_wait_r<PAIR>(&sfree[slot], ((rph >> slot) & 1u) ^ 1u, 8, crank, tile, c);   // its previous store has read it (first use: free)
          rph ^= 1u << slot;
        }
        {
          // narrow: chunk buffer [128][32 B] per plane, 32-byte swizzle (16-byte cell j of row r at j ^ ((r >> 2) & 1));
          // wide: group box [128][64 B] per plane, 64-byte swizzle (cell j of row r at j ^ ((r >> 1) & 3)), this chunk = cells 2u, 2u+1
          uint8_t* hp;
          uint32_t c0, c1, lo_off;
          if (p.epi_wide) {
            const uint32_t sw = (row >> 1) & 3;
            hp = sb + row * 64;
            c0 = ((2 * u) ^ sw) << 4;
            c1 = ((2 * u + 1) ^ sw) << 4;
            lo_off = 2 * kEpiPlaneBytes;
          } else {
            const uint32_t sw = (row >> 2) & 1;
            hp = sb + u * p.epi_chunk_bytes + row * 32;
            c0 = sw << 4;
            c1 = (1 ^ sw) << 4;
            lo_off = kEpiPlaneBytes;
          }
          epilogue_chunk16_smem<SPLIT, SWISH>(p, v, reinterpret_cast<uint4*>(hp + c0), reinterpret_cast<uint4*>(hp + c1),
                                       reinterpret_cast<uint4*>(hp + lo_off + c0), reinterpret_cast<uint4*>(hp + lo_off + c1), n,
                                       has_res, res_lo, amax);
        }
        if (u == grp - 1 || c == my_n - 1) {   // group complete: hand it to the output TMA warp
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive(&gready[slot]);
          if (++slot == nslots) slot = 0;
        }
      };

      if (ACC) {
        float sums[kAccMaxChunks * 16];
#pragma unroll
        for (int i = 0; i < kAccMaxChunks * 16; ++i) sums[i] = 0.0f;
        const int nq = (p.num_kb + p.acc_kb - 1) / p.acc_kb;
        for (int q = 0; q < nq; ++q) {
          const int cbuf = ecbuf;
          mbar_wait_r<PAIR>(&c_full[cbuf], ecphase, 5, crank, tile, q);
          if (++ecbuf == p.acc_ring) {
            ecbuf = 0;
            ecphase ^= 1;
          }
          tc_fence_after();
          acc_fold<false, PAIR>(sums, tmem_base + lane_off + cbuf * p.acc_stride + c_beg * 16, my_n, &c_empty[cbuf], lane);
        }
        // the correction accumulator (hi*lo + lo*hi) is folded into the sums right away, which hands the tile's TMEM
        // stage back before the output stage starts
        mbar_wait_r<PAIR>(&tmem_full[as], aphase, 6, crank, tile, 0);
        tc_fence_after();
        acc_fold<true, PAIR>(sums, tmem_base + lane_off + (p.acc_ring + as) * p.acc_stride + c_beg * 16, my_n, &tmem_empty[as], lane);
#pragma unroll
        for (int c = 0; c < kAccMaxChunks; ++c) {
          if (c < my_n) {
            float v[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = fmaf(sums[(ACC ? c : 0) * 16 + i], p.acc_delta, sums[(ACC ? c : 0) * 16 + i]);
            chunk_out(c, v);
          }
        }
      } else {
        mbar_wait(&tmem_full[as], aphase);
        tc_fence_after();
        const uint32_t tacc = tmem_base + lane_off + as * acc_stage_cols + c_beg * 16;
        const uint32_t tacc1 = tacc + 128;
        for (int c = 0; c < my_n; ++c) {
          uint32_t a0[16], a1[16];
          tmem_ld_32x32b_x16(tacc + c * 16, a0);
          if (SPLIT) tmem_ld_32x32b_x16(tacc1 + c * 16, a1);
          tmem_ld_wait();
          float v[16];
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            v[i] = __uint_as_float(a0[i]);
            if (SPLIT) {
              v[i] = fmaf(v[i], p.acc_delta, v[i]);   // the same compensation for the single-chunk (K <= 64) split layers
              v[i] = fmaf(__uint_as_float(a1[i]), kLoInv, v[i]);
            }
          }
          chunk_out(c, v);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tmem_empty[as]);
      }
      if (++as == 2) {
        as = 0;
        aphase ^= 1;
      }
      // inf included; a NaN can only follow an inf, which an earlier launch has flagged
      if (p.range_flag != nullptr && amax > 65504.f) atomicOr(p.range_flag, 1u);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync();   // neither CTA retires (shared memory, TMEM, barriers) while its peer may still signal it
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_pair(tmem_base, kTmemCols);
    else tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t,
                                   const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_encode_tiled = nullptr;
EncodeIm2colFn g_encode_im2col = nullptr;
int g_driver_version = 0;

void small_tensor_fixup(CUtensorMap* m, size_t bytes) {
  // Driver <= 13.1 mis-encodes maps of tensors smaller than 128 KiB (bit 21 of the 2nd qword); the
  // vendored CuTe applies the same fix-up (cute/atom/copy_traits_sm90_tma.hpp).
  if (g_driver_version <= 13010 && bytes < 131072) reinterpret_cast<uint64_t*>(m)[1] &= ~(1ull << 21);
}

int encode_2d(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t row_stride_bytes,
              uint32_t box_inner, uint32_t box_outer, CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {row_stride_bytes};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode_tiled(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, swz,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed: " + std::to_string(static_cast<int>(r)));
    return -1;
  }
  small_tensor_fixup(m, static_cast<size_t>(outer) * row_stride_bytes);
  return 0;
}

}  // namespace

struct ConvPlan {
  CUtensorMap tmA_hi, tmA_lo, tmB_hi, tmB_lo, tmO_hi, tmO_lo, tmR_hi, tmR_lo;
  ConvTcParams p;
  bool split;
  bool acc;
  bool pair;   // CTA pairs (cta_group::2): clusters of two CTAs share 256-row tiles
  int grid;
  size_t smem_bytes;
};

int conv_tc_init() {
  if (g_encode_tiled && g_encode_im2col) return 0;
  B2_CUDA(cudaDriverGetVersion(&g_driver_version));
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  B2_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
  B2_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled not available");
  g_encode_tiled = reinterpret_cast<EncodeTiledFn>(fn);
  fn = nullptr;
  B2_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &q));
  B2_CHECK(fn != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeIm2col not available");
  g_encode_im2col = reinterpret_cast<EncodeIm2colFn>(fn);
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<false, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<true, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  B2_CUDA(cudaFuncSetAttribute(conv_tc_kernel<true, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  return 0;
}

static int pick_block_n(int cout_pad, bool split) {
  const int cap = split ? 128 : 256;
  if (cout_pad <= cap) return cout_pad;
  for (int bn = cap; bn >= 16; bn -= 16)
    if (cout_pad % bn == 0) return bn;
  return 16;
}

static int plan_build(ConvPlan* pl, const ConvDesc& d, const ConvWeights& w, const ConvIO& io, bool split,
                      int num_sms, int force_a_mode) {
  B2_CHECK(conv_tc_init() == 0, "conv_tc_init failed");
  B2_CHECK(d.Cin % kBlockK == 0, "conv_tc: Cin must be a multiple of 64");
  B2_CHECK(w.Cout_pad % 16 == 0, "conv_tc: Cout_pad must be a multiple of 16");
  B2_CHECK(w.K == d.R * d.S * d.Cin, "conv_tc: packed weight K mismatch");
  B2_CHECK(!split || (io.in_lo && w.w_lo), "conv_tc: split precision needs lo planes");
  ConvTcParams& p = pl->p;
  const int Ho = d.Ho(), Wo = d.Wo();
  B2_CHECK(Ho > 0 && Wo > 0, "conv_tc: empty output");
  p.M = d.B * Ho * Wo;
  p.Ho = Ho;
  p.Wo = Wo;
  p.HoWo = Ho * Wo;
  p.stride = d.stride;
  p.dil = d.dil;
  p.lower_h = -d.pad_t;
  p.lower_w = -d.pad_l;
  p.S = d.S;
  p.cin_blocks = d.Cin / kBlockK;
  p.num_kb = d.R * d.S * p.cin_blocks;
  p.block_n = pick_block_n(w.Cout_pad, split);
  p.num_n_blocks = w.Cout_pad / p.block_n;
  B2_CHECK(p.num_n_blocks * p.block_n == w.Cout_pad, "conv_tc: Cout_pad not divisible by block_n");
  const int num_m_blocks = (p.M + kBlockM - 1) / kBlockM;
  p.num_tiles = num_m_blocks * p.num_n_blocks;
  // CTA pairs: an SM takes operands in at ~51 B/clk (tools/l2_fill_probe.cu), a 128x128 split tile needs 85 B/clk at full
  // tensor-pipe rate; sharing the B tile between the two CTAs of a pair brings that to 64.  Layers with at least
  // B2_PAIR K-blocks (the operand-bound ones), split + ACC, ReLU / linear epilogue.
  pl->pair = false;
  if (const char* e = getenv("B2_PAIR")) {
    const int acc_kb_plan = d.acc_kb > 0 ? d.acc_kb : kAccChunkKb;
    const bool acc_plan = split && d.acc_kb >= 0 && p.num_kb > acc_kb_plan;
    pl->pair = acc_plan && atoi(e) > 0 && p.num_kb >= atoi(e) && p.block_n == 128 && d.relu != 2 && num_m_blocks >= 2 &&
               num_sms >= 2;
  }
  p.num_pair_tiles = ((num_m_blocks + 1) / 2) * p.num_n_blocks;
  p.idesc = make_idesc_f16(pl->pair ? 2 * kBlockM : kBlockM, p.block_n);
  p.b_bytes = static_cast<uint32_t>(pl->pair ? p.block_n / 2 : p.block_n) * kBlockK * 2;   // per CTA
  p.stage_bytes = (kABytes + p.b_bytes) * (split ? 2 : 1);
  // TMA-staged epilogue: fp16 plane output with a 1:1 row mapping (no placement offset, no shifted residual)
  {
    const bool one_to_one = d.off_h == 0 && d.off_w == 0 && d.out_H == Ho && d.out_W == Wo;
    const bool res_ok = io.res_hi == nullptr || (d.res_shift == 0 && d.res_H == d.out_H && d.res_W == d.out_W);
    p.epi_mode = (io.out_f32 == nullptr && one_to_one && res_ok && d.force_epi_mode != 0) ? 1 : 0;
  }
  // staging rings (one per column half of the tile).  A group = epi_grp chunks of 16 columns that share one fence /
  // barrier / TMA-store round; a ring = epi_slots groups.  With a residual: three slots (the prefetch runs two groups
  // ahead); without: two.  Two-chunk groups are used when that still leaves three pipeline stages (two with a residual:
  // those layers are bound by the output stage, not by operand latency).
  {
    const int nch = p.block_n >> 4;
    const bool has_res = io.res_hi != nullptr;
    p.epi_chunk_bytes = static_cast<uint32_t>(kEpiPlaneBytes) * (split ? 2 : 1);
    p.epi_slots = has_res ? 3 : 2;
    p.epi_grp = ((nch + 1) / 2 >= 2) ? 2 : 1;
    auto stages_for = [&](int grp) {
      const int epi = kEpiHalves * p.epi_slots * grp * static_cast<int>(p.epi_chunk_bytes);
      return (kSmemBudget - epi) / static_cast<int>(p.stage_bytes);
    };
    if (p.epi_grp == 2 && stages_for(2) < (has_res ? 2 : 3) && stages_for(1) > stages_for(2)) p.epi_grp = 1;
    // two-chunk groups move as one 32-column box per plane when every group of both halves is full
    p.epi_wide = (p.epi_mode == 1 && p.epi_grp == 2 && nch % 4 == 0) ? 1 : 0;
    if (p.epi_mode != 1) {   // direct mode: no staging ring
      p.epi_grp = 1;
      p.epi_slots = 0;
    }
  }
  const int epi_bytes = kEpiHalves * p.epi_slots * p.epi_grp * static_cast<int>(p.epi_chunk_bytes);
  p.num_stages = (kSmemBudget - epi_bytes) / static_cast<int>(p.stage_bytes);
  if (p.num_stages > kMaxStages) p.num_stages = kMaxStages;
  B2_CHECK(p.num_stages >= 2, "conv_tc: tile too large for shared memory");
  p.epi_off = static_cast<uint32_t>(p.num_stages) * p.stage_bytes;
  p.out_hi = io.out_hi;
  p.out_lo = io.out_lo;
  p.out_f32 = io.out_f32;
  p.ldc = d.ldc;
  p.out_H = d.out_H;
  p.out_W = d.out_W;
  p.off_h = d.off_h;
  p.off_w = d.off_w;
  B2_CHECK(d.ldc >= w.Cout_pad && d.ldc % 8 == 0, "conv_tc: ldc must cover Cout_pad");
  B2_CHECK(Ho + d.off_h <= d.out_H && Wo + d.off_w <= d.out_W, "conv_tc: output does not fit buffer");
  p.bias = w.bias;
  p.res_hi = io.res_hi;
  p.res_lo = io.res_lo;
  p.ldr = d.ldr;
  p.res_H = d.res_H;
  p.res_W = d.res_W;
  p.res_shift = d.res_shift;
  p.relu = d.relu;
  pl->split = split;
  p.range_flag = io.range_flag;
  // accurate accumulation: on by default in split precision when K spans more than one chunk
  p.acc_kb = d.acc_kb > 0 ? d.acc_kb : kAccChunkKb;
  // experiment hook (round 2): longer chunks on the CTA-pair layers only -- every chunk hand-off of a pair crosses the two
  // SMs twice (commit multicast out, "drained" arrive back), which a two-deep ring of one-K-block chunks does not cover
  if (const char* e = getenv("B2_PAIR_ACC_KB")) if (pl->pair && atoi(e) > 0 && p.num_kb > atoi(e)) p.acc_kb = atoi(e);
  pl->acc = split && d.acc_kb >= 0 && p.num_kb > p.acc_kb;
  p.acc_delta = p.acc_kb >= 2 ? kAccDelta2 : kAccDelta;
  p.acc_stride = p.block_n == 64 ? 64 : 128;
  p.acc_ring = p.block_n == 64 ? kAccRingMax : 2;   // (ring + 2 correction accumulators) * stride <= 512 columns
  pl->grid = p.num_tiles < num_sms ? p.num_tiles : num_sms;
  if (pl->pair) {
    B2_CHECK(pl->acc && p.acc_ring == 2, "conv_tc: CTA pairs need the ACC scheme on 128-column tiles");
    const int pairs = num_sms / 2;
    pl->grid = 2 * (p.num_pair_tiles < pairs ? p.num_pair_tiles : pairs);
  }
  pl->smem_bytes = static_cast<size_t>(p.num_stages) * p.stage_bytes + epi_bytes + 1024 /*align*/ + 512 /*barriers*/;
  const int in_ld = d.in_ld > 0 ? d.in_ld : d.Cin;
  const bool plain = (d.R == 1 && d.S == 1 && d.stride == 1 && d.pad_t == 0 && d.pad_b == 0 && d.pad_l == 0 &&
                      d.pad_r == 0 && d.in_H == d.in_pitch_H && d.in_W == d.in_pitch_W);
  p.a_mode = plain ? 0 : 1;
  if (force_a_mode >= 0) {
    B2_CHECK(force_a_mode == 1 || plain, "conv_tc: tiled A mode needs a plain 1x1 conv");
    p.a_mode = force_a_mode;
  }
  const size_t in_bytes = static_cast<size_t>(d.B) * d.in_pitch_H * d.in_pitch_W * in_ld * 2;
  for (int plane = 0; plane < (split ? 2 : 1); ++plane) {
    CUtensorMap* mA = plane == 0 ? &pl->tmA_hi : &pl->tmA_lo;
    CUtensorMap* mB = plane == 0 ? &pl->tmB_hi : &pl->tmB_lo;
    const __half* a = plane == 0 ? io.in_hi : io.in_lo;
    const __half* b = plane == 0 ? w.w_hi : w.w_lo;
    if (p.a_mode == 0) {
      if (encode_2d(mA, a, d.Cin, static_cast<uint64_t>(d.B) * d.in_H * d.in_W, static_cast<uint64_t>(in_ld) * 2,
                    kBlockK, kBlockM))
        return -1;
    } else {
      cuuint64_t dims[4] = {static_cast<cuuint64_t>(d.Cin), static_cast<cuuint64_t>(d.in_W),
                            static_cast<cuuint64_t>(d.in_H), static_cast<cuuint64_t>(d.B)};
      cuuint64_t strides[3] = {static_cast<cuuint64_t>(in_ld) * 2,
                               static_cast<cuuint64_t>(d.in_pitch_W) * in_ld * 2,
                               static_cast<cuuint64_t>(d.in_pitch_H) * d.in_pitch_W * in_ld * 2};
      // bounding box of filter base positions: lower = -pad, upper = pad_after - (k-1)*dilation  {W, H}
      int lower[2] = {-d.pad_l, -d.pad_t};
      int upper[2] = {d.pad_r - (d.S - 1) * d.dil, d.pad_b - (d.R - 1) * d.dil};
      cuuint32_t estr[4] = {1, static_cast<cuuint32_t>(d.stride), static_cast<cuuint32_t>(d.stride), 1};
      CUresult r = g_encode_im2col(mA, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(a), dims, strides,
                                   lower, upper, kBlockK, kBlockM, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeIm2col failed: " + std::to_string(static_cast<int>(r)) + " (Cin=" +
                  std::to_string(d.Cin) + " W=" + std::to_string(d.in_W) + " H=" + std::to_string(d.in_H) + ")");
        return -1;
      }
      small_tensor_fixup(mA, in_bytes);
    }
    if (encode_2d(mB, b, w.K, w.Cout_pad, static_cast<uint64_t>(w.K) * 2, kBlockK, pl->pair ? p.block_n / 2 : p.block_n))
      return -1;
  }
  if (!split) {
    pl->tmA_lo = pl->tmA_hi;
    pl->tmB_lo = pl->tmB_hi;
  }
  pl->tmO_hi = pl->tmO_lo = pl->tmR_hi = pl->tmR_lo = pl->tmB_hi;   // valid placeholders for the direct mode
  if (p.epi_mode == 1) {
    const uint64_t rows = static_cast<uint64_t>(p.M);
    const uint32_t ebox = p.epi_wide ? 32 : 16;
    const CUtensorMapSwizzle eswz = p.epi_wide ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
    if (encode_2d(&pl->tmO_hi, io.out_hi, w.Cout_pad, rows, static_cast<uint64_t>(d.ldc) * 2, ebox, kBlockM, eswz))
      return -1;
    pl->tmO_lo = pl->tmO_hi;
    if (split && io.out_lo &&
        encode_2d(&pl->tmO_lo, io.out_lo, w.Cout_pad, rows, static_cast<uint64_t>(d.ldc) * 2, ebox, kBlockM, eswz))
      return -1;
    pl->tmR_hi = pl->tmR_lo = pl->tmO_hi;
    if (io.res_hi) {
      if (encode_2d(&pl->tmR_hi, io.res_hi, w.Cout_pad, rows, static_cast<uint64_t>(d.ldr) * 2, ebox, kBlockM, eswz))
        return -1;
      pl->tmR_lo = pl->tmR_hi;
      if (split && io.res_lo &&
          encode_2d(&pl->tmR_lo, io.res_lo, w.Cout_pad, rows, static_cast<uint64_t>(d.ldr) * 2, ebox, kBlockM, eswz))
        return -1;
    }
  }
  return 0;
}

ConvPlan* conv_tc_plan_create(const ConvDesc& d, const ConvWeights& w, const ConvIO& io, bool split, int num_sms) {
  ConvPlan* pl = new ConvPlan();
  if (plan_build(pl, d, w, io, split, num_sms, d.force_a_mode) != 0) {
    delete pl;
    return nullptr;
  }
  return pl;
}

void conv_tc_plan_destroy(ConvPlan* p) { delete p; }

static long long g_pair_launches = 0;   // launches that took the CTA-pair path (tests check that the opt-in hook is live)
long long conv_tc_pair_launches() { return g_pair_launches; }

int conv_tc_launch(const ConvPlan* pl, cudaStream_t stream) {
  const bool sw = pl->p.relu == 2;
#define B2_CONV_LAUNCH(S, A, W)                                                                                          \
  conv_tc_kernel<S, A, W><<<pl->grid, kThreads, pl->smem_bytes, stream>>>(pl->tmA_hi, pl->tmA_lo, pl->tmB_hi, pl->tmB_lo, \
                                                                          pl->tmO_hi, pl->tmO_lo, pl->tmR_hi, pl->tmR_lo, pl->p)
  if (pl->pair) {
    ++g_pair_launches;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(pl->grid);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = pl->smem_bytes;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    B2_CUDA(cudaLaunchKernelEx(&cfg, conv_tc_kernel<true, true, false, true>, pl->tmA_hi, pl->tmA_lo, pl->tmB_hi, pl->tmB_lo,
                               pl->tmO_hi, pl->tmO_lo, pl->tmR_hi, pl->tmR_lo, pl->p));
#ifdef B2_PAIR_DIAG
    {   // bring-up variant only (never inside a graph capture): report a wait that timed out
      B2_CUDA(cudaStreamSynchronize(stream));
      unsigned int diag[2] = {0, 0};
      B2_CUDA(cudaMemcpyFromSymbol(diag, g_pair_diag, sizeof(diag)));
      if (diag[0] != 0) {
        fprintf(stderr, "conv_tc PAIR: wait timed out: role %u rank %u tile %u kb %u (grid %d, pair tiles %d, kb %d, stages %d, epi_mode %d)\n",
                diag[0] >> 28, (diag[0] >> 27) & 1u, (diag[0] >> 8) & 0x7FFFFu, diag[0] & 0xFFu, pl->grid, pl->p.num_pair_tiles,
                pl->p.num_kb, pl->p.num_stages, pl->p.epi_mode);
        unsigned int zero[2] = {0, 0};
        B2_CUDA(cudaMemcpyToSymbol(g_pair_diag, zero, sizeof(zero)));
        set_error("conv_tc PAIR: barrier wait timed out");
        return -1;
      }
    }
#endif
  } else if (pl->split && pl->acc) {
    if (sw) B2_CONV_LAUNCH(true, true, true);
    else B2_CONV_LAUNCH(true, true, false);
  } else if (pl->split) {
    if (sw) B2_CONV_LAUNCH(true, false, true);
    else B2_CONV_LAUNCH(true, false, false);
  } else {
    if (sw) B2_CONV_LAUNCH(false, false, true);
    else B2_CONV_LAUNCH(false, false, false);
  }
#undef B2_CONV_LAUNCH
  B2_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace b2
