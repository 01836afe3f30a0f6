// Detector head tail fused into one tcgen05 kernel: convPb (1x1, 256 -> 65, folded BN) + softmax over the 65
// channels + dustbin drop + depth-to-space (pixel_shuffle 8) + validity-mask multiply.
//
// Reference: models/model_utils/heads.py:22-28 (convPb, softmax, [:, :-1], pixel_shuffle, squeeze) and
// engine_solvers/export.py:70 (prob *= mask).  The 65 logits of a cell never leave the SM unless the caller asks for
// them (model.forward returns "logits"; the homography-adaptation export does not).
//
// GEMM view: M = 128 cells (8 wide x 16 high, TMEM lane = cell), N = 80 (65 padded to the next legal UMMA N for M = 128),
// K = 256 = 4 channel blocks x 4 K-steps.  One epilogue thread owns one cell: it reads the 65 fp32 logits from TMEM,
// computes exp(l - max) / sum exactly like softmax_d2s_kernel, and writes the cell's 8 x 8 block of the heatmap
// (times the mask) with float4 stores.  Warp roles: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 and 6-9 two
// epilogue groups that alternate tiles (one per TMEM accumulator), so one group's exp / store phase overlaps the
// other's TMEM reads; the mask bytes of a cell are fetched before the accumulator wait (they do not depend on the
// MMAs), which takes their DRAM latency off the per-row store loop.  Bias through one extra MMA against a constant
// ones operand.
#include <cuda.h>
#include <math.h>

#include <vector>

#include "spn_common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcptx;

constexpr int kTW = 8, kTH = 16;
constexpr int kN = 80;                              // 65 logits padded to a multiple of 16
constexpr int kBlk = 2 * kN * 16;                   // operand-B block of one K-step: [chunk 2][n 80][8] = 2560 B
constexpr int kWBytes = 16 * kBlk + kBlk;           // 4 channel blocks x 4 K-steps + bias block = 43520 B
constexpr uint32_t kChStride = (uint32_t)kTH * kTW * 16;   // 2048 B between 8-channel groups of a slab
constexpr int kSlabBytes = 8 * kTH * kTW * 16;      // 16384 B: 64 channels of 128 cells
constexpr int kOnesBytes = 4096;
constexpr int kStages = 8;
constexpr int kThreads = 320;   // TMA, MMA, 2 x 4 epilogue warps

struct HeadParams {
  int n_img, Hc, Wc, tiles_x, tiles_y;
  int is_bf16;
  const void* wimg;
  const uint8_t* __restrict__ mask;   // [n][H][W] or null
  float* __restrict__ logits;         // [n][65][Hc][Wc] or null
  float* __restrict__ prob;           // [n][H][W]
};

__global__ void __launch_bounds__(kThreads, 1)
head_tc_kernel(const __grid_constant__ CUtensorMap tmap, const HeadParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full[kStages], bar_empty[kStages], bar_w, bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_s;

  griddep_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint8_t* wsm = smem;
  uint8_t* ones = smem + ((kWBytes + 1023) & ~1023);
  uint8_t* slab0 = ones + kOnesBytes;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int n_tiles = p.n_img * tiles_per_img;

  if (threadIdx.x == 0) {
    for (int i = 0; i < kStages; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_w, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {
    const uint32_t one2 = p.is_bf16 ? 0x3F803F80u : 0x3C003C00u;
    for (int i = threadIdx.x; i < kOnesBytes / 16; i += kThreads)
      reinterpret_cast<uint4*>(ones)[i] = i < 128 ? make_uint4(one2, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: 2 accumulators x 80 columns at column 0 and 128
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(256));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(&bar_w, (uint32_t)kWBytes);
      for (int o = 0; o < kWBytes; o += kBlk) bulk_load(wsm + o, (const uint8_t*)p.wimg + o, kBlk, &bar_w);
    }
    griddep_wait();  // convPa's output comes from the previous kernel; every store of this CTA follows these loads
    int stage = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      const int n = t / tiles_per_img, r = t - n * tiles_per_img;
      const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
      for (int cb = 0; cb < 4; ++cb) {
        mbar_wait(&bar_empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bar_full[stage], (uint32_t)kSlabBytes);
          tma_load_4d(slab0 + (size_t)stage * kSlabBytes, &tmap, &bar_full[stage], tx * kTW * 8, ty * kTH, cb * 8, n);
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    const uint32_t fmt = p.is_bf16 ? 1u : 0u;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (((uint32_t)kN >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t a_hi = ((uint32_t)(kTW * 16) >> 4) | (1u << 14);   // SBO = one row of 8 cells (128 B)
    const uint32_t a_lo_c = (kChStride >> 4) << 16;
    const uint32_t b_hi = (128u >> 4) | (1u << 14);
    const uint32_t b_lo_c = (((uint32_t)kN * 16) >> 4) << 16;          // LBO = 1280 B between the two K chunks
    const uint32_t o_lo = (smem_u32(ones) >> 4) | ((2048u >> 4) << 16);
    mbar_wait(&bar_w, 0);
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    const uint32_t w_addr = smem_u32(wsm), slab_addr = smem_u32(slab0);
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
      mbar_wait(&bar_tempty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * 128;
      for (int cb = 0; cb < 4; ++cb) {
        mbar_wait(&bar_full[stage], phase);
        tc_fence_after();
        const uint32_t a_lo = ((slab_addr + (uint32_t)stage * kSlabBytes) >> 4) | a_lo_c;
        const uint32_t b_lo = ((w_addr + (uint32_t)cb * (4 * kBlk)) >> 4) | b_lo_c;
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16_2w(d_tmem, a_lo + (((uint32_t)kk * 2 * kChStride) >> 4), a_hi, b_lo + (((uint32_t)kk * kBlk) >> 4), b_hi, idesc,
                        (cb | kk) ? 1u : 0u);
          umma_commit(&bar_empty[stage]);
          if (cb == 3) {
            umma_f16_2w(d_tmem, o_lo, (128u >> 4) | (1u << 14), ((w_addr + 16u * kBlk) >> 4) | b_lo_c, b_hi, idesc, 1u);  // + bias
            umma_commit(&bar_tfull[acc]);
          }
        }
        __syncwarp();
        if (++stage == kStages) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    // ===================== epilogue: one thread = one 8x8 cell; group = accumulator =====================
    const int q = warp & 3;                 // TMEM lane quarter this warp may read
    const int grp = (warp - 2) >> 2;        // 0: warps 2-5, 1: warps 6-9
    const int g = q * 4 + (lane >> 3), r = lane & 7;
    const int H = p.Hc * 8, W = p.Wc * 8;
    const size_t cells = (size_t)p.Hc * p.Wc;
    int i = grp;
    for (int t = blockIdx.x + grp * gridDim.x; t < n_tiles; t += 2 * gridDim.x, i += 2) {
      const uint32_t acc_phase = (uint32_t)(i >> 1) & 1u;
      const int n = t / tiles_per_img, rr = t - n * tiles_per_img;
      const int ty = rr / p.tiles_x, tx = rr - ty * p.tiles_x;
      const int cy = ty * kTH + g, cx = tx * kTW + r;
      const bool live = cy < p.Hc && cx < p.Wc;
      const size_t o0 = ((size_t)n * H + cy * 8) * W + cx * 8;
      uint2 mm[8];
      if (p.mask && live) {
#pragma unroll
        for (int dy = 0; dy < 8; ++dy) mm[dy] = __ldg(reinterpret_cast<const uint2*>(p.mask + o0 + (size_t)dy * W));
      }
      mbar_wait(&bar_tfull[grp], acc_phase);
      tc_fence_after();
      uint32_t v[80];
      const uint32_t taddr = tmem_base + (uint32_t)grp * 128 + ((uint32_t)(q * 32) << 16);
#pragma unroll
      for (int c0 = 0; c0 < 80; c0 += 16) tmem_ld16(taddr + c0, v + c0);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&bar_tempty[grp]);
      if (!live) continue;
      if (p.logits) {
        float* lp = p.logits + (size_t)n * 65 * cells + (size_t)cy * p.Wc + cx;
#pragma unroll
        for (int c = 0; c < 65; ++c) lp[(size_t)c * cells] = __uint_as_float(v[c]);
      }
      float m = -INFINITY;
#pragma unroll
      for (int c = 0; c < 65; ++c) m = fmaxf(m, __uint_as_float(v[c]));
      float s = 0.f;
#pragma unroll
      for (int c = 0; c < 65; ++c) {
        // fast exp (ex2.approx): this kernel only runs in the 16-bit operand modes, whose parity gate is 5e-3
        const float e = __expf(__uint_as_float(v[c]) - m);
        v[c] = __float_as_uint(e);
        s += e;
      }
      const float inv_s = 1.0f / s;
#pragma unroll
      for (int dy = 0; dy < 8; ++dy) {
        const size_t o = o0 + (size_t)dy * W;
        float pr[8];
#pragma unroll
        for (int dx = 0; dx < 8; ++dx) pr[dx] = __uint_as_float(v[dy * 8 + dx]) * inv_s;
        if (p.mask) {
#pragma unroll
          for (int dx = 0; dx < 4; ++dx) {
            pr[dx] *= (float)((mm[dy].x >> (8 * dx)) & 0xff);
            pr[4 + dx] *= (float)((mm[dy].y >> (8 * dx)) & 0xff);
          }
        }
        *reinterpret_cast<float4*>(p.prob + o) = make_float4(pr[0], pr[1], pr[2], pr[3]);
        *reinterpret_cast<float4*>(p.prob + o + 4) = make_float4(pr[4], pr[5], pr[6], pr[7]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256));
  }
}

}  // namespace

// operand-B image of convPb for head_tc_kernel (1x1, 256 -> 65): [cb 4][kk 4][chunk 2][n 80][8] + bias block
int spn_head_pack_layer(spn_ctx* ctx, int layer, const float* h_wfold, const float* h_bfold) {
  SpnLayer& L = ctx->layers[layer];
  if (layer != SPN_L_CONVPB || L.ks != 1 || L.cin != 256 || L.cout != 65) return SPN_OK;
  for (int bf = 0; bf < 2; ++bf) {
    std::vector<uint16_t> img(kWBytes / 2, 0);
    for (int cb = 0; cb < 4; ++cb)
      for (int kk = 0; kk < 4; ++kk)
        for (int j = 0; j < 2; ++j)
          for (int co = 0; co < 65; ++co)
            for (int e = 0; e < 8; ++e) {
              const int ci = cb * 64 + kk * 16 + j * 8 + e;
              img[(size_t)(cb * 4 + kk) * (kBlk / 2) + ((size_t)j * kN + co) * 8 + e] = to16(h_wfold[(size_t)co * 256 + ci], bf);
            }
    uint16_t* bb = img.data() + (size_t)16 * (kBlk / 2);
    for (int co = 0; co < 65; ++co) {
      const uint16_t hi = to16(h_bfold[co], bf);
      bb[(size_t)co * 8] = hi;
      bb[(size_t)co * 8 + 1] = to16(h_bfold[co] - from16(hi, bf), bf);
    }
    if (L.w16f[bf]) { cudaFree(L.w16f[bf]); L.w16f[bf] = nullptr; }
    SPN_CUDA(cudaMalloc(&L.w16f[bf], img.size() * 2));
    SPN_CUDA(cudaMemcpy(L.w16f[bf], img.data(), img.size() * 2, cudaMemcpyHostToDevice));
  }
  return SPN_OK;
}

// in: convPa output, C8 [n][32][Hc][Wc][8]; writes prob [n][8Hc][8Wc] (x mask) and optionally logits.
int spn_launch_head_tc(spn_ctx* ctx, int mode, const void* in, int n_img, int Hc, int Wc, const uint8_t* d_mask, float* d_logits,
                       float* d_prob, cudaStream_t s) {
  const SpnLayer& L = ctx->layers[SPN_L_CONVPB];
  const int bf = mode == SPN_MODE_BF16 ? 1 : 0;
  if (!L.w16f[bf]) { spn_set_error("convPb has no fused-head weights"); return SPN_E_STATE; }
  HeadParams p;
  memset(&p, 0, sizeof(p));
  p.n_img = n_img; p.Hc = Hc; p.Wc = Wc; p.tiles_x = spn_cdiv(Wc, kTW); p.tiles_y = spn_cdiv(Hc, kTH); p.is_bf16 = bf;
  p.wimg = L.w16f[bf]; p.mask = d_mask; p.logits = d_logits; p.prob = d_prob;
  const size_t dyn = (size_t)((kWBytes + 1023) & ~1023) + kOnesBytes + (size_t)kStages * kSlabBytes + 1024;
  CUtensorMap tmap;
  int rc = spn_c8_tensor_map(ctx, &tmap, in, n_img, 256, Hc, Wc, kTW, kTH, bf);
  if (rc) return rc;
  SPN_CUDA(cudaFuncSetAttribute(head_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  const long long tiles = (long long)n_img * p.tiles_x * p.tiles_y;
  const int grid = (int)(tiles < ctx->sm_count ? tiles : ctx->sm_count);
  SpnProfScope prof(ctx, SPN_L_CONVPB, s);
  SPN_CUDA(spn_launch_pdl(head_tc_kernel, dim3(grid), dim3(kThreads), dyn, s, tmap, p));
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
