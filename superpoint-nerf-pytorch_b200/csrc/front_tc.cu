// Fused front end of the fast path: homography warp -> block_1 (3x3, 1->64) -> block_2 (3x3, 64->64, ReLU, 2x2 pool)
// in ONE tcgen05 kernel.  Neither the warped image (614 KB / homography) nor block_1's output (9.8 MB / forward, the
// largest tensor of the network) ever reaches HBM: the kernel reads the fp32 source image through L2 and writes
// block_2's pooled C8 output (2.5 MB / forward).
//
// Reference semantics fused here: K.warp_perspective(image, H, bilinear) (engine_solvers/export.py:51) +
// VGG_Block 1 and 2 (models/model_utils/VGG_Backbone.py:23-36, 60-63).
//
// Per CTA tile (8 x 16 output pixels of block_2 before pooling = M 128), pipelined over tiles by warp role:
//   P  warps 10-17  bilinear-sample the 12 x 20 warped-image patch, build block_1's im2col operand A1
//                   (256 rows = the 10 x 18 halo pixels (180 used), K = 9 taps padded to 16, fp16) in SMEM;
//                   four groups of two warps that take tiles round robin
//   M  warps 0, 1   two issuers, one per tile parity, taking turns (bar_turn).  MMA1: D1 = A1 . W1 (2 x M128 N64 K16)
//                   into TMEM, issued kAhead = 3 tiles AHEAD of
//                   MMA2: D2 += slab(tap) . W2(tap) (36 x M128 N64 K16, weights resident in SMEM), rolled tap loop
//   E1 warps 6-9    D1 (bias already added through A1's ones columns, rows outside the image exactly 0 = block_2's
//                   zero padding) -> ReLU -> fp16 -> the slab
//                   [chunk][halo row][halo col][8] that MMA2's nine shifted descriptors read
//   E2 warps 2-5    D2 (bias2 added by one extra MMA against a constant ones operand) -> fp16 + ReLU in one cvt -> 2x2
//                   max-pool (two shfl.xor) -> 16-byte C8 stores
//   warp 0          also the weight loader (cp.async.bulk)
// All hand-offs are mbarriers with one arrival per warp (generic-proxy SMEM writes are published to the tensor core
// with fence.proxy.async).  How the role balance was found: DESIGN.md section 3.2.
#include "spn_common.cuh"
#include "spn_geom.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcptx;
using namespace spngeom;

constexpr int kTW = 8, kTH = 16;
constexpr int kPW = kTW + 2, kPH = kTH + 2;          // block_1 halo tile: 10 x 18 = 180 pixels
constexpr int kHalo = kPW * kPH;
constexpr int kQW = kTW + 4, kQH = kTH + 4;          // warped-image patch: 12 x 20 = 240 pixels
constexpr uint32_t kChStride = (uint32_t)kHalo * 16;  // slab bytes between 8-channel groups (2880)
constexpr int kSlabBytes = 8 * kHalo * 16;            // 23040
constexpr int kStageBytes = (kSlabBytes + 1023) & ~1023;
constexpr int kW2Bytes = 9 * 8192 + 2048;             // block_2 weights, one 64-channel slice, + its bias block
constexpr int kOnesBytes = 4096;                      // constant operand A of the bias MMA
constexpr int kW1Bytes = 2 * 64 * 16;                 // block_1 weights as operand B: [chunk 2][cout 64][8]
constexpr int kA1Rows = 256;
constexpr int kA1Bytes = 2 * kA1Rows * 16;            // [chunk 2][row 256][8 halfs]
constexpr int kStages = 4;
constexpr int kNA1 = 3;                               // D1 buffers (TMEM)
constexpr int kThreads = 576;                         // 18 warps
constexpr int kAhead = 3;                             // block_1's MMAs are issued this many tiles ahead of block_2's
constexpr int kPGroups = 4;                           // P role: the 8 warps 10-17 split into groups that take tiles round robin
constexpr int kPGroup = 256 / kPGroups;               // threads per group
constexpr int kPSamples = (12 * 20 + kPGroup - 1) / kPGroup, kPRows = (10 * 18 + kPGroup - 1) / kPGroup;   // per thread and tile
constexpr int kNA1s = kPGroups;                       // A1 / patch buffers (SMEM): one per P group

struct FrontParams {
  const float* images;   // [n_src][H][W] fp32
  const float* hinv;     // [n_src][n_h][9] pixel-space H^-1, or null (plain forward: slot == source image)
  int n_h;               // homographies per source image (slot = src * (n_h + 1) + j, j == 0 is the identity)
  int slot_begin, n_slots;
  int H, W, tiles_x, tiles_y;
  unsigned long long magic_tpi, magic_tx, magic_nh1;   // fast_div magics for tiles_per_img, tiles_x and n_h + 1
  int is_bf16;
  const void* w1img;     // operand-B image of block_1 (taps + bias rows)
  const void* w2img;     // operand-B image of block_2 (72 KB) followed by its 2 KB bias block
  void* out;             // C8 [n_slots][8][H/2][W/2][8]
};

__device__ __forceinline__ uint16_t to16(float v, int bf) {
  if (bf) {
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __half h = __float2half_rn(v);
  return *reinterpret_cast<uint16_t*>(&h);
}

__global__ void __launch_bounds__(kThreads, 1) front_tc_kernel(const FrontParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_w, bar_a1_full[kNA1s], bar_a1_empty[kNA1s], bar_d1_full[kNA1], bar_d1_empty[kNA1],
      bar_slab_full[kStages], bar_slab_empty[kStages], bar_d2_full[2], bar_d2_empty[2], bar_turn[2];
  __shared__ uint32_t tmem_base_s;
  __shared__ __align__(16) uint16_t patch_s[kNA1s][kQH * kQW];

  uint8_t* w2s = smem;                                  // 75776
  uint8_t* w1s = smem + kW2Bytes;                       // 2048
  uint8_t* a1s = w1s + kW1Bytes;                        // kNA1s x 8192  (at 77824)
  uint8_t* ones = a1s + kNA1s * kA1Bytes;               // 4096
  uint8_t* slab0 = ones + kOnesBytes;                   // kStages x 23552  (1024-aligned: every block above is a multiple of 1 KB... 2 KB)

  griddep_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int n_tiles = p.n_slots * tiles_per_img;

  // Shared-memory traffic is a first-order cost here: an M128 x N64 MMA fetches 6 KB of operands per 48 cycles = the
  // whole 128 B/cycle of the shared-memory pipe, so every other wavefront (st.shared, mbarrier arrivals and polls)
  // takes its cycle from the MMA stream.  Barriers are therefore arrived on by ONE lane per warp after __syncwarp
  // (4 arrivals instead of 128 per hand-off).
  if (threadIdx.x == 0) {
    mbar_init(&bar_w, 1);
    for (int i = 0; i < kNA1s; ++i) { mbar_init(&bar_a1_full[i], kPGroup / 32); mbar_init(&bar_a1_empty[i], 1); }
    for (int i = 0; i < kNA1; ++i) {
      mbar_init(&bar_d1_full[i], 1);   mbar_init(&bar_d1_empty[i], 4);
    }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_d2_full[i], 1); mbar_init(&bar_d2_empty[i], 4); }
    for (int i = 0; i < kStages; ++i) { mbar_init(&bar_slab_full[i], 4); mbar_init(&bar_slab_empty[i], 1); }
    for (int i = 0; i < 2; ++i) mbar_init(&bar_turn[i], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    mbar_arrive(&bar_turn[0]);  // issuer 0 owns the first turn
  }
  // A1 rows >= 180 are never written again: zero both buffers once
  for (int i = threadIdx.x; i < kNA1s * kA1Bytes / 16; i += kThreads) reinterpret_cast<uint4*>(a1s)[i] = make_uint4(0, 0, 0, 0);
  if (warp == 1) {  // TMEM: D2 2 x 64 columns + D1 3 buffers x 2 halves x 64 columns = 512 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  {
    const uint32_t one2 = p.is_bf16 ? 0x3F803F80u : 0x3C003C00u;
    for (int i = threadIdx.x; i < kOnesBytes / 16; i += kThreads)
      reinterpret_cast<uint4*>(ones)[i] = i < 128 ? make_uint4(one2, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the fills above are read by the tensor core
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  const uint32_t fmt = p.is_bf16 ? 1u : 0u;
  const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);

  if (warp <= 1) {
    // ===================== MMA issuers (warp 0 also loads the weights) =====================
    // Two issuing warps, one per tile parity: while one of them is blocked feeding the tensor pipe with its tile's 37
    // MMAs, the other one does the per-tile bookkeeping (barrier waits, fences, commits, block_1's MMAs) of the next
    // tile, so the pipe does not drain between tiles (its instruction queue is only a few MMAs deep).
    if (warp == 0) {
      if (elect_one()) {
        mbar_expect_tx(&bar_w, (uint32_t)(kW2Bytes + kW1Bytes));
        for (int o = 0; o + 8192 <= kW2Bytes; o += 8192) bulk_load(w2s + o, (const uint8_t*)p.w2img + o, 8192, &bar_w);
        bulk_load(w2s + 9 * 8192, (const uint8_t*)p.w2img + 9 * 8192, 2048, &bar_w);
        bulk_load(w1s, p.w1img, kW1Bytes, &bar_w);
      }
      __syncwarp();
    }
    const int par = warp;
    mbar_wait(&bar_w, 0);
    const uint32_t hi_a1 = (128u >> 4) | (1u << 14);                  // SBO 128 B (8 rows x 16 B), version 1
    const uint32_t lo_a1_c = ((uint32_t)(kA1Rows * 16) >> 4) << 16;   // LBO 4096 B between the two K chunks
    const uint32_t hi_b = (128u >> 4) | (1u << 14);
    const uint32_t lo_b_c = (1024u >> 4) << 16;
    const uint32_t hi_a2 = ((uint32_t)(kPW * 16) >> 4) | (1u << 14);  // SBO = one halo row (160 B)
    const uint32_t lo_a2_c = (kChStride >> 4) << 16;
    const uint32_t w1_lo = (smem_u32(w1s) >> 4) | lo_b_c, w2_lo = (smem_u32(w2s) >> 4) | lo_b_c;
    const uint32_t a1_addr = smem_u32(a1s), slab_addr = smem_u32(slab0);
    const uint32_t d1_col = tmem_base + 128;

    auto issue_mma1 = [&](int i) {  // block_1 for local tile i: D1[b][h] = A1[b] rows h*128.. times W1
      const int b = i % kNA1, ba = i % kNA1s;
      const uint32_t ph = (uint32_t)(i / kNA1) & 1u;
      mbar_wait(&bar_a1_full[ba], (uint32_t)(i / kNA1s) & 1u);
      mbar_wait(&bar_d1_empty[b], ph ^ 1u);
      tc_fence_after();
      if (elect_one()) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t a_lo = ((a1_addr + (uint32_t)ba * kA1Bytes + (uint32_t)h * 128 * 16) >> 4) | lo_a1_c;
          umma_f16_2w(d1_col + (uint32_t)(b * 2 + h) * 64, a_lo, hi_a1, w1_lo, hi_b, idesc, 0u);
        }
        umma_commit(&bar_a1_empty[ba]);
        umma_commit(&bar_d1_full[b]);
      }
      __syncwarp();
    };

    // Per issuer: MMA2(i) is followed by MMA1(i + kAhead).  block_1 of a tile is issued kAhead = 3 tiles ahead of its
    // block_2 (as far as the three D1 buffers and the four slab stages allow), so E1 has two tile times to turn D1 into
    // the slab (2117 -> 2069 cycles per tile against two tiles ahead).
    if ((int)(blockIdx.x + par * gridDim.x) < n_tiles) issue_mma1(par);
    if (par == 0 && (int)(blockIdx.x + 2 * gridDim.x) < n_tiles) issue_mma1(2);
    for (int i = par, t = blockIdx.x + par * gridDim.x; t < n_tiles; t += 2 * gridDim.x, i += 2) {
      const int stage = i % kStages, acc = i & 1;
      const uint32_t sph = (uint32_t)(i / kStages) & 1u, aph = (uint32_t)(i >> 1) & 1u;
      mbar_wait(&bar_slab_full[stage], sph);
      mbar_wait(&bar_d2_empty[acc], aph ^ 1u);
      // The two issuers take turns: block_2 of tile i+1 is not issued before the last MMA of tile i is in the queue.
      // Without the turn both warps issue at once whenever their operands are ready, the MMAs of two tiles interleave
      // (alternating accumulators), both accumulators complete together and the pipe then idles while they drain.
      mbar_wait(&bar_turn[par], aph);
      tc_fence_after();
      if (elect_one()) {
        // One ROLLED loop over the nine taps (4 MMAs per iteration, descriptors advanced by loop-carried adds).  Fully
        // unrolled, ptxas hoists the preparation of all 37 descriptor pairs to the top of the block, runs out of
        // uniform registers and spills them (MOV.SPILL / R2UR.FILL): ~10 instructions and several exposed latencies
        // per MMA, which made the issuing thread - not the tensor pipe - the pace of this stream (tools/mma_seq.cu:
        // the same 39 MMAs issue in 1873 cycles from a lean loop, 2845 with a few extra instructions per MMA).
        uint32_t a_t = ((slab_addr + (uint32_t)stage * kStageBytes) >> 4) | lo_a2_c;
        uint32_t b_t = w2_lo;
        const uint32_t d2 = tmem_base + (uint32_t)acc * 64;
        int kx = 0;
#pragma unroll 1
        for (int tap = 0; tap < 9; ++tap) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16_2w(d2, a_t + (uint32_t)kk * ((2 * kChStride) >> 4), hi_a2, b_t + (uint32_t)kk * (2048u >> 4), hi_b, idesc,
                        (tap | kk) ? 1u : 0u);
          b_t += 8192u >> 4;
          if (++kx == 3) { kx = 0; a_t += kPW - 2; } else { a_t += 1; }   // next tap: +1 pixel, or the next halo row
        }
        umma_commit(&bar_slab_empty[stage]);
        // + bias2: D2 += ones[128 x 16] . biasB[64 x 16]
        umma_f16_2w(d2, (smem_u32(ones) >> 4) | ((2048u >> 4) << 16), (128u >> 4) | (1u << 14), w2_lo + ((9u * 8192u) >> 4), hi_b,
                    idesc, 1u);
        umma_commit(&bar_d2_full[acc]);
        mbar_arrive(&bar_turn[par ^ 1]);   // the bias MMA is in the queue: the other issuer's turn
      }
      __syncwarp();
      if (t + kAhead * (int)gridDim.x < n_tiles) issue_mma1(i + kAhead);   // kAhead == 3: the other issuer's next tile
    }
  } else if (warp >= 10 && warp < 18) {
    // ===================== P: warped patch + im2col operand of block_1 =====================
    // kPGroups groups of warps take tiles round robin.  A tile's P work is one long dependent chain (coordinates ->
    // four L2 loads -> interpolation -> patch -> barrier -> im2col rows -> fence), ~2300 cycles when all eight warps
    // work on the same tile in lock step, which made P the pace of the kernel (ncu source page: P never waited for a
    // free A1 buffer while the MMA issuers waited for operands; role knock-outs in SM cycles, DESIGN.md section 3.2:
    // 2230 cycles per tile with P, 1971 without, 1969 for the MMA stream alone).  With g groups each has g tile times
    // per tile and the samples of a thread overlap their loads.
    const int grp = (warp - 10) / (8 / kPGroups);
    const int pt = threadIdx.x - 320 - grp * kPGroup;  // 0..kPGroup-1
    griddep_wait();  // the output buffer may still be read by the previous chunk's kernels; every store follows P's data
    float hm[9] = {1.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 1.f};
    int hm_slot = -1;
    for (int i = grp, t = blockIdx.x + grp * gridDim.x; t < n_tiles; t += kPGroups * gridDim.x, i += kPGroups) {
      const int b = i % kNA1s;
      const uint32_t ph = (uint32_t)(i / kNA1s) & 1u;
      const int ls = fast_div(t, p.magic_tpi), rr = t - ls * tiles_per_img;
      const int ty = fast_div(rr, p.magic_tx), tx = rr - ty * p.tiles_x;
      const int slot = p.slot_begin + ls;
      const int src = p.hinv ? fast_div(slot, p.magic_nh1) : slot;
      const int j = p.hinv ? slot - src * (p.n_h + 1) : 0;
      const float* img = p.images + (size_t)src * p.H * p.W;
      if (j > 0 && slot != hm_slot) {  // warp-uniform; a CTA's consecutive tiles mostly belong to the same slot
        const float* hp = p.hinv + ((size_t)src * p.n_h + (j - 1)) * 9;
#pragma unroll
        for (int k = 0; k < 9; ++k) hm[k] = __ldg(hp + k);
        hm_slot = slot;
      }
      // 1. the 12 x 20 patch of the warped image around the tile (zero outside the frame = block_1's padding):
      //    kPSamples samples per thread, their loads in flight together; the values are only stored once A1[b] /
      //    patch_s[b] are free (MMA1 of tile i - kNA1s has consumed them)
      float pv[kPSamples];
#pragma unroll
      for (int k = 0; k < kPSamples; ++k) {
        const int s = pt + k * kPGroup;
        const int py = s / kQW, px = s - py * kQW;
        const int y = ty * kTH - 2 + py, x = tx * kTW - 2 + px;
        float v = 0.f;
        if (s < kQH * kQW && y >= 0 && y < p.H && x >= 0 && x < p.W) {
          if (j == 0) {
            v = __ldg(&img[(size_t)y * p.W + x]);
          } else {
            float sx, sy;
            apply_h(hm, (float)x, (float)y, sx, sy);
            v = bilinear_zero_nb(img, sx, sy, p.H, p.W);
          }
        }
        pv[k] = v;
      }
      mbar_wait(&bar_a1_empty[b], ph ^ 1u);
#pragma unroll
      for (int k = 0; k < kPSamples; ++k)
        if (pt + k * kPGroup < kQH * kQW) patch_s[b][pt + k * kPGroup] = to16(pv[k], p.is_bf16);
      switch (grp) {  // one named barrier per group
        case 0: asm volatile("bar.sync 1, %0;" ::"n"(kPGroup) : "memory"); break;
        case 1: asm volatile("bar.sync 2, %0;" ::"n"(kPGroup) : "memory"); break;
        case 2: asm volatile("bar.sync 3, %0;" ::"n"(kPGroup) : "memory"); break;
        default: asm volatile("bar.sync 4, %0;" ::"n"(kPGroup) : "memory"); break;
      }
      // 2. A1 row r = halo pixel (hy, hx): its 3x3 neighbourhood (K 0..8), then two constant-one columns that
      //    multiply the (hi, lo) bias rows of W1.  Halo pixels outside the image get an all-zero row, so block_1's
      //    output there is exactly 0 = block_2's zero padding.
      const uint32_t one16 = p.is_bf16 ? 0x3F80u : 0x3C00u;
#pragma unroll
      for (int k = 0; k < kPRows; ++k) {
        const int r = pt + k * kPGroup;
        if (r >= kHalo) break;
        const int hy = r / kPW, hx = r - hy * kPW;
        const int gy = ty * kTH - 1 + hy, gx = tx * kTW - 1 + hx;
        uint4 c0 = make_uint4(0u, 0u, 0u, 0u), c1 = make_uint4(0u, 0u, 0u, 0u);
        if (gy >= 0 && gy < p.H && gx >= 0 && gx < p.W) {
          const uint16_t* q = &patch_s[b][hy * kQW + hx];
          c0.x = q[0] | ((uint32_t)q[1] << 16);
          c0.y = q[2] | ((uint32_t)q[kQW] << 16);
          c0.z = q[kQW + 1] | ((uint32_t)q[kQW + 2] << 16);
          c0.w = q[2 * kQW] | ((uint32_t)q[2 * kQW + 1] << 16);
          c1.x = q[2 * kQW + 2] | (one16 << 16);
          c1.y = one16;
        }
        uint8_t* dst = a1s + (size_t)b * kA1Bytes + (size_t)r * 16;
        *reinterpret_cast<uint4*>(dst) = c0;                    // taps 0..7
        *reinterpret_cast<uint4*>(dst + kA1Rows * 16) = c1;     // tap 8, one, one, zero padding
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_a1_full[b]);   // one arrival per warp (see the note on shared-memory traffic above)
    }
  } else if (warp >= 6 && warp < 10) {
    // ===================== E1: block_1 epilogue -> block_2's input slab =====================
    const int q = warp & 3;
    int i = 0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
      const int b = i % kNA1, stage = i % kStages;
      const uint32_t ph = (uint32_t)(i / kNA1) & 1u, sph = (uint32_t)(i / kStages) & 1u;
      mbar_wait(&bar_d1_full[b], ph);
      mbar_wait(&bar_slab_empty[stage], sph ^ 1u);
      tc_fence_after();
      uint8_t* slab = slab0 + (size_t)stage * kStageBytes;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        if (h * 128 + q * 32 >= kHalo) continue;  // warp-uniform: this lane quarter holds no halo pixel
        const int r = h * 128 + q * 32 + lane;
        uint32_t v[64];
        const uint32_t taddr = tmem_base + 128 + (uint32_t)(b * 2 + h) * 64 + ((uint32_t)(q * 32) << 16);
        tmem_ld32(taddr, v);
        tmem_ld32(taddr + 32, v + 32);
        tmem_ld_wait();
        if (r < kHalo) {  // bias is already inside D1 (ones columns of A1): ReLU + 16-bit pack + 8 x 16-byte stores
#pragma unroll
          for (int c8 = 0; c8 < 8; ++c8) {
            uint32_t w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const int c = c8 * 8 + 2 * e;
              w[e] = pack2_relu(__uint_as_float(v[c]), __uint_as_float(v[c + 1]), p.is_bf16);
            }
            *reinterpret_cast<uint4*>(slab + (size_t)c8 * kChStride + (size_t)r * 16) = make_uint4(w[0], w[1], w[2], w[3]);
          }
        }
      }
      tc_fence_before();
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(&bar_d1_empty[b]);
        mbar_arrive(&bar_slab_full[stage]);
      }
    }
  } else {
    // ===================== E2: block_2 epilogue (bias, ReLU, 2x2 max-pool, C8 store) =====================
    const int q = warp & 3;
    const int g = q * 4 + (lane >> 3), r = lane & 7;
    const int Ho = p.H >> 1, Wo = p.W >> 1;
    for (int i = 0, t = blockIdx.x; t < n_tiles; t += gridDim.x, ++i) {
      const int acc = i & 1;
      const uint32_t aph = (uint32_t)(i >> 1) & 1u;
      const int ls = fast_div(t, p.magic_tpi), rr = t - ls * tiles_per_img;
      const int ty = fast_div(rr, p.magic_tx), tx = rr - ty * p.tiles_x;
      const int y = ty * kTH + g, x = tx * kTW + r;
      mbar_wait(&bar_d2_full[acc], aph);
      tc_fence_after();
      uint32_t v[64];
      const uint32_t taddr = tmem_base + (uint32_t)acc * 64 + ((uint32_t)(q * 32) << 16);
      tmem_ld32(taddr, v);
      tmem_ld32(taddr + 32, v + 32);
      tmem_ld_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_d2_empty[acc]);
      uint32_t h2[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) h2[c] = pack2_relu(__uint_as_float(v[2 * c]), __uint_as_float(v[2 * c + 1]), p.is_bf16);
#pragma unroll
      for (int c = 0; c < 32; ++c) {  // bias is already in D2; ReLU was applied by the conversion (it commutes with the pool)
        h2[c] = max2(h2[c], __shfl_xor_sync(0xffffffffu, h2[c], 1), p.is_bf16);
        h2[c] = max2(h2[c], __shfl_xor_sync(0xffffffffu, h2[c], 8), p.is_bf16);
      }
      if (y < p.H && x < p.W && (g & 1) == 0 && (r & 1) == 0) {
        uint4* o = reinterpret_cast<uint4*>(p.out);
        const int oy = y >> 1, ox = x >> 1;
#pragma unroll
        for (int jj = 0; jj < 8; ++jj)
          o[(((size_t)ls * 8 + jj) * Ho + oy) * Wo + ox] = make_uint4(h2[4 * jj], h2[4 * jj + 1], h2[4 * jj + 2], h2[4 * jj + 3]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

}  // namespace

// d_out: C8 [n_slots][8][H/2][W/2][8]; weights of block_1 / block_2 from the context.
int spn_front_tc_launch(spn_ctx* ctx, const float* d_images, const float* d_hinv, int n_h, int slot_begin, int n_slots, int H,
                        int W, int mode, const void* w1img, void* d_out, cudaStream_t s) {
  const int bf = mode == SPN_MODE_BF16 ? 1 : 0;
  const SpnLayer& L2 = ctx->layers[SPN_L_BLOCK2];
  SPN_REQUIRE(L2.cin == 64 && L2.cout == 64 && L2.ks == 3 && L2.w16[bf], "front end needs block_2 = 3x3 conv 64->64 with packed weights");
  FrontParams p;
  memset(&p, 0, sizeof(p));
  p.images = d_images; p.hinv = d_hinv; p.n_h = n_h; p.slot_begin = slot_begin; p.n_slots = n_slots;
  p.H = H; p.W = W; p.tiles_x = spn_cdiv(W, kTW); p.tiles_y = spn_cdiv(H, kTH); p.is_bf16 = bf;
  p.magic_tpi = fast_div_magic(p.tiles_x * p.tiles_y); p.magic_tx = fast_div_magic(p.tiles_x); p.magic_nh1 = fast_div_magic(n_h + 1);
  SPN_REQUIRE((long long)n_slots * p.tiles_x * p.tiles_y * (p.tiles_x * p.tiles_y) < (1ll << 40), "too many tiles for one launch");
  SPN_REQUIRE((long long)(slot_begin + n_slots) * (n_h + 1) < (1ll << 40) && (long long)H * W < (1ll << 31), "slot range / image too large");
  p.w1img = w1img; p.w2img = L2.w16[bf];
  p.out = d_out;
  const size_t dyn = (size_t)kW2Bytes + kW1Bytes + kNA1s * kA1Bytes + kOnesBytes + (size_t)kStages * kStageBytes + 1024;
  const long long tiles = (long long)n_slots * p.tiles_x * p.tiles_y;
  const int grid = (int)(tiles < ctx->sm_count ? tiles : ctx->sm_count);
  SPN_CUDA(cudaFuncSetAttribute(front_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  SpnProfScope prof(ctx, SPN_L_BLOCK2, s);
  SPN_CUDA(spn_launch_pdl(front_tc_kernel, dim3(grid), dim3(kThreads), dyn, s, p));
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
