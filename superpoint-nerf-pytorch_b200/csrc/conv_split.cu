// Strict mode ON THE TENSOR CORES (SPN_MODE_F16X3): every convolution product a.w is evaluated as
//      a_hi.w_hi + a_hi.w_lo + a_lo.w_hi        with x_hi = fp16(x), x_lo = fp16(x - x_hi)
// (the dropped a_lo.w_lo term is ~2^-22 relative), accumulated in fp32 TMEM by tcgen05.mma kind::f16 - three MMAs per
// product, i.e. 3x the tensor work of the fast mode, for fp32-grade results (1e-4 parity gate; the FFMA strict path
// of conv_fp32.cu stays as the CUDA-core cross-check).  Activations travel between layers as TWO C8 fp16 tensors (hi, lo);
// weights are resident in shared memory as hi and lo operand-B images.
//
// Reference semantics: VGG_Block.forward (models/model_utils/VGG_Backbone.py:23-36) in fp32.
//
// Kernels (structure of conv_fold.cu / conv_tc.cu, see those files for the tile / descriptor conventions):
//   conv1_split_kernel            block_1 (Cin = 1) on CUDA cores, fp32 math, writes the (hi, lo) pair
//   conv_split_fold_kernel<NCO>   3x3 layers, horizontal taps folded into N = 3 * NCO.  NCO = 64 for 64 input channels,
//                                 NCO = 32 for 128 (hi + lo weights of a 64-wide slice would not fit in shared memory).
//                                 Per tile and 64-channel block three "virtual" K blocks are streamed: (hi slab, W_hi),
//                                 (hi slab, W_lo), (lo slab, W_hi).  Epilogue: shift-add in fp32, 2x2 max-pool and ReLU in
//                                 fp32, split into (hi, lo), two 16-byte C8 stores per channel group.
//   conv_split_1x1_kernel         1x1 heads (convPb, convDb), N = 64 slices, fp32 NCHW output.
#include <cuda.h>

#include <vector>

#include "spn_common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcptx;

__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
  const __half ha = __float2half_rn(a), hb = __float2half_rn(b);
  const __half la = __float2half_rn(a - __half2float(ha)), lb = __float2half_rn(b - __half2float(hb));
  hi = (uint32_t)__half_as_ushort(ha) | ((uint32_t)__half_as_ushort(hb) << 16);
  lo = (uint32_t)__half_as_ushort(la) | ((uint32_t)__half_as_ushort(lb) << 16);
}

// ------------------------------------------------------------------------------------------------ block_1
constexpr int kC1Px = 5, kC1Rows = 8;
__global__ void __launch_bounds__(256)
conv1_split_kernel(const float* __restrict__ img, const float* __restrict__ w /*[9][64]*/, const float* __restrict__ bias,
                   void* __restrict__ out_hi, void* __restrict__ out_lo, int B, int H, int W) {
  constexpr int TWp = 32 * kC1Px;
  __shared__ float rows[kC1Rows + 2][TWp + 2];
  __shared__ __align__(16) float ws[9 * 64 + 64];
  const int lane = threadIdx.x & 31, cg = threadIdx.x >> 5;
  const int x0 = blockIdx.x * TWp, y0 = blockIdx.y * kC1Rows, n = blockIdx.z;
  const float* im = img + (size_t)n * H * W;
  for (int i = threadIdx.x; i < 9 * 64 + 64; i += 256) ws[i] = i < 576 ? __ldg(&w[i]) : __ldg(&bias[i - 576]);
  for (int i = threadIdx.x; i < (kC1Rows + 2) * (TWp + 2); i += 256) {
    const int r = i / (TWp + 2), c = i - r * (TWp + 2);
    const int yy = y0 + r - 1, xx = x0 + c - 1;
    rows[r][c] = (yy >= 0 && yy < H && xx >= 0 && xx < W) ? __ldg(&im[(size_t)yy * W + xx]) : 0.f;
  }
  __syncthreads();
  float wr[9][8], bb[8];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int c = 0; c < 8; ++c) wr[t][c] = ws[t * 64 + cg * 8 + c];
#pragma unroll
  for (int c = 0; c < 8; ++c) bb[c] = ws[576 + cg * 8 + c];
  for (int ry = 0; ry < kC1Rows; ++ry) {
    const int y = y0 + ry;
    if (y >= H) break;
    const size_t row = (((size_t)n * 8 + cg) * H + y) * W;
#pragma unroll
    for (int k = 0; k < kC1Px; ++k) {
      const int xl = lane + 32 * k, x = x0 + xl;
      if (x >= W) break;
      float acc[8];
#pragma unroll
      for (int c = 0; c < 8; ++c) acc[c] = bb[c];
#pragma unroll
      for (int ky = 0; ky < 3; ++ky)
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const float v = rows[ry + ky][xl + kx];
#pragma unroll
          for (int c = 0; c < 8; ++c) acc[c] = fmaf(v, wr[ky * 3 + kx][c], acc[c]);
        }
      uint4 qh, ql;
      split2(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f), qh.x, ql.x);
      split2(fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f), qh.y, ql.y);
      split2(fmaxf(acc[4], 0.f), fmaxf(acc[5], 0.f), qh.z, ql.z);
      split2(fmaxf(acc[6], 0.f), fmaxf(acc[7], 0.f), qh.w, ql.w);
      reinterpret_cast<uint4*>(out_hi)[row + x] = qh;
      reinterpret_cast<uint4*>(out_lo)[row + x] = ql;
    }
  }
}

// ------------------------------------------------------------------------------------------------ 3x3, kx folded
constexpr int kTWs = 16, kTWv = 14, kTH = 8;
constexpr int kPH = kTH + 2;
constexpr uint32_t kChStride = (uint32_t)kPH * kTWs * 16;
constexpr int kSlabBytes = 8 * kPH * kTWs * 16;   // 20480
constexpr int kOnesBytes = 4096;
constexpr int kFoldThreads = 320;
constexpr int kMaxStages = 6;

struct SplitFoldParams {
  int n_img, H, W;
  int cin_blocks, cout_slices, cout;
  int relu, pool;
  int tiles_x, tiles_y, stages;
  void* out_hi;
  void* out_lo;
  const void* wimg;   // per slice: [W_hi: cin block][ky 3][k-step 4][chunk 2][n = kx*NCO+co][8], same for W_lo, bias block
};

template <int NCO>
__global__ void __launch_bounds__(kFoldThreads, 1)
conv_split_fold_kernel(const __grid_constant__ CUtensorMap tmap_hi, const __grid_constant__ CUtensorMap tmap_lo, const SplitFoldParams p) {
  constexpr int N = 3 * NCO;
  constexpr int kBlk = 2 * N * 16;
  constexpr int kAccStride = NCO == 64 ? 192 : 128;   // TMEM columns between the two accumulators
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full[kMaxStages], bar_empty[kMaxStages], bar_w, bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wbytes = (2 * p.cin_blocks * 12 + 1) * kBlk;
  uint8_t* wsm = smem;
  uint8_t* ones = smem + ((wbytes + 1023) & ~1023);
  uint8_t* slab0 = ones + kOnesBytes;
  const int slice = blockIdx.x % p.cout_slices;
  const int cta_in_slice = blockIdx.x / p.cout_slices, ctas_per_slice = gridDim.x / p.cout_slices;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int n_tiles = p.n_img * tiles_per_img;
  const int upt = 3 * p.cin_blocks;   // virtual K blocks per tile

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_w, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < kOnesBytes / 16; i += kFoldThreads)
    reinterpret_cast<uint4*>(ones)[i] = i < 128 ? make_uint4(0x3C003C00u, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      mbar_expect_tx(&bar_w, (uint32_t)wbytes);
      const uint8_t* wsrc = (const uint8_t*)p.wimg + (size_t)slice * wbytes;
      for (int o = 0; o < wbytes; o += kBlk) bulk_load(wsm + o, wsrc + o, kBlk, &bar_w);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice) {
      const int n = t / tiles_per_img, r = t - n * tiles_per_img;
      const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
      for (int u = 0; u < upt; ++u) {
        const int cb = u / 3, v = u - cb * 3;   // v: 0 (hi, W_hi)  1 (hi, W_lo)  2 (lo, W_hi)
        mbar_wait(&bar_empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bar_full[stage], (uint32_t)kSlabBytes);
          tma_load_4d(slab0 + (size_t)stage * kSlabBytes, v == 2 ? &tmap_lo : &tmap_hi, &bar_full[stage], (tx * kTWv - 1) * 8,
                      ty * kTH - 1, cb * 8, n);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc = (1u << 4) | (((uint32_t)N >> 3) << 17) | ((128u >> 4) << 24);   // fp16 x fp16 -> fp32, M 128
    const uint32_t a_hi = (128u >> 4) | (1u << 14);
    const uint32_t a_lo_c = (kChStride >> 4) << 16;
    const uint32_t b_hi = (128u >> 4) | (1u << 14);
    const uint32_t b_lo_c = (((uint32_t)N * 16u) >> 4) << 16;
    const uint32_t o_lo = (smem_u32(ones) >> 4) | ((2048u >> 4) << 16);
    mbar_wait(&bar_w, 0);
    const uint32_t w_addr = smem_u32(wsm), slab_addr = smem_u32(slab0);
    int stage = 0, i = 0;
    uint32_t phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice, ++i) {
      const int acc = i & 1;
      mbar_wait(&bar_tempty[acc], ((uint32_t)(i >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * kAccStride;
      for (int u = 0; u < upt; ++u) {
        const int cb = u / 3, v = u - cb * 3;
        mbar_wait(&bar_full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_lo = ((slab_addr + (uint32_t)stage * kSlabBytes) >> 4) | a_lo_c;
          const uint32_t b_lo = ((w_addr + (uint32_t)((v == 1 ? p.cin_blocks : 0) + cb) * (12 * kBlk)) >> 4) | b_lo_c;
#pragma unroll
          for (int m = 0; m < 12; ++m) {
            const int ky = m >> 2, kk = m & 3;
            const uint32_t aoff = ((uint32_t)ky * (kTWs * 16) + (uint32_t)kk * 2 * kChStride) >> 4;
            const uint32_t boff = ((uint32_t)(ky * 4 + kk) * kBlk) >> 4;
            umma_f16_2w(d_tmem, a_lo + aoff, a_hi, b_lo + boff, b_hi, idesc, (u | m) ? 1u : 0u);
          }
          umma_commit(&bar_empty[stage]);
          if (u == upt - 1) {
            const uint32_t bb_lo = ((w_addr + (uint32_t)(2 * p.cin_blocks) * (12 * kBlk)) >> 4) | b_lo_c;
            umma_f16_2w(d_tmem, o_lo, a_hi, bb_lo, b_hi, idesc, 1u);   // + bias (hi, lo halves) in the kx = 1 column block
            umma_commit(&bar_tfull[acc]);
          }
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ===================== epilogue: two groups alternate tiles =====================
    const int group = (warp - 2) >> 2;
    const int q = warp & 3;
    const int r = 2 * q + (lane >> 4), x = lane & 15;
    const int Ho = p.pool ? p.H >> 1 : p.H, Wo = p.pool ? p.W >> 1 : p.W;
    const int cgroups = p.cout_slices * (NCO / 8);
    int i = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice, ++i) {
      if ((i & 1) != group) continue;
      const int acc = i & 1;
      const uint32_t acc_phase = (uint32_t)(i >> 1) & 1u;
      const int n = t / tiles_per_img, rr = t - n * tiles_per_img;
      const int ty = rr / p.tiles_x, tx = rr - ty * p.tiles_x;
      const int y = ty * kTH + r, gx = tx * kTWv - 1 + x;
      mbar_wait(&bar_tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * kAccStride + ((uint32_t)(q * 32) << 16);
      bool writer = x >= 1 && x <= kTWv && gx < p.W && y < p.H;
      int oy = y, ox = gx;
      if (p.pool) {
        writer = writer && (x & 1) && ((lane >> 4) == 0);
        oy = y >> 1; ox = gx >> 1;
      }
#pragma unroll 1
      for (int c0 = 0; c0 < NCO; c0 += 32) {
        uint32_t f0[32], f1[32], f2[32];
        tmem_ld32(taddr + c0, f0);
        tmem_ld32(taddr + NCO + c0, f1);
        tmem_ld32(taddr + 2 * NCO + c0, f2);
        tmem_ld_wait();
        if (c0 + 32 >= NCO) {   // last chunk read: the accumulator may be overwritten
          tc_fence_before();
          mbar_arrive(&bar_tempty[acc]);
        }
        float a[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          a[c] = __shfl_up_sync(0xffffffffu, __uint_as_float(f0[c]), 1) + __uint_as_float(f1[c]) +
                 __shfl_down_sync(0xffffffffu, __uint_as_float(f2[c]), 1);
          if (p.pool) {
            a[c] = fmaxf(a[c], __shfl_down_sync(0xffffffffu, a[c], 1));
            a[c] = fmaxf(a[c], __shfl_xor_sync(0xffffffffu, a[c], 16));
          }
          if (p.relu) a[c] = fmaxf(a[c], 0.f);
        }
        if (writer) {
          uint4* oh = reinterpret_cast<uint4*>(p.out_hi);
          uint4* ol = reinterpret_cast<uint4*>(p.out_lo);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int cgp = slice * (NCO / 8) + (c0 >> 3) + j;
            if (cgp * 8 < p.cout) {
              uint4 qh, ql;
              split2(a[8 * j], a[8 * j + 1], qh.x, ql.x);
              split2(a[8 * j + 2], a[8 * j + 3], qh.y, ql.y);
              split2(a[8 * j + 4], a[8 * j + 5], qh.z, ql.z);
              split2(a[8 * j + 6], a[8 * j + 7], qh.w, ql.w);
              const size_t o = (((size_t)n * cgroups + cgp) * Ho + oy) * Wo + ox;
              oh[o] = qh;
              ol[o] = ql;
            }
          }
        }
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

// ------------------------------------------------------------------------------------------------ 1x1 heads
constexpr int kTW1 = 8, kTH1 = 16;
constexpr int k1Threads = 192;
constexpr int kWBlk1 = 8192;        // [k-step 4][chunk 2][cout 64][8]
constexpr int kBias1 = 2048;
constexpr int kSlab1 = 8 * kTH1 * kTW1 * 16;   // 16384

struct Split1x1Params {
  int n_img, H, W, cin_blocks, cout_slices, cout, stages, tiles_x, tiles_y;
  float* out;          // NCHW fp32
  const void* wimg;    // per slice: [W_hi: cin block][8 KB], [W_lo: ...], bias block
};

__global__ void __launch_bounds__(k1Threads, 1)
conv_split_1x1_kernel(const __grid_constant__ CUtensorMap tmap_hi, const __grid_constant__ CUtensorMap tmap_lo, const Split1x1Params p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full[kMaxStages], bar_empty[kMaxStages], bar_w, bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_s;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t ch_stride = (uint32_t)kTH1 * kTW1 * 16;
  const int wbytes = 2 * p.cin_blocks * kWBlk1 + kBias1;
  uint8_t* wsm = smem;
  uint8_t* ones = smem + ((wbytes + 1023) & ~1023);
  uint8_t* slab0 = ones + kOnesBytes;
  const int slice = blockIdx.x % p.cout_slices;
  const int cta_in_slice = blockIdx.x / p.cout_slices, ctas_per_slice = gridDim.x / p.cout_slices;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int n_tiles = p.n_img * tiles_per_img;
  const int upt = 3 * p.cin_blocks;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_w, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int i = threadIdx.x; i < kOnesBytes / 16; i += k1Threads)
    reinterpret_cast<uint4*>(ones)[i] = i < 128 ? make_uint4(0x3C003C00u, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(128));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    if (elect_one()) {
      mbar_expect_tx(&bar_w, (uint32_t)wbytes);
      const uint8_t* wsrc = (const uint8_t*)p.wimg + (size_t)slice * wbytes;
      for (int o = 0; o + kWBlk1 <= wbytes; o += kWBlk1) bulk_load(wsm + o, wsrc + o, kWBlk1, &bar_w);
      bulk_load(wsm + wbytes - kBias1, wsrc + wbytes - kBias1, kBias1, &bar_w);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice) {
      const int n = t / tiles_per_img, r = t - n * tiles_per_img;
      const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
      for (int u = 0; u < upt; ++u) {
        const int cb = u / 3, v = u - cb * 3;
        mbar_wait(&bar_empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bar_full[stage], (uint32_t)kSlab1);
          tma_load_4d(slab0 + (size_t)stage * kSlab1, v == 2 ? &tmap_lo : &tmap_hi, &bar_full[stage], tx * kTW1 * 8, ty * kTH1, cb * 8, n);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    const uint32_t idesc = (1u << 4) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t a_hi = ((uint32_t)(kTW1 * 16) >> 4) | (1u << 14), b_hi = (128u >> 4) | (1u << 14);
    const uint32_t a_lo_c = (ch_stride >> 4) << 16, b_lo_c = (1024u >> 4) << 16;
    mbar_wait(&bar_w, 0);
    const uint32_t w_addr = smem_u32(wsm), slab_addr = smem_u32(slab0);
    int stage = 0, i = 0;
    uint32_t phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice, ++i) {
      const int acc = i & 1;
      mbar_wait(&bar_tempty[acc], ((uint32_t)(i >> 1) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * 64;
      for (int u = 0; u < upt; ++u) {
        const int cb = u / 3, v = u - cb * 3;
        mbar_wait(&bar_full[stage], phase);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t a_lo = ((slab_addr + (uint32_t)stage * kSlab1) >> 4) | a_lo_c;
          const uint32_t b_lo = ((w_addr + (uint32_t)((v == 1 ? p.cin_blocks : 0) + cb) * kWBlk1) >> 4) | b_lo_c;
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_f16_2w(d_tmem, a_lo + (((uint32_t)kk * 2 * ch_stride) >> 4), a_hi, b_lo + (((uint32_t)kk * 2048) >> 4), b_hi, idesc,
                        (u | kk) ? 1u : 0u);
          umma_commit(&bar_empty[stage]);
          if (u == upt - 1) {
            const uint32_t o_lo = (smem_u32(ones) >> 4) | ((2048u >> 4) << 16);
            const uint32_t bb_lo = ((w_addr + (uint32_t)(2 * p.cin_blocks) * kWBlk1) >> 4) | b_lo_c;
            umma_f16_2w(d_tmem, o_lo, (128u >> 4) | (1u << 14), bb_lo, b_hi, idesc, 1u);
            umma_commit(&bar_tfull[acc]);
          }
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    const int q = warp & 3;
    const int g = q * 4 + (lane >> 3), r = lane & 7;
    int i = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice, ++i) {
      const int acc = i & 1;
      const int n = t / tiles_per_img, rr = t - n * tiles_per_img;
      const int ty = rr / p.tiles_x, tx = rr - ty * p.tiles_x;
      const int y = ty * kTH1 + g, x = tx * kTW1 + r;
      mbar_wait(&bar_tfull[acc], (uint32_t)(i >> 1) & 1u);
      tc_fence_after();
      uint32_t v[64];
      const uint32_t taddr = tmem_base + (uint32_t)acc * 64 + ((uint32_t)(q * 32) << 16);
      tmem_ld32(taddr, v);
      tmem_ld32(taddr + 32, v + 32);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&bar_tempty[acc]);
      if (y < p.H && x < p.W) {
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          const int co = slice * 64 + c;
          if (co < p.cout) p.out[(((size_t)n * p.cout + co) * p.H + y) * p.W + x] = __uint_as_float(v[c]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128));
  }
}

// ------------------------------------------------------------------------------------------------ layout conversions (layer-level API)
__global__ void nchw_to_c8_split_kernel(const float* __restrict__ in, void* __restrict__ hi, void* __restrict__ lo, int B, int C, int H, int W) {
  const size_t total = (size_t)B * (C / 8) * H * W;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int x = i % W, y = (i / W) % H;
  const int cgp = (i / ((size_t)W * H)) % (C / 8);
  const int n = i / ((size_t)W * H * (C / 8));
  float v[8];
  for (int e = 0; e < 8; ++e) v[e] = in[(((size_t)n * C + cgp * 8 + e) * H + y) * W + x];
  uint4 qh, ql;
  split2(v[0], v[1], qh.x, ql.x); split2(v[2], v[3], qh.y, ql.y); split2(v[4], v[5], qh.z, ql.z); split2(v[6], v[7], qh.w, ql.w);
  reinterpret_cast<uint4*>(hi)[i] = qh;
  reinterpret_cast<uint4*>(lo)[i] = ql;
}
__global__ void c8_split_to_nchw_kernel(const void* __restrict__ hi, const void* __restrict__ lo, float* __restrict__ out, int B, int C, int H, int W) {
  const size_t total = (size_t)B * (C / 8) * H * W;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int x = i % W, y = (i / W) % H;
  const int cgp = (i / ((size_t)W * H)) % (C / 8);
  const int n = i / ((size_t)W * H * (C / 8));
  const uint4 qh = reinterpret_cast<const uint4*>(hi)[i], ql = reinterpret_cast<const uint4*>(lo)[i];
  const uint32_t h4[4] = {qh.x, qh.y, qh.z, qh.w}, l4[4] = {ql.x, ql.y, ql.z, ql.w};
  for (int e = 0; e < 4; ++e) {
    const __half2 th = *reinterpret_cast<const __half2*>(&h4[e]), tl = *reinterpret_cast<const __half2*>(&l4[e]);
    out[(((size_t)n * C + cgp * 8 + 2 * e) * H + y) * W + x] = __half2float(th.x) + __half2float(tl.x);
    out[(((size_t)n * C + cgp * 8 + 2 * e + 1) * H + y) * W + x] = __half2float(th.y) + __half2float(tl.y);
  }
}

int fold_nco(const SpnLayer& L) { return L.cin == 64 ? 64 : 32; }

// one 3x3 layer: (in_hi, in_lo) C8 -> (out_hi, out_lo) C8 (pooled or not)
int launch_split_fold(spn_ctx* ctx, int layer, const void* in_hi, const void* in_lo, void* out_hi, void* out_lo, int n_img, int H, int W,
                      bool relu, bool pool, cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  if (!L.w16x) { spn_set_error("layer %d has no split (f16x3) weights", layer); return SPN_E_STATE; }
  const int nco = fold_nco(L);
  const int kBlk = 2 * 3 * nco * 16;
  SplitFoldParams p;
  memset(&p, 0, sizeof(p));
  p.n_img = n_img; p.H = H; p.W = W; p.cin_blocks = L.cin / 64; p.cout_slices = (L.cout + nco - 1) / nco; p.cout = L.cout;
  p.relu = relu; p.pool = pool; p.tiles_x = spn_cdiv(W, kTWv); p.tiles_y = spn_cdiv(H, kTH);
  const int wbytes = (2 * p.cin_blocks * 12 + 1) * kBlk;
  const int wres = ((wbytes + 1023) & ~1023) + kOnesBytes;
  p.stages = (227 * 1024 - 2048 - wres - 1024) / kSlabBytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  SPN_REQUIRE(p.stages >= 2, "split layer %d does not fit in shared memory (%d weight bytes)", layer, wbytes);
  p.out_hi = out_hi; p.out_lo = out_lo; p.wimg = L.w16x;
  const size_t dyn = (size_t)wres + (size_t)p.stages * kSlabBytes + 1024;
  CUtensorMap th, tl;
  int rc = spn_c8_tensor_map(ctx, &th, in_hi, n_img, L.cin, H, W, kTWs, kPH, 0);
  if (rc) return rc;
  if ((rc = spn_c8_tensor_map(ctx, &tl, in_lo, n_img, L.cin, H, W, kTWs, kPH, 0))) return rc;
  const long long work = (long long)n_img * p.tiles_x * p.tiles_y * p.cout_slices;
  int grid = ctx->sm_count;
  if (work < grid) grid = (int)work;
  grid = grid / p.cout_slices * p.cout_slices;
  if (grid < p.cout_slices) grid = p.cout_slices;
  SpnProfScope prof(ctx, layer, s);
  if (nco == 64) {
    SPN_CUDA(cudaFuncSetAttribute(conv_split_fold_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    conv_split_fold_kernel<64><<<grid, kFoldThreads, dyn, s>>>(th, tl, p);
  } else {
    SPN_CUDA(cudaFuncSetAttribute(conv_split_fold_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    conv_split_fold_kernel<32><<<grid, kFoldThreads, dyn, s>>>(th, tl, p);
  }
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

// one 1x1 layer: (in_hi, in_lo) C8 -> fp32 NCHW
int launch_split_1x1(spn_ctx* ctx, int layer, const void* in_hi, const void* in_lo, float* out, int n_img, int H, int W, cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  if (!L.w16x) { spn_set_error("layer %d has no split (f16x3) weights", layer); return SPN_E_STATE; }
  Split1x1Params p;
  memset(&p, 0, sizeof(p));
  p.n_img = n_img; p.H = H; p.W = W; p.cin_blocks = L.cin / 64; p.cout_slices = (L.cout + 63) / 64; p.cout = L.cout;
  p.tiles_x = spn_cdiv(W, kTW1); p.tiles_y = spn_cdiv(H, kTH1);
  const int wbytes = 2 * p.cin_blocks * kWBlk1 + kBias1;
  const int wres = ((wbytes + 1023) & ~1023) + kOnesBytes;
  p.stages = (227 * 1024 - 2048 - wres - 1024) / kSlab1;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  SPN_REQUIRE(p.stages >= 2, "split 1x1 layer %d does not fit in shared memory", layer);
  p.out = out; p.wimg = L.w16x;
  const size_t dyn = (size_t)wres + (size_t)p.stages * kSlab1 + 1024;
  CUtensorMap th, tl;
  int rc = spn_c8_tensor_map(ctx, &th, in_hi, n_img, L.cin, H, W, kTW1, kTH1, 0);
  if (rc) return rc;
  if ((rc = spn_c8_tensor_map(ctx, &tl, in_lo, n_img, L.cin, H, W, kTW1, kTH1, 0))) return rc;
  const long long work = (long long)n_img * p.tiles_x * p.tiles_y * p.cout_slices;
  int grid = ctx->sm_count;
  if (work < grid) grid = (int)work;
  grid = grid / p.cout_slices * p.cout_slices;
  if (grid < p.cout_slices) grid = p.cout_slices;
  SPN_CUDA(cudaFuncSetAttribute(conv_split_1x1_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  SpnProfScope prof(ctx, layer, s);
  conv_split_1x1_kernel<<<grid, k1Threads, dyn, s>>>(th, tl, p);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

struct SplitPlan {
  size_t a, b, feat, head, logits, total;   // bytes of ONE half (hi or lo); every activation buffer holds hi then lo
};
SplitPlan split_plan(int B, int H, int W) {
  SplitPlan p;
  const size_t hw = (size_t)H * W;
  p.a = (size_t)B * 64 * hw * 2;
  p.b = (size_t)B * 64 * hw / 4 * 2;
  p.feat = (size_t)B * 128 * hw / 64 * 2;
  p.head = (size_t)B * 256 * hw / 64 * 2;
  p.logits = (size_t)B * 65 * hw / 64 * 4;
  p.total = 2 * (p.a + p.b + p.feat + p.head) + p.logits + 4096;
  return p;
}

}  // namespace

// hi / lo operand-B images of one layer (fp16 only): see the kernel comments for the layouts
int spn_split_pack_layer(spn_ctx* ctx, int layer, const float* w, const float* b) {
  SpnLayer& L = ctx->layers[layer];
  if (L.w16x) { cudaFree(L.w16x); L.w16x = nullptr; }
  if (L.cin % 64 != 0) return SPN_OK;
  std::vector<uint16_t> img;
  auto hi_of = [&](float v) { return to16(v, 0); };
  auto lo_of = [&](float v) { return to16(v - from16(to16(v, 0), 0), 0); };
  if (L.ks == 3) {
    const int nco = fold_nco(L), N = 3 * nco, blk = 2 * N * 8 /* halfs */, cbs = L.cin / 64, slices = (L.cout + nco - 1) / nco;
    const size_t per_slice = (size_t)(2 * cbs * 12 + 1) * blk;
    img.assign(per_slice * slices, 0);
    for (int sl = 0; sl < slices; ++sl) {
      uint16_t* base = img.data() + per_slice * sl;
      for (int part = 0; part < 2; ++part)
        for (int cb = 0; cb < cbs; ++cb)
          for (int ky = 0; ky < 3; ++ky)
            for (int kk = 0; kk < 4; ++kk) {
              uint16_t* bl = base + ((size_t)((part * cbs + cb) * 3 + ky) * 4 + kk) * blk;
              for (int j = 0; j < 2; ++j)
                for (int kx = 0; kx < 3; ++kx)
                  for (int co = 0; co < nco; ++co)
                    for (int e = 0; e < 8; ++e) {
                      const int c = sl * nco + co, ci = cb * 64 + kk * 16 + j * 8 + e;
                      if (c >= L.cout) continue;
                      const float v = w[((size_t)c * L.cin + ci) * 9 + ky * 3 + kx];
                      bl[((size_t)j * N + kx * nco + co) * 8 + e] = part ? lo_of(v) : hi_of(v);
                    }
            }
      uint16_t* bb = base + (size_t)(2 * cbs * 12) * blk;
      for (int co = 0; co < nco; ++co) {
        const int c = sl * nco + co;
        if (c >= L.cout) continue;
        bb[((size_t)nco + co) * 8] = hi_of(b[c]);
        bb[((size_t)nco + co) * 8 + 1] = lo_of(b[c]);
      }
    }
  } else {
    const int cbs = L.cin / 64, slices = (L.cout + 63) / 64;
    const size_t per_slice = (size_t)2 * cbs * (kWBlk1 / 2) + kBias1 / 2;
    img.assign(per_slice * slices, 0);
    for (int sl = 0; sl < slices; ++sl) {
      uint16_t* base = img.data() + per_slice * sl;
      for (int part = 0; part < 2; ++part)
        for (int cb = 0; cb < cbs; ++cb)
          for (int kk = 0; kk < 4; ++kk)
            for (int j = 0; j < 2; ++j)
              for (int co = 0; co < 64; ++co)
                for (int e = 0; e < 8; ++e) {
                  const int c = sl * 64 + co, ci = cb * 64 + kk * 16 + j * 8 + e;
                  if (c >= L.cout) continue;
                  const float v = w[(size_t)c * L.cin + ci];
                  base[(size_t)(part * cbs + cb) * (kWBlk1 / 2) + (size_t)kk * 1024 + ((size_t)j * 64 + co) * 8 + e] = part ? lo_of(v) : hi_of(v);
                }
      uint16_t* bb = base + (size_t)2 * cbs * (kWBlk1 / 2);
      for (int co = 0; co < 64; ++co) {
        const int c = sl * 64 + co;
        if (c >= L.cout) continue;
        bb[(size_t)co * 8] = hi_of(b[c]);
        bb[(size_t)co * 8 + 1] = lo_of(b[c]);
      }
    }
  }
  SPN_CUDA(cudaMalloc(&L.w16x, img.size() * 2));
  SPN_CUDA(cudaMemcpy(L.w16x, img.data(), img.size() * 2, cudaMemcpyHostToDevice));
  return SPN_OK;
}

// VGG_BACKBONE.forward in split mode: leaves the (hi, lo) feature map in the workspace (ctx->feat = hi, lo follows)
int spn_split_encoder(spn_ctx* ctx, const float* d_images, int B, int H, int W, cudaStream_t s) {
  const float* w1 = spn_tc_block1_weights(ctx);
  if (!w1) { spn_set_error("block_1 has no weights"); return SPN_E_STATE; }
  const SplitPlan pl = split_plan(B, H, W);
  int rc = spn_ensure_ws(ctx, pl.total, s);
  if (rc) return rc;
  char* A = ctx->ws;               // hi at A, lo at A + pl.a
  char* Bq = A + 2 * pl.a;
  char* F = Bq + 2 * pl.b;
  {
    SpnProfScope prof(ctx, SPN_L_BLOCK1, s);
    dim3 g(spn_cdiv(W, 32 * kC1Px), spn_cdiv(H, kC1Rows), B);
    conv1_split_kernel<<<g, 256, 0, s>>>(d_images, w1, ctx->layers[0].bias, A, A + pl.a, B, H, W);
    SPN_CHECK_LAUNCH(ctx);
  }
  // every buffer is used with the (hi, lo) halves at distance = that tensor's own size
  auto half = [&](int ch, int h, int w) { return (size_t)B * ch * h * w * 2; };
  if ((rc = launch_split_fold(ctx, 1, A, A + pl.a, Bq, Bq + half(64, H / 2, W / 2), B, H, W, true, true, s))) return rc;
  if ((rc = launch_split_fold(ctx, 2, Bq, Bq + half(64, H / 2, W / 2), A, A + half(64, H / 2, W / 2), B, H / 2, W / 2, true, false, s))) return rc;
  if ((rc = launch_split_fold(ctx, 3, A, A + half(64, H / 2, W / 2), Bq, Bq + half(64, H / 4, W / 4), B, H / 2, W / 2, true, true, s))) return rc;
  if ((rc = launch_split_fold(ctx, 4, Bq, Bq + half(64, H / 4, W / 4), A, A + half(128, H / 4, W / 4), B, H / 4, W / 4, true, false, s))) return rc;
  if ((rc = launch_split_fold(ctx, 5, A, A + half(128, H / 4, W / 4), Bq, Bq + half(128, H / 8, W / 8), B, H / 4, W / 4, true, true, s))) return rc;
  if ((rc = launch_split_fold(ctx, 6, Bq, Bq + half(128, H / 8, W / 8), A, A + half(128, H / 8, W / 8), B, H / 8, W / 8, true, false, s))) return rc;
  if ((rc = launch_split_fold(ctx, 7, A, A + half(128, H / 8, W / 8), F, F + pl.feat, B, H / 8, W / 8, true, false, s))) return rc;
  ctx->feat = F;
  return SPN_OK;
}

// convPa + convPb (or convDa + convDb) in split mode: fp32 NCHW output
int spn_split_head(spn_ctx* ctx, int layer_a, int layer_b, int B, int H, int W, float* d_out, cudaStream_t s) {
  const SplitPlan pl = split_plan(B, H, W);
  char* F = (char*)ctx->feat;
  char* Hd = ctx->ws + 2 * pl.a + 2 * pl.b + 2 * pl.feat;
  const int Hc = H / 8, Wc = W / 8;
  int rc = launch_split_fold(ctx, layer_a, F, F + pl.feat, Hd, Hd + pl.head, B, Hc, Wc, true, false, s);
  if (rc) return rc;
  return launch_split_1x1(ctx, layer_b, Hd, Hd + pl.head, d_out, B, Hc, Wc, s);
}

float* spn_split_logits_scratch(spn_ctx* ctx, int B, int H, int W) {
  const SplitPlan pl = split_plan(B, H, W);
  return (float*)(ctx->ws + 2 * (pl.a + pl.b + pl.feat + pl.head));
}

// layer-level entry (spn_conv_layer, mode F16X3): NCHW fp32 in / out
int spn_split_conv_layer(spn_ctx* ctx, int layer, const float* d_in, int B, int H, int W, bool relu, bool pool, float* d_out, cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  const int Ho = pool ? H / 2 : H, Wo = pool ? W / 2 : W;
  const size_t in_half = (size_t)B * L.cin * H * W * 2;
  const int cpad = (L.cout + 7) / 8 * 8;
  const size_t out_half = (size_t)B * cpad * Ho * Wo * 2;
  int rc = spn_ensure_ws(ctx, 2 * in_half + 2 * out_half + 4096, s);
  if (rc) return rc;
  char* ih = ctx->ws;
  char* il = ih + in_half;
  char* oh = il + in_half;
  char* ol = oh + out_half;
  const size_t nin = (size_t)B * (L.cin / 8) * H * W;
  nchw_to_c8_split_kernel<<<(unsigned)((nin + 255) / 256), 256, 0, s>>>(d_in, ih, il, B, L.cin, H, W);
  SPN_CHECK_LAUNCH(ctx);
  if (L.ks == 1) {
    SPN_REQUIRE(!relu && !pool, "split 1x1 layers are the heads' output convolutions (no ReLU / pool)");
    return launch_split_1x1(ctx, layer, ih, il, d_out, B, H, W, s);
  }
  SPN_REQUIRE(L.cout % 8 == 0, "split 3x3 layers need Cout %% 8 == 0");
  if ((rc = launch_split_fold(ctx, layer, ih, il, oh, ol, B, H, W, relu, pool, s))) return rc;
  const size_t nout = (size_t)B * (L.cout / 8) * Ho * Wo;
  c8_split_to_nchw_kernel<<<(unsigned)((nout + 255) / 256), 256, 0, s>>>(oh, ol, d_out, B, L.cout, Ho, Wo);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
