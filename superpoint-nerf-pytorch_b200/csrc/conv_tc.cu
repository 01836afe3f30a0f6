// tcgen05 1x1 convolution with fp32 NCHW output: the 1x1 heads convDb and, on the unfused path (option fuse_head = 0),
// convPb, and the single-layer entry point spn_conv_layer for 1x1 layers.  fp16/bf16 operands, fp32 accumulation in TMEM.
// The 3x3 layers run in conv_fold.cu (block_3..8, convPa, convDa) and front_tc.cu (block_1 + block_2).
//
// Data layout in HBM ("C8"): act[n][C/8][H][W][8] halfs - i.e. 16-byte channel groups, pixels contiguous along W.
// This is exactly the UMMA no-swizzle K-major operand layout (core matrix = 8 rows x 16 bytes), so ONE TMA box
//   (W: 8 pixels) x (H: 16 rows) x (8 channel groups)                    [tile of 64 input channels]
// lands in shared memory as slab[chunk][row][col][8] and is read directly as operand A.
//
// GEMM view per CTA tile: M = 128 pixels (8 wide x 16 high; TMEM lane = pixel), N = 64 output channels (one
// "slice"; a CTA keeps its slice's weights for all K resident in SMEM), K = Cin.  MMA = tcgen05.mma
// cta_group::1 kind::f16 M128 N64 K16, A and B from SMEM descriptors (SWIZZLE_NONE, LBO = channel-group stride,
// SBO = 8-row-group stride), D = 64 fp32 TMEM columns, double buffered so the epilogue of tile i overlaps the MMAs
// of tile i+1.
//
// Warp roles (192 threads, persistent, one CTA per SM): warp 0 = TMA producer (weights once via cp.async.bulk,
// then one 16 KB slab per (tile, 64-channel block) through a ring of mbarriers), warp 1 = MMA issuer (one elected
// lane) + TMEM allocator, warps 2-5 = epilogue (tcgen05.ld -> optional ReLU -> fp32 NCHW stores).
#include <cuda.h>

#include <string>
#include <vector>

#include "spn_common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcptx;

constexpr int kTW = 8, kTH = 16;              // output tile: 8 x 16 pixels = 128 GEMM rows
constexpr int kThreads = 192;
constexpr int kWBlockBytes = 8192;            // weights of one cin block: 4 k-steps x 2 chunks x 64 cout x 16 B
constexpr int kSlabBytes = 8 * kTH * kTW * 16;  // one TMA box: 8 channel groups x 16 rows x 8 pixels x 16 B
constexpr uint32_t kChStride = (uint32_t)kTH * kTW * 16;  // bytes between 8-channel groups inside a slab
constexpr int kMaxStages = 6;
constexpr int kBiasBlockBytes = 2048;         // bias as operand B: [chunk 2][cout 64][8], k 0 / 1 = hi / lo halves
constexpr int kOnesBytes = 4096;              // constant operand A of the bias MMA: [chunk 2][128 rows][8]

struct TcParams {
  int n_img, H, W;        // input == conv-output spatial size
  int cin_blocks;         // Cin / 64
  int cout_slices;        // ceil(Cout / 64)
  int cout;               // real number of output channels
  int relu;
  int is_bf16;
  int tiles_x, tiles_y;
  int stages;
  float* out;             // NCHW fp32 [n][cout][H][W]
  const void* wimg;       // [cout_slices][cin_blocks][4][2][64][8] halfs + per slice the bias block
};

// Constant A operand of the bias MMA: row r = (1, 1, 0, ..., 0) in K chunk 0, zeros in chunk 1.
__device__ __forceinline__ void fill_ones_operand(uint8_t* ones, int is_bf16, int tid, int nthreads) {
  const uint32_t one2 = is_bf16 ? 0x3F803F80u : 0x3C003C00u;
  for (int i = tid; i < kOnesBytes / 16; i += nthreads)
    reinterpret_cast<uint4*>(ones)[i] = i < 128 ? make_uint4(one2, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ------------------------------------------------------------------------------------------------ main kernel
__global__ void __launch_bounds__(kThreads, 1)
conv1x1_tc_kernel(const __grid_constant__ CUtensorMap tmap, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full[kMaxStages], bar_empty[kMaxStages], bar_w, bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_s;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wbytes = p.cin_blocks * kWBlockBytes + kBiasBlockBytes;
  uint8_t* wsm = smem;                                    // this CTA's weight slice (+ bias block), resident
  uint8_t* ones = smem + ((wbytes + 1023) & ~1023);       // constant A operand of the bias MMA
  uint8_t* slab0 = ones + kOnesBytes;

  const int slice = blockIdx.x % p.cout_slices;
  const int cta_in_slice = blockIdx.x / p.cout_slices, ctas_per_slice = gridDim.x / p.cout_slices;
  const int tiles_per_img = p.tiles_x * p.tiles_y;
  const int n_tiles = p.n_img * tiles_per_img;

  if (threadIdx.x == 0) {
    for (int i = 0; i < p.stages; ++i) { mbar_init(&bar_full[i], 1); mbar_init(&bar_empty[i], 1); }
    mbar_init(&bar_w, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_tfull[i], 1); mbar_init(&bar_tempty[i], 128); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  fill_ones_operand(ones, p.is_bf16, threadIdx.x, kThreads);
  if (warp == 1) {  // TMEM: 2 accumulators x 64 fp32 columns
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(128));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;

  if (warp == 0) {
    // ===================== TMA producer (warp-uniform loop, one elected lane issues) =====================
    if (elect_one()) {
      mbar_expect_tx(&bar_w, (uint32_t)wbytes);
      const uint8_t* wsrc = (const uint8_t*)p.wimg + (size_t)slice * wbytes;
      for (int o = 0; o + kWBlockBytes <= wbytes; o += kWBlockBytes) bulk_load(wsm + o, wsrc + o, kWBlockBytes, &bar_w);
      bulk_load(wsm + wbytes - kBiasBlockBytes, wsrc + wbytes - kBiasBlockBytes, kBiasBlockBytes, &bar_w);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice) {
      const int n = t / tiles_per_img, r = t - n * tiles_per_img;
      const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
      for (int cb = 0; cb < p.cin_blocks; ++cb) {
        mbar_wait(&bar_empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bar_full[stage], (uint32_t)kSlabBytes);
          tma_load_4d(slab0 + (size_t)stage * kSlabBytes, &tmap, &bar_full[stage], tx * kTW * 8, ty * kTH, cb * 8, n);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (warp-uniform loop; descriptors differ only in their low word) =====================
    // instruction descriptor: D=f32, A=B=f16|bf16, both K-major, N=64, M=128
    const uint32_t fmt = p.is_bf16 ? 1u : 0u;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((64u >> 3) << 17) | ((128u >> 4) << 24);
    // operand A (slab): LBO = stride between 8-channel groups, SBO = stride between 8-pixel rows of the tile;
    // operand B (weights): LBO = 1024 B between the two K chunks, SBO = 128 B between groups of 8 output channels
    const uint32_t a_lbo = kChStride, a_sbo = (uint32_t)kTW * 16;
    const uint32_t b_lbo = 1024u, b_sbo = 128u;
    const uint32_t a_hi = (a_sbo >> 4) | (1u << 14), b_hi = (b_sbo >> 4) | (1u << 14);  // SBO | descriptor version 1
    const uint32_t a_lo_c = (a_lbo >> 4) << 16, b_lo_c = (b_lbo >> 4) << 16;
    mbar_wait(&bar_w, 0);
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0;
    const uint32_t w_addr = smem_u32(wsm), slab_addr = smem_u32(slab0);
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice) {
      mbar_wait(&bar_tempty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * 64;
      for (int cb = 0; cb < p.cin_blocks; ++cb) {
        mbar_wait(&bar_full[stage], phase);
        tc_fence_after();
        const uint32_t a_lo = ((slab_addr + (uint32_t)stage * kSlabBytes) >> 4) | a_lo_c;
        const uint32_t b_lo = ((w_addr + (uint32_t)cb * kWBlockBytes) >> 4) | b_lo_c;
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const uint32_t aoff = ((uint32_t)kk * 2 * kChStride) >> 4;
            const uint32_t boff = ((uint32_t)kk * 2048) >> 4;
            umma_f16_2w(d_tmem, a_lo + aoff, a_hi, b_lo + boff, b_hi, idesc, (cb | kk) ? 1u : 0u);
          }
          umma_commit(&bar_empty[stage]);  // frees the slab once these MMAs have read it
          if (cb == p.cin_blocks - 1) {
            // + bias: D += ones[128 x 16] . biasB[64 x 16]  (k 0/1 = hi/lo halves of the folded bias)
            const uint32_t o_lo = (smem_u32(ones) >> 4) | ((2048u >> 4) << 16);
            const uint32_t bb_lo = ((w_addr + (uint32_t)p.cin_blocks * kWBlockBytes) >> 4) | b_lo_c;
            umma_f16_2w(d_tmem, o_lo, (128u >> 4) | (1u << 14), bb_lo, b_hi, idesc, 1u);
            umma_commit(&bar_tfull[acc]);  // accumulator complete -> epilogue
          }
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    // ===================== epilogue (4 warps; warp%4 selects the TMEM lane quarter) =====================
    const int q = warp & 3;
    const int g = q * 4 + (lane >> 3), r = lane & 7;   // pixel (row g, col r) of the 16 x 8 tile
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice) {
      const int n = t / tiles_per_img, rr = t - n * tiles_per_img;
      const int ty = rr / p.tiles_x, tx = rr - ty * p.tiles_x;
      const int y = ty * kTH + g, x = tx * kTW + r;
      mbar_wait(&bar_tfull[acc], acc_phase);
      tc_fence_after();
      uint32_t v[64];
      const uint32_t taddr = tmem_base + (uint32_t)acc * 64 + ((uint32_t)(q * 32) << 16);
      tmem_ld32(taddr, v);
      tmem_ld32(taddr + 32, v + 32);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&bar_tempty[acc]);  // TMEM accumulator is free again
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }

      if (y < p.H && x < p.W) {
#pragma unroll
        for (int c = 0; c < 64; ++c) {
          const int co = slice * 64 + c;
          if (co < p.cout) {
            float a = __uint_as_float(v[c]);  // bias is already in D
            if (p.relu) a = fmaxf(a, 0.f);
            p.out[(((size_t)n * p.cout + co) * p.H + y) * p.W + x] = a;
          }
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

// ------------------------------------------------------------------------------------------------ CUDA-core helpers
// block_1 (Cin = 1): fp32 image -> C8 16-bit activations, 64 channels.  K = 9 is too small for a tensor-core tile;
// the kernel is bound by the 128 B/pixel it writes.  One warp = one 8-channel group (its 72 folded weights live in
// registers), lane = pixel, kPx pixels per thread at stride 32 so that every store instruction writes 512 contiguous
// bytes; the 3x3 input window comes from a shared-memory row tile.
constexpr int kC1Px = 5;   // 160 pixels per block row: 320 = 2 blocks, 160 = 1 block
constexpr int kC1Rows = 8; // image rows per block (amortises the weight fetch)
__global__ void __launch_bounds__(256)
conv1_c8_kernel(const float* __restrict__ img, const float* __restrict__ w /*[9][64]*/, const float* __restrict__ bias,
                void* __restrict__ out, int B, int H, int W, int is_bf16) {
  constexpr int TWp = 32 * kC1Px;
  __shared__ float rows[kC1Rows + 2][TWp + 2];
  __shared__ __align__(16) float ws[9 * 64 + 64];
  const int lane = threadIdx.x & 31, cg = threadIdx.x >> 5;  // channel group 0..7
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
  for (int t = 0; t < 9; ++t) {
    const float4 a = *reinterpret_cast<const float4*>(&ws[t * 64 + cg * 8]);
    const float4 b = *reinterpret_cast<const float4*>(&ws[t * 64 + cg * 8 + 4]);
    wr[t][0] = a.x; wr[t][1] = a.y; wr[t][2] = a.z; wr[t][3] = a.w;
    wr[t][4] = b.x; wr[t][5] = b.y; wr[t][6] = b.z; wr[t][7] = b.w;
  }
#pragma unroll
  for (int c = 0; c < 8; ++c) bb[c] = ws[576 + cg * 8 + c];
  for (int ry = 0; ry < kC1Rows; ++ry) {
    const int y = y0 + ry;
    if (y >= H) break;
    uint4* o = reinterpret_cast<uint4*>(out) + (((size_t)n * 8 + cg) * H + y) * W;
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
      uint4 q;
      q.x = pack2(fmaxf(acc[0], 0.f), fmaxf(acc[1], 0.f), is_bf16);
      q.y = pack2(fmaxf(acc[2], 0.f), fmaxf(acc[3], 0.f), is_bf16);
      q.z = pack2(fmaxf(acc[4], 0.f), fmaxf(acc[5], 0.f), is_bf16);
      q.w = pack2(fmaxf(acc[6], 0.f), fmaxf(acc[7], 0.f), is_bf16);
      o[x] = q;
    }
  }
}

// layout conversions for the single-layer entry point (spn_conv_layer): NCHW fp32 <-> C8 16-bit
__global__ void nchw_to_c8_kernel(const float* __restrict__ in, void* __restrict__ out, int B, int C, int H, int W, int is_bf16) {
  const size_t total = (size_t)B * (C / 8) * H * W;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int x = i % W;
  const int y = (i / W) % H;
  const int cgp = (i / ((size_t)W * H)) % (C / 8);
  const int n = i / ((size_t)W * H * (C / 8));
  float v[8];
  for (int e = 0; e < 8; ++e) v[e] = in[(((size_t)n * C + cgp * 8 + e) * H + y) * W + x];
  uint4 o;
  o.x = pack2(v[0], v[1], is_bf16); o.y = pack2(v[2], v[3], is_bf16);
  o.z = pack2(v[4], v[5], is_bf16); o.w = pack2(v[6], v[7], is_bf16);
  reinterpret_cast<uint4*>(out)[i] = o;
}
__global__ void c8_to_nchw_kernel(const void* __restrict__ in, float* __restrict__ out, int B, int C, int H, int W, int is_bf16) {
  const size_t total = (size_t)B * (C / 8) * H * W;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int x = i % W;
  const int y = (i / W) % H;
  const int cgp = (i / ((size_t)W * H)) % (C / 8);
  const int n = i / ((size_t)W * H * (C / 8));
  const uint4 q = reinterpret_cast<const uint4*>(in)[i];
  const uint32_t w4[4] = {q.x, q.y, q.z, q.w};
  for (int e = 0; e < 4; ++e) {
    float a, b;
    if (is_bf16) {
      const __nv_bfloat162 t = *reinterpret_cast<const __nv_bfloat162*>(&w4[e]);
      a = __bfloat162float(t.x); b = __bfloat162float(t.y);
    } else {
      const __half2 t = *reinterpret_cast<const __half2*>(&w4[e]);
      a = __half2float(t.x); b = __half2float(t.y);
    }
    out[(((size_t)n * C + cgp * 8 + 2 * e) * H + y) * W + x] = a;
    out[(((size_t)n * C + cgp * 8 + 2 * e + 1) * H + y) * W + x] = b;
  }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

struct TcState {
  EncodeTiledFn encode = nullptr;
  float* w1 = nullptr;      // block_1 weights [9][64] fp32 (BN folded)
  void* w1img[2] = {nullptr, nullptr};  // block_1 as tcgen05 operand B: [chunk 2][cout 64][8] (K = 9 taps padded to 16)
};

TcState* tc_state(spn_ctx* ctx) {
  if (!ctx->tc) ctx->tc = new TcState();
  return (TcState*)ctx->tc;
}

int get_encode(TcState* st) {
  if (st->encode) return SPN_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  SPN_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) {
    spn_set_error("cuTensorMapEncodeTiled not available from the driver");
    return SPN_E_CUDA;
  }
  st->encode = (EncodeTiledFn)fn;
  return SPN_OK;
}

// One 1x1 tensor-core conv layer: in (C8, [n][cin/8][H][W][8]) -> out (NCHW fp32 [n][cout][H][W]).
int launch_conv1x1_tc(spn_ctx* ctx, int layer, int mode, const void* in, float* out, int n_img, int H, int W, bool relu,
                      cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  const int bf = mode == SPN_MODE_BF16 ? 1 : 0;
  if (!L.w16[bf]) { spn_set_error("layer %d has no tensor-core weights", layer); return SPN_E_STATE; }
  SPN_REQUIRE(L.cin % 64 == 0, "tensor-core conv needs Cin %% 64 == 0 (layer %d has %d)", layer, L.cin);

  TcParams p;
  memset(&p, 0, sizeof(p));
  p.n_img = n_img; p.H = H; p.W = W;
  p.cin_blocks = L.cin / 64;
  p.cout_slices = (L.cout + 63) / 64;
  p.cout = L.cout;
  p.relu = relu; p.is_bf16 = bf;
  p.tiles_x = spn_cdiv(W, kTW); p.tiles_y = spn_cdiv(H, kTH);
  const int wbytes = p.cin_blocks * kWBlockBytes + kBiasBlockBytes;
  const int wres = ((wbytes + 1023) & ~1023) + kOnesBytes;
  const int max_dyn = 227 * 1024 - 2048;  // leave room for the static barriers / bias
  p.stages = (max_dyn - wres - 1024) / kSlabBytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  SPN_REQUIRE(p.stages >= 2, "layer %d does not fit in shared memory (weights %d bytes)", layer, wbytes);
  p.out = out; p.wimg = L.w16[bf];
  const size_t dyn = (size_t)wres + (size_t)p.stages * kSlabBytes + 1024;

  CUtensorMap tmap;
  int rc = spn_c8_tensor_map(ctx, &tmap, in, n_img, L.cin, H, W, kTW, kTH, bf);
  if (rc) return rc;
  SPN_CUDA(cudaFuncSetAttribute(conv1x1_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  const long long work = (long long)n_img * p.tiles_x * p.tiles_y * p.cout_slices;
  int grid = ctx->sm_count;
  if (work < grid) grid = (int)work;
  grid = grid / p.cout_slices * p.cout_slices;
  if (grid < p.cout_slices) grid = p.cout_slices;
  SpnProfScope prof(ctx, layer, s);
  conv1x1_tc_kernel<<<grid, kThreads, dyn, s>>>(tmap, p);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

struct TcPlan {
  size_t a, b, feat, head, total;  // region sizes in bytes (each followed by a kSpnGap guard gap)
  size_t off_b, off_feat, off_head, off_logits;
};
TcPlan tc_plan(int B, int H, int W) {
  TcPlan p;
  const size_t hw = (size_t)H * W;
  p.a = (size_t)B * 64 * hw * 2;           // block_1 out (largest)
  p.b = (size_t)B * 64 * hw / 4 * 2;       // pooled block_2 out
  p.feat = (size_t)B * 128 * hw / 64 * 2;
  p.head = (size_t)B * 256 * hw / 64 * 2;  // convPa / convDa out
  const size_t logits = (size_t)B * 65 * hw / 64 * 4;
  p.off_b = p.a + kSpnGap;
  p.off_feat = p.off_b + p.b + kSpnGap;
  p.off_head = p.off_feat + p.feat + kSpnGap;
  p.off_logits = p.off_head + p.head + kSpnGap;
  p.total = p.off_logits + logits + 4096;
  return p;
}

// option "ws_guard": paint the four gaps before a pass and remember them for spn_check_guards
int paint_gaps(spn_ctx* ctx, const TcPlan& pl, cudaStream_t s) {
  if (!ctx->opt_ws_guard) return SPN_OK;
  ctx->guard_gaps.clear();
  for (size_t off : {pl.off_b, pl.off_feat, pl.off_head, pl.off_logits}) {
    char* g = ctx->ws + off - kSpnGap;
    SPN_CUDA(cudaMemsetAsync(g, kSpnGuardByte, kSpnGap, s));
    ctx->guard_gaps.push_back({g, kSpnGap});
  }
  return SPN_OK;
}

}  // namespace

const float* spn_tc_block1_weights(spn_ctx* ctx) { return tc_state(ctx)->w1; }

int spn_tc_pack_layer(spn_ctx* ctx, int layer, const float* h_wfold, const float* h_bfold, cudaStream_t s) {
  TcState* st = tc_state(ctx);
  SpnLayer& L = ctx->layers[layer];
  SPN_CUDA(cudaStreamSynchronize(s));
  if (layer == SPN_L_BLOCK1) {
    SPN_REQUIRE(L.cin == 1 && L.cout == 64 && L.ks == 3, "block_1 must be a 3x3 conv 1->64");
    std::vector<float> w(9 * 64);
    for (int co = 0; co < 64; ++co)
      for (int t = 0; t < 9; ++t) w[t * 64 + co] = h_wfold[(size_t)co * 9 + t];
    if (!st->w1) SPN_CUDA(cudaMalloc((void**)&st->w1, w.size() * sizeof(float)));
    SPN_CUDA(cudaMemcpy(st->w1, w.data(), w.size() * sizeof(float), cudaMemcpyHostToDevice));
    for (int bf = 0; bf < 2; ++bf) {
      // K = 16: k 0..8 = the nine taps, k 9 / 10 = the bias as a (hi, lo) pair of 16-bit values multiplied by the
      // constant-one columns the front end puts into A1 (so block_1's epilogue needs no bias add)
      std::vector<uint16_t> img(2 * 64 * 8, 0);
      for (int co = 0; co < 64; ++co) {
        for (int t = 0; t < 9; ++t) img[((size_t)(t / 8) * 64 + co) * 8 + (t % 8)] = to16(h_wfold[(size_t)co * 9 + t], bf);
        const uint16_t hi = to16(h_bfold[co], bf);
        img[((size_t)1 * 64 + co) * 8 + 1] = hi;
        img[((size_t)1 * 64 + co) * 8 + 2] = to16(h_bfold[co] - from16(hi, bf), bf);
      }
      if (!st->w1img[bf]) SPN_CUDA(cudaMalloc(&st->w1img[bf], img.size() * 2));
      SPN_CUDA(cudaMemcpy(st->w1img[bf], img.data(), img.size() * 2, cudaMemcpyHostToDevice));
    }
    return SPN_OK;
  }
  if (L.cin % 64 != 0) return SPN_OK;  // not a tensor-core layer
  if (L.ks == 1 || layer == SPN_L_BLOCK2) {  // the 1x1 kernel's weights, and block_2's that front_tc_kernel reads
    const int taps = L.ks * L.ks, slices = (L.cout + 63) / 64, cbs = L.cin / 64;
    // operand-B image: [slice][cin block][tap][k-step 4][chunk 2][cout 64][8 cin]  (SWIZZLE_NONE K-major core matrices)
    // followed, per slice, by the bias block [chunk 2][cout 64][8]: k 0 = hi, k 1 = lo 16-bit halves of the folded bias
    const size_t n16 = (size_t)slices * ((size_t)cbs * taps * 4 * 2 * 64 * 8 + 2 * 64 * 8);
    for (int bf = 0; bf < 2; ++bf) {
      std::vector<uint16_t> img(n16, 0);
      size_t o = 0;
      for (int sl = 0; sl < slices; ++sl) {
        for (int cb = 0; cb < cbs; ++cb)
          for (int t = 0; t < taps; ++t)
            for (int kk = 0; kk < 4; ++kk)
              for (int j = 0; j < 2; ++j)
                for (int co = 0; co < 64; ++co)
                  for (int e = 0; e < 8; ++e, ++o) {
                    const int c = sl * 64 + co, ci = cb * 64 + kk * 16 + j * 8 + e;
                    if (c < L.cout) img[o] = to16(h_wfold[((size_t)c * L.cin + ci) * taps + t], bf);
                  }
        for (int co = 0; co < 64; ++co) {
          const int c = sl * 64 + co;
          if (c < L.cout) {
            const uint16_t hi = to16(h_bfold[c], bf);
            img[o + (size_t)co * 8] = hi;
            img[o + (size_t)co * 8 + 1] = to16(h_bfold[c] - from16(hi, bf), bf);
          }
        }
        o += 2 * 64 * 8;
      }
      if (L.w16[bf]) { cudaFree(L.w16[bf]); L.w16[bf] = nullptr; }
      SPN_CUDA(cudaMalloc(&L.w16[bf], n16 * 2));
      SPN_CUDA(cudaMemcpy(L.w16[bf], img.data(), n16 * 2, cudaMemcpyHostToDevice));
    }
  }
  int rc = spn_fold_pack_layer(ctx, layer, h_wfold, h_bfold);
  if (rc) return rc;
  return spn_head_pack_layer(ctx, layer, h_wfold, h_bfold);
}

int spn_c8_tensor_map(spn_ctx* ctx, CUtensorMap* map, const void* base, int n_img, int C, int H, int W, int box_w, int box_h,
                      int bf16) {
  TcState* st = tc_state(ctx);
  int rc = get_encode(st);
  if (rc) return rc;
  const cuuint64_t dims[4] = {(cuuint64_t)W * 8, (cuuint64_t)H, (cuuint64_t)(C / 8), (cuuint64_t)n_img};
  const cuuint64_t strides[3] = {(cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)(C / 8) * H * W * 16};
  const cuuint32_t box[4] = {(cuuint32_t)box_w * 8, (cuuint32_t)box_h, 8, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult cr = st->encode(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<void*>(base),
                           dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                           CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) {
    spn_set_error("cuTensorMapEncodeTiled failed (%d) for a C8 tensor of %d x %d x %d x %d", (int)cr, n_img, C, H, W);
    return SPN_E_CUDA;
  }
  return SPN_OK;
}

// Encoder over `n_slots` forwards.  d_hinv == nullptr: slot i is image i (plain forward).  Otherwise slot =
// src*(n_h+1)+j is image `src` warped by homography j-1 (j == 0: the image itself) and the warp is fused in.
int spn_tc_encoder_slots(spn_ctx* ctx, const float* d_images, const float* d_hinv, int n_h, int slot_begin, int n_slots,
                         int H, int W, int mode, cudaStream_t s) {
  TcState* st = tc_state(ctx);
  if (!st->w1) { spn_set_error("block_1 has no weights"); return SPN_E_STATE; }
  const int B = n_slots;
  const TcPlan pl = tc_plan(B, H, W);
  int rc = spn_ensure_ws(ctx, pl.total, s);
  if (rc) return rc;
  if ((rc = paint_gaps(ctx, pl, s))) return rc;
  char* A = ctx->ws;
  char* Bq = A + pl.off_b;
  char* F = A + pl.off_feat;
  const int bf = mode == SPN_MODE_BF16 ? 1 : 0;
  if (!ctx->opt_fuse_front) {
    SPN_REQUIRE(!d_hinv, "option fuse_front = 0: the unfused path takes already-warped images");
    {
      SpnProfScope prof(ctx, SPN_L_BLOCK1, s);
      dim3 g(spn_cdiv(W, 32 * kC1Px), spn_cdiv(H, kC1Rows), B);
      conv1_c8_kernel<<<g, 256, 0, s>>>(d_images + (size_t)slot_begin * H * W, st->w1, ctx->layers[0].bias, A, B, H, W, bf);
      SPN_CHECK_LAUNCH(ctx);
    }
    if ((rc = spn_launch_conv_fold(ctx, 1, mode, A, Bq, B, H, W, true, true, s))) return rc;
  } else {
    // warp + block_1 + block_2 in one kernel (front_tc.cu): block_1's output never reaches HBM
    rc = spn_front_tc_launch(ctx, d_images, d_hinv, n_h, slot_begin, n_slots, H, W, mode, st->w1img[bf], Bq, s);
    if (rc) return rc;
  }
  if ((rc = spn_launch_conv_fold(ctx, 2, mode, Bq, A, B, H / 2, W / 2, true, false, s))) return rc;
  if ((rc = spn_launch_conv_fold(ctx, 3, mode, A, Bq, B, H / 2, W / 2, true, true, s))) return rc;
  if ((rc = spn_launch_conv_fold(ctx, 4, mode, Bq, A, B, H / 4, W / 4, true, false, s))) return rc;
  if ((rc = spn_launch_conv_fold(ctx, 5, mode, A, Bq, B, H / 4, W / 4, true, true, s))) return rc;
  if ((rc = spn_launch_conv_fold(ctx, 6, mode, Bq, A, B, H / 8, W / 8, true, false, s))) return rc;
  if ((rc = spn_launch_conv_fold(ctx, 7, mode, A, F, B, H / 8, W / 8, true, false, s))) return rc;
  ctx->feat = F;
  return SPN_OK;
}

int spn_tc_encoder(spn_ctx* ctx, const float* d_images, int B, int H, int W, int mode, cudaStream_t s) {
  return spn_tc_encoder_slots(ctx, d_images, nullptr, 0, 0, B, H, W, mode, s);
}

int spn_tc_detector_head(spn_ctx* ctx, int B, int H, int W, int mode, float* d_logits, cudaStream_t s) {
  const TcPlan pl = tc_plan(B, H, W);
  char* head = ctx->ws + pl.off_head;
  int rc;
  if ((rc = spn_launch_conv_fold(ctx, SPN_L_CONVPA, mode, ctx->feat, head, B, H / 8, W / 8, true, false, s))) return rc;
  return launch_conv1x1_tc(ctx, SPN_L_CONVPB, mode, head, d_logits, B, H / 8, W / 8, false, s);
}

// convPa, then convPb + softmax + depth-to-space + mask in one kernel (head_tc.cu)
int spn_tc_detector_head_fused(spn_ctx* ctx, int B, int H, int W, int mode, const uint8_t* d_mask, float* d_logits, float* d_prob,
                               cudaStream_t s) {
  const TcPlan pl = tc_plan(B, H, W);
  char* head = ctx->ws + pl.off_head;
  int rc;
  if ((rc = spn_launch_conv_fold(ctx, SPN_L_CONVPA, mode, ctx->feat, head, B, H / 8, W / 8, true, false, s))) return rc;
  return spn_launch_head_tc(ctx, mode, head, B, H / 8, W / 8, d_mask, d_logits, d_prob, s);
}

int spn_tc_descriptor_head(spn_ctx* ctx, int B, int H, int W, int mode, float* d_desc_raw, cudaStream_t s) {
  const TcPlan pl = tc_plan(B, H, W);
  char* head = ctx->ws + pl.off_head;
  int rc;
  if ((rc = spn_launch_conv_fold(ctx, SPN_L_CONVDA, mode, ctx->feat, head, B, H / 8, W / 8, true, false, s))) return rc;
  return launch_conv1x1_tc(ctx, SPN_L_CONVDB, mode, head, d_desc_raw, B, H / 8, W / 8, false, s);
}

float* spn_tc_logits_scratch(spn_ctx* ctx, int B, int H, int W) {
  const TcPlan pl = tc_plan(B, H, W);
  return (float*)(ctx->ws + pl.off_logits);
}

// single VGG_Block through the tensor-core path with NCHW fp32 in/out (layout conversion on both sides)
int spn_tc_conv_layer(spn_ctx* ctx, int layer, int mode, const float* d_in, int B, int H, int W, bool relu, bool pool,
                      float* d_out, cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  const int bf = mode == SPN_MODE_BF16 ? 1 : 0;
  const int Ho = pool ? H / 2 : H, Wo = pool ? W / 2 : W;
  const int cout_pad = (L.cout + 63) / 64 * 64;
  const size_t in_b = (size_t)B * L.cin * H * W * 2, out_b = (size_t)B * cout_pad * Ho * Wo * 2;
  int rc = spn_ensure_ws(ctx, in_b + out_b + 2048, s);
  if (rc) return rc;
  char* cin8 = ctx->ws;
  char* cout8 = ctx->ws + ((in_b + 1023) & ~(size_t)1023);
  const size_t n_in = (size_t)B * (L.cin / 8) * H * W;
  nchw_to_c8_kernel<<<(unsigned)((n_in + 255) / 256), 256, 0, s>>>(d_in, cin8, B, L.cin, H, W, bf);
  SPN_CHECK_LAUNCH(ctx);
  if (L.ks == 1) return launch_conv1x1_tc(ctx, layer, mode, cin8, d_out, B, H, W, relu, s);
  if ((rc = spn_launch_conv_fold(ctx, layer, mode, cin8, cout8, B, H, W, relu, pool, s))) return rc;
  // C8 buffer has cout_slices*64 channels; only the first cout are meaningful
  SPN_REQUIRE(L.cout % 64 == 0, "spn_conv_layer (tensor-core, 3x3) needs Cout %% 64 == 0");
  const size_t n_out = (size_t)B * (L.cout / 8) * Ho * Wo;
  c8_to_nchw_kernel<<<(unsigned)((n_out + 255) / 256), 256, 0, s>>>(cout8, d_out, B, L.cout, Ho, Wo, bf);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

void spn_tc_destroy(spn_ctx* ctx) {
  TcState* st = (TcState*)ctx->tc;
  if (!st) return;
  if (st->w1) cudaFree(st->w1);
  for (auto& w : st->w1img) if (w) cudaFree(w);
  delete st;
  ctx->tc = nullptr;
}
