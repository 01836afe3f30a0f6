// 3x3 tcgen05 convolution with the horizontal filter taps folded into the MMA's N dimension.
//
// Why: an M128 x N64 x K16 MMA needs 6 KB of shared-memory operands per 32 tensor cycles and is capped by the
// 128 B/cycle shared-memory pipe at 2/3 of the tensor peak (tools/mma_rate.cu: 48.1 cycles per MMA measured for
// N = 64, 64.1 / 96.1 / 128.1 for N = 128 / 192 / 256, i.e. full rate from N = 128 up).  N is the layer's output
// channel slice (64), so instead of shifting the A operand for each of the nine taps this kernel computes, per
// vertical tap ky and 16-channel K step,
//      F[pixel p, (kx, co)] += in[p + ky row shift, ci] . W[ky, kx, ci, co]           (ONE MMA, N = 3 x 64 = 192)
// with the UNSHIFTED pixel p for all three kx, and applies the horizontal shift when the accumulator is read back:
//      out[y, x, co] = F[(y, x-1), (0, co)] + F[(y, x), (1, co)] + F[(y, x+1), (2, co)]   (two warp shuffles per value).
// 12 MMAs of N = 192 (+1 bias MMA) replace 36 MMAs of N = 64: same FLOPs, A is read from shared memory 3x less often
// and the tensor pipe is no longer starved.
//
// Tile: 8 rows x 16 pixels (M = 128, TMEM lane = 16*row + x); the two edge columns of a tile have no x-neighbour inside
// the tile, so 14 of the 16 columns are valid outputs and tiles advance by 14 pixels in x (origin x0 = 14*tx - 1, which
// keeps the valid range even-aligned for the fused 2x2 max-pool).  Slab = 10 rows x 16 pixels x 64 channels = 20 KB per
// TMA box, rows contiguous so that the 128 GEMM rows are one contiguous run (SBO = 128 B) and a vertical tap is a
// +256 B start-address offset.  Pooling partners (x+-1: lane+-1, y+-1: lane^16) stay inside one warp.
//
// Warp roles (320 threads, persistent, 1 CTA/SM): warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 / 6-9 two epilogue
// groups that alternate tiles (the epilogue does 3x the TMEM reads and 2 shuffles per output value, so one group alone
// would not keep up with a full-rate MMA stream).
#include <cuda.h>

#include <vector>

#include "spn_common.cuh"
#include "tc_ptx.cuh"

namespace {

using namespace tcptx;

constexpr int kTWs = 16, kTWv = 14, kTH = 8;         // slab width, valid output width, rows
constexpr int kPH = kTH + 2;                          // slab rows
constexpr uint32_t kChStride = (uint32_t)kPH * kTWs * 16;   // 2560 B between 8-channel groups
constexpr int kSlabBytes = 8 * kPH * kTWs * 16;       // 20480
constexpr int kBlkBytes = 2 * 192 * 16;               // operand-B block of one (cin block, ky, k-step): [chunk 2][n 192][8]
constexpr int kOnesBytes = 4096;
constexpr int kThreads = 320;
constexpr int kMaxStages = 6;

struct FoldParams {
  int n_img, H, W;
  int cin_blocks, cout_slices, cout;
  int relu, pool, is_bf16;
  int tiles_x, tiles_y, stages;
  void* out;           // C8 [n][cout_slices*8][Ho][Wo][8]
  const void* wimg;    // per slice: [cin block][ky 3][k-step 4][chunk 2][n = kx*64+co 192][8] + bias block [2][192][8]
};

__global__ void __launch_bounds__(kThreads, 1)
conv_fold_kernel(const __grid_constant__ CUtensorMap tmap, const FoldParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar_full[kMaxStages], bar_empty[kMaxStages], bar_w, bar_tfull[2], bar_tempty[2];
  __shared__ uint32_t tmem_base_s;

  griddep_launch_dependents();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wbytes = p.cin_blocks * 12 * kBlkBytes + kBlkBytes;
  uint8_t* wsm = smem;
  uint8_t* ones = smem + ((wbytes + 1023) & ~1023);
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
  {  // constant A operand of the bias MMA: row = (1, 1, 0, ...) in K chunk 0, zeros in chunk 1
    const uint32_t one2 = p.is_bf16 ? 0x3F803F80u : 0x3C003C00u;
    for (int i = threadIdx.x; i < kOnesBytes / 16; i += kThreads)
      reinterpret_cast<uint4*>(ones)[i] = i < 128 ? make_uint4(one2, 0u, 0u, 0u) : make_uint4(0u, 0u, 0u, 0u);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {  // TMEM: 2 accumulators x 192 fp32 columns
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
      for (int o = 0; o < wbytes; o += kBlkBytes) bulk_load(wsm + o, wsrc + o, kBlkBytes, &bar_w);
    }
    griddep_wait();  // the activations come from the previous kernel; every store of this CTA follows these loads
    int stage = 0;
    uint32_t phase = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice) {
      const int n = t / tiles_per_img, r = t - n * tiles_per_img;
      const int ty = r / p.tiles_x, tx = r - ty * p.tiles_x;
      for (int cb = 0; cb < p.cin_blocks; ++cb) {
        mbar_wait(&bar_empty[stage], phase ^ 1);
        if (elect_one()) {
          mbar_expect_tx(&bar_full[stage], (uint32_t)kSlabBytes);
          tma_load_4d(slab0 + (size_t)stage * kSlabBytes, &tmap, &bar_full[stage], (tx * kTWv - 1) * 8, ty * kTH - 1, cb * 8, n);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // The tensor pipe's instruction queue is only a few MMAs deep, so whatever the issuing warp does between two
    // MMAs beyond that depth leaves the pipe idle.  The waits for the NEXT unit (a unit = one 64-channel block of one
    // tile = 12 MMAs) are therefore taken in the middle of the current unit's MMAs, and the commits at its end:
    // two short bookkeeping stretches per unit, each covered by the MMAs already queued.
    const uint32_t fmt = p.is_bf16 ? 1u : 0u;
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((192u >> 3) << 17) | ((128u >> 4) << 24);  // N 192, M 128
    const uint32_t a_hi = (128u >> 4) | (1u << 14);                 // A: SBO = 128 B (8 consecutive pixels)
    const uint32_t a_lo_c = (kChStride >> 4) << 16;                 //    LBO = 8-channel group stride
    const uint32_t b_hi = (128u >> 4) | (1u << 14);                 // B: SBO = 128 B (8 consecutive n)
    const uint32_t b_lo_c = ((192u * 16u) >> 4) << 16;              //    LBO = 3072 B between the two K chunks
    const uint32_t o_lo = (smem_u32(ones) >> 4) | ((2048u >> 4) << 16);
    mbar_wait(&bar_w, 0);
    const uint32_t w_addr = smem_u32(wsm), slab_addr = smem_u32(slab0);
    const int my_tiles = cta_in_slice < n_tiles ? (n_tiles - cta_in_slice + ctas_per_slice - 1) / ctas_per_slice : 0;
    const int n_units = my_tiles * p.cin_blocks;
    int stage = 0, i = 0, cb = 0;
    uint32_t phase = 0;
    if (n_units > 0) {
      mbar_wait(&bar_tempty[0], 1u);
      mbar_wait(&bar_full[0], 0u);
      tc_fence_after();
    }
    for (int u = 0; u < n_units; ++u) {
      const int acc = i & 1;
      const bool last_cb = cb == p.cin_blocks - 1;
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * 192;
      const uint32_t a_lo = ((slab_addr + (uint32_t)stage * kSlabBytes) >> 4) | a_lo_c;
      const uint32_t b_lo = ((w_addr + (uint32_t)cb * (12 * kBlkBytes)) >> 4) | b_lo_c;
      if (elect_one()) {
#pragma unroll
        for (int m = 0; m < 8; ++m) {
          const int ky = m >> 2, kk = m & 3;
          const uint32_t aoff = ((uint32_t)ky * (kTWs * 16) + (uint32_t)kk * 2 * kChStride) >> 4;
          const uint32_t boff = ((uint32_t)(ky * 4 + kk) * kBlkBytes) >> 4;
          umma_f16_2w(d_tmem, a_lo + aoff, a_hi, b_lo + boff, b_hi, idesc, (cb | m) ? 1u : 0u);
        }
      }
      __syncwarp();
      int nstage = stage + 1;
      uint32_t nphase = phase;
      if (nstage == p.stages) { nstage = 0; nphase ^= 1u; }
      if (u + 1 < n_units) {  // the next unit's operands and accumulator, while 8 MMAs are in the queue
        // With 128 input channels a tile is 25 MMAs and the kernel is tensor-bound: take the accumulator wait here too.
        // With 64 it is bound by the epilogues' TMEM reads (96 KB per tile against 13 MMAs): the accumulator of tile
        // i+1 is usually not free yet, so tile i is issued completely first (its epilogue can then start at once).
        if (last_cb && p.cin_blocks > 1) mbar_wait(&bar_tempty[(i + 1) & 1], ((uint32_t)((i + 1) >> 1) & 1u) ^ 1u);
        mbar_wait(&bar_full[nstage], nphase);
        tc_fence_after();
      }
      if (elect_one()) {
#pragma unroll
        for (int m = 8; m < 12; ++m) {
          const int ky = m >> 2, kk = m & 3;
          const uint32_t aoff = ((uint32_t)ky * (kTWs * 16) + (uint32_t)kk * 2 * kChStride) >> 4;
          const uint32_t boff = ((uint32_t)(ky * 4 + kk) * kBlkBytes) >> 4;
          umma_f16_2w(d_tmem, a_lo + aoff, a_hi, b_lo + boff, b_hi, idesc, 1u);
        }
        umma_commit(&bar_empty[stage]);
        if (last_cb) {
          const uint32_t bb_lo = ((w_addr + (uint32_t)p.cin_blocks * (12 * kBlkBytes)) >> 4) | b_lo_c;
          umma_f16_2w(d_tmem, o_lo, a_hi, bb_lo, b_hi, idesc, 1u);  // + bias (lives in the kx = 1 column block)
          umma_commit(&bar_tfull[acc]);
        }
      }
      __syncwarp();
      if (u + 1 < n_units && last_cb && p.cin_blocks == 1) {
        mbar_wait(&bar_tempty[(i + 1) & 1], ((uint32_t)((i + 1) >> 1) & 1u) ^ 1u);
        tc_fence_after();
      }
      stage = nstage;
      phase = nphase;
      if (last_cb) { cb = 0; ++i; } else { ++cb; }
    }
  } else {
    // ===================== epilogue: group 0 (warps 2-5) takes even tiles, group 1 (warps 6-9) odd tiles =====================
    const int group = (warp - 2) >> 2;
    const int q = warp & 3;                       // TMEM lane quarter of this warp
    const int r = 2 * q + (lane >> 4), x = lane & 15;   // tile row / column of this thread's pixel
    const int Ho = p.pool ? p.H >> 1 : p.H, Wo = p.pool ? p.W >> 1 : p.W;
    const int cgroups = p.cout_slices * 8;
    int i = 0;
    for (int t = cta_in_slice; t < n_tiles; t += ctas_per_slice, ++i) {
      if ((i & 1) != group) continue;
      const int acc = i & 1;                      // == group
      const uint32_t acc_phase = (uint32_t)(i >> 1) & 1u;
      const int n = t / tiles_per_img, rr = t - n * tiles_per_img;
      const int ty = rr / p.tiles_x, tx = rr - ty * p.tiles_x;
      const int y = ty * kTH + r, gx = tx * kTWv - 1 + x;
      mbar_wait(&bar_tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + (uint32_t)acc * 192 + ((uint32_t)(q * 32) << 16);
      uint32_t h2[32];
#pragma unroll
      for (int c0 = 0; c0 < 64; c0 += 32) {
        uint32_t f0[32], f1[32], f2[32];
        tmem_ld32(taddr + c0, f0);
        tmem_ld32(taddr + 64 + c0, f1);
        tmem_ld32(taddr + 128 + c0, f2);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < 32; c += 2) {
          // out(x) = F(x-1, kx=0) + F(x, kx=1) + F(x+1, kx=2): neighbours are lane-1 / lane+1 (same tile row for x in 1..14)
          float a = __shfl_up_sync(0xffffffffu, __uint_as_float(f0[c]), 1) + __uint_as_float(f1[c]);
          float b = __shfl_up_sync(0xffffffffu, __uint_as_float(f0[c + 1]), 1) + __uint_as_float(f1[c + 1]);
          a += __shfl_down_sync(0xffffffffu, __uint_as_float(f2[c]), 1);
          b += __shfl_down_sync(0xffffffffu, __uint_as_float(f2[c + 1]), 1);
          h2[(c0 + c) >> 1] = p.relu ? pack2_relu(a, b, p.is_bf16) : pack2(a, b, p.is_bf16);   // ReLU commutes with the pool below
        }
      }
      tc_fence_before();
      mbar_arrive(&bar_tempty[acc]);
      bool writer = x >= 1 && x <= kTWv && gx < p.W && y < p.H;
      int oy = y, ox = gx;
      if (p.pool) {
#pragma unroll
        for (int c = 0; c < 32; ++c) {
          h2[c] = max2(h2[c], __shfl_down_sync(0xffffffffu, h2[c], 1), p.is_bf16);   // (x, x+1), x odd = gx even
          h2[c] = max2(h2[c], __shfl_xor_sync(0xffffffffu, h2[c], 16), p.is_bf16);   // rows 2q, 2q+1
        }
        writer = writer && (x & 1) && ((lane >> 4) == 0);
        oy = y >> 1; ox = gx >> 1;
      }
      if (writer) {
        uint4* o = reinterpret_cast<uint4*>(p.out);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (slice * 64 + j * 8 < p.cout)
            o[(((size_t)n * cgroups + slice * 8 + j) * Ho + oy) * Wo + ox] = make_uint4(h2[4 * j], h2[4 * j + 1], h2[4 * j + 2], h2[4 * j + 3]);
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

// operand-B image of a 3x3 layer for conv_fold_kernel (both 16-bit types)
int spn_fold_pack_layer(spn_ctx* ctx, int layer, const float* h_wfold, const float* h_bfold) {
  SpnLayer& L = ctx->layers[layer];
  if (L.ks != 3 || L.cin % 64 != 0) return SPN_OK;
  const int slices = (L.cout + 63) / 64, cbs = L.cin / 64;
  const size_t per_slice = ((size_t)cbs * 12 + 1) * (kBlkBytes / 2);
  for (int bf = 0; bf < 2; ++bf) {
    std::vector<uint16_t> img(per_slice * slices, 0);
    for (int sl = 0; sl < slices; ++sl) {
      uint16_t* base = img.data() + per_slice * sl;
      for (int cb = 0; cb < cbs; ++cb)
        for (int ky = 0; ky < 3; ++ky)
          for (int kk = 0; kk < 4; ++kk) {
            uint16_t* blk = base + ((size_t)(cb * 3 + ky) * 4 + kk) * (kBlkBytes / 2);
            for (int j = 0; j < 2; ++j)
              for (int kx = 0; kx < 3; ++kx)
                for (int co = 0; co < 64; ++co)
                  for (int e = 0; e < 8; ++e) {
                    const int c = sl * 64 + co, ci = cb * 64 + kk * 16 + j * 8 + e;
                    if (c < L.cout)
                      blk[((size_t)j * 192 + kx * 64 + co) * 8 + e] = to16(h_wfold[((size_t)c * L.cin + ci) * 9 + ky * 3 + kx], bf);
                  }
          }
      uint16_t* bb = base + (size_t)cbs * 12 * (kBlkBytes / 2);  // bias block: n = 64 + co (kx = 1), k 0 / 1 = hi / lo
      for (int co = 0; co < 64; ++co) {
        const int c = sl * 64 + co;
        if (c < L.cout) {
          const uint16_t hi = to16(h_bfold[c], bf);
          bb[((size_t)64 + co) * 8] = hi;
          bb[((size_t)64 + co) * 8 + 1] = to16(h_bfold[c] - from16(hi, bf), bf);
        }
      }
    }
    if (L.w16f[bf]) { cudaFree(L.w16f[bf]); L.w16f[bf] = nullptr; }
    SPN_CUDA(cudaMalloc(&L.w16f[bf], img.size() * 2));
    SPN_CUDA(cudaMemcpy(L.w16f[bf], img.data(), img.size() * 2, cudaMemcpyHostToDevice));
  }
  return SPN_OK;
}

int spn_launch_conv_fold(spn_ctx* ctx, int layer, int mode, const void* in, void* out, int n_img, int H, int W, bool relu,
                         bool pool, cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  const int bf = mode == SPN_MODE_BF16 ? 1 : 0;
  if (!L.w16f[bf]) { spn_set_error("layer %d has no folded tensor-core weights", layer); return SPN_E_STATE; }
  FoldParams p;
  memset(&p, 0, sizeof(p));
  p.n_img = n_img; p.H = H; p.W = W;
  p.cin_blocks = L.cin / 64; p.cout_slices = (L.cout + 63) / 64; p.cout = L.cout;
  p.relu = relu; p.pool = pool; p.is_bf16 = bf;
  p.tiles_x = spn_cdiv(W, kTWv); p.tiles_y = spn_cdiv(H, kTH);
  const int wbytes = p.cin_blocks * 12 * kBlkBytes + kBlkBytes;
  const int wres = ((wbytes + 1023) & ~1023) + kOnesBytes;
  const int max_dyn = 227 * 1024 - 2048;
  p.stages = (max_dyn - wres - 1024) / kSlabBytes;
  if (p.stages > kMaxStages) p.stages = kMaxStages;
  SPN_REQUIRE(p.stages >= 2, "layer %d does not fit in shared memory", layer);
  p.out = out; p.wimg = L.w16f[bf];
  const size_t dyn = (size_t)wres + (size_t)p.stages * kSlabBytes + 1024;

  CUtensorMap tmap;
  int rc = spn_c8_tensor_map(ctx, &tmap, in, n_img, L.cin, H, W, kTWs, kPH, bf);
  if (rc) return rc;
  SPN_CUDA(cudaFuncSetAttribute(conv_fold_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  const long long work = (long long)n_img * p.tiles_x * p.tiles_y * p.cout_slices;
  int grid = ctx->sm_count;
  if (work < grid) grid = (int)work;
  grid = grid / p.cout_slices * p.cout_slices;
  if (grid < p.cout_slices) grid = p.cout_slices;
  SpnProfScope prof(ctx, layer, s);
  SPN_CUDA(spn_launch_pdl(conv_fold_kernel, dim3(grid), dim3(kThreads), dyn, s, tmap, p));
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
