// Strict-mode (fp32 FFMA) convolution + the softmax / dustbin-drop / depth-to-space kernel.
//
// conv: VGG_Block.forward = conv(k, stride 1, pad k/2) + BN(eval) + ReLU + MaxPool(2,2)
//       (reference models/model_utils/VGG_Backbone.py:23-36) with BN folded into the weights.
//       NCHW fp32 in and out, i.e. the reference's own layout.  This is the 1e-4 parity path; the
//       throughput path is the tcgen05 implicit GEMM in front_tc.cu / conv_fold.cu / conv_tc.cu.
// softmax_d2s: Detector_head.forward lines heads.py:25-28 (softmax over 65, drop channel 64,
//       pixel_shuffle(8), squeeze) optionally multiplied by the validity mask (export.py:70).
#include "spn_common.cuh"

namespace {

constexpr int kTW = 32, kTH = 16, kCiChunk = 8, kCoTile = 16, kSW = 36;

template <int KS, bool POOL>
__global__ void __launch_bounds__(256)
conv_fp32_kernel(const float* __restrict__ in, const float* __restrict__ wpk, const float* __restrict__ bias,
                 float* __restrict__ out, int Cin, int Cout, int cout_pad, int H, int W, int tiles_x, int relu) {
  constexpr int TAPS = KS * KS;
  constexpr int HALO = KS / 2;
  constexpr int SH = kTH + 2 * HALO;
  __shared__ __align__(16) float in_s[kCiChunk][SH][kSW];
  __shared__ __align__(16) float w_s[kCiChunk][TAPS][kCoTile];

  const int tile = blockIdx.x;
  const int tx0 = (tile % tiles_x) * kTW, ty0 = (tile / tiles_x) * kTH;
  const int co0 = blockIdx.y * kCoTile;
  const int b = blockIdx.z;
  const int tid = threadIdx.x;
  const int strip = tid & 127, cg = tid >> 7;
  const int sx = strip & 7, sy = strip >> 3;
  const int x0 = sx * 4;

  float acc[4][8];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

  const float* inb = in + (size_t)b * Cin * H * W;
  for (int c0 = 0; c0 < Cin; c0 += kCiChunk) {
    const int nci = min(kCiChunk, Cin - c0);
    for (int i = tid; i < nci * SH * kSW; i += 256) {
      int ci = i / (SH * kSW);
      int rem = i - ci * (SH * kSW);
      int r = rem / kSW, c = rem - r * kSW;
      int gy = ty0 + r - HALO, gx = tx0 + c - HALO;
      float v = 0.f;
      if (c < kTW + 2 * HALO && gy >= 0 && gy < H && gx >= 0 && gx < W) v = __ldg(&inb[((size_t)(c0 + ci) * H + gy) * W + gx]);
      in_s[ci][r][c] = v;
    }
    for (int i = tid; i < nci * TAPS * kCoTile; i += 256) {
      int ci = i / (TAPS * kCoTile);
      int rem = i - ci * (TAPS * kCoTile);
      int t = rem / kCoTile, co = rem - t * kCoTile;
      w_s[ci][t][co] = __ldg(&wpk[((size_t)(c0 + ci) * TAPS + t) * cout_pad + co0 + co]);
    }
    __syncthreads();
    for (int ci = 0; ci < nci; ++ci) {
#pragma unroll
      for (int ky = 0; ky < KS; ++ky) {
        float r[4 + KS - 1];
        const float4 a = *reinterpret_cast<const float4*>(&in_s[ci][sy + ky][x0]);
        r[0] = a.x; r[1] = a.y; r[2] = a.z; r[3] = a.w;
        if (KS == 3) {
          const float2 b2 = *reinterpret_cast<const float2*>(&in_s[ci][sy + ky][x0 + 4]);
          r[4] = b2.x; r[5] = b2.y;
        }
#pragma unroll
        for (int kx = 0; kx < KS; ++kx) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            const float4 w = *reinterpret_cast<const float4*>(&w_s[ci][ky * KS + kx][cg * 8 + h * 4]);
#pragma unroll
            for (int px = 0; px < 4; ++px) {
              acc[px][h * 4 + 0] = fmaf(r[px + kx], w.x, acc[px][h * 4 + 0]);
              acc[px][h * 4 + 1] = fmaf(r[px + kx], w.y, acc[px][h * 4 + 1]);
              acc[px][h * 4 + 2] = fmaf(r[px + kx], w.z, acc[px][h * 4 + 2]);
              acc[px][h * 4 + 3] = fmaf(r[px + kx], w.w, acc[px][h * 4 + 3]);
            }
          }
        }
      }
    }
    __syncthreads();
  }

  const int y = ty0 + sy, x = tx0 + x0;
#pragma unroll
  for (int co = 0; co < 8; ++co) {
    const int cidx = co0 + cg * 8 + co;  // warp-uniform
    if (cidx >= Cout) break;
    const float bv = __ldg(&bias[cidx]);
    float v[4];
#pragma unroll
    for (int px = 0; px < 4; ++px) {
      v[px] = acc[px][co] + bv;
      if (relu) v[px] = fmaxf(v[px], 0.f);
    }
    if (!POOL) {
      if (y < H) {
        float* o = out + (((size_t)b * Cout + cidx) * H + y) * W + x;
        if ((W & 3) == 0 && x + 3 < W) {
          *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
          for (int px = 0; px < 4; ++px)
            if (x + px < W) o[px] = v[px];
        }
      }
    } else {
      float m0 = fmaxf(v[0], v[1]), m1 = fmaxf(v[2], v[3]);
      m0 = fmaxf(m0, __shfl_xor_sync(0xffffffffu, m0, 8));  // row partner sy^1 lives in lane^8
      m1 = fmaxf(m1, __shfl_xor_sync(0xffffffffu, m1, 8));
      const int Ho = H >> 1, Wo = W >> 1;
      const int oy = y >> 1, ox = x >> 1;
      if ((sy & 1) == 0 && oy < Ho) {
        float* o = out + (((size_t)b * Cout + cidx) * Ho + oy) * Wo + ox;
        if (ox < Wo) o[0] = m0;
        if (ox + 1 < Wo) o[1] = m1;
      }
    }
  }
}

__global__ void __launch_bounds__(128)
softmax_d2s_kernel(const float* __restrict__ logits, const uint8_t* __restrict__ mask, float* __restrict__ prob,
                   int B, int Hc, int Wc) {
  const int cells = Hc * Wc;
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * cells) return;
  const int b = idx / cells, cell = idx - b * cells;
  const int cy = cell / Wc, cx = cell - cy * Wc;
  const float* lp = logits + (size_t)b * 65 * cells + cell;
  float v[65];
  float m = -INFINITY;
#pragma unroll
  for (int c = 0; c < 65; ++c) {
    v[c] = __ldg(lp + (size_t)c * cells);
    m = fmaxf(m, v[c]);
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < 65; ++c) {
    v[c] = expf(v[c] - m);
    s += v[c];
  }
  const int H = Hc * 8, W = Wc * 8;
#pragma unroll
  for (int dy = 0; dy < 8; ++dy) {
    const size_t o = ((size_t)b * H + cy * 8 + dy) * W + cx * 8;
    float p[8];
#pragma unroll
    for (int dx = 0; dx < 8; ++dx) p[dx] = v[dy * 8 + dx] / s;
    if (mask) {
      const uint2 mm = *reinterpret_cast<const uint2*>(mask + o);
#pragma unroll
      for (int dx = 0; dx < 4; ++dx) {
        p[dx] *= (float)((mm.x >> (8 * dx)) & 0xff);
        p[4 + dx] *= (float)((mm.y >> (8 * dx)) & 0xff);
      }
    }
    *reinterpret_cast<float4*>(prob + o) = make_float4(p[0], p[1], p[2], p[3]);
    *reinterpret_cast<float4*>(prob + o + 4) = make_float4(p[4], p[5], p[6], p[7]);
  }
}

}  // namespace

int spn_conv_fp32(spn_ctx* ctx, int layer, const float* in, float* out, int B, int H, int W, bool relu, bool pool,
                  cudaStream_t s) {
  const SpnLayer& L = ctx->layers[layer];
  if (!L.w32) {
    spn_set_error("layer %d has no weights (call spn_pack_weights first)", layer);
    return SPN_E_STATE;
  }
  SPN_REQUIRE(!pool || L.ks == 3, "pooling only fused into 3x3 layers");
  const int tiles_x = spn_cdiv(W, kTW), tiles_y = spn_cdiv(H, kTH);
  dim3 grid(tiles_x * tiles_y, L.cout_pad / kCoTile, B), block(256);
  SpnProfScope prof(ctx, layer, s);
  if (L.ks == 3) {
    if (pool)
      conv_fp32_kernel<3, true><<<grid, block, 0, s>>>(in, L.w32, L.bias, out, L.cin, L.cout, L.cout_pad, H, W, tiles_x, relu);
    else
      conv_fp32_kernel<3, false><<<grid, block, 0, s>>>(in, L.w32, L.bias, out, L.cin, L.cout, L.cout_pad, H, W, tiles_x, relu);
  } else {
    conv_fp32_kernel<1, false><<<grid, block, 0, s>>>(in, L.w32, L.bias, out, L.cin, L.cout, L.cout_pad, H, W, tiles_x, relu);
  }
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

int spn_softmax_d2s(spn_ctx* ctx, const float* logits, int B, int Hc, int Wc, const uint8_t* mask, float* prob,
                    cudaStream_t s) {
  const int n = B * Hc * Wc;
  SpnProfScope prof(ctx, SPN_PROF_SOFTMAX, s);
  softmax_d2s_kernel<<<spn_cdiv(n, 128), 128, 0, s>>>(logits, mask, prob, B, Hc, Wc);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
