// The L2 distance tile of the descriptor matchers on tcgen05, shared by nn_match_tc_kernel (eval.cu) and
// match_pairs_kernel (match.cu) so that both compute every distance with the same operations:
//   - the fp32 descriptors are split into fp16 (hi, lo) halves on the way into shared memory and the dot product is
//     accumulated as hi*hi + hi*lo + lo*hi in fp32 TMEM (error ~2^-22, i.e. fp32 quality on L2-normalised descriptors);
//   - |row|^2 is an fp32 FMA chain per 64-element K step, the steps summed in order;
//   - d^2 = max(fma(-2, q.t, |q|^2 + |t|^2), 0).
#pragma once
#include "tc_ptx.cuh"

namespace nntc {

using namespace tcptx;

constexpr int kMT = 128;            // query rows per CTA (TMEM lanes)
constexpr int kNT = 128;            // train rows per tile (accumulator columns)
constexpr int kKC = 64;             // K elements staged per step (4 MMA K-steps of 16)
constexpr int kPlane = kMT * 16;    // bytes of one 8-element K chunk for 128 rows: [row][8 halfs]
constexpr int kOpBytes = (kKC / 8) * kPlane;   // 16 KB: one operand (hi or lo) of one K step
constexpr size_t kSmemBytes = 4 * (size_t)kOpBytes + 1024;   // A hi, A lo, B hi, B lo + alignment slack

// rows [row0, row0 + 128) x K [k0, k0 + 64) of src (row-major fp32, `n` valid rows) -> hi / lo fp16 operand images
// [chunk 8][row 128][8]; returns this thread's partial |row|^2 (thread = row).
__device__ __forceinline__ float stage_operand(const float* __restrict__ src, int n, int C, int row0, int k0, uint8_t* hi, uint8_t* lo) {
  const int r = threadIdx.x;
  const bool live = row0 + r < n;
  const float4* g = reinterpret_cast<const float4*>(src + (size_t)(row0 + r) * C + k0);
  float ss = 0.f;
#pragma unroll
  for (int c = 0; c < kKC / 8; ++c) {
    float v[8];
    if (live) {
      const float4 a = __ldg(g + 2 * c), b = __ldg(g + 2 * c + 1);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = 0.f;
    }
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const __half h0 = __float2half_rn(v[2 * e]), h1 = __float2half_rn(v[2 * e + 1]);
      const __half l0 = __float2half_rn(v[2 * e] - __half2float(h0)), l1 = __float2half_rn(v[2 * e + 1] - __half2float(h1));
      h[e] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
      l[e] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
      ss = fmaf(v[2 * e], v[2 * e], ss);
      ss = fmaf(v[2 * e + 1], v[2 * e + 1], ss);
    }
    *reinterpret_cast<uint4*>(hi + (size_t)c * kPlane + (size_t)r * 16) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + (size_t)c * kPlane + (size_t)r * 16) = make_uint4(l[0], l[1], l[2], l[3]);
  }
  return ss;
}

// The 128 x 128 dot-product tile q[q0, q0 + 128) . t[t0, t0 + 128) over all C into the TMEM accumulator at tmem_base
// (128 columns), K step by K step through the four 16 KB operand buffers at smem.  All 128 threads call it; on return
// every MMA has completed.  na / nb: this thread's |q row|^2 and |t row|^2 (thread = row of the tile).
__device__ __forceinline__ void dot_tile(const float* qb, int nq, int q0, const float* tb, int nt, int t0, int C, uint8_t* smem,
                                         uint64_t* bar, uint32_t& phase, uint32_t tmem_base, float& na, float& nb) {
  uint8_t* a_hi = smem;
  uint8_t* a_lo = smem + kOpBytes;
  uint8_t* b_hi = smem + 2 * kOpBytes;
  uint8_t* b_lo = smem + 3 * kOpBytes;
  // instruction descriptor: fp16 x fp16 -> fp32, M = 128, N = 128, both operands K-major
  const uint32_t idesc = (1u << 4) | ((uint32_t)(kNT >> 3) << 17) | ((uint32_t)(kMT >> 4) << 24);
  const uint32_t d_hi = (128u >> 4) | (1u << 14);                    // SBO: 8 rows x 16 B
  const uint32_t lbo = ((uint32_t)kPlane >> 4) << 16;               // LBO: next 8-element K chunk
  na = 0.f;
  nb = 0.f;
  for (int k0 = 0; k0 < C; k0 += kKC) {
    na += stage_operand(qb, nq, C, q0, k0, a_hi, a_lo);
    nb += stage_operand(tb, nt, C, t0, k0, b_hi, b_lo);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy stores -> tensor-core reads
    __syncthreads();
    if (threadIdx.x == 0) {
      tc_fence_after();
#pragma unroll
      for (int kk = 0; kk < kKC / 16; ++kk) {
        const uint32_t off = ((uint32_t)kk * 2 * kPlane) >> 4;
        const uint32_t ah = ((smem_u32(a_hi) >> 4) + off) | lbo, al = ((smem_u32(a_lo) >> 4) + off) | lbo;
        const uint32_t bh = ((smem_u32(b_hi) >> 4) + off) | lbo, bl = ((smem_u32(b_lo) >> 4) + off) | lbo;
        umma_f16_2w(tmem_base, ah, d_hi, bh, d_hi, idesc, (k0 | kk) ? 1u : 0u);   // hi . hi
        umma_f16_2w(tmem_base, ah, d_hi, bl, d_hi, idesc, 1u);                    // hi . lo
        umma_f16_2w(tmem_base, al, d_hi, bh, d_hi, idesc, 1u);                    // lo . hi
      }
      umma_commit(bar);
    }
    mbar_wait(bar, phase);   // the MMAs have read this step's operands: the buffers may be refilled
    phase ^= 1;
  }
  tc_fence_after();
}

__device__ __forceinline__ float dist2(uint32_t dot_bits, float na, float nb) {
  return fmaxf(fmaf(-2.0f, __uint_as_float(dot_bits), na + nb), 0.f);
}

}  // namespace nntc
