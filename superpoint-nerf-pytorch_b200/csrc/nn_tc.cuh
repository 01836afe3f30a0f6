// The L2 distance tile of the descriptor matchers on tcgen05, shared by nn_match_tc_kernel (eval.cu),
// match_pairs_kernel (match.cu) and knn_kernel (retrieval.cu) so that all compute every distance with the same operations:
//   - the fp32 descriptors are split into fp16 (hi, lo) halves on the way into shared memory and the dot product is
//     accumulated as hi*hi + hi*lo + lo*hi in fp32 TMEM (error ~2^-22, i.e. fp32 quality on L2-normalised descriptors);
//   - the tensor core truncates each accumulation to fp32, a bias that grows with the number of MMAs into one
//     accumulator.  So each chunk of kChunk K elements starts a fresh accumulator, and the chunks after the first are
//     added into the first in fp32 (round to nearest) on the CUDA cores.  Up to C = kChunk there is one chunk and no add;
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
constexpr int kChunk = 256;         // K elements per tensor-core accumulator (multiple of kKC)

// TMEM columns a kernel allocates for dot_tile: the result tile, and for C > kChunk a second tile for the later chunks.
__host__ __device__ constexpr uint32_t tmem_cols(int C) { return C > kChunk ? 2 * kNT : kNT; }

// run += chunk over this warp's 32 lanes x 128 columns, in fp32 with round to nearest, 32 columns at a time.
__device__ __forceinline__ void add_chunk(uint32_t run, uint32_t chunk) {
#pragma unroll 1
  for (int c0 = 0; c0 < kNT; c0 += 32) {
    uint32_t a[32], b[32];
    tmem_ld32(run + c0, a);
    tmem_ld32(chunk + c0, b);
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < 32; ++c) a[c] = __float_as_uint(__fadd_rn(__uint_as_float(a[c]), __uint_as_float(b[c])));
    tmem_st32(run + c0, a);
  }
  tmem_st_wait();
}

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
// (128 columns; tmem_cols(C) allocated, the columns after the first 128 hold the chunk in flight), K step by K step
// through the four 16 KB operand buffers at smem.  All 128 threads call it; on return every MMA and every chunk add
// has completed.  na / nb: this thread's |q row|^2 and |t row|^2 (thread = row of the tile).
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
  const uint32_t lanes = (uint32_t)((threadIdx.x >> 5) * 32) << 16;   // this warp's TMEM lanes
  na = 0.f;
  nb = 0.f;
  for (int k0 = 0; k0 < C; k0 += kKC) {
    const int kc = k0 % kChunk;                                           // K offset inside the chunk
    const uint32_t acc = k0 < kChunk ? tmem_base : tmem_base + kNT;      // chunk 0 accumulates in the result tile
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
        umma_f16_2w(acc, ah, d_hi, bh, d_hi, idesc, (kc | kk) ? 1u : 0u);   // hi . hi
        umma_f16_2w(acc, ah, d_hi, bl, d_hi, idesc, 1u);                    // hi . lo
        umma_f16_2w(acc, al, d_hi, bh, d_hi, idesc, 1u);                    // lo . hi
      }
      umma_commit(bar);
    }
    mbar_wait(bar, phase);   // the MMAs have completed and read this step's operands: the buffers may be refilled
    phase ^= 1;
    if (k0 >= kChunk && (kc + kKC == kChunk || k0 + kKC == C)) {   // a later chunk is complete: add it to the result
      tc_fence_after();
      add_chunk(tmem_base + lanes, tmem_base + kNT + lanes);
      tc_fence_before();     // the next chunk's MMAs overwrite the chunk tile after the __syncthreads of its first step
    }
  }
  tc_fence_after();
}

__device__ __forceinline__ float dist2(uint32_t dot_bits, float na, float nb) {
  return fmaxf(fmaf(-2.0f, __uint_as_float(dot_bits), na + nb), 0.f);
}

}  // namespace nntc
