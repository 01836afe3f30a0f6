// spn_match_pairs (include/spn_match.h): nearest-neighbour matching with mutual check, ratio test and distance
// threshold over a pool of descriptor sets.
//
//   match_pairs_kernel   one 128-thread CTA per (pair, 128-query block of a).  It walks b's rows in ascending 128-row
//                        tiles; each tile is the same tcgen05 distance tile as nn_match_tc_kernel (nn_tc.cuh), so every
//                        distance has the same bits as there.  Thread = query row keeps (best, best_j, second) in
//                        registers with strict '<' in ascending j: ties go to the lower index, no atomics, the same
//                        result run to run.  The reverse pass (query = b, train = a) only writes b's nearest row of a
//                        into scratch; the forward pass applies the mutual, ratio and threshold filters in its epilogue.
#include <math.h>

#include "spn_common.cuh"
#include "nn_tc.cuh"
#include "../../include/spn_match.h"

namespace {

using namespace nntc;

constexpr int kMaxN = 1 << 20, kMaxCap = 16384, kMaxPairs = 65535;

struct PairParams {
  const float* desc;     // [N][cap][C]
  const int* count;      // [N]
  const int* pairs;      // [P][2] (a, b), uploaded
  int cap, C;
  int reverse;           // 1: query set = b, train set = a; writes nearest[] only
  int* nearest;          // [P][cap]: nearest row of a for every row of b (written by the reverse pass, read with mutual)
  int mutual;
  float ratio, max_dist;
  int* match;            // [P][cap]
  float* dist;           // [P][cap]
};

__global__ void __launch_bounds__(128, 1) match_pairs_kernel(const PairParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];   // A hi, A lo, B hi, B lo: 4 x 16 KB
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ float nb_s[kNT];
  const int q = blockIdx.y;
  const int ia = p.pairs[2 * q], ib = p.pairs[2 * q + 1];
  const int qs = p.reverse ? ib : ia, ts = p.reverse ? ia : ib;
  const int nq = min(max(p.count[qs], 0), p.cap), nt = min(max(p.count[ts], 0), p.cap);
  const int q0 = blockIdx.x * kMT;
  const int i = q0 + (int)threadIdx.x;
  const size_t out = (size_t)q * p.cap + i;
  if (q0 >= nq || nt == 0) {   // uniform per CTA: nothing to match in this block
    if (!p.reverse && i < p.cap) { p.match[out] = -1; p.dist[out] = 0.f; }
    return;
  }
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(128));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_s;
  const float* qb = p.desc + (size_t)qs * p.cap * p.C;
  const float* tb = p.desc + (size_t)ts * p.cap * p.C;
  float best = INFINITY, second = INFINITY;
  int best_j = 0;
  uint32_t phase = 0;
  for (int t0 = 0; t0 < nt; t0 += kNT) {
    float na, nb;
    dot_tile(qb, nq, q0, tb, nt, t0, p.C, smem, &bar, phase, tmem_base, na, nb);
    nb_s[threadIdx.x] = nb;
    __syncthreads();
#pragma unroll 1
    for (int c0 = 0; c0 < kNT; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
      tmem_ld_wait();
#pragma unroll
      for (int c = 0; c < 32; ++c) {
        const int j = t0 + c0 + c;
        const float d2 = dist2(v[c], na, nb_s[c0 + c]);
        if (j < nt) {
          if (d2 < best) { second = best; best = d2; best_j = j; }
          else if (d2 < second) second = d2;
        }
      }
    }
    tc_fence_before();
    __syncthreads();   // TMEM and nb_s are read: the next tile may overwrite them
    tc_fence_after();
  }
  if (p.reverse) {
    if (i < nq) p.nearest[out] = best_j;
  } else if (i < p.cap) {
    int m = -1;
    float d = 0.f;
    if (i < nq) {
      const float d1 = sqrtf(best);
      bool keep = !p.mutual || p.nearest[(size_t)q * p.cap + best_j] == i;
      if (p.ratio > 0.f) keep = keep && d1 < __fmul_rn(p.ratio, sqrtf(second));
      keep = keep && d1 <= p.max_dist;
      if (keep) { m = best_j; d = d1; }
    }
    p.match[out] = m;
    p.dist[out] = d;
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(128));
  }
}

}  // namespace

extern "C" int spn_match_pairs(spn_ctx* ctx, const float* d_desc, const int32_t* d_count, int N, int cap, int C,
                               const int32_t* h_pairs, int P, int mutual, float ratio, float max_dist, int32_t* d_match,
                               float* d_dist, spn_stream stream) {
  SPN_REQUIRE(ctx && d_desc && d_count, "spn_match_pairs: null pointer");
  SPN_REQUIRE(N > 0 && N <= kMaxN, "spn_match_pairs: N = %d descriptor sets outside [1, %d]", N, kMaxN);
  SPN_REQUIRE(cap > 0 && cap <= kMaxCap, "spn_match_pairs: cap = %d outside [1, %d]", cap, kMaxCap);
  SPN_REQUIRE(C > 0 && C % kKC == 0, "spn_match_pairs: C = %d must be a positive multiple of %d", C, kKC);
  SPN_REQUIRE(P >= 0 && P <= kMaxPairs, "spn_match_pairs: P = %d pairs outside [0, %d]", P, kMaxPairs);
  SPN_REQUIRE(ratio >= 0.f && ratio <= 1.f, "spn_match_pairs: ratio must be in [0, 1] (0: no ratio test), got %g", (double)ratio);
  SPN_REQUIRE(!isnan(max_dist), "spn_match_pairs: max_dist must not be NaN (+inf: no threshold)");
  if (P == 0) return SPN_OK;
  SPN_REQUIRE(h_pairs && d_match && d_dist, "spn_match_pairs: null pointer (h_pairs / outputs)");
  for (int q = 0; q < P; ++q)
    SPN_REQUIRE(h_pairs[2 * q] >= 0 && h_pairs[2 * q] < N && h_pairs[2 * q + 1] >= 0 && h_pairs[2 * q + 1] < N,
                "spn_match_pairs: pair %d = (%d, %d) has a set index outside [0, %d)", q, h_pairs[2 * q], h_pairs[2 * q + 1], N);
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t pair_bytes = (size_t)P * 2 * sizeof(int32_t);
  const size_t near_bytes = mutual ? (size_t)P * cap * sizeof(int32_t) : 0;
  int rc = spn_ensure_aux(ctx, pair_bytes + near_bytes, s);
  if (rc) return rc;
  // pageable source: the call returns once the bytes are staged
  SPN_CUDA(cudaMemcpyAsync(ctx->aux, h_pairs, pair_bytes, cudaMemcpyHostToDevice, s));
  SPN_CUDA(cudaFuncSetAttribute(match_pairs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
  PairParams p;
  p.desc = d_desc; p.count = d_count; p.pairs = (const int*)ctx->aux; p.cap = cap; p.C = C;
  p.nearest = mutual ? (int*)(ctx->aux + pair_bytes) : nullptr;
  p.mutual = mutual ? 1 : 0; p.ratio = ratio; p.max_dist = max_dist; p.match = d_match; p.dist = d_dist;
  const dim3 grid(spn_cdiv(cap, kMT), P);
  if (mutual) {
    p.reverse = 1;
    match_pairs_kernel<<<grid, 128, kSmemBytes, s>>>(p);   // nearest row of a for every row of b
    SPN_CHECK_LAUNCH(ctx);
  }
  p.reverse = 0;
  match_pairs_kernel<<<grid, 128, kSmemBytes, s>>>(p);     // every row of a: nearest, second, filters
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
