// spn_knn and spn_residual_sums (include/spn_retrieval.h): the kernels of vocabulary-based image retrieval.
//
//   knn_kernel             one 128-thread CTA per 128-query block.  It walks the train rows in ascending 128-row tiles,
//                          each the tcgen05 distance tile of the matchers (nn_tc.cuh), so every d^2 has the bits it has
//                          in spn_match_pairs.  Thread = query row keeps a sorted top-k list in shared memory (slot-major,
//                          so the 128 threads of a slot hit 128 consecutive words) and inserts only on a strict '<' in
//                          ascending j: ties go to the lower index, no atomics.
//   residual_sums_kernel   one 256-thread CTA per (image, block of 32 words, block of 256 channels).  Thread = channel
//                          walks the image's rows in ascending order and adds x_i - c_w into its column of a shared
//                          accumulator [32 words][256 channels]: one owner per output element, the order of the header.
#include <math.h>

#include "spn_common.cuh"
#include "nn_tc.cuh"
#include "../../include/spn_retrieval.h"

namespace {

using namespace nntc;

constexpr int kMaxK = 128, kMaxC = 65536, kMaxRows = 1 << 26;
constexpr int kWB = 32, kRC = 256;            // residual sums: words and channels per CTA
constexpr int kMaxCap = 1 << 20, kMaxWords = 65536;

struct KnnParams {
  const float* query;    // [nq][C]
  const float* train;    // [nt][C]
  int nq, nt, C, k;
  int exclude_self;
  int* index;            // [nq][k]
  float* dist2;          // [nq][k]
};

// Sorted insert of (d2, j) into this thread's list (slot s at [s * kMT]); the caller has checked d2 < the k-th entry.
__device__ __forceinline__ float topk_insert(float* td, int* ti, int k, float d2, int j) {
  int s = k - 1;
  while (s > 0) {
    const float prev = td[(s - 1) * kMT];
    if (!(prev > d2)) break;   // an equal distance was seen first, at a lower index: it stays in front
    td[s * kMT] = prev;
    ti[s * kMT] = ti[(s - 1) * kMT];
    --s;
  }
  td[s * kMT] = d2;
  ti[s * kMT] = j;
  return td[(k - 1) * kMT];
}

__global__ void __launch_bounds__(128, 1) knn_kernel(const KnnParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];   // A hi, A lo, B hi, B lo (4 x 16 KB), then the top-k lists
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ float nb_s[kNT];
  float* td = reinterpret_cast<float*>(smem + kSmemBytes) + threadIdx.x;   // [k][128] distances
  int* ti = reinterpret_cast<int*>(td - threadIdx.x + p.k * kMT) + threadIdx.x;   // [k][128] indices
  const int q0 = blockIdx.x * kMT;
  const int i = q0 + (int)threadIdx.x;
  const int skip = p.exclude_self ? i : -1;
  for (int s = 0; s < p.k; ++s) { td[s * kMT] = INFINITY; ti[s * kMT] = -1; }
  float kth = INFINITY;
  if (p.nt > 0) {   // uniform per CTA
    const int warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
      mbar_init(&bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 0) {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(tmem_cols(p.C)));
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_base_s;
    uint32_t phase = 0;
    for (int t0 = 0; t0 < p.nt; t0 += kNT) {
      float na, nb;
      dot_tile(p.query, p.nq, q0, p.train, p.nt, t0, p.C, smem, &bar, phase, tmem_base, na, nb);
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
          if (j < p.nt && d2 < kth && j != skip) kth = topk_insert(td, ti, p.k, d2, j);
        }
      }
      tc_fence_before();
      __syncthreads();   // TMEM and nb_s are read: the next tile may overwrite them
      tc_fence_after();
    }
    if (warp == 0) {
      tc_fence_after();
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols(p.C)));
    }
  }
  if (i < p.nq) {
    const size_t o = (size_t)i * p.k;
    for (int s = 0; s < p.k; ++s) {
      p.index[o + s] = ti[s * kMT];
      p.dist2[o + s] = td[s * kMT];
    }
  }
}

struct ResidualParams {
  const float* desc;     // [N][cap][C]
  const int* count;      // [N]
  const int* assign;     // [N][cap]
  const float* words;    // [K][C]
  int cap, C, K;
  float* sums;           // [N][K][C]
  int* n;                // [N][K]
};

__global__ void __launch_bounds__(kRC) residual_sums_kernel(const ResidualParams p) {
  __shared__ float acc[kWB][kRC];
  __shared__ int word_s[kRC];
  __shared__ int num[kWB];
  const int img = blockIdx.x, w0 = blockIdx.y * kWB, c = blockIdx.z * kRC + (int)threadIdx.x;
  const int nw = min(kWB, p.K - w0);
  const bool counter = threadIdx.x == 0 && blockIdx.z == 0;
  const bool live = c < p.C;
#pragma unroll
  for (int w = 0; w < kWB; ++w) acc[w][threadIdx.x] = 0.f;
  if (counter) for (int w = 0; w < kWB; ++w) num[w] = 0;
  const int cnt = min(max(p.count[img], 0), p.cap);
  const int* a = p.assign + (size_t)img * p.cap;
  const float* x = p.desc + (size_t)img * p.cap * p.C + (live ? c : 0);
  const float* cw = p.words + (size_t)w0 * p.C + (live ? c : 0);
  for (int i0 = 0; i0 < cnt; i0 += kRC) {
    __syncthreads();   // word_s of the previous chunk is read
    if (i0 + (int)threadIdx.x < cnt) {
      const int aw = a[i0 + threadIdx.x];   // compared before the subtraction, so no assignment can overflow
      word_s[threadIdx.x] = aw >= w0 && aw < w0 + nw ? aw - w0 : -1;
    }
    __syncthreads();
    const int m = min(kRC, cnt - i0);
    for (int r = 0; r < m; ++r) {
      const int w = word_s[r];
      if (w < 0) continue;
      if (live) acc[w][threadIdx.x] = __fadd_rn(acc[w][threadIdx.x], __fsub_rn(x[(size_t)(i0 + r) * p.C], cw[(size_t)w * p.C]));
      if (counter) ++num[w];
    }
  }
  for (int w = 0; w < nw; ++w) {
    const size_t o = (size_t)img * p.K + w0 + w;
    if (live) p.sums[o * p.C + c] = acc[w][threadIdx.x];
    if (counter) p.n[o] = num[w];
  }
}

}  // namespace

extern "C" int spn_knn(spn_ctx* ctx, const float* d_query, int nq, const float* d_train, int nt, int C, int k, int exclude_self,
                       int32_t* d_index, float* d_dist2, spn_stream stream) {
  SPN_REQUIRE(ctx, "spn_knn: null pointer (ctx)");
  SPN_REQUIRE(k >= 1 && k <= kMaxK, "spn_knn: k = %d outside [1, %d]", k, kMaxK);
  SPN_REQUIRE(C > 0 && C % kKC == 0 && C <= kMaxC, "spn_knn: C = %d must be a positive multiple of %d up to %d", C, kKC, kMaxC);
  SPN_REQUIRE(nq >= 0 && nq <= kMaxRows, "spn_knn: nq = %d query rows outside [0, %d]", nq, kMaxRows);
  SPN_REQUIRE(nt >= 0 && nt <= kMaxRows, "spn_knn: nt = %d train rows outside [0, %d]", nt, kMaxRows);
  SPN_REQUIRE(!exclude_self || nq == nt, "spn_knn: exclude_self needs the same set as query and train (nq = %d, nt = %d)", nq, nt);
  if (nq == 0) return SPN_OK;
  SPN_REQUIRE(d_query && (d_train || nt == 0) && d_index && d_dist2, "spn_knn: null pointer (query / train / outputs)");
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t smem = kSmemBytes + (size_t)k * kMT * (sizeof(float) + sizeof(int32_t));
  SPN_CUDA(cudaFuncSetAttribute(knn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  KnnParams p;
  p.query = d_query; p.train = d_train; p.nq = nq; p.nt = nt; p.C = C; p.k = k; p.exclude_self = exclude_self ? 1 : 0;
  p.index = d_index; p.dist2 = d_dist2;
  knn_kernel<<<spn_cdiv(nq, kMT), 128, smem, s>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_residual_sums(spn_ctx* ctx, const float* d_desc, const int32_t* d_count, const int32_t* d_assign,
                                 const float* d_words, int N, int cap, int C, int K, float* d_sums, int32_t* d_n,
                                 spn_stream stream) {
  SPN_REQUIRE(ctx, "spn_residual_sums: null pointer (ctx)");
  SPN_REQUIRE(N >= 0 && N <= kMaxRows, "spn_residual_sums: N = %d images outside [0, %d]", N, kMaxRows);
  SPN_REQUIRE(cap > 0 && cap <= kMaxCap, "spn_residual_sums: cap = %d outside [1, %d]", cap, kMaxCap);
  SPN_REQUIRE(C > 0 && C <= kMaxC, "spn_residual_sums: C = %d outside [1, %d]", C, kMaxC);
  SPN_REQUIRE(K > 0 && K <= kMaxWords, "spn_residual_sums: K = %d words outside [1, %d]", K, kMaxWords);
  if (N == 0) return SPN_OK;
  SPN_REQUIRE(d_desc && d_count && d_assign && d_words && d_sums && d_n, "spn_residual_sums: null pointer (inputs / outputs)");
  SpnDeviceGuard guard(ctx->device);
  ResidualParams p;
  p.desc = d_desc; p.count = d_count; p.assign = d_assign; p.words = d_words; p.cap = cap; p.C = C; p.K = K;
  p.sums = d_sums; p.n = d_n;
  residual_sums_kernel<<<dim3(N, spn_cdiv(K, kWB), spn_cdiv(C, kRC)), kRC, 0, (cudaStream_t)stream>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
