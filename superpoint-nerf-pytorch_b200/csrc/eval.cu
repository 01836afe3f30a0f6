// On-GPU evaluation of the exports (SURVEY.md section 8f-3): the keypoint selection, repeatability counting and
// mutual-nearest-neighbour descriptor matching of the reference's evaluation scripts
//   evaluations/detector_evaluation.py:145-238   compute_repeatability
//   evaluations/descriptor_evaluation.py:17-90   keep_shared_points, compute_homography (matching part)
// The RANSAC homography fit that follows the matching stays with cv2 on the host, as in the reference.
//
//   select_keypoints_kernel   np.where(prob > 0) + warp_keypoints / keep_true_keypoints / filter_keypoints (fp64, as
//                             numpy) + select_k_best (ascending by probability, last k): one CTA per map, candidates
//                             compacted into shared memory and bitonic-sorted as 64-bit (prob bits, pixel index) keys
//   repeat_count_kernel       N1 x N2 Euclidean distances in fp64, nearest-neighbour counts within the threshold
//   nn_match_tc_kernel        cv2.BFMatcher(NORM_L2): the N1 x N2 x 256 distance matrix as a tcgen05 GEMM (the tile is
//                             in nn_tc.cuh, shared with match.cu).  The fp32
//                             descriptors are split into fp16 (hi, lo) halves on the way into shared memory and the dot
//                             product is accumulated as hi*hi + hi*lo + lo*hi in fp32 TMEM (error ~2^-22, i.e. fp32
//                             quality on L2-normalised descriptors); the epilogue forms |a|^2 + |b|^2 - 2 a.b per
//                             accumulator row and publishes the row-wise arg-min with one 64-bit atomicMin
//                             (distance bits, index): ties go to the lower index like cv2.
//   cross_check_kernel        crossCheck=True: keep (i, j) iff j is i's nearest and i is j's nearest
//   posed_reproject_kernel    spn_posed_reproject (include/spn_posed.h): one CTA per (pair, direction); every keypoint
//                             through depth and both poses in explicitly rounded fp64, the visibility / occlusion test,
//                             the visible points compacted in keypoint order with a ballot and block scan
#include <math.h>

#include "spn_common.cuh"
#include "nn_tc.cuh"
#include "tc_ptx.cuh"
#include "../../include/spn_posed.h"

namespace {

using namespace tcptx;

// ------------------------------------------------------------------------------------------------ keypoint selection
constexpr int kSelCap = 16384;   // candidates per map held in shared memory (128 KB of 64-bit keys)
constexpr int kSelThreads = 1024;

struct SelParams {
  const float* prob;     // [B][H][W]
  const double* warp;    // [B][9] or null: homography applied to (x = col, y = row, 1)
  int H, W;
  int bound_h, bound_w;  // the warped point must satisfy 0 <= row' < bound_h, 0 <= col' < bound_w
  int emit_warped;       // 0: output the original integer (row, col); 1: output the warped (row', col')
  int keep_k;
  double* pts;           // [B][keep_k][2]
  float* score;          // [B][keep_k]
  int* count;            // [B] points written; [B + b] = candidates before select_k_best (diagnostic / overflow check)
};

__device__ __forceinline__ void warp_point(const double* h, double x, double y, double& wx, double& wy) {
  const double z = h[6] * x + h[7] * y + h[8];
  wx = (h[0] * x + h[1] * y + h[2]) / z;
  wy = (h[3] * x + h[4] * y + h[5]) / z;
}

__global__ void __launch_bounds__(kSelThreads, 1) select_keypoints_kernel(const SelParams p) {
  extern __shared__ unsigned long long keys[];  // kSelCap
  __shared__ int n_s, warp_tot[kSelThreads / 32];
  __shared__ double hm[9];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float* pr = p.prob + (size_t)b * p.H * p.W;
  if (tid == 0) n_s = 0;
  if (tid < 9 && p.warp) hm[tid] = p.warp[(size_t)b * 9 + tid];
  __syncthreads();
  const int npx = p.H * p.W;
  // ordered compaction (row-major, like np.where): chunks of kSelThreads pixels, block-wide exclusive scan of the flags
  for (int base = 0; base < npx; base += kSelThreads) {
    const int i = base + tid;
    bool ok = false;
    float v = 0.f;
    if (i < npx) {
      v = pr[i];
      ok = v > 0.f;
      if (ok && p.warp) {
        const int y = i / p.W, x = i - y * p.W;
        double wx, wy;
        warp_point(hm, (double)x, (double)y, wx, wy);
        ok = wy >= 0.0 && wy < (double)p.bound_h && wx >= 0.0 && wx < (double)p.bound_w;
      }
    }
    const unsigned m = __ballot_sync(0xffffffffu, ok);
    if (lane == 0) warp_tot[wid] = __popc(m);
    __syncthreads();
    int off = n_s;
    for (int w = 0; w < wid; ++w) off += warp_tot[w];
    const int pos = off + __popc(m & ((1u << lane) - 1u));
    if (ok && pos < kSelCap) keys[pos] = ((unsigned long long)__float_as_uint(v) << 32) | (unsigned)i;
    __syncthreads();
    if (tid == 0) {
      int t = 0;
      for (int w = 0; w < kSelThreads / 32; ++w) t += warp_tot[w];
      n_s += t;
    }
    __syncthreads();
  }
  const int n_all = n_s;
  const int n = min(n_all, kSelCap);
  int n2 = 1;
  while (n2 < n) n2 <<= 1;
  for (int i = n + tid; i < n2; i += kSelThreads) keys[i] = ~0ull;
  __syncthreads();
  // bitonic sort, ascending (positive floats order like their bit patterns; ties by pixel index)
  for (int k = 2; k <= n2; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = tid; i < n2; i += kSelThreads) {
        const int l = i ^ j;
        if (l > i) {
          const unsigned long long a = keys[i], c = keys[l];
          const bool up = (i & k) == 0;
          if ((a > c) == up) { keys[i] = c; keys[l] = a; }
        }
      }
      __syncthreads();
    }
  const int kk = min(p.keep_k, n);
  for (int i = tid; i < kk; i += kSelThreads) {  // select_k_best: ascending by probability, the last kk
    const unsigned long long key = keys[n - kk + i];
    const int px = (int)(key & 0xffffffffu);
    const int y = px / p.W, x = px - y * p.W;
    double oy = (double)y, ox = (double)x;
    if (p.warp && p.emit_warped) warp_point(hm, (double)x, (double)y, ox, oy);
    p.pts[((size_t)b * p.keep_k + i) * 2] = oy;
    p.pts[((size_t)b * p.keep_k + i) * 2 + 1] = ox;
    p.score[(size_t)b * p.keep_k + i] = __uint_as_float((unsigned)(key >> 32));
  }
  if (tid == 0) {
    p.count[b] = kk;
    p.count[gridDim.x + b] = n_all;
  }
}

// ------------------------------------------------------------------------------------------------ repeatability counts
// out[b] = {N1, N2, count1, count2}: count1 = #points of set 1 whose nearest point of set 2 is within thresh, and
// vice versa (detector_evaluation.py:214-233).
__global__ void __launch_bounds__(256) repeat_count_kernel(const double* __restrict__ p1, const int* __restrict__ n1,
                                                           const double* __restrict__ p2, const int* __restrict__ n2, int cap,
                                                           double thresh, int* __restrict__ out) {
  __shared__ int c1, c2;
  const int b = blockIdx.x;
  const int N1 = n1[b], N2 = n2[b];
  if (threadIdx.x == 0) { c1 = 0; c2 = 0; }
  __syncthreads();
  const double* a = p1 + (size_t)b * cap * 2;
  const double* c = p2 + (size_t)b * cap * 2;
  int l1 = 0, l2 = 0;
  if (N2 > 0)
    for (int i = threadIdx.x; i < N1; i += blockDim.x) {
      double best = 1e300;
      for (int j = 0; j < N2; ++j) {
        const double dy = a[2 * i] - c[2 * j], dx = a[2 * i + 1] - c[2 * j + 1];
        best = fmin(best, sqrt(dy * dy + dx * dx));
      }
      l1 += best <= thresh;
    }
  if (N1 > 0)
    for (int j = threadIdx.x; j < N2; j += blockDim.x) {
      double best = 1e300;
      for (int i = 0; i < N1; ++i) {
        const double dy = a[2 * i] - c[2 * j], dx = a[2 * i + 1] - c[2 * j + 1];
        best = fmin(best, sqrt(dy * dy + dx * dx));
      }
      l2 += best <= thresh;
    }
  atomicAdd(&c1, l1);
  atomicAdd(&c2, l2);
  __syncthreads();
  if (threadIdx.x == 0) {
    out[4 * b] = N1; out[4 * b + 1] = N2; out[4 * b + 2] = c1; out[4 * b + 3] = c2;
  }
}

// ------------------------------------------------------------------------------------------------ NN matching on tcgen05
using namespace nntc;

struct MatchParams {
  const float* q;        // [B][qcap][C] query descriptors
  const float* t;        // [B][tcap][C] train descriptors
  const int* nq;         // [B]
  const int* nt;         // [B]
  int qcap, tcap, C;
  unsigned long long* best;   // [B][qcap]: (distance^2 bits << 32) | train index, initialised to ~0
};

__global__ void __launch_bounds__(128, 1) nn_match_tc_kernel(const MatchParams p) {
  extern __shared__ __align__(1024) uint8_t smem[];   // A hi, A lo, B hi, B lo: 4 x 16 KB
  __shared__ __align__(8) uint64_t bar;
  __shared__ uint32_t tmem_base_s;
  __shared__ float nb_s[kNT];
  const int b = blockIdx.z;
  const int q0 = blockIdx.y * kMT, t0 = blockIdx.x * kNT;
  const int nq = p.nq[b], nt = p.nt[b];
  if (q0 >= nq || t0 >= nt) return;   // uniform per CTA
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
  const float* qb = p.q + (size_t)b * p.qcap * p.C;
  const float* tb = p.t + (size_t)b * p.tcap * p.C;
  float na, nb;
  uint32_t phase = 0;
  dot_tile(qb, nq, q0, tb, nt, t0, p.C, smem, &bar, phase, tmem_base, na, nb);
  nb_s[threadIdx.x] = nb;
  __syncthreads();
  // epilogue: thread = query row = TMEM lane; arg-min of |a|^2 + |b|^2 - 2 a.b over this CTA's 128 train rows
  float best = INFINITY;
  int best_j = 0;
#pragma unroll 1
  for (int c0 = 0; c0 < kNT; c0 += 32) {
    uint32_t v[32];
    tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, v);
    tmem_ld_wait();
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      const int j = t0 + c0 + c;
      const float d2 = dist2(v[c], na, nb_s[c0 + c]);
      if (j < nt && d2 < best) { best = d2; best_j = j; }
    }
  }
  if (q0 + (int)threadIdx.x < nq)
    atomicMin(&p.best[(size_t)b * p.qcap + q0 + threadIdx.x], ((unsigned long long)__float_as_uint(best) << 32) | (unsigned)best_j);
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols(p.C)));
  }
}

__global__ void fill_u64_kernel(unsigned long long* p, size_t n, unsigned long long v) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) p[i] = v;
}

__global__ void cross_check_kernel(const unsigned long long* __restrict__ bq, const unsigned long long* __restrict__ bt,
                                   const int* __restrict__ nq, const int* __restrict__ nt, int qcap, int tcap,
                                   int* __restrict__ match, float* __restrict__ dist) {
  const int b = blockIdx.y, i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= qcap) return;
  int m = -1;
  float d = 0.f;
  if (i < nq[b] && nt[b] > 0) {
    const unsigned long long k = bq[(size_t)b * qcap + i];
    const int j = (int)(k & 0xffffffffu);
    if ((int)(bt[(size_t)b * tcap + j] & 0xffffffffu) == i) {
      m = j;
      d = sqrtf(__uint_as_float((unsigned)(k >> 32)));
    }
  }
  match[(size_t)b * qcap + i] = m;
  dist[(size_t)b * qcap + i] = d;
}

// ------------------------------------------------------------------------------------------------ posed reprojection
// Every operation is a separately rounded intrinsic so that a numpy restatement in the same order (oracle/posed_oracle.py)
// gives the same bits: nvcc would otherwise contract a * b + c into an FMA.
constexpr int kPosedThreads = 256;

__device__ __forceinline__ double dmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ double dadd(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ double dsub(double a, double b) { return __dsub_rn(a, b); }

// row of a 3x3 product: (m0 x + m1 y) + m2 z
__device__ __forceinline__ double drow(const double* m, double x, double y, double z) {
  return dadd(dadd(dmul(m[0], x), dmul(m[1], y)), dmul(m[2], z));
}

__device__ __forceinline__ double dnorm3(double x, double y, double z) {
  return __dsqrt_rn(dadd(dadd(dmul(x, x), dmul(y, y)), dmul(z, z)));
}

// inverse of a 3x3 fp32 matrix: the adjugate divided by the determinant, in fp64 (labels.cu inverse3x3 without the
// final rounding to float)
__device__ void inverse3x3_d(const float* m, double* o) {
  const double a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], h = m[7], i = m[8];
  const double c00 = dsub(dmul(e, i), dmul(f, h)), c01 = dsub(dmul(f, g), dmul(d, i)), c02 = dsub(dmul(d, h), dmul(e, g));
  const double det = dadd(dadd(dmul(a, c00), dmul(b, c01)), dmul(c, c02));
  o[0] = __ddiv_rn(c00, det); o[1] = __ddiv_rn(dsub(dmul(c, h), dmul(b, i)), det); o[2] = __ddiv_rn(dsub(dmul(b, f), dmul(c, e)), det);
  o[3] = __ddiv_rn(c01, det); o[4] = __ddiv_rn(dsub(dmul(a, i), dmul(c, g)), det); o[5] = __ddiv_rn(dsub(dmul(c, d), dmul(a, f)), det);
  o[6] = __ddiv_rn(c02, det); o[7] = __ddiv_rn(dsub(dmul(b, g), dmul(a, h)), det); o[8] = __ddiv_rn(dsub(dmul(a, e), dmul(b, d)), det);
}

struct PosedParams {
  const int32_t* kp;        // [V][max_kp][2] (row, col)
  const int32_t* kp_count;  // [V]
  const float* depth;       // [V][H][W]
  const float* K;           // [V][9]
  const float* R;           // [V][9]
  const float* t;           // [V][3]
  const int* pairs;         // [P][2] (a, b), uploaded
  int H, W, max_kp;
  double depth_tol;
  double* proj;             // [P][max_kp][2]
  int* vis;                 // [P][2][max_kp]
  double* set1;             // [P][max_kp][2]
  double* set2;             // [P][max_kp][2]
  int* set_count;           // [P][2]
};

// blockIdx.x = 2 q + dir.  dir 0: keypoints of a into b (proj, vis[q][0], set 1 at the projected positions); dir 1:
// keypoints of b into a (vis[q][1], set 2 at b's own integer positions).
__global__ void __launch_bounds__(kPosedThreads) posed_reproject_kernel(const PosedParams p) {
  __shared__ double Ks[9], Kinv[9], Rs[9], Rinv[9], ts[3], tdst[3];
  __shared__ int warp_n[kPosedThreads / 32];
  __shared__ int base;
  const int q = blockIdx.x >> 1, dir = blockIdx.x & 1;
  const int a = p.pairs[2 * q], b = p.pairs[2 * q + 1];
  const int src = dir ? b : a, dst = dir ? a : b;
  if (threadIdx.x == 0) {
    inverse3x3_d(p.K + src * 9, Kinv);
    inverse3x3_d(p.R + dst * 9, Rinv);
    for (int e = 0; e < 9; ++e) { Ks[e] = p.K[dst * 9 + e]; Rs[e] = p.R[src * 9 + e]; }
    for (int e = 0; e < 3; ++e) { ts[e] = p.t[src * 3 + e]; tdst[e] = p.t[dst * 3 + e]; }
    base = 0;
  }
  __syncthreads();
  const int H = p.H, W = p.W, max_kp = p.max_kp;
  const int n = min(max(p.kp_count[src], 0), max_kp);
  const int32_t* P = p.kp + (size_t)src * max_kp * 2;
  const float* Dsrc = p.depth + (size_t)src * H * W;
  const float* Ddst = p.depth + (size_t)dst * H * W;
  int* vis = p.vis + ((size_t)q * 2 + dir) * max_kp;
  double* proj = p.proj + (size_t)q * max_kp * 2;
  double* set = (dir ? p.set2 : p.set1) + (size_t)q * max_kp * 2;
  const double nan = __longlong_as_double(0x7ff8000000000000ll);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c0 = 0; c0 < max_kp; c0 += kPosedThreads) {   // slots past n are written too (vis 0, proj NaN)
    const int i = c0 + threadIdx.x;
    bool visible = false;
    int r = 0, c = 0;
    double row = nan, col = nan;
    if (i < n) {
      r = P[2 * i];
      c = P[2 * i + 1];
      if (r >= 0 && r < H && c >= 0 && c < W) {
        const double d = (double)Dsrc[(size_t)r * W + c];
        const double x = (double)c, y = (double)r;
        const double ray0 = dadd(dadd(dmul(Kinv[0], x), dmul(Kinv[1], y)), Kinv[2]);
        const double ray1 = dadd(dadd(dmul(Kinv[3], x), dmul(Kinv[4], y)), Kinv[5]);
        const double ray2 = dadd(dadd(dmul(Kinv[6], x), dmul(Kinv[7], y)), Kinv[8]);
        const double nrm = dnorm3(ray0, ray1, ray2);
        const double X0 = dmul(__ddiv_rn(ray0, nrm), d), X1 = dmul(__ddiv_rn(ray1, nrm), d), X2 = dmul(__ddiv_rn(ray2, nrm), d);
        const double w0 = dsub(dadd(drow(Rs, X0, X1, X2), ts[0]), tdst[0]);
        const double w1 = dsub(dadd(drow(Rs + 3, X0, X1, X2), ts[1]), tdst[1]);
        const double w2 = dsub(dadd(drow(Rs + 6, X0, X1, X2), ts[2]), tdst[2]);
        const double Y0 = drow(Rinv, w0, w1, w2), Y1 = drow(Rinv + 3, w0, w1, w2), Y2 = drow(Rinv + 6, w0, w1, w2);
        const double p0 = drow(Ks, Y0, Y1, Y2), p1 = drow(Ks + 3, Y0, Y1, Y2), p2 = drow(Ks + 6, Y0, Y1, Y2);
        row = __ddiv_rn(p1, p2);
        col = __ddiv_rn(p0, p2);
        if (!isfinite(row) || !isfinite(col)) { row = nan; col = nan; }
        if (isfinite(d) && d > 0.0 && Y2 > 0.0 && row >= 0.0 && row <= (double)(H - 1) && col >= 0.0 && col <= (double)(W - 1)) {
          const int nr = (int)floor(dadd(row, 0.5)), nc = (int)floor(dadd(col, 0.5));
          const double db = (double)Ddst[(size_t)nr * W + nc];
          visible = isfinite(db) && db > 0.0 && fabs(dsub(dnorm3(Y0, Y1, Y2), db)) <= dmul(p.depth_tol, db);
        }
      }
    }
    if (i < max_kp) {
      vis[i] = visible ? 1 : 0;
      if (dir == 0) { proj[2 * i] = row; proj[2 * i + 1] = col; }
    }
    // ordered compaction of the visible points (block-wide exclusive scan of the flags)
    const unsigned ballot = __ballot_sync(0xffffffffu, visible);
    if (lane == 0) warp_n[warp] = __popc(ballot);
    __syncthreads();
    int s = base + __popc(ballot & ((1u << lane) - 1u)), total = 0;
    for (int w = 0; w < kPosedThreads / 32; ++w) {
      s += w < warp ? warp_n[w] : 0;
      total += warp_n[w];
    }
    if (visible) {
      set[2 * s] = dir ? (double)r : row;
      set[2 * s + 1] = dir ? (double)c : col;
    }
    __syncthreads();
    if (threadIdx.x == 0) base += total;
    __syncthreads();
  }
  const int count = base;
  for (int i = count + threadIdx.x; i < max_kp; i += kPosedThreads) { set[2 * i] = nan; set[2 * i + 1] = nan; }
  if (threadIdx.x == 0) p.set_count[2 * q + dir] = count;
}

}  // namespace

extern "C" int spn_select_keypoints(spn_ctx* ctx, const float* d_prob, int B, int H, int W, const double* h_warp, int bound_h,
                                    int bound_w, int emit_warped, int keep_k, double* d_pts, float* d_score, int32_t* d_count,
                                    spn_stream stream) {
  SPN_REQUIRE(ctx && d_prob && d_pts && d_score && d_count, "spn_select_keypoints: null pointer");
  SPN_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0 && keep_k > 0 && keep_k <= kSelCap, "spn_select_keypoints: bad shape / keep_k (<= %d)", kSelCap);
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  SelParams p;
  memset(&p, 0, sizeof(p));
  p.prob = d_prob; p.H = H; p.W = W; p.bound_h = bound_h; p.bound_w = bound_w; p.emit_warped = emit_warped; p.keep_k = keep_k;
  p.pts = d_pts; p.score = d_score; p.count = d_count;
  if (h_warp) {
    int rc = spn_ensure_aux(ctx, (size_t)B * 9 * sizeof(double), s);
    if (rc) return rc;
    SPN_CUDA(cudaMemcpyAsync(ctx->aux, h_warp, (size_t)B * 9 * sizeof(double), cudaMemcpyHostToDevice, s));
    p.warp = (const double*)ctx->aux;
  }
  const size_t dyn = (size_t)kSelCap * sizeof(unsigned long long);
  SPN_CUDA(cudaFuncSetAttribute(select_keypoints_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  select_keypoints_kernel<<<B, kSelThreads, dyn, s>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_repeatability_counts(spn_ctx* ctx, const double* d_pts1, const int32_t* d_n1, const double* d_pts2,
                                        const int32_t* d_n2, int B, int cap, double thresh, int32_t* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_pts1 && d_n1 && d_pts2 && d_n2 && d_out, "spn_repeatability_counts: null pointer");
  SPN_REQUIRE(B > 0 && B <= 65535 && cap > 0, "spn_repeatability_counts: bad shape");
  SpnDeviceGuard guard(ctx->device);
  repeat_count_kernel<<<B, 256, 0, (cudaStream_t)stream>>>(d_pts1, d_n1, d_pts2, d_n2, cap, thresh, d_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_mutual_nn_match(spn_ctx* ctx, const float* d_desc1, const int32_t* d_n1, const float* d_desc2,
                                   const int32_t* d_n2, int B, int cap1, int cap2, int C, int32_t* d_match, float* d_dist,
                                   spn_stream stream) {
  SPN_REQUIRE(ctx && d_desc1 && d_n1 && d_desc2 && d_n2 && d_match && d_dist, "spn_mutual_nn_match: null pointer");
  SPN_REQUIRE(B > 0 && B <= 65535 && cap1 > 0 && cap2 > 0 && C > 0 && C % kKC == 0, "spn_mutual_nn_match: bad shape (C must be a multiple of %d)", kKC);
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n1 = (size_t)B * cap1, n2 = (size_t)B * cap2;
  int rc = spn_ensure_aux(ctx, (n1 + n2) * sizeof(unsigned long long), s);
  if (rc) return rc;
  unsigned long long* bq = (unsigned long long*)ctx->aux;
  unsigned long long* bt = bq + n1;
  fill_u64_kernel<<<(unsigned)((n1 + n2 + 255) / 256), 256, 0, s>>>(bq, n1 + n2, ~0ull);
  SPN_CHECK_LAUNCH(ctx);
  const size_t dyn = kSmemBytes;
  SPN_CUDA(cudaFuncSetAttribute(nn_match_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  MatchParams p;
  p.q = d_desc1; p.t = d_desc2; p.nq = d_n1; p.nt = d_n2; p.qcap = cap1; p.tcap = cap2; p.C = C; p.best = bq;
  nn_match_tc_kernel<<<dim3(spn_cdiv(cap2, kNT), spn_cdiv(cap1, kMT), B), 128, dyn, s>>>(p);   // nearest train row of every query row
  SPN_CHECK_LAUNCH(ctx);
  p.q = d_desc2; p.t = d_desc1; p.nq = d_n2; p.nt = d_n1; p.qcap = cap2; p.tcap = cap1; p.best = bt;
  nn_match_tc_kernel<<<dim3(spn_cdiv(cap1, kNT), spn_cdiv(cap2, kMT), B), 128, dyn, s>>>(p);   // and the other direction
  SPN_CHECK_LAUNCH(ctx);
  cross_check_kernel<<<dim3(spn_cdiv(cap1, 128), B), 128, 0, s>>>(bq, bt, d_n1, d_n2, cap1, cap2, d_match, d_dist);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_posed_reproject(spn_ctx* ctx, const int32_t* d_kp, const int32_t* d_kp_count, int max_kp, const float* d_depth,
                                   const float* d_K, const float* d_R, const float* d_t, int V, int H, int W, int P,
                                   const int32_t* h_pairs, double depth_tol, double* d_proj, int32_t* d_vis, double* d_set1,
                                   double* d_set2, int32_t* d_set_count, spn_stream stream) {
  SPN_REQUIRE(ctx && d_kp && d_kp_count && d_depth && d_K && d_R && d_t, "spn_posed_reproject: null pointer");
  SPN_REQUIRE(V > 0 && H > 0 && W > 0 && H <= 32767 && W <= 32767, "spn_posed_reproject: bad shape V=%d H=%d W=%d (need V > 0, 0 < H, W <= 32767)", V, H, W);
  SPN_REQUIRE(max_kp > 0, "spn_posed_reproject: max_kp must be > 0 (got %d)", max_kp);
  SPN_REQUIRE(P >= 0 && P <= 65535, "spn_posed_reproject: P = %d pairs outside [0, 65535]", P);
  SPN_REQUIRE(isfinite(depth_tol) && depth_tol >= 0.0, "spn_posed_reproject: depth_tol must be finite and >= 0 (got %g)", depth_tol);
  if (P == 0) return SPN_OK;
  SPN_REQUIRE(h_pairs && d_proj && d_vis && d_set1 && d_set2 && d_set_count, "spn_posed_reproject: null pointer (h_pairs / outputs)");
  for (int q = 0; q < P; ++q)
    SPN_REQUIRE(h_pairs[2 * q] >= 0 && h_pairs[2 * q] < V && h_pairs[2 * q + 1] >= 0 && h_pairs[2 * q + 1] < V,
                "spn_posed_reproject: pair %d = (%d, %d) has a view index outside [0, %d)", q, h_pairs[2 * q], h_pairs[2 * q + 1], V);
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t bytes = (size_t)P * 2 * sizeof(int32_t);
  int rc = spn_ensure_aux(ctx, bytes, s);
  if (rc) return rc;
  // pageable source: the call returns once the bytes are staged
  SPN_CUDA(cudaMemcpyAsync(ctx->aux, h_pairs, bytes, cudaMemcpyHostToDevice, s));
  PosedParams p;
  p.kp = d_kp; p.kp_count = d_kp_count; p.depth = d_depth; p.K = d_K; p.R = d_R; p.t = d_t; p.pairs = (const int*)ctx->aux;
  p.H = H; p.W = W; p.max_kp = max_kp; p.depth_tol = depth_tol;
  p.proj = d_proj; p.vis = d_vis; p.set1 = d_set1; p.set2 = d_set2; p.set_count = d_set_count;
  posed_reproject_kernel<<<2 * P, kPosedThreads, 0, s>>>(p);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
