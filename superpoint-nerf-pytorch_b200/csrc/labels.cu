// Train-time label building that shares the hot path's data (SURVEY.md section 8f-4): the detector-loss labels of
// utils/losses.py:13-27 of the reference, one thread per 8x8 cell.
//   labels = argmax_c( cat([2 * pixel_unshuffle(kpts_heatmap, 8), 1]) + noise ),  noise ~ U(0, 0.1)   (random tie break)
//   valid  = prod_c( pixel_unshuffle(valid_mask, 8) )
// With a caller-supplied noise tensor the labels are bit-identical to torch.argmax on the same noise (first maximum
// wins); without one a counter-based generator keyed by (seed, element index) draws the tie-break noise.
#include "spn_common.cuh"

namespace {

__device__ __forceinline__ uint64_t mix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

__global__ void __launch_bounds__(128) detector_labels_kernel(const int32_t* __restrict__ kmap, const int32_t* __restrict__ valid,
                                                              const float* __restrict__ noise, uint64_t seed, int B, int Hc, int Wc,
                                                              int64_t* __restrict__ labels, float* __restrict__ valid_cells) {
  const int cell = blockIdx.x * blockDim.x + threadIdx.x;
  const int n_cells = B * Hc * Wc;
  if (cell >= n_cells) return;
  const int b = cell / (Hc * Wc), r = cell - b * Hc * Wc;
  const int cy = r / Wc, cx = r - cy * Wc;
  const int W = Wc * 8;
  const size_t base = ((size_t)b * Hc * 8 + cy * 8) * W + cx * 8;
  float best = -1.f;
  int best_c = 0;
  int ok = 1;
  for (int c = 0; c < 65; ++c) {
    float v = 1.0f;   // dustbin
    if (c < 64) {
      const size_t o = base + (size_t)(c >> 3) * W + (c & 7);
      v = 2.0f * (float)kmap[o];
      if (valid) ok &= valid[o] != 0;
    }
    float nz;
    if (noise) {
      nz = noise[((size_t)b * 65 + c) * Hc * Wc + r];
    } else {
      const uint64_t h = mix64(mix64(seed) ^ (((uint64_t)cell * 65 + c) + 1));
      nz = 0.1f * (float)((h >> 40) * (1.0 / 16777216.0));
    }
    v += nz;
    if (v > best) { best = v; best_c = c; }
  }
  labels[cell] = best_c;
  valid_cells[cell] = (float)ok;
}

}  // namespace

extern "C" int spn_detector_labels(spn_ctx* ctx, const int32_t* d_kpts_heatmap, const int32_t* d_valid_mask, const float* d_noise,
                                   uint64_t seed, int B, int H, int W, int64_t* d_labels, float* d_valid_cells, spn_stream stream) {
  SPN_REQUIRE(ctx && d_kpts_heatmap && d_labels && d_valid_cells, "spn_detector_labels: null pointer");
  SPN_REQUIRE(B > 0 && H > 0 && W > 0 && H % 8 == 0 && W % 8 == 0, "spn_detector_labels: H, W must be positive multiples of 8");
  SpnDeviceGuard guard(ctx->device);
  const int cells = B * (H / 8) * (W / 8);
  detector_labels_kernel<<<spn_cdiv(cells, 128), 128, 0, (cudaStream_t)stream>>>(d_kpts_heatmap, d_valid_mask, d_noise, seed, B, H / 8,
                                                                                 W / 8, d_labels, d_valid_cells);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// ExportNeRFDetections.step splat (engine_solvers/export.py:271-283 of the reference): for every (destination point u_i,
// source point w_i) pair IN ORDER, copy the 3x3 patch of the source heatmap around w_i onto the 3x3 patch around u_i
// (a single pixel when either point is within one pixel of the border); later pairs overwrite earlier ones.  The
// sequential "last writer wins" rule is reproduced in parallel with an owner map: pass 1 records, per destination
// pixel, the highest pair index that covers it (atomicMax), pass 2 gathers the value that pair would have written.
namespace {

__device__ __forceinline__ bool nerf_border(int u0, int u1, int w0, int w1, int H, int W) {
  return u0 <= 1 || u1 <= 1 || u0 >= H - 1 || u1 >= W - 1 || w0 <= 1 || w1 <= 1 || w0 >= H - 1 || w1 >= W - 1;
}

__global__ void nerf_owner_kernel(const float* __restrict__ dst, const int32_t* __restrict__ src, int n, int H, int W,
                                  unsigned* __restrict__ owner) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int u0 = (int)dst[2 * i], u1 = (int)dst[2 * i + 1];   // python int(): truncation toward zero
  const int w0 = src[2 * i], w1 = src[2 * i + 1];
  if (u0 < 0 || u0 >= H || u1 < 0 || u1 >= W) return;
  if (nerf_border(u0, u1, w0, w1, H, W)) {
    atomicMax(&owner[u0 * W + u1], (unsigned)i + 1u);
  } else {
    for (int dy = -1; dy <= 1; ++dy)
      for (int dx = -1; dx <= 1; ++dx) atomicMax(&owner[(u0 + dy) * W + u1 + dx], (unsigned)i + 1u);
  }
}

__global__ void nerf_gather_kernel(const float* __restrict__ prob, const float* __restrict__ dst, const int32_t* __restrict__ src, int H,
                                   int W, const unsigned* __restrict__ owner, float* __restrict__ out) {
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= H * W) return;
  const unsigned o = owner[p];
  float v = 0.f;
  if (o) {
    const int i = (int)o - 1;
    const int u0 = (int)dst[2 * i], u1 = (int)dst[2 * i + 1];
    const int w0 = src[2 * i], w1 = src[2 * i + 1];
    const int y = p / W, x = p - y * W;
    v = prob[(w0 + (y - u0)) * W + w1 + (x - u1)];   // (y - u0, x - u1) is (0, 0) in the single-pixel case
  }
  out[p] = v;
}

}  // namespace

extern "C" int spn_nerf_splat(spn_ctx* ctx, const float* d_prob_src, const float* d_dst_pts, const int32_t* d_src_pts, int n_pairs, int H,
                              int W, float* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_prob_src && d_out && (n_pairs == 0 || (d_dst_pts && d_src_pts)), "spn_nerf_splat: null pointer");
  SPN_REQUIRE(n_pairs >= 0 && H > 2 && W > 2, "spn_nerf_splat: bad shape");
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = spn_ensure_aux(ctx, (size_t)H * W * sizeof(unsigned), s);
  if (rc) return rc;
  unsigned* owner = (unsigned*)ctx->aux;
  SPN_CUDA(cudaMemsetAsync(owner, 0, (size_t)H * W * sizeof(unsigned), s));
  if (n_pairs) {
    nerf_owner_kernel<<<spn_cdiv(n_pairs, 128), 128, 0, s>>>(d_dst_pts, d_src_pts, n_pairs, H, W, owner);
    SPN_CHECK_LAUNCH(ctx);
  }
  nerf_gather_kernel<<<spn_cdiv(H * W, 256), 256, 0, s>>>(d_prob_src, d_dst_pts, d_src_pts, H, W, owner, d_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// spn_nerf_fuse (include/spn_nerf.h): every (target j, source k) pair of a batch in two kernels.
//   nerf_reproject_kernel  one CTA per pair: the keypoints of k through warp_points_NeRF's depth rule and fp32 chain,
//                          filter_points, the survivors compacted IN ORDER (block scan) into the scratch buffer as
//                          (destination, source) records - survivor s is paired with the s-th original keypoint.
//   nerf_fuse_kernel       one CTA per (32x64 output tile, target): walks the target's pairs in summation order; per
//                          pair it rebuilds the tile's owner map in shared memory (atomicMax on the record index, the
//                          rule of nerf_owner_kernel) and every pixel adds its owner's source value to a register
//                          accumulator.  No float atomics, no per-pair maps in global memory, deterministic.
#include "../../include/spn_nerf.h"

namespace {

constexpr int kFuseTileH = 32, kFuseTileW = 64, kFuseThreads = 256, kReprojThreads = 256;
constexpr unsigned kRecSingle = 0x80000000u;   // record flag: single-pixel copy
constexpr unsigned kRecSkip = 0xFFFFFFFFu;     // record whose paired source keypoint lies outside the image

// one row of a 3x3 fp32 product (cuBLAS-style FMA chain)
__device__ __forceinline__ float dot3(const float* m, float a, float b, float c) {
  return fmaf(m[2], c, fmaf(m[1], b, __fmul_rn(m[0], a)));
}

// torch.linalg.inv of a 3x3: adjugate in fp64, rounded once to fp32
__device__ void inverse3x3(const float* m, float* o) {
  const double a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], h = m[7], i = m[8];
  const double c00 = e * i - f * h, c01 = f * g - d * i, c02 = d * h - e * g;
  const double det = a * c00 + b * c01 + c * c02;
  o[0] = (float)(c00 / det); o[1] = (float)((c * h - b * i) / det); o[2] = (float)((b * f - c * e) / det);
  o[3] = (float)(c01 / det); o[4] = (float)((a * i - c * g) / det); o[5] = (float)((c * d - a * f) / det);
  o[6] = (float)(c02 / det); o[7] = (float)((b * g - a * h) / det); o[8] = (float)((a * e - b * d) / det);
}

__global__ void __launch_bounds__(kReprojThreads) nerf_reproject_kernel(
    const int32_t* __restrict__ kp, const int32_t* __restrict__ kp_count, const float* __restrict__ depth, const float* __restrict__ Kmat,
    const float* __restrict__ Rmat, const float* __restrict__ Tvec, const int* __restrict__ pair_src, const int* __restrict__ pair_view,
    int H, int W, int max_kp, int* __restrict__ surv_count, uint2* __restrict__ surv) {
  __shared__ float Kj[9], Kinv[9], Rk[9], tk[3], Rjinv[9], Rjt[3];
  __shared__ int warp_n[kReprojThreads / 32];
  __shared__ int base;
  const int q = blockIdx.x;
  const int k = pair_src[q], j = pair_view[q];
  if (threadIdx.x == 0) {
    for (int e = 0; e < 9; ++e) { Kj[e] = Kmat[j * 9 + e]; Rk[e] = Rmat[k * 9 + e]; }
    for (int e = 0; e < 3; ++e) tk[e] = Tvec[k * 3 + e];
    inverse3x3(Kj, Kinv);
    inverse3x3(Rmat + j * 9, Rjinv);
    const float* tj = Tvec + j * 3;
    for (int r = 0; r < 3; ++r) Rjt[r] = dot3(Rjinv + 3 * r, tj[0], tj[1], tj[2]);   // inv(R_j) @ t_j
    base = 0;
  }
  __syncthreads();
  const int n = min(max(kp_count[k], 0), max_kp);
  const int32_t* P = kp + (size_t)k * max_kp * 2;
  const float* D = depth + (size_t)k * H * W;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int c0 = 0; c0 < n; c0 += kReprojThreads) {
    const int i = c0 + threadIdx.x;
    bool keep = false;
    int u0 = 0, u1 = 0;
    if (i < n) {
      const int r = P[2 * i], c = P[2 * i + 1];
      if (r >= 0 && r < H && c >= 0 && c < W) {
        // depth rule of warp_points_NeRF (5x5 min / max pooling; max_pool2d propagates NaN)
        float dv = D[r * W + c];
        if (!(r <= 2 || c <= 2 || r >= H - 2 || c >= W - 2)) {
          float mn = dv, mx = dv;
          bool nan = false;
          for (int dy = -2; dy <= 2; ++dy)
            for (int dx = -2; dx <= 2; ++dx) {
              const float v = D[(r + dy) * W + c + dx];
              nan |= v != v;
              mn = fminf(mn, v);
              mx = fmaxf(mx, v);
            }
          if (nan) dv = __int_as_float(0x7fc00000);
          else if (!(__fsub_rn(mx, mn) < 0.03f)) dv = mn;
        }
        const float x = (float)c, y = (float)r;
        float a0 = dot3(Kinv, x, y, 1.f), a1 = dot3(Kinv + 3, x, y, 1.f), a2 = dot3(Kinv + 6, x, y, 1.f);
        const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(a0, a0), __fmul_rn(a1, a1)), __fmul_rn(a2, a2)));
        a0 = __fmul_rn(__fdiv_rn(a0, nrm), dv);
        a1 = __fmul_rn(__fdiv_rn(a1, nrm), dv);
        a2 = __fmul_rn(__fdiv_rn(a2, nrm), dv);
        const float b0 = __fadd_rn(dot3(Rk, a0, a1, a2), tk[0]), b1 = __fadd_rn(dot3(Rk + 3, a0, a1, a2), tk[1]),
                    b2 = __fadd_rn(dot3(Rk + 6, a0, a1, a2), tk[2]);
        const float e0 = __fsub_rn(dot3(Rjinv, b0, b1, b2), Rjt[0]), e1 = __fsub_rn(dot3(Rjinv + 3, b0, b1, b2), Rjt[1]),
                    e2 = __fsub_rn(dot3(Rjinv + 6, b0, b1, b2), Rjt[2]);
        const float p0 = dot3(Kj, e0, e1, e2), p1 = dot3(Kj + 3, e0, e1, e2), p2 = dot3(Kj + 6, e0, e1, e2);
        const float row = __fdiv_rn(p1, p2), col = __fdiv_rn(p0, p2);
        if (row >= 0.f && row < (float)(H - 1) && col >= 0.f && col < (float)(W - 1)) {   // filter_points
          keep = true;
          u0 = (int)row;   // python int(): truncation
          u1 = (int)col;
        }
      }
    }
    const unsigned ballot = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_n[warp] = __popc(ballot);
    __syncthreads();
    int s = base + __popc(ballot & ((1u << lane) - 1u)), total = 0;
    for (int w = 0; w < kReprojThreads / 32; ++w) {
      s += w < warp ? warp_n[w] : 0;
      total += warp_n[w];
    }
    if (keep) {
      const int w0 = P[2 * s], w1 = P[2 * s + 1];   // survivor s goes with the s-th original keypoint (export.py:269-271)
      uint2 rec;
      rec.x = ((unsigned)u0 << 16) | (unsigned)u1;
      if (w0 < 0 || w0 >= H || w1 < 0 || w1 >= W) {
        rec.y = kRecSkip;
      } else {
        rec.y = ((unsigned)w0 << 16) | (unsigned)w1 | (nerf_border(u0, u1, w0, w1, H, W) ? kRecSingle : 0u);
      }
      surv[(size_t)q * max_kp + s] = rec;
    }
    __syncthreads();
    if (threadIdx.x == 0) base += total;
    __syncthreads();
  }
  if (threadIdx.x == 0) surv_count[q] = base;
}

__global__ void __launch_bounds__(kFuseThreads) nerf_fuse_kernel(const float* __restrict__ prob, const int* __restrict__ tgt_view,
                                                                 const int* __restrict__ offsets, const int* __restrict__ pair_src,
                                                                 const int* __restrict__ surv_count, const uint2* __restrict__ surv,
                                                                 int H, int W, int max_kp, int tiles_x, float* __restrict__ out) {
  constexpr int kPix = kFuseTileH * kFuseTileW, kPer = kPix / kFuseThreads;
  __shared__ unsigned owner[kPix];
  const int t = blockIdx.y;
  const int ty0 = (blockIdx.x / tiles_x) * kFuseTileH, tx0 = (blockIdx.x % tiles_x) * kFuseTileW;
  const float* Pj = prob + (size_t)tgt_view[t] * H * W;
  float acc[kPer];
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    const int p = threadIdx.x + e * kFuseThreads;
    const int y = ty0 + p / kFuseTileW, x = tx0 + p % kFuseTileW;
    acc[e] = (y < H && x < W) ? Pj[y * W + x] : 0.f;
    owner[p] = 0u;
  }
  __syncthreads();
  const int q0 = offsets[t], q1 = offsets[t + 1];
  for (int q = q0; q < q1; ++q) {
    const int n = surv_count[q];
    const uint2* S = surv + (size_t)q * max_kp;
    for (int i = threadIdx.x; i < n; i += kFuseThreads) {
      const uint2 r = S[i];
      if (r.y == kRecSkip) continue;
      const int ly = (int)(r.x >> 16) - ty0, lx = (int)(r.x & 0xffffu) - tx0;
      if (r.y & kRecSingle) {
        if ((unsigned)ly < (unsigned)kFuseTileH && (unsigned)lx < (unsigned)kFuseTileW) atomicMax(&owner[ly * kFuseTileW + lx], (unsigned)i + 1u);
      } else if (ly >= -1 && ly <= kFuseTileH && lx >= -1 && lx <= kFuseTileW) {
        for (int dy = -1; dy <= 1; ++dy)
          for (int dx = -1; dx <= 1; ++dx) {
            const int yy = ly + dy, xx = lx + dx;
            if ((unsigned)yy < (unsigned)kFuseTileH && (unsigned)xx < (unsigned)kFuseTileW) atomicMax(&owner[yy * kFuseTileW + xx], (unsigned)i + 1u);
          }
      }
    }
    __syncthreads();
    const float* Pk = prob + (size_t)pair_src[q] * H * W;
#pragma unroll
    for (int e = 0; e < kPer; ++e) {
      const int p = threadIdx.x + e * kFuseThreads;
      const unsigned o = owner[p];
      if (o) {
        owner[p] = 0u;   // cleared for the next pair by the thread that reads it
        const uint2 r = S[o - 1];
        const int y = ty0 + p / kFuseTileW, x = tx0 + p % kFuseTileW;
        const int u0 = (int)(r.x >> 16), u1 = (int)(r.x & 0xffffu);
        const int w0 = (int)((r.y >> 16) & 0x7fffu), w1 = (int)(r.y & 0xffffu);
        acc[e] += Pk[(w0 + (y - u0)) * W + w1 + (x - u1)];   // (y - u0, x - u1) is (0, 0) for a single-pixel copy
      }
    }
    __syncthreads();
  }
  const float inv = 1.0f / (float)(1 + q1 - q0);   // torch: tensor / python float = tensor * (1 / float)
  float* O = out + (size_t)t * H * W;
#pragma unroll
  for (int e = 0; e < kPer; ++e) {
    const int p = threadIdx.x + e * kFuseThreads;
    const int y = ty0 + p / kFuseTileW, x = tx0 + p % kFuseTileW;
    if (y < H && x < W) O[y * W + x] = __fmul_rn(acc[e], inv);
  }
}

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

}  // namespace

extern "C" int spn_nerf_fuse(spn_ctx* ctx, const float* d_prob, const int32_t* d_kp, const int32_t* d_kp_count, int max_kp,
                             const float* d_depth, const float* d_K, const float* d_R, const float* d_t, int V, int H, int W,
                             int n_targets, const int32_t* h_targets, const int32_t* h_pair_offsets, const int32_t* h_pair_src,
                             float* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_prob && d_kp && d_kp_count && d_depth && d_K && d_R && d_t && h_pair_offsets, "spn_nerf_fuse: null pointer");
  SPN_REQUIRE(V > 0 && H > 2 && W > 2 && H <= 32767 && W <= 32767, "spn_nerf_fuse: bad shape V=%d H=%d W=%d (need V > 0, 2 < H, W <= 32767)", V, H, W);
  SPN_REQUIRE(max_kp > 0, "spn_nerf_fuse: max_kp must be > 0 (got %d)", max_kp);
  SPN_REQUIRE(n_targets >= 0 && n_targets <= 65535, "spn_nerf_fuse: n_targets %d outside [0, 65535]", n_targets);
  SPN_REQUIRE(n_targets == 0 || (h_targets && d_out), "spn_nerf_fuse: null pointer (h_targets / d_out)");   // no targets: empty output
  SPN_REQUIRE(h_pair_offsets[0] == 0, "spn_nerf_fuse: h_pair_offsets[0] must be 0 (got %d)", h_pair_offsets[0]);
  for (int t = 0; t < n_targets; ++t) {
    SPN_REQUIRE(h_targets[t] >= 0 && h_targets[t] < V, "spn_nerf_fuse: target %d has view index %d outside [0, %d)", t, h_targets[t], V);
    SPN_REQUIRE(h_pair_offsets[t + 1] >= h_pair_offsets[t], "spn_nerf_fuse: h_pair_offsets not monotone at target %d (%d -> %d)", t,
                h_pair_offsets[t], h_pair_offsets[t + 1]);
  }
  const int n_pairs = h_pair_offsets[n_targets];
  SPN_REQUIRE(n_pairs == 0 || h_pair_src, "spn_nerf_fuse: null pointer (h_pair_src)");
  for (int q = 0; q < n_pairs; ++q)
    SPN_REQUIRE(h_pair_src[q] >= 0 && h_pair_src[q] < V, "spn_nerf_fuse: pair %d has source view index %d outside [0, %d)", q, h_pair_src[q], V);
  if (n_targets == 0) return SPN_OK;
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  // scratch: [pair_src | pair_view | tgt_view | offsets] (int32, uploaded) | surv_count [n_pairs] | surv [n_pairs][max_kp]
  std::vector<int32_t> tab(2 * (size_t)n_pairs + n_targets + n_targets + 1);
  int32_t* p_src = tab.data();
  int32_t* p_view = p_src + n_pairs;
  int32_t* p_tgt = p_view + n_pairs;
  int32_t* p_off = p_tgt + n_targets;
  for (int t = 0; t < n_targets; ++t) {
    p_tgt[t] = h_targets[t];
    for (int q = h_pair_offsets[t]; q < h_pair_offsets[t + 1]; ++q) { p_src[q] = h_pair_src[q]; p_view[q] = h_targets[t]; }
  }
  for (int t = 0; t <= n_targets; ++t) p_off[t] = h_pair_offsets[t];
  const size_t tab_bytes = align256(tab.size() * sizeof(int32_t));
  const size_t cnt_bytes = align256((size_t)n_pairs * sizeof(int));
  const size_t surv_bytes = (size_t)n_pairs * max_kp * sizeof(uint2);
  int rc = spn_ensure_aux(ctx, tab_bytes + cnt_bytes + surv_bytes, s);
  if (rc) return rc;
  char* base = ctx->aux;
  const int* d_tab = (const int*)base;
  int* d_cnt = (int*)(base + tab_bytes);
  uint2* d_surv = (uint2*)(base + tab_bytes + cnt_bytes);
  // pageable source: the call returns once the bytes are staged, so the vector may go out of scope
  SPN_CUDA(cudaMemcpyAsync(base, tab.data(), tab.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
  if (n_pairs) {
    nerf_reproject_kernel<<<n_pairs, kReprojThreads, 0, s>>>(d_kp, d_kp_count, d_depth, d_K, d_R, d_t, d_tab, d_tab + n_pairs, H, W,
                                                             max_kp, d_cnt, d_surv);
    SPN_CHECK_LAUNCH(ctx);
  }
  const int tiles_x = spn_cdiv(W, kFuseTileW), tiles_y = spn_cdiv(H, kFuseTileH);
  nerf_fuse_kernel<<<dim3(tiles_x * tiles_y, n_targets), kFuseThreads, 0, s>>>(d_prob, d_tab + 2 * n_pairs, d_tab + 2 * n_pairs + n_targets,
                                                                               d_tab, d_cnt, d_surv, H, W, max_kp, tiles_x, d_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
