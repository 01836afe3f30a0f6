// Homography kernels: batched bilinear warp + eroded validity mask, the fused inverse-warp / count-normalised
// aggregation over homographies, the device homography sampler and a batched 3x3 inverse.
//
// Reference semantics (superpoint/superpoint/engine_solvers/export.py:42-114 and kornia 0.7.0 as restated in
// oracle/kornia_shim.py): warp_perspective(src, M)(p) = interp(src, M^-1 p), align_corners=True, zeros padding,
// nearest = round-half-even.  Source coordinates are evaluated with kornia's own normalised-space fp32 chain
// (spn_geom.cuh: kornia_src) from the matrices Ainv = torch.inverse(normalize_homography(M)), so validity masks,
// counts and bilinear samples are bit-identical to the reference's CPU run when Ainv is the reference's (the Python
// binding computes it with the same torch calls); erosion = min over the elliptical structuring element
// cv2.getStructuringElement(MORPH_ELLIPSE, (2m,2m)) with origin (m,m) and a geodesic border (pixels outside the
// image never erode).
//
// Both kernels are HBM/L2-bandwidth bound (a few FLOPs per byte): they are tiled 32x8 pixels per CTA with the
// raw validity bits of the tile + erosion halo staged in shared memory, coalesced row-major global accesses, and
// grids of (tiles x slots) CTAs = many multiples of the 148 SMs.
#include <math.h>

#include "spn_common.cuh"
#include "spn_geom.cuh"

namespace {

using namespace spngeom;

constexpr int kTileW = 32, kTileH = 8, kMaxKs = 16;
constexpr int kRawH = kTileH + kMaxKs - 1, kRawW = kTileW + kMaxKs;  // 23 x 48

struct ErodeK {
  int ks;              // structuring element is ks x ks
  int org;             // origin = ks/2
  uint32_t rw_magic;   // ceil(2^32 / (kTileW + ks - 1)): row of a linearised halo index by one multiply-high
  uint32_t rows[kMaxKs];
};

// cv2.getStructuringElement(MORPH_ELLIPSE, (ks,ks)) restated (export.py:59).
ErodeK make_ellipse(int margin) {
  ErodeK e;
  memset(&e, 0, sizeof(e));
  if (margin == 0) {  // no erosion (compute_valid_mask with erosion = 0): the 1x1 structuring element
    e.ks = 1;
    e.org = 0;
    e.rw_magic = (uint32_t)(((1ull << 32) + kTileW - 1) / kTileW);
    e.rows[0] = 1u;
    return e;
  }
  const int ks = 2 * margin;
  e.ks = ks;
  e.org = ks / 2;
  e.rw_magic = (uint32_t)(((1ull << 32) + (kTileW + ks - 1) - 1) / (kTileW + ks - 1));
  const int r = ks / 2, c = ks / 2;
  const double inv_r2 = r ? 1.0 / ((double)r * r) : 0.0;
  for (int i = 0; i < ks; ++i) {
    const int dy = i - r;
    int j1 = 0, j2 = 0;
    if (abs(dy) <= r) {
      const int dx = (int)lrint(c * sqrt((r * r - dy * dy) * inv_r2));
      j1 = max(c - dx, 0);
      j2 = min(c + dx + 1, ks);
    }
    for (int j = j1; j < j2; ++j) e.rows[i] |= 1u << j;
  }
  return e;
}

// ---- tile classification -----------------------------------------------------------------------------------
// The set of pixels p whose source coordinate M p satisfies a bound (sx >= a, sx <= b, ...) is a half-plane in p as
// long as the homogeneous z stays positive, so for a rectangle of pixels it suffices to test its four corners:
//   all four corners inside the source image (with a safety margin)  -> every pixel of the rectangle is valid,
//   all four corners beyond the same source edge (with a margin)     -> every pixel is invalid and samples to zero,
//   all four corners at least one pixel inside the source image      -> additionally every bilinear tap is in bounds
//                                                                       ("deep": the aggregate's unchecked fast path).
// Only tiles cut by the border of the warped quad need the per-pixel validity bits and the erosion.
enum { kTileMixed = 0, kTileInside = 1, kTileOutside = 2, kTileDeep = 3 };

__device__ __forceinline__ int classify_tile(const float* a, const KGrid& g, const ErodeK& ek, int tx0, int ty0, int H, int W,
                                             bool want_deep = false) {
  // halo rectangle clipped to the image (out-of-image neighbours never erode: geodesic border)
  const int xa = max(tx0 - ek.org, 0), xb = min(tx0 + kTileW - 1 + (ek.ks - ek.org - 1), W - 1);
  const int ya = max(ty0 - ek.org, 0), yb = min(ty0 + kTileH - 1 + (ek.ks - ek.org - 1), H - 1);
  const float mg = 1e-2f;
  bool zok = true, in = true, deep = true, l = true, r = true, t = true, b = true;
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const float xn = __ldg(&g.xs[(c & 1) ? xb : xa]), yn = __ldg(&g.ys[(c & 2) ? yb : ya]);
    const float z = fmaf(a[6], xn, fmaf(a[7], yn, a[8]));
    float sx, sy;
    kornia_src(a, xn, yn, g.hw, g.hh, sx, sy);
    zok = zok && z > 1e-3f;
    in = in && sx >= -0.5f + mg && sx <= (float)W - 0.5f - mg && sy >= -0.5f + mg && sy <= (float)H - 0.5f - mg;
    deep = deep && sx >= mg && sx <= (float)W - 1.0f - mg && sy >= mg && sy <= (float)H - 1.0f - mg;
    l = l && sx < -1.0f - mg;
    r = r && sx > (float)W + mg;
    t = t && sy < -1.0f - mg;
    b = b && sy > (float)H + mg;
  }
  if (!zok) return kTileMixed;
  if (in) return (deep && want_deep) ? kTileDeep : kTileInside;
  if (l || r || t || b) return kTileOutside;
  return kTileMixed;
}

// Raw (un-eroded) validity bits of the tile + halo, linearised row-major (rw = kTileW + ks - 1 columns), one ballot
// per 32 positions; positions outside the image count as valid (geodesic border).
constexpr int kRawWords = (kRawH * kRawW + 31) / 32 + 1;

__device__ __forceinline__ void fill_raw_bits(uint32_t* bits, const float* a, const KGrid& g, const ErodeK& ek, int tx0,
                                              int ty0, int H, int W) {
  const int rh = kTileH + ek.ks - 1, rw = kTileW + ek.ks - 1;
  const int n = rh * rw;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  for (int base = warp * 32; base < n + 32; base += nwarps * 32) {  // + 32: one zero-padded word past the end
    const int i = base + lane;
    int v = 0;
    if (i < n) {
      const int ry = (int)__umulhi((unsigned)i, ek.rw_magic), rx = i - ry * rw;  // i < 2^11: exact
      const int y = ty0 + ry - ek.org, x = tx0 + rx - ek.org;
      v = 1;
      if (x >= 0 && x < W && y >= 0 && y < H) {
        float sx, sy;
        kornia_src(a, __ldg(&g.xs[x]), __ldg(&g.ys[y]), g.hw, g.hh, sx, sy);
        v = inside_nearest(sx, sy, H, W);
      }
    }
    const unsigned b = __ballot_sync(0xffffffffu, v);
    if (lane == 0) bits[base >> 5] = b;
  }
}

// `rows` = the structuring element's row masks in shared memory (a kernel parameter indexed by a loop counter would
// be spilled to local memory).
__device__ __forceinline__ int eroded_bits(const uint32_t* bits, const uint32_t* rows, int ks, int tx, int ty) {
  const int rw = kTileW + ks - 1;
  int ok = 1;
  int o = ty * rw + tx;
  for (int i = 0; i < ks; ++i, o += rw) {
    const uint32_t lo = bits[o >> 5], hi = bits[(o >> 5) + 1];
    const uint32_t w = __funnelshift_r(lo, hi, o & 31);
    const uint32_t rm = rows[i];
    ok &= ((w & rm) == rm);
  }
  return ok;
}

// One block per (row of tiles, slot).  The first threads classify the row's tiles (one thread per tile, four corner
// projections each); the block then walks the tiles: uniform ones are a plain store, tiles cut by the warped quad's
// border go through the validity bits + erosion (bit buffers double buffered: one barrier per mixed tile).
constexpr int kMaxRowTiles = 256;

__global__ void __launch_bounds__(256)
warp_batch_kernel(const float* __restrict__ images, const float* __restrict__ ainv, KGrid g, int n_h, int H, int W,
                  int tiles_x, ErodeK ek, float* __restrict__ warped, uint8_t* __restrict__ mask) {
  __shared__ uint32_t bits[2][kRawWords];
  __shared__ float m[9];
  __shared__ uint32_t rows_s[kMaxKs];
  __shared__ uint8_t cls_s[kMaxRowTiles];
  const int slot = blockIdx.y;
  const int img = slot / (n_h + 1), j = slot - img * (n_h + 1);
  const int ty0 = blockIdx.x * kTileH;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int y = ty0 + ty;
  const float* src = images + (size_t)img * H * W;
  const size_t orow = ((size_t)slot * H + y) * W;
  // mask-only calls (the fused encoder warps on the fly): uniform tiles are written as 16-byte chunks of the 8 image
  // rows of this block (one contiguous span), only tiles cut by the quad border take the per-pixel path below
  const bool vec = warped == nullptr && (W & 15) == 0;
  const int chunks_per_row = W >> 4, block_rows = min(kTileH, H - ty0);
  if (j == 0) {  // identity forward (export.py:93): the image itself, no mask
    if (vec) {
      for (int c = threadIdx.x; c < block_rows * chunks_per_row; c += blockDim.x)
        reinterpret_cast<uint4*>(mask + ((size_t)slot * H + ty0) * W)[c] = make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u);
      return;
    }
    if (y < H)
      for (int x = tx; x < W; x += 32) {
        if (warped) warped[orow + x] = __ldg(&src[(size_t)y * W + x]);
        mask[orow + x] = 1;
      }
    return;
  }
  if (threadIdx.x < 9) m[threadIdx.x] = __ldg(&ainv[((size_t)img * n_h + (j - 1)) * 9 + threadIdx.x]);
  if (threadIdx.x >= 32 && threadIdx.x < 32 + kMaxKs) rows_s[threadIdx.x - 32] = ek.rows[threadIdx.x - 32];
  __syncthreads();
  for (int t = threadIdx.x; t < tiles_x; t += blockDim.x) cls_s[t] = (uint8_t)classify_tile(m, g, ek, t * kTileW, ty0, H, W);
  const float yn = y < H ? __ldg(&g.ys[y]) : 0.f;
  __syncthreads();
  if (vec)
    for (int c = threadIdx.x; c < block_rows * chunks_per_row; c += blockDim.x) {
      const int r = c / chunks_per_row, xc = c - r * chunks_per_row;
      const int cls = cls_s[xc >> 1];  // a 16-pixel chunk lies inside one 32-pixel tile
      if (cls == kTileMixed) continue;
      const uint32_t v = cls == kTileOutside ? 0u : 0x01010101u;
      reinterpret_cast<uint4*>(mask + ((size_t)slot * H + ty0) * W)[c] = make_uint4(v, v, v, v);
    }
  int nmixed = 0;
  for (int t = 0; t < tiles_x; ++t) {
    const int cls = cls_s[t];  // block-uniform
    if (vec && cls != kTileMixed) continue;
    const int tx0 = t * kTileW, x = tx0 + tx;
    const bool in_img = x < W && y < H;
    if (cls == kTileOutside) {
      if (in_img) {
        if (warped) warped[orow + x] = 0.f;
        mask[orow + x] = 0;
      }
      continue;
    }
    int mk = 1;
    if (cls == kTileMixed) {
      uint32_t* bb = bits[nmixed & 1];
      ++nmixed;
      fill_raw_bits(bb, m, g, ek, tx0, ty0, H, W);
      __syncthreads();
      mk = eroded_bits(bb, rows_s, ek.ks, tx, ty);
    }
    if (in_img) {
      if (warped) {  // null: mask only (the fused encoder warps on the fly)
        float sx, sy;
        kornia_src(m, __ldg(&g.xs[x]), yn, g.hw, g.hh, sx, sy);
        warped[orow + x] = bilinear_zero_exact(src, sx, sy, H, W);
      }
      mask[orow + x] = (uint8_t)mk;
    }
  }
}

struct DeepTaps {
  float v00, v01, v10, v11, ax, ay;
};

// Issue the four loads of one bilinear sample whose taps are all inside the image (tile class "deep").
__device__ __forceinline__ DeepTaps deep_taps(const float* __restrict__ pimg, const float4* __restrict__ hs4,
                                              const float* __restrict__ hs, int j, int hw, int W, float xn, float yn,
                                              float ghw, float ghh) {
  const float4 r0 = hs4[j * 3], r1 = hs4[j * 3 + 1];
  const float m8 = hs[j * 12 + 8];
  // kornia_src on the rows held in registers (tile class "deep" guarantees z > 1e-3: the |z| > 1e-8 select is moot)
  const float qx = __fadd_rn(fmaf(r0.y, yn, __fmul_rn(r0.x, xn)), r0.z);
  const float qy = __fadd_rn(fmaf(r1.x, yn, __fmul_rn(r0.w, xn)), r1.y);
  const float qz = __fadd_rn(fmaf(r1.w, yn, __fmul_rn(r1.z, xn)), m8);
  const float sc = rcp_normal(__fadd_rn(qz, 1e-8f));
  const float sx = __fmul_rn(__fadd_rn(__fmul_rn(sc, qx), 1.0f), ghw), sy = __fmul_rn(__fadd_rn(__fmul_rn(sc, qy), 1.0f), ghh);
  const float flx = floorf(sx), fly = floorf(sy);
  const float* p = pimg + ((j + 1) * hw + (int)fly * W + (int)flx);
  DeepTaps t;
  t.v00 = __ldg(p);
  t.v01 = __ldg(p + 1);
  t.v10 = __ldg(p + W);
  t.v11 = __ldg(p + W + 1);
  t.ax = __fsub_rn(sx, flx);
  t.ay = __fsub_rn(sy, fly);
  return t;
}

// ATen's CPU bilinear arithmetic (spn_geom.cuh: bilinear_combine) on taps already in registers
__device__ __forceinline__ float deep_value(const DeepTaps& t) {
  const float e = __fsub_rn(1.0f, t.ax), s = __fsub_rn(1.0f, t.ay);
  return fmaf(t.v11, __fmul_rn(t.ay, t.ax),
              fmaf(t.v10, __fmul_rn(t.ay, e), fmaf(t.v01, __fmul_rn(s, t.ax), __fmul_rn(t.v00, __fmul_rn(s, e)))));
}

// One block per 32 x 8 output tile of one image.  The homographies are first classified for this tile; the "deep"
// ones (most of them: whole tile valid, all taps in bounds) run as a barrier-free loop with two samples in flight per
// thread; the tiles cut by a warped border go through the validity bits + erosion.
__global__ void __launch_bounds__(256, 4)
ha_aggregate_kernel(const float* __restrict__ probs, const float* __restrict__ hmat, KGrid g, int n_h, int H, int W,
                    int tiles_x, ErodeK ek, int agg_max, float* __restrict__ out) {
  extern __shared__ float4 hs4[];  // n_h homographies padded to 12 floats, then three byte arrays of n_h entries
  __shared__ uint32_t bits[2][kRawWords];
  __shared__ uint32_t rows_s[kMaxKs];
  __shared__ int n_list[2];
  float* hs = reinterpret_cast<float*>(hs4);
  uint8_t* cls_s = reinterpret_cast<uint8_t*>(hs + n_h * 12);
  uint8_t* deep_s = cls_s + ((n_h + 15) & ~15);
  uint8_t* rest_s = deep_s + ((n_h + 15) & ~15);
  const int img = blockIdx.y;
  const int tx0 = (blockIdx.x % tiles_x) * kTileW, ty0 = (blockIdx.x / tiles_x) * kTileH;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int x = tx0 + tx, y = ty0 + ty;
  const bool in_img = x < W && y < H;
  const float xn = in_img ? __ldg(&g.xs[x]) : 0.f, yn = in_img ? __ldg(&g.ys[y]) : 0.f;
  for (int i = threadIdx.x; i < n_h * 9; i += blockDim.x) hs[(i / 9) * 12 + i % 9] = __ldg(&hmat[(size_t)img * n_h * 9 + i]);
  if (threadIdx.x < kMaxKs) rows_s[threadIdx.x] = ek.rows[threadIdx.x];
  const float* pimg = probs + (size_t)img * (n_h + 1) * H * W;
  const int hw = H * W;
  float acc = 0.f, cnt = 1.f, mx = 0.f;
  if (in_img) {
    acc = __ldg(&pimg[y * W + x]);
    mx = acc;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < n_h; j += blockDim.x)
    cls_s[j] = (uint8_t)classify_tile(hs + j * 12, g, ek, tx0, ty0, H, W, true);
  __syncthreads();
  if (threadIdx.x < 32) {  // ordered compaction into the two work lists (outside tiles contribute nothing: dropped)
    int nd = 0, nr = 0;
    for (int base = 0; base < n_h; base += 32) {
      const int j = base + threadIdx.x;
      const int c = j < n_h ? cls_s[j] : kTileOutside;
      const unsigned md = __ballot_sync(0xffffffffu, c == kTileDeep);
      const unsigned mr = __ballot_sync(0xffffffffu, c == kTileMixed || c == kTileInside);
      const unsigned lt = (1u << threadIdx.x) - 1u;
      if (c == kTileDeep) deep_s[nd + __popc(md & lt)] = (uint8_t)j;
      if (c == kTileMixed || c == kTileInside) rest_s[nr + __popc(mr & lt)] = (uint8_t)j;
      nd += __popc(md);
      nr += __popc(mr);
    }
    if (threadIdx.x == 0) {
      n_list[0] = nd;
      n_list[1] = nr;
    }
  }
  __syncthreads();
  const int n_deep = n_list[0], n_rest = n_list[1];
  if (in_img) {
    int k = 0;
    for (; k + 3 < n_deep; k += 4) {  // four samples (16 loads) in flight per thread
      const DeepTaps a = deep_taps(pimg, hs4, hs, deep_s[k], hw, W, xn, yn, g.hw, g.hh);
      const DeepTaps b = deep_taps(pimg, hs4, hs, deep_s[k + 1], hw, W, xn, yn, g.hw, g.hh);
      const DeepTaps c = deep_taps(pimg, hs4, hs, deep_s[k + 2], hw, W, xn, yn, g.hw, g.hh);
      const DeepTaps d = deep_taps(pimg, hs4, hs, deep_s[k + 3], hw, W, xn, yn, g.hw, g.hh);
      const float va = deep_value(a), vb = deep_value(b), vc = deep_value(c), vd = deep_value(d);
      acc += va;
      acc += vb;
      acc += vc;
      acc += vd;
      mx = fmaxf(fmaxf(mx, fmaxf(va, vb)), fmaxf(vc, vd));
    }
    for (; k < n_deep; ++k) {
      const float va = deep_value(deep_taps(pimg, hs4, hs, deep_s[k], hw, W, xn, yn, g.hw, g.hh));
      acc += va;
      mx = fmaxf(mx, va);
    }
    cnt += (float)n_deep;
  }
  int nmixed = 0;
  for (int k = 0; k < n_rest; ++k) {
    const int j = rest_s[k];
    const float* m = hs + j * 12;
    int c = 1;
    if (cls_s[j] == kTileMixed) {        // block-uniform
      uint32_t* bb = bits[nmixed & 1];   // double buffered: one barrier per mixed homography
      ++nmixed;
      fill_raw_bits(bb, m, g, ek, tx0, ty0, H, W);
      __syncthreads();
      c = eroded_bits(bb, rows_s, ek.ks, tx, ty);
    }
    if (in_img && c) {
      float sx, sy;
      kornia_src(m, xn, yn, g.hw, g.hh, sx, sy);
      const float v = bilinear_zero_exact(pimg + (j + 1) * hw, sx, sy, H, W);
      acc += v;
      cnt += 1.f;
      mx = fmaxf(mx, v);
    }
  }
  if (in_img) out[((size_t)img * H + y) * W + x] = agg_max ? mx : acc / cnt;
}

// ---------------- device homography sampler (homographic_augmentation.py:21-106) ----------------

struct Rng {
  uint64_t key, ctr;
  __device__ double uniform() {  // (0,1)
    const uint64_t r = splitmix64(key ^ splitmix64(ctr++));
    return ((double)(r >> 11) + 0.5) * (1.0 / 9007199254740992.0);
  }
  __device__ double truncnorm(double loc, double scale) {  // scipy.stats.truncnorm(-2, 2, loc, scale)
    const double lo = 0.022750131948179195, hi = 0.9772498680518208;  // Phi(-2), Phi(2)
    return loc + scale * normcdfinv(lo + uniform() * (hi - lo));
  }
  __device__ int randint(int n) { return min((int)(uniform() * n), n - 1); }
};

__device__ void inv3x3(const float* a, float* o) {
  const float c00 = a[4] * a[8] - a[5] * a[7], c01 = a[5] * a[6] - a[3] * a[8], c02 = a[3] * a[7] - a[4] * a[6];
  const float det = a[0] * c00 + a[1] * c01 + a[2] * c02;
  const float id = 1.0f / det;
  o[0] = c00 * id; o[1] = (a[2] * a[7] - a[1] * a[8]) * id; o[2] = (a[1] * a[5] - a[2] * a[4]) * id;
  o[3] = c01 * id; o[4] = (a[0] * a[8] - a[2] * a[6]) * id; o[5] = (a[2] * a[3] - a[0] * a[5]) * id;
  o[6] = c02 * id; o[7] = (a[1] * a[6] - a[0] * a[7]) * id; o[8] = (a[0] * a[4] - a[1] * a[3]) * id;
}

__device__ bool all_in_unit(const double (*p)[2]) {
  bool ok = true;
  for (int i = 0; i < 4; ++i) ok = ok && p[i][0] >= 0.0 && p[i][0] <= 1.0 && p[i][1] >= 0.0 && p[i][1] <= 1.0;
  return ok;
}

__global__ void sample_homographies_kernel(spn_homography_params prm, uint64_t seed, uint64_t first, int count, int H,
                                           int W, float* __restrict__ out_h, float* __restrict__ out_hinv) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  Rng rng{splitmix64(seed) ^ splitmix64(0xD1B54A32D192ED03ull * (first + i + 1)), 0};
  const double pr = prm.patch_ratio, margin = (1.0 - pr) / 2.0;
  double p1[4][2] = {{margin, margin}, {margin, margin + pr}, {margin + pr, margin + pr}, {margin + pr, margin}};
  double p2[4][2];
  for (int k = 0; k < 4; ++k) { p2[k][0] = p1[k][0]; p2[k][1] = p1[k][1]; }
  if (prm.perspective) {
    double ax = prm.perspective_amplitude_x, ay = prm.perspective_amplitude_y;
    if (!prm.allow_artifacts) { ax = fmin(ax, margin); ay = fmin(ay, margin); }
    const double dy = rng.truncnorm(0.0, ay / 2), dl = rng.truncnorm(0.0, ax / 2), dr = rng.truncnorm(0.0, ax / 2);
    p2[0][0] += dl; p2[0][1] += dy;
    p2[1][0] += dl; p2[1][1] -= dy;
    p2[2][0] += dr; p2[2][1] += dy;
    p2[3][0] += dr; p2[3][1] -= dy;
  }
  if (prm.scaling) {
    const int ns = min(prm.n_scales, 31);
    double sc[32];
    sc[0] = 1.0;
    for (int k = 1; k <= ns; ++k) sc[k] = rng.truncnorm(1.0, prm.scaling_amplitude / 2);
    double cx = 0, cy = 0;
    for (int k = 0; k < 4; ++k) { cx += p2[k][0]; cy += p2[k][1]; }
    cx /= 4; cy /= 4;
    int valid[32], nv = 0;
    for (int k = (prm.allow_artifacts ? 1 : 0); k <= ns; ++k) {
      double q[4][2];
      for (int t = 0; t < 4; ++t) { q[t][0] = (p2[t][0] - cx) * sc[k] + cx; q[t][1] = (p2[t][1] - cy) * sc[k] + cy; }
      if (prm.allow_artifacts || all_in_unit(q)) valid[nv++] = k;
    }
    const int idx = nv ? valid[rng.randint(nv)] : 0;
    for (int t = 0; t < 4; ++t) { p2[t][0] = (p2[t][0] - cx) * sc[idx] + cx; p2[t][1] = (p2[t][1] - cy) * sc[idx] + cy; }
  }
  if (prm.translation) {
    double tminx = 1e30, tminy = 1e30, tmaxx = 1e30, tmaxy = 1e30;
    for (int t = 0; t < 4; ++t) {
      tminx = fmin(tminx, p2[t][0]); tminy = fmin(tminy, p2[t][1]);
      tmaxx = fmin(tmaxx, 1.0 - p2[t][0]); tmaxy = fmin(tmaxy, 1.0 - p2[t][1]);
    }
    if (prm.allow_artifacts) {
      tminx += prm.translation_overflow; tminy += prm.translation_overflow;
      tmaxx += prm.translation_overflow; tmaxy += prm.translation_overflow;
    }
    const double dx = -tminx + rng.uniform() * (tmaxx + tminx), dy = -tminy + rng.uniform() * (tmaxy + tminy);
    for (int t = 0; t < 4; ++t) { p2[t][0] += dx; p2[t][1] += dy; }
  }
  if (prm.rotation) {
    const int na = min(prm.n_angles, 63);
    double cx = 0, cy = 0;
    for (int k = 0; k < 4; ++k) { cx += p2[k][0]; cy += p2[k][1]; }
    cx /= 4; cy /= 4;
    int valid[64], nv = 0;
    for (int k = (prm.allow_artifacts ? 1 : 0); k <= na; ++k) {
      const double ang = k == 0 ? 0.0 : (na > 1 ? -prm.max_angle + (2.0 * prm.max_angle) * (k - 1) / (na - 1) : -prm.max_angle);
      const double c = cos(ang), s = sin(ang);
      double q[4][2];
      for (int t = 0; t < 4; ++t) {  // (p - c) @ [[cos, -sin], [sin, cos]]
        const double ux = p2[t][0] - cx, uy = p2[t][1] - cy;
        q[t][0] = ux * c + uy * s + cx;
        q[t][1] = -ux * s + uy * c + cy;
      }
      if (prm.allow_artifacts || all_in_unit(q)) valid[nv++] = k;
    }
    const int idx = nv ? valid[rng.randint(nv)] : 0;
    const double ang = idx == 0 ? 0.0 : (na > 1 ? -prm.max_angle + (2.0 * prm.max_angle) * (idx - 1) / (na - 1) : -prm.max_angle);
    const double c = cos(ang), s = sin(ang);
    for (int t = 0; t < 4; ++t) {
      const double ux = p2[t][0] - cx, uy = p2[t][1] - cy;
      p2[t][0] = ux * c + uy * s + cx;
      p2[t][1] = -ux * s + uy * c + cy;
    }
  }
  // to pixels (x * W, y * H), rounded to fp32 like np.float32(pts) before cv2.getPerspectiveTransform
  double a[8][9];
  for (int t = 0; t < 4; ++t) {
    const double sx = (double)(float)(p1[t][0] * W), sy = (double)(float)(p1[t][1] * H);
    const double dx = (double)(float)(p2[t][0] * W), dy = (double)(float)(p2[t][1] * H);
    double* r0 = a[t];
    double* r1 = a[t + 4];
    r0[0] = sx; r0[1] = sy; r0[2] = 1; r0[3] = 0; r0[4] = 0; r0[5] = 0; r0[6] = -sx * dx; r0[7] = -sy * dx; r0[8] = dx;
    r1[0] = 0; r1[1] = 0; r1[2] = 0; r1[3] = sx; r1[4] = sy; r1[5] = 1; r1[6] = -sx * dy; r1[7] = -sy * dy; r1[8] = dy;
  }
  for (int c = 0; c < 8; ++c) {  // Gaussian elimination, partial pivoting (cv2 solves with DECOMP_LU)
    int piv = c;
    for (int r = c + 1; r < 8; ++r)
      if (fabs(a[r][c]) > fabs(a[piv][c])) piv = r;
    if (piv != c)
      for (int k = 0; k < 9; ++k) { const double t = a[c][k]; a[c][k] = a[piv][k]; a[piv][k] = t; }
    const double d = 1.0 / a[c][c];
    for (int r = c + 1; r < 8; ++r) {
      const double f = a[r][c] * d;
      for (int k = c; k < 9; ++k) a[r][k] -= f * a[c][k];
    }
  }
  double sol[8];
  for (int r = 7; r >= 0; --r) {
    double s = a[r][8];
    for (int k = r + 1; k < 8; ++k) s -= a[r][k] * sol[k];
    sol[r] = s / a[r][r];
  }
  float M[9], Hm[9], Hi[9];
  for (int k = 0; k < 8; ++k) M[k] = (float)sol[k];
  M[8] = 1.0f;
  inv3x3(M, Hm);   // homography = torch.inverse(M)           (homographic_augmentation.py:104)
  inv3x3(Hm, Hi);  // H_inv = torch.inverse(H)                (export.py:49)
  for (int k = 0; k < 9; ++k) {
    out_h[(size_t)i * 9 + k] = Hm[k];
    out_hinv[(size_t)i * 9 + k] = Hi[k];
  }
}

__global__ void invert3x3_kernel(const float* __restrict__ in, int count, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float a[9], o[9];
  for (int k = 0; k < 9; ++k) a[k] = in[(size_t)i * 9 + k];
  inv3x3(a, o);
  for (int k = 0; k < 9; ++k) out[(size_t)i * 9 + k] = o[k];
}

// kornia normalize_homography + inverse for a batch of pixel-space homographies (the matrices K.warp_perspective
// builds internally at export.py:51-55,72): fwd = inverse(N (M N^-1)) samples the source of warp(., M);
// bwd = the same for M^-1 (export.py:49).  N = normal_transform_pixel(H, W); products in the reference's order (no
// FMA); the 3x3 inverses use the adjugate, which agrees with the reference's LAPACK inverse to a few ulp, not bit for
// bit (for bit-exact masks the caller passes matrices computed with the reference's own torch.inverse).
__device__ void mm3_ref(const float* A, const float* B, float* C) {
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      C[i * 3 + j] = __fadd_rn(__fadd_rn(__fmul_rn(A[i * 3], B[j]), __fmul_rn(A[i * 3 + 1], B[3 + j])), __fmul_rn(A[i * 3 + 2], B[6 + j]));
}

__global__ void kornia_matrices_kernel(const float* __restrict__ h, int count, int H, int W, float* __restrict__ fwd,
                                       float* __restrict__ bwd) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const float ax = __fdiv_rn(2.0f, (float)(W - 1)), ay = __fdiv_rn(2.0f, (float)(H - 1));
  const float n[9] = {ax, 0.f, -1.f, 0.f, ay, -1.f, 0.f, 0.f, 1.f};
  const float rx = __frcp_rn(ax), ry = __frcp_rn(ay);
  const float ni[9] = {rx, 0.f, rx, 0.f, ry, ry, 0.f, 0.f, 1.f};
  float m[9], mi[9], t[9], a[9], o[9];
  for (int k = 0; k < 9; ++k) m[k] = h[(size_t)i * 9 + k];
  inv3x3(m, mi);
  mm3_ref(m, ni, t);
  mm3_ref(n, t, a);
  inv3x3(a, o);
  for (int k = 0; k < 9; ++k) fwd[(size_t)i * 9 + k] = o[k];
  mm3_ref(mi, ni, t);
  mm3_ref(n, t, a);
  inv3x3(a, o);
  for (int k = 0; k < 9; ++k) bwd[(size_t)i * 9 + k] = o[k];
}

// Loader pre-processing (data/COCO.py:66-76, data/HPatches.py:64-72): bilinear resize (align_corners=False, no
// antialias, i.e. F.interpolate as kornia.resize calls it) + centre crop (zero pad if the resized image is smaller)
// + division by 255, fused; source is the decoded grayscale image as uint8 or float32.
template <typename T>
__global__ void __launch_bounds__(256)
resize_crop_kernel(const T* __restrict__ src, int H0, int W0, int nh, int nw, int top, int left, int H, int W,
                   float divisor, float* __restrict__ out) {
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= W || y >= H) return;
  const int ry = y + top, rx = x + left;  // coordinates in the resized image
  float v = 0.f;
  if (ry >= 0 && ry < nh && rx >= 0 && rx < nw) {
    const float sy = fmaxf(((float)H0 / (float)nh) * ((float)ry + 0.5f) - 0.5f, 0.f);
    const float sx = fmaxf(((float)W0 / (float)nw) * ((float)rx + 0.5f) - 0.5f, 0.f);
    const int y0 = (int)sy, x0 = (int)sx;
    const int y1 = y0 + (y0 < H0 - 1 ? 1 : 0), x1 = x0 + (x0 < W0 - 1 ? 1 : 0);
    const float ly1 = sy - (float)y0, lx1 = sx - (float)x0, ly0 = 1.f - ly1, lx0 = 1.f - lx1;
    const float v00 = (float)src[(size_t)y0 * W0 + x0], v01 = (float)src[(size_t)y0 * W0 + x1];
    const float v10 = (float)src[(size_t)y1 * W0 + x0], v11 = (float)src[(size_t)y1 * W0 + x1];
    v = ly0 * (lx0 * v00 + lx1 * v01) + ly1 * (lx0 * v10 + lx1 * v11);
  }
  out[(size_t)y * W + x] = v / divisor;
}

}  // namespace

extern "C" int spn_resize_crop(spn_ctx* ctx, const void* d_src, int src_is_u8, int H0, int W0, int new_h, int new_w,
                               int crop_top, int crop_left, int H, int W, float divisor, float* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_src && d_out, "spn_resize_crop: null pointer");
  SpnDeviceGuard guard(ctx->device);
  SPN_REQUIRE(H0 > 0 && W0 > 0 && new_h > 0 && new_w > 0 && H > 0 && W > 0 && divisor != 0.f, "spn_resize_crop: bad shape");
  dim3 grid(spn_cdiv(W, 32), spn_cdiv(H, 8));
  if (src_is_u8)
    resize_crop_kernel<uint8_t><<<grid, 256, 0, (cudaStream_t)stream>>>((const uint8_t*)d_src, H0, W0, new_h, new_w, crop_top,
                                                                         crop_left, H, W, divisor, d_out);
  else
    resize_crop_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>((const float*)d_src, H0, W0, new_h, new_w, crop_top, crop_left,
                                                                       H, W, divisor, d_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

// kornia create_meshgrid coordinates, tabulated per image size: xs[i] = (i / (W-1) - 0.5) * 2 in IEEE fp32, the
// reference's operation order (linspace(0, W-1, W) is exact integers).  Cached per (H, W) in the context.
static int kornia_grid(spn_ctx* ctx, int H, int W, cudaStream_t s, KGrid* out) {
  SPN_REQUIRE(H >= 2 && W >= 2, "kornia grid needs H, W >= 2");
  for (auto& e : ctx->grids)
    if (e.H == H && e.W == W) {
      *out = KGrid{e.tab, e.tab + W, 0.5f * (float)(W - 1), 0.5f * (float)(H - 1)};
      return SPN_OK;
    }
  std::vector<float> host((size_t)W + H);
  for (int i = 0; i < W; ++i) {
    volatile float q = (float)i / (float)(W - 1);
    volatile float d = q - 0.5f;
    host[i] = d * 2.0f;
  }
  for (int i = 0; i < H; ++i) {
    volatile float q = (float)i / (float)(H - 1);
    volatile float d = q - 0.5f;
    host[W + i] = d * 2.0f;
  }
  SpnGridTab e;
  e.H = H; e.W = W; e.tab = nullptr;
  SPN_CUDA(cudaMalloc((void**)&e.tab, host.size() * sizeof(float)));
  // pageable source: the copy is staged before the call returns, so `host` may go out of scope
  SPN_CUDA(cudaMemcpyAsync(e.tab, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice, s));
  ctx->grids.push_back(e);
  *out = KGrid{e.tab, e.tab + W, 0.5f * (float)(W - 1), 0.5f * (float)(H - 1)};
  return SPN_OK;
}

extern "C" int spn_kornia_matrices(spn_ctx* ctx, const float* d_h, int count, int H, int W, float* d_ainv_fwd,
                                   float* d_ainv_bwd, spn_stream stream) {
  SPN_REQUIRE(ctx && d_h && d_ainv_fwd && d_ainv_bwd && count >= 0, "spn_kornia_matrices: bad argument");
  SPN_REQUIRE(H >= 2 && W >= 2, "spn_kornia_matrices: H, W must be >= 2");
  SpnDeviceGuard guard(ctx->device);
  if (count == 0) return SPN_OK;
  kornia_matrices_kernel<<<spn_cdiv(count, 128), 128, 0, (cudaStream_t)stream>>>(d_h, count, H, W, d_ainv_fwd, d_ainv_bwd);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_warp_batch(spn_ctx* ctx, const float* d_images, int n_images, const float* d_ainv, int n_h, int H,
                              int W, int margin, float* d_warped, uint8_t* d_mask, spn_stream stream) {
  SPN_REQUIRE(ctx && d_images && d_mask, "spn_warp_batch: null pointer");
  SpnDeviceGuard guard(ctx->device);
  SPN_REQUIRE(n_images > 0 && n_h >= 0 && H > 0 && W > 0, "spn_warp_batch: bad shape");
  SPN_REQUIRE(n_h == 0 || d_ainv, "spn_warp_batch: d_ainv is null");
  KGrid kg;
  {
    const int rc = kornia_grid(ctx, H, W, (cudaStream_t)stream, &kg);
    if (rc) return rc;
  }
  // the reference's valid_border_margin == 0 path is shape-broken (SURVEY.md section 8 a2): unsupported
  SPN_REQUIRE(margin >= 0 && 2 * margin <= kMaxKs, "spn_warp_batch: valid_border_margin must be in [0,%d]", kMaxKs / 2);
  SPN_REQUIRE((size_t)n_images * (n_h + 1) <= 65535, "spn_warp_batch: too many slots per launch");
  const ErodeK ek = make_ellipse(margin);
  const int tiles_x = spn_cdiv(W, kTileW), tiles_y = spn_cdiv(H, kTileH);
  SPN_REQUIRE(tiles_x <= kMaxRowTiles, "spn_warp_batch: W must be <= %d", kMaxRowTiles * kTileW);
  dim3 grid(tiles_y, n_images * (n_h + 1));
  SpnProfScope prof(ctx, SPN_PROF_WARP, (cudaStream_t)stream);
  warp_batch_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_images, d_ainv, kg, n_h, H, W, tiles_x, ek, d_warped, d_mask);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_ha_aggregate(spn_ctx* ctx, const float* d_probs, const float* d_h, int n_images, int n_h, int H,
                                int W, int margin, int aggregation, float* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_probs && d_out, "spn_ha_aggregate: null pointer");
  SpnDeviceGuard guard(ctx->device);
  KGrid kg;
  {
    const int rc = kornia_grid(ctx, H, W, (cudaStream_t)stream, &kg);
    if (rc) return rc;
  }
  SPN_REQUIRE(n_images > 0 && n_images <= 65535 && n_h >= 0 && H > 0 && W > 0, "spn_ha_aggregate: bad shape");
  SPN_REQUIRE(n_h == 0 || d_h, "spn_ha_aggregate: d_h is null");
  SPN_REQUIRE(margin >= 1 && 2 * margin <= kMaxKs, "spn_ha_aggregate: valid_border_margin must be in [1,%d]", kMaxKs / 2);
  SPN_REQUIRE(aggregation == 0 || aggregation == 1, "spn_ha_aggregate: aggregation must be 0 (sum) or 1 (max)");
  SPN_REQUIRE(n_h <= 255, "spn_ha_aggregate: at most 255 homographies per image");
  SPN_REQUIRE((size_t)(n_h + 1) * H * W < (1u << 30), "spn_ha_aggregate: (n_h + 1) * H * W must be below 2^30");
  const ErodeK ek = make_ellipse(margin);
  const int tiles_x = spn_cdiv(W, kTileW), tiles_y = spn_cdiv(H, kTileH);
  dim3 grid(tiles_x * tiles_y, n_images);
  SpnProfScope prof(ctx, SPN_PROF_AGGREGATE, (cudaStream_t)stream);
  ha_aggregate_kernel<<<grid, 256, n_h * 12 * sizeof(float) + 3 * ((n_h + 15) & ~15), (cudaStream_t)stream>>>(d_probs, d_h, kg, n_h, H, W, tiles_x, ek,
                                                                                     aggregation, d_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_sample_homographies(spn_ctx* ctx, const spn_homography_params* params, uint64_t seed,
                                       uint64_t first_index, int count, int H, int W, float* d_h, float* d_hinv,
                                       spn_stream stream) {
  SPN_REQUIRE(ctx && params && d_h && d_hinv, "spn_sample_homographies: null pointer");
  SpnDeviceGuard guard(ctx->device);
  SPN_REQUIRE(count >= 0 && H > 0 && W > 0, "spn_sample_homographies: bad shape");
  SPN_REQUIRE(params->n_scales >= 1 && params->n_scales <= 31 && params->n_angles >= 1 && params->n_angles <= 63,
              "spn_sample_homographies: n_scales must be in [1,31], n_angles in [1,63]");
  if (count == 0) return SPN_OK;
  SpnProfScope prof(ctx, SPN_PROF_SAMPLER, (cudaStream_t)stream);
  sample_homographies_kernel<<<spn_cdiv(count, 64), 64, 0, (cudaStream_t)stream>>>(*params, seed, first_index, count, H,
                                                                                    W, d_h, d_hinv);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}

extern "C" int spn_invert3x3(spn_ctx* ctx, const float* d_in, int count, float* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_in && d_out && count >= 0, "spn_invert3x3: bad argument");
  SpnDeviceGuard guard(ctx->device);
  if (count == 0) return SPN_OK;
  invert3x3_kernel<<<spn_cdiv(count, 128), 128, 0, (cudaStream_t)stream>>>(d_in, count, d_out);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
