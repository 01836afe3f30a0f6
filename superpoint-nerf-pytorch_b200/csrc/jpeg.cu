// Baseline JPEG -> grayscale decoder of the export loader (include/spn_jpeg.h).
//
// spn_jpeg_plan parses the headers on the host into a flat plan; spn_jpeg_decode_gray runs two kernels:
//   jpeg_entropy_kernel  one thread per image walks the entropy-coded segment (byte unstuffing, RSTn markers inline),
//                        decodes every block of every component and stores the luma blocks' 16-bit coefficients in
//                        natural order; chroma is parsed and dropped.  A serial chain per image: latency bound.
//   jpeg_idct_kernel     one thread per luma block: dequantisation + ISLOW inverse DCT + level shift, cropped to the
//                        image, written into the image's uint8 plane.
// The arithmetic is libjpeg-turbo's where the two can differ: jdhuff.c for the entropy decoder (DC predictor in int,
// stored as 16 bits; AC positions past 63 land on 63 as jpeg_natural_order's padding does) and the x86-64 SIMD ISLOW
// IDCT (jidctint-sse2/avx2: 16-bit lanes) for the transform.
#include "spn_common.cuh"
#include "../../include/spn_jpeg.h"

#include <algorithm>

namespace {

constexpr uint32_t kPlanMagic = 0x4750534au;  // "JSPG"

struct JpegHuff {         // one decoding table (1424 bytes)
  uint16_t lut[512];      // 9-bit lookahead: (code length << 8) | symbol, 0 = longer code
  int32_t maxcode[18];    // largest code of each length, -1 if none (libjpeg's maxcode; [17] is a sentinel)
  int32_t valoff[18];     // symbol index of the first code of each length minus that code
  uint8_t val[256];       // symbols in code order
};

struct JpegImage {        // one image of the plan (136 bytes)
  int32_t status, height, width, bw, bh, mcus_x, mcus_y, restart;
  int32_t ncomp, luma_pos, luma_h, luma_v;
  int32_t nblk[4];        // blocks per MCU of each scan component
  int32_t dc[4], ac[4];   // byte offsets of the Huffman tables in the plan
  int32_t quant, pad;     // byte offset of the luma quantisation table (64 int16, natural order)
  int64_t data_begin, data_end;   // entropy-coded segment, absolute offsets in d_data
  int64_t coef_block;     // first block of the image in d_coef (64 coefficients each)
  int64_t out_off;        // byte offset of the H x W plane in d_out
};
static_assert(sizeof(JpegImage) == 136, "plan layout");
static_assert(sizeof(JpegHuff) % 16 == 0, "plan layout");

struct PlanHead {
  uint32_t magic;
  int32_t n;
  int64_t bytes;
};

// zigzag index -> natural index, padded with 63 like libjpeg's jpeg_natural_order so that a corrupt run cannot go past
#define SPN_JPEG_NATURAL_ORDER                                                                                         \
  {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13,         \
   6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,         \
   39, 46, 53, 60, 61, 54, 47, 55, 62, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63, 63}
__constant__ uint8_t kNaturalDev[80] = SPN_JPEG_NATURAL_ORDER;
[[maybe_unused]] const uint8_t kNaturalHost[80] = SPN_JPEG_NATURAL_ORDER;

__host__ __device__ inline int natural_order(int k) {
#ifdef __CUDA_ARCH__
  return kNaturalDev[k];
#else
  return kNaturalHost[k];
#endif
}

// ---------------------------------------------------------------------------------------------------------------------
// entropy decoder

struct BitReader {
  const uint8_t* p;       // next byte to read
  const uint8_t* end;
  uint64_t acc;           // valid bits are the top `nbits`
  int nbits;
  int nfake;              // zero bits appended after a marker / the end (they are at the bottom of the valid bits)
  int marker;             // marker code that stopped the reader, -1 = none yet

  __host__ __device__ void fill() {
    if (marker < 0 && p + 4 <= end) {   // fast path: four bytes, none of them 0xFF
      uint32_t w = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3];
      if (((w & 0x7F7F7F7Fu) + 0x01010101u & w & 0x80808080u) == 0) {
        acc |= (uint64_t)w << (32 - nbits);
        nbits += 32;
        p += 4;
        return;
      }
    }
    while (nbits <= 56) {
      int c = 0;
      if (marker < 0) {
        if (p >= end) {
          marker = 0x100;               // out of data: libjpeg's fake EOI
        } else if ((c = *p++) == 0xFF) {
          while (p < end && *p == 0xFF) ++p;   // fill bytes
          if (p >= end) { marker = 0x100; c = 0; }
          else if (*p == 0) { ++p; }           // stuffed 0xFF00 -> data byte 0xFF
          else { marker = *p++; c = 0; }
        }
      }
      if (marker >= 0) nfake += 8;
      acc |= (uint64_t)c << (56 - nbits);
      nbits += 8;
    }
  }
  __host__ __device__ uint32_t peek(int n) const { return (uint32_t)(acc >> (64 - n)); }
  __host__ __device__ void skip(int n) { acc <<= n; nbits -= n; }
};

__host__ __device__ inline int huff_decode(BitReader& br, const JpegHuff* __restrict__ h) {
  const uint32_t e = h->lut[br.peek(9)];
  if (e) {
    br.skip(e >> 8);
    return e & 0xFF;
  }
  const uint32_t code16 = br.peek(16);
  for (int l = 10; l <= 16; ++l) {
    const int32_t code = (int32_t)(code16 >> (16 - l));
    if (code <= h->maxcode[l]) {
      br.skip(l);
      return h->val[(code + h->valoff[l]) & 0xFF];
    }
  }
  return -1;
}

__host__ __device__ inline int extend(uint32_t v, int s) {   // HUFF_EXTEND
  return (v < (1u << (s - 1))) ? (int)v - (1 << s) + 1 : (int)v;
}

// Decodes image i of the plan into coef (blocks of 64 int16, natural order); blk: 64 int16 of scratch, 16-byte aligned.
// Returns the image's status.
__host__ __device__ int jpeg_entropy_image(const uint8_t* __restrict__ plan, const uint8_t* __restrict__ data, int i,
                                           int16_t* __restrict__ coef, int64_t coef_blocks, int16_t* __restrict__ blk) {
  const JpegImage& im = reinterpret_cast<const JpegImage*>(plan + sizeof(PlanHead))[i];
  if (im.status != SPN_JPEG_OK) return im.status;
  const int64_t nblocks = (int64_t)im.bw * im.bh;
  if (im.coef_block < 0 || im.coef_block + nblocks > coef_blocks) return SPN_JPEG_BAD_PLAN;
  int16_t* out = coef + im.coef_block * 64;
  BitReader br{data + im.data_begin, data + im.data_end, 0, 0, 0, -1};
  int dc_pred = 0;
  int rst_next = 0, to_go = im.restart;
  const int n_mcu = im.mcus_x * im.mcus_y;
  for (int m = 0; m < n_mcu; ++m) {
    if (im.restart && to_go == 0) {   // libjpeg process_restart: drop buffered bits, expect RSTn, reset predictors
      br.acc = 0;
      br.nbits = br.nfake = 0;
      if (br.marker < 0) {
        while (br.p < br.end && *br.p != 0xFF) ++br.p;   // extraneous bytes are discarded (libjpeg warns)
        while (br.p < br.end && *br.p == 0xFF) ++br.p;
        br.marker = br.p < br.end ? *br.p++ : 0x100;
      }
      if (br.marker != 0xD0 + rst_next) return SPN_JPEG_BAD_RESTART;
      br.marker = -1;
      rst_next = (rst_next + 1) & 7;
      to_go = im.restart;
      dc_pred = 0;
    }
    const int mx = m % im.mcus_x, my = m / im.mcus_x;
    for (int c = 0; c < im.ncomp; ++c) {
      const bool luma = c == im.luma_pos;
      const JpegHuff* dc = reinterpret_cast<const JpegHuff*>(plan + im.dc[c]);
      const JpegHuff* ac = reinterpret_cast<const JpegHuff*>(plan + im.ac[c]);
      for (int b = 0; b < im.nblk[c]; ++b) {
        if (br.nbits < 32) br.fill();
        int s = huff_decode(br, dc);
        if (s < 0) return SPN_JPEG_BAD_CODE;
        int diff = 0;
        if (s) {
          if (br.nbits < 16) br.fill();
          diff = extend(br.peek(s), s);
          br.skip(s);
        }
        if (luma) {
#ifdef __CUDA_ARCH__
#pragma unroll
          for (int q = 0; q < 8; ++q) reinterpret_cast<uint4*>(blk)[q] = make_uint4(0, 0, 0, 0);
#else
          for (int q = 0; q < 64; ++q) blk[q] = 0;
#endif
          dc_pred = (int)((unsigned)diff + (unsigned)dc_pred);
          blk[0] = (int16_t)dc_pred;
          for (int k = 1; k < 64; ++k) {
            if (br.nbits < 32) br.fill();
            int rs = huff_decode(br, ac);
            if (rs < 0) return SPN_JPEG_BAD_CODE;
            const int r = rs >> 4;
            s = rs & 15;
            if (s) {
              k += r;
              const int v = extend(br.peek(s), s);
              br.skip(s);
              blk[natural_order(k)] = (int16_t)v;
            } else {
              if (r != 15) break;
              k += 15;
            }
          }
          const int bx = mx * im.luma_h + b % im.luma_h, by = my * im.luma_v + b / im.luma_h;
          int16_t* dst = out + ((int64_t)by * im.bw + bx) * 64;
#ifdef __CUDA_ARCH__
          const uint4* src4 = reinterpret_cast<const uint4*>(blk);
          uint4* dst4 = reinterpret_cast<uint4*>(dst);
#pragma unroll
          for (int q = 0; q < 8; ++q) dst4[q] = src4[q];
#else
          for (int q = 0; q < 64; ++q) dst[q] = blk[q];
#endif
        } else {
          for (int k = 1; k < 64; ++k) {
            if (br.nbits < 32) br.fill();
            int rs = huff_decode(br, ac);
            if (rs < 0) return SPN_JPEG_BAD_CODE;
            const int r = rs >> 4;
            s = rs & 15;
            if (s) {
              k += r;
              br.skip(s);
            } else {
              if (r != 15) break;
              k += 15;
            }
          }
        }
        if (br.nbits < br.nfake) return SPN_JPEG_PREMATURE_END;   // used bits that were never in the file
      }
    }
    if (im.restart) --to_go;
  }
  return SPN_JPEG_OK;
}

// One single-thread CTA per image: the decode is one dependent chain, so an image gets a warp scheduler slot of its own
// rather than sharing a diverging warp with 31 others.
__global__ void __launch_bounds__(1) jpeg_entropy_kernel(const uint8_t* __restrict__ plan, const uint8_t* __restrict__ data,
                                                         int n, int16_t* __restrict__ coef, int64_t coef_blocks,
                                                         int32_t* __restrict__ status) {
  __shared__ __align__(16) int16_t blk[64];
  const int i = blockIdx.x;
  const PlanHead* h = reinterpret_cast<const PlanHead*>(plan);
  status[i] = (h->magic != kPlanMagic || h->n != n) ? SPN_JPEG_BAD_PLAN : jpeg_entropy_image(plan, data, i, coef, coef_blocks, blk);
}

// ---------------------------------------------------------------------------------------------------------------------
// ISLOW inverse DCT as libjpeg-turbo's x86-64 SIMD kernel computes it: 16-bit dequantisation products, 16-bit sums of
// the inputs that are added before a multiply, pass-1 results saturated to int16 (packssdw), output saturated to int8
// and shifted by 128 (packsswb + paddb).  A block whose rows 1-7 are all zero takes the kernel's shortcut: pass 1 is
// (int16)(dequantised row 0 << 2).

constexpr int F0298 = 2446, F0390 = 3196, F0541 = 4433, F0765 = 6270, F0899 = 7373, F1175 = 9633, F1501 = 12299,
              F1847 = 15137, F1961 = 16069, F2053 = 16819, F2562 = 20995, F3072 = 25172;

__host__ __device__ inline int16_t sat16(int v) { return (int16_t)(v < -32768 ? -32768 : v > 32767 ? 32767 : v); }

// 1-D 8-point ISLOW on 16-bit inputs; out[] before the descale
__host__ __device__ inline void islow_1d(const int16_t in0, const int16_t in1, const int16_t in2, const int16_t in3,
                                         const int16_t in4, const int16_t in5, const int16_t in6, const int16_t in7,
                                         int out[8]) {
  const int tmp3e = in2 * (F0541 + F0765) + in6 * F0541;
  const int tmp2e = in2 * F0541 + in6 * (F0541 - F1847);
  const int t0 = (int)(int16_t)(in0 + in4) * (1 << 13);
  const int t1 = (int)(int16_t)(in0 - in4) * (1 << 13);
  const int tmp10 = t0 + tmp3e, tmp13 = t0 - tmp3e, tmp11 = t1 + tmp2e, tmp12 = t1 - tmp2e;
  const int z3 = (int16_t)(in7 + in3), z4 = (int16_t)(in5 + in1);
  const int z3p = z3 * (F1175 - F1961) + z4 * F1175;
  const int z4p = z3 * F1175 + z4 * (F1175 - F0390);
  const int o0 = in7 * (F0298 - F0899) + in1 * (-F0899) + z3p;
  const int o3 = in7 * (-F0899) + in1 * (F1501 - F0899) + z4p;
  const int o1 = in5 * (F2053 - F2562) + in3 * (-F2562) + z4p;
  const int o2 = in5 * (-F2562) + in3 * (F3072 - F2562) + z3p;
  out[0] = tmp10 + o3; out[7] = tmp10 - o3;
  out[1] = tmp11 + o2; out[6] = tmp11 - o2;
  out[2] = tmp12 + o1; out[5] = tmp12 - o1;
  out[3] = tmp13 + o0; out[4] = tmp13 - o0;
}

// coef and q: 64 values in natural order; pix: 8x8 row-major
__host__ __device__ inline void jpeg_idct_block(const int16_t* __restrict__ coef, const int16_t* __restrict__ q,
                                                uint8_t pix[64]) {
  int16_t dq[64], ws[64];
  bool ac_zero = true;
#pragma unroll
  for (int k = 0; k < 64; ++k) {
    dq[k] = (int16_t)(coef[k] * q[k]);
    if (k >= 8 && coef[k] != 0) ac_zero = false;
  }
  if (ac_zero) {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const int16_t v = (int16_t)(dq[c] * 4);
#pragma unroll
      for (int r = 0; r < 8; ++r) ws[r * 8 + c] = v;
    }
  } else {
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      int o[8];
      islow_1d(dq[c], dq[8 + c], dq[16 + c], dq[24 + c], dq[32 + c], dq[40 + c], dq[48 + c], dq[56 + c], o);
#pragma unroll
      for (int r = 0; r < 8; ++r) ws[r * 8 + c] = sat16((o[r] + (1 << 10)) >> 11);
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    int o[8];
    const int16_t* w = ws + r * 8;
    islow_1d(w[0], w[1], w[2], w[3], w[4], w[5], w[6], w[7], o);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      int v = (o[c] + (1 << 17)) >> 18;
      v = v < -128 ? -128 : v > 127 ? 127 : v;
      pix[r * 8 + c] = (uint8_t)(v + 128);
    }
  }
}

__global__ void __launch_bounds__(128) jpeg_idct_kernel(const uint8_t* __restrict__ plan, const int16_t* __restrict__ coef,
                                                        uint8_t* __restrict__ out, const int32_t* __restrict__ status) {
  const int i = blockIdx.y;
  if (status[i] != SPN_JPEG_OK) return;
  const JpegImage& im = reinterpret_cast<const JpegImage*>(plan + sizeof(PlanHead))[i];
  __shared__ int16_t q[64];
  if (threadIdx.x < 64) q[threadIdx.x] = reinterpret_cast<const int16_t*>(plan + im.quant)[threadIdx.x];
  __syncthreads();
  const int H = im.height, W = im.width, bw = im.bw;
  const int vis_w = (W + 7) >> 3, vis_h = (H + 7) >> 3;   // blocks that hold image pixels
  uint8_t* dst = out + im.out_off;
  const int64_t nvis = (int64_t)vis_w * vis_h;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < nvis; t += (int64_t)gridDim.x * blockDim.x) {
    const int bx = (int)(t % vis_w), by = (int)(t / vis_w);
    const int16_t* src = coef + (im.coef_block + (int64_t)by * bw + bx) * 64;
    int16_t c[64];
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
#pragma unroll
    for (int k = 0; k < 8; ++k) reinterpret_cast<uint4*>(c)[k] = __ldg(s4 + k);
    uint8_t pix[64];
    jpeg_idct_block(c, q, pix);
    const int x0 = bx * 8, y0 = by * 8;
    const int cw = min(8, W - x0), ch = min(8, H - y0);
    for (int r = 0; r < ch; ++r) {
      uint8_t* row = dst + (int64_t)(y0 + r) * W + x0;
      if (cw == 8 && ((uintptr_t)row & 7) == 0) {
        *reinterpret_cast<uint2*>(row) = *reinterpret_cast<const uint2*>(pix + r * 8);
      } else {
        for (int x = 0; x < cw; ++x) row[x] = pix[r * 8 + x];
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// host parser

struct HuffSpec {
  bool present = false;
  uint8_t bits[17] = {};
  uint8_t val[256] = {};
};

struct Frame {
  int status = SPN_JPEG_OK;
  int height = 0, width = 0, nc = 0;
  int id[4] = {}, h[4] = {}, v[4] = {}, tq[4] = {};
  int scan_n = 0, scan_comp[4] = {}, td[4] = {}, ta[4] = {};
  int restart = 0;
  int16_t quant[4][64] = {};
  bool quant_present[4] = {};
  HuffSpec dc[4], ac[4];
  bool jfif = false, adobe = false;
  int adobe_transform = 0;
  int64_t data_begin = 0, data_end = 0;
};

static int u16(const uint8_t* p) { return (p[0] << 8) | p[1]; }

// libjpeg's jpeg_make_d_derived_tbl, checks included (over-subscribed code space, more than 256 symbols, DC symbols > 15)
static bool build_huff(const HuffSpec& s, bool is_dc, JpegHuff* t) {
  memset(t, 0, sizeof(*t));
  int count = 0;
  for (int l = 1; l <= 16; ++l) count += s.bits[l];
  if (count > 256) return false;
  int huffsize[257], huffcode[257], p = 0;
  for (int l = 1; l <= 16; ++l)
    for (int i = 0; i < s.bits[l]; ++i) huffsize[p++] = l;
  huffsize[p] = 0;
  int code = 0, si = huffsize[0];
  p = 0;
  while (huffsize[p]) {
    while (huffsize[p] == si) huffcode[p++] = code++;
    if (code >= (1 << si)) return false;
    code <<= 1;
    ++si;
  }
  p = 0;
  for (int l = 1; l <= 16; ++l) {
    if (s.bits[l]) {
      t->valoff[l] = p - huffcode[p];
      p += s.bits[l];
      t->maxcode[l] = huffcode[p - 1];
    } else {
      t->maxcode[l] = -1;
    }
  }
  t->maxcode[17] = 0xFFFFF;
  memcpy(t->val, s.val, 256);
  p = 0;
  for (int l = 1; l <= 9; ++l)
    for (int i = 0; i < s.bits[l]; ++i, ++p) {
      const int lo = huffcode[p] << (9 - l), hi = (huffcode[p] + 1) << (9 - l);
      for (int x = lo; x < hi; ++x) t->lut[x] = (uint16_t)((l << 8) | s.val[p]);
    }
  if (is_dc)
    for (int i = 0; i < count; ++i)
      if (s.val[i] > 15) return false;
  return true;
}

// Parses one file up to the end of its first scan.  Never reads outside [0, len).
static void parse_jpeg(const uint8_t* d, int64_t len, Frame& f) {
  auto fail = [&](int st) { f.status = st; };
  if (len < 4 || d[0] != 0xFF || d[1] != 0xD8) return fail(SPN_JPEG_MALFORMED);
  int64_t p = 2;
  bool have_sof = false;
  for (;;) {
    if (p >= len) return fail(SPN_JPEG_MALFORMED);
    if (d[p] != 0xFF) return fail(SPN_JPEG_UNSUPPORTED);   // garbage between segments (libjpeg skips it with a warning)
    while (p < len && d[p] == 0xFF) ++p;                   // fill bytes
    if (p >= len) return fail(SPN_JPEG_MALFORMED);
    const int m = d[p++];
    if (m == 0xD8 || m == 0xD9 || (m >= 0xD0 && m <= 0xD7) || m == 0x01) return fail(SPN_JPEG_MALFORMED);
    if (p + 2 > len) return fail(SPN_JPEG_MALFORMED);
    const int L = u16(d + p);
    if (L < 2 || p + L > len) return fail(SPN_JPEG_MALFORMED);
    const uint8_t* s = d + p + 2;
    const int sl = L - 2;
    p += L;
    if (m == 0xC0 || m == 0xC1) {                             // SOF0 / SOF1
      if (have_sof || sl < 6) return fail(SPN_JPEG_MALFORMED);
      have_sof = true;
      f.height = u16(s + 1);
      f.width = u16(s + 3);
      f.nc = s[5];
      if (f.nc < 1 || sl != 6 + 3 * f.nc) return fail(SPN_JPEG_MALFORMED);
      if (s[0] != 8 || f.nc > 4) return fail(SPN_JPEG_UNSUPPORTED);
      if (f.height <= 0 || f.width <= 0 || f.height > 65500 || f.width > 65500) return fail(SPN_JPEG_MALFORMED);
      for (int c = 0; c < f.nc; ++c) {
        f.id[c] = s[6 + 3 * c];
        f.h[c] = s[7 + 3 * c] >> 4;
        f.v[c] = s[7 + 3 * c] & 15;
        f.tq[c] = s[8 + 3 * c];
        if (f.h[c] < 1 || f.h[c] > 4 || f.v[c] < 1 || f.v[c] > 4 || f.tq[c] > 3) return fail(SPN_JPEG_MALFORMED);
      }
    } else if (m >= 0xC2 && m <= 0xCF && m != 0xC4) {
      if (m != 0xC8 && m != 0xCC && sl >= 5) {                  // a frame header: report its size
        f.height = u16(s + 1);
        f.width = u16(s + 3);
      }
      return fail(SPN_JPEG_UNSUPPORTED);                     // progressive, lossless, hierarchical, arithmetic
    } else if (m == 0xC4) {                                   // DHT
      int q = 0;
      while (q < sl) {
        if (q + 17 > sl) return fail(SPN_JPEG_MALFORMED);
        const int tc = s[q] >> 4, th = s[q] & 15;
        if (tc > 1 || th > 3) return fail(SPN_JPEG_MALFORMED);
        HuffSpec& hs = tc ? f.ac[th] : f.dc[th];
        hs = HuffSpec();
        int count = 0;
        for (int l = 1; l <= 16; ++l) count += (hs.bits[l] = s[q + l]);
        q += 17;
        if (count > 256 || q + count > sl) return fail(SPN_JPEG_MALFORMED);
        memcpy(hs.val, s + q, count);
        hs.present = true;
        q += count;
      }
    } else if (m == 0xDB) {                                   // DQT
      int q = 0;
      while (q < sl) {
        const int pq = s[q] >> 4, tq = s[q] & 15;
        if (pq > 1 || tq > 3) return fail(SPN_JPEG_MALFORMED);
        ++q;
        if (q + 64 * (pq + 1) > sl) return fail(SPN_JPEG_MALFORMED);
        bool too_big = false;
        for (int k = 0; k < 64; ++k) {
          const int v = pq ? u16(s + q + 2 * k) : s[q + k];
          too_big |= v > 32767;
          f.quant[tq][natural_order(k)] = (int16_t)v;
        }
        if (too_big) return fail(SPN_JPEG_UNSUPPORTED);
        f.quant_present[tq] = true;
        q += 64 * (pq + 1);
      }
    } else if (m == 0xDD) {                                   // DRI
      if (sl != 2) return fail(SPN_JPEG_MALFORMED);
      f.restart = u16(s);
    } else if (m == 0xE0) {
      if (sl >= 14 && s[0] == 'J' && s[1] == 'F' && s[2] == 'I' && s[3] == 'F' && s[4] == 0) f.jfif = true;
    } else if (m == 0xEE) {
      if (sl >= 12 && s[0] == 'A' && s[1] == 'd' && s[2] == 'o' && s[3] == 'b' && s[4] == 'e') {
        f.adobe = true;
        f.adobe_transform = s[11];
      }
    } else if (m == 0xDA) {                                   // SOS
      if (!have_sof) return fail(SPN_JPEG_MALFORMED);
      const int ns = sl >= 1 ? s[0] : 0;
      if (ns < 1 || ns > 4 || sl != 4 + 2 * ns) return fail(SPN_JPEG_MALFORMED);
      f.scan_n = ns;
      for (int j = 0; j < ns; ++j) {
        int c = 0;
        while (c < f.nc && f.id[c] != s[1 + 2 * j]) ++c;
        if (c == f.nc) return fail(SPN_JPEG_MALFORMED);
        for (int k = 0; k < j; ++k)
          if (f.scan_comp[k] == c) return fail(SPN_JPEG_UNSUPPORTED);
        f.scan_comp[j] = c;
        f.td[j] = s[2 + 2 * j] >> 4;
        f.ta[j] = s[2 + 2 * j] & 15;
        if (f.td[j] > 3 || f.ta[j] > 3) return fail(SPN_JPEG_MALFORMED);
      }
      const uint8_t* t = s + 1 + 2 * ns;
      if (t[0] != 0 || t[1] != 63 || t[2] != 0) return fail(SPN_JPEG_UNSUPPORTED);
      f.data_begin = p;
      break;
    } else if (m >= 0xE0 || m == 0xFE) {
      // APPn / COM
    } else {
      return fail(SPN_JPEG_UNSUPPORTED);                     // DNL, DHP, EXP, JPGn, reserved
    }
  }
  // end of the entropy-coded segment: the first marker other than RSTn.  A file that ends before it, or before the EOI
  // that follows it, goes to the host: torchvision's source manager raises when libjpeg asks for bytes past the end,
  // which jpeg_finish_decompress does while it looks for the EOI.
  int64_t q = f.data_begin;
  for (;;) {
    const uint8_t* ff = (const uint8_t*)memchr(d + q, 0xFF, (size_t)(len - q));
    if (!ff) return fail(SPN_JPEG_UNSUPPORTED);
    int64_t r = ff - d;
    while (r < len && d[r] == 0xFF) ++r;
    if (r >= len) return fail(SPN_JPEG_UNSUPPORTED);
    if (d[r] == 0 || (d[r] >= 0xD0 && d[r] <= 0xD7)) { q = r + 1; continue; }
    f.data_end = ff - d;
    q = r;
    break;
  }
  // after the scan: only RSTn / APPn / COM up to the EOI keeps it a single-scan file the device decodes
  while (q < len) {
    const int m = d[q++];
    if (m == 0xD9) return;
    if (m >= 0xD0 && m <= 0xD7) {
    } else if (m >= 0xE0 || m == 0xFE) {
      if (q + 2 > len) break;
      q += u16(d + q);
    } else {
      return fail(SPN_JPEG_UNSUPPORTED);                     // another scan, or tables for one
    }
    while (q < len && d[q] != 0xFF) ++q;
    while (q < len && d[q] == 0xFF) ++q;
  }
  fail(SPN_JPEG_UNSUPPORTED);                               // no EOI
}

// Scope checks on a parsed frame (status stays SPN_JPEG_OK only for what the kernels decode exactly).
static void check_scope(Frame& f) {
  if (f.status != SPN_JPEG_OK) return;
  if (f.nc == 2 || f.nc == 4) return (void)(f.status = SPN_JPEG_UNSUPPORTED);     // no gray conversion / CMYK, YCCK
  if (f.nc == 3) {
    bool rgb;
    if (f.jfif) rgb = false;
    else if (f.adobe) rgb = f.adobe_transform == 0;
    else rgb = f.id[0] == 'R' && f.id[1] == 'G' && f.id[2] == 'B';
    if (rgb) return (void)(f.status = SPN_JPEG_UNSUPPORTED);
  }
  if (f.scan_n != f.nc) return (void)(f.status = SPN_JPEG_UNSUPPORTED);          // sequential, more than one scan
  for (int j = 0; j < f.scan_n; ++j) {
    const int c = f.scan_comp[j];
    if (!f.quant_present[f.tq[c]]) return (void)(f.status = SPN_JPEG_MALFORMED);
    if (!f.dc[f.td[j]].present || !f.ac[f.ta[j]].present) return (void)(f.status = SPN_JPEG_UNSUPPORTED);
  }
  if (f.nc > 1) {
    int hmax = 0, vmax = 0, blocks = 0;
    for (int c = 0; c < f.nc; ++c) {
      hmax = std::max(hmax, f.h[c]);
      vmax = std::max(vmax, f.v[c]);
      blocks += f.h[c] * f.v[c];
    }
    if (blocks > 10) return (void)(f.status = SPN_JPEG_MALFORMED);               // libjpeg: JERR_BAD_MCU_SIZE
    if (f.h[0] != hmax || f.v[0] != vmax) return (void)(f.status = SPN_JPEG_UNSUPPORTED);   // luma would be upsampled
  }
}

}  // namespace

extern "C" int spn_jpeg_plan(const uint8_t* h_data, const int64_t* h_offsets, int n, void* h_plan, int64_t* plan_bytes,
                             int64_t* h_info, int64_t* h_totals) {
  SPN_REQUIRE(h_offsets && plan_bytes && h_info && h_totals, "spn_jpeg_plan: null pointer");
  SPN_REQUIRE(n >= 1 && n <= 65535, "spn_jpeg_plan: n = %d (1..65535)", n);
  SPN_REQUIRE(h_data || h_offsets[n] == h_offsets[0], "spn_jpeg_plan: h_data is null");
  for (int i = 0; i < n; ++i)
    SPN_REQUIRE(h_offsets[i] >= 0 && h_offsets[i + 1] >= h_offsets[i], "spn_jpeg_plan: offsets must be non-decreasing");
  std::vector<JpegImage> imgs(n);
  std::vector<std::vector<JpegHuff>> tabs(n);
  int64_t bytes = sizeof(PlanHead) + (int64_t)n * sizeof(JpegImage);
  int64_t coef_blocks = 0, out_bytes = 0;
  Frame* f = new Frame;
  for (int i = 0; i < n; ++i) {
    *f = Frame();
    parse_jpeg(h_data + h_offsets[i], h_offsets[i + 1] - h_offsets[i], *f);
    check_scope(*f);
    JpegImage& im = imgs[i];
    memset(&im, 0, sizeof(im));
    im.status = f->status;
    im.height = f->height;
    im.width = f->width;
    im.coef_block = -1;
    im.out_off = -1;
    if (im.status == SPN_JPEG_OK) {
      if (f->nc == 1) {
        im.mcus_x = im.bw = (f->width + 7) / 8;
        im.mcus_y = im.bh = (f->height + 7) / 8;
        im.luma_h = im.luma_v = 1;
        im.nblk[0] = 1;
      } else {
        im.luma_h = f->h[0];
        im.luma_v = f->v[0];
        im.mcus_x = (f->width + 8 * im.luma_h - 1) / (8 * im.luma_h);
        im.mcus_y = (f->height + 8 * im.luma_v - 1) / (8 * im.luma_v);
        im.bw = im.mcus_x * im.luma_h;
        im.bh = im.mcus_y * im.luma_v;
      }
      im.ncomp = f->scan_n;
      im.restart = f->restart;
      im.data_begin = h_offsets[i] + f->data_begin;
      im.data_end = h_offsets[i] + f->data_end;
      int slot_dc[4] = {-1, -1, -1, -1}, slot_ac[4] = {-1, -1, -1, -1};
      // table block of this image: luma quantisation (128 bytes, padded to a JpegHuff) then the Huffman tables it uses
      tabs[i].emplace_back();
      memcpy(&tabs[i][0], f->quant[f->tq[0]], 128);
      bool ok = true;
      for (int j = 0; j < f->scan_n && ok; ++j) {
        const int c = f->scan_comp[j];
        if (c == 0) im.luma_pos = j;
        if (f->nc > 1) im.nblk[j] = f->h[c] * f->v[c];
        if (slot_dc[f->td[j]] < 0) {
          slot_dc[f->td[j]] = (int)tabs[i].size();
          tabs[i].emplace_back();
          ok &= build_huff(f->dc[f->td[j]], true, &tabs[i].back());
        }
        if (slot_ac[f->ta[j]] < 0) {
          slot_ac[f->ta[j]] = (int)tabs[i].size();
          tabs[i].emplace_back();
          ok &= build_huff(f->ac[f->ta[j]], false, &tabs[i].back());
        }
        im.dc[j] = slot_dc[f->td[j]];
        im.ac[j] = slot_ac[f->ta[j]];
      }
      if (!ok) {
        im.status = SPN_JPEG_MALFORMED;
        tabs[i].clear();
      } else {
        im.quant = (int32_t)bytes;
        for (int j = 0; j < f->scan_n; ++j) {
          im.dc[j] = (int32_t)(bytes + (int64_t)im.dc[j] * sizeof(JpegHuff));
          im.ac[j] = (int32_t)(bytes + (int64_t)im.ac[j] * sizeof(JpegHuff));
        }
        bytes += (int64_t)tabs[i].size() * sizeof(JpegHuff);
        im.coef_block = coef_blocks;
        coef_blocks += (int64_t)im.bw * im.bh;
        im.out_off = out_bytes;
        out_bytes += (int64_t)im.height * im.width;
      }
    }
    int64_t* info = h_info + (int64_t)i * SPN_JPEG_INFO_FIELDS;
    info[SPN_JPEG_INFO_STATUS] = im.status;
    info[SPN_JPEG_INFO_HEIGHT] = im.height;
    info[SPN_JPEG_INFO_WIDTH] = im.width;
    info[SPN_JPEG_INFO_BLOCKS] = im.status == SPN_JPEG_OK ? (int64_t)im.bw * im.bh : 0;
    info[SPN_JPEG_INFO_OUT_OFFSET] = im.out_off;
  }
  delete f;
  SPN_REQUIRE(bytes < (int64_t(1) << 31), "spn_jpeg_plan: plan of %lld bytes is too large (split the batch)", (long long)bytes);
  h_totals[0] = coef_blocks * 128;
  h_totals[1] = out_bytes;
  const int64_t cap = *plan_bytes;
  *plan_bytes = bytes;
  if (!h_plan) return SPN_OK;
  SPN_REQUIRE(cap >= bytes, "spn_jpeg_plan: plan buffer of %lld bytes, %lld needed", (long long)cap, (long long)bytes);
  uint8_t* out = static_cast<uint8_t*>(h_plan);
  PlanHead head{kPlanMagic, n, bytes};
  memcpy(out, &head, sizeof(head));
  memcpy(out + sizeof(PlanHead), imgs.data(), (size_t)n * sizeof(JpegImage));
  for (int i = 0; i < n; ++i)
    if (!tabs[i].empty()) memcpy(out + imgs[i].quant, tabs[i].data(), tabs[i].size() * sizeof(JpegHuff));
  return SPN_OK;
}

extern "C" int spn_jpeg_decode_gray(spn_ctx* ctx, const void* d_plan, const uint8_t* d_data, int n, int16_t* d_coef,
                                    int64_t coef_bytes, uint8_t* d_out, int32_t* d_status, spn_stream stream) {
  SPN_REQUIRE(ctx && d_plan && d_data && d_out && d_status, "spn_jpeg_decode_gray: null pointer");
  SPN_REQUIRE(n >= 1 && n <= 65535, "spn_jpeg_decode_gray: n = %d (1..65535)", n);
  SPN_REQUIRE(coef_bytes >= 0 && (coef_bytes == 0 || d_coef), "spn_jpeg_decode_gray: bad coefficient buffer");
  SPN_REQUIRE(((uintptr_t)d_coef & 15) == 0 && ((uintptr_t)d_plan & 15) == 0, "spn_jpeg_decode_gray: d_plan and d_coef must be 16-byte aligned");
  SpnDeviceGuard guard(ctx->device);
  cudaStream_t s = (cudaStream_t)stream;
  jpeg_entropy_kernel<<<n, 1, 0, s>>>((const uint8_t*)d_plan, d_data, n, d_coef, coef_bytes / 128, d_status);
  SPN_CHECK_LAUNCH(ctx);
  // 16 CTAs per image cover a 1080p luma plane in 4 strides; the grid never exceeds a few thousand CTAs per batch
  jpeg_idct_kernel<<<dim3(16, n), 128, 0, s>>>((const uint8_t*)d_plan, d_coef, d_out, d_status);
  SPN_CHECK_LAUNCH(ctx);
  return SPN_OK;
}
