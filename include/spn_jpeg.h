/* spn_jpeg.h - baseline JPEG -> grayscale decoder of the export loader (part of libspn_b200.so).
 *
 * Decodes what torchvision.io.decode_image(data, ImageReadMode.GRAY) decodes (libjpeg-turbo, JCS_GRAYSCALE output,
 * ISLOW IDCT) and gives the same bytes: the luma component of the scan after the inverse DCT, cropped to the image
 * size.  The IDCT follows the host decoder's x86-64 SIMD ISLOW kernel (16-bit lanes: 16-bit dequantisation products,
 * 16-bit sums before the multiplies, pass-1 results saturated to 16 bits, output saturated to 0..255), which is what
 * decode_image runs on x86-64; within 16-bit range it is the same arithmetic as jidctint.c.
 *
 * Decoded on the device: SOF0 / SOF1 (8-bit samples, Huffman coding), one scan holding every component (interleaved,
 * or a single component), sampling factors 1-4 with the luma component at the largest factors, restart intervals,
 * 8-bit DQT and 16-bit DQT with values <= 32767.  Everything else is reported as SPN_JPEG_UNSUPPORTED (progressive,
 * arithmetic, 12-bit, lossless, CMYK / YCCK / RGB, more than one scan, no EOI after the scan) or SPN_JPEG_MALFORMED; the
 * caller decodes those on the host.
 *
 * Conventions are those of spn_b200.h: return 0 or a negative SPN_E_* code with spn_last_error(), caller-owned
 * buffers, no allocation, no synchronisation.  These entry points do not use the context's workspace, so a loader
 * context may decode on a side stream while a model context runs.
 */
#ifndef SPN_JPEG_H
#define SPN_JPEG_H

#include "spn_b200.h"

#ifdef __cplusplus
extern "C" {
#endif

/* per-image status: spn_jpeg_plan reports 0..2, spn_jpeg_decode_gray writes 0..6 into d_status */
enum {
  SPN_JPEG_OK = 0,
  SPN_JPEG_UNSUPPORTED = 1, /* a valid file outside the device decoder's scope: decode it on the host */
  SPN_JPEG_MALFORMED = 2,   /* the header parser rejected it                                           */
  SPN_JPEG_BAD_CODE = 3,    /* entropy data: a Huffman code that is not in the table                   */
  SPN_JPEG_PREMATURE_END = 4, /* entropy data: a marker or the end of the file before the last block    */
  SPN_JPEG_BAD_RESTART = 5, /* entropy data: the expected RSTn marker is missing                       */
  SPN_JPEG_BAD_PLAN = 6     /* the plan does not match n or coef_bytes                                 */
};

/* per-image fields of h_info */
enum { SPN_JPEG_INFO_STATUS = 0, SPN_JPEG_INFO_HEIGHT, SPN_JPEG_INFO_WIDTH, SPN_JPEG_INFO_BLOCKS, SPN_JPEG_INFO_OUT_OFFSET,
       SPN_JPEG_INFO_FIELDS };

/* Host only.  Parses the headers of n JPEG files held back to back in h_data: file i is bytes
 * [h_offsets[i], h_offsets[i+1]) (h_offsets has n+1 entries).  Never reads outside those ranges.
 *   h_info [n][SPN_JPEG_INFO_FIELDS]: status, height, width, luma blocks (8x8, MCU padding included) and the byte offset
 *     of the image's H x W luma plane in d_out (-1 unless status is SPN_JPEG_OK; the planes of the decodable images are
 *     packed in order).  Height and width are reported whenever the frame header was read.
 *   h_totals [2]: bytes of d_coef and of d_out that spn_jpeg_decode_gray needs.
 *   *plan_bytes: in = capacity of h_plan, out = size of the plan.  h_plan == NULL asks for the size only; a smaller
 *     capacity is SPN_E_INVALID.  The plan is a flat blob (image descriptors, Huffman lookup tables, quantisation
 *     tables, restart interval, entropy-data range, coefficient and output offsets) to be copied to the device as is. */
SPN_API int spn_jpeg_plan(const uint8_t* h_data, const int64_t* h_offsets, int n, void* h_plan, int64_t* plan_bytes,
                          int64_t* h_info, int64_t* h_totals);

/* Decodes every image the plan marks SPN_JPEG_OK: d_plan is the blob of spn_jpeg_plan, d_data the same bytes as h_data,
 * d_coef scratch of coef_bytes (>= h_totals[0]) bytes, d_out the luma planes (>= h_totals[1] bytes).  Two kernels on
 * `stream`: the entropy decoder (one thread per image, luma coefficients to d_coef) and the IDCT (luma planes to
 * d_out).  d_status [n] int32 receives the plan status, or the entropy decoder's error: an image whose status is not 0
 * has undefined pixels in d_out and must be decoded on the host.  1 <= n <= 65535. */
SPN_API int spn_jpeg_decode_gray(spn_ctx* ctx, const void* d_plan, const uint8_t* d_data, int n, int16_t* d_coef,
                                 int64_t coef_bytes, uint8_t* d_out, int32_t* d_status, spn_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPN_JPEG_H */
