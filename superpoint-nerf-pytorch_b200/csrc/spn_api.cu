// C-ABI entry points (include/spn_b200.h): context, weight packing, encoder / head orchestration.
#include <stdarg.h>

#include <vector>

#include "spn_common.cuh"

static thread_local char g_err[1024] = "";

void spn_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" const char* spn_last_error(void) { return g_err; }
extern "C" int spn_version(void) { return 100; }

static int grow(char** buf, size_t* have, size_t need, cudaStream_t s) {
  if (need <= *have) return SPN_OK;
  // growing the workspace is the one place that synchronises (first call with a larger shape)
  SPN_CUDA(cudaStreamSynchronize(s));
  if (*buf) SPN_CUDA(cudaFree(*buf - kSpnGuard));
  *buf = nullptr;
  *have = 0;
  const size_t sz = (need + (size_t(1) << 20)) & ~((size_t(1) << 20) - 1);
  char* base = nullptr;
  cudaError_t e = cudaMalloc((void**)&base, sz + 2 * kSpnGuard);
  if (e != cudaSuccess) {
    spn_set_error("cudaMalloc(%zu) failed: %s", sz + 2 * kSpnGuard, cudaGetErrorString(e));
    return SPN_E_NOMEM;
  }
  SPN_CUDA(cudaMemsetAsync(base, kSpnGuardByte, kSpnGuard, s));                 // guard bands (spn_check_guards)
  SPN_CUDA(cudaMemsetAsync(base + kSpnGuard + sz, kSpnGuardByte, kSpnGuard, s));
  *buf = base + kSpnGuard;
  *have = sz;
  return SPN_OK;
}

int spn_ensure_ws(spn_ctx* ctx, size_t bytes, cudaStream_t s) {
  const char* old = ctx->ws;
  int rc = grow(&ctx->ws, &ctx->ws_bytes, bytes, s);
  if (ctx->ws != old) ctx->feat_mode = -1;  // feature map lived in the old workspace
  return rc;
}
int spn_ensure_aux(spn_ctx* ctx, size_t bytes, cudaStream_t s) { return grow(&ctx->aux, &ctx->aux_bytes, bytes, s); }

extern "C" int spn_create(spn_ctx** out, int device) {
  if (!out) { spn_set_error("spn_create: out is null"); return SPN_E_INVALID; }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    spn_set_error("spn_create: no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
    return SPN_E_CUDA;
  }
  SPN_REQUIRE(device >= 0 && device < n, "spn_create: device %d out of range [0,%d)", device, n);
  SpnDeviceGuard guard(device);
  cudaDeviceProp prop;
  SPN_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    spn_set_error("spn_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return SPN_E_CUDA;
  }
  spn_ctx* c = new spn_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  *out = c;
  return SPN_OK;
}

extern "C" int spn_destroy(spn_ctx* ctx) {
  if (!ctx) return SPN_OK;
  SpnDeviceGuard guard(ctx->device);
  cudaDeviceSynchronize();
  spn_tc_destroy(ctx);
  for (auto& g : ctx->grids) cudaFree(g.tab);
  for (auto& L : ctx->layers) {
    if (L.w32) cudaFree(L.w32);
    if (L.bias) cudaFree(L.bias);
    for (auto& p : L.w16) if (p) cudaFree(p);
    for (auto& p : L.w16f) if (p) cudaFree(p);
    if (L.w16x) cudaFree(L.w16x);
  }
  if (ctx->ws) cudaFree(ctx->ws - kSpnGuard);
  if (ctx->aux) cudaFree(ctx->aux - kSpnGuard);
  delete ctx;
  return SPN_OK;
}

extern "C" int spn_set_option(spn_ctx* ctx, const char* name, int value) {
  SPN_REQUIRE(ctx && name, "spn_set_option: null pointer");
  struct { const char* n; int* v; } opts[] = {{"fuse_front", &ctx->opt_fuse_front}, {"fuse_head", &ctx->opt_fuse_head},
                                               {"ws_guard", &ctx->opt_ws_guard}};
  for (auto& o : opts)
    if (!strcmp(o.n, name)) { *o.v = value; return SPN_OK; }
  spn_set_error("spn_set_option: unknown option '%s' (fuse_front, fuse_head, ws_guard)", name);
  return SPN_E_INVALID;
}

extern "C" int64_t spn_launch_count(spn_ctx* ctx) { return ctx ? ctx->launches : -1; }

namespace {
__global__ void count_guard_damage_kernel(const unsigned char* __restrict__ p, size_t n, unsigned long long* __restrict__ bad) {
  unsigned local = 0;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    local += p[i] != (unsigned char)kSpnGuardByte;
  for (int o = 16; o > 0; o >>= 1) local += __shfl_xor_sync(0xffffffffu, local, o);
  if ((threadIdx.x & 31) == 0 && local) atomicAdd(bad, (unsigned long long)local);
}
}  // namespace

// Counts the guard bytes that no longer hold the pattern: the bands around the workspace and the scratch buffer, and
// (option "ws_guard") the gaps between the regions the last encoder pass carved.  Synchronises the device.
extern "C" int spn_check_guards(spn_ctx* ctx, int64_t* h_bad) {
  SPN_REQUIRE(ctx && h_bad, "spn_check_guards: null pointer");
  SpnDeviceGuard guard(ctx->device);
  unsigned long long* d_bad = nullptr;
  SPN_CUDA(cudaDeviceSynchronize());
  SPN_CUDA(cudaMalloc((void**)&d_bad, sizeof(*d_bad)));
  SPN_CUDA(cudaMemset(d_bad, 0, sizeof(*d_bad)));
  std::vector<std::pair<const char*, size_t>> spans;
  if (ctx->ws) { spans.push_back({ctx->ws - kSpnGuard, kSpnGuard}); spans.push_back({ctx->ws + ctx->ws_bytes, kSpnGuard}); }
  if (ctx->aux) { spans.push_back({ctx->aux - kSpnGuard, kSpnGuard}); spans.push_back({ctx->aux + ctx->aux_bytes, kSpnGuard}); }
  if (ctx->opt_ws_guard)
    for (auto& g : ctx->guard_gaps) spans.push_back({g.first, g.second});
  for (auto& sp : spans) count_guard_damage_kernel<<<32, 256>>>((const unsigned char*)sp.first, sp.second, d_bad);
  unsigned long long bad = 0;
  cudaError_t e = cudaMemcpy(&bad, d_bad, sizeof(bad), cudaMemcpyDeviceToHost);
  cudaFree(d_bad);
  if (e != cudaSuccess) { spn_set_error("spn_check_guards: %s", cudaGetErrorString(e)); return SPN_E_CUDA; }
  *h_bad = (int64_t)bad;
  return SPN_OK;
}

extern "C" int spn_profile_enable(spn_ctx* ctx, int enable) {
  SPN_REQUIRE(ctx, "spn_profile_enable: null ctx");
  ctx->prof_on = enable != 0;
  return SPN_OK;
}

extern "C" int spn_profile_read(spn_ctx* ctx, float* h_ms, int64_t* h_count) {
  SPN_REQUIRE(ctx && h_ms && h_count, "spn_profile_read: null pointer");
  for (int i = 0; i < SPN_PROF_SLOTS; ++i) { h_ms[i] = 0.f; h_count[i] = 0; }
  for (auto& r : ctx->prof) {
    float ms = 0.f;
    SPN_CUDA(cudaEventSynchronize(r.b));
    SPN_CUDA(cudaEventElapsedTime(&ms, r.a, r.b));
    if (r.slot >= 0 && r.slot < SPN_PROF_SLOTS) { h_ms[r.slot] += ms; h_count[r.slot] += 1; }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  ctx->prof.clear();
  return SPN_OK;
}

extern "C" int spn_pack_weights(spn_ctx* ctx, int layer, const float* h_w, const float* h_b, const float* h_gamma,
                                const float* h_beta, const float* h_mean, const float* h_var, float eps, int cout,
                                int cin, int ksize, spn_stream stream) {
  SPN_REQUIRE(ctx && h_w, "spn_pack_weights: null pointer");
  SPN_REQUIRE(layer >= 0 && layer < SPN_NUM_LAYERS, "spn_pack_weights: layer %d out of range", layer);
  SPN_REQUIRE((ksize == 1 || ksize == 3) && cin > 0 && cout > 0, "spn_pack_weights: unsupported conv %dx%d %d->%d", ksize, ksize, cin, cout);
  cudaStream_t s = (cudaStream_t)stream;
  SpnDeviceGuard guard(ctx->device);
  const int taps = ksize * ksize;
  const int cout_pad = (cout + 15) / 16 * 16;
  // fold eval-mode BatchNorm (VGG_Backbone.py:28-29): y = (conv + b - mean) * gamma / sqrt(var + eps) + beta
  std::vector<float> wf((size_t)cout * cin * taps), bf(cout);
  std::vector<float> wpk((size_t)cin * taps * cout_pad, 0.f), bpk(cout_pad, 0.f);
  for (int co = 0; co < cout; ++co) {
    double scale = 1.0, shift = 0.0;
    const double b0 = h_b ? (double)h_b[co] : 0.0;
    if (h_gamma && h_beta && h_mean && h_var) {
      scale = (double)h_gamma[co] / sqrt((double)h_var[co] + (double)eps);
      shift = (double)h_beta[co] - (double)h_mean[co] * scale;
    }
    bf[co] = (float)(b0 * scale + shift);
    bpk[co] = bf[co];
    for (int ci = 0; ci < cin; ++ci)
      for (int t = 0; t < taps; ++t) {
        const float v = (float)((double)h_w[((size_t)co * cin + ci) * taps + t] * scale);
        wf[((size_t)co * cin + ci) * taps + t] = v;
        wpk[((size_t)ci * taps + t) * cout_pad + co] = v;
      }
  }
  SpnLayer& L = ctx->layers[layer];
  SPN_CUDA(cudaStreamSynchronize(s));
  if (L.w32) { cudaFree(L.w32); L.w32 = nullptr; }
  if (L.bias) { cudaFree(L.bias); L.bias = nullptr; }
  SPN_CUDA(cudaMalloc((void**)&L.w32, wpk.size() * sizeof(float)));
  SPN_CUDA(cudaMalloc((void**)&L.bias, bpk.size() * sizeof(float)));
  SPN_CUDA(cudaMemcpy(L.w32, wpk.data(), wpk.size() * sizeof(float), cudaMemcpyHostToDevice));
  SPN_CUDA(cudaMemcpy(L.bias, bpk.data(), bpk.size() * sizeof(float), cudaMemcpyHostToDevice));
  L.cin = cin; L.cout = cout; L.ks = ksize; L.cout_pad = cout_pad;
  ctx->feat_mode = -1;
  int rc = spn_tc_pack_layer(ctx, layer, wf.data(), bf.data(), s);
  if (rc) return rc;
  return spn_split_pack_layer(ctx, layer, wf.data(), bf.data());
}

// workspace carve-up for the strict (NCHW fp32) path, in floats
struct Fp32Plan {
  size_t bufA, bufB, feat, total;
};
static Fp32Plan fp32_plan(int B, int H, int W) {
  Fp32Plan p;
  const size_t hw = (size_t)H * W;
  p.bufA = (size_t)B * 64 * hw;      // block_1 out (largest), later layers ping-pong
  p.bufB = (size_t)B * 64 * hw / 4;  // pooled outputs
  p.feat = (size_t)B * 128 * hw / 64;
  p.total = p.bufA + p.bufB + p.feat + (size_t)B * 80 * hw / 64;  // + logits scratch
  return p;
}

static int check_image_shape(int B, int H, int W) {
  SPN_REQUIRE(B > 0 && B <= 65535, "batch %d out of range", B);
  SPN_REQUIRE(H >= 8 && W >= 8 && H % 8 == 0 && W % 8 == 0, "H and W must be positive multiples of 8 (got %dx%d)", H, W);
  return SPN_OK;
}

extern "C" int spn_encoder_forward(spn_ctx* ctx, const float* d_images, int B, int H, int W, int mode,
                                   spn_stream stream) {
  SPN_REQUIRE(ctx && d_images, "spn_encoder_forward: null pointer");
  int rc = check_image_shape(B, H, W);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  SpnDeviceGuard guard(ctx->device);
  for (int l = SPN_L_BLOCK1; l <= SPN_L_BLOCK8; ++l)
    if (!ctx->layers[l].w32) { spn_set_error("spn_encoder_forward: layer %d has no weights", l); return SPN_E_STATE; }
  if (mode == SPN_MODE_F16 || mode == SPN_MODE_BF16) {
    rc = spn_tc_encoder(ctx, d_images, B, H, W, mode, s);
    if (rc) return rc;
  } else if (mode == SPN_MODE_F16X3) {
    rc = spn_split_encoder(ctx, d_images, B, H, W, s);
    if (rc) return rc;
  } else {
    SPN_REQUIRE(mode == SPN_MODE_FP32, "spn_encoder_forward: unknown mode %d", mode);
    const Fp32Plan p = fp32_plan(B, H, W);
    rc = spn_ensure_ws(ctx, p.total * sizeof(float), s);
    if (rc) return rc;
    float* A = (float*)ctx->ws;
    float* Bq = A + p.bufA;
    float* F = Bq + p.bufB;
    // VGG_BACKBONE.forward (VGG_Backbone.py:60-71): pools after blocks 2, 4, 6
    if ((rc = spn_conv_fp32(ctx, 0, d_images, A, B, H, W, true, false, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 1, A, Bq, B, H, W, true, true, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 2, Bq, A, B, H / 2, W / 2, true, false, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 3, A, Bq, B, H / 2, W / 2, true, true, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 4, Bq, A, B, H / 4, W / 4, true, false, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 5, A, Bq, B, H / 4, W / 4, true, true, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 6, Bq, A, B, H / 8, W / 8, true, false, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, 7, A, F, B, H / 8, W / 8, true, false, s))) return rc;
    ctx->feat = F;
  }
  ctx->feat_B = B; ctx->feat_H = H; ctx->feat_W = W; ctx->feat_mode = mode;
  return SPN_OK;
}

extern "C" int spn_encoder_forward_ha(spn_ctx* ctx, const float* d_images, int n_images, const float* d_hinv, int n_h,
                                      int slot_begin, int n_slots, int H, int W, int mode, spn_stream stream) {
  SPN_REQUIRE(ctx && d_images, "spn_encoder_forward_ha: null pointer");
  SPN_REQUIRE(n_h >= 0 && (n_h == 0 || d_hinv), "spn_encoder_forward_ha: d_hinv is null");
  SPN_REQUIRE(n_images > 0 && slot_begin >= 0 && n_slots > 0 && (long long)slot_begin + n_slots <= (long long)n_images * (n_h + 1),
              "spn_encoder_forward_ha: slot range [%d,%d) outside %d images x %d slots", slot_begin, slot_begin + n_slots, n_images, n_h + 1);
  int rc = check_image_shape(n_slots, H, W);
  if (rc) return rc;
  SPN_REQUIRE(mode == SPN_MODE_F16 || mode == SPN_MODE_BF16,
              "spn_encoder_forward_ha: the fused warp+encoder exists for the tensor-core modes only (fp32: spn_warp_batch + spn_encoder_forward)");
  cudaStream_t s = (cudaStream_t)stream;
  SpnDeviceGuard guard(ctx->device);
  for (int l = SPN_L_BLOCK1; l <= SPN_L_BLOCK8; ++l)
    if (!ctx->layers[l].w32) { spn_set_error("spn_encoder_forward_ha: layer %d has no weights", l); return SPN_E_STATE; }
  // n_h == 0 still goes through the slot path (slot == image)
  rc = spn_tc_encoder_slots(ctx, d_images, n_h ? d_hinv : nullptr, n_h, slot_begin, n_slots, H, W, mode, s);
  if (rc) return rc;
  ctx->feat_B = n_slots; ctx->feat_H = H; ctx->feat_W = W; ctx->feat_mode = mode;
  return SPN_OK;
}

static int check_feat(spn_ctx* ctx, int B, int H, int W, int mode, const char* who) {
  if (ctx->feat_mode != mode || ctx->feat_B != B || ctx->feat_H != H || ctx->feat_W != W) {
    spn_set_error("%s: no feature map for B=%d H=%d W=%d mode=%d (call spn_encoder_forward first)", who, B, H, W, mode);
    return SPN_E_STATE;
  }
  return SPN_OK;
}

extern "C" int spn_detector_head_forward(spn_ctx* ctx, int B, int H, int W, int mode, const uint8_t* d_mask,
                                         float* d_logits, float* d_prob, spn_stream stream) {
  SPN_REQUIRE(ctx && d_prob, "spn_detector_head_forward: null pointer");
  int rc = check_feat(ctx, B, H, W, mode, "spn_detector_head_forward");
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  SpnDeviceGuard guard(ctx->device);
  const SpnLayer& Pb = ctx->layers[SPN_L_CONVPB];
  if (!ctx->layers[SPN_L_CONVPA].w32 || !Pb.w32) { spn_set_error("detector head has no weights"); return SPN_E_STATE; }
  SPN_REQUIRE(Pb.cout == 65, "detector head must have 65 output channels (grid_size 8), got %d", Pb.cout);
  const int Hc = H / 8, Wc = W / 8;
  float* logits = d_logits;
  if (mode == SPN_MODE_F16X3) {
    if (!logits) logits = spn_split_logits_scratch(ctx, B, H, W);
    if ((rc = spn_split_head(ctx, SPN_L_CONVPA, SPN_L_CONVPB, B, H, W, logits, s))) return rc;
  } else if (mode == SPN_MODE_FP32) {
    const Fp32Plan p = fp32_plan(B, H, W);
    float* A = (float*)ctx->ws;
    if (!logits) logits = A + p.bufA + p.bufB + p.feat;
    if ((rc = spn_conv_fp32(ctx, SPN_L_CONVPA, (const float*)ctx->feat, A, B, Hc, Wc, true, false, s))) return rc;
    if ((rc = spn_conv_fp32(ctx, SPN_L_CONVPB, A, logits, B, Hc, Wc, false, false, s))) return rc;
  } else {
    if (ctx->opt_fuse_head && ctx->layers[SPN_L_CONVPB].w16f[mode == SPN_MODE_BF16 ? 1 : 0])
      return spn_tc_detector_head_fused(ctx, B, H, W, mode, d_mask, d_logits, d_prob, s);  // convPb + softmax fused
    if (!logits) logits = spn_tc_logits_scratch(ctx, B, H, W);
    if ((rc = spn_tc_detector_head(ctx, B, H, W, mode, logits, s))) return rc;
  }
  return spn_softmax_d2s(ctx, logits, B, Hc, Wc, d_mask, d_prob, s);
}

extern "C" int spn_descriptor_head_forward(spn_ctx* ctx, int B, int H, int W, int mode, float* d_desc_raw,
                                           spn_stream stream) {
  SPN_REQUIRE(ctx && d_desc_raw, "spn_descriptor_head_forward: null pointer");
  int rc = check_feat(ctx, B, H, W, mode, "spn_descriptor_head_forward");
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  SpnDeviceGuard guard(ctx->device);
  if (!ctx->layers[SPN_L_CONVDA].w32 || !ctx->layers[SPN_L_CONVDB].w32) {
    spn_set_error("descriptor head has no weights (model_name != 'superpoint'?)");
    return SPN_E_STATE;
  }
  const int Hc = H / 8, Wc = W / 8;
  if (mode == SPN_MODE_F16X3) return spn_split_head(ctx, SPN_L_CONVDA, SPN_L_CONVDB, B, H, W, d_desc_raw, s);
  if (mode == SPN_MODE_FP32) {
    float* A = (float*)ctx->ws;
    if ((rc = spn_conv_fp32(ctx, SPN_L_CONVDA, (const float*)ctx->feat, A, B, Hc, Wc, true, false, s))) return rc;
    return spn_conv_fp32(ctx, SPN_L_CONVDB, A, d_desc_raw, B, Hc, Wc, false, false, s);
  }
  return spn_tc_descriptor_head(ctx, B, H, W, mode, d_desc_raw, s);
}

extern "C" int spn_conv_layer(spn_ctx* ctx, int layer, int mode, const float* d_in, int B, int H, int W, int relu,
                              int pool, float* d_out, spn_stream stream) {
  SPN_REQUIRE(ctx && d_in && d_out, "spn_conv_layer: null pointer");
  SPN_REQUIRE(layer >= 0 && layer < SPN_NUM_LAYERS && ctx->layers[layer].w32, "spn_conv_layer: layer %d has no weights", layer);
  SPN_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0, "spn_conv_layer: bad shape");
  SPN_REQUIRE(!pool || (H % 2 == 0 && W % 2 == 0 && ctx->layers[layer].ks == 3), "spn_conv_layer: pooling needs even H, W and a 3x3 layer");
  cudaStream_t s = (cudaStream_t)stream;
  SpnDeviceGuard guard(ctx->device);
  ctx->feat_mode = -1;  // the workspace is reused
  if (mode == SPN_MODE_FP32 || ctx->layers[layer].cin % 64 != 0) return spn_conv_fp32(ctx, layer, d_in, d_out, B, H, W, relu != 0, pool != 0, s);
  if (mode == SPN_MODE_F16X3) return spn_split_conv_layer(ctx, layer, d_in, B, H, W, relu != 0, pool != 0, d_out, s);
  SPN_REQUIRE(mode == SPN_MODE_F16 || mode == SPN_MODE_BF16, "spn_conv_layer: unknown mode %d", mode);
  return spn_tc_conv_layer(ctx, layer, mode, d_in, B, H, W, relu != 0, pool != 0, d_out, s);
}

// SuperPoint.forward + keypoint extraction in ONE call (models/SuperPoint.py:17-30 followed by what every consumer does
// with the output: nonzero(prob_heatmap_nms) and desc[:, y, x], evaluations/descriptor_evaluation.py:55-69): encoder,
// detector head, box_nms + top-k ONCE (map, pred and the row-major keypoint list from the same pass), descriptor head,
// descriptors evaluated only at the keypoints.  Everything is enqueued back to back on `stream` from one host call.
extern "C" int spn_detect_describe(spn_ctx* ctx, const float* d_images, int B, int H, int W, int mode, float nms_size, float iou,
                                   float det_thresh, int top_k, int interp, float* d_logits, float* d_prob, float* d_nms,
                                   int32_t* d_pred, int32_t* d_kp, int32_t* d_kp_count, int max_kp, float* d_desc_raw,
                                   float* d_desc_sparse, spn_stream stream) {
  SPN_REQUIRE(ctx && d_images && d_prob && d_kp && d_kp_count && max_kp > 0, "spn_detect_describe: null pointer / max_kp");
  SPN_REQUIRE((d_desc_raw != nullptr) == (d_desc_sparse != nullptr), "spn_detect_describe: d_desc_raw and d_desc_sparse go together");
  int rc = spn_encoder_forward(ctx, d_images, B, H, W, mode, stream);
  if (rc) return rc;
  if ((rc = spn_detector_head_forward(ctx, B, H, W, mode, nullptr, d_logits, d_prob, stream))) return rc;
  if (d_desc_raw && (rc = spn_descriptor_head_forward(ctx, B, H, W, mode, d_desc_raw, stream))) return rc;
  if (nms_size > 0.f) {
    if ((rc = spn_box_nms_topk(ctx, d_prob, B, H, W, nms_size, iou, det_thresh, top_k, det_thresh, d_nms, d_pred, d_kp, d_kp_count,
                               max_kp, stream))) return rc;
  } else {
    spn_set_error("spn_detect_describe: nms_size must be > 0 (the keypoint list comes from the NMS pass)");
    return SPN_E_INVALID;
  }
  if (d_desc_raw)
    return spn_sample_descriptors(ctx, d_desc_raw, B, 256, H / 8, W / 8, 8, d_kp, d_kp_count, max_kp, interp, d_desc_sparse, stream);
  return SPN_OK;
}
