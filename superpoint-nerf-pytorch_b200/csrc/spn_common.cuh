// Shared declarations for the sm_100a kernels behind include/spn_b200.h.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/spn_b200.h"

struct SpnLayer {
  int cin = 0, cout = 0, ks = 0, cout_pad = 0;
  float* w32 = nullptr;    // [cin][ks*ks][cout_pad] fp32, BN folded
  float* bias = nullptr;   // [cout_pad] fp32, BN folded
  void* w16[2] = {nullptr, nullptr};  // tcgen05 operand-B images (fp16, bf16) of the 1x1 layers and block_2, see conv_tc.cu
  void* w16f[2] = {nullptr, nullptr}; // same for the kx-folded 3x3 kernel (N = 192), see conv_fold.cu
  void* w16x = nullptr;               // (hi, lo) fp16 operand-B images of the split strict mode, see conv_split.cu
};

struct SpnProfRec {
  int slot;
  cudaEvent_t a, b;
};

struct SpnGridTab {  // kornia create_meshgrid coordinates of one image size: xs[W] then ys[H] (geometry.cu)
  int H, W;
  float* tab;
};

// Makes the context's GPU current for the duration of an entry point and restores the caller's device afterwards
// (PyTorch's current device must not change behind its back).
struct SpnDeviceGuard {
  int prev = -1;
  explicit SpnDeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev); else prev = -1;
  }
  ~SpnDeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

struct spn_ctx {
  bool prof_on = false;
  std::vector<SpnGridTab> grids;
  std::vector<SpnProfRec> prof;
  int device = 0;
  int sm_count = 148;
  SpnLayer layers[SPN_NUM_LAYERS];
  char* ws = nullptr;       // activation workspace
  size_t ws_bytes = 0;
  char* aux = nullptr;      // small scratch (nms status, ...)
  size_t aux_bytes = 0;
  // feature map state left by spn_encoder_forward
  int feat_B = 0, feat_H = 0, feat_W = 0, feat_mode = -1;
  void* feat = nullptr;     // points into ws
  int64_t launches = 0;
  void* tc = nullptr;       // tcgen05 path state (conv_tc.cu)
  // options (spn_set_option)
  int opt_fuse_front = 1;   // warp + block_1 + block_2 in one kernel (front_tc.cu)
  int opt_fuse_head = 1;    // convPb + softmax + depth-to-space in one kernel (head_tc.cu)
  int opt_ws_guard = 0;     // paint the gaps between the carved workspace regions before every encoder pass (spn_check_guards)
  std::vector<std::pair<char*, size_t>> guard_gaps;   // the gaps painted by the last pass
};

void spn_set_error(const char* fmt, ...);

#define SPN_CUDA(call)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (call);                                                                   \
    if (e_ != cudaSuccess) {                                                                   \
      spn_set_error("%s:%d %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));      \
      return SPN_E_CUDA;                                                                       \
    }                                                                                          \
  } while (0)

#define SPN_CHECK_LAUNCH(ctx)                                                                  \
  do {                                                                                         \
    (ctx)->launches++;                                                                         \
    cudaError_t e_ = cudaGetLastError();                                                       \
    if (e_ != cudaSuccess) {                                                                   \
      spn_set_error("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e_));  \
      return SPN_E_CUDA;                                                                       \
    }                                                                                          \
  } while (0)

#define SPN_REQUIRE(cond, ...)                                                                 \
  do {                                                                                         \
    if (!(cond)) {                                                                             \
      spn_set_error(__VA_ARGS__);                                                              \
      return SPN_E_INVALID;                                                                    \
    }                                                                                          \
  } while (0)

// CUDA-event bracket around a group of launches, active only after spn_profile_enable(ctx, 1)
struct SpnProfScope {
  spn_ctx* c;
  cudaStream_t s;
  SpnProfRec r;
  bool on;
  SpnProfScope(spn_ctx* ctx, int slot, cudaStream_t st) : c(ctx), s(st), on(ctx->prof_on) {
    if (!on) return;
    r.slot = slot;
    on = cudaEventCreate(&r.a) == cudaSuccess && cudaEventCreate(&r.b) == cudaSuccess;
    if (on) cudaEventRecord(r.a, s);
  }
  ~SpnProfScope() {
    if (!on) return;
    cudaEventRecord(r.b, s);
    c->prof.push_back(r);
  }
};

// Launch with programmatic stream serialization: the kernel may begin (prologue: barriers, TMEM, weights) while the
// previous kernel of the stream drains; it must execute griddepcontrol.wait before touching anything that kernel
// wrote or read.
template <typename... KArgs, typename... Args>
inline cudaError_t spn_launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t dyn, cudaStream_t s, Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = dyn;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// Both growable buffers carry a kSpnGuard-byte band of kSpnGuardByte before and after the usable range (painted when the
// buffer is allocated); the tensor-core workspace plan leaves kSpnGap bytes between its regions.  No kernel may ever
// write there: spn_check_guards counts the bytes that changed (the in-repo substitute for compute-sanitizer, which is
// closed on the GPU pool).
constexpr size_t kSpnGuard = 64 * 1024, kSpnGap = 4096;
constexpr int kSpnGuardByte = 0xA5;
int spn_ensure_ws(spn_ctx* ctx, size_t bytes, cudaStream_t s);
int spn_ensure_aux(spn_ctx* ctx, size_t bytes, cudaStream_t s);

// Host-side 16-bit conversions for packing operand images (bf16 != 0: bfloat16, else fp16), round to nearest even.
inline uint16_t to16(float f, int bf16) {
  if (bf16) {
    __nv_bfloat16 h = __float2bfloat16_rn(f);
    return *reinterpret_cast<uint16_t*>(&h);
  }
  __half h = __float2half_rn(f);
  return *reinterpret_cast<uint16_t*>(&h);
}
inline float from16(uint16_t h, int bf16) {
  if (bf16) return __bfloat162float(*reinterpret_cast<__nv_bfloat16*>(&h));
  return __half2float(*reinterpret_cast<__half*>(&h));
}

// ---- kernels implemented in the other translation units ----
int spn_conv_fp32(spn_ctx* ctx, int layer, const float* in, float* out, int B, int H, int W, bool relu, bool pool,
                  cudaStream_t s);
int spn_softmax_d2s(spn_ctx* ctx, const float* logits, int B, int Hc, int Wc, const uint8_t* mask, float* prob,
                    cudaStream_t s);

// tcgen05 path (conv_tc.cu)
int spn_tc_pack_layer(spn_ctx* ctx, int layer, const float* h_wfold, const float* h_bfold, cudaStream_t s);
int spn_tc_encoder(spn_ctx* ctx, const float* d_images, int B, int H, int W, int mode, cudaStream_t s);
int spn_tc_detector_head(spn_ctx* ctx, int B, int H, int W, int mode, float* d_logits, cudaStream_t s);
int spn_tc_descriptor_head(spn_ctx* ctx, int B, int H, int W, int mode, float* d_desc_raw, cudaStream_t s);
void spn_tc_destroy(spn_ctx* ctx);
int spn_head_pack_layer(spn_ctx* ctx, int layer, const float* h_wfold, const float* h_bfold);
int spn_launch_head_tc(spn_ctx* ctx, int mode, const void* in, int n_img, int Hc, int Wc, const uint8_t* d_mask, float* d_logits,
                       float* d_prob, cudaStream_t s);
int spn_tc_detector_head_fused(spn_ctx* ctx, int B, int H, int W, int mode, const uint8_t* d_mask, float* d_logits, float* d_prob,
                               cudaStream_t s);
// TMA map of a C8 activation tensor [n_img][C/8][H][W][8] (fp16, or bf16 if bf16 != 0) whose box is box_w pixels x
// box_h rows x 64 channels of one image; reads outside the tensor are zero-filled (the convolutions' padding).
int spn_c8_tensor_map(spn_ctx* ctx, CUtensorMap* map, const void* base, int n_img, int C, int H, int W, int box_w, int box_h,
                      int bf16);
int spn_fold_pack_layer(spn_ctx* ctx, int layer, const float* h_wfold, const float* h_bfold);
int spn_launch_conv_fold(spn_ctx* ctx, int layer, int mode, const void* in, void* out, int n_img, int H, int W, bool relu,
                         bool pool, cudaStream_t s);
int spn_tc_encoder_slots(spn_ctx* ctx, const float* d_images, const float* d_hinv, int n_h, int slot_begin, int n_slots,
                         int H, int W, int mode, cudaStream_t s);
int spn_front_tc_launch(spn_ctx* ctx, const float* d_images, const float* d_hinv, int n_h, int slot_begin, int n_slots, int H,
                        int W, int mode, const void* w1img, void* d_out, cudaStream_t s);
// split strict mode on the tensor cores (conv_split.cu)
int spn_split_pack_layer(spn_ctx* ctx, int layer, const float* w, const float* b);
int spn_split_encoder(spn_ctx* ctx, const float* d_images, int B, int H, int W, cudaStream_t s);
int spn_split_head(spn_ctx* ctx, int layer_a, int layer_b, int B, int H, int W, float* d_out, cudaStream_t s);
float* spn_split_logits_scratch(spn_ctx* ctx, int B, int H, int W);
int spn_split_conv_layer(spn_ctx* ctx, int layer, const float* d_in, int B, int H, int W, bool relu, bool pool, float* d_out, cudaStream_t s);
const float* spn_tc_block1_weights(spn_ctx* ctx);
float* spn_tc_logits_scratch(spn_ctx* ctx, int B, int H, int W);
int spn_tc_conv_layer(spn_ctx* ctx, int layer, int mode, const float* d_in, int B, int H, int W, bool relu, bool pool,
                      float* d_out, cudaStream_t s);

static inline int spn_cdiv(int a, int b) { return (a + b - 1) / b; }
