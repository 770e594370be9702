// Shared declarations for the paacb kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "../../include/paacb.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "paacb is written for sm_100a (B200) only"
#endif

namespace paacb {

// One conv / fc layer viewed as an implicit GEMM: Y[M, N] = im2col(X)[M, K] * W[K, N].
// X is NHWC [b, H, W, C]; W is HWIO = row-major [K = R*S*C, N = Cout]; Y is NHWC [b, OH, OW, Cout].
// An fc layer is H = W = R = S = 1, C = in, N = out.
struct LayerGeom {
  int H, W, C;        // input
  int R, S, stride;   // filter
  int OH, OW, N;      // output (N = Cout)
  int K;              // R*S*C
  int in_u8;          // input is the uint8 state tensor (scaled by 1/255 on load)
  int index;          // layer index (0 = conv1); selects the profiling slot
  int64_t w_off, b_off;   // offsets into the flat parameter buffer
  int64_t in_act_off;     // offset of the input activation in the forward workspace, per sample (floats); -1: states
  int64_t out_act_off;    // offset of the output activation, per sample
};

// per-step scalars that ride along with K1 (paacb_observe_u8); all nullptr for plain paacb_preprocess_u8
struct StepScalars {
  const float* rewards_in;   // [n] device or pinned+mapped host memory (the runners' shared arrays)
  const float* over_in;      // [n] episode-over flags (0/1)
  float* rewards_out;        // [n] row t of the rollout buffers
  float* over_out;
  int over_is_reset;         // over_in[n] != 0 resets environment n's stack (needs 4 frame pairs per environment)
};

struct ResizeTables {
  uint8_t row[PAACB_OBS];
  uint8_t col[PAACB_OBS];
};

// profiling slots: one per kernel family per layer (paacb_profile_read)
enum KernelId {
  K_PREPROCESS = 0, K_FWD0 = 1, K_HEADS_FWD = 5, K_LOSS = 6, K_HEADS_BWD = 7, K_WGRAD0 = 8, K_DGRAD0 = 12,
  K_SUMSQ = 16, K_RMSPROP = 17, K_PACK = 18, K_COUNT = 19
};
constexpr int kMaxProfEvents = 8192;

// "done once per device" flag for per-device state such as cudaFuncSetAttribute (function attributes belong to the device
// that was current when they were set): one bit per device index, set/read atomically (the setup itself is idempotent).
struct DeviceOnce {
  unsigned long long mask[2] = {0ull, 0ull};
  bool done(int device) const { return (__atomic_load_n(&mask[(device >> 6) & 1], __ATOMIC_ACQUIRE) >> (device & 63)) & 1ull; }
  void mark(int device) { __atomic_fetch_or(&mask[(device >> 6) & 1], 1ull << (device & 63), __ATOMIC_RELEASE); }
};

struct TensorInfo {
  char name[40];
  int64_t offset;
  int ndim;
  int64_t shape[4];
  int64_t fan_in;
};

}  // namespace paacb

struct paacb_ctx {
  int arch;
  int num_actions;
  int device;
  int math;
  int num_sms;
  int n_layers;                 // conv layers + the hidden fc
  paacb::LayerGeom layer[4];
  int feat;                     // hidden fc width F
  int64_t act_floats_per_sample;   // sum of activation sizes of all layers
  int64_t relu1_words_per_sample;  // forward workspace, after the activations: one 32-bit word per conv1 output position, bit c = (channel c > 0)
  int64_t actor_w_off, actor_b_off, critic_w_off, critic_b_off;
  int64_t param_count;
  int n_tensors;
  paacb::TensorInfo tensor[PAACB_MAX_TENSORS];
  paacb::ResizeTables tabs;
  mutable int64_t launches;
  // optional per-kernel CUDA-event timing on the launching stream (bench.py's roofline numbers)
  mutable int prof_on;
  mutable int prof_n;
  mutable cudaEvent_t* prof_ev;       // 2 * kMaxProfEvents events, created on first enable
  mutable int* prof_kid;
  mutable double prof_ms[paacb::K_COUNT];
  mutable int64_t prof_cnt[paacb::K_COUNT];
  // context-owned workspace of the tcgen05 path: weights prepacked as swizzled tf32 operand images (hi, lo)
  uint32_t* wpack_hi;
  uint32_t* wpack_lo;
  uint32_t* wpack_d_hi;         // the transposed / per-stride-class images the data-gradient kernels read
  uint32_t* wpack_d_lo;
  // bf16-split path (PAACB_MATH_BF16X3): weights as (hi, lo) bf16 images, forward (transposed) and data-gradient layouts
  uint16_t* wb_f_hi;
  uint16_t* wb_f_lo;
  uint16_t* wb_d_hi;
  uint16_t* wb_d_lo;
  int8_t* wq_i8;                // conv1 forward: three int8 digit images of the weights [3][Cout][K] + per-channel scale
  float* wq_scale;
  // forward weight images are cached between calls: valid for the parameter buffer `fwd_img_src` until the parameters change
  // (paacb_clip_rmsprop refreshes them in-stream; paacb_params_changed() invalidates them)
  mutable int fwd_img_valid;
  mutable const float* fwd_img_src;
  // fused optimizer: self-resetting grid barrier (arrival counter + generation word in device memory, zeroed at creation)
  // and the co-resident grid size of the cooperative kernel on this context's device (-1: not queried yet)
  unsigned int* opt_counter;
  mutable int opt_fused_blocks;
  int opt_two_pass;             // PAACB_OPT_TWO_PASS=1: the two-launch optimizer (sumsq + update)
  // K1: memory type of the frame buffers seen so far (address >> 21 -> host?)
  static constexpr int kK1Cache = 8;
  mutable int k1_cache_n;
  mutable uintptr_t k1_cache_key[kK1Cache];
  mutable int k1_cache_host[kK1Cache];
  int sm_reserve;               // paacb_set_sm_reserve: SMs the persistent conv weight-gradient kernels leave free (multi-GPU)
};

namespace paacb {

void set_error(const char* fmt, ...);

#define PAACB_CHECK_ARG(cond, msg)                         \
  do {                                                     \
    if (!(cond)) {                                         \
      paacb::set_error("%s: %s", __func__, msg);           \
      return PAACB_EINVAL;                                 \
    }                                                      \
  } while (0)

void prof_drain(const paacb_ctx* ctx);

// kernel<<<grid, block, smem, st>>>(args...) with the programmatic-stream-serialization attribute (tc_ptx.cuh)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kernel(void (*kern)(KArgs...), unsigned grid, unsigned block, size_t smem, cudaStream_t st,
                                 Args&&... args) {
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// bracket a kernel launch: PAACB_LAUNCH_BEGIN(ctx, kid, st); kernel<<<...>>>(...); PAACB_LAUNCH_END(ctx, kid, st);
#define PAACB_LAUNCH_BEGIN(ctx, kid, st)                                               \
  do {                                                                                 \
    if ((ctx)->prof_on) {                                                              \
      if ((ctx)->prof_n >= paacb::kMaxProfEvents) paacb::prof_drain(ctx);              \
      cudaEventRecord((ctx)->prof_ev[2 * (ctx)->prof_n], st);                          \
    }                                                                                  \
  } while (0)

#define PAACB_LAUNCH_END(ctx, kid, st)                                                 \
  do {                                                                                 \
    cudaError_t e__ = cudaPeekAtLastError();                                           \
    if (e__ != cudaSuccess) {                                                          \
      paacb::set_error("%s: launch failed: %s", __func__, cudaGetErrorString(e__));    \
      return PAACB_ECUDA;                                                              \
    }                                                                                  \
    (ctx)->launches++;                                                                 \
    if ((ctx)->prof_on) {                                                              \
      cudaEventRecord((ctx)->prof_ev[2 * (ctx)->prof_n + 1], st);                      \
      (ctx)->prof_kid[(ctx)->prof_n++] = (kid);                                        \
    }                                                                                  \
  } while (0)

// ---- launchers implemented in the .cu files (all asynchronous on `st`) --------------------------
int launch_preprocess(const paacb_ctx* ctx, const uint8_t* frames, int pairs, const uint8_t* reset,
                      const uint8_t* prev, uint8_t* next, int64_t n, const StepScalars& sc, cudaStream_t st);

// SIMT fp32 implicit GEMMs (gemm_simt.cu)
int launch_conv_fwd_simt(const paacb_ctx* ctx, const LayerGeom& g, const void* x, const float* w, const float* bias,
                         float* y, int64_t batch, cudaStream_t st);
// dx[b,H,W,C] = (dz (*) W^T) * (x_act > 0)   (x_act == nullptr: no mask)
int launch_conv_dgrad_simt(const paacb_ctx* ctx, const LayerGeom& g, const float* dz, const float* w, const float* x_act,
                           float* dx, int64_t batch, cudaStream_t st);
// dw[K,N] += im2col(x)^T dz ; db[N] += colsum(dz)    (dw, db must be zeroed by the caller)
int launch_conv_wgrad_simt(const paacb_ctx* ctx, const LayerGeom& g, const void* x, const float* dz, float* dw, float* db,
                           int64_t batch, cudaStream_t st);

// heads (heads.cu)
// h == nullptr: the hidden activation is given as bf16-split planes (h_hi, h_lo)
int launch_heads_fwd(const paacb_ctx* ctx, const float* h, const uint16_t* h_hi, const uint16_t* h_lo, const float* wa, const float* ba, const float* wc,
                     const float* bc, int64_t batch, float* pi, float* v, const float* uniforms, const uint64_t* rng,
                     uint64_t draw, int64_t first_sample, int32_t* actions, float* onehot, cudaStream_t st);
int launch_rng_advance(const paacb_ctx* ctx, uint64_t* rng, uint64_t n, cudaStream_t st);
// dh == nullptr: dh is written as bf16-split planes (dh_hi, dh_lo) and its column sums are added to dbh
int launch_heads_bwd(const paacb_ctx* ctx, const float* h, const uint16_t* h_hi, const uint16_t* h_lo, uint16_t* dh_hi,
                     uint16_t* dh_lo, float* dbh, const float* wa, const float* wc, const float* dlogits,
                     const float* dv, int64_t batch, float* dh, float* dwa, float* dba, float* dwc, float* dbc,
                     cudaStream_t st);

// loss (loss.cu)
int launch_returns_loss_grad(const paacb_ctx* ctx, const float* rewards, const float* over, const float* values,
                             const float* boot, const int32_t* actions, const float* pi, const float* v, int T,
                             int64_t N, double gamma, float beta, float* y, float* adv, float* dlogits, float* dv,
                             float* loss, cudaStream_t st);

// optimizer (optim.cu)
int64_t optimizer_ws_floats(const paacb_ctx* ctx);
// d_lr != nullptr: the learning rate is read from device memory at run time instead of `lr`
int launch_clip_rmsprop(const paacb_ctx* ctx, float* params, float* ms, float* mom, const float* grads, float gscale,
                        float lr, const float* d_lr, float rho, float eps, float momentum, float clip, int clip_type,
                        float* norm_out, float* ws, cudaStream_t st);

int launch_grad_stats(const paacb_ctx* ctx, const float* grads, float gscale, float* ws, double* out4, cudaStream_t st);

// tcgen05 path (gemm_tc.cu); returns PAACB_EUNSUPPORTED when a layer/mode is not covered
int launch_pack_weights(const paacb_ctx* ctx, const LayerGeom& g, const float* w, cudaStream_t st);
int launch_pack_dgrad_weights(const paacb_ctx* ctx, const LayerGeom& g, const float* w, cudaStream_t st);
int launch_conv_dgrad_tc(const paacb_ctx* ctx, const LayerGeom& g, const float* dz, const float* x_act, float* dx,
                         int64_t batch, int split3, cudaStream_t st);
int launch_conv_wgrad_tc(const paacb_ctx* ctx, const LayerGeom& g, const void* x, const float* dz, float* dw, float* db,
                         int64_t batch, int split3, cudaStream_t st);
int launch_conv_fwd_tc(const paacb_ctx* ctx, const LayerGeom& g, const void* x, const float* w, const float* bias,
                       float* y, int64_t batch, int split3, cudaStream_t st);

}  // namespace paacb
