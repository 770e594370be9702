// extern "C" entry points of libpaacb.so (see include/paacb.h for the contract of each).
#include <stdarg.h>
#include <stdlib.h>
#include "common.cuh"
#include "tc2.cuh"

namespace paacb {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Pillow NEAREST column table for 160 -> 84 (floor((x + 0.5) * 160 / 84) except x = 52 -> 99, x = 73 -> 139).
static const uint8_t kDefaultCol[PAACB_OBS] = {
    0,   2,   4,   6,   8,   10,  12,  14,  16,  18,  20,  21,  23,  25,  27,  29,  31,  33,  35,  37,  39,
    40,  42,  44,  46,  48,  50,  52,  54,  56,  58,  60,  61,  63,  65,  67,  69,  71,  73,  75,  77,  79,
    80,  82,  84,  86,  88,  90,  92,  94,  96,  98,  99,  101, 103, 105, 107, 109, 111, 113, 115, 117, 119,
    120, 122, 124, 126, 128, 130, 132, 134, 136, 138, 139, 141, 143, 145, 147, 149, 151, 153, 155, 157, 159};

static void add_tensor(paacb_ctx* c, const char* name, int64_t& off, int ndim, int64_t s0, int64_t s1, int64_t s2,
                       int64_t s3, int64_t fan_in) {
  TensorInfo& t = c->tensor[c->n_tensors++];
  snprintf(t.name, sizeof(t.name), "%s", name);
  t.offset = off;
  t.ndim = ndim;
  t.shape[0] = s0; t.shape[1] = s1; t.shape[2] = s2; t.shape[3] = s3;
  t.fan_in = fan_in;
  int64_t n = 1;
  for (int i = 0; i < ndim; ++i) n *= t.shape[i];
  off += n;
}

static void add_conv(paacb_ctx* c, const char* name, int k, int cout, int stride, int& h, int& w, int& ch,
                     int64_t& poff, int64_t& aoff) {
  LayerGeom& g = c->layer[c->n_layers];
  g.H = h; g.W = w; g.C = ch; g.R = k; g.S = k; g.stride = stride;
  g.OH = (h - k) / stride + 1; g.OW = (w - k) / stride + 1; g.N = cout;
  g.K = k * k * ch;
  g.in_u8 = (c->n_layers == 0);
  g.index = c->n_layers;
  g.in_act_off = (c->n_layers == 0) ? -1 : c->layer[c->n_layers - 1].out_act_off;
  g.out_act_off = aoff;
  aoff += (int64_t)g.OH * g.OW * g.N;
  char nm[40];
  g.w_off = poff;
  snprintf(nm, sizeof(nm), "%s_weights", name);
  add_tensor(c, nm, poff, 4, k, k, ch, cout, g.K);
  g.b_off = poff;
  snprintf(nm, sizeof(nm), "%s_biases", name);
  add_tensor(c, nm, poff, 1, cout, 0, 0, 0, g.K);
  h = g.OH; w = g.OW; ch = cout;
  c->n_layers++;
}

// Fold the recorded (start, stop) event pairs into the per-kernel accumulators.  Synchronises on the
// last recorded event, so it is only called from paacb_profile_read or when the event pool is full.
void prof_drain(const paacb_ctx* ctx) {
  if (ctx->prof_n == 0) return;
  cudaEventSynchronize(ctx->prof_ev[2 * (ctx->prof_n - 1) + 1]);
  for (int i = 0; i < ctx->prof_n; ++i) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->prof_ev[2 * i], ctx->prof_ev[2 * i + 1]) == cudaSuccess) {
      ctx->prof_ms[ctx->prof_kid[i]] += ms;
      ctx->prof_cnt[ctx->prof_kid[i]]++;
    }
  }
  cudaGetLastError();
  ctx->prof_n = 0;
}

// Every launch goes to the CURRENT device; kernel attributes, tensor maps and the context's own buffers belong to
// ctx->device.  A mismatch would silently run on the wrong GPU, so it is an argument error.
int check_current_device(const paacb_ctx* ctx, const char* who) {
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess) {
    cudaGetLastError();
    set_error("%s: cudaGetDevice failed", who);
    return PAACB_ECUDA;
  }
  if (cur != ctx->device) {
    set_error("%s: the current CUDA device is %d but the context was created for device %d (cudaSetDevice first)", who, cur,
              ctx->device);
    return PAACB_EINVAL;
  }
  return PAACB_OK;
}
#define PAACB_CHECK_DEVICE(ctx)                                              \
  do {                                                                       \
    const int rc__ = paacb::check_current_device((ctx), __func__);           \
    if (rc__ != PAACB_OK) return rc__;                                       \
  } while (0)

}  // namespace paacb

using namespace paacb;

extern "C" {

int paacb_version(void) { return PAACB_VERSION; }
const char* paacb_last_error(void) { return g_err; }

int paacb_create(paacb_ctx** out, int arch, int num_actions, int device) {
  PAACB_CHECK_ARG(out != nullptr, "out is NULL");
  PAACB_CHECK_ARG(arch == PAACB_ARCH_NIPS || arch == PAACB_ARCH_NATURE, "arch must be PAACB_ARCH_NIPS or PAACB_ARCH_NATURE");
  PAACB_CHECK_ARG(num_actions >= 2 && num_actions <= PAACB_MAX_ACTIONS, "num_actions out of range [2, 18]");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    set_error("paacb_create: no CUDA device (this library has no CPU path)");
    return PAACB_ECUDA;
  }
  PAACB_CHECK_ARG(device >= 0 && device < ndev, "device index out of range");
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) { set_error("cudaGetDeviceProperties failed"); return PAACB_ECUDA; }
  if (prop.major != 10) {
    set_error("paacb_create: device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    return PAACB_EUNSUPPORTED;
  }
  paacb_ctx* c = new paacb_ctx();
  memset(c, 0, sizeof(*c));
  c->arch = arch; c->num_actions = num_actions; c->device = device; c->math = PAACB_MATH_FP32;
  c->num_sms = prop.multiProcessorCount;
  c->opt_fused_blocks = -1;
  const char* tp = getenv("PAACB_OPT_TWO_PASS");
  c->opt_two_pass = (tp != nullptr) ? atoi(tp) : 0;
  int h = PAACB_OBS, w = PAACB_OBS, ch = PAACB_STACK;
  int64_t poff = 0, aoff = 0;
  if (arch == PAACB_ARCH_NIPS) {                       // networks.py:145-149
    add_conv(c, "conv1", 8, 16, 4, h, w, ch, poff, aoff);
    add_conv(c, "conv2", 4, 32, 2, h, w, ch, poff, aoff);
  } else {                                             // networks.py:161-167
    add_conv(c, "conv1", 8, 32, 4, h, w, ch, poff, aoff);
    add_conv(c, "conv2", 4, 64, 2, h, w, ch, poff, aoff);
    add_conv(c, "conv3", 3, 64, 1, h, w, ch, poff, aoff);
  }
  {  // hidden fc over the (h, w, c)-flattened activation (networks.py:6-9)
    const int fin = h * w * ch;
    const int fout = (arch == PAACB_ARCH_NIPS) ? 256 : 512;
    LayerGeom& g = c->layer[c->n_layers];
    g.H = 1; g.W = 1; g.C = fin; g.R = 1; g.S = 1; g.stride = 1; g.OH = 1; g.OW = 1; g.N = fout; g.K = fin;
    g.in_u8 = 0;
    g.index = c->n_layers;
    g.in_act_off = c->layer[c->n_layers - 1].out_act_off;
    g.out_act_off = aoff;
    aoff += fout;
    const char* nm = (arch == PAACB_ARCH_NIPS) ? "fc3" : "fc4";
    char buf[40];
    g.w_off = poff;
    snprintf(buf, sizeof(buf), "%s_weights", nm);
    add_tensor(c, buf, poff, 2, fin, fout, 0, 0, fin);
    g.b_off = poff;
    snprintf(buf, sizeof(buf), "%s_biases", nm);
    add_tensor(c, buf, poff, 1, fout, 0, 0, 0, fin);
    c->n_layers++;
    c->feat = fout;
  }
  c->act_floats_per_sample = aoff;
  c->relu1_words_per_sample = (int64_t)c->layer[0].OH * c->layer[0].OW;
  c->actor_w_off = poff;  add_tensor(c, "actor_output_weights", poff, 2, c->feat, num_actions, 0, 0, c->feat);
  c->actor_b_off = poff;  add_tensor(c, "actor_output_biases", poff, 1, num_actions, 0, 0, 0, c->feat);
  c->critic_w_off = poff; add_tensor(c, "critic_output_weights", poff, 2, c->feat, 1, 0, 0, c->feat);
  c->critic_b_off = poff; add_tensor(c, "critic_output_biases", poff, 1, 1, 0, 0, 0, c->feat);
  c->param_count = poff;
  for (int y = 0; y < PAACB_OBS; ++y) {
    c->tabs.row[y] = (uint8_t)(((2 * y + 1) * 5) / 4);   // floor((y + 0.5) * 2.5)
    c->tabs.col[y] = kDefaultCol[y];
  }
  {  // the grid-barrier counter of the fused optimizer kernel (context-owned, like the weight images)
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(device);
    if (cudaMalloc(&c->opt_counter, 256) == cudaSuccess) {
      cudaMemset(c->opt_counter, 0, 256);
    } else {
      cudaGetLastError();
      c->opt_counter = nullptr;          // falls back to the two-launch optimizer
    }
    cudaSetDevice(cur);
  }
  *out = c;
  return PAACB_OK;
}

int paacb_destroy(paacb_ctx* ctx) {
  if (ctx == nullptr) return PAACB_OK;
  if (ctx->prof_ev != nullptr) {
    for (int i = 0; i < 2 * kMaxProfEvents; ++i) cudaEventDestroy(ctx->prof_ev[i]);
    delete[] ctx->prof_ev;
    delete[] ctx->prof_kid;
  }
  if (ctx->opt_counter != nullptr) cudaFree(ctx->opt_counter);
  if (ctx->wpack_hi != nullptr) cudaFree(ctx->wpack_hi);
  if (ctx->wpack_lo != nullptr) cudaFree(ctx->wpack_lo);
  if (ctx->wpack_d_hi != nullptr) cudaFree(ctx->wpack_d_hi);
  if (ctx->wpack_d_lo != nullptr) cudaFree(ctx->wpack_d_lo);
  if (ctx->wb_f_hi != nullptr) cudaFree(ctx->wb_f_hi);
  if (ctx->wb_f_lo != nullptr) cudaFree(ctx->wb_f_lo);
  if (ctx->wb_d_hi != nullptr) cudaFree(ctx->wb_d_hi);
  if (ctx->wb_d_lo != nullptr) cudaFree(ctx->wb_d_lo);
  if (ctx->wq_i8 != nullptr) cudaFree(ctx->wq_i8);
  if (ctx->wq_scale != nullptr) cudaFree(ctx->wq_scale);
  delete ctx;
  return PAACB_OK;
}

int paacb_profile_enable(paacb_ctx* ctx, int on) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  if (on && ctx->prof_ev == nullptr) {
    ctx->prof_ev = new cudaEvent_t[2 * kMaxProfEvents];
    ctx->prof_kid = new int[kMaxProfEvents];
    for (int i = 0; i < 2 * kMaxProfEvents; ++i) {
      if (cudaEventCreate(&ctx->prof_ev[i]) != cudaSuccess) { set_error("cudaEventCreate failed"); return PAACB_ECUDA; }
    }
  }
  if (!on) prof_drain(ctx);
  ctx->prof_on = on ? 1 : 0;
  return PAACB_OK;
}

int paacb_profile_reset(paacb_ctx* ctx) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  prof_drain(ctx);
  for (int i = 0; i < K_COUNT; ++i) { ctx->prof_ms[i] = 0.0; ctx->prof_cnt[i] = 0; }
  return PAACB_OK;
}

int paacb_profile_slots(void) { return K_COUNT; }

int paacb_profile_read(const paacb_ctx* ctx, int slot, char* name, int name_cap, double* total_ms, int64_t* launches) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  PAACB_CHECK_ARG(slot >= 0 && slot < K_COUNT, "slot out of range");
  prof_drain(ctx);
  if (name && name_cap > 0) {
    const char* base = "";
    int layer = -1;
    if (slot == K_PREPROCESS) base = "preprocess_u8";
    else if (slot < K_HEADS_FWD) { base = "fwd"; layer = slot - K_FWD0; }
    else if (slot == K_HEADS_FWD) base = "heads_fwd";
    else if (slot == K_LOSS) base = "returns_loss_grad";
    else if (slot == K_HEADS_BWD) base = "heads_bwd";
    else if (slot < K_DGRAD0) { base = "wgrad"; layer = slot - K_WGRAD0; }
    else if (slot < K_SUMSQ) { base = "dgrad"; layer = slot - K_DGRAD0; }
    else if (slot == K_SUMSQ) base = "grad_sumsq";
    else if (slot == K_RMSPROP) base = "clip_rmsprop";
    else base = "pack_weights";
    if (layer >= 0) {
      if (layer < ctx->n_layers) {
        char lname[40];
        snprintf(lname, sizeof(lname), "%s", ctx->tensor[2 * layer].name);      // "<layer>_weights"
        char* us = strrchr(lname, '_');
        if (us) *us = 0;
        snprintf(name, (size_t)name_cap, "%s_%s", lname, base);
      } else {
        snprintf(name, (size_t)name_cap, "unused");
      }
    } else {
      snprintf(name, (size_t)name_cap, "%s", base);
    }
  }
  if (total_ms) *total_ms = ctx->prof_ms[slot];
  if (launches) *launches = ctx->prof_cnt[slot];
  return PAACB_OK;
}

int paacb_set_math(paacb_ctx* ctx, int math_mode) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  PAACB_CHECK_ARG(math_mode == PAACB_MATH_FP32 || math_mode == PAACB_MATH_TF32X3 || math_mode == PAACB_MATH_TF32 ||
                  math_mode == PAACB_MATH_BF16X3, "unknown math mode");
  ctx->fwd_img_valid = 0;
  if (math_mode == PAACB_MATH_BF16X3) {
    if (!bf16x3_supported(ctx)) {
      set_error("paacb_set_math: PAACB_MATH_BF16X3 does not cover this architecture (use PAACB_MATH_TF32X3)");
      return PAACB_EUNSUPPORTED;
    }
    if (ctx->wb_f_hi == nullptr) {
      int cur = 0;
      cudaGetDevice(&cur);
      cudaSetDevice(ctx->device);
      const size_t bytes = (size_t)ctx->param_count * sizeof(uint16_t) + 256;
      const cudaError_t e1 = cudaMalloc(&ctx->wb_f_hi, bytes);
      const cudaError_t e2 = cudaMalloc(&ctx->wb_f_lo, bytes);
      const cudaError_t e3 = cudaMalloc(&ctx->wb_d_hi, bytes);
      const cudaError_t e4 = cudaMalloc(&ctx->wb_d_lo, bytes);
      const cudaError_t e5 = cudaMalloc(&ctx->wq_i8, (size_t)3 * ctx->layer[0].N * ctx->layer[0].K);
      const cudaError_t e6 = cudaMalloc(&ctx->wq_scale, (size_t)ctx->layer[0].N * sizeof(float));
      cudaSetDevice(cur);
      if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess || e5 != cudaSuccess || e6 != cudaSuccess) {
        cudaGetLastError();
        set_error("paacb_set_math: cannot allocate %zu bytes for the bf16 weight images", 4 * bytes);
        return PAACB_ECUDA;
      }
    }
    ctx->math = math_mode;
    return PAACB_OK;
  }
  if (math_mode != PAACB_MATH_FP32 && ctx->wpack_hi == nullptr) {
    // context-owned workspace (like a TMA descriptor): the prepacked tf32 weight images, 2 x P words
    int cur = 0;
    cudaGetDevice(&cur);
    cudaSetDevice(ctx->device);
    const size_t bytes = (size_t)ctx->param_count * sizeof(uint32_t);
    const cudaError_t e1 = cudaMalloc(&ctx->wpack_hi, bytes);
    const cudaError_t e2 = cudaMalloc(&ctx->wpack_lo, bytes);
    const cudaError_t e3 = cudaMalloc(&ctx->wpack_d_hi, bytes);
    const cudaError_t e4 = cudaMalloc(&ctx->wpack_d_lo, bytes);
    if (ctx->wq_i8 == nullptr && ctx->layer[0].N == 16) {      // NIPS: the first layer runs on the int8 pipe (tc2_conv1.cu)
      if (cudaMalloc(&ctx->wq_i8, (size_t)3 * ctx->layer[0].N * ctx->layer[0].K) != cudaSuccess ||
          cudaMalloc(&ctx->wq_scale, (size_t)ctx->layer[0].N * sizeof(float)) != cudaSuccess) {
        cudaGetLastError();
        ctx->wq_i8 = nullptr;                                    // falls back to the tf32 kernel
      }
    }
    cudaSetDevice(cur);
    if (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess || e4 != cudaSuccess) {
      cudaGetLastError();
      set_error("paacb_set_math: cannot allocate %zu bytes for packed weights", 2 * bytes);
      return PAACB_ECUDA;
    }
  }
  ctx->math = math_mode;
  return PAACB_OK;
}

int paacb_get_math(const paacb_ctx* ctx) { return ctx ? ctx->math : PAACB_EINVAL; }

int paacb_set_sm_reserve(paacb_ctx* ctx, int n_sms) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  PAACB_CHECK_ARG(n_sms >= 0 && n_sms < ctx->num_sms, "n_sms out of range");
  ctx->sm_reserve = n_sms;
  return PAACB_OK;
}

int paacb_params_changed(paacb_ctx* ctx) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  ctx->fwd_img_valid = 0;
  ctx->fwd_img_src = nullptr;
  return PAACB_OK;
}

// the operand images of the forward for the parameters at d_params: bf16 hi/lo transposes + conv1 int8 digits (bf16x3), or
// the pre-swizzled tf32 images (+ NIPS conv1 int8 digits) of the tf32 modes.  Cached in the context between calls.
static int pack_forward_images(const paacb_ctx* ctx, const float* d_params, cudaStream_t st) {
  if (ctx->math == PAACB_MATH_BF16X3) {
    // forward AND data-gradient images: the backward then starts with no pack kernel in front of its first GEMM (the
    // kernels of a backward are launched as programmatic dependents of each other and load their weights early)
    const int rc = launch_pack_bf16_weights(ctx, d_params, st);
    return rc != PAACB_OK ? rc : launch_pack_bf16_dgrad_weights(ctx, d_params, st);
  }
  if (ctx->math == PAACB_MATH_FP32) return PAACB_OK;
  for (int l = 0; l < ctx->n_layers; ++l) {
    const LayerGeom& g = ctx->layer[l];
    const int rc = launch_pack_weights(ctx, g, d_params + g.w_off, st);
    if (rc != PAACB_OK) return rc;
  }
  if (ctx->layer[0].N == 16 && ctx->wq_i8 != nullptr) {          // NIPS conv1 runs on the int8 pipe (tc2_conv1.cu)
    const int rc = launch_pack_conv1_i8(ctx, d_params, st);
    if (rc != PAACB_OK && rc != PAACB_EUNSUPPORTED) return rc;
  }
  return PAACB_OK;
}
static int ensure_forward_images(const paacb_ctx* ctx, const float* d_params, cudaStream_t st) {
  if (ctx->fwd_img_valid && ctx->fwd_img_src == d_params) return PAACB_OK;
  const int rc = pack_forward_images(ctx, d_params, st);
  if (rc == PAACB_OK) {
    ctx->fwd_img_valid = 1;
    ctx->fwd_img_src = d_params;
  }
  return rc;
}

int paacb_set_resize_tables(paacb_ctx* ctx, const int32_t* row84, const int32_t* col84) {
  PAACB_CHECK_ARG(ctx && row84 && col84, "NULL argument");
  for (int i = 0; i < PAACB_OBS; ++i) {
    PAACB_CHECK_ARG(row84[i] >= 0 && row84[i] < PAACB_FRAME_H && col84[i] >= 0 && col84[i] < PAACB_FRAME_W,
                    "table entry out of range");
    ctx->tabs.row[i] = (uint8_t)row84[i];
    ctx->tabs.col[i] = (uint8_t)col84[i];
  }
  return PAACB_OK;
}

int64_t paacb_param_count(const paacb_ctx* ctx) { return ctx ? ctx->param_count : PAACB_EINVAL; }
int paacb_num_tensors(const paacb_ctx* ctx) { return ctx ? ctx->n_tensors : PAACB_EINVAL; }

int paacb_tensor_info(const paacb_ctx* ctx, int index, char* name, int name_cap, int64_t* offset, int* ndim,
                      int64_t shape[4], int64_t* fan_in) {
  PAACB_CHECK_ARG(ctx != nullptr, "ctx is NULL");
  PAACB_CHECK_ARG(index >= 0 && index < ctx->n_tensors, "tensor index out of range");
  const TensorInfo& t = ctx->tensor[index];
  if (name && name_cap > 0) snprintf(name, (size_t)name_cap, "%s", t.name);
  if (offset) *offset = t.offset;
  if (ndim) *ndim = t.ndim;
  if (shape) for (int i = 0; i < 4; ++i) shape[i] = t.shape[i];
  if (fan_in) *fan_in = t.fan_in;
  return PAACB_OK;
}

int64_t paacb_forward_workspace_floats(const paacb_ctx* ctx, int64_t batch) {
  // activations as fp32, or as two bf16 planes per tensor (PAACB_MATH_BF16X3): the same bytes; then the ReLU bit mask of the
  // first conv layer (one word per output position; written by conv1's forward, read by conv2's data gradient)
  if (ctx == nullptr) return PAACB_EINVAL;
  return (ctx->act_floats_per_sample + (ctx->math == PAACB_MATH_BF16X3 ? ctx->relu1_words_per_sample : 0)) * batch;
}
int64_t paacb_backward_workspace_floats(const paacb_ctx* ctx, int64_t batch) {
  return ctx ? ctx->act_floats_per_sample * batch : PAACB_EINVAL;
}
int64_t paacb_optimizer_workspace_floats(const paacb_ctx* ctx) { return ctx ? optimizer_ws_floats(ctx) : PAACB_EINVAL; }
int64_t paacb_launch_count(const paacb_ctx* ctx) { return ctx ? ctx->launches : PAACB_EINVAL; }

static int preprocess_impl(const paacb_ctx* ctx, const uint8_t* d_frames, int pairs_per_env, const uint8_t* d_reset,
                           const uint8_t* d_prev, uint8_t* d_next, int64_t n_envs, const StepScalars& sc, paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_frames && d_prev && d_next, "NULL argument");
  PAACB_CHECK_DEVICE(ctx);
  PAACB_CHECK_ARG(pairs_per_env == 1 || pairs_per_env == PAACB_STACK, "pairs_per_env must be 1 or 4");
  PAACB_CHECK_ARG((d_reset == nullptr && !(sc.over_in != nullptr && sc.over_is_reset)) || pairs_per_env == PAACB_STACK,
                  "reset flags need pairs_per_env == 4");
  PAACB_CHECK_ARG(n_envs >= 0 && n_envs < (1LL << 31), "n_envs out of range");
  PAACB_CHECK_ARG(((uintptr_t)d_frames & 15) == 0 && ((uintptr_t)d_prev & 15) == 0 && ((uintptr_t)d_next & 15) == 0,
                  "buffers must be 16-byte aligned");
  return launch_preprocess(ctx, d_frames, pairs_per_env, d_reset, d_prev, d_next, n_envs, sc, (cudaStream_t)stream);
}

int paacb_preprocess_u8(const paacb_ctx* ctx, const uint8_t* d_frames, int pairs_per_env, const uint8_t* d_reset,
                        const uint8_t* d_prev, uint8_t* d_next, int64_t n_envs, paacb_stream stream) {
  const StepScalars none = {nullptr, nullptr, nullptr, nullptr, 0};
  return preprocess_impl(ctx, d_frames, pairs_per_env, d_reset, d_prev, d_next, n_envs, none, stream);
}

int paacb_observe_u8(const paacb_ctx* ctx, const uint8_t* d_frames, int pairs_per_env, const uint8_t* d_reset,
                     const uint8_t* d_prev, uint8_t* d_next, int64_t n_envs, const float* d_rewards_in,
                     const float* d_over_in, float* d_rewards_out, float* d_over_out, int over_is_reset, paacb_stream stream) {
  PAACB_CHECK_ARG(d_rewards_in && d_over_in && d_rewards_out && d_over_out, "NULL reward / episode-over buffer");
  const StepScalars sc = {d_rewards_in, d_over_in, d_rewards_out, d_over_out, over_is_reset ? 1 : 0};
  return preprocess_impl(ctx, d_frames, pairs_per_env, d_reset, d_prev, d_next, n_envs, sc, stream);
}

static int run_layer_fwd(const paacb_ctx* ctx, int l, const float* d_params, const uint8_t* d_states, int64_t batch,
                         float* ws, const WsSlice& slice, cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  const void* x = (l == 0) ? (const void*)d_states
                           : (const void*)(ws + g.in_act_off * slice.cap + slice.first * (int64_t)g.H * g.W * g.C);
  float* y = ws + g.out_act_off * slice.cap + slice.first * (int64_t)g.OH * g.OW * g.N;
  if (ctx->math != PAACB_MATH_FP32 && l == 0 && g.N == 16 && ctx->wq_i8 != nullptr) {
    // NIPS conv1: uint8 pixels x int8 weight digits (tc2_conv1.cu; the digit image is part of the cached forward images)
    const int rc = launch_conv1_fwd_i8_f32(ctx, d_params, d_states, y, batch, st);
    if (rc != PAACB_EUNSUPPORTED) return rc;
  }
  if (ctx->math != PAACB_MATH_FP32) {
    const int rc = launch_conv_fwd_tc(ctx, g, x, d_params + g.w_off, d_params + g.b_off, y, batch,
                                      ctx->math == PAACB_MATH_TF32X3, st);
    if (rc != PAACB_EUNSUPPORTED) return rc;
  }
  return launch_conv_fwd_simt(ctx, g, x, d_params + g.w_off, d_params + g.b_off, y, batch, st);
}

static int forward_impl(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch, float* d_fwd_ws,
                        int64_t ws_capacity, int64_t ws_first, float* d_pi, float* d_v, const float* d_uniforms,
                        const uint64_t* d_rng, uint64_t draw, int64_t first_sample, int32_t* d_actions, float* d_onehot,
                        paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_params && d_states && d_fwd_ws && d_pi && d_v, "NULL argument");
  PAACB_CHECK_DEVICE(ctx);
  PAACB_CHECK_ARG(batch >= 0 && batch * (int64_t)ctx->layer[0].OH * ctx->layer[0].OW < (1LL << 40), "batch out of range");
  PAACB_CHECK_ARG(ws_first >= 0 && ws_capacity >= 0 && ws_first + batch <= ws_capacity,
                  "samples [ws_first, ws_first + batch) must lie inside the workspace capacity");
  PAACB_CHECK_ARG(d_uniforms == nullptr || d_rng == nullptr, "give injected uniforms OR a device rng state, not both");
  // every per-sample tensor is a multiple of 32 elements (Nature: of 64), so any sample offset keeps the planes 16-byte aligned
  const WsSlice slice = {ws_capacity, ws_first};
  PAACB_CHECK_ARG(((uintptr_t)d_params & 15) == 0 && ((uintptr_t)d_states & 15) == 0 && ((uintptr_t)d_fwd_ws & 15) == 0,
                  "params / states / workspace must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (batch == 0) return PAACB_OK;
  int rc = ensure_forward_images(ctx, d_params, st);
  if (rc != PAACB_OK) return rc;
  if (ctx->math == PAACB_MATH_BF16X3) {
    const int L = ctx->n_layers;
    for (int l = 0; l < L - 1 && rc == PAACB_OK; ++l) rc = launch_conv_fwd_bf16(ctx, l, d_params, d_states, d_fwd_ws, batch, slice, st);
    if (rc == PAACB_OK) rc = launch_fc_fwd_bf16(ctx, L - 1, d_params, d_fwd_ws, batch, slice, st);
    if (rc != PAACB_OK) return rc;
    const Planes hp = layer_planes(d_fwd_ws, ctx->layer[L - 1].out_act_off, ctx->feat, slice);
    return launch_heads_fwd(ctx, nullptr, reinterpret_cast<const uint16_t*>(hp.hi), reinterpret_cast<const uint16_t*>(hp.lo),
                            d_params + ctx->actor_w_off, d_params + ctx->actor_b_off, d_params + ctx->critic_w_off,
                            d_params + ctx->critic_b_off, batch, d_pi, d_v, d_uniforms, d_rng, draw, first_sample, d_actions,
                            d_onehot, st);
  }
  for (int l = 0; l < ctx->n_layers; ++l) {
    rc = run_layer_fwd(ctx, l, d_params, d_states, batch, d_fwd_ws, slice, st);
    if (rc != PAACB_OK) return rc;
  }
  const float* h = d_fwd_ws + ctx->layer[ctx->n_layers - 1].out_act_off * slice.cap + slice.first * (int64_t)ctx->feat;
  return launch_heads_fwd(ctx, h, nullptr, nullptr, d_params + ctx->actor_w_off, d_params + ctx->actor_b_off,
                          d_params + ctx->critic_w_off, d_params + ctx->critic_b_off, batch, d_pi, d_v, d_uniforms, d_rng, draw,
                          first_sample, d_actions, d_onehot, st);
}

int paacb_policy_forward(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                         float* d_fwd_ws, float* d_pi, float* d_v, const float* d_uniforms, int32_t* d_actions,
                         float* d_onehot, paacb_stream stream) {
  return forward_impl(ctx, d_params, d_states, batch, d_fwd_ws, batch, 0, d_pi, d_v, d_uniforms, nullptr, 0, 0, d_actions,
                      d_onehot, stream);
}

int paacb_policy_forward_at(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                            float* d_fwd_ws, int64_t ws_capacity, int64_t ws_first, float* d_pi, float* d_v,
                            const float* d_uniforms, int32_t* d_actions, float* d_onehot, paacb_stream stream) {
  return forward_impl(ctx, d_params, d_states, batch, d_fwd_ws, ws_capacity, ws_first, d_pi, d_v, d_uniforms, nullptr, 0, 0,
                      d_actions, d_onehot, stream);
}

int paacb_policy_forward_sample(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                                float* d_fwd_ws, int64_t ws_capacity, int64_t ws_first, float* d_pi, float* d_v,
                                const uint64_t* d_rng, uint64_t draw_index, int64_t first_sample, int32_t* d_actions,
                                float* d_onehot, paacb_stream stream) {
  PAACB_CHECK_ARG(d_rng != nullptr && (d_actions != nullptr || d_onehot != nullptr), "NULL rng state / no output for the actions");
  PAACB_CHECK_ARG(((uintptr_t)d_rng & 7) == 0 && first_sample >= 0, "rng state must be 8-byte aligned, first_sample >= 0");
  return forward_impl(ctx, d_params, d_states, batch, d_fwd_ws, ws_capacity, ws_first, d_pi, d_v, nullptr, d_rng, draw_index,
                      first_sample, d_actions, d_onehot, stream);
}

int paacb_rng_advance(const paacb_ctx* ctx, uint64_t* d_rng, uint64_t n, paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_rng && ((uintptr_t)d_rng & 7) == 0, "NULL / misaligned rng state");
  PAACB_CHECK_DEVICE(ctx);
  return launch_rng_advance(ctx, d_rng, n, (cudaStream_t)stream);
}

int paacb_returns_loss_grad(const paacb_ctx* ctx, const float* d_rewards, const float* d_episode_over,
                            const float* d_values, const float* d_bootstrap_v, const int32_t* d_actions,
                            const float* d_pi, const float* d_v, int t_max, int64_t n_envs, double gamma,
                            float entropy_beta, float* d_y, float* d_adv, float* d_dlogits, float* d_dv,
                            float* d_loss, paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_rewards && d_episode_over && d_values && d_bootstrap_v && d_actions && d_pi && d_v &&
                  d_y && d_adv && d_dlogits && d_dv && d_loss, "NULL argument");
  PAACB_CHECK_ARG(t_max >= 1 && n_envs >= 0, "t_max / n_envs out of range");
  PAACB_CHECK_DEVICE(ctx);
  return launch_returns_loss_grad(ctx, d_rewards, d_episode_over, d_values, d_bootstrap_v, d_actions, d_pi, d_v,
                                  t_max, n_envs, gamma, entropy_beta, d_y, d_adv, d_dlogits, d_dv, d_loss,
                                  (cudaStream_t)stream);
}

// bf16x3: head gradients, every data gradient (they also produce the conv / fc BIAS gradients) and the fc weight gradient
static int backward_bf16_tail(const paacb_ctx* ctx, const float* d_params, const float* d_fwd_ws, const float* d_dlogits,
                              const float* d_dv, float* d_bwd_ws, float* d_grads, int64_t batch, cudaStream_t st) {
  const int L = ctx->n_layers;
  {
    const Planes hp = layer_planes(const_cast<float*>(d_fwd_ws), ctx->layer[L - 1].out_act_off, ctx->feat, batch);
    const Planes dhp = layer_planes(d_bwd_ws, ctx->layer[L - 1].out_act_off, ctx->feat, batch);
    int rc = launch_heads_bwd(ctx, nullptr, reinterpret_cast<const uint16_t*>(hp.hi), reinterpret_cast<const uint16_t*>(hp.lo),
                              reinterpret_cast<uint16_t*>(dhp.hi), reinterpret_cast<uint16_t*>(dhp.lo),
                              d_grads + ctx->layer[L - 1].b_off, d_params + ctx->actor_w_off, d_params + ctx->critic_w_off,
                              d_dlogits, d_dv, batch, nullptr, d_grads + ctx->actor_w_off, d_grads + ctx->actor_b_off,
                              d_grads + ctx->critic_w_off, d_grads + ctx->critic_b_off, st);
    // (the data-gradient images of the weights are cached with the forward images; the forward that produced d_fwd_ws made them)
    if (rc == PAACB_OK && !(ctx->fwd_img_valid && ctx->fwd_img_src == d_params)) rc = launch_pack_bf16_dgrad_weights(ctx, d_params, st);
    // data gradients first (they produce the dZ planes and the bias gradients), then the weight gradients
    if (rc == PAACB_OK) rc = launch_fc_dgrad_bf16(ctx, L - 1, d_fwd_ws, d_bwd_ws, d_grads, batch, st);
    for (int l = L - 2; l >= 1 && rc == PAACB_OK; --l) rc = launch_conv_dgrad_bf16(ctx, l, d_fwd_ws, d_bwd_ws, d_grads, batch, st);
    if (rc == PAACB_OK) rc = launch_fc_wgrad_bf16(ctx, L - 1, d_fwd_ws, d_bwd_ws, d_grads, batch, st);
    return rc;
  }
}

// fp32 / tf32 modes, layer by layer from the top: `do_tail` = heads + the hidden fc layer (its weight gradient and the data
// gradient below it), `do_head` = the conv layers
static int backward_generic(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                            const float* d_fwd_ws, const float* d_dlogits, const float* d_dv, float* d_bwd_ws, float* d_grads,
                            bool do_tail, bool do_head, cudaStream_t st) {
  const int L = ctx->n_layers;
  int rc = PAACB_OK;
  const float* h = d_fwd_ws + ctx->layer[L - 1].out_act_off * batch;
  float* dh = d_bwd_ws + ctx->layer[L - 1].out_act_off * batch;
  if (do_tail) {
    rc = launch_heads_bwd(ctx, h, nullptr, nullptr, nullptr, nullptr, nullptr, d_params + ctx->actor_w_off, d_params + ctx->critic_w_off, d_dlogits, d_dv, batch,
                          dh, d_grads + ctx->actor_w_off, d_grads + ctx->actor_b_off, d_grads + ctx->critic_w_off,
                          d_grads + ctx->critic_b_off, st);
    if (rc != PAACB_OK) return rc;
  }
  const bool tc = (ctx->math != PAACB_MATH_FP32) && batch > 0;
  const int split3 = ctx->math == PAACB_MATH_TF32X3;
  if (tc && do_tail) {
    for (int l = 1; l < L; ++l) {
      rc = launch_pack_dgrad_weights(ctx, ctx->layer[l], d_params + ctx->layer[l].w_off, st);
      if (rc != PAACB_OK) return rc;
    }
  }
  for (int l = L - 1; l >= 0; --l) {
    if ((l == L - 1) ? !do_tail : !do_head) continue;
    const LayerGeom& g = ctx->layer[l];
    const void* x = (l == 0) ? (const void*)d_states : (const void*)(d_fwd_ws + g.in_act_off * batch);
    const float* dz = d_bwd_ws + g.out_act_off * batch;
    rc = tc ? launch_conv_wgrad_tc(ctx, g, x, dz, d_grads + g.w_off, d_grads + g.b_off, batch, split3, st) : PAACB_EUNSUPPORTED;
    if (rc == PAACB_EUNSUPPORTED) rc = launch_conv_wgrad_simt(ctx, g, x, dz, d_grads + g.w_off, d_grads + g.b_off, batch, st);
    if (rc != PAACB_OK) return rc;
    if (l > 0) {
      float* dx = d_bwd_ws + g.in_act_off * batch;
      rc = tc ? launch_conv_dgrad_tc(ctx, g, dz, (const float*)x, dx, batch, split3, st) : PAACB_EUNSUPPORTED;
      if (rc == PAACB_EUNSUPPORTED) rc = launch_conv_dgrad_simt(ctx, g, dz, d_params + g.w_off, (const float*)x, dx, batch, st);
      if (rc != PAACB_OK) return rc;
    }
  }
  return PAACB_OK;
}

int paacb_backward(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                   const float* d_fwd_ws, const float* d_dlogits, const float* d_dv, float* d_bwd_ws, float* d_grads,
                   paacb_stream stream) {
  return paacb_backward_part(ctx, d_params, d_states, batch, d_fwd_ws, d_dlogits, d_dv, d_bwd_ws, d_grads, PAACB_BWD_ALL,
                             stream);
}

int64_t paacb_grad_tail_offset(const paacb_ctx* ctx) {
  return ctx ? ctx->layer[ctx->n_layers - 1].w_off : PAACB_EINVAL;
}

int paacb_backward_part(const paacb_ctx* ctx, const float* d_params, const uint8_t* d_states, int64_t batch,
                        const float* d_fwd_ws, const float* d_dlogits, const float* d_dv, float* d_bwd_ws, float* d_grads,
                        int part, paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_params && d_states && d_fwd_ws && d_dlogits && d_dv && d_bwd_ws && d_grads, "NULL argument");
  PAACB_CHECK_ARG(((uintptr_t)d_bwd_ws & 15) == 0 && ((uintptr_t)d_grads & 15) == 0, "workspace / grads must be 16-byte aligned");
  PAACB_CHECK_ARG(part == PAACB_BWD_ALL || part == PAACB_BWD_TAIL || part == PAACB_BWD_HEAD, "unknown part");
  PAACB_CHECK_DEVICE(ctx);
  cudaStream_t st = (cudaStream_t)stream;
  const bool do_tail = part != PAACB_BWD_HEAD, do_head = part != PAACB_BWD_TAIL;
  if (do_tail && cudaMemsetAsync(d_grads, 0, (size_t)ctx->param_count * sizeof(float), st) != cudaSuccess) {
    set_error("paacb_backward: memset failed");
    return PAACB_ECUDA;
  }
  const int L = ctx->n_layers;
  if (ctx->math == PAACB_MATH_BF16X3) {
    if (batch == 0) return PAACB_OK;
    int rc = PAACB_OK;
    if (do_tail) {
      rc = backward_bf16_tail(ctx, d_params, d_fwd_ws, d_dlogits, d_dv, d_bwd_ws, d_grads, batch, st);
      if (rc != PAACB_OK) return rc;
    }
    // weight gradients of the conv layers: nothing downstream depends on them, so they come last and a caller can
    // all-reduce the tail of the gradient buffer while they run
    for (int l = L - 2; l >= 0 && rc == PAACB_OK && do_head; --l) rc = launch_conv_wgrad_bf16(ctx, l, d_states, d_fwd_ws, d_bwd_ws, d_grads, batch, st);
    return rc;
  }
  return backward_generic(ctx, d_params, d_states, batch, d_fwd_ws, d_dlogits, d_dv, d_bwd_ws, d_grads, do_tail, do_head, st);
}

static int clip_rmsprop_impl(const paacb_ctx* ctx, float* d_params, float* d_ms, float* d_mom, const float* d_grads,
                             float grad_scale, float lr, const float* d_lr, float rho, float eps, float momentum, float clip_norm,
                             int clip_type, float* d_norm_out, float* d_opt_ws, paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_params && d_ms && d_mom && d_grads && d_opt_ws, "NULL argument");
  PAACB_CHECK_DEVICE(ctx);
  PAACB_CHECK_ARG(clip_type == PAACB_CLIP_IGNORE || clip_type == PAACB_CLIP_GLOBAL,
                  "clip_type must be ignore or global ('local' is broken in the reference, actor_learner.py:62-63)");
  PAACB_CHECK_ARG(clip_type == PAACB_CLIP_IGNORE || clip_norm > 0.f, "clip_norm must be positive");
  PAACB_CHECK_ARG((((uintptr_t)d_params | (uintptr_t)d_ms | (uintptr_t)d_mom | (uintptr_t)d_grads | (uintptr_t)d_opt_ws) & 15) == 0,
                  "buffers must be 16-byte aligned");
  int rc = launch_clip_rmsprop(ctx, d_params, d_ms, d_mom, d_grads, grad_scale, lr, d_lr, rho, eps, momentum, clip_norm,
                               clip_type, d_norm_out, d_opt_ws, (cudaStream_t)stream);
  if (rc == PAACB_OK && ctx->math != PAACB_MATH_FP32) {
    // the library just changed the parameters: refresh the cached forward images in stream order (also inside a captured
    // graph), so the next forwards -- T acting forwards, the bootstrap and the training forward -- need no pack
    rc = pack_forward_images(ctx, d_params, (cudaStream_t)stream);
    ctx->fwd_img_valid = (rc == PAACB_OK);
    ctx->fwd_img_src = d_params;
  }
  return rc;
}

int paacb_clip_rmsprop(const paacb_ctx* ctx, float* d_params, float* d_ms, float* d_mom, const float* d_grads,
                       float grad_scale, float lr, float rho, float eps, float momentum, float clip_norm,
                       int clip_type, float* d_norm_out, float* d_opt_ws, paacb_stream stream) {
  return clip_rmsprop_impl(ctx, d_params, d_ms, d_mom, d_grads, grad_scale, lr, nullptr, rho, eps, momentum, clip_norm, clip_type,
                           d_norm_out, d_opt_ws, stream);
}

int paacb_clip_rmsprop_dlr(const paacb_ctx* ctx, float* d_params, float* d_ms, float* d_mom, const float* d_grads,
                           float grad_scale, const float* d_lr, float rho, float eps, float momentum, float clip_norm,
                           int clip_type, float* d_norm_out, float* d_opt_ws, paacb_stream stream) {
  PAACB_CHECK_ARG(d_lr != nullptr, "d_lr is NULL");
  return clip_rmsprop_impl(ctx, d_params, d_ms, d_mom, d_grads, grad_scale, 0.f, d_lr, rho, eps, momentum, clip_norm, clip_type,
                           d_norm_out, d_opt_ws, stream);
}

int paacb_grad_stats(const paacb_ctx* ctx, const float* d_grads, float grad_scale, float* d_opt_ws, double* d_out4,
                     paacb_stream stream) {
  PAACB_CHECK_ARG(ctx && d_grads && d_opt_ws && d_out4, "NULL argument");
  PAACB_CHECK_ARG(((uintptr_t)d_opt_ws & 15) == 0 && ((uintptr_t)d_out4 & 7) == 0, "workspace / output misaligned");
  PAACB_CHECK_DEVICE(ctx);
  return launch_grad_stats(ctx, d_grads, grad_scale, d_opt_ws, d_out4, (cudaStream_t)stream);
}

int paacb_host_register(void* host_ptr, size_t bytes, void** d_ptr) {
  PAACB_CHECK_ARG(host_ptr && d_ptr && bytes > 0, "NULL argument");
  cudaError_t e = cudaHostRegister(host_ptr, bytes, cudaHostRegisterMapped | cudaHostRegisterPortable);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaHostRegister(%zu bytes) failed: %s", bytes, cudaGetErrorString(e));
    return PAACB_ECUDA;
  }
  e = cudaHostGetDevicePointer(d_ptr, host_ptr, 0);
  if (e != cudaSuccess) {
    cudaGetLastError();
    cudaHostUnregister(host_ptr);
    set_error("cudaHostGetDevicePointer failed: %s", cudaGetErrorString(e));
    return PAACB_ECUDA;
  }
  return PAACB_OK;
}

int paacb_host_unregister(void* host_ptr) {
  PAACB_CHECK_ARG(host_ptr != nullptr, "NULL argument");
  const cudaError_t e = cudaHostUnregister(host_ptr);
  if (e != cudaSuccess) {
    cudaGetLastError();
    set_error("cudaHostUnregister failed: %s", cudaGetErrorString(e));
    return PAACB_ECUDA;
  }
  return PAACB_OK;
}

}  // extern "C"
