// bf16-split tensor-core path, part 4: the first conv layer forward as an INT8 patch-resident implicit GEMM.
//
//   Y[p, co] = relu( (1/255) * sum_{kh, kw, c} X[p; kh, kw, c] * W[kh, kw, c, co] + b[co] )      networks.py:115, 12-21
//
// The layer's input is the uint8 state itself.  Instead of converting 28 KB of pixels per sample to a floating type
// (the first version spent more time on that than on the MMAs), the pixels feed tcgen05.mma.kind::i8 as they are and the
// WEIGHTS are moved to integers: per output channel, w = s_c/63 * (d0 + d1/64 + d2/4096) with three signed digits
// |d0| <= 63, |d1|, |d2| <= 32 -- a fixed-point image of w with error <= 2^-19 of the channel's largest weight (the
// bf16-split weights of the other layers carry 2^-18 of EACH weight).  The three digit images are three groups of N
// columns of ONE MMA (N = 96): int32 accumulation is exact (|acc| <= 255 * 63 * 256 < 2^22), and the epilogue forms
// s_c / (63 * 255) * (acc0 + acc1/64 + acc2/4096) + b in fp32.
//
// A row of the GEMM is an output position, enumerated over the input grid as in tc2_conv.cu: the patch of a tile is
// 9 rows of each of the 4 row-parity planes of the state (input row ih = 4 q + rho), landed by the TMA engine WITHOUT
// swizzle as 16-byte units (4 pixels x 4 channels).  Consecutive output positions are 16 bytes apart and a filter row
// (8 pixels x 4 channels = 32 bytes = one K = 32 MMA) spans two consecutive units, which is exactly the no-swizzle
// K-major canonical layout with LBO = 16 (the second 16-byte K chunk of row r IS the first chunk of row r + 1) and
// SBO = 128: the overlapping windows of the convolution cost nothing.  Filter row kh is plane kh & 3 at a row offset.
#include "tc2_conv1.cuh"

namespace paacb {

// weights -> three int8 digit images + per-channel scale.  One block per output channel, one thread per k.
__global__ void __launch_bounds__(256) pack_conv1_i8_kernel(const float* __restrict__ w, int nc, int8_t* __restrict__ wq,
                                                            float* __restrict__ wscale) {
  __shared__ float red[8];
  const int c = blockIdx.x, k = threadIdx.x;
  const float v = __ldg(w + k * nc + c);
  float m = fabsf(v);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((k & 31) == 0) red[k >> 5] = m;
  __syncthreads();
  float s = red[0];
#pragma unroll
  for (int i = 1; i < 8; ++i) s = fmaxf(s, red[i]);
  // double arithmetic: the digits must reproduce x = 63 w / s to 2^-13 absolute
  const double x = (s > 0.f) ? 63.0 * (double)v / (double)s : 0.0;
  const double d0 = rint(x);
  const double r1 = (x - d0) * 64.0;
  const double d1 = rint(r1);
  const double d2 = rint((r1 - d1) * 64.0);
  wq[(0 * nc + c) * 256 + k] = (int8_t)d0;
  wq[(1 * nc + c) * 256 + k] = (int8_t)d1;
  wq[(2 * nc + c) * 256 + k] = (int8_t)d2;
  if (k == 0) wscale[c] = s / (63.0f * 255.0f);
}

int launch_pack_conv1_i8(const paacb_ctx* ctx, const float* params, cudaStream_t st) {
  const LayerGeom& g = ctx->layer[0];
  if (g.K != 256 || (g.N != 16 && g.N != 32) || ctx->wq_i8 == nullptr) return PAACB_EUNSUPPORTED;
  PAACB_LAUNCH_BEGIN(ctx, K_PACK, st);
  pack_conv1_i8_kernel<<<g.N, 256, 0, st>>>(params + g.w_off, g.N, ctx->wq_i8, ctx->wq_scale);
  PAACB_LAUNCH_END(ctx, K_PACK, st);
  return PAACB_OK;
}

template <int NC, bool F32OUT>
static int launch_conv1_inst(const paacb_ctx* ctx, const float* params, const uint8_t* states, uint8_t* out_hi, uint8_t* out_lo,
                             float* out_f32, uint16_t* relu_bits, int64_t batch, cudaStream_t st) {
  const LayerGeom& g = ctx->layer[0];
  if (g.C != 4 || g.stride != 4 || g.R != 8 || g.S != 8 || g.N != NC || g.H != 84 || g.W != 84 || g.OH != kC1_OH)
    return PAACB_EUNSUPPORTED;
  const int64_t plane_rows = batch * kC1_HQ;
  if (plane_rows * kC1_WU >= (1LL << 31) - 256) return PAACB_EUNSUPPORTED;
  Conv1Params p;
  memset(&p, 0, sizeof(p));
  // an image row (84 pixels x 4 channels = 336 bytes) is ONE inner box row of 84 32-bit words (box dimensions are limited
  // to 256 elements); plane row q = ih / 4 and row parity rho are separate dimensions (ih = 4 q + rho), parity slowest,
  // so one box lands the four parity planes of a tile one after the other
  const uint64_t adims[3] = {84u, (uint64_t)batch * kC1_HQ, 4u};
  const uint64_t astr[2] = {4u * 336u, 336u};
  const uint32_t abox[3] = {84u, (uint32_t)kC1_ROWS, 4u};
  int rc = encode_tmap(&p.tmA, states, 4, 3, adims, astr, abox, 0);
  const uint64_t wdims[2] = {256u, (uint64_t)C1<NC>::ND};
  const uint64_t wstr[1] = {256u};
  const uint32_t wbox[2] = {128u, (uint32_t)C1<NC>::ND};
  if (rc == PAACB_OK) rc = encode_tmap(&p.tmW, ctx->wq_i8, 1, 2, wdims, wstr, wbox, 128);
  if (rc != PAACB_OK) return rc;
  p.num_tiles = (int)((plane_rows + kC1_TROWS - 1) / kC1_TROWS);
  p.batch = (int)batch;
  p.bias = params + g.b_off;
  p.wscale = ctx->wq_scale;
  p.out_hi = out_hi;
  p.out_lo = out_lo;
  p.out_f32 = out_f32;
  p.relu_bits = relu_bits;
  constexpr int SMEM = kC1_SMEM_FIXED + C1<NC>::WBYTES;
  static DeviceOnce attr_set;   // kernel attributes are per device: one bit per device index
  if (!attr_set.done(ctx->device)) {
    if (cudaFuncSetAttribute(conv1_i8_kernel<NC, F32OUT>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM) != cudaSuccess) {
      cudaGetLastError();
      set_error("conv1_i8: cannot set %d bytes of dynamic shared memory", SMEM);
      return PAACB_ECUDA;
    }
    // one persistent CTA per SM: ask for the largest shared-memory carve-out whatever the kernel's own request (measured
    // on conv1 forward: the same code ran 10 % slower when its request dropped from 160 KB to 86 KB)
    cudaFuncSetAttribute(conv1_i8_kernel<NC, F32OUT>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    cudaGetLastError();
    attr_set.mark(ctx->device);
  }
  const unsigned grid = (unsigned)(p.num_tiles < ctx->num_sms ? p.num_tiles : ctx->num_sms);
  PAACB_LAUNCH_BEGIN(ctx, K_FWD0, st);
  conv1_i8_kernel<NC, F32OUT><<<grid, C1<NC>::THREADS, SMEM, st>>>(p);
  PAACB_LAUNCH_END(ctx, K_FWD0, st);
  return PAACB_OK;
}

// bf16-split pipeline (both architectures): planes out
int launch_conv1_fwd_i8(const paacb_ctx* ctx, const float* params, const uint8_t* states, void* fwd_ws, int64_t batch,
                        const WsSlice& slice, cudaStream_t st) {
  const LayerGeom& g = ctx->layer[0];
  const Planes out = layer_planes(fwd_ws, g.out_act_off, (int64_t)g.OH * g.OW * g.N, slice);
  uint16_t* bits = reinterpret_cast<uint16_t*>(relu1_bits(fwd_ws, ctx, slice));
  if (g.N == 16)      // NIPS: 16 channels = one 32-byte sector per position and plane
    return launch_conv1_inst<16, false>(ctx, params, states, out.hi, out.lo, nullptr, bits, batch, st);
  return launch_conv1_inst<32, false>(ctx, params, states, out.hi, out.lo, nullptr, bits, batch, st);
}

// NIPS (16 output channels), tf32 pipeline: fp32 activations out.  The int8 digit scheme is exact to 2^-19 of the largest
// weight of a channel, tighter than the tf32 split of the layers that follow.
int launch_conv1_fwd_i8_f32(const paacb_ctx* ctx, const float* params, const uint8_t* states, float* y, int64_t batch,
                            cudaStream_t st) {
  if (ctx->layer[0].N != 16 || ctx->wq_i8 == nullptr) return PAACB_EUNSUPPORTED;
  return launch_conv1_inst<16, true>(ctx, params, states, nullptr, nullptr, y, nullptr, batch, st);
}

}  // namespace paacb
