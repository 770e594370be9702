// bf16-split tensor-core path, part 2: streaming GEMM for the fully connected layer (forward, data-gradient and
// weight-gradient).  Both operands are re-staged per 64-wide K-block by the TMA engine (there is no spatial reuse to
// exploit in an fc layer); three kind::f16 MMAs per K-step evaluate hi*hi + hi*lo + lo*hi (tc2_conv.cu).
//
//   forward : H[m, n]  = relu(sum_k X[m, k] W[k, n] + b[n])        A = X planes [M, K] (K-major), B = W^T image [N, K]
//   dgrad   : dX[m, c] = (sum_n dZ[m, n] W[c, n]) * [X[m, c] > 0]  A = dZ planes [M, N],          B = W image   [C, N]
//   wgrad   : dW[k, n] += sum_m X[m, k] dZ[m, n]                   A = X planes, B = dZ planes, both MN-major: the
//             reduction index (samples) is the slow index of both as they lie in HBM, so the tiles are used as they
//             land -- no transposition anywhere (the previous kernel transposed through registers with 4-byte stores).
// Persistent CTA per SM: warp 0 TMA producer, warp 1 MMA issuer, warps 2-5 epilogue; double-buffered TMEM accumulator.
#include "tc2_stream.cuh"

namespace paacb {

template <int BN, int MODE>
static int launch_stream(const paacb_ctx* ctx, const StreamParams& p, int slot, cudaStream_t st) {
  using Cfg = StreamCfg<BN, MODE>;
  static DeviceOnce attr_set;   // kernel attributes are per device: one bit per device index
  if (!attr_set.done(ctx->device)) {
    if (cudaFuncSetAttribute(stream_gemm_kernel<BN, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) !=
        cudaSuccess) {
      cudaGetLastError();
      set_error("stream_gemm<%d,%d>: cannot set %d bytes of dynamic shared memory", BN, MODE, Cfg::SMEM_BYTES);
      return PAACB_ECUDA;
    }
    // one persistent CTA per SM: ask for the largest shared-memory carve-out whatever the kernel's own request (measured
    // on conv1 forward: the same code ran 10 % slower when its request dropped from 160 KB to 86 KB)
    cudaFuncSetAttribute(stream_gemm_kernel<BN, MODE>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    cudaGetLastError();
    attr_set.mark(ctx->device);
  }
  const int units = p.m_tiles * p.n_tiles * p.k_splits;
  const unsigned grid = (unsigned)(units < ctx->num_sms ? units : ctx->num_sms);
  PAACB_LAUNCH_BEGIN(ctx, slot, st);
  launch_kernel(stream_gemm_kernel<BN, MODE>, grid, kStreamThreads, Cfg::SMEM_BYTES, st, p);
  PAACB_LAUNCH_END(ctx, slot, st);
  return PAACB_OK;
}

static int map2d(CUtensorMap* out, const void* base, uint64_t inner, uint64_t rows, uint32_t box_inner, uint32_t box_rows) {
  const uint64_t dims[2] = {inner, rows};
  const uint64_t strides[1] = {inner * 2};
  const uint32_t box[2] = {box_inner, box_rows};
  return encode_tmap_bf16(out, base, 2, dims, strides, box, 128);
}

int launch_fc_fwd_bf16(const paacb_ctx* ctx, int l, const float* params, void* fwd_ws, int64_t batch, const WsSlice& slice,
                       cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  // K need not be a multiple of the 64-wide K-block (NIPS: 2592 = 40.5 blocks): the TMA engine zero-fills BOTH operands
  // beyond K, so the ragged tail contributes nothing.  Row pitches must be multiples of 16 bytes.
  if (g.K % 8 != 0 || g.N % kFcBN != 0) return PAACB_EUNSUPPORTED;
  StreamParams p;
  memset(&p, 0, sizeof(p));
  const Planes x = layer_planes(fwd_ws, g.in_act_off, g.K, slice);
  const Planes y = layer_planes(fwd_ws, g.out_act_off, g.N, slice);
  int rc = map2d(&p.tmA[0], x.hi, (uint64_t)g.K, (uint64_t)batch, 64, 128);
  if (rc == PAACB_OK) rc = map2d(&p.tmA[1], x.lo, (uint64_t)g.K, (uint64_t)batch, 64, 128);
  if (rc == PAACB_OK) rc = map2d(&p.tmB[0], ctx->wb_f_hi + g.w_off, (uint64_t)g.K, (uint64_t)g.N, 64, kFcBN);
  if (rc == PAACB_OK) rc = map2d(&p.tmB[1], ctx->wb_f_lo + g.w_off, (uint64_t)g.K, (uint64_t)g.N, 64, kFcBN);
  if (rc != PAACB_OK) return rc;
  p.m_tiles = (int)((batch + 127) / 128);
  p.n_tiles = g.N / kFcBN;
  p.k_splits = 1;
  p.kblocks_total = p.kblocks_per_split = (g.K + 63) / 64;
  p.M = (int)batch;
  p.N = g.N;
  p.ldo = g.N;
  p.bias = params + g.b_off;
  p.out_hi = y.hi;
  p.out_lo = y.lo;
  return launch_stream<kFcBN, ST_FWD>(ctx, p, K_FWD0 + l, st);
}

int launch_fc_dgrad_bf16(const paacb_ctx* ctx, int l, const void* fwd_ws, void* bwd_ws, float* grads, int64_t batch,
                         cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  const LayerGeom& gp = ctx->layer[l - 1];
  if (g.N % 64 != 0 || g.K % 32 != 0) return PAACB_EUNSUPPORTED;
  StreamParams p;
  memset(&p, 0, sizeof(p));
  const Planes dz = layer_planes(bwd_ws, g.out_act_off, g.N, batch);
  const Planes dx = layer_planes(bwd_ws, gp.out_act_off, g.K, batch);
  const Planes xa = layer_planes(const_cast<void*>(fwd_ws), gp.out_act_off, g.K, batch);
  int rc = map2d(&p.tmA[0], dz.hi, (uint64_t)g.N, (uint64_t)batch, 64, 128);
  if (rc == PAACB_OK) rc = map2d(&p.tmA[1], dz.lo, (uint64_t)g.N, (uint64_t)batch, 64, 128);
  if (rc == PAACB_OK) rc = map2d(&p.tmB[0], ctx->wb_d_hi + g.w_off, (uint64_t)g.N, (uint64_t)g.K, 64, kFcBN);
  if (rc == PAACB_OK) rc = map2d(&p.tmB[1], ctx->wb_d_lo + g.w_off, (uint64_t)g.N, (uint64_t)g.K, 64, kFcBN);
  if (rc != PAACB_OK) return rc;
  p.m_tiles = (int)((batch + 127) / 128);
  p.n_tiles = (g.K + kFcBN - 1) / kFcBN;
  p.k_splits = 1;
  p.kblocks_total = p.kblocks_per_split = g.N / 64;
  p.M = (int)batch;
  p.N = g.K;
  p.ldo = g.K;
  p.out_hi = dx.hi;
  p.out_lo = dx.lo;
  p.mask_hi = xa.hi;
  p.dbias = grads + gp.b_off;
  p.dbias_mod = gp.N;
  return launch_stream<kFcBN, ST_DGRAD>(ctx, p, K_DGRAD0 + l, st);
}

int launch_fc_wgrad_bf16(const paacb_ctx* ctx, int l, const void* fwd_ws, const void* bwd_ws, float* grads, int64_t batch,
                         cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  if (g.N % kFcBN != 0 || g.K % 32 != 0) return PAACB_EUNSUPPORTED;      // ragged k-tiles: OOB columns of X read zeros
  StreamParams p;
  memset(&p, 0, sizeof(p));
  const Planes x = layer_planes(const_cast<void*>(fwd_ws), g.in_act_off, g.K, batch);
  const Planes dz = layer_planes(const_cast<void*>(bwd_ws), g.out_act_off, g.N, batch);
  int rc = map2d(&p.tmA[0], x.hi, (uint64_t)g.K, (uint64_t)batch, 64, 64);
  if (rc == PAACB_OK) rc = map2d(&p.tmA[1], x.lo, (uint64_t)g.K, (uint64_t)batch, 64, 64);
  if (rc == PAACB_OK) rc = map2d(&p.tmB[0], dz.hi, (uint64_t)g.N, (uint64_t)batch, 64, 64);
  if (rc == PAACB_OK) rc = map2d(&p.tmB[1], dz.lo, (uint64_t)g.N, (uint64_t)batch, 64, 64);
  if (rc != PAACB_OK) return rc;
  p.m_tiles = (g.K + 127) / 128;
  p.n_tiles = g.N / kFcBN;
  p.kblocks_total = (int)((batch + 63) / 64);
  // reduction splits: the (k-tile, n-tile, split) units are spread over one persistent CTA per SM; pick the split count
  // (2..3 units per SM: every unit ends with 16 K fp32 atomics, about a fifth of a 2,000-sample mainloop) whose last wave
  // is fullest (3 splits left 32 % of the SMs idle in the last wave of the fc layer)
  const int tiles = p.m_tiles * p.n_tiles;
  int splits = 1;
  double best = 0.0;
  for (int s = 1; s <= 64; ++s) {
    const int units = tiles * s;
    if (units < 2 * ctx->num_sms && s < 64) continue;
    if (units > 3 * ctx->num_sms && splits > 1) break;
    const int waves = (units + ctx->num_sms - 1) / ctx->num_sms;
    const double eff = (double)units / ((double)waves * ctx->num_sms);
    if (eff > best + 1e-9) { best = eff; splits = s; }
  }
  if (splits > p.kblocks_total) splits = p.kblocks_total;
  if (splits < 1) splits = 1;
  p.kblocks_per_split = (p.kblocks_total + splits - 1) / splits;
  p.k_splits = (p.kblocks_total + p.kblocks_per_split - 1) / p.kblocks_per_split;
  p.M = g.K;
  p.N = g.N;
  p.ldo = g.N;
  p.dw = grads + g.w_off;
  return launch_stream<kFcBN, ST_WGRAD>(ctx, p, K_WGRAD0 + l, st);
}

}  // namespace paacb
