// bf16-split tensor-core path, part 1: patch-resident implicit GEMMs for the conv layers (forward and data-gradient),
// plus the small producers of their operands (uint8 -> bf16 states, packed weight images) and the tensor-map helper.
//
// Design (sm_100a; see DESIGN.md section 3.2):
//  * Activations live in HBM as TWO bf16 planes, value = hi + lo (|x - hi - lo| <= 2^-18 |x|).  A product is evaluated as
//    hi*hi + hi*lo + lo*hi in three kind::f16 MMAs with fp32 accumulation in TMEM: the dropped lo*lo term and the
//    residuals are ~2^-17 relative, an order of magnitude inside the 1e-4 parity bar, at twice the MMA rate and half
//    the operand bytes of the tf32x3 scheme.  uint8 pixels are exact in bf16 (conv1 needs two MMAs per K-step).
//  * No im2col, neither in HBM nor in shared memory.  The activation patch a tile of 128 output positions needs is
//    landed ONCE by the TMA engine, row-parity plane by row-parity plane, as rows of s*C consecutive channels
//    (32 B for conv1, 128 B for conv2/conv3).  Output positions are enumerated over the (padded) INPUT grid, so the
//    operand of filter tap (kh, kw) is the same patch at a byte offset: every tap is just another start address in
//    the MMA's shared-memory descriptor (the absolute-address swizzle that makes this legal was measured, tc_ptx.cuh).
//    Shared-memory fill traffic is 1x the input instead of the 4-9x an im2col-style tile pipeline re-reads.
//  * The layer's weights (both bf16 pieces, <= 144 KB) stay resident in shared memory for the whole kernel.
//  * Persistent CTA per SM: warp 0 = TMA producer, warp 1 = MMA issuer (one elected lane), warps 2-5 = epilogue
//    (tcgen05.ld, bias + ReLU or ReLU-mask, bf16 split, 16-byte stores; bias gradients as warp-transposed column sums).
//    Accumulators are double-buffered in TMEM; patch slots form an mbarrier ring.
#include "tc2_conv.cuh"

namespace paacb {

// ------------------------------------------------------------------------------------------------
// tensor maps
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
    else
      cudaGetLastError();
  }
  return fn;
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                     const uint32_t* box, int swizzle_bytes) {
  return encode_tmap(out, base, 2, rank, dims, strides_bytes, box, swizzle_bytes);
}

int encode_tmap(CUtensorMap* out, const void* base, int elem_bytes, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                const uint32_t* box, int swizzle_bytes) {
  EncodeTiledFn fn = encode_fn();
  if (fn == nullptr) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return PAACB_ECUDA;
  }
  cuuint64_t gd[5];
  cuuint64_t gs[5];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) {
    gd[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gs[i - 1] = strides_bytes[i - 1];
  }
  const CUtensorMapSwizzle sw = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  const CUtensorMapDataType dt = elem_bytes == 1 ? CU_TENSOR_MAP_DATA_TYPE_UINT8
                                 : elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
  const CUresult r = fn(out, dt, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): rank %d dims %llu,%llu,%llu,%llu box %u,%u,%u,%u", (int)r, rank,
              (unsigned long long)gd[0], (unsigned long long)(rank > 1 ? gd[1] : 0), (unsigned long long)(rank > 2 ? gd[2] : 0),
              (unsigned long long)(rank > 3 ? gd[3] : 0), bx[0], rank > 1 ? bx[1] : 0, rank > 2 ? bx[2] : 0, rank > 3 ? bx[3] : 0);
    return PAACB_ECUDA;
  }
  return PAACB_OK;
}

bool bf16x3_supported(const paacb_ctx* ctx) { return ctx->arch == PAACB_ARCH_NATURE || ctx->arch == PAACB_ARCH_NIPS; }

// ------------------------------------------------------------------------------------------------
// operand producers
// ------------------------------------------------------------------------------------------------
// forward image: Wp[n][k] = W[k][n] as (hi, lo) bf16, row-major [N][K] (the B operand, K-major).  32 x 32 tiles through
// shared memory so that both the fp32 reads and the bf16 writes are coalesced (the fc layer has 1.6 M weights and the
// image is rebuilt on every forward call).
__global__ void __launch_bounds__(256) pack_bf16_transpose_kernel(const float* __restrict__ w, int K, int N,
                                                                  uint16_t* __restrict__ hi, uint16_t* __restrict__ lo) {
  __shared__ float tile[32][33];
  const int k0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;       // 8 rows per pass
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int k = k0 + r, n = n0 + tx;
    tile[r][tx] = (k < K && n < N) ? __ldg(w + (int64_t)k * N + n) : 0.f;
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 32; r += 8) {
    const int n = n0 + r, k = k0 + tx;
    if (n < N && k < K) {
      uint16_t h, l;
      split_bf16(tile[tx][r], h, l);
      hi[(int64_t)n * K + k] = h;
      lo[(int64_t)n * K + k] = l;
    }
  }
}
// same orientation as stored (fc data-gradient: rows = inputs, K = outputs)
__global__ void pack_bf16_copy_kernel(const float* __restrict__ w, int64_t total, uint16_t* __restrict__ hi,
                                      uint16_t* __restrict__ lo) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    uint16_t h, l;
    split_bf16(__ldg(w + i), h, l);
    hi[i] = h;
    lo[i] = l;
  }
}
// conv data-gradient image: Wd[cls][ci][(tj*I + ti)*Cout + co] = W[ph + s*tj][pw + s*ti][ci][co], cls = ph*s + pw
__global__ void pack_bf16_dgrad_kernel(const float* __restrict__ w, LayerGeom g, int J, int I, uint16_t* __restrict__ hi,
                                       uint16_t* __restrict__ lo) {
  const int s = g.stride;
  const int Kd = J * I * g.N;
  const int64_t total = (int64_t)s * s * g.C * Kd;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int kd = (int)(i % Kd);
    const int64_t rest = i / Kd;
    const int ci = (int)(rest % g.C), cls = (int)(rest / g.C);
    const int tap = kd / g.N, co = kd - tap * g.N;
    const int tj = tap / I, ti = tap - tj * I;
    const int kh = cls / s + s * tj, kw = cls % s + s * ti;
    uint16_t h, l;
    split_bf16(__ldg(w + ((int64_t)(kh * g.S + kw) * g.C + ci) * g.N + co), h, l);
    hi[i] = h;
    lo[i] = l;
  }
}

int launch_pack_bf16_weights(const paacb_ctx* ctx, const float* params, cudaStream_t st) {
  const int rc = launch_pack_conv1_i8(ctx, params, st);      // conv1 runs on the int8 pipe (tc2_conv1.cu)
  if (rc != PAACB_OK) return rc;
  for (int l = 1; l < ctx->n_layers; ++l) {
    const LayerGeom& g = ctx->layer[l];
    const dim3 grid((unsigned)((g.N + 31) / 32), (unsigned)((g.K + 31) / 32));
    PAACB_LAUNCH_BEGIN(ctx, K_PACK, st);
    pack_bf16_transpose_kernel<<<grid, 256, 0, st>>>(params + g.w_off, g.K, g.N, ctx->wb_f_hi + g.w_off, ctx->wb_f_lo + g.w_off);
    PAACB_LAUNCH_END(ctx, K_PACK, st);
  }
  return PAACB_OK;
}

int launch_pack_bf16_dgrad_weights(const paacb_ctx* ctx, const float* params, cudaStream_t st) {
  for (int l = 1; l < ctx->n_layers; ++l) {
    const LayerGeom& g = ctx->layer[l];
    const int64_t total = (int64_t)g.K * g.N;
    PAACB_LAUNCH_BEGIN(ctx, K_PACK, st);
    if (g.R == 1 && g.S == 1) {
      pack_bf16_copy_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(params + g.w_off, total, ctx->wb_d_hi + g.w_off,
                                                                             ctx->wb_d_lo + g.w_off);
    } else {
      const int s = g.stride;
      pack_bf16_dgrad_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(params + g.w_off, g, g.R / s, g.S / s,
                                                                              ctx->wb_d_hi + g.w_off, ctx->wb_d_lo + g.w_off);
    }
    PAACB_LAUNCH_END(ctx, K_PACK, st);
  }
  return PAACB_OK;
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
template <int G>
static int launch_convk(const paacb_ctx* ctx, const ConvKParams& p, int slot, cudaStream_t st) {
  // always the successor of another kernel of the same forward / backward: programmatic dependent launch (tc_ptx.cuh)
  using Cfg = ConvKCfg<G>;
  static DeviceOnce attr_set;   // kernel attributes are per device: one bit per device index
  if (!attr_set.done(ctx->device)) {
    if (cudaFuncSetAttribute(convk_kernel<G>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess) {
      cudaGetLastError();
      set_error("convk<%d>: cannot set %d bytes of dynamic shared memory", G, Cfg::SMEM_BYTES);
      return PAACB_ECUDA;
    }
    // one persistent CTA per SM: ask for the largest shared-memory carve-out whatever the kernel's own request (measured
    // on conv1 forward: the same code ran 10 % slower when its request dropped from 160 KB to 86 KB)
    cudaFuncSetAttribute(convk_kernel<G>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    cudaGetLastError();
    attr_set.mark(ctx->device);
  }
  const unsigned grid = (unsigned)(p.num_tiles < ctx->num_sms ? p.num_tiles : ctx->num_sms);
  PAACB_LAUNCH_BEGIN(ctx, slot, st);
  launch_kernel(convk_kernel<G>, grid, Cfg::THREADS, Cfg::SMEM_BYTES, st, p);
  PAACB_LAUNCH_END(ctx, slot, st);
  return PAACB_OK;
}

static int weight_maps(const paacb_ctx* ctx, const uint16_t* hi, const uint16_t* lo, const LayerGeom& g, uint64_t kdim,
                       uint64_t rows, uint32_t box_rows, CUtensorMap* out) {
  const uint64_t dims[2] = {kdim, rows};
  const uint64_t strides[1] = {kdim * 2};
  const uint32_t box[2] = {64, box_rows};
  int rc = encode_tmap_bf16(&out[0], hi + g.w_off, 2, dims, strides, box, 128);
  if (rc != PAACB_OK) return rc;
  return encode_tmap_bf16(&out[1], lo + g.w_off, 2, dims, strides, box, 128);
}

int launch_conv_fwd_bf16(const paacb_ctx* ctx, int l, const float* params, const uint8_t* states, void* fwd_ws, int64_t batch,
                         const WsSlice& slice, cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  ConvKParams p;
  memset(&p, 0, sizeof(p));
  p.batch = (int)batch;
  p.bias = params + g.b_off;
  p.in_scale = g.in_u8 ? 0.003921568859368563f : 1.0f;
  const Planes out = layer_planes(fwd_ws, g.out_act_off, (int64_t)g.OH * g.OW * g.N, slice);
  p.out_hi = out.hi;
  p.out_lo = out.lo;
  const uint8_t* in_hi;
  const uint8_t* in_lo;
  if (l == 0) {
    in_hi = in_lo = nullptr;                    // conv1 converts the uint8 states itself
  } else {
    const Planes in = layer_planes(fwd_ws, g.in_act_off, (int64_t)g.H * g.W * g.C, slice);
    in_hi = in.hi;
    in_lo = in.lo;
  }
  const int s = g.stride;
  const uint64_t unit = (uint64_t)s * g.C;                      // elements per unit
  const uint64_t wu = (uint64_t)g.W / s, hq = (uint64_t)g.H / s;
  const uint64_t dims[4] = {unit, wu, (uint64_t)s, (uint64_t)batch * hq};
  const uint64_t strides[3] = {unit * 2, (uint64_t)g.W * g.C * 2, (uint64_t)s * g.W * g.C * 2};
  int rc;
#define PAACB_FWD_CASE(GE)                                                                                         \
  {                                                                                                                \
    using Ge = Geo<GE>;                                                                                            \
    if ((int)unit * 2 != Ge::UB || (int)wu != Ge::WU || (int)hq != Ge::HQ || g.N != Ge::BN || g.K != Ge::KB * 64 ||  \
        s != Ge::PARTS || g.OH != Ge::OH || g.OW != Ge::OW)                                                        \
      break;                                                                                                       \
    const uint32_t box[4] = {(uint32_t)unit, (uint32_t)Ge::WU, 1u, (uint32_t)Ge::BOX_ROWS};                        \
    rc = encode_tmap_bf16(&p.tmA[0], in_hi, 4, dims, strides, box, Ge::UB);                                        \
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmA[1], in_lo, 4, dims, strides, box, Ge::UB);                    \
    if (rc == PAACB_OK) rc = weight_maps(ctx, ctx->wb_f_hi, ctx->wb_f_lo, g, (uint64_t)g.K, (uint64_t)g.N, Ge::BN, p.tmW); \
    if (rc != PAACB_OK) return rc;                                                                                 \
    const int64_t q_total = batch * Ge::HQ * Ge::WU;                                                               \
    if (q_total >= (1LL << 31) - 256) return PAACB_EUNSUPPORTED;                                                   \
    p.num_tiles = (int)((q_total + 127) / 128);                                                                    \
    return launch_convk<GE>(ctx, p, K_FWD0 + l, st);                                                               \
  }
  if (l == 0) return launch_conv1_fwd_i8(ctx, params, states, fwd_ws, batch, slice, st);
  // (each case leaves its do-while with `break` when the layer's geometry is not the one it was written for)
  if (l == 1) do PAACB_FWD_CASE(G_FWD2) while (0);
  if (l == 1) do PAACB_FWD_CASE(G_FWD2N) while (0);
  if (l == 2) do {
    // conv3, two whole samples per tile (Geo<G_FWD3P>): the source planes as (channels, x, y, sample); one box = the 7 input
    // rows kh .. kh + 6 of two samples; a box that runs past the last sample is zero-filled
    using Ge = Geo<G_FWD3P>;
    if (g.C * 2 != Ge::UB || g.W != Ge::WU || g.H != Ge::HQ || g.N != Ge::BN || g.K != Ge::KB * 64 || s != 1 || g.R != Ge::PARTS ||
        g.S != 3 || g.OH != Ge::OH || g.OW != Ge::OW)
      break;
    const uint64_t pdims[4] = {(uint64_t)g.C, (uint64_t)g.W, (uint64_t)g.H, (uint64_t)batch};
    const uint64_t pstr[3] = {(uint64_t)g.C * 2, (uint64_t)g.W * g.C * 2, (uint64_t)g.H * g.W * g.C * 2};
    const uint32_t pbox[4] = {(uint32_t)g.C, (uint32_t)g.W, (uint32_t)Ge::OH, (uint32_t)GeoPack<G_FWD3P>::SAMPLES};
    static_assert(Ge::BOX_ROWS == Ge::OH * GeoPack<G_FWD3P>::SAMPLES, "box bytes");
    rc = encode_tmap_bf16(&p.tmA[0], in_hi, 4, pdims, pstr, pbox, Ge::UB);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmA[1], in_lo, 4, pdims, pstr, pbox, Ge::UB);
    if (rc == PAACB_OK) rc = weight_maps(ctx, ctx->wb_f_hi, ctx->wb_f_lo, g, (uint64_t)g.K, (uint64_t)g.N, Ge::BN, p.tmW);
    if (rc != PAACB_OK) return rc;
    p.num_tiles = (int)((batch + GeoPack<G_FWD3P>::SAMPLES - 1) / GeoPack<G_FWD3P>::SAMPLES);
    return launch_convk<G_FWD3P>(ctx, p, K_FWD0 + l, st);
  } while (0);
#undef PAACB_FWD_CASE
  return PAACB_EUNSUPPORTED;
}

// dX of layer l's input: A = dZ planes of layer l (bwd_ws), output = dZ planes of layer l-1, masked by layer l-1's activation
int launch_conv_dgrad_bf16(const paacb_ctx* ctx, int l, const void* fwd_ws, void* bwd_ws, float* grads, int64_t batch,
                           cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  const LayerGeom& gp = ctx->layer[l - 1];
  ConvKParams p;
  memset(&p, 0, sizeof(p));
  p.batch = (int)batch;
  p.num_tiles = (int)batch;
  const Planes dz = layer_planes(bwd_ws, g.out_act_off, (int64_t)g.OH * g.OW * g.N, batch);
  const Planes dx = layer_planes(bwd_ws, gp.out_act_off, (int64_t)g.H * g.W * g.C, batch);
  const Planes xa = layer_planes(const_cast<void*>(fwd_ws), gp.out_act_off, (int64_t)g.H * g.W * g.C, batch);
  p.out_hi = dx.hi;
  p.out_lo = dx.lo;
  p.mask_hi = xa.hi;
  if (l == 1) p.mask_bits = relu1_bits(const_cast<void*>(fwd_ws), ctx, WsSlice{batch, 0});     // conv1's ReLU mask as bit words
  p.dbias = grads + gp.b_off;
  const uint64_t dims[4] = {(uint64_t)g.N, (uint64_t)g.OW, (uint64_t)g.OH, (uint64_t)batch};
  const uint64_t strides[3] = {(uint64_t)g.N * 2, (uint64_t)g.OW * g.N * 2, (uint64_t)g.OH * g.OW * g.N * 2};
  int rc;
#define PAACB_DG_CASE(GE)                                                                                          \
  {                                                                                                                \
    using Ge = Geo<GE>;                                                                                            \
    const int s = g.stride;                                                                                        \
    if (g.N * 2 != Ge::UB || g.C != Ge::CH || s != Ge::S || g.H != Ge::XH || g.W != Ge::XW ||                       \
        (g.R / s) * (g.S / s) * g.N != Ge::KB * 64 || s * s * g.C != Ge::NACC * Ge::BN ||                           \
        (g.R - 1) / s != Ge::PAD || g.OH + 2 * Ge::PAD > Ge::BOX_ROWS + 0 || (g.H + s - 1) / s != Ge::OH)          \
      break;                                                                                                       \
    const uint32_t box[4] = {(uint32_t)g.N, (uint32_t)Ge::WU, (uint32_t)Ge::BOX_ROWS, 1u};                          \
    rc = encode_tmap_bf16(&p.tmA[0], dz.hi, 4, dims, strides, box, Ge::UB);                                        \
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmA[1], dz.lo, 4, dims, strides, box, Ge::UB);                    \
    if (rc == PAACB_OK)                                                                                            \
      rc = weight_maps(ctx, ctx->wb_d_hi, ctx->wb_d_lo, g, (uint64_t)(g.R / s) * (g.S / s) * g.N,                  \
                       (uint64_t)s * s * g.C, Ge::BN, p.tmW);                                                      \
    if (rc == PAACB_OK && Ge::STAGED) {                                                                            \
      const uint64_t od[4] = {(uint64_t)2 * g.C, (uint64_t)g.W / 2, 2u, (uint64_t)batch * (g.H / 2)};              \
      const uint64_t os[3] = {(uint64_t)2 * g.C * 2, (uint64_t)g.W * g.C * 2, (uint64_t)2 * g.W * g.C * 2};        \
      const uint32_t ob[4] = {(uint32_t)(2 * g.C), (uint32_t)(g.W / 2), 1u, (uint32_t)(g.H / 2)};                  \
      rc = encode_tmap_bf16(&p.tmOut, dx.hi, 4, od, os, ob, 128);                                                  \
    }                                                                                                              \
    if (rc != PAACB_OK) return rc;                                                                                 \
    return launch_convk<GE>(ctx, p, K_DGRAD0 + l, st);                                                             \
  }
  if (g.stride == 1) do PAACB_DG_CASE(G_DG3) while (0);
  if (g.stride == 2) do PAACB_DG_CASE(G_DG2) while (0);
  if (g.stride == 2) do PAACB_DG_CASE(G_DG2N) while (0);
#undef PAACB_DG_CASE
  return PAACB_EUNSUPPORTED;
}

}  // namespace paacb
