// K5 + K6: actor / critic heads, softmax, categorical sampling; and the heads' backward.
//
// Forward replaces networks.py:84-89 (softmax layer), policy_v_network.py:24-26,37 (critic, reshape)
// and paac.py:34-45 / :27 (sampling, one-hot).  One warp per sample: lanes stride the F hidden
// features, accumulate the A+1 dot products against head weights staged in shared memory, butterfly
// reduce, then every lane holds the logits; softmax is exp(z - max) / sum as TF's Softmax op.
// Sampling is inverse-CDF on a caller-supplied uniform (fp32 running sum, last bucket open-ended).
//
// Backward: dWa = h^T dlogits, dba = colsum(dlogits), dWc = h^T dv, dbc = sum(dv),
//           dh = (dlogits Wa^T + dv Wc^T) * [h > 0]   (ReLU mask of the hidden layer fused).
#include "common.cuh"
#include "tc_ptx.cuh"
#include <cuda_bf16.h>

namespace paacb {

// bf16-split activations (PAACB_MATH_BF16X3): value = float(hi) + float(lo)
__device__ __forceinline__ float split_load(const uint16_t* hi, const uint16_t* lo, int64_t i) {
  return __uint_as_float((uint32_t)__ldg(hi + i) << 16) + __uint_as_float((uint32_t)__ldg(lo + i) << 16);
}


constexpr int kMaxA = PAACB_MAX_ACTIONS;
constexpr int kHeadWarps = 8;

// ---- K6: the uniform of a sampling decision ---------------------------------------------------------------------
// Either injected by the caller (d_uniforms; tests and reference-style host sampling) or drawn IN the kernel from
// Philox4x32-10 (Salmon et al., SC'11; the generator behind curand / torch.cuda): counter = (sample index, draw index),
// key = seed, u = (first output word >> 8) * 2^-24 in [0, 1).  Stateless: every (seed, draw, sample) has one value
// whatever the launch geometry or the slicing of the environments.  oracle/sampling.py restates it in NumPy.
struct SampleSrc {
  const float* uniforms;        // injected uniforms [b] or nullptr
  const uint64_t* rng;          // device {seed, draw base} or nullptr
  uint64_t draw;                // added to the draw base
  int64_t first;                // global index of sample 0 of this call (environment slices)
};
__device__ __forceinline__ uint32_t mulhilo32(uint32_t a, uint32_t b, uint32_t& hi) {
  const uint64_t p = (uint64_t)a * b;
  hi = (uint32_t)(p >> 32);
  return (uint32_t)p;
}
__device__ __forceinline__ uint32_t philox4x32_10_x(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0, hi1;
    const uint32_t lo0 = mulhilo32(0xD2511F53u, c0, hi0);
    const uint32_t lo1 = mulhilo32(0xCD9E8D57u, c2, hi1);
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c0;
}
__device__ __forceinline__ float sample_uniform(const SampleSrc& s, int64_t b) {
  if (s.uniforms != nullptr) return __ldg(s.uniforms + b);
  const uint64_t seed = s.rng[0], d = s.rng[1] + s.draw, i = (uint64_t)(s.first + b);
  const uint32_t x = philox4x32_10_x((uint32_t)i, (uint32_t)(i >> 32), (uint32_t)d, (uint32_t)(d >> 32), (uint32_t)seed,
                                     (uint32_t)(seed >> 32));
  return (float)(x >> 8) * 5.9604644775390625e-08f;      // 2^-24
}
// paacb_rng_advance: draw base += n, in stream order (one launch per update; the base lives in device memory so that a
// captured CUDA graph of the rollout replays with fresh uniforms)
__global__ void rng_advance_kernel(uint64_t* rng, uint64_t n) { rng[1] += n; }

__global__ void __launch_bounds__(kHeadWarps * 32)
heads_fwd_kernel(const float* __restrict__ h, const uint16_t* __restrict__ h_hi, const uint16_t* __restrict__ h_lo,
                 const float* __restrict__ wa, const float* __restrict__ ba,
                 const float* __restrict__ wc, const float* __restrict__ bc, int64_t batch, int F, int A,
                 float* __restrict__ pi, float* __restrict__ v, const SampleSrc smp,
                 int32_t* __restrict__ actions, float* __restrict__ onehot) {
  extern __shared__ float sw[];              // [F][A+1]: actor columns then the critic column
  const int A1 = A + 1;
  for (int i = threadIdx.x; i < F * A1; i += blockDim.x) {
    const int f = i / A1, a = i - f * A1;
    sw[i] = (a < A) ? __ldg(wa + (int64_t)f * A + a) : __ldg(wc + f);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t b = (int64_t)blockIdx.x * kHeadWarps + warp; b < batch; b += (int64_t)gridDim.x * kHeadWarps) {
    float acc[kMaxA + 1];
#pragma unroll
    for (int a = 0; a <= kMaxA; ++a) acc[a] = 0.f;
    for (int f = lane; f < F; f += 32) {
      const float hv = (h != nullptr) ? __ldg(h + b * F + f) : split_load(h_hi, h_lo, b * F + f);
      const float* wr = sw + f * A1;
#pragma unroll
      for (int a = 0; a <= kMaxA; ++a)
        if (a < A1) acc[a] = fmaf(hv, wr[a], acc[a]);
    }
#pragma unroll
    for (int a = 0; a <= kMaxA; ++a) {
      if (a < A1) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[a] += __shfl_xor_sync(0xffffffffu, acc[a], o);
      }
    }
    // every lane now holds all A+1 sums; lanes 0..A-1 keep their own logit
    float z = -INFINITY, val = 0.f;
#pragma unroll
    for (int a = 0; a <= kMaxA; ++a) {
      if (a < A && lane == a) z = acc[a] + __ldg(ba + a);
      if (a == A) val = acc[a] + __ldg(bc);
    }
    float mx = z;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float e = (lane < A) ? expf(z - mx) : 0.f;
    float sum = e;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float p = e / sum;
    if (lane < A) pi[b * A + lane] = p;
    if (lane == 0) v[b] = val;
    if (smp.uniforms != nullptr || smp.rng != nullptr) {
      const float u = sample_uniform(smp, b);
      // fp32 running sum in index order: c_j = c_{j-1} + p_j; action = first j < A-1 with u < c_j
      int act = A - 1;
      float c = 0.f;
      bool done = false;
      for (int j = 0; j < A - 1; ++j) {
        c += __shfl_sync(0xffffffffu, p, j);
        if (!done && u < c) { act = j; done = true; }
      }
      if (actions != nullptr && lane == 0) actions[b] = act;
      if (onehot != nullptr && lane < A) onehot[b * A + lane] = (lane == act) ? 1.f : 0.f;
    }
  }
}

constexpr int kHbThreads = 256;
constexpr int kHbChunk = 128;    // samples per CTA

template <int FPT>   // features per thread: F = FPT * 256
__global__ void __launch_bounds__(kHbThreads)
heads_bwd_kernel(const float* __restrict__ h, const uint16_t* __restrict__ h_hi, const uint16_t* __restrict__ h_lo,
                 uint16_t* __restrict__ dh_hi, uint16_t* __restrict__ dh_lo, float* __restrict__ dbh,
                 const float* __restrict__ wa, const float* __restrict__ wc,
                 const float* __restrict__ dlogits, const float* __restrict__ dv, int64_t batch, int F, int A,
                 float* __restrict__ dh, float* __restrict__ dwa, float* __restrict__ dba, float* __restrict__ dwc,
                 float* __restrict__ dbc) {
  __shared__ float sd[kHbChunk][kMaxA + 2];      // dlogits row then dv
  const int A1 = A + 1;
  const int tid = threadIdx.x;
  const int64_t b0 = (int64_t)blockIdx.x * kHbChunk;
  const int nb = (int)((batch - b0 < kHbChunk) ? batch - b0 : kHbChunk);
  for (int i = tid; i < nb * A1; i += kHbThreads) {
    const int r = i / A1, a = i - r * A1;
    sd[r][a] = (a < A) ? __ldg(dlogits + (b0 + r) * A + a) : __ldg(dv + b0 + r);
  }
  float wreg[FPT][kMaxA + 1];
  float gacc[FPT][kMaxA + 1];
  float dsum[FPT];
#pragma unroll
  for (int q = 0; q < FPT; ++q) {
    const int f = tid + q * kHbThreads;
    dsum[q] = 0.f;
#pragma unroll
    for (int a = 0; a <= kMaxA; ++a) {
      gacc[q][a] = 0.f;
      wreg[q][a] = 0.f;
      if (f < F && a < A) wreg[q][a] = __ldg(wa + (int64_t)f * A + a);
      if (f < F && a == A) wreg[q][a] = __ldg(wc + f);
    }
  }
  __syncthreads();
  for (int r = 0; r < nb; ++r) {
#pragma unroll
    for (int q = 0; q < FPT; ++q) {
      const int f = tid + q * kHbThreads;
      if (f < F) {
        const int64_t hi_ = (b0 + r) * F + f;
        const float hv = (h != nullptr) ? __ldg(h + hi_) : split_load(h_hi, h_lo, hi_);
        float g = 0.f;
#pragma unroll
        for (int a = 0; a <= kMaxA; ++a) {
          if (a < A1) {
            const float d = sd[r][a];
            gacc[q][a] = fmaf(hv, d, gacc[q][a]);
            g = fmaf(d, wreg[q][a], g);
          }
        }
        const float gm = hv > 0.f ? g : 0.f;
        if (dh != nullptr) {
          dh[hi_] = gm;
        } else {      // bf16-split planes for the tensor-core data/weight-gradient kernels; db of the hidden layer here
          const __nv_bfloat16 gh = __float2bfloat16_rn(gm);
          dh_hi[hi_] = __bfloat16_as_ushort(gh);
          dh_lo[hi_] = __bfloat16_as_ushort(__float2bfloat16_rn(gm - __bfloat162float(gh)));
          dsum[q] += gm;
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < FPT; ++q) {
    const int f = tid + q * kHbThreads;
    if (f < F) {
#pragma unroll
      for (int a = 0; a <= kMaxA; ++a) {
        if (a < A) atomicAdd(dwa + (int64_t)f * A + a, gacc[q][a]);
        if (a == A) atomicAdd(dwc + f, gacc[q][a]);
      }
      if (dbh != nullptr) atomicAdd(dbh + f, dsum[q]);
    }
  }
  if (tid < A1) {
    float s = 0.f;
    for (int r = 0; r < nb; ++r) s += sd[r][tid];
    if (tid < A) atomicAdd(dba + tid, s); else atomicAdd(dbc, s);
  }
}

// ------------------------------------------------------------------------------------------------
// bf16-split fast paths (F = 512): 8-byte plane loads, conflict-free 16-byte weight reads, more loads in flight.
// The first versions read the planes 2 bytes at a time in 16 dependent iterations per sample and sat at 6 % of HBM.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void unpack4(uint2 hi, uint2 lo, float (&x)[4]) {
  x[0] = __uint_as_float(hi.x << 16) + __uint_as_float(lo.x << 16);
  x[1] = __uint_as_float(hi.x & 0xffff0000u) + __uint_as_float(lo.x & 0xffff0000u);
  x[2] = __uint_as_float(hi.y << 16) + __uint_as_float(lo.y << 16);
  x[3] = __uint_as_float(hi.y & 0xffff0000u) + __uint_as_float(lo.y & 0xffff0000u);
}

// kHsF = hidden width: 512 (Nature) or 256 (NIPS)
template <int kHsF>
__global__ void __launch_bounds__(kHeadWarps * 32)
heads_fwd_split_kernel(const uint16_t* __restrict__ h_hi, const uint16_t* __restrict__ h_lo, const float* __restrict__ wa,
                       const float* __restrict__ ba, const float* __restrict__ wc, const float* __restrict__ bc, int64_t batch,
                       int A, float* __restrict__ pi, float* __restrict__ v, const SampleSrc smp,
                       int32_t* __restrict__ actions, float* __restrict__ onehot) {
  extern __shared__ __align__(16) float sw[];          // [A+1][F]: actor rows then the critic row
  const int A1 = A + 1;
  pdl_launch_dependents();                             // tc_ptx.cuh: launched as a programmatic dependent of the fc GEMM
  for (int i = threadIdx.x; i < kHsF * A1; i += blockDim.x) {
    const int a = i / kHsF, f = i - a * kHsF;
    sw[i] = (a < A) ? __ldg(wa + (int64_t)f * A + a) : __ldg(wc + f);
  }
  __syncthreads();
  pdl_wait();                                          // the head weights above depend on no kernel of this forward
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int64_t b = (int64_t)blockIdx.x * kHeadWarps + warp; b < batch; b += (int64_t)gridDim.x * kHeadWarps) {
    // lane's features: 128 * j + 4 * lane + e  (j < F / 128, e = 0..3): every warp load covers 256 contiguous bytes of a plane
    constexpr int NJ = kHsF / 128;
    float x[NJ][4];
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      const int64_t o = b * kHsF + 128 * j + 4 * lane;
      unpack4(__ldg(reinterpret_cast<const uint2*>(h_hi + o)), __ldg(reinterpret_cast<const uint2*>(h_lo + o)), x[j]);
    }
    float acc[kMaxA + 1];
#pragma unroll
    for (int a = 0; a <= kMaxA; ++a) {
      acc[a] = 0.f;
      if (a < A1) {
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
          const float4 w = *reinterpret_cast<const float4*>(sw + a * kHsF + 128 * j + 4 * lane);
          acc[a] = fmaf(x[j][0], w.x, fmaf(x[j][1], w.y, fmaf(x[j][2], w.z, fmaf(x[j][3], w.w, acc[a]))));
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc[a] += __shfl_xor_sync(0xffffffffu, acc[a], o);
      }
    }
    float z = -INFINITY, val = 0.f;
#pragma unroll
    for (int a = 0; a <= kMaxA; ++a) {
      if (a < A && lane == a) z = acc[a] + __ldg(ba + a);
      if (a == A) val = acc[a] + __ldg(bc);
    }
    float mx = z;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    const float e = (lane < A) ? expf(z - mx) : 0.f;
    float sum = e;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float p = e / sum;
    if (lane < A) pi[b * A + lane] = p;
    if (lane == 0) v[b] = val;
    if (smp.uniforms != nullptr || smp.rng != nullptr) {
      const float u = sample_uniform(smp, b);
      int act = A - 1;
      float c = 0.f;
      bool done = false;
      for (int j = 0; j < A - 1; ++j) {
        c += __shfl_sync(0xffffffffu, p, j);
        if (!done && u < c) { act = j; done = true; }
      }
      if (actions != nullptr && lane == 0) actions[b] = act;
      if (onehot != nullptr && lane < A) onehot[b * A + lane] = (lane == act) ? 1.f : 0.f;
    }
  }
}

// thread t owns the adjacent features 2t, 2t + 1 (one 32-bit word of each plane); 4 samples in flight
template <int kHsF>
__global__ void __launch_bounds__(kHsF / 2)
heads_bwd_split_kernel(const uint16_t* __restrict__ h_hi, const uint16_t* __restrict__ h_lo, uint16_t* __restrict__ dh_hi,
                       uint16_t* __restrict__ dh_lo, float* __restrict__ dbh, const float* __restrict__ wa,
                       const float* __restrict__ wc, const float* __restrict__ dlogits, const float* __restrict__ dv,
                       int64_t batch, int rows, int A, float* __restrict__ dwa, float* __restrict__ dba, float* __restrict__ dwc,
                       float* __restrict__ dbc) {
  // rows (<= kHbChunk) samples per CTA, chosen by the launcher (128: half the atomics per parameter of 64; a one-wave grid of
  // 70-row CTAs measured 10 % slower on the same box)
  __shared__ float sd[kHbChunk][kMaxA + 2];
  const int A1 = A + 1;
  const int tid = threadIdx.x;
  const int64_t b0 = (int64_t)blockIdx.x * rows;
  const int nb = (int)((batch - b0 < rows) ? batch - b0 : rows);
  for (int i = tid; i < rows * A1; i += kHsF / 2) {
    const int r = i / A1, a = i - r * A1;
    sd[r][a] = (r < nb) ? ((a < A) ? __ldg(dlogits + (b0 + r) * A + a) : __ldg(dv + b0 + r)) : 0.f;   // zero rows past the batch
  }
  const int f0 = 2 * tid;
  float w0[kMaxA + 1], w1[kMaxA + 1], g0[kMaxA + 1], g1[kMaxA + 1];
#pragma unroll
  for (int a = 0; a <= kMaxA; ++a) {
    g0[a] = g1[a] = w0[a] = w1[a] = 0.f;
    if (a < A) { w0[a] = __ldg(wa + (int64_t)f0 * A + a); w1[a] = __ldg(wa + (int64_t)(f0 + 1) * A + a); }
    if (a == A) { w0[a] = __ldg(wc + f0); w1[a] = __ldg(wc + f0 + 1); }
  }
  float ds0 = 0.f, ds1 = 0.f;
  __syncthreads();
  const uint32_t* hh = reinterpret_cast<const uint32_t*>(h_hi) + (b0 * kHsF + f0) / 2;
  const uint32_t* hl = reinterpret_cast<const uint32_t*>(h_lo) + (b0 * kHsF + f0) / 2;
  uint32_t* oh = reinterpret_cast<uint32_t*>(dh_hi) + (b0 * kHsF + f0) / 2;
  uint32_t* ol = reinterpret_cast<uint32_t*>(dh_lo) + (b0 * kHsF + f0) / 2;
  for (int r0 = 0; r0 < nb; r0 += 4) {
    uint32_t wh[4], wl[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool in = r0 + u < nb;
      wh[u] = in ? __ldg(hh + (int64_t)(r0 + u) * (kHsF / 2)) : 0u;
      wl[u] = in ? __ldg(hl + (int64_t)(r0 + u) * (kHsF / 2)) : 0u;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int r = r0 + u;
      if (r < nb) {
        const float x0 = __uint_as_float(wh[u] << 16) + __uint_as_float(wl[u] << 16);
        const float x1 = __uint_as_float(wh[u] & 0xffff0000u) + __uint_as_float(wl[u] & 0xffff0000u);
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int a = 0; a <= kMaxA; ++a) {
          if (a < A1) {
            const float d = sd[r][a];
            g0[a] = fmaf(x0, d, g0[a]);
            g1[a] = fmaf(x1, d, g1[a]);
            s0 = fmaf(d, w0[a], s0);
            s1 = fmaf(d, w1[a], s1);
          }
        }
        s0 = x0 > 0.f ? s0 : 0.f;                       // ReLU of the hidden layer
        s1 = x1 > 0.f ? s1 : 0.f;
        const __nv_bfloat162 hi2 = __floats2bfloat162_rn(s0, s1);
        const uint32_t hw = *reinterpret_cast<const uint32_t*>(&hi2);
        const __nv_bfloat162 lo2 = __floats2bfloat162_rn(s0 - __uint_as_float(hw << 16), s1 - __uint_as_float(hw & 0xffff0000u));
        oh[(int64_t)r * (kHsF / 2)] = hw;
        ol[(int64_t)r * (kHsF / 2)] = *reinterpret_cast<const uint32_t*>(&lo2);
        ds0 += s0;
        ds1 += s1;
      }
    }
  }
#pragma unroll
  for (int a = 0; a <= kMaxA; ++a) {
    if (a < A) { atomicAdd(dwa + (int64_t)f0 * A + a, g0[a]); atomicAdd(dwa + (int64_t)(f0 + 1) * A + a, g1[a]); }
    if (a == A) { atomicAdd(dwc + f0, g0[a]); atomicAdd(dwc + f0 + 1, g1[a]); }
  }
  if (dbh != nullptr) { atomicAdd(dbh + f0, ds0); atomicAdd(dbh + f0 + 1, ds1); }
  if (tid < A1) {
    float s = 0.f;
    for (int r = 0; r < nb; ++r) s += sd[r][tid];
    if (tid < A) atomicAdd(dba + tid, s); else atomicAdd(dbc, s);
  }
}

int launch_heads_fwd(const paacb_ctx* ctx, const float* h, const uint16_t* h_hi, const uint16_t* h_lo, const float* wa, const float* ba, const float* wc,
                     const float* bc, int64_t batch, float* pi, float* v, const float* uniforms, const uint64_t* rng,
                     uint64_t draw, int64_t first_sample, int32_t* actions, float* onehot, cudaStream_t st) {
  if (batch == 0) return PAACB_OK;
  const int F = ctx->feat, A = ctx->num_actions;
  // one sample per warp, up to 8 CTAs per SM: the kernel is latency-bound per sample, and wider is faster (measured: four
  // samples per warp on 2 CTAs per SM, to amortise the weight staging, took 0.175 instead of 0.130 ms per step on the same box)
  int64_t blocks = (batch + kHeadWarps - 1) / kHeadWarps;
  const int64_t cap = (int64_t)ctx->num_sms * 8;
  if (blocks > cap) blocks = cap;
  const size_t smem = (size_t)F * (A + 1) * sizeof(float);
  const SampleSrc smp = {uniforms, rng, draw, first_sample};
  if (h == nullptr && (F == 512 || F == 256)) {
    PAACB_LAUNCH_BEGIN(ctx, K_HEADS_FWD, st);
    if (F == 512)
      launch_kernel(heads_fwd_split_kernel<512>, (unsigned)blocks, kHeadWarps * 32, smem, st, h_hi, h_lo, wa, ba, wc, bc,
                    batch, A, pi, v, smp, actions, onehot);
    else
      launch_kernel(heads_fwd_split_kernel<256>, (unsigned)blocks, kHeadWarps * 32, smem, st, h_hi, h_lo, wa, ba, wc, bc,
                    batch, A, pi, v, smp, actions, onehot);
    PAACB_LAUNCH_END(ctx, K_HEADS_FWD, st);
    return PAACB_OK;
  }
  PAACB_LAUNCH_BEGIN(ctx, K_HEADS_FWD, st);
  heads_fwd_kernel<<<(unsigned)blocks, kHeadWarps * 32, smem, st>>>(h, h_hi, h_lo, wa, ba, wc, bc, batch, F, A, pi, v, smp,
                                                                     actions, onehot);
  PAACB_LAUNCH_END(ctx, K_HEADS_FWD, st);
  return PAACB_OK;
}

int launch_heads_bwd(const paacb_ctx* ctx, const float* h, const uint16_t* h_hi, const uint16_t* h_lo, uint16_t* dh_hi,
                     uint16_t* dh_lo, float* dbh, const float* wa, const float* wc, const float* dlogits,
                     const float* dv, int64_t batch, float* dh, float* dwa, float* dba, float* dwc, float* dbc,
                     cudaStream_t st) {
  if (batch == 0) return PAACB_OK;
  const int F = ctx->feat, A = ctx->num_actions;
  unsigned blocks = (unsigned)((batch + kHbChunk - 1) / kHbChunk);
  const int rows = kHbChunk;
  if (F > 2 * kHbThreads) { set_error("heads_bwd: hidden width > 512 unsupported"); return PAACB_EUNSUPPORTED; }
  if (h == nullptr && dh == nullptr && (F == 512 || F == 256)) {
    PAACB_LAUNCH_BEGIN(ctx, K_HEADS_BWD, st);
    if (F == 512)
      heads_bwd_split_kernel<512><<<(unsigned)((batch + rows - 1) / rows), 256, 0, st>>>(h_hi, h_lo, dh_hi, dh_lo, dbh, wa, wc, dlogits, dv, batch, rows, A, dwa, dba,
                                                          dwc, dbc);
    else
      heads_bwd_split_kernel<256><<<(unsigned)((batch + rows - 1) / rows), 128, 0, st>>>(h_hi, h_lo, dh_hi, dh_lo, dbh, wa, wc, dlogits, dv, batch, rows, A, dwa, dba,
                                                          dwc, dbc);
    PAACB_LAUNCH_END(ctx, K_HEADS_BWD, st);
    return PAACB_OK;
  }
  PAACB_LAUNCH_BEGIN(ctx, K_HEADS_BWD, st);
  if (F <= kHbThreads)
    heads_bwd_kernel<1><<<blocks, kHbThreads, 0, st>>>(h, h_hi, h_lo, dh_hi, dh_lo, dbh, wa, wc, dlogits, dv, batch, F, A, dh, dwa, dba, dwc, dbc);
  else
    heads_bwd_kernel<2><<<blocks, kHbThreads, 0, st>>>(h, h_hi, h_lo, dh_hi, dh_lo, dbh, wa, wc, dlogits, dv, batch, F, A, dh, dwa, dba, dwc, dbc);
  PAACB_LAUNCH_END(ctx, K_HEADS_BWD, st);
  return PAACB_OK;
}

int launch_rng_advance(const paacb_ctx* ctx, uint64_t* rng, uint64_t n, cudaStream_t st) {
  PAACB_LAUNCH_BEGIN(ctx, K_HEADS_FWD, st);
  rng_advance_kernel<<<1, 1, 0, st>>>(rng, n);
  PAACB_LAUNCH_END(ctx, K_HEADS_FWD, st);
  return PAACB_OK;
}

}  // namespace paacb
