// Streaming GEMM of the fully connected layer (forward, data gradient, weight gradient): parameters and the kernel.
// Design: tc2_stream.cu.
#pragma once
#include "tc2.cuh"

namespace paacb {

enum { ST_FWD = 0, ST_DGRAD = 1, ST_WGRAD = 2 };

struct StreamParams {
  CUtensorMap tmA[2];
  CUtensorMap tmB[2];
  int m_tiles, n_tiles, k_splits;
  int kblocks_per_split;     // 64-wide reduction blocks per unit
  int kblocks_total;
  int M, N;                  // valid output rows / columns
  int ldo;                   // output row length in elements
  const float* bias;
  uint8_t* out_hi;
  uint8_t* out_lo;
  const uint8_t* mask_hi;
  float* dbias;              // dgrad: += column sums, column c -> dbias[c % dbias_mod]
  int dbias_mod;
  float* dw;                 // wgrad target (fp32, atomics)
};

template <int BN, int MODE>
struct StreamCfg {
  static constexpr bool MN = (MODE == ST_WGRAD);
  static constexpr int A_PIECE = 128 * 128;                 // 128 rows x 64 k (K-major) or 2 x (64 rows x 64 m) (MN-major)
  static constexpr int B_PIECE = BN * 128;
  static constexpr int STAGE_BYTES = 2 * A_PIECE + 2 * B_PIECE;
  static constexpr int STAGES = (200 * 1024) / STAGE_BYTES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + (2 * STAGES + 4) * 8 + 16;
  static constexpr int TMEM_COLS = 4 * BN;                  // two buffers of [A_hi*B_hi + A_lo*B_hi | A_hi*B_lo]
  static_assert(2 * BN <= 256, "MMA N");
  static_assert(STAGES >= 2, "pipeline too shallow");
};

constexpr int kStreamThreads = 192;
constexpr int kFcBN = 128;               // output columns per unit of the fc GEMMs

__device__ __forceinline__ float warp_transpose_sum32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool up = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = up ? v[i] : v[i + off];
      const float keep = up ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

template <int BN, int MODE>
__global__ void __launch_bounds__(kStreamThreads, 1) stream_gemm_kernel(const __grid_constant__ StreamParams p) {
  const int cta = (int)blockIdx.x, ncta = (int)gridDim.x;   // persistent CTAs: this one's index, their count
  using Cfg = StreamCfg<BN, MODE>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr bool MN = Cfg::MN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tfull_bar = bars + 2 * STAGES;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  const int units = p.m_tiles * p.n_tiles * p.k_splits;

  pdl_launch_dependents();                        // tc_ptx.cuh: the next kernel's prologue may run under this kernel's tail
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 128);
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmB[0]);
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_slot;

  // unit -> (split, m-tile, n-tile); n fastest so that CTAs running together share the A tile in L2
  auto decode = [&](int u, int& split, int& mt, int& nt) {
    nt = u % p.n_tiles;
    const int rest = u / p.n_tiles;
    mt = rest % p.m_tiles;
    split = rest / p.m_tiles;
  };
  auto kb_range = [&](int split, int& kb0, int& kb1) {
    kb0 = split * p.kblocks_per_split;
    kb1 = kb0 + p.kblocks_per_split;
    if (kb1 > p.kblocks_total) kb1 = p.kblocks_total;
  };

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = cta; u < units; u += ncta) {
        int split, mt, nt, kb0, kb1;
        decode(u, split, mt, nt);
        kb_range(split, kb0, kb1);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          mbar_arrive_expect_tx(&full_bar[stage], Cfg::STAGE_BYTES);
          uint8_t* st = smem + stage * Cfg::STAGE_BYTES;
#pragma unroll
          for (int piece = 0; piece < 2; ++piece) {
            uint8_t* a = st + piece * Cfg::A_PIECE;
            uint8_t* b = st + 2 * Cfg::A_PIECE + piece * Cfg::B_PIECE;
            if constexpr (MN) {
              // boxes of (64 columns, 64 reduction rows): A columns = weight rows k, B columns = output channels n
#pragma unroll
              for (int i = 0; i < 2; ++i) tma_load_2d(a + i * 8192, &p.tmA[piece], mt * 128 + i * 64, kb * 64, &full_bar[stage]);
#pragma unroll
              for (int i = 0; i < BN / 64; ++i) tma_load_2d(b + i * 8192, &p.tmB[piece], nt * BN + i * 64, kb * 64, &full_bar[stage]);
            } else {
              tma_load_2d(a, &p.tmA[piece], kb * 64, mt * 128, &full_bar[stage]);      // box (64 k, 128 rows)
              tma_load_2d(b, &p.tmB[piece], kb * 64, nt * BN, &full_bar[stage]);       // box (64 k, BN rows)
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one_sync();
    // B_hi and B_lo lie back to back in the stage: one MMA of N = 2 * BN evaluates A_hi * [B_hi | B_lo] (A is read from
    // shared memory once), a second of N = BN adds A_lo * B_hi into the first half; the epilogue adds the halves.
    constexpr uint32_t idesc_full = make_idesc_bf16(2 * BN, MN ? 1 : 0, MN ? 1 : 0);
    constexpr uint32_t idesc_half = make_idesc_bf16(BN, MN ? 1 : 0, MN ? 1 : 0);
    const uint64_t desc0 = MN ? make_smem_desc(0, 8192, 1024, SWZ_128B) : make_smem_desc(0, 16, 1024, SWZ_128B);
    constexpr uint32_t kstep_bytes = MN ? 2048u : 32u;
    int stage = 0;
    uint32_t phase = 0;
    int tl = 0;
    for (int u = cta; u < units; u += ncta, ++tl) {
      int split, mt, nt, kb0, kb1;
      decode(u, split, mt, nt);
      kb_range(split, kb0, kb1);
      const int ab = tl & 1;
      const uint32_t aph = (uint32_t)((tl >> 1) & 1);
      mbar_wait(&tempty_bar[ab], aph ^ 1u);
      tc_fence_after();
      const uint32_t d = tmem_base + (uint32_t)(ab * 2 * BN);
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after();
        if (leader) {
          const uint32_t st = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint32_t a_hi = st, a_lo = st + Cfg::A_PIECE;
          const uint32_t b_hi = st + 2 * Cfg::A_PIECE;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {
            const uint32_t o = (uint32_t)ks * kstep_bytes;
            const uint64_t bd = desc_with_addr(desc0, b_hi + o);
            umma_bf16(d, desc_with_addr(desc0, a_hi + o), bd, idesc_full, (kb > kb0 || ks > 0) ? 1u : 0u);
            umma_bf16(d, desc_with_addr(desc0, a_lo + o), bd, idesc_half, 1u);
          }
          umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
      if (leader) umma_commit(&tfull_bar[ab]);
      __syncwarp();
    }
  } else {
    // =========================== epilogue ===========================
    const int ew = warp & 3;
    const int r = ew * 32 + lane;
    // dgrad bias sums kept in registers across tiles when the column -> channel map is tile-invariant
    // (channel = column % 64 and tiles start at multiples of 64): bsum[j] belongs to channel 32 * j + lane
    // (per-thread sums over this thread's rows; the transposed warp reduction runs once at the end of the kernel)
    float bs[MODE == ST_DGRAD ? 2 : 1][32];
#pragma unroll
    for (int i = 0; i < (MODE == ST_DGRAD ? 2 : 1); ++i)
#pragma unroll
      for (int j = 0; j < 32; ++j) bs[i][j] = 0.f;
    const bool reg_sums = (MODE == ST_DGRAD) && p.dbias != nullptr && p.dbias_mod == 64;
    int tl = 0;
    for (int u = cta; u < units; u += ncta, ++tl) {
      int split, mt, nt;
      decode(u, split, mt, nt);
      const int ab = tl & 1;
      const uint32_t aph = (uint32_t)((tl >> 1) & 1);
      const int m = mt * 128 + r;
      const bool ok = m < p.M;
      // dgrad: prefetch the ReLU-mask words of this row before waiting for the MMAs (their latency overlaps the mainloop)
      uint4 mk[MODE == ST_DGRAD ? BN / 32 : 1][4];
      if constexpr (MODE == ST_DGRAD) {
#pragma unroll
        for (int c = 0; c < BN / 32; ++c) {
          const int n0 = nt * BN + c * 32;
#pragma unroll
          for (int j = 0; j < 4; ++j) mk[c][j] = make_uint4(0u, 0u, 0u, 0u);
          if (ok && n0 < p.N) {
            const uint8_t* mp = p.mask_hi + ((int64_t)m * p.ldo + n0) * 2;
            ldg256(mp, mk[c][0], mk[c][1]);
            ldg256(mp + 32, mk[c][2], mk[c][3]);
          }
        }
      }
      mbar_wait(&tfull_bar[ab], aph);
      tc_fence_after();
#pragma unroll
      for (int c0 = 0; c0 < BN; c0 += 32) {
        const int n0 = nt * BN + c0;
        uint32_t v[32], v2[32];
        const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(ab * 2 * BN + c0);
        tmem_ld32(tcol, v);
        tmem_ld32(tcol + (uint32_t)BN, v2);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v2[j]));
        if (n0 >= p.N) continue;                 // warp-uniform: N is a multiple of 32
        if constexpr (MODE == ST_WGRAD) {
          if (ok) {
            float4* dst = reinterpret_cast<float4*>(p.dw + (int64_t)m * p.ldo + n0);      // RED.ADD.F32x4
#pragma unroll
            for (int j = 0; j < 8; ++j)
              atomicAdd(dst + j, make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]), __uint_as_float(v[4 * j + 2]),
                                             __uint_as_float(v[4 * j + 3])));
          }
        } else {
          const int64_t obase = (int64_t)m * p.ldo + n0;
          float o[32];
          if constexpr (MODE == ST_DGRAD) {
            uint32_t mw[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 q = mk[c0 / 32][j];
              mw[4 * j] = q.x; mw[4 * j + 1] = q.y; mw[4 * j + 2] = q.z; mw[4 * j + 3] = q.w;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const uint32_t a0 = mw[j] & 0xffffu, a1 = mw[j] >> 16;
              o[2 * j] = (ok && a0 != 0u && a0 < 0x8000u) ? __uint_as_float(v[2 * j]) : 0.f;
              o[2 * j + 1] = (ok && a1 != 0u && a1 < 0x8000u) ? __uint_as_float(v[2 * j + 1]) : 0.f;
            }
          } else {
            const float4* b4 = reinterpret_cast<const float4*>(p.bias + n0);        // n0 is a multiple of 32: 16-byte aligned if bias is
#pragma unroll
            for (int j = 0; j < 8; ++j) {                                            // warp-uniform address: one broadcast 16-byte load per 4 columns
              const float4 bb = __ldg(b4 + j);
              o[4 * j] = fmaxf(__uint_as_float(v[4 * j]) + bb.x, 0.f);
              o[4 * j + 1] = fmaxf(__uint_as_float(v[4 * j + 1]) + bb.y, 0.f);
              o[4 * j + 2] = fmaxf(__uint_as_float(v[4 * j + 2]) + bb.z, 0.f);
              o[4 * j + 3] = fmaxf(__uint_as_float(v[4 * j + 3]) + bb.w, 0.f);
            }
          }
          if (ok) {
            uint32_t hw[16], lw[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) split_bf16x2(o[2 * j], o[2 * j + 1], hw[j], lw[j]);
            uint8_t* dh = p.out_hi + obase * 2;
            uint8_t* dl = p.out_lo + obase * 2;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              stg256(dh + 32 * j, hw + 8 * j);
              stg256(dl + 32 * j, lw + 8 * j);
            }
          }
          if constexpr (MODE == ST_DGRAD) {
            if (p.dbias != nullptr) {
              if (reg_sums) {
#pragma unroll
                for (int j = 0; j < 32; ++j) bs[(c0 >> 5) & 1][j] += o[j];
              } else {
                const float s = warp_transpose_sum32(o, lane);
                atomicAdd(p.dbias + ((n0 + lane) % p.dbias_mod), s);
              }
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[ab]);
    }
    if constexpr (MODE == ST_DGRAD) {
      if (reg_sums) {
        atomicAdd(p.dbias + lane, warp_transpose_sum32(bs[0], lane));
        atomicAdd(p.dbias + 32 + lane, warp_transpose_sum32(bs[1], lane));
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

}  // namespace paacb
