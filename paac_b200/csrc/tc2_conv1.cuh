// conv1 forward on the int8 tensor pipe: parameters, geometry and the kernel.  Design notes: tc2_conv1.cu.
#pragma once
#include "tc2.cuh"

namespace paacb {

// NC = output channels: 32 (Nature; bf16-split planes out) or 16 (NIPS; fp32 out, the tf32 pipeline's activation format)
template <int NC>
struct C1 {
  static constexpr int ND = 3 * NC;                          // MMA N: three digit images
  static constexpr int WBYTES = 2 * ND * 128;                // K = 256 bytes per row: two 128-byte K-blocks of ND rows
  static constexpr int EPI_WARPS = 8 * (NC / 16);            // 2 accumulator buffers x (NC / 16) channel groups x 4 TMEM lane quarters
  static constexpr int THREADS = 64 + 32 * EPI_WARPS;
  static_assert(NC == 16 || NC == 32, "conv1 has 16 or 32 output channels");
  static_assert(WBYTES % 1024 == 0, "1024-byte aligned regions");
};
constexpr int kC1_WU = 21, kC1_HQ = 21, kC1_OH = 20, kC1_OW = 20;
// A tile is SIX plane rows (6 x 21 = 126 of the 128 MMA rows): a thread's position inside its plane row is a kernel constant.
// Epilogue history, all measured (profiles/r01_*): (1) 16-byte stores from registers at a 64-byte lane stride: 16 L1
// wavefronts per store instruction, l1tex at 72 % with DRAM at 47 % -- 0.95 ms per step; (2) a swizzled staging tile
// drained by TMA stores, two tiles in flight: 0.89-0.92 ms, half of it the per-tile skeleton (two 256-thread barriers, a
// proxy fence and the wait for the TMA engine); (3) 16 epilogue warps, each thread owning 16 channels of one position =
// exactly ONE 256-bit store (a full 32-byte sector) per plane, no shared memory, no barrier: 0.64 ms.
constexpr int kC1_TROWS = 6;
constexpr int kC1_ROWS = kC1_TROWS + 1;                // + 1 plane row for the filter rows kh >= 4
constexpr int kC1_PLANE = 16 * kC1_WU * kC1_ROWS;      // 2,352 bytes per parity plane patch
constexpr int kC1_BOX = 4 * kC1_PLANE;                 // one TMA box per tile: [4 parities][7 plane rows][336 bytes]
constexpr int kC1_SLOT = 10240;                        // >= 3 planes + (127 + 21 + 2) units: the two spare MMA rows read stale bytes
constexpr int kC1_NSLOTS = 6;                            // six tiles of patches in flight
constexpr int kC1_SMEM_FIXED = kC1_NSLOTS * kC1_SLOT + 256 + 1024 + (2 * kC1_NSLOTS + 5) * 8 + 16;   // + C1<NC>::WBYTES
constexpr int kC1_TMEM = 256;                            // two accumulator buffers of <= 96 columns at 0 and 128
static_assert((kC1_NSLOTS * kC1_SLOT) % 1024 == 0, "1024-byte aligned regions");
static_assert(3 * kC1_PLANE + (127 + kC1_WU + 2) * 16 <= kC1_SLOT, "slot holds every byte an MMA row can address");

struct Conv1Params {
  CUtensorMap tmA;         // uint8 states as (84 words = one 336-byte image row, b * 21 plane rows, 4 row parities)
  CUtensorMap tmW;         // int8 digit image [96 rows = (digit, co)][256 k]
  int num_tiles;
  int batch;
  const float* bias;
  const float* wscale;     // [NC]: s_c / (63 * 255)
  float* out_f32;          // fp32 output [b, 20, 20, NC] (F32OUT variants) instead of the planes
  uint8_t* out_hi;
  uint8_t* out_lo;
  uint16_t* relu_bits;     // [b][2 planes][400 positions] uint16, plane h bit relu1_bit_pos(c) = (channel 16 h + c > 0); nullptr: not wanted (tc2.cuh)
};

// D[tmem] (+)= A[smem] * B[smem], kind::i8 (uint8 x int8 -> int32), K = 32 per instruction
__device__ __forceinline__ void umma_i8(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D = int32, A = unsigned 8-bit, B = signed 8-bit, both K-major, M = 128
__host__ __device__ constexpr uint32_t make_idesc_i8(int n) {
  return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}

// An epilogue thread owns 16 channels of one tile row: NC / 16 warps share a tile row (Nature: 16 epilogue warps hide the
// TMEM / shared-memory / barrier / store latencies of an HBM-bound kernel).
template <int NC, bool F32OUT>
__global__ void __launch_bounds__(C1<NC>::THREADS, 1) conv1_i8_kernel(const __grid_constant__ Conv1Params p) {
  const int cta = (int)blockIdx.x, ncta = (int)gridDim.x;   // persistent CTAs: this one's index, their count
  constexpr int kC1_ND = C1<NC>::ND, kC1_WBYTES = C1<NC>::WBYTES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* ring = smem;
  uint8_t* wsm = smem + kC1_NSLOTS * kC1_SLOT;
  float2* s_sb = reinterpret_cast<float2*>(wsm + kC1_WBYTES);       // per channel: (scale, bias)
  uint64_t* bars = reinterpret_cast<uint64_t*>(wsm + kC1_WBYTES + 256);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kC1_NSLOTS;
  uint64_t* w_bar = bars + 2 * kC1_NSLOTS;
  uint64_t* tfull_bar = w_bar + 1;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty_bar + 2);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;

  pdl_launch_dependents();                        // tc_ptx.cuh: the next kernel's prologue may run under this kernel's tail
  if (tid == 0) {
    for (int s = 0; s < kC1_NSLOTS; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(w_bar, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 128 * (NC / 16));
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.tmA);
    tma_prefetch_desc(&p.tmW);
    mbar_arrive_expect_tx(w_bar, kC1_WBYTES);     // the weights depend on no kernel of this forward: loaded before pdl_wait
    tma_load_2d(wsm, &p.tmW, 0, 0, w_bar);
    tma_load_2d(wsm + kC1_ND * 128, &p.tmW, 128, 0, w_bar);
  }
  if (tid >= 64 && tid < 64 + NC) s_sb[tid - 64] = make_float2(__ldg(p.wscale + tid - 64), __ldg(p.bias + tid - 64));
  if (warp == 1) tmem_alloc(tmem_slot, kC1_TMEM);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (elect_one_sync()) {
      int slot = 0;
      uint32_t phase = 0;
      for (int tile = cta; tile < p.num_tiles; tile += ncta) {
        mbar_wait(&empty_bar[slot], phase ^ 1u);
        mbar_arrive_expect_tx(&full_bar[slot], kC1_BOX);
        tma_load_3d(ring + slot * kC1_SLOT, &p.tmA, 0, tile * kC1_TROWS, 0, &full_bar[slot]);
        if (++slot == kC1_NSLOTS) { slot = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one_sync();
    constexpr uint32_t idesc = make_idesc_i8(kC1_ND);
    const uint64_t adesc0 = make_smem_desc(0, 16, 128, SWZ_NONE);       // rows 16 B apart, K chunks 16 B apart (overlapping windows)
    const uint64_t bdesc0 = make_smem_desc(0, 16, 1024, SWZ_128B);
    const uint32_t ring_a = smem_u32(ring), w_a = smem_u32(wsm);
    mbar_wait(w_bar, 0);
    int slot = 0;
    uint32_t phase = 0;
    int tl = 0;
    for (int tile = cta; tile < p.num_tiles; tile += ncta, ++tl) {
      const int ab = tl & 1;
      const uint32_t aph = (uint32_t)((tl >> 1) & 1);
      mbar_wait(&tempty_bar[ab], aph ^ 1u);
      tc_fence_after();
      const uint32_t d0 = tmem_base + (uint32_t)(ab * 128);
      mbar_wait(&full_bar[slot], phase);
      tc_fence_after();
      if (leader) {
#pragma unroll
        for (int kh = 0; kh < 8; ++kh) {           // filter row kh: parity plane kh & 3, one plane row further down for kh >= 4
          const uint32_t a = ring_a + (uint32_t)(slot * kC1_SLOT + (kh & 3) * kC1_PLANE + (kh >> 2) * kC1_WU * 16);
          const uint64_t bd = desc_with_addr(bdesc0, w_a + (uint32_t)((kh / 4) * (kC1_ND * 128) + (kh % 4) * 32));
          umma_i8(d0, desc_with_addr(adesc0, a), bd, idesc, kh ? 1u : 0u);
        }
        umma_commit(&empty_bar[slot]);
      }
      __syncwarp();
      if (++slot == kC1_NSLOTS) { slot = 0; phase ^= 1u; }
      if (leader) umma_commit(&tfull_bar[ab]);
      __syncwarp();
    }
  } else {
    // =========================== epilogue ===========================
    const int ew = warp & 3;
    const int r = ew * 32 + lane;                   // MMA row = unit r of the tile's 6 x 21 units
    const int grp = ((warp - 2) >> 2) & 1;          // epilogue group = accumulator buffer it drains
    const int cg = (warp - 2) >> 3;                 // this thread's 16-channel group
    const int pr = r / kC1_WU, ju = r - pr * kC1_WU;
    const bool rowok = (r < kC1_TROWS * kC1_WU) && (ju < kC1_OW);
    for (int tl = grp, tile = cta + grp * ncta; tile < p.num_tiles; tile += 2 * ncta, tl += 2) {
      const uint32_t aph = (uint32_t)((tl >> 1) & 1);
      const uint32_t g = (uint32_t)tile * kC1_TROWS + (uint32_t)pr;           // global plane row
      const uint32_t n = g / (uint32_t)kC1_HQ;
      const bool ok = rowok && ((int)(g - n * (uint32_t)kC1_HQ) < kC1_OH) && ((int)n < p.batch);
      mbar_wait(&tfull_bar[grp], aph);
      tc_fence_after();
      uint32_t v0[16], v1[16], v2[16];
      const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(grp * 128 + cg * 16);
      tmem_ld16(tcol, v0);
      tmem_ld16(tcol + (uint32_t)NC, v1);
      tmem_ld16(tcol + (uint32_t)(2 * NC), v2);
      tmem_ld_wait();
      tc_fence_before();
      mbar_arrive(&tempty_bar[grp]);           // the accumulator is in registers: release the buffer before the arithmetic
      uint32_t hw[8], lw[8];
      float of[F32OUT ? 16 : 1];
      const float4* sb4 = reinterpret_cast<const float4*>(s_sb) + cg * 8;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 sb = sb4[j];              // (scale, bias) of channels 2j, 2j + 1: one broadcast 16-byte load
        float o[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          // |acc| < 2^22: int -> float exactly on the integer + FMA pipes (the conversion pipe issues at a quarter rate)
          const float f0 = __uint_as_float(v0[2 * j + e] + 0x4B400000u) - 12582912.0f;
          const float f1 = __uint_as_float(v1[2 * j + e] + 0x4B400000u) - 12582912.0f;
          const float f2 = __uint_as_float(v2[2 * j + e] + 0x4B400000u) - 12582912.0f;
          const float t = fmaf(f2, 1.0f / 4096.0f, fmaf(f1, 1.0f / 64.0f, f0));
          o[e] = fmaxf(fmaf(t, e ? sb.z : sb.x, e ? sb.w : sb.y), 0.f);
        }
        if constexpr (F32OUT) { of[2 * j] = o[0]; of[2 * j + 1] = o[1]; }
        else split_bf16x2(o[0], o[1], hw[j], lw[j]);
      }
      if (ok) {                 // 16 channels = one full 32-byte sector per plane
        const uint32_t oh = g - n * (uint32_t)kC1_HQ;
        if constexpr (!F32OUT) {
          if (p.relu_bits != nullptr) {
            // the ReLU mask conv2's data gradient needs, as bits.  The outputs are >= +0, so "hi > 0" is "the bf16 half is not
            // zero", and w + 0x7fff7fff sets bit 15 / bit 31 exactly when the low / high half of w is non-zero (a positive bf16
            // is <= 0x7f80: no carry between the halves).  Word j's two flags are shifted to bits 15 - j / 31 - j and OR-ed:
            // three instructions per pair of channels in this ALU-bound epilogue; relu1_bit_pos() is the resulting layout.
            const int64_t px = (int64_t)n * (2 * kC1_OH * kC1_OW) + oh * kC1_OW + ju;      // plane 0 of sample n
            uint32_t acc = 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) acc |= ((hw[j] + 0x7fff7fffu) >> j) & (0x80008000u >> j);
            const uint32_t bits = ((acc >> 8) & 0xffu) | ((acc >> 16) & 0xff00u);
            p.relu_bits[px + cg * (kC1_OH * kC1_OW)] = (uint16_t)bits;
          }
        }
        const int64_t oe = (((int64_t)n * kC1_OH + oh) * kC1_OW + ju) * NC + cg * 16;      // element index
        if constexpr (F32OUT) {
          stg256(p.out_f32 + oe, reinterpret_cast<const uint32_t*>(of));
          stg256(p.out_f32 + oe + 8, reinterpret_cast<const uint32_t*>(of) + 8);
        } else {
          stg256(p.out_hi + oe * 2, hw);
          stg256(p.out_lo + oe * 2, lw);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kC1_TMEM);
  }
}

}  // namespace paacb
