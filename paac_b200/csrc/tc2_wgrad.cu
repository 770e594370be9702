// bf16-split tensor-core path, part 3: conv weight gradients as patch-resident GEMMs with MN-major operands.
//
//   dW[k = (kh, kw, ci), co] = sum over (sample, oh, ow) of  X[sample, s*oh + kh, s*ow + kw, ci] * dZ[sample, oh, ow, co]
//
// The 128-row MMA dimension is a tile of k, N = Cout, and the reduction runs over output positions.  Both operands
// have the reduction index as their slow (row) index in HBM, which is exactly the MN-major shared-memory layout, so
// the TMA boxes are used as they land.  As in tc2_conv.cu the positions are enumerated over the INPUT grid
// (row-parity plane by row-parity plane) so every filter tap is a start-address offset into ONE resident input patch;
// dZ is fetched with a box one row/column larger than the tensor so the positions that are not real outputs read
// zeros (TMA out-of-bounds fill), and the rows of a slot the box never writes are zeroed once at kernel start.
// All k-tile accumulators of the layer stay in TMEM for the whole kernel (conv2: 4 x 64 columns, conv3: 5 x 64,
// conv1: 2 x 64); every CTA reduces a contiguous range of samples and adds its partial sums to dW with fp32 atomics
// once, at the end.  Bias gradients are produced by the kernels that write dZ (tc2_conv.cu, tc2_stream.cu, heads.cu).
#include "tc2.cuh"

namespace paacb {

template <int L>
struct Wg;

// conv1: X = bf16 states [b,84,84,4] (exact, one piece), dZ1 [b,20,20,32].  Stage = half a sample (224 positions).
// Units are 32 B (4 pixels x 4 channels): MN groups of 16 k.  The 8 groups of a 128-row MMA are the 4 row-parity planes
// (kh & 3; LBO = plane slot stride) for kw / 4 = 0 followed by the SAME 4 planes one unit (4 pixels) further for
// kw / 4 = 1: the converter warps write every unit twice, into slot p and, shifted by 32 bytes, into slot p + 4, so one
// MMA covers what were two half-empty k-tiles (the kernel is bound by its MMA count -- half the k-tiles took half the
// time -- while conversion and loads are free).  k-tile kt = kh / 4.
template <>
struct Wg<0> {
  static constexpr int A_PARTS = 8, A_PIECES = 1, A_SLOT = 9216, A_BOX = 16 * 2 * 21 * 13, B_SLOT = 16384, B_BOX = 64 * 21 * 12;
  static constexpr int STAGES = 2, KT = 2, BN = 32, KSTEPS = 14, A_KSTEP = 512, B_KSTEP = 1024;
  static constexpr int A_SWZ = SWZ_32B, A_SBO = 256, B_SWZ = SWZ_64B, B_SBO = 512;
  static constexpr int STAGES_PER_SAMPLE = 2, SAMPLES_PER_STAGE = 1;
  static constexpr int K = 256, KIND = 0, LAYER = 0, MROWS = 128, CONCAT_KT = 2;
  __device__ static constexpr int pos(int t) { return 16 * t; }
  __device__ static int a_off(int kt) { return kt * 21 * 32; }                               // within plane 0's slot
  __device__ static int a_lbo(int) { return A_SLOT; }
  // row m of k-tile kt -> weight row k = kh * 32 + kw * 4 + c: group g = m >> 4 is (kw / 4 = g >> 2, kh & 3 = g & 3)
  __device__ static int k_of(int kt, int m) { return (4 * kt + ((m >> 4) & 3)) * 32 + (m >> 6) * 16 + (m & 15); }
};
// conv2: X1 [b,20,20,32] (hi, lo), dZ2 [b,9,9,64].  Stage = one sample, 100 positions (10 x 10 over the parity plane).
template <>
struct Wg<1> {
  static constexpr int A_PARTS = 2, A_PIECES = 2, A_SLOT = 15360, A_BOX = 128 * 10 * 12, B_SLOT = 14336, B_BOX = 128 * 10 * 10;
  // K-steps: dZ2 is 9 x 9 inside the 10 x 10 enumeration, so the last position that carries data is 10 * 8 + 8 = 88:
  // 6 steps of 16 positions, not 7
  static constexpr int STAGES = 2, KT = 4, BN = 64, KSTEPS = 6, A_KSTEP = 2048, B_KSTEP = 2048;
  static constexpr int A_SWZ = SWZ_128B, A_SBO = 1024, B_SWZ = SWZ_128B, B_SBO = 1024;
  static constexpr int STAGES_PER_SAMPLE = 1, SAMPLES_PER_STAGE = 1;
  static constexpr int K = 512, KIND = 1, LAYER = 1, MROWS = 128, CONCAT_KT = 4;
  __device__ static constexpr int pos(int t) { return 16 * t; }
  __device__ static int a_off(int kt) { return (kt >> 1) * 10 * 128; }                       // kh = kt: plane kt & 1, row offset kt / 2
  __device__ static int a_lbo(int) { return 128; }
  __device__ static int k_of(int kt, int m) { return kt * 128 + m; }
};
// conv3: X2 [b,9,9,64] (hi, lo), dZ3 [b,7,7,64].  Stage = two samples, 162 positions (9 x 9 each).
template <>
struct Wg<2> {
  static constexpr int A_PARTS = 1, A_PIECES = 2, A_SLOT = 24576, A_BOX = 128 * 9 * 21, B_SLOT = 22528, B_BOX = 128 * 9 * 9 * 2;
  // K-steps: the reduction index of an MMA is 16 CONSECUTIVE positions starting anywhere (a start address, like a tap), so
  // the positions that carry no data are skipped: dZ3 is 7 x 7 inside the 9 x 9 enumeration, its last data position is
  // 9 * 6 + 6 = 60 -> 4 steps per sample starting at the sample's position 0 (8 per stage instead of the 11 a flat walk
  // over 162 positions takes).  TMEM: 3 k-tiles accumulate [X_hi^T dZ_hi + X_lo^T dZ_hi | X_hi^T dZ_lo] (two MMAs per
  // step, N = 128 and N = 64), the other 2 a single 64-column sum (three MMAs of N = 64): 3 * 128 + 2 * 64 = 512 columns.
  static constexpr int STAGES = 2, KT = 5, BN = 64, KSTEPS = 8, A_KSTEP = 2048, B_KSTEP = 2048;
  static constexpr int A_SWZ = SWZ_128B, A_SBO = 1024, B_SWZ = SWZ_128B, B_SBO = 1024;
  static constexpr int STAGES_PER_SAMPLE = 1, SAMPLES_PER_STAGE = 2;
  static constexpr int K = 576, KIND = 2, LAYER = 2, MROWS = 128, CONCAT_KT = 3;
  __device__ static constexpr int pos(int t) { return (t >> 2) * 81 + (t & 3) * 16; }
  __device__ static int tap_off(int tap) { return ((tap / 3) * 9 + (tap % 3)) * 128; }
  __device__ static int a_off(int kt) { return tap_off(2 * kt); }
  __device__ static int a_lbo(int kt) { return kt < 4 ? tap_off(2 * kt + 1) - tap_off(2 * kt) : 128; }
  __device__ static int k_of(int kt, int m) { return (kt * 128 + m < K) ? kt * 128 + m : -1; }
};

// ---- NIPS (networks.py:145-146): the same two kernels with narrower dZ operands ----
// conv1, 16 output channels: dZ1 [b,20,20,16] rows are 32 B (SWIZZLE_32B MN-major, like the X operand); everything on the X
// side (converter warps, merged k-tiles) is unchanged.
template <>
struct Wg<3> {
  static constexpr int A_PARTS = 8, A_PIECES = 1, A_SLOT = 9216, A_BOX = 16 * 2 * 21 * 13, B_SLOT = 8192, B_BOX = 32 * 21 * 12;
  static constexpr int STAGES = 2, KT = 2, BN = 16, KSTEPS = 14, A_KSTEP = 512, B_KSTEP = 512;
  static constexpr int A_SWZ = SWZ_32B, A_SBO = 256, B_SWZ = SWZ_32B, B_SBO = 256;
  static constexpr int STAGES_PER_SAMPLE = 2, SAMPLES_PER_STAGE = 1;
  static constexpr int K = 256, KIND = 0, LAYER = 0, MROWS = 128, CONCAT_KT = 2;
  __device__ static constexpr int pos(int t) { return 16 * t; }
  __device__ static int a_off(int kt) { return kt * 21 * 32; }
  __device__ static int a_lbo(int) { return A_SLOT; }
  __device__ static int k_of(int kt, int m) { return (4 * kt + ((m >> 4) & 3)) * 32 + (m >> 6) * 16 + (m & 15); }
};
// conv2: X1 [b,20,20,16] (hi, lo), dZ2 [b,9,9,32].  Units are 64 B (2 pixels x 16 channels): an MN group of a SWIZZLE_64B
// operand is 32 k = (kw pair, ci), so filter row kh is TWO groups (this unit and the next, LBO = 64) = 64 rows of the
// 128-row MMA; the other two groups read the units after them and are discarded (k_of = -1).  One k-tile per kh: the layer
// has a quarter of Nature's conv2 MACs and costs the same MMA count -- still 4x faster than the tf32 kernel it replaces.
template <>
struct Wg<4> {
  static constexpr int A_PARTS = 2, A_PIECES = 2, A_SLOT = 8192, A_BOX = 64 * 10 * 12, B_SLOT = 7168, B_BOX = 64 * 10 * 10;
  static constexpr int STAGES = 2, KT = 4, BN = 32, KSTEPS = 6, A_KSTEP = 1024, B_KSTEP = 1024;      // 6 steps: see Wg<1>
  static constexpr int A_SWZ = SWZ_64B, A_SBO = 512, B_SWZ = SWZ_64B, B_SBO = 512;
  static constexpr int STAGES_PER_SAMPLE = 1, SAMPLES_PER_STAGE = 1;
  static constexpr int K = 256, KIND = 1, LAYER = 1, MROWS = 64, CONCAT_KT = 4;
  __device__ static constexpr int pos(int t) { return 16 * t; }
  __device__ static int a_off(int kt) { return (kt >> 1) * 10 * 64; }                        // kh = kt: plane kt & 1, row offset kt / 2
  __device__ static int a_lbo(int) { return 64; }
  __device__ static int k_of(int kt, int m) { return m < 64 ? kt * 64 + m : -1; }
};

struct Wg2Params {
  CUtensorMap tmA[2];
  CUtensorMap tmB[2];
  int stages_total;
  int batch;
  const uint8_t* a_u8;    // conv1: the uint8 states [b, 84, 84, 4], converted to bf16 in shared memory, instead of tmA
  float* dw;              // [K, BN] fp32
  float w_scale;          // 1/255 for the uint8 layer (the operand holds the raw pixel values), else 1
};

template <int L>
struct Wg2Cfg {
  using W = Wg<L>;
  static constexpr int A_STAGE = W::A_PARTS * W::A_PIECES * W::A_SLOT;
  static constexpr int B_STAGE = 2 * W::B_SLOT;
  static constexpr int A_BYTES = W::STAGES * A_STAGE;
  static constexpr int DATA_BYTES = A_BYTES + W::STAGES * B_STAGE;
  static constexpr bool U8_A = (W::KIND == 0);                 // conv1: nine converter warps produce the X operand from the uint8 states
  static constexpr int TX_BYTES = (U8_A ? 0 : W::A_PARTS * W::A_PIECES * W::A_BOX) + 2 * W::B_BOX;
  static constexpr int CONV_THREADS = 288;               // conv1: nine converter warps, one 32-byte unit of each plane per thread (273 units)
  static constexpr int THREADS = 192 + (U8_A ? CONV_THREADS : 0);
  static constexpr int SMEM_BYTES = DATA_BYTES + 1024 + (2 * W::STAGES + 1) * 8 + 16;
  // dZ_hi and dZ_lo slots lie back to back: one MMA of N = 2 * BN evaluates X_hi^T * [dZ_hi | dZ_lo] (X is read from shared
  // memory once), a second of N = BN adds X_lo^T * dZ_hi.  The first CONCAT_KT k-tiles work that way (2 * BN columns each);
  // conv3's 5 x 128 columns do not fit in TMEM: its last two k-tiles keep three MMAs of N = BN per K-step (BN columns).
  static constexpr int NCAT = W::CONCAT_KT;
  __host__ __device__ static constexpr int acc_col(int kt) { return kt < NCAT ? kt * 2 * W::BN : NCAT * 2 * W::BN + (kt - NCAT) * W::BN; }
  static constexpr int ACC_TOTAL = NCAT * 2 * W::BN + (W::KT - NCAT) * W::BN;
  static constexpr int TMEM_COLS = (ACC_TOTAL <= 128) ? 128 : ((ACC_TOTAL <= 256) ? 256 : 512);
  static_assert(ACC_TOTAL <= 512, "TMEM columns");
  static_assert(W::A_BOX <= W::A_SLOT && W::B_BOX <= W::B_SLOT, "slot too small");
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
};


template <int L>
__global__ void __launch_bounds__(Wg2Cfg<L>::THREADS, 1) wgrad2_kernel(const __grid_constant__ Wg2Params p) {
  using W = Wg<L>;
  using Cfg = Wg2Cfg<L>;
  constexpr int STAGES = W::STAGES;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* a_sm = smem;                                  // [STAGES][A_PARTS][A_PIECES][A_SLOT]
  uint8_t* b_sm = smem + Cfg::A_BYTES;                   // [STAGES][2][B_SLOT]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::DATA_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* done_bar = bars + 2 * STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  // contiguous range of stages of this CTA
  const int per = (p.stages_total + (int)gridDim.x - 1) / (int)gridDim.x;
  const int s_begin = (int)blockIdx.x * per;
  const int s_end = (s_begin + per < p.stages_total) ? s_begin + per : p.stages_total;

  pdl_launch_dependents();                        // tc_ptx.cuh: the next kernel's prologue may run under this kernel's tail
  // zero the operand area once: rows of a slot the TMA boxes never write must read as 0 (dZ) / finite (X)
  for (int i = tid * 16; i < Cfg::DATA_BYTES; i += Cfg::THREADS * 16) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0u, 0u, 0u, 0u);
  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], Cfg::U8_A ? 1 + Cfg::CONV_THREADS : 1);      // TMA producer (+ the converter threads)
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(done_bar, 1);
    fence_barrier_init();
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmB[0]);
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                                     // the shared-memory zero fill above ran under the previous kernel's tail
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (elect_one_sync()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int s = s_begin; s < s_end; ++s) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        mbar_arrive_expect_tx(&full_bar[stage], Cfg::TX_BYTES);
        uint8_t* a = a_sm + stage * Cfg::A_STAGE;
        uint8_t* b = b_sm + stage * Cfg::B_STAGE;
        if constexpr (W::KIND == 0) {
          const int n = s >> 1, h = s & 1;
#pragma unroll
          (void)a;                                    // the X operand is written by the converter warps
#pragma unroll
          for (int piece = 0; piece < 2; ++piece) tma_load_4d(b + piece * W::B_SLOT, &p.tmB[piece], 0, 0, 10 * h, n, &full_bar[stage]);
          // two stages only: ask for the dZ boxes of the stage after next to be in L2 when their slot frees
          if (s + 2 < s_end) {
#pragma unroll
            for (int piece = 0; piece < 2; ++piece) tma_prefetch_4d(&p.tmB[piece], 0, 0, 10 * ((s + 2) & 1), (s + 2) >> 1);
          }
        } else if constexpr (W::KIND == 1) {
#pragma unroll
          for (int part = 0; part < 2; ++part)
#pragma unroll
            for (int piece = 0; piece < 2; ++piece)
              tma_load_4d(a + (part * 2 + piece) * W::A_SLOT, &p.tmA[piece], 0, 0, part, s * 10, &full_bar[stage]);
#pragma unroll
          for (int piece = 0; piece < 2; ++piece) tma_load_4d(b + piece * W::B_SLOT, &p.tmB[piece], 0, 0, 0, s, &full_bar[stage]);
        } else {
#pragma unroll
          for (int piece = 0; piece < 2; ++piece) tma_load_3d(a + piece * W::A_SLOT, &p.tmA[piece], 0, 0, s * 18, &full_bar[stage]);
#pragma unroll
          for (int piece = 0; piece < 2; ++piece) tma_load_4d(b + piece * W::B_SLOT, &p.tmB[piece], 0, 0, 0, s * 2, &full_bar[stage]);
        }
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one_sync();
    constexpr uint32_t idesc = make_idesc_bf16(W::BN, 1, 1);
    constexpr uint32_t idesc_full = make_idesc_bf16(2 * W::BN, 1, 1);
    const uint64_t bdesc_cat = make_smem_desc(0, W::B_SLOT, W::B_SBO, W::B_SWZ);      // N = 2 BN: the second 64-wide atom is the lo slot
    const uint64_t bdesc_one = make_smem_desc(0, 16, W::B_SBO, W::B_SWZ);
    int stage = 0;
    uint32_t phase = 0;
    for (int s = s_begin; s < s_end; ++s) {
      mbar_wait(&full_bar[stage], phase);
      tc_fence_after();
      if (leader) {
        const uint32_t a_st = smem_u32(a_sm + stage * Cfg::A_STAGE);
        const uint32_t b_st = smem_u32(b_sm + stage * Cfg::B_STAGE);
        uint32_t a_rel = 0, b_rel = 0;
        if constexpr (W::KIND == 0) {
          if (s & 1) { a_rel = 14 * 32; b_rel = 14 * 2 * W::BN; }      // second half of the sample starts at position 224 = 10 * 21 + 14
        }
        const uint32_t first = (s == s_begin) ? 0u : 1u;
#pragma unroll
        for (int kt = 0; kt < W::KT; ++kt) {
          const uint32_t d = tmem_base + (uint32_t)Cfg::acc_col(kt);
          const bool cat = kt < Cfg::NCAT;
          const uint64_t bdesc0 = cat ? bdesc_cat : bdesc_one;
          const uint64_t adesc0 = make_smem_desc(0, (uint32_t)W::a_lbo(kt), W::A_SBO, W::A_SWZ);
          uint32_t a_hi, a_lo = 0;
          if constexpr (W::KIND == 0) {
            a_hi = a_st + a_rel + (uint32_t)W::a_off(kt);
          } else if constexpr (W::KIND == 1) {
            a_hi = a_st + (uint32_t)((kt & 1) * 2 * W::A_SLOT) + (uint32_t)W::a_off(kt);
            a_lo = a_hi + W::A_SLOT;
          } else {
            a_hi = a_st + (uint32_t)W::a_off(kt);
            a_lo = a_hi + W::A_SLOT;
          }
          const uint32_t b_hi = b_st + b_rel, b_lo = b_hi + W::B_SLOT;
#pragma unroll
          for (int t = 0; t < W::KSTEPS; ++t) {
            const uint32_t ao = (uint32_t)(W::pos(t) * (W::A_KSTEP / 16)), bo = (uint32_t)(W::pos(t) * (W::B_KSTEP / 16));
            if (cat) {
              umma_bf16(d, desc_with_addr(adesc0, a_hi + ao), desc_with_addr(bdesc0, b_hi + bo), idesc_full, t > 0 ? 1u : first);
            } else {
              umma_bf16(d, desc_with_addr(adesc0, a_hi + ao), desc_with_addr(bdesc0, b_hi + bo), idesc, t > 0 ? 1u : first);
              umma_bf16(d, desc_with_addr(adesc0, a_hi + ao), desc_with_addr(bdesc0, b_lo + bo), idesc, 1u);
            }
            if constexpr (W::A_PIECES == 2)
              umma_bf16(d, desc_with_addr(adesc0, a_lo + ao), desc_with_addr(bdesc0, b_hi + bo), idesc, 1u);
          }
        }
        umma_commit(&empty_bar[stage]);
      }
      __syncwarp();
      if (++stage == STAGES) { stage = 0; phase ^= 1u; }
    }
    if (leader) umma_commit(done_bar);
    __syncwarp();
  } else if (Cfg::U8_A && warp >= 6) {
    // =========================== uint8 -> bf16 converters (conv1) ===========================
    // A stage needs 13 plane rows of each of the 4 row-parity planes: 273 units (4 pixels x 4 channels) per plane.
    // 288 threads: thread c converts unit c of every plane (with 256 threads the first warp carried a second unit and was the
    // critical path of every stage), loaded one stage ahead into registers.
    if constexpr (Cfg::U8_A) {
      constexpr int UNITS = 13 * 21;
      constexpr int UPT = (UNITS + Cfg::CONV_THREADS - 1) / Cfg::CONV_THREADS;      // units per thread and plane
      const int ct = tid - 192;
      auto load_stage = [&](int s, uint4 (&b)[4][UPT]) {
        const int row0 = (s >> 1) * 21 + 10 * (s & 1);
#pragma unroll
        for (int i = 0; i < UPT; ++i) {
          const int w = ct + i * Cfg::CONV_THREADS;
          const int R = row0 + w / 21, u = w % 21;
          const int n = R / 21, q = R - n * 21;
          const bool ok = (w < UNITS) && (s < s_end) && (n < p.batch);
#pragma unroll
          for (int part = 0; part < 4; ++part) {
            b[part][i] = make_uint4(0u, 0u, 0u, 0u);
            if (ok) b[part][i] = __ldg(reinterpret_cast<const uint4*>(p.a_u8 + (((int64_t)n * 84 + 4 * q + part) * 84 + 4 * u) * 4));
          }
        }
      };
      int stage = 0;
      uint32_t phase = 0;
      auto store_stage = [&](const uint4 (&b)[4][UPT]) {
        mbar_wait(&empty_bar[stage], phase ^ 1u);
        const uint32_t base = smem_u32(a_sm + stage * Cfg::A_STAGE);
#pragma unroll
        for (int part = 0; part < 4; ++part) {
#pragma unroll
          for (int i = 0; i < UPT; ++i) {
            const int w = ct + i * Cfg::CONV_THREADS;
            if (w < UNITS) {
              const uint32_t wd[4] = {b[part][i].x, b[part][i].y, b[part][i].z, b[part][i].w};
              uint32_t o[8];
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float f0 = u8_to_f32(wd[j], 0), f1 = u8_to_f32(wd[j], 1), f2 = u8_to_f32(wd[j], 2), f3 = u8_to_f32(wd[j], 3);
                o[2 * j] = (__float_as_uint(f0) >> 16) | (__float_as_uint(f1) & 0xffff0000u);
                o[2 * j + 1] = (__float_as_uint(f2) >> 16) | (__float_as_uint(f3) & 0xffff0000u);
              }
              const uint32_t a0 = base + (uint32_t)(part * W::A_SLOT) + (uint32_t)w * 32u;
              const uint32_t sw = ((a0 >> 7) & 1u) << 4;       // SWIZZLE_32B on the absolute address
              asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a0 ^ sw), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
              asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"((a0 + 16u) ^ sw), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
              if (w > 0) {                                     // the same unit, one unit earlier in slot part + 4 (kw / 4 = 1)
                const uint32_t a1 = a0 + (uint32_t)(4 * W::A_SLOT) - 32u;
                const uint32_t sw1 = ((a1 >> 7) & 1u) << 4;
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a1 ^ sw1), "r"(o[0]), "r"(o[1]), "r"(o[2]), "r"(o[3]) : "memory");
                asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"((a1 + 16u) ^ sw1), "r"(o[4]), "r"(o[5]), "r"(o[6]), "r"(o[7]) : "memory");
              }
            }
          }
        }
        fence_proxy_async();
        mbar_arrive(&full_bar[stage]);
        if (++stage == STAGES) { stage = 0; phase ^= 1u; }
      };
      uint4 bufa[4][UPT], bufb[4][UPT];
      int s = s_begin;
      load_stage(s, bufa);
      load_stage(s + 1, bufb);
      for (; s < s_end; s += 2) {
        store_stage(bufa);
        load_stage(s + 2, bufa);
        if (s + 1 < s_end) {
          store_stage(bufb);
          load_stage(s + 3, bufb);
        }
      }
    }
  } else if (s_end > s_begin) {
    // =========================== epilogue: add this CTA's partial sums into dW ===========================
    const int ew = warp & 3;
    const int m = ew * 32 + lane;
    mbar_wait(done_bar, 0);
    tc_fence_after();
#pragma unroll 1
    for (int kt = 0; kt < W::KT; ++kt) {
      const int k = W::k_of(kt, m);
      if constexpr (W::BN == 16) {
        // 16 output channels: the accumulator is [X^T dZ_hi (16 columns) | X^T dZ_lo (16 columns)], one 32-column load
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)Cfg::acc_col(kt), v);
        tmem_ld_wait();
        if (k >= 0) {
          float4* dst = reinterpret_cast<float4*>(p.dw + (int64_t)k * W::BN);
#pragma unroll
          for (int j = 0; j < 4; ++j)
            atomicAdd(dst + j, make_float4((__uint_as_float(v[4 * j]) + __uint_as_float(v[16 + 4 * j])) * p.w_scale,
                                           (__uint_as_float(v[4 * j + 1]) + __uint_as_float(v[16 + 4 * j + 1])) * p.w_scale,
                                           (__uint_as_float(v[4 * j + 2]) + __uint_as_float(v[16 + 4 * j + 2])) * p.w_scale,
                                           (__uint_as_float(v[4 * j + 3]) + __uint_as_float(v[16 + 4 * j + 3])) * p.w_scale));
        }
        continue;
      }
#pragma unroll
      for (int c0 = 0; c0 < W::BN; c0 += 32) {
        uint32_t v[32];
        const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(Cfg::acc_col(kt) + c0);
        tmem_ld32(tcol, v);
        if (kt < Cfg::NCAT) {
          uint32_t v2[32];
          tmem_ld32(tcol + (uint32_t)W::BN, v2);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v2[j]));
        } else {
          tmem_ld_wait();
        }
        if (k >= 0) {
          // 16-byte vector reductions (RED.ADD.F32x4): a quarter of the requests the 148 CTAs send to the same dW addresses
          float4* dst = reinterpret_cast<float4*>(p.dw + (int64_t)k * W::BN + c0);
#pragma unroll
          for (int j = 0; j < 8; ++j)
            atomicAdd(dst + j, make_float4(__uint_as_float(v[4 * j]) * p.w_scale, __uint_as_float(v[4 * j + 1]) * p.w_scale,
                                           __uint_as_float(v[4 * j + 2]) * p.w_scale, __uint_as_float(v[4 * j + 3]) * p.w_scale));
        }
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

template <int L>
static int launch_wg2(const paacb_ctx* ctx, const Wg2Params& p, cudaStream_t st) {
  using Cfg = Wg2Cfg<L>;
  static DeviceOnce attr_set;   // kernel attributes are per device: one bit per device index
  if (!attr_set.done(ctx->device)) {
    if (cudaFuncSetAttribute(wgrad2_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES) != cudaSuccess) {
      cudaGetLastError();
      set_error("wgrad2<%d>: cannot set %d bytes of dynamic shared memory", L, Cfg::SMEM_BYTES);
      return PAACB_ECUDA;
    }
    // one persistent CTA per SM: ask for the largest shared-memory carve-out whatever the kernel's own request (measured
    // on conv1 forward: the same code ran 10 % slower when its request dropped from 160 KB to 86 KB)
    cudaFuncSetAttribute(wgrad2_kernel<L>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    cudaGetLastError();
    attr_set.mark(ctx->device);
  }
  // multi-GPU: the gradient tail is being all-reduced while these kernels run; one persistent CTA per SM with the maximum
  // shared-memory carve-out would leave the collective's CTAs nowhere to go until a whole kernel retires
  const int sms = ctx->num_sms - ctx->sm_reserve > 0 ? ctx->num_sms - ctx->sm_reserve : 1;
  const unsigned grid = (unsigned)(p.stages_total < sms ? p.stages_total : sms);
  PAACB_LAUNCH_BEGIN(ctx, K_WGRAD0 + Wg<L>::LAYER, st);
  launch_kernel(wgrad2_kernel<L>, grid, Cfg::THREADS, Cfg::SMEM_BYTES, st, p);
  PAACB_LAUNCH_END(ctx, K_WGRAD0 + Wg<L>::LAYER, st);
  return PAACB_OK;
}

int launch_conv_wgrad_bf16(const paacb_ctx* ctx, int l, const uint8_t* states, const void* fwd_ws, const void* bwd_ws,
                           float* grads, int64_t batch, cudaStream_t st) {
  const LayerGeom& g = ctx->layer[l];
  if (batch == 0) return PAACB_OK;
  Wg2Params p;
  memset(&p, 0, sizeof(p));
  p.batch = (int)batch;
  p.dw = grads + g.w_off;
  p.w_scale = g.in_u8 ? 0.003921568859368563f : 1.0f;
  const uint8_t* x_hi;
  const uint8_t* x_lo;
  if (l == 0) {
    x_hi = x_lo = nullptr;                       // conv1 converts the uint8 states itself
  } else {
    const Planes x = layer_planes(const_cast<void*>(fwd_ws), g.in_act_off, (int64_t)g.H * g.W * g.C, batch);
    x_hi = x.hi;
    x_lo = x.lo;
  }
  const Planes dz = layer_planes(const_cast<void*>(bwd_ws), g.out_act_off, (int64_t)g.OH * g.OW * g.N, batch);
  const int s = g.stride;
  const uint64_t unit = (uint64_t)s * g.C, wu = (uint64_t)g.W / s, hq = (uint64_t)g.H / s;
  const uint64_t bdims[4] = {(uint64_t)g.N, (uint64_t)g.OW, (uint64_t)g.OH, (uint64_t)batch};
  const uint64_t bstr[3] = {(uint64_t)g.N * 2, (uint64_t)g.OW * g.N * 2, (uint64_t)g.OH * g.OW * g.N * 2};
  int rc;
  if (l == 0) {
    if (g.C != 4 || s != 4 || g.R != 8 || (g.N != 32 && g.N != 16) || g.H != 84 || g.OH != 20) return PAACB_EUNSUPPORTED;
    const uint32_t bbox[4] = {(uint32_t)g.N, 21u, 12u, 1u};
    (void)x_lo; (void)x_hi; (void)unit; (void)wu; (void)hq;
    p.a_u8 = states;
    rc = encode_tmap_bf16(&p.tmB[0], dz.hi, 4, bdims, bstr, bbox, 2 * g.N);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[1], dz.lo, 4, bdims, bstr, bbox, 2 * g.N);
    if (rc != PAACB_OK) return rc;
    p.stages_total = (int)batch * 2;
    return g.N == 32 ? launch_wg2<0>(ctx, p, st) : launch_wg2<3>(ctx, p, st);
  }
  if (l == 1 && g.C == 16) {      // NIPS conv2
    if (s != 2 || g.R != 4 || g.N != 32 || g.H != 20 || g.OH != 9) return PAACB_EUNSUPPORTED;
    const uint64_t adims[4] = {unit, wu, (uint64_t)s, (uint64_t)batch * hq};
    const uint64_t astr[3] = {unit * 2, (uint64_t)g.W * g.C * 2, (uint64_t)s * g.W * g.C * 2};
    const uint32_t abox[4] = {32u, 10u, 1u, 12u};
    const uint32_t bbox[4] = {32u, 10u, 10u, 1u};
    rc = encode_tmap_bf16(&p.tmA[0], x_hi, 4, adims, astr, abox, 64);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmA[1], x_lo, 4, adims, astr, abox, 64);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[0], dz.hi, 4, bdims, bstr, bbox, 64);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[1], dz.lo, 4, bdims, bstr, bbox, 64);
    if (rc != PAACB_OK) return rc;
    p.stages_total = (int)batch;
    return launch_wg2<4>(ctx, p, st);
  }
  if (l == 1) {
    if (g.C != 32 || s != 2 || g.R != 4 || g.N != 64 || g.H != 20 || g.OH != 9) return PAACB_EUNSUPPORTED;
    const uint64_t adims[4] = {unit, wu, (uint64_t)s, (uint64_t)batch * hq};
    const uint64_t astr[3] = {unit * 2, (uint64_t)g.W * g.C * 2, (uint64_t)s * g.W * g.C * 2};
    const uint32_t abox[4] = {64u, 10u, 1u, 12u};
    const uint32_t bbox[4] = {64u, 10u, 10u, 1u};
    rc = encode_tmap_bf16(&p.tmA[0], x_hi, 4, adims, astr, abox, 128);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmA[1], x_lo, 4, adims, astr, abox, 128);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[0], dz.hi, 4, bdims, bstr, bbox, 128);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[1], dz.lo, 4, bdims, bstr, bbox, 128);
    if (rc != PAACB_OK) return rc;
    p.stages_total = (int)batch;
    return launch_wg2<1>(ctx, p, st);
  }
  if (l == 2) {
    if (g.C != 64 || s != 1 || g.R != 3 || g.N != 64 || g.H != 9 || g.OH != 7) return PAACB_EUNSUPPORTED;
    const uint64_t adims[3] = {64u, 9u, (uint64_t)batch * 9};
    const uint64_t astr[2] = {128u, 1152u};
    const uint32_t abox[3] = {64u, 9u, 21u};
    const uint32_t bbox[4] = {64u, 9u, 9u, 2u};
    rc = encode_tmap_bf16(&p.tmA[0], x_hi, 3, adims, astr, abox, 128);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmA[1], x_lo, 3, adims, astr, abox, 128);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[0], dz.hi, 4, bdims, bstr, bbox, 128);
    if (rc == PAACB_OK) rc = encode_tmap_bf16(&p.tmB[1], dz.lo, 4, bdims, bstr, bbox, 128);
    if (rc != PAACB_OK) return rc;
    p.stages_total = (int)((batch + 1) / 2);
    return launch_wg2<2>(ctx, p, st);
  }
  return PAACB_EUNSUPPORTED;
}

}  // namespace paacb
