// Patch-resident implicit GEMMs of the conv layers (forward and data gradient): geometry, parameters and the kernel.
// Design: tc2_conv.cu.
#pragma once
#include "tc2.cuh"

namespace paacb {

// ------------------------------------------------------------------------------------------------
// geometry of the five patch-resident GEMMs of the Nature network
// ------------------------------------------------------------------------------------------------
enum { G_FWD2 = 1, G_DG3 = 3, G_DG2 = 4,                    // Nature; conv1 forward has its own int8 kernel (tc2_conv1.cu)
       G_FWD2N = 5, G_DG2N = 6,                             // NIPS conv2 (networks.py:146): 64-byte units, SWIZZLE_64B
       G_FWD3P = 7 };                                       // conv3 forward, two whole samples per tile (below)

template <int G>
struct Geo;

// conv2 forward: [b,20,20,32] 4x4 stride 2 -> [b,9,9,64].  Unit = 2 pixels x 32 channels = 128 B; 2 row-parity planes.
template <>
struct Geo<G_FWD2> {
  static constexpr bool DGRAD = false, A_LO = true, STAGED = false, MASK_BITS = false;
  static constexpr int UB = 128, SWZ = SWZ_128B, PARTS = 2, WU = 10, HQ = 10, BOX_ROWS = 15, SLOT = 19456, NSLOTS = 5;
  static constexpr int NACC = 1, BN = 64, KS = 16, KB = 8, OH = 9, OW = 9;
  static constexpr int CH = 64, PIX = 1;
  __host__ __device__ static constexpr int aoff(int t) { return ((t / 8) * 10 + ((t / 4) % 2)) * 128 + (t % 4) * 32; }
  __host__ __device__ static constexpr int jw(int part, int t) { return ((part + 2 * (t / 8)) * 2 + ((t / 4) % 2)) * 4 + (t % 4); }
};
// conv3 forward: [b,9,9,64] 3x3 stride 1 -> [b,7,7,64].  Unit = 1 pixel x 64 channels = 128 B.  PACKED: enumerating the 9 x 9
// INPUT grid, as conv2's forward does, would make only 7 x 7 positions outputs (60 % of the MMA rows).  A row group of an MMA
// operand is 8 consecutive 128-byte units and the groups lie at a uniform stride (the descriptor's SBO, any multiple of 16
// bytes: probe A_k128_sbo1152) -- so group g = output row (sample g / 7, oh = g % 7), its 8 units = ow 0..7 (7 outputs), stride
// 9 units, over a patch copy that holds ONLY the 7 input rows kh .. kh + 6 of each sample: the TMA box {64 ch, 9, 7 rows from
// kh, 2 samples} lands exactly that, densely.  One copy per filter row kh (PARTS = 3; the 2nd and 3rd are L2 hits), tap (kh, kw)
// = copy kh at a byte offset of kw units.  A tile = two whole samples = 14 of 16 groups x 7 of 8 units: 77 % of the MMA rows,
// 0.5 instead of 0.63 tiles per sample.
template <>
struct Geo<G_FWD3P> {
  static constexpr bool DGRAD = false, A_LO = true, STAGED = false, MASK_BITS = false;
  static constexpr int UB = 128, SWZ = SWZ_128B, PARTS = 3, WU = 9, HQ = 9, BOX_ROWS = 14, SLOT = 16384, NSLOTS = 5;
  static constexpr int NACC = 1, BN = 64, KS = 12, KB = 9, OH = 7, OW = 7;
  static constexpr int CH = 64, PIX = 1;
  __host__ __device__ static constexpr int aoff(int t) { return (t / 4) * 128 + (t % 4) * 32; }
  __host__ __device__ static constexpr int jw(int part, int t) { return part * 12 + t; }
};
// PACKED geometries: samples per tile; row-group stride of the A descriptor in units
template <int G> struct GeoPack { static constexpr int SAMPLES = 0; };
template <> struct GeoPack<G_FWD3P> { static constexpr int SAMPLES = 2; };

// conv3 data-gradient: dZ3 [b,7,7,64] -> dX [b,9,9,64]; one sample per tile, positions enumerated 11 wide over the
// zero-padded dZ (TMA out-of-bounds fill), tap (kh, kw) reads position q + (2-kh)*11 + (2-kw).
template <>
struct Geo<G_DG3> {
  static constexpr bool DGRAD = true, A_LO = true, STAGED = false, MASK_BITS = false;
  static constexpr int UB = 128, SWZ = SWZ_128B, PARTS = 1, WU = 11, HQ = 9, BOX_ROWS = 11, SLOT = 16384, NSLOTS = 4;
  static constexpr int NACC = 1, BN = 64, KS = 36, KB = 9, OH = 9, OW = 9;       // OH/OW: valid rows/cols of the enumeration
  static constexpr int PAD = 2, S = 1, XH = 9, XW = 9;
  static constexpr int CH = 64, PIX = 1;      // output channels per pixel, pixels per accumulator row
  __host__ __device__ static constexpr int aoff(int t) { return ((2 - (t / 4) / 3) * 11 + (2 - (t / 4) % 3)) * 128 + (t % 4) * 32; }
  __host__ __device__ static constexpr int jw(int, int t) { return t; }
};
// conv2 data-gradient: dZ2 [b,9,9,64] -> dX [b,20,20,32]; the four stride-parity classes are four accumulators over
// the same resident dZ patch (class (ph, pw), tap (tj, ti) reads position q + (1-tj)*11 + (1-ti)).
// STAGED epilogue: a thread's outputs of the two classes (ph, 0), (ph, 1) are one 128-byte row (2 pixels x 32 channels)
// of a [10 x 10 rows] x 128 B tile per output-row parity ph; written straight to HBM every warp store touched 32
// different cache lines (the first version was bound by LSU wavefronts: 34 % tensor-pipe activity).  The rows go to a
// swizzled shared-memory tile instead and the TMA engine stores the tile.
template <>
struct Geo<G_DG2> {
  static constexpr bool DGRAD = true, A_LO = true, STAGED = true, MASK_BITS = true;      // mask = conv1's ReLU bit words
  static constexpr int UB = 128, SWZ = SWZ_128B, PARTS = 1, WU = 11, HQ = 10, BOX_ROWS = 11, SLOT = 16384, NSLOTS = 4;
  static constexpr int NACC = 4, BN = 32, KS = 16, KB = 4, OH = 10, OW = 10;
  static constexpr int PAD = 1, S = 2, XH = 20, XW = 20;
  static constexpr int CH = 32, PIX = 1;
  __host__ __device__ static constexpr int aoff(int t) { return ((1 - (t / 4) / 2) * 11 + (1 - (t / 4) % 2)) * 128 + (t % 4) * 32; }
  __host__ __device__ static constexpr int jw(int, int t) { return t; }
};

// NIPS conv2 forward: [b,20,20,16] 4x4 stride 2 -> [b,9,9,32].  Unit = 2 pixels x 16 channels = 64 B (SWIZZLE_64B rows); one
// K = 16 MMA is exactly one pixel's 16 channels, so filter tap (kh, kw) = plane kh & 1, row offset kh >> 1, unit offset
// kw >> 1, 32-byte half kw & 1.
template <>
struct Geo<G_FWD2N> {
  static constexpr bool DGRAD = false, A_LO = true, STAGED = false, MASK_BITS = false;
  static constexpr int UB = 64, SWZ = SWZ_64B, PARTS = 2, WU = 10, HQ = 10, BOX_ROWS = 15, SLOT = 10240, NSLOTS = 6;
  static constexpr int NACC = 1, BN = 32, KS = 8, KB = 4, OH = 9, OW = 9;
  static constexpr int CH = 32, PIX = 1;
  __host__ __device__ static constexpr int aoff(int t) { return ((t / 4) * 10 + ((t / 2) % 2)) * 64 + (t % 2) * 32; }
  __host__ __device__ static constexpr int jw(int part, int t) { return (part + 2 * (t / 4)) * 4 + 2 * ((t / 2) % 2) + (t % 2); }
};
// NIPS conv2 data-gradient: dZ2 [b,9,9,32] -> dX [b,20,20,16].  The four stride-parity classes (ph, pw) x 16 input channels are
// TWO accumulators of 32 columns: accumulator ph holds (pw, ci) = the two horizontally adjacent output pixels 2 qw, 2 qw + 1,
// which are 32 contiguous elements of the NHWC output -- the packed data-gradient image is row-ordered (ph, pw, ci) already,
// and a thread's 32 columns are one 64-byte run of each output plane (direct 256-bit stores, no staging tile).
template <>
struct Geo<G_DG2N> {
  static constexpr bool DGRAD = true, A_LO = true, STAGED = false, MASK_BITS = true;     // mask = conv1's ReLU bit words
  static constexpr int UB = 64, SWZ = SWZ_64B, PARTS = 1, WU = 11, HQ = 10, BOX_ROWS = 11, SLOT = 8192, NSLOTS = 6;
  static constexpr int NACC = 2, BN = 32, KS = 8, KB = 2, OH = 10, OW = 10;
  static constexpr int PAD = 1, S = 2, XH = 20, XW = 20;
  static constexpr int CH = 16, PIX = 2;      // output channels per pixel, pixels per accumulator row
  __host__ __device__ static constexpr int aoff(int t) { return ((1 - (t / 2) / 2) * 11 + (1 - (t / 2) % 2)) * 64 + (t % 2) * 32; }
  __host__ __device__ static constexpr int jw(int, int t) { return t; }
};

struct ConvKParams {
  CUtensorMap tmA[2];      // source planes (hi, lo); forward: dims (unit, units/row, row parity, plane rows); dgrad: (C, OW, OH, b)
  CUtensorMap tmW[2];      // packed weights (hi, lo): dims (K, rows)
  CUtensorMap tmOut;       // staged epilogue: output hi plane as (2 px x C, W/2, row parity, b * H/2)
  int num_tiles;
  int batch;
  const float* bias;       // forward
  float in_scale;          // forward: applied to the accumulator (1/255 for the uint8 layer, networks.py:115)
  uint8_t* out_hi;         // output planes (bf16)
  uint8_t* out_lo;
  const uint8_t* mask_hi;  // dgrad: hi plane of the activation whose ReLU is differentiated (same shape as the output)
  const uint32_t* mask_bits;   // conv2's data gradient: the same mask as bit planes, uint16 [b][2][XH * XW] (tc2.cuh: relu1_bits)
  float* dbias;            // dgrad: += column sums of the output (the bias gradient of the layer that produced that activation)
};

template <int G>
struct ConvKCfg {
  using Ge = Geo<G>;
  static constexpr int RING_BYTES = Ge::NSLOTS * Ge::SLOT;
  // resident weights: per 64-wide K-block one K-major tile of 2 * NT rows: the hi pieces of all accumulators, then the
  // lo pieces.  One MMA of N = 2 * NT evaluates A_hi * [W_hi | W_lo] (the operand A is read from shared memory once:
  // with N <= 64 an SS-mode MMA is bound by its 4 KB A read, not by the tensor pipe), a second of N = NT adds A_lo * W_hi.
  static constexpr int NT = Ge::NACC * Ge::BN;
  static constexpr int KB_BYTES = 2 * NT * 128;
  static constexpr int W_BYTES = Ge::KB * KB_BYTES;
  static constexpr int BOX_BYTES = Ge::UB * Ge::WU * Ge::BOX_ROWS;
  static constexpr int STG_TILE = 13 * 1024;                                // 100 rows x 128 B, 1024-byte aligned
  static constexpr int STG_BYTES = Ge::STAGED ? 2 * STG_TILE : 0;            // one tile of the hi plane per output-row parity
  static constexpr int NBARS = 2 * Ge::NSLOTS + 1 + 4 + 1;
  static constexpr int SMEM_BYTES = RING_BYTES + W_BYTES + STG_BYTES + 1024 /* alignment slack */ + NBARS * 8 + 16 + 256 /* forward: bias row */;
  static constexpr int TMEM_COLS = 4 * NT;                                  // two accumulator buffers of 2 * NT columns
  static_assert(BOX_BYTES <= Ge::SLOT && Ge::SLOT % 1024 == 0, "slot too small");
  // TMA warp, MMA warp, two epilogue groups of four warps (one per accumulator buffer; the staged epilogue splits every
  // tile between the groups: output-row parity 0 / 1)
  static constexpr int THREADS = 64 + 256;
  static_assert(SMEM_BYTES <= 227 * 1024, "shared memory budget");
  static_assert(TMEM_COLS == 128 || TMEM_COLS == 256 || TMEM_COLS == 512, "TMEM columns");
  static_assert(2 * NT <= 256, "MMA N");
};


// lane j of the warp ends up with the sum over the warp's 32 lanes of v[j] (31 shuffles)
__device__ __forceinline__ float warp_transpose_sum(float (&v)[32], int lane) {
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

template <int G>
__global__ void __launch_bounds__(ConvKCfg<G>::THREADS, 1) convk_kernel(const __grid_constant__ ConvKParams p) {
  const int cta = (int)blockIdx.x, ncta = (int)gridDim.x;   // persistent CTAs: this one's index, their count
  using Ge = Geo<G>;
  using Cfg = ConvKCfg<G>;
  constexpr int NSLOTS = Ge::NSLOTS, BN = Ge::BN, NACC = Ge::NACC;
  constexpr int PACK = GeoPack<G>::SAMPLES;       // > 0: whole samples per tile, one patch copy per filter row
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* ring = smem;
  uint8_t* wsm = smem + Cfg::RING_BYTES;
  uint8_t* stg = wsm + Cfg::W_BYTES;              // staged epilogue tiles
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg + Cfg::STG_BYTES);
  uint64_t* full_bar = bars;                      // [NSLOTS] TMA -> MMA
  uint64_t* empty_bar = bars + NSLOTS;            // [NSLOTS] MMA commit -> TMA
  uint64_t* w_bar = bars + 2 * NSLOTS;            // weights resident
  uint64_t* tfull_bar = w_bar + 1;                // [2] MMA commit -> epilogue
  uint64_t* tempty_bar = tfull_bar + 2;           // [2] epilogue -> MMA
  uint64_t* mask_bar = tempty_bar + 2;            // staged epilogue: the staging tiles have been read out by the TMA stores
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mask_bar + 1);
  float* s_bias = reinterpret_cast<float*>(bars + Cfg::NBARS + 2);      // forward: the layer's bias row (16-byte aligned)

  const int tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;

  pdl_launch_dependents();                        // the next kernel's prologue may run under this kernel's tail (tc_ptx.cuh)
  if (tid == 0) {
    for (int s = 0; s < NSLOTS; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(w_bar, 1);
    mbar_init(mask_bar, 1);
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], Ge::STAGED ? 256 : 128);     // the epilogue warps that drain buffer s
    }
    fence_barrier_init();
    tma_prefetch_desc(&p.tmA[0]);
    tma_prefetch_desc(&p.tmW[0]);
    // the layer's weights depend on no kernel of this forward / backward: their loads start before the wait below
    mbar_arrive_expect_tx(w_bar, Cfg::W_BYTES);
    for (int piece = 0; piece < 2; ++piece)
      for (int acc = 0; acc < NACC; ++acc)
        for (int kb = 0; kb < Ge::KB; ++kb)
          tma_load_2d(wsm + kb * Cfg::KB_BYTES + (piece * NACC + acc) * (BN * 128), &p.tmW[piece], kb * 64, acc * BN, w_bar);
  }
  if (warp == 1) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  if constexpr (!Ge::DGRAD) {
    if (tid >= 64 && tid < 64 + BN) s_bias[tid - 64] = __ldg(p.bias + tid - 64);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  pdl_wait();                                     // everything below reads or writes what other kernels produce / consume
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // =========================== TMA producer ===========================
    if (elect_one_sync()) {
      int slot = 0;
      uint32_t phase = 0;
      for (int tile = cta; tile < p.num_tiles; tile += ncta) {
        // (requesting the boxes of the tile after next into L2 with cp.async.bulk.prefetch.tensor was measured: 3 % slower; the
        // packed conv3 geometry with the NEXT tile's two samples prefetched: 0.603 -> 0.617 ms per step;
        // prefetch.global.L2 of the tile after next by the idle epilogue threads, one per 128-byte line: conv2 0.76-0.79 -> 0.79-0.83,
        // conv3 unchanged -- these kernels do not wait for first-touch DRAM latency)
        // slot order: (part, piece) with the piece fastest; PACKED: piece slowest (all taps of A_hi, then all taps of A_lo: the
        // MMA order of the input-grid conv3 forward it replaced, so that the accumulators hold the same bits)
        constexpr int NPIECE = Ge::A_LO ? 2 : 1;
#pragma unroll 1
        for (int it = 0; it < Ge::PARTS * NPIECE; ++it) {
          const int part = PACK > 0 ? it % Ge::PARTS : it / NPIECE;
          const int piece = PACK > 0 ? it / Ge::PARTS : it % NPIECE;
          {
            mbar_wait(&empty_bar[slot], phase ^ 1u);
            mbar_arrive_expect_tx(&full_bar[slot], Cfg::BOX_BYTES);
            uint8_t* dst = ring + slot * Ge::SLOT;
            if constexpr (Ge::DGRAD) {
              tma_load_4d(dst, &p.tmA[piece], 0, -Ge::PAD, -Ge::PAD, tile, &full_bar[slot]);
            } else if constexpr (PACK > 0) {
              tma_load_4d(dst, &p.tmA[piece], 0, 0, part, PACK * tile, &full_bar[slot]);     // input rows part .. part + OH - 1
            } else {
              const int row0 = (int)(((int64_t)tile * 128) / Ge::WU);
              tma_load_4d(dst, &p.tmA[piece], 0, 0, part, row0, &full_bar[slot]);
            }
            if (++slot == NSLOTS) { slot = 0; phase ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =========================== MMA issuer ===========================
    const bool leader = elect_one_sync();
    constexpr uint32_t idesc_full = make_idesc_bf16(2 * Cfg::NT, 0, 0);
    constexpr uint32_t idesc_half = make_idesc_bf16(Cfg::NT, 0, 0);
    const uint64_t adesc0 = make_smem_desc(0, 16, (PACK > 0 ? Ge::WU : 8) * Ge::UB, Ge::SWZ);
    const uint64_t bdesc0 = make_smem_desc(0, 16, 1024, SWZ_128B);
    const uint32_t ring_a = smem_u32(ring);
    const uint32_t w_a = smem_u32(wsm);
    mbar_wait(w_bar, 0);
    int slot = 0;
    uint32_t phase = 0;
    int tl = 0;
    for (int tile = cta; tile < p.num_tiles; tile += ncta, ++tl) {
      const int ab = tl & 1;
      const uint32_t aph = (uint32_t)((tl >> 1) & 1);
      mbar_wait(&tempty_bar[ab], aph ^ 1u);
      tc_fence_after();
      uint32_t rel = 0;
      if constexpr (!Ge::DGRAD && PACK == 0) rel = (uint32_t)(((int64_t)tile * 128) % Ge::WU) * Ge::UB;
      const uint32_t d0 = tmem_base + (uint32_t)(ab * 2 * Cfg::NT);
      constexpr int NPIECE = Ge::A_LO ? 2 : 1;
#pragma unroll
      for (int it = 0; it < Ge::PARTS * NPIECE; ++it) {
        const int part = PACK > 0 ? it % Ge::PARTS : it / NPIECE;       // same slot order as the producer
        const int piece = PACK > 0 ? it / Ge::PARTS : it % NPIECE;
        {
          mbar_wait(&full_bar[slot], phase);
          tc_fence_after();
          if (leader) {
            const uint32_t a_base = ring_a + (uint32_t)(slot * Ge::SLOT) + rel;
#pragma unroll
            for (int t = 0; t < Ge::KS; ++t) {
              const uint64_t ad = desc_with_addr(adesc0, a_base + (uint32_t)Ge::aoff(t));
              const int jw = Ge::jw(part, t);
              const uint64_t bd = desc_with_addr(bdesc0, w_a + (uint32_t)((jw / 4) * Cfg::KB_BYTES + (jw % 4) * 32));
              if (piece == 0) umma_bf16(d0, ad, bd, idesc_full, (part | t) ? 1u : 0u);    // A_hi * [W_hi | W_lo]
              else umma_bf16(d0, ad, bd, idesc_half, 1u);                                             // A_lo * W_hi
            }
            umma_commit(&empty_bar[slot]);
          }
          __syncwarp();
          if (++slot == NSLOTS) { slot = 0; phase ^= 1u; }
        }
      }
      if (leader) umma_commit(&tfull_bar[ab]);
      __syncwarp();
    }
  } else if (Ge::STAGED) {
    // =========================== staged epilogue (conv2 data-gradient) ===========================
    if constexpr (Ge::STAGED) {
      const int ew = warp & 3;
      const int r = ew * 32 + lane;
      const int qh = r / Ge::WU, qw = r - qh * Ge::WU;
      const bool ok = (qh < Ge::OH) && (qw < Ge::OW);
      const uint32_t srow = (uint32_t)(qh * Ge::OW + qw);                  // row of the 100 x 128 B staging tile
      const uint32_t stg_a = smem_u32(stg);
      const int ph = (warp - 2) >> 2;                                       // this warp's output-row parity: classes (ph, 0), (ph, 1)
      const bool io = (tid == 64 + 128 * ph);                               // issues the TMA stores of this group's tile
      float bsum = 0.f;
      // The ReLU mask of this thread's two output pixels is TWO 32-bit words (bit c = channel c > 0, written by conv1's
      // forward epilogue), carried one tile ahead in two registers.  History: (1) the 64-byte hi-plane rows of both pixels
      // loaded cold at the top of the tile: a DRAM round trip per tile; (2) the rows carried one tile ahead in registers: 32
      // registers this kernel does not have -- the spill put a local-memory load on the critical path right after the MMA
      // barrier, 18 % of all stall samples; (3) rows loaded at the top of the tile behind an L2 prefetch issued a tile earlier:
      // still 11 % of the samples on the first use of the mask (the kernel is epilogue-bound, so nothing hides an L2 hit),
      // -17 % with the loads switched off (profiles/r02_ablations_dgrad.json); (4) bits.
      // (plane h of sample `tile`: uint16 [XH * XW]; this thread's two pixels are adjacent: one 32-bit load per plane)
      const uint16_t* bits16 = reinterpret_cast<const uint16_t*>(p.mask_bits);
      const int pxo = (Ge::S * qh + ph) * Ge::XW + Ge::S * qw;
      auto load_bits = [&](int tile) {
        const uint16_t* b = bits16 + (int64_t)tile * (2 * Ge::XH * Ge::XW) + pxo;
        return make_uint2(__ldg(reinterpret_cast<const uint32_t*>(b)), __ldg(reinterpret_cast<const uint32_t*>(b + Ge::XH * Ge::XW)));
      };
      uint2 mb_next = make_uint2(0u, 0u);
      if (ok && cta < p.num_tiles) mb_next = load_bits(cta);
      int tl = 0;
      for (int tile = cta; tile < p.num_tiles; tile += ncta, ++tl) {
        const int ab = tl & 1;
        const uint32_t aph = (uint32_t)((tl >> 1) & 1);
        const uint2 mb = mb_next;
        if (ok && tile + ncta < p.num_tiles) mb_next = load_bits(tile + ncta);
        mbar_wait(&tfull_bar[ab], aph);
        tc_fence_after();
        float o[2][32];
#pragma unroll
        for (int pw = 0; pw < 2; ++pw) {
          uint32_t v[32], v2[32];
          const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(ab * 2 * Cfg::NT + (ph * 2 + pw) * BN);
          tmem_ld32(tcol, v);
          tmem_ld32(tcol + (uint32_t)Cfg::NT, v2);
          tmem_ld_wait();
          // pixel pw: channels 0-15 in half pw of mb.x, channels 16-31 in half pw of mb.y (0 for rows that are no output pixels)
          const uint32_t word = ((pw ? mb.x >> 16 : mb.x) & 0xffffu) | (pw ? mb.y & 0xffff0000u : mb.y << 16);
#pragma unroll
          for (int e = 0; e < 32; ++e)
            o[pw][e] = ((word >> (16 * (e / 16) + relu1_bit_pos(e % 16))) & 1u) ? __uint_as_float(v[e]) + __uint_as_float(v2[e]) : 0.f;
        }
        tc_fence_before();
        mbar_arrive(&tempty_bar[ab]);                                       // accumulator drained: the MMAs of tile tl + 2 may start
        // This group's 100 x 128 B staging tile carries the hi plane only (the rest of shared memory is needed for a
        // 4-deep patch ring: with 2 slots the kernel was bound by the TMA round trip).  io = the group's first thread.
        uint8_t* tile_p = stg + ph * Cfg::STG_TILE;
        const uint32_t t_row = stg_a + (uint32_t)(ph * Cfg::STG_TILE) + srow * 128u;
        uint32_t lw[2][16];
        if (io) tma_store_wait_read();                                      // previous tile's hi plane has been read out
        named_bar_sync(1 + ph, 128);
#pragma unroll
        for (int pw = 0; pw < 2; ++pw) {
          uint32_t hw[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) split_bf16x2(o[pw][2 * j], o[pw][2 * j + 1], hw[j], lw[pw][j]);
          if (ok) {
#pragma unroll
            for (int c = 0; c < 4; ++c)                                     // 16-byte chunk pw * 4 + c of the row, swizzled
              sts128(t_row + ((((uint32_t)(pw * 4 + c)) ^ (srow & 7u)) << 4), make_uint4(hw[4 * c], hw[4 * c + 1], hw[4 * c + 2], hw[4 * c + 3]));
          }
        }
        fence_proxy_async();                                                // staging writes -> visible to the TMA engine
        named_bar_sync(1 + ph, 128);
        if (io) {
          tma_store_4d(&p.tmOut, tile_p, 0, 0, ph, tile * Ge::OH);
          tma_store_commit();
        }
        // bias gradient: channel = lane for both classes: add the classes first, ONE transposed warp reduction per tile
        // (this kernel has no registers left for per-thread column sums; the shuffles overlap the TMA engine reading the tile)
#pragma unroll
        for (int j = 0; j < 32; ++j) o[0][j] += o[1][j];
        bsum += warp_transpose_sum(o[0], lane);
        if (ok) {
          // lo plane: this thread's two pixels are one 128-byte row of the plane -- four 256-bit stores straight from
          // registers while the TMA engine drains the hi tile (there is no shared memory for a second staging tile; sending
          // the lo plane through the same tile after the hi plane costs two more barriers and a second wait per tile)
          uint8_t* dl = p.out_lo + ((((int64_t)tile * Ge::XH + Ge::S * qh + ph) * Ge::XW + Ge::S * qw) * BN) * 2;
#pragma unroll
          for (int pw = 0; pw < 2; ++pw)
#pragma unroll
            for (int c = 0; c < 2; ++c) stg256(dl + pw * 64 + c * 32, &lw[pw][8 * c]);
        }
      }
      if (io) tma_store_wait_all();
      if (p.dbias != nullptr) atomicAdd(p.dbias + lane, bsum);
    }
  } else {
    // =========================== epilogue ===========================
    const int ew = warp & 3;                     // TMEM lane quarter this warp may access
    const int r = ew * 32 + lane;                // tile row of this thread
    const int grp = (warp - 2) >> 2;             // epilogue group = accumulator buffer it drains (tiles tl with tl & 1 == grp)
    // (per-thread column sums reduced once at the end -- what tc2_stream.cu's dgrad does -- cost this kernel 42 registers
    // it does not have: conv3's data gradient got 7 % slower with them)
    float bsum[NACC == 1 ? BN / 32 : 1];
#pragma unroll
    for (int i = 0; i < (NACC == 1 ? BN / 32 : 1); ++i) bsum[i] = 0.f;
    for (int tl = grp, tile = cta + grp * ncta; tile < p.num_tiles; tile += 2 * ncta, tl += 2) {
      const int ab = grp;
      const uint32_t aph = (uint32_t)((tl >> 1) & 1);
      // row -> output pixel
      bool ok;
      int64_t pix = 0;          // forward: output pixel index; dgrad: (sample, qh, qw) resolved per class below
      int qh = 0, qw = 0;
      if constexpr (Ge::DGRAD) {
        qh = r / Ge::WU;
        qw = r - qh * Ge::WU;
        ok = (qh < Ge::OH) && (qw < Ge::OW);
      } else if constexpr (PACK > 0) {
        const int g = r >> 3, ju = r & 7;                             // row group = (sample, output row), unit = output column
        const int n = PACK * tile + g / Ge::OH;
        const int oh = g % Ge::OH;
        ok = (g < PACK * Ge::OH) && (ju < Ge::OW) && (n < p.batch);
        pix = ((int64_t)n * Ge::OH + oh) * Ge::OW + ju;
      } else {
        const uint32_t q = (uint32_t)tile * 128u + (uint32_t)r;      // < 2^31 (checked by the launcher)
        const uint32_t prow = q / (uint32_t)Ge::WU;
        const int ju = (int)(q - prow * (uint32_t)Ge::WU);
        const uint32_t n = prow / (uint32_t)Ge::HQ;
        const int oh = (int)(prow - n * (uint32_t)Ge::HQ);
        ok = (ju < Ge::OW) && (oh < Ge::OH) && ((int)n < p.batch);
        pix = ((int64_t)n * Ge::OH + oh) * Ge::OW + ju;
      }
      // dgrad: the ReLU-mask words of the whole tile row do not depend on the accumulator: fetch them before waiting
      // for the MMAs so that their DRAM latency overlaps the mainloop (they were the top stall of the first version)
      uint4 mk[(Ge::DGRAD && !Ge::MASK_BITS) ? NACC : 1][(Ge::DGRAD && !Ge::MASK_BITS) ? BN / 32 : 1][4];
      uint32_t mbits[Ge::MASK_BITS ? NACC : 1];   // MASK_BITS (PIX == 2, CH = 16): the 16 flags of the two pixels of an accumulator row
      if constexpr (Ge::DGRAD && Ge::MASK_BITS) {
        static_assert(!Ge::MASK_BITS || Ge::STAGED || (Ge::PIX == 2 && Ge::CH == 16 && BN == 32), "bit masks: two pixels of 16 channels per row");
#pragma unroll
        for (int acc = 0; acc < NACC; ++acc) {
          const int ih = Ge::S * qh + acc, iw = Ge::S * qw;
          mbits[acc] = 0u;
          if (ok)      // plane 0 of sample `tile`: pixels iw, iw + 1 are one aligned 32-bit word
            mbits[acc] = __ldg(reinterpret_cast<const uint32_t*>(reinterpret_cast<const uint16_t*>(p.mask_bits) +
                                                                 (int64_t)tile * (2 * Ge::XH * Ge::XW) + ih * Ge::XW + iw));
        }
      } else if constexpr (Ge::DGRAD) {
#pragma unroll
        for (int acc = 0; acc < NACC; ++acc) {
          // accumulator -> output pixel: PIX == 1: class (acc / 2, acc % 2) of a stride-2 layer; PIX == 2: row parity acc, the
          // 32 columns are the pixels 2 qw, 2 qw + 1 (CH channels each)
          const int ih = Ge::S * qh + (NACC > 1 ? (Ge::PIX == 2 ? acc : acc / 2) : 0);
          const int iw = Ge::S * qw + ((NACC > 1 && Ge::PIX == 1) ? acc % 2 : 0);
          const int64_t ob = (((int64_t)tile * Ge::XH + ih) * Ge::XW + iw) * Ge::CH;
#pragma unroll
          for (int c = 0; c < BN / 32; ++c) {
#pragma unroll
            for (int j = 0; j < 4; ++j) mk[acc][c][j] = make_uint4(0u, 0u, 0u, 0u);
            if (ok) {
              ldg256(p.mask_hi + (ob + c * 32) * 2, mk[acc][c][0], mk[acc][c][1]);
              ldg256(p.mask_hi + (ob + c * 32) * 2 + 32, mk[acc][c][2], mk[acc][c][3]);
            }
          }
        }
      }
      mbar_wait(&tfull_bar[ab], aph);
      tc_fence_after();
      if constexpr (!Ge::DGRAD) {
        // forward: the whole accumulator row goes to registers first and the buffer is handed back to the MMA warp BEFORE
        // the arithmetic and the stores (the data-gradient variants have no registers for that: they release it at the end)
        uint32_t av[BN / 32][32];
#pragma unroll
        for (int c = 0; c < BN / 32; ++c) {
          uint32_t v2[32];
          const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(ab * 2 * Cfg::NT + c * 32);
          tmem_ld32(tcol, av[c]);                               // A_hi * W_hi + A_lo * W_hi
          tmem_ld32(tcol + (uint32_t)Cfg::NT, v2);              // A_hi * W_lo
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) av[c][j] = __float_as_uint(__uint_as_float(av[c][j]) + __uint_as_float(v2[j]));
        }
        tc_fence_before();
        mbar_arrive(&tempty_bar[ab]);
        const float4* b4 = reinterpret_cast<const float4*>(s_bias);
        uint32_t hw[BN / 32][16], lw[BN / 32][16];
#pragma unroll
        for (int c = 0; c < BN / 32; ++c) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 bb = b4[c * 8 + j];                    // broadcast 16-byte shared-memory load: 4 channels
            const float o0 = fmaxf(fmaf(__uint_as_float(av[c][4 * j]), p.in_scale, bb.x), 0.f);
            const float o1 = fmaxf(fmaf(__uint_as_float(av[c][4 * j + 1]), p.in_scale, bb.y), 0.f);
            const float o2 = fmaxf(fmaf(__uint_as_float(av[c][4 * j + 2]), p.in_scale, bb.z), 0.f);
            const float o3 = fmaxf(fmaf(__uint_as_float(av[c][4 * j + 3]), p.in_scale, bb.w), 0.f);
            split_bf16x2(o0, o1, hw[c][2 * j], lw[c][2 * j]);
            split_bf16x2(o2, o3, hw[c][2 * j + 1], lw[c][2 * j + 1]);
          }
        }
        if (ok) {
#pragma unroll
          for (int c = 0; c < BN / 32; ++c) {
            uint8_t* dh = p.out_hi + (pix * BN + c * 32) * 2;
            uint8_t* dl = p.out_lo + (pix * BN + c * 32) * 2;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              stg256(dh + 32 * j, hw[c] + 8 * j);
              stg256(dl + 32 * j, lw[c] + 8 * j);
            }
          }
        }
        continue;
      }
#pragma unroll
      for (int acc = 0; acc < NACC; ++acc) {
        int64_t obase;          // element index of this row's first output channel
        if constexpr (Ge::DGRAD) {
          const int ih = Ge::S * qh + (NACC > 1 ? (Ge::PIX == 2 ? acc : acc / 2) : 0);
          const int iw = Ge::S * qw + ((NACC > 1 && Ge::PIX == 1) ? acc % 2 : 0);
          obase = (((int64_t)tile * Ge::XH + ih) * Ge::XW + iw) * Ge::CH;
        } else {
          obase = pix * BN;
        }
#pragma unroll
        for (int c0 = 0; c0 < BN; c0 += 32) {
          uint32_t v[32], v2[32];
          const uint32_t tcol = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(ab * 2 * Cfg::NT + acc * BN + c0);
          tmem_ld32(tcol, v);                                   // A_hi * W_hi + A_lo * W_hi
          tmem_ld32(tcol + (uint32_t)Cfg::NT, v2);              // A_hi * W_lo
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(v2[j]));
          float o[32];
          if constexpr (Ge::DGRAD && Ge::MASK_BITS) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {      // column j = pixel j / CH, channel j % CH; rows that are no output pixels carry 0 bits
              o[j] = ((mbits[acc] >> (16 * (j / Ge::CH) + relu1_bit_pos(j % Ge::CH))) & 1u) ? __uint_as_float(v[j]) : 0.f;
            }
          } else if constexpr (Ge::DGRAD) {
            uint32_t mw[16];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const uint4 m = mk[acc][c0 / 32][j];
              mw[4 * j] = m.x; mw[4 * j + 1] = m.y; mw[4 * j + 2] = m.z; mw[4 * j + 3] = m.w;
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              // bf16 > 0  <=>  sign clear and magnitude non-zero
              const uint32_t a0 = mw[j] & 0xffffu, a1 = mw[j] >> 16;
              o[2 * j] = (ok && a0 != 0u && a0 < 0x8000u) ? __uint_as_float(v[2 * j]) : 0.f;
              o[2 * j + 1] = (ok && a1 != 0u && a1 < 0x8000u) ? __uint_as_float(v[2 * j + 1]) : 0.f;
            }
          }
          if (ok) {
            uint32_t hw[16], lw[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) split_bf16x2(o[2 * j], o[2 * j + 1], hw[j], lw[j]);
            uint8_t* dh = p.out_hi + (obase + c0) * 2;
            uint8_t* dl = p.out_lo + (obase + c0) * 2;
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              stg256(dh + 32 * j, hw + 8 * j);
              stg256(dl + 32 * j, lw + 8 * j);
            }
          }
          if constexpr (Ge::DGRAD) {
            const float s = warp_transpose_sum(o, lane);      // column c0 + lane over this warp's 32 rows
            bsum[NACC == 1 ? c0 / 32 : 0] += s;
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[ab]);
    }
    if constexpr (Ge::DGRAD) {
      if (p.dbias != nullptr) {
        // column -> channel: PIX == 2 packs two pixels of CH channels into one accumulator row
#pragma unroll
        for (int i = 0; i < (NACC == 1 ? BN / 32 : 1); ++i) atomicAdd(p.dbias + (i * 32 + lane) % Ge::CH, bsum[i]);
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
