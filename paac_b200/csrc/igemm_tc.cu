// tcgen05 (5th-generation tensor core) implicit GEMMs for the conv / fc layers, sm_100a: forward and data-gradient.
//
//   forward : Y[m, n]  = act( in_scale * sum_k im2col(X)[m, k] W[k, n] + bias[n] )     networks.py:12-21, 49-60, 115
//   dgrad   : dX[p, c] = ( sum_{tap, co} dZ[p - tap, co] W[tap, c, co] ) * [X[p, c] > 0]  (TF autodiff: Conv2DBackpropInput,
//             MatMul grad, ReluGrad; one GEMM per stride-parity class so no zero taps are multiplied)
//
// One persistent CTA per SM, warp-specialised (13 warps):
//   warps 0-7   A producers: two groups of 128 threads alternate K-blocks.  Thread r of a group owns tile row r.  It
//               gathers the 32 consecutive k of its row (128 contiguous bytes of NHWC fp32, or 32 bytes of the uint8
//               state) with cp.async into a thread-private, bank-swizzled staging slot in shared memory, DEPTH
//               K-blocks ahead (no registers held, no scoreboard wait at the loop back-edge -- the first version kept
//               the prefetch in registers and ptxas serialised it); when a K-block has landed the thread reads its row
//               back, converts to tf32 (round-to-nearest on the integer pipe; in TF32X3 mode also the residual
//               lo = rna(a - hi)) and writes the row straight into TENSOR MEMORY with tcgen05.st (lane = row,
//               32 columns = the 32 k).  The MMA reads A from TMEM: the operand never occupies a shared-memory
//               operand tile and costs the MMA no shared-memory bandwidth.  im2col is never materialised.
//   warp  8     lane 0 issues tcgen05.mma.cta_group::1.kind::tf32 (M = 128, N = BN, K = 8) into a TMEM accumulator;
//               tcgen05.commit releases the stage / publishes the accumulator.
//   warps 9-12  epilogue: tcgen05.ld the accumulator rows (32 lanes per warp), then scale + bias + ReLU (forward) or
//               ReLU-mask + scatter to the input pixel (dgrad), 16-byte stores.
// B (weights) is prepacked once per call into the exact swizzled shared-memory image of every (class, n-tile, k-block),
// so a single cp.async.bulk (TMA engine) per stage lands it, completing on the stage's mbarrier.  Accumulators are
// double-buffered in TMEM so the epilogue of tile i overlaps the mainloop of tile i+1.
//
// TF32X3: A = Ahi + Alo, B = Bhi + Blo, D += Alo*Bhi + Ahi*Blo + Ahi*Bhi (fp32 accumulate in TMEM): the dropped
// Alo*Blo term is ~2^-22 relative, which is what meets the 1e-4 parity bar that plain TF32 (2^-11 operand rounding)
// does not.  For the uint8 input layer the pixel values 0..255 are exact in tf32 (no lo part) and the 1/255 scale is
// applied to the accumulator.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace paacb {

enum { TC_FWD_U8 = 0, TC_FWD_F32 = 1, TC_DGRAD = 2 };

// ------------------------------------------------------------------------------------------------
// weight prepack: fp32 weights -> swizzled K-major images of tf32 hi and lo, one per (class, n-tile, k-block)
// image word index: (img * BN + row) * 32 + ((chunk ^ (row & 7)) * 4 + e),  k = kb*32 + chunk*4 + e
// ------------------------------------------------------------------------------------------------
__global__ void pack_fwd_weights_kernel(const float* __restrict__ w, int K, int N, int BN, uint32_t* __restrict__ hi,
                                        uint32_t* __restrict__ lo) {
  const int KB = K / 32;
  const int64_t total = (int64_t)N * (K / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int n = (int)(i % N);
    const int k4 = (int)(i / N);              // group of 4 consecutive k
    const int kb = k4 >> 3, chunk = k4 & 7;
    const int nt = n / BN, row = n - nt * BN;
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float v = __ldg(w + (int64_t)(k4 * 4 + e) * N + n);
      h[e] = tf32_rna(v);
      l[e] = tf32_rna(v - __uint_as_float(h[e]));
    }
    const int64_t dst = (((int64_t)nt * KB + kb) * BN + row) * 32 + ((chunk ^ (row & 7)) << 2);
    *reinterpret_cast<uint4*>(hi + dst) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + dst) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// dgrad operand: B_cls[k = (tj, ti, co), c] = W[ph + s*tj, pw + s*ti, c, co] (zero when the tap is outside the filter)
__global__ void pack_dgrad_weights_kernel(const float* __restrict__ w, LayerGeom g, int BN, int J, int I,
                                          uint32_t* __restrict__ hi, uint32_t* __restrict__ lo) {
  const int s = g.stride;
  const int Kd = J * I * g.N;                 // g.N = Cout
  const int KB = Kd / 32;
  const int n_tiles = g.C / BN;
  const int64_t total = (int64_t)s * s * g.C * (Kd / 4);
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int k4 = (int)(i % (Kd / 4));       // co fastest: coalesced reads of HWIO
    const int64_t rest = i / (Kd / 4);
    const int c = (int)(rest % g.C);
    const int cls = (int)(rest / g.C);
    const int ph = cls / s, pw = cls - ph * s;
    const int k = k4 * 4;
    const int tap = k / g.N, co = k - tap * g.N;
    const int tj = tap / I, ti = tap - tj * I;
    const int kh = ph + s * tj, kw = pw + s * ti;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (kh < g.R && kw < g.S) v = __ldg(reinterpret_cast<const float4*>(w + ((int64_t)(kh * g.S + kw) * g.C + c) * g.N + co));
    const float f[4] = {v.x, v.y, v.z, v.w};
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      h[e] = tf32_rna(f[e]);
      l[e] = tf32_rna(f[e] - __uint_as_float(h[e]));
    }
    const int kb = k4 >> 3, chunk = k4 & 7;
    const int nt = c / BN, row = c - nt * BN;
    const int64_t img = ((int64_t)cls * n_tiles + nt) * KB + kb;
    const int64_t dst = (img * BN + row) * 32 + ((chunk ^ (row & 7)) << 2);
    *reinterpret_cast<uint4*>(hi + dst) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo + dst) = make_uint4(l[0], l[1], l[2], l[3]);
  }
}

// ------------------------------------------------------------------------------------------------
// the implicit-GEMM kernel
// ------------------------------------------------------------------------------------------------
constexpr int kTcGroups = 2;                // producer groups of 128 threads (4 warps) that take K-blocks round-robin
constexpr int kTcThreads = kTcGroups * 128 + 32 + 128;
constexpr int kTcMmaWarp = kTcGroups * 4;   // warps [0, 4*NG) produce, warp 4*NG issues MMAs, the next four run the epilogue
constexpr int kMaxKB = 128;                 // K-blocks per tile the per-K-block table can hold

struct TcParams {
  const void* x;          // fwd: layer input (uint8 states or fp32 NHWC); dgrad: dZ of this layer [b, OH, OW, Cout]
  const uint32_t* b_hi;   // prepacked operand images
  const uint32_t* b_lo;
  const float* bias;      // fwd
  const float* xact;      // dgrad: activation feeding this layer (ReLU mask) or nullptr
  float* y;               // fwd: output [M, N]; dgrad: dX [b, H, W, C]
  LayerGeom g;
  uint32_t M;             // GEMM rows (per class)
  uint32_t m_tiles;       // per class
  int n_tiles;
  int classes;            // dgrad: stride^2
  int kblocks;
  int Hq, Wq, I;          // dgrad: class grid and taps per row
  float in_scale;
  int relu;
};

constexpr int kSmemBudget = 224 * 1024;      // B stages + cp.async staging (the per-SM maximum is 227 KB incl. static)

template <int BN, int MODE, bool SPLIT, int KSUB>
struct TcCfg {
  // One pipeline stage covers KSUB consecutive 32-wide K-blocks: the producer/MMA handshake (mbarrier round trip,
  // tcgen05.wait::st, fences) costs ~700 cycles per stage whatever its payload, so narrow tiles use larger stages.
  static constexpr bool U8 = (MODE == TC_FWD_U8);
  static constexpr bool A_LO = SPLIT && !U8;
  static constexpr int B_BYTES = BN * 128;                                      // one 32-wide K-block image of B
  static constexpr int STAGE_BYTES = KSUB * B_BYTES * (SPLIT ? 2 : 1);          // shared memory per pipeline stage (B only)
  static constexpr int ACOLS = A_LO ? 64 : 32;                                  // TMEM columns per 32-wide K-block of A
  static constexpr int SCOLS = KSUB * ACOLS;                                    // TMEM columns per A stage
  static constexpr int ROWB = U8 ? 32 : 128;                                    // bytes of one row of one 32-wide K-block
  static constexpr int NV = ROWB / 16;                                          // 16-byte chunks per row per K-block
  static constexpr int NG = kTcGroups;
  static constexpr int S_TMEM = ((512 - 2 * BN) / SCOLS) > 4 ? 4 : ((512 - 2 * BN) / SCOLS);
  static constexpr int STAGES = S_TMEM;
  static constexpr int STG_UNIT = NG * 128 * ROWB * KSUB;                       // staging bytes per unit of depth
  static constexpr int D_FIT = (kSmemBudget - STAGES * STAGE_BYTES) / STG_UNIT;
  static constexpr int DEPTH = D_FIT > (U8 ? 6 : 3) ? (U8 ? 6 : 3) : D_FIT;    // stages in flight per producer thread
  static constexpr int STG_BYTES = STG_UNIT * DEPTH;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + STG_BYTES + 1024 /* alignment slack */ + 256 /* barriers */;
  static constexpr int TMEM_COLS = 512;
  static_assert(STAGES >= 2 && DEPTH >= 1, "pipeline does not fit");
};

template <int BN, int MODE, bool SPLIT, int KSUB>
__global__ void __launch_bounds__(kTcThreads, 1) igemm_tc_kernel(const TcParams p) {
  using Cfg = TcCfg<BN, MODE, SPLIT, KSUB>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int NV = Cfg::NV, DEPTH = Cfg::DEPTH, NG = Cfg::NG;
  extern __shared__ uint8_t smem_raw[];
  __shared__ int kb_tab[kMaxKB];                // per-K-block source element offsets (no division in the hot loop)
  __shared__ int kb_tap[kMaxKB];                // dgrad: (tj << 8) | ti of the K-block's filter tap
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* stg_base = smem + STAGES * Cfg::STAGE_BYTES;                        // cp.async staging rings
  uint64_t* bars = reinterpret_cast<uint64_t*>(stg_base + Cfg::STG_BYTES);
  uint64_t* full_bar = bars;                    // [STAGES]  producers (128 + 1) -> MMA
  uint64_t* empty_bar = bars + STAGES;          // [STAGES]  MMA commit -> producers
  uint64_t* tfull_bar = bars + 2 * STAGES;      // [2]       MMA commit -> epilogue
  uint64_t* tempty_bar = bars + 2 * STAGES + 2; // [2]       epilogue (128) -> MMA
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const LayerGeom& g = p.g;
  const uint32_t tiles_per_class = p.m_tiles * (uint32_t)p.n_tiles;
  const uint32_t total_tiles = tiles_per_class * (uint32_t)p.classes;
  const int my_tiles = (int)((total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);   // tiles of this CTA
  const int KB = p.kblocks;                     // 32-wide K-blocks per tile
  const int KBS = KB / KSUB;                    // pipeline stages per tile

  if (tid == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 128 + 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tfull_bar[s], 1);
      mbar_init(&tempty_bar[s], 128);
    }
    fence_barrier_init();
  }
  for (int kb = tid; kb < KB; kb += kTcThreads) {
    const int k0 = kb * 32;
    if constexpr (MODE == TC_DGRAD) {
      const int tap = k0 / g.N, co0 = k0 - tap * g.N;
      const int tj = tap / p.I, ti = tap - tj * p.I;
      kb_tab[kb] = co0 - (tj * g.OW + ti) * g.N;
      kb_tap[kb] = (tj << 8) | ti;
    } else {
      const int SC = g.S * g.C;
      const int kh = k0 / SC, off = k0 - kh * SC;
      kb_tab[kb] = kh * g.W * g.C + off;
    }
  }
  if (warp == kTcMmaWarp) tmem_alloc(tmem_slot, Cfg::TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  constexpr uint32_t kAcol0 = 2 * BN;           // first TMEM column of the A stages (A_TMEM)

  if (warp < kTcMmaWarp) {
    // =========================== A producers (+ B bulk copy) ===========================
    const int grp = warp >> 2;                 // owns iterations it with it % NG == grp
    const int wq4 = warp & 3;                  // this warp stages, converts and writes tile rows 32*wq4 .. 32*wq4+31
    const int lane = tid & 31;
    const uint32_t ohw = (uint32_t)(g.OH * g.OW);
    const int total_it = my_tiles * KBS;
    // COALESCED staging: the NVR lanes that share a row fetch its NVR consecutive 16-byte chunks, so one warp-wide
    // cp.async touches 32/NVR rows = 32/NVR cache lines (a lane-per-row gather would touch 32 lines per instruction
    // and is bound by the L1 wavefront rate: measured 4x slower).  Lane l later reads back ROW l of the warp's slab.
    constexpr int NVR = Cfg::NV;               // 16-byte chunks per row per K-block (8 fp32 / 2 uint8)
    constexpr int RPI = 32 / NVR;              // rows covered by one warp-wide cp.async
    constexpr int NI = 32 / RPI;               // cp.async instructions per K-block per lane
    constexpr int ESZ = Cfg::U8 ? 1 : 4;
    const int my_chunk = lane % NVR;
    const int my_row0 = lane / NVR;            // instruction j stages slab row j*RPI + my_row0
    constexpr uint32_t kSlot = KSUB * 32 * Cfg::ROWB;    // one depth slot of this warp's slab: [KSUB][32 rows][ROWB]
    const uint32_t slab = smem_u32(stg_base) + (uint32_t)((grp * 4 + wq4) * DEPTH) * kSlot;
    auto swz_of = [](int row) -> uint32_t { return Cfg::U8 ? (uint32_t)((row >> 2) & 1) : (uint32_t)(row & 7); };

    // load-stream position (advances by NG K-blocks per owned iteration) and per-tile state of the NI rows this lane stages
    int ld_tl = 0, ld_kb = grp * KSUB;
    while (ld_kb >= KB) { ld_kb -= KB; ++ld_tl; }
    int cached_tile = -1;
    int64_t base_j[NI];        // element offset of the row's first k (fwd) / of dZ[smp, hq, wq, 0] (dgrad)
    int hw_j[NI];              // dgrad: (hq << 16) | wq
    uint32_t ok_mask = 0;      // bit j: row j*RPI + my_row0 exists
    int img_base = 0;          // (class * n_tiles + n_tile) * KB
    int img_of[DEPTH];

    auto issue = [&](int d, int& img) {
      if (ld_tl != cached_tile) {
        cached_tile = ld_tl;
        const uint32_t t = blockIdx.x + (uint32_t)ld_tl * gridDim.x;
        const uint32_t cls = t / tiles_per_class;
        const uint32_t tc = t - cls * tiles_per_class;
        const uint32_t mt = tc / (uint32_t)p.n_tiles;
        const int nt = (int)(tc - mt * (uint32_t)p.n_tiles);
        img_base = ((int)cls * p.n_tiles + nt) * KB;
        ok_mask = 0;
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          const uint32_t m = mt * 128u + (uint32_t)(wq4 * 32 + j * RPI + my_row0);
          base_j[j] = 0;
          hw_j[j] = 0;
          if (m < p.M) {
            ok_mask |= 1u << j;
            if constexpr (MODE == TC_DGRAD) {
              const uint32_t hw = (uint32_t)(p.Hq * p.Wq);
              const uint32_t sm = m / hw;
              const uint32_t rem = m - sm * hw;
              const uint32_t hq = rem / (uint32_t)p.Wq, wq = rem - hq * (uint32_t)p.Wq;
              hw_j[j] = (int)((hq << 16) | wq);
              base_j[j] = (((int64_t)sm * g.OH + hq) * g.OW + wq) * (int64_t)g.N;
            } else {
              const uint32_t sm = m / ohw;
              const uint32_t rem = m - sm * ohw;
              const uint32_t oh = rem / (uint32_t)g.OW, ow = rem - oh * (uint32_t)g.OW;
              base_j[j] = (((int64_t)sm * g.H + (int64_t)oh * g.stride) * g.W + (int64_t)ow * g.stride) * g.C;
            }
          }
        }
      }
      img = img_base + ld_kb;
      const uint8_t* xb = reinterpret_cast<const uint8_t*>(p.x);
#pragma unroll
      for (int sb = 0; sb < KSUB; ++sb) {
        const int tab = kb_tab[ld_kb + sb];
        const int tap = (MODE == TC_DGRAD) ? kb_tap[ld_kb + sb] : 0;
        const uint32_t dst0 = slab + (uint32_t)d * kSlot + (uint32_t)(sb * 32 * Cfg::ROWB);
#pragma unroll
        for (int j = 0; j < NI; ++j) {
          bool ok = (ok_mask >> j) & 1u;
          if constexpr (MODE == TC_DGRAD) {
            // k = (tj, ti, co): the row reads dZ[smp, hq - tj, wq - ti, co0 .. co0 + 32); tab = co0 - (tj*OW + ti)*Cout
            const int oh = (hw_j[j] >> 16) - (tap >> 8), ow = (hw_j[j] & 0xffff) - (tap & 0xff);
            ok = ok && oh >= 0 && ow >= 0 && oh < g.OH && ow < g.OW;
          }
          const uint8_t* src = ok ? xb + (base_j[j] + tab) * ESZ + my_chunk * 16 : xb;   // !ok: 0 bytes read, zero fill
          const int row = j * RPI + my_row0;
          cp_async16(dst0 + (uint32_t)(row * Cfg::ROWB) + (((uint32_t)my_chunk ^ swz_of(row)) << 4), src, ok ? 16u : 0u);
        }
      }
      ld_kb += NG * KSUB;
      while (ld_kb >= KB) { ld_kb -= KB; ++ld_tl; }
    };

    int pstage = grp;
    uint32_t pphase = 0;
    while (pstage >= STAGES) { pstage -= STAGES; pphase ^= 1u; }

#pragma unroll
    for (int u = 0; u < DEPTH; ++u) {
      if (grp + NG * u < total_it) issue(u, img_of[u]);
      cp_async_commit();
    }
    for (int base = grp; base < total_it; base += NG * DEPTH) {
#pragma unroll
      for (int u = 0; u < DEPTH; ++u) {
        const int it = base + NG * u;
        if (it < total_it) {
          cp_async_wait<DEPTH - 1>();          // this lane's copies for iteration `it` have landed in slot u ...
          __syncwarp();                        // ... and so have the other lanes' (the slab row is written by NVR lanes)
          uint4 b[KSUB][NV];
#pragma unroll
          for (int sb = 0; sb < KSUB; ++sb) {
            const uint32_t rowp = slab + (uint32_t)u * kSlot + (uint32_t)(sb * 32 * Cfg::ROWB) + (uint32_t)(lane * Cfg::ROWB);
#pragma unroll
            for (int c = 0; c < NV; ++c) b[sb][c] = lds128(rowp + (((uint32_t)c ^ swz_of(lane)) << 4));
          }
          __syncwarp();                        // every lane has read its rows: slot u may be refilled
          const int img = img_of[u];
          if (it + NG * DEPTH < total_it) issue(u, img_of[u]);
          cp_async_commit();

          mbar_wait(&empty_bar[pstage], pphase ^ 1u);
          if (wq4 == 0 && elect_one_sync()) {
            uint8_t* b_hi = smem + (size_t)pstage * Cfg::STAGE_BYTES;
            mbar_arrive_expect_tx(&full_bar[pstage], Cfg::STAGE_BYTES);
            bulk_g2s(b_hi, p.b_hi + (int64_t)img * (BN * 32), KSUB * Cfg::B_BYTES, &full_bar[pstage]);
            if constexpr (SPLIT)
              bulk_g2s(b_hi + KSUB * Cfg::B_BYTES, p.b_lo + (int64_t)img * (BN * 32), KSUB * Cfg::B_BYTES, &full_bar[pstage]);
          }
          // this thread's row of the A operand goes straight into tensor memory: lane = row, 32 columns per K-block
#pragma unroll
          for (int sb = 0; sb < KSUB; ++sb) {
            const uint32_t taddr = tmem_base + ((uint32_t)(wq4 * 32) << 16) + kAcol0 + (uint32_t)(pstage * Cfg::SCOLS + sb * Cfg::ACOLS);
            uint32_t hi[32];
            if constexpr (Cfg::U8) {
              const uint32_t wds[8] = {b[sb][0].x, b[sb][0].y, b[sb][0].z, b[sb][0].w, b[sb][1].x, b[sb][1].y, b[sb][1].z, b[sb][1].w};
#pragma unroll
              for (int c = 0; c < 8; ++c) {     // small integers are exact in tf32
                hi[c * 4 + 0] = __float_as_uint(u8_to_f32(wds[c], 0));
                hi[c * 4 + 1] = __float_as_uint(u8_to_f32(wds[c], 1));
                hi[c * 4 + 2] = __float_as_uint(u8_to_f32(wds[c], 2));
                hi[c * 4 + 3] = __float_as_uint(u8_to_f32(wds[c], 3));
              }
              tmem_st32(taddr, hi);
            } else {
              // TF32X3: hi = a with the 13 low mantissa bits cleared (1 LOP), lo = a - hi exactly (1 FADD); the tensor
              // core reads only the tf32 bits of lo, an error of 2^-21 |a|.  Plain TF32 rounds to nearest (2 integer ops).
#pragma unroll
              for (int c = 0; c < 8; ++c) {
                hi[c * 4 + 0] = Cfg::A_LO ? (b[sb][c].x & 0xFFFFE000u) : tf32_rna_bits(b[sb][c].x);
                hi[c * 4 + 1] = Cfg::A_LO ? (b[sb][c].y & 0xFFFFE000u) : tf32_rna_bits(b[sb][c].y);
                hi[c * 4 + 2] = Cfg::A_LO ? (b[sb][c].z & 0xFFFFE000u) : tf32_rna_bits(b[sb][c].z);
                hi[c * 4 + 3] = Cfg::A_LO ? (b[sb][c].w & 0xFFFFE000u) : tf32_rna_bits(b[sb][c].w);
              }
              tmem_st32(taddr, hi);
              if constexpr (Cfg::A_LO) {
                uint32_t lo[32];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                  lo[c * 4 + 0] = __float_as_uint(__uint_as_float(b[sb][c].x) - __uint_as_float(hi[c * 4 + 0]));
                  lo[c * 4 + 1] = __float_as_uint(__uint_as_float(b[sb][c].y) - __uint_as_float(hi[c * 4 + 1]));
                  lo[c * 4 + 2] = __float_as_uint(__uint_as_float(b[sb][c].z) - __uint_as_float(hi[c * 4 + 2]));
                  lo[c * 4 + 3] = __float_as_uint(__uint_as_float(b[sb][c].w) - __uint_as_float(hi[c * 4 + 3]));
                }
                tmem_st32(taddr + 32u, lo);
              }
            }
          }
          tmem_st_wait();                      // tcgen05.st complete ...
          tc_fence_before();                   // ... and ordered before the arrive the MMA thread observes
          mbar_arrive(&full_bar[pstage]);
          pstage += NG;
          while (pstage >= STAGES) { pstage -= STAGES; pphase ^= 1u; }
        }
      }
    }
    cp_async_wait<0>();
  } else if (warp == kTcMmaWarp) {
    // =========================== MMA issuer ===========================
    // The whole warp walks the loop (warp-uniform control flow, so descriptors and addresses live in uniform
    // registers); one elected lane issues.  Issuing from inside a divergent `if (lane == 0)` made the compiler wrap
    // every tcgen05.mma in an ELECT / BRA.U.ANY sequence (~90 cycles per MMA: the first version's real bottleneck).
    {
      constexpr uint32_t idesc = make_idesc_tf32(BN);
      const bool leader = elect_one_sync();
      int stage = 0;
      uint32_t phase = 0;
      for (int tl = 0; tl < my_tiles; ++tl) {
        const int acc = tl & 1;
        const uint32_t acc_phase = (uint32_t)((tl >> 1) & 1);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BN);
        for (int kb = 0; kb < KBS; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t b_st = smem_u32(smem + (size_t)stage * Cfg::STAGE_BYTES);
          if (leader) {
#pragma unroll
            for (int sb = 0; sb < KSUB; ++sb) {
              const uint32_t b_hi = b_st + (uint32_t)(sb * Cfg::B_BYTES), b_lo = b_hi + (uint32_t)(KSUB * Cfg::B_BYTES);
#pragma unroll
              for (int ks = 0; ks < 4; ++ks) {   // K = 8 tf32 per instruction: 32 bytes of smem (B) / 8 TMEM columns (A)
                const uint32_t ko = (uint32_t)ks * 32u;
                uint32_t accum = (kb > 0 || sb > 0 || ks > 0) ? 1u : 0u;
                const uint32_t a_hi = tmem_base + kAcol0 + (uint32_t)(stage * Cfg::SCOLS + sb * Cfg::ACOLS) + (uint32_t)ks * 8u;
                if constexpr (SPLIT) {
                  if constexpr (Cfg::A_LO) {
                    umma_tf32_ts(d_tmem, a_hi + 32u, make_sw128_desc(b_hi + ko), idesc, accum);
                    accum = 1u;
                  }
                  umma_tf32_ts(d_tmem, a_hi, make_sw128_desc(b_lo + ko), idesc, accum);
                  accum = 1u;
                }
                umma_tf32_ts(d_tmem, a_hi, make_sw128_desc(b_hi + ko), idesc, accum);
              }
            }
            umma_commit(&empty_bar[stage]);      // stage reusable once these MMAs retire
          }
          __syncwarp();
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (leader) umma_commit(&tfull_bar[acc]);   // accumulator complete
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue ===========================
    const int ew = warp & 3;                   // TMEM lane quarter this warp may access
    const int lane = tid & 31;
    for (int tl = 0; tl < my_tiles; ++tl) {
      const int acc = tl & 1;
      const uint32_t acc_phase = (uint32_t)((tl >> 1) & 1);
      const uint32_t t = blockIdx.x + (uint32_t)tl * gridDim.x;
      const uint32_t cls = t / tiles_per_class;
      const uint32_t tc = t - cls * tiles_per_class;
      const uint32_t mt = tc / (uint32_t)p.n_tiles;
      const int nt = (int)(tc - mt * (uint32_t)p.n_tiles);
      const uint32_t m = mt * 128u + (uint32_t)(ew * 32 + lane);
      bool ok = m < p.M;
      int64_t out_base = 0;
      if constexpr (MODE == TC_DGRAD) {
        if (ok) {
          const int s = g.stride;
          const int ph = (int)cls / s, pw = (int)cls - ph * s;
          const uint32_t hw = (uint32_t)(p.Hq * p.Wq);
          const uint32_t sm = m / hw;
          const uint32_t rem = m - sm * hw;
          const int qh = (int)(rem / (uint32_t)p.Wq), qw = (int)(rem - (uint32_t)qh * (uint32_t)p.Wq);
          const int h = ph + s * qh, wv = pw + s * qw;
          ok = (h < g.H) && (wv < g.W);
          out_base = (((int64_t)sm * g.H + h) * g.W + wv) * (int64_t)g.C + nt * BN;
        }
      } else {
        out_base = (int64_t)m * g.N + nt * BN;
      }
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN);
      constexpr int CW = BN < 32 ? BN : 32;     // columns per TMEM load (16 for the NIPS layers with 16 channels)
#pragma unroll
      for (int c0 = 0; c0 < BN; c0 += CW) {
        uint32_t v[32];
        if constexpr (CW == 16) {
          uint32_t v16[16];
          tmem_ld16(taddr, v16);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) { v[j] = v16[j]; v[j + 16] = 0u; }
        } else {
          tmem_ld32(taddr + (uint32_t)c0, v);
          tmem_ld_wait();
        }
        if (ok) {
          float* dst = p.y + out_base + c0;
          if constexpr (MODE == TC_DGRAD) {
            const float* xa = (p.xact != nullptr) ? p.xact + out_base + c0 : nullptr;
#pragma unroll
            for (int j = 0; j < CW; j += 4) {
              float4 o = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                                     __uint_as_float(v[j + 3]));
              if (xa != nullptr) {
                const float4 a = __ldg(reinterpret_cast<const float4*>(xa + j));
                o.x = a.x > 0.f ? o.x : 0.f; o.y = a.y > 0.f ? o.y : 0.f;
                o.z = a.z > 0.f ? o.z : 0.f; o.w = a.w > 0.f ? o.w : 0.f;
              }
              *reinterpret_cast<float4*>(dst + j) = o;
            }
          } else {
            const float* bp = p.bias + nt * BN + c0;
#pragma unroll
            for (int j = 0; j < CW; j += 4) {
              float4 o;
              o.x = fmaf(__uint_as_float(v[j + 0]), p.in_scale, __ldg(bp + j + 0));
              o.y = fmaf(__uint_as_float(v[j + 1]), p.in_scale, __ldg(bp + j + 1));
              o.z = fmaf(__uint_as_float(v[j + 2]), p.in_scale, __ldg(bp + j + 2));
              o.w = fmaf(__uint_as_float(v[j + 3]), p.in_scale, __ldg(bp + j + 3));
              if (p.relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
              *reinterpret_cast<float4*>(dst + j) = o;
            }
          }
        }
      }
      tc_fence_before();
      mbar_arrive(&tempty_bar[acc]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kTcMmaWarp) {
    tc_fence_after();
    tmem_dealloc(tmem_base, Cfg::TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------------
// launchers
// ------------------------------------------------------------------------------------------------
template <int BN, int MODE, bool SPLIT, int KSUB>
static int launch_tc_inst2(const paacb_ctx* ctx, const TcParams& p, int slot, cudaStream_t st) {
  using Cfg = TcCfg<BN, MODE, SPLIT, KSUB>;
  static DeviceOnce attr_set;   // kernel attributes are per device: one bit per device index
  if (!attr_set.done(ctx->device)) {
    if (cudaFuncSetAttribute(igemm_tc_kernel<BN, MODE, SPLIT, KSUB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             Cfg::SMEM_BYTES) != cudaSuccess) {
      cudaGetLastError();
      set_error("igemm_tc: cannot set %d bytes of dynamic shared memory", Cfg::SMEM_BYTES);
      return PAACB_ECUDA;
    }
    attr_set.mark(ctx->device);
  }
  const uint32_t tiles = p.m_tiles * (uint32_t)p.n_tiles * (uint32_t)p.classes;
  const unsigned grid = tiles < (uint32_t)ctx->num_sms ? tiles : (unsigned)ctx->num_sms;
  PAACB_LAUNCH_BEGIN(ctx, slot, st);
  igemm_tc_kernel<BN, MODE, SPLIT, KSUB><<<grid, kTcThreads, Cfg::SMEM_BYTES, st>>>(p);
  PAACB_LAUNCH_END(ctx, slot, st);
  return PAACB_OK;
}

template <int BN, int MODE>
static int launch_tc_inst(const paacb_ctx* ctx, const TcParams& p, int slot, int split3, cudaStream_t st) {
  // K-blocks per pipeline stage: 4 for the uint8 layer (32-byte rows: small stages are all handshake); the fp32
  // layers measured faster with single-K-block stages (deeper TMEM / smem pipelines, fewer live registers)
  constexpr int KS = (MODE == TC_FWD_U8) ? 4 : 1;
  if (KS > 1 && p.kblocks % KS == 0) {
    return split3 ? launch_tc_inst2<BN, MODE, true, KS>(ctx, p, slot, st) : launch_tc_inst2<BN, MODE, false, KS>(ctx, p, slot, st);
  }
  return split3 ? launch_tc_inst2<BN, MODE, true, 1>(ctx, p, slot, st) : launch_tc_inst2<BN, MODE, false, 1>(ctx, p, slot, st);
}

static int pick_bn(int n) { return (n % 128 == 0) ? 128 : ((n % 64 == 0) ? 64 : ((n % 32 == 0) ? 32 : ((n % 16 == 0) ? 16 : 0))); }

int launch_pack_weights(const paacb_ctx* ctx, const LayerGeom& g, const float* w, cudaStream_t st) {
  if (ctx->wpack_hi == nullptr) return PAACB_EUNSUPPORTED;
  const int bn = pick_bn(g.N);
  if (bn != 0 && g.K % 32 == 0) {
    const int64_t total = (int64_t)g.N * (g.K / 4);
    PAACB_LAUNCH_BEGIN(ctx, K_PACK, st);
    pack_fwd_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w, g.K, g.N, bn, ctx->wpack_hi + g.w_off,
                                                                             ctx->wpack_lo + g.w_off);
    PAACB_LAUNCH_END(ctx, K_PACK, st);
  }
  return PAACB_OK;
}

int launch_pack_dgrad_weights(const paacb_ctx* ctx, const LayerGeom& g, const float* w, cudaStream_t st) {
  if (ctx->wpack_d_hi == nullptr) return PAACB_EUNSUPPORTED;
  const int s = g.stride;
  const int J = (g.R + s - 1) / s, I = (g.S + s - 1) / s;
  const int bn = pick_bn(g.C);
  if (bn == 0 || g.N % 32 != 0 || (int64_t)s * s * J * I != (int64_t)g.R * g.S) return PAACB_OK;   // layer stays on the SIMT path
  const int64_t total = (int64_t)s * s * g.C * (J * I * g.N / 4);
  PAACB_LAUNCH_BEGIN(ctx, K_PACK, st);
  pack_dgrad_weights_kernel<<<(unsigned)((total + 255) / 256), 256, 0, st>>>(w, g, bn, J, I, ctx->wpack_d_hi + g.w_off,
                                                                            ctx->wpack_d_lo + g.w_off);
  PAACB_LAUNCH_END(ctx, K_PACK, st);
  return PAACB_OK;
}

int launch_conv_fwd_tc(const paacb_ctx* ctx, const LayerGeom& g, const void* x, const float* w, const float* bias,
                       float* y, int64_t batch, int split3, cudaStream_t st) {
  (void)w;
  const int bn = pick_bn(g.N);
  const int64_t M = batch * g.OH * g.OW;
  if ((g.S * g.C) % 32 != 0 || g.K % 32 != 0 || g.K / 32 > kMaxKB || bn == 0 || ctx->wpack_hi == nullptr ||
      M >= (1LL << 31) - 256)
    return PAACB_EUNSUPPORTED;
  if (M == 0) return PAACB_OK;
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.x = x;
  p.b_hi = ctx->wpack_hi + g.w_off;
  p.b_lo = ctx->wpack_lo + g.w_off;
  p.bias = bias;
  p.y = y;
  p.g = g;
  p.M = (uint32_t)M;
  p.m_tiles = (uint32_t)((M + 127) / 128);
  p.n_tiles = g.N / bn;
  p.classes = 1;
  p.kblocks = g.K / 32;
  p.in_scale = g.in_u8 ? 0.003921568859368563f : 1.0f;
  p.relu = 1;
  const int slot = K_FWD0 + g.index;
  if (g.in_u8) {
    if (bn == 16) return launch_tc_inst<16, TC_FWD_U8>(ctx, p, slot, split3, st);
    if (bn == 32) return launch_tc_inst<32, TC_FWD_U8>(ctx, p, slot, split3, st);
    if (bn == 64) return launch_tc_inst<64, TC_FWD_U8>(ctx, p, slot, split3, st);
    return PAACB_EUNSUPPORTED;
  }
  if (bn == 16) return launch_tc_inst<16, TC_FWD_F32>(ctx, p, slot, split3, st);
  if (bn == 32) return launch_tc_inst<32, TC_FWD_F32>(ctx, p, slot, split3, st);
  if (bn == 64) return launch_tc_inst<64, TC_FWD_F32>(ctx, p, slot, split3, st);
  return launch_tc_inst<128, TC_FWD_F32>(ctx, p, slot, split3, st);
}

int launch_conv_dgrad_tc(const paacb_ctx* ctx, const LayerGeom& g, const float* dz, const float* x_act, float* dx,
                         int64_t batch, int split3, cudaStream_t st) {
  const int s = g.stride;
  const int J = (g.R + s - 1) / s, I = (g.S + s - 1) / s;
  const int bn = pick_bn(g.C);
  const int Hq = (g.H + s - 1) / s, Wq = (g.W + s - 1) / s;
  const int64_t M = batch * Hq * Wq;
  if (bn == 0 || g.N % 32 != 0 || g.N > 65535 || g.in_u8 || ctx->wpack_d_hi == nullptr || J * I * g.N / 32 > kMaxKB ||
      (int64_t)s * s * J * I != (int64_t)g.R * g.S || M >= (1LL << 31) - 256 || J > 127 || I > 127)
    return PAACB_EUNSUPPORTED;
  if (M == 0) return PAACB_OK;
  TcParams p;
  memset(&p, 0, sizeof(p));
  p.x = dz;
  p.b_hi = ctx->wpack_d_hi + g.w_off;
  p.b_lo = ctx->wpack_d_lo + g.w_off;
  p.xact = x_act;
  p.y = dx;
  p.g = g;
  p.Hq = Hq;
  p.Wq = Wq;
  p.I = I;
  p.M = (uint32_t)M;
  p.m_tiles = (uint32_t)((M + 127) / 128);
  p.n_tiles = g.C / bn;
  p.classes = s * s;
  p.kblocks = J * I * g.N / 32;
  p.in_scale = 1.0f;
  const int slot = K_DGRAD0 + g.index;
  if (bn == 16) return launch_tc_inst<16, TC_DGRAD>(ctx, p, slot, split3, st);
  if (bn == 32) return launch_tc_inst<32, TC_DGRAD>(ctx, p, slot, split3, st);
  if (bn == 64) return launch_tc_inst<64, TC_DGRAD>(ctx, p, slot, split3, st);
  return launch_tc_inst<128, TC_DGRAD>(ctx, p, slot, split3, st);
}

}  // namespace paacb
