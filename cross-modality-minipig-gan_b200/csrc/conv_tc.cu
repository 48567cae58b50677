// tcgen05 implicit-GEMM convolution for sm_100a (rank 2 NHWC and rank 3 NDHWC, bf16 operands, fp32 TMEM accumulators).
//
// Replaces cuDNN's convolution forward / backward-data / backward-filter behind nn.Conv2d / nn.ConvTranspose2d for
// the discriminator (/root/reference/code/GAN/GAN_final.py:167-189 -- 90 % of the step FLOPs) and the >=16-channel
// generator layers (MONAI Convolution via GAN_final.py:106-114).
//
// Formulation ("tap GEMM"): for a tile of 128 output pixels (a tw x th x tn box of the output grid)
//     out[p, n] = sum_{tap} sum_{c} In[pix(p) + off(tap), c] * W[tap][n][c]
//  * A operand: one TMA 4-D box (KC channels, tw, th, tn) of the NHWC input per (tap, channel chunk); it lands in
//    shared memory as 128 rows x KC bf16, K-major, hardware-swizzled (128/64/32 B) -- exactly the canonical UMMA
//    layout, so the im2col matrix is never materialised.  Zero padding and ragged tile edges come from TMA's
//    out-of-bounds zero fill (coordinates may be negative).  Stride-2 convolutions read through four "parity"
//    tensor maps (base offset (ph,pw), element strides doubled), stride-2 backward-data / ConvTranspose writes four
//    output parity classes, each an ordinary stride-1 tap list.
//  * B operand: TMA 3-D box (KC, 1 tap, BN) of the packed weights [N][tap][C] (K-major).
//  * D: 128 x BN fp32 in TMEM, double buffered (2 x BN columns) so the epilogue of tile i overlaps the MMAs of
//    tile i+1.  Persistent CTAs (one per SM), warp-specialised: warp 0 TMA producer, warp 1 MMA issuer,
//    warp 2 TMEM allocator, warps 4-7 epilogue (TMEM -> registers -> +bias -> bf16 -> global, plus the batch-norm
//    partial sums via a register transpose-reduce).
//  * Weight gradient: D[cy, cx] += dY^T X per tap, both operands MN-major straight from the NHWC tensors
//    (pixels are the K dimension), accumulators for a group of taps live in TMEM, split over pixel ranges and
//    reduced with fp32 atomics into the flat gradient buffer.
#include <cudaTypedefs.h>
#include <algorithm>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"
#include "tc_common.cuh"

namespace mpgan {
namespace tc {

constexpr int MAXT = 64;     // 4 x 4 x 4 taps (rank 3, D layers 3 / 4)
constexpr int MAXCLS = 8;    // output parity classes of a stride-2 rank-3 data gradient
constexpr int kSmemLimit = 227 * 1024;

// Activation tensor maps of one launch: one for stride 1; for stride-2 gathers one per input parity class
// (4 in rank 2, 8 in rank 3).  Passed as ONE __grid_constant__ kernel parameter and indexed by the tap's class.
struct ActMaps { CUtensorMap m[8]; };

struct TapGemmParams {
  int ncls;
  int cls_tap_begin[MAXCLS + 1];
  int cls_od[MAXCLS], cls_oh[MAXCLS], cls_ow[MAXCLS];
  long long cls_out_off[MAXCLS];
  signed char tap_map[MAXT];
  short tap_dd[MAXT], tap_dh[MAXT], tap_dw[MAXT], tap_slab[MAXT];
  int nkc;
  int tiles_w, tiles_h, tiles_d, tiles_n;      // tiles_d / td_log2: rank 3 only (1 / 0 otherwise)
  int tw_log2, th_log2, td_log2;
  int nimg;
  int n_total, n_tiles;
  int cls_minor;       // tile order: the parity classes of one spatial tile are consecutive (equal tap counts only)
  int mt;              // 128-pixel tiles per weight stage (1, or 2 for large BN = 128 layers)
  int lane_parallel;   // taps of a tile are loaded by different lanes (needs max taps per class * nkc <= STAGES)
  long long out_sn, out_sd, out_sh, out_sw;
  bf16* out;
  const float* bias;
  double* stats;
  const bf16* res;     // optional tensor added to the result before rounding (same grid / classes as out)
  long long res_sn, res_sd, res_sh, res_sw;
  long long cls_res_off[MAXCLS];
  int wide;            // output rows are 32-byte aligned: 256-bit stores
  const float* slope;  // optional device scalar: PReLU applied to (acc + bias) before the residual (inference fusion)
};

struct WgradParams {
  int ntaps;
  signed char tap_map[MAXT];
  short tap_dd[MAXT], tap_dh[MAXT], tap_dw[MAXT];
  int taps_per_group, ngroups, m_blocks, splits;
  int tiles_w, tiles_h, tiles_d, tiles_n, tw_log2, th_log2, td_log2;
  int cx, cy;
  int cx_blocks;       // X-channel blocks of NX columns each (cx = cx_blocks * NX; > 1 only for NX = 256)
  int nprod;           // TMA producer warps (1..7)
  float* dw;
};

template <int KC> struct SwizzleOf;
template <> struct SwizzleOf<64> { static constexpr uint32_t layout = 2, sbo = 1024; };
template <> struct SwizzleOf<32> { static constexpr uint32_t layout = 4, sbo = 512; };
template <> struct SwizzleOf<16> { static constexpr uint32_t layout = 6, sbo = 256; };

// Epilogue organisation.  BN <= 64 (generator layers: few MMAs per tile, so the per-tile latency chain of the
// epilogue is the bottleneck): 8 epilogue warps in two groups -- alternate tiles (BN <= 32) or alternate 32-column
// chunks (BN = 64) --, up to 8 TMEM accumulators in flight, BatchNorm statistics in per-thread registers.
// BN >= 128 (discriminator layers, MMA bound): 4 epilogue warps, double-buffered accumulator.
template <int BN> struct EpiCfg {
  static constexpr bool REG = BN <= 64;
  static constexpr int EW = REG ? 8 : 4;                       // epilogue warps
  static constexpr int THREADS = 128 + 32 * EW;
  static constexpr int NACC = REG ? (512 / BN > 8 ? 8 : 512 / BN) : 2;
  static constexpr int CH = BN >= 32 ? 32 : 16;                // columns per tcgen05.ld
  static constexpr int NCH = BN / CH;
  static constexpr uint32_t ARRIVALS = REG ? (NCH == 1 ? 4u : 8u) : 4u;
};

// MT = 128-pixel tiles that share one weight stage ("supertile", consecutive along w).  A 128-column MMA reads as
// many weight bytes as activation bytes, so with MT = 1 the BN = 128 layers (D layer 3 data gradient) were bound by the
// L2 -> shared-memory stream (125 B/clk/SM); MT = 2 reuses every weight stage twice (94 B/clk, like the BN = 256 layers).
template <int BN, int KC, int MT_> struct TapCfg {
  static constexpr int MT = MT_;
  static constexpr int A_TILE = 128 * KC * 2;
  static constexpr int A_BYTES = MT * A_TILE;
  static constexpr int B_TX = BN * KC * 2;
  static constexpr int B_BYTES = B_TX < 1024 ? 1024 : B_TX;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_BYTES = 1024;  // full/empty[<=32] + tfull/tempty[<=8] + tmem slot
  static constexpr int STAT_BYTES = EpiCfg<BN>::EW * 2 * 512 * 4;   // per-epilogue-warp stats[2*n_total<=1024 floats]
  static constexpr int AUX_BYTES = BAR_BYTES + STAT_BYTES + 512 * 4;  // barriers + stats slots + bias[n_total<=512]
  static constexpr int MAX_STAGES = (kSmemLimit - 1024 - AUX_BYTES) / STAGE_BYTES;
  // small-channel layers are TMA-latency bound: keep up to 32 stages (>= 3 tiles of a 3x3 layer) in flight
  static constexpr int STAGES = MAX_STAGES > 32 ? 32 : MAX_STAGES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + AUX_BYTES;
  static constexpr int TMEM_COLS = EpiCfg<BN>::NACC * MT * BN < 32 ? 32 : EpiCfg<BN>::NACC * MT * BN;
  static_assert(TMEM_COLS <= 512, "accumulators exceed TMEM");
  static_assert(STAGES >= 2, "pipeline too shallow");
};

// fp32 x4 reduction into global memory (address 16-byte aligned)
__device__ __forceinline__ void red_add_v4(float* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(__uint_as_float(a)),
               "f"(__uint_as_float(b)), "f"(__uint_as_float(c)), "f"(__uint_as_float(d))
               : "memory");
}

// lane l ends up with sum over the warp's lanes of v[l]
__device__ __forceinline__ float warp_transpose_reduce32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int j = 0; j < off; ++j) {
      float send = upper ? v[j] : v[j + off];
      float keep = upper ? v[j + off] : v[j];
      v[j] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// Decoded position of one tile of the persistent sequence (R3: rank-3 tensors, one more tile dimension).
struct TileIdx { int nt, twi, thi, tdi, tni, cls; };
template <bool R3> struct TapWalk {
  static constexpr int ND = R3 ? 6 : 5;
  TileWalk<ND> w;
  int minor;
  __device__ __forceinline__ void init(const TapGemmParams& P, int tile0, int step) {
    minor = P.cls_minor;
    if constexpr (R3) {
      const int rmaj[6] = {P.n_tiles, P.tiles_w, P.tiles_h, P.tiles_d, P.tiles_n, 1 << 30};
      const int rmin[6] = {P.ncls, P.n_tiles, P.tiles_w, P.tiles_h, P.tiles_d, 1 << 30};
      if (minor) w.init(tile0, step, rmin); else w.init(tile0, step, rmaj);
    } else {
      const int rmaj[5] = {P.n_tiles, P.tiles_w, P.tiles_h, P.tiles_n, 1 << 30};
      const int rmin[5] = {P.ncls, P.n_tiles, P.tiles_w, P.tiles_h, 1 << 30};
      if (minor) w.init(tile0, step, rmin); else w.init(tile0, step, rmaj);
    }
  }
  __device__ __forceinline__ void next() { w.next(); }
  __device__ __forceinline__ TileIdx get() const {
    const int o = minor ? 1 : 0;   // class-minor order puts the class digit first
    TileIdx t;
    t.nt = w.d[o]; t.twi = w.d[o + 1]; t.thi = w.d[o + 2];
    t.tdi = R3 ? w.d[o + 3] : 0;
    t.tni = w.d[o + (R3 ? 4 : 3)];
    t.cls = minor ? w.d[0] : w.d[ND - 1];
    return t;
  }
};

template <int BN, int KC, int MT_, bool R3>
__global__ void __launch_bounds__(EpiCfg<BN>::THREADS, 1)
tapgemm_kernel(const __grid_constant__ TapGemmParams P, const __grid_constant__ ActMaps tmA,
               const __grid_constant__ CUtensorMap tmB) {
  using Cfg = TapCfg<BN, KC, MT_>;
  using Epi = EpiCfg<BN>;
  constexpr int STAGES = Cfg::STAGES;
  constexpr int NACC = Epi::NACC;
  constexpr int MT = Cfg::MT;
  // No static shared memory in this kernel, so the dynamic window starts at the CTA's (1024-byte aligned) base; using
  // the symbol directly (instead of a manually aligned pointer) lets the compiler emit LDS/STS rather than generic
  // loads and stores for every shared-memory access of the epilogue.
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint64_t* tempty = tfull + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 8);
  float* s_stats = reinterpret_cast<float*>(smem + STAGES * Cfg::STAGE_BYTES + Cfg::BAR_BYTES);
  float* s_bias = s_stats + Epi::EW * 2 * 512;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmA.m[0]);
    prefetch_tmap(&tmB);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&tfull[i], 1); mbar_init(&tempty[i], Epi::ARRIVALS); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  // (layers wider than 512 output channels -- the patch discriminator's Linear as a 1x1 convolution -- carry neither a
  //  bias nor statistics: the 512 bias slots are then all zero and indexed modulo 512)
  const int n_slots = P.n_total < 512 ? P.n_total : 512;
  if (P.stats) for (int i = threadIdx.x; i < Epi::EW * 2 * P.n_total; i += blockDim.x) s_stats[i] = 0.f;
  pdl_wait();      // PDL: barrier init / TMEM allocation / descriptor prefetch above overlap the previous kernel
  pdl_launch();
  for (int i = threadIdx.x; i < n_slots; i += blockDim.x) s_bias[i] = P.bias ? __ldg(&P.bias[i]) : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int tn_log2 = 7 - P.tw_log2 - P.th_log2 - (R3 ? P.td_log2 : 0);
  const int per_cls = P.tiles_n * (R3 ? P.tiles_d : 1) * P.tiles_h * P.tiles_w * P.n_tiles;
  const int total_tiles = per_cls * P.ncls;

  if (warp == 0) {
    if (!P.lane_parallel) {
    if (elect_one()) {  // ================= TMA producer (one thread) =================
      int stage = 0;
      uint32_t phase = 0;
      TapWalk<R3> tw5;
      tw5.init(P, (int)blockIdx.x, (int)gridDim.x);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, tw5.next()) {
        const TileIdx t = tw5.get();
        const int w0 = (t.twi * MT) << P.tw_log2, h0 = t.thi << P.th_log2, d0 = t.tdi << P.td_log2, n0 = t.tni << tn_log2;
        for (int tap = P.cls_tap_begin[t.cls]; tap < P.cls_tap_begin[t.cls + 1]; ++tap) {
          const CUtensorMap* mA = &tmA.m[P.tap_map[tap]];
          const int cw = w0 + P.tap_dw[tap], chh = h0 + P.tap_dh[tap], cd = d0 + P.tap_dd[tap], slab = P.tap_slab[tap];
          for (int kc = 0; kc < P.nkc; ++kc) {
            mbar_wait(&empty[stage], phase ^ 1);
            uint8_t* sA = smem + stage * Cfg::STAGE_BYTES;
            uint8_t* sB = sA + Cfg::A_BYTES;
            mbar_expect_tx(&full[stage], Cfg::A_BYTES + Cfg::B_TX);
#pragma unroll
            for (int sub = 0; sub < MT; ++sub) {
              if constexpr (R3) tma_load_5d(sA + sub * Cfg::A_TILE, mA, &full[stage], kc * KC, cw + (sub << P.tw_log2), chh, cd, n0);
              else tma_load_4d(sA + sub * Cfg::A_TILE, mA, &full[stage], kc * KC, cw + (sub << P.tw_log2), chh, n0);
            }
            tma_load_3d(sB, &tmB, &full[stage], kc * KC, slab, t.nt * BN);
            if (++stage == STAGES) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
    } else {
    // ================= TMA producer: lane l loads tap l of every tile =================
    // A single issuing thread needs ~40 dependent scalar instructions per (tap, chunk) -- for the generator's layers
    // (9 taps of 128 x 16..64 channels per tile) that, not bandwidth, was the tile rate.  The taps of a tile use
    // consecutive ring stages, so each lane owns one tap, waits for its own stage and issues its own two TMA loads.
    int cur_cls = -1, ntaps = 0, dd = 0, dh = 0, dw = 0, slab = 0;
    const CUtensorMap* mA = &tmA.m[0];
    uint32_t cnt = 0;   // ring position of the tile's first stage (identical in all lanes)
    TapWalk<R3> tw5;
    tw5.init(P, (int)blockIdx.x, (int)gridDim.x);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, tw5.next()) {
      const TileIdx t = tw5.get();
      if (t.cls != cur_cls) {
        cur_cls = t.cls;
        const int tb = P.cls_tap_begin[t.cls];
        ntaps = P.cls_tap_begin[t.cls + 1] - tb;
        if (lane < ntaps) {
          const int tap = tb + lane;
          mA = &tmA.m[P.tap_map[tap]];
          dd = P.tap_dd[tap]; dh = P.tap_dh[tap]; dw = P.tap_dw[tap]; slab = P.tap_slab[tap];
        }
      }
      if (lane < ntaps) {
        const int cw = ((t.twi * MT) << P.tw_log2) + dw, chh = (t.thi << P.th_log2) + dh, cd = (t.tdi << P.td_log2) + dd,
                  n0 = t.tni << tn_log2;
        for (int kc = 0; kc < P.nkc; ++kc) {
          const uint32_t a = cnt + (uint32_t)(lane * P.nkc + kc);
          const uint32_t stage = a % (uint32_t)STAGES;
          const uint32_t phase = (a / (uint32_t)STAGES) & 1u;
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sA = smem + stage * Cfg::STAGE_BYTES;
          uint8_t* sB = sA + Cfg::A_BYTES;
          mbar_expect_tx(&full[stage], Cfg::A_BYTES + Cfg::B_TX);
#pragma unroll
          for (int sub = 0; sub < MT; ++sub) {
            if constexpr (R3) tma_load_5d(sA + sub * Cfg::A_TILE, mA, &full[stage], kc * KC, cw + (sub << P.tw_log2), chh, cd, n0);
            else tma_load_4d(sA + sub * Cfg::A_TILE, mA, &full[stage], kc * KC, cw + (sub << P.tw_log2), chh, n0);
          }
          tma_load_3d(sB, &tmB, &full[stage], kc * KC, slab, t.nt * BN);
        }
      }
      cnt += (uint32_t)(ntaps * P.nkc);
      __syncwarp();   // no lane runs a tile ahead: with taps*chunks <= STAGES the stage parity stays unambiguous
    }
    }
  } else if (warp == 1) {
    if (elect_one()) {  // ================= MMA issuer =================
      constexpr uint32_t idesc = make_idesc_bf16(128, BN, 0, 0);
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      TileWalk<2> tw2;
      { const int radix[2] = {P.cls_minor ? P.ncls : per_cls, 1 << 30}; tw2.init((int)blockIdx.x, (int)gridDim.x, radix); }
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it, tw2.next()) {
        const int cls = P.cls_minor ? tw2.d[0] : tw2.d[1];
        const int buf = it % NACC;
        const uint32_t par = (uint32_t)(it / NACC) & 1u;
        mbar_wait(&tempty[buf], par ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(buf * MT * BN);
        const int kiters = (P.cls_tap_begin[cls + 1] - P.cls_tap_begin[cls]) * P.nkc;
        for (int ki = 0; ki < kiters; ++ki) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint32_t b_addr = a_addr + Cfg::A_BYTES;
#pragma unroll
          for (int k = 0; k < KC / 16; ++k) {
            const uint64_t bdesc = make_smem_desc(b_addr + k * 32, 16, SwizzleOf<KC>::sbo, SwizzleOf<KC>::layout);
#pragma unroll
            for (int sub = 0; sub < MT; ++sub) {
              const uint64_t adesc = make_smem_desc(a_addr + sub * Cfg::A_TILE + k * 32, 16, SwizzleOf<KC>::sbo,
                                                    SwizzleOf<KC>::layout);
              umma_bf16(d_tmem + (uint32_t)(sub * BN), adesc, bdesc, idesc, (ki | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(&empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull[buf]);
      }
    }
  } else if (warp >= 4) {  // ================= epilogue =================
    const int ew = warp - 4;
    const int q = ew & 3;           // TMEM lane quarter (== warp % 4)
    const int half = ew >> 2;       // second warp group (BN <= 64 only)
    const int row = q * 32 + lane;
    const int tw_mask = (1 << P.tw_log2) - 1, th_mask = (1 << P.th_log2) - 1, td_mask = R3 ? (1 << P.td_log2) - 1 : 0;
    const int lw = row & tw_mask, lh = (row >> P.tw_log2) & th_mask;
    const int ld = R3 ? (row >> (P.tw_log2 + P.th_log2)) & td_mask : 0;
    const int ln = row >> (P.tw_log2 + P.th_log2 + (R3 ? P.td_log2 : 0));
    constexpr int CH = Epi::CH;
    float* sl = s_stats + ew * 2 * P.n_total;
    if constexpr (Epi::REG) {
      constexpr int NCH = Epi::NCH;               // 1 (BN = 16, 32) or 2 (BN = 64)
      const int c0 = NCH == 2 ? half * CH : 0;
      unsigned long long s1[CH / 2], s2[CH / 2];   // packed fp32 pairs
#pragma unroll
      for (int j = 0; j < CH / 2; ++j) { s1[j] = 0ull; s2[j] = 0ull; }
      int stat_base = -1;                         // channel block the register statistics belong to
      auto flush = [&]() {                        // once per kernel unless the layer has several BN-column blocks
        float v[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = j < CH ? ((j & 1) ? unpack_f32x2(s1[j / 2]).y : unpack_f32x2(s1[j / 2]).x) : 0.f;
        const float t1 = warp_transpose_reduce32(v, lane);
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = j < CH ? ((j & 1) ? unpack_f32x2(s2[j / 2]).y : unpack_f32x2(s2[j / 2]).x) : 0.f;
        const float t2 = warp_transpose_reduce32(v, lane);
        if (lane < CH) { sl[stat_base + c0 + lane] += t1; sl[P.n_total + stat_base + c0 + lane] += t2; }
#pragma unroll
        for (int j = 0; j < CH / 2; ++j) { s1[j] = 0ull; s2[j] = 0ull; }
      };
      int it = 0;
      TapWalk<R3> tw5;
      tw5.init(P, (int)blockIdx.x, (int)gridDim.x);
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it, tw5.next()) {
        if (NCH == 1 && (it & 1) != half) continue;
        const TileIdx t = tw5.get();
        const int nt = t.nt, cls = t.cls;
        const int ow = (t.twi << P.tw_log2) + lw, oh = (t.thi << P.th_log2) + lh, od = (t.tdi << P.td_log2) + ld,
                  img = (t.tni << tn_log2) + ln;
        const bool valid = img < P.nimg && oh < P.cls_oh[cls] && ow < P.cls_ow[cls] && (!R3 || od < P.cls_od[cls]);
        const int nbase = nt * BN;
        bf16* orow = P.out + P.cls_out_off[cls] + (long long)img * P.out_sn + (long long)oh * P.out_sh +
                     (long long)ow * P.out_sw + (R3 ? (long long)od * P.out_sd : 0LL) + nbase + c0;
        if (P.stats && nbase != stat_base) {
          if (stat_base >= 0) flush();
          stat_base = nbase;
        }
        const int buf = it % NACC;
        const uint32_t par = (uint32_t)(it / NACC) & 1u;
        mbar_wait(&tfull[buf], par);
        tc_fence_after();
        const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + c0);
        uint32_t r[CH];
        if (CH == 32) tmem_ld_32x32(t_addr, r);
        else tmem_ld_32x16(t_addr, r);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&tempty[buf]);   // values are in registers: the accumulator is free again
        const bf16* rrow = P.res ? P.res + P.cls_res_off[cls] + (long long)img * P.res_sn + (long long)oh * P.res_sh +
                                       (long long)ow * P.res_sw + (R3 ? (long long)od * P.res_sd : 0LL) + nbase + c0
                                 : nullptr;
        epi_chunk_store<CH>(r, s_bias + ((nbase + c0) & 511), orow, valid, P.stats != nullptr, s1, s2, rrow, P.wide != 0, P.slope);
      }
      if (P.stats && stat_base >= 0) flush();
    } else {
    int it = 0;
    TapWalk<R3> tw5;
    tw5.init(P, (int)blockIdx.x, (int)gridDim.x);
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x, ++it, tw5.next()) {
      const TileIdx t = tw5.get();
      const int nt = t.nt, twi = t.twi, thi = t.thi, tni = t.tni, cls = t.cls;
      const int od = (t.tdi << P.td_log2) + ld;
      const int nbase = nt * BN;
      const int buf = it % NACC;
      const uint32_t par = (uint32_t)(it / NACC) & 1u;
      mbar_wait(&tfull[buf], par);
      tc_fence_after();
#pragma unroll 1
      for (int sub = 0; sub < MT; ++sub) {
      const int ow = ((twi * MT + sub) << P.tw_log2) + lw, oh = (thi << P.th_log2) + lh, img = (tni << tn_log2) + ln;
      const bool valid = img < P.nimg && oh < P.cls_oh[cls] && ow < P.cls_ow[cls] && (!R3 || od < P.cls_od[cls]);
      bf16* orow = P.out + P.cls_out_off[cls] + (long long)img * P.out_sn + (long long)oh * P.out_sh +
                   (long long)ow * P.out_sw + (R3 ? (long long)od * P.out_sd : 0LL) + nbase;
      const uint32_t t_addr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * MT + sub) * BN);
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += CH) {
        uint32_t r[32];
        if (CH == 32) tmem_ld_32x32(t_addr + c0, r);
        else tmem_ld_32x16(t_addr + c0, r);
        tmem_ld_wait();
        float v[32];
#pragma unroll
        for (int j = 0; j < CH; ++j) v[j] = __uint_as_float(r[j]) + s_bias[((nbase + c0) & 511) + j];
        if (P.slope) {
          const float a = __ldg(P.slope);
#pragma unroll
          for (int j = 0; j < CH; ++j) v[j] = v[j] > 0.f ? v[j] : a * v[j];
        }
        if (P.res && valid) {
          const bf16* rrow = P.res + P.cls_res_off[cls] + (long long)img * P.res_sn + (long long)oh * P.res_sh +
                             (long long)ow * P.res_sw + (R3 ? (long long)od * P.res_sd : 0LL) + nbase + c0;
#pragma unroll
          for (int j = 0; j < CH / 8; ++j) {
            const uint4 q = *reinterpret_cast<const uint4*>(rrow + j * 8);
            const uint32_t u[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              v[8 * j + 2 * e] += __uint_as_float(u[e] << 16);
              v[8 * j + 2 * e + 1] += __uint_as_float(u[e] & 0xffff0000u);
            }
          }
        }
        uint32_t packed[CH / 2];
#pragma unroll
        for (int j = 0; j < CH / 2; ++j) {
          __nv_bfloat162 h = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
          packed[j] = *reinterpret_cast<uint32_t*>(&h);
          if (P.stats) {  // statistics of the values as stored
            float2 f = __bfloat1622float2(h);
            v[2 * j] = valid ? f.x : 0.f;
            v[2 * j + 1] = valid ? f.y : 0.f;
          }
        }
        if (valid) {
          if (P.wide) {
#pragma unroll
            for (int j = 0; j < CH / 16; ++j)
              st_global_256(orow + c0 + j * 16, packed[8 * j], packed[8 * j + 1], packed[8 * j + 2], packed[8 * j + 3],
                            packed[8 * j + 4], packed[8 * j + 5], packed[8 * j + 6], packed[8 * j + 7]);
          } else {
#pragma unroll
            for (int j = 0; j < CH / 8; ++j)
              *reinterpret_cast<uint4*>(orow + c0 + j * 8) =
                  make_uint4(packed[4 * j], packed[4 * j + 1], packed[4 * j + 2], packed[4 * j + 3]);
          }
        }
        if (P.stats) {
          float sq[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (j >= CH) v[j] = 0.f;
            sq[j] = v[j] * v[j];
          }
          float s1 = warp_transpose_reduce32(v, lane);
          float s2 = warp_transpose_reduce32(sq, lane);
          if (lane < CH) {  // slot owned by (this warp, this lane): fixed accumulation order, run-to-run reproducible
            sl[nbase + c0 + lane] += s1;
            sl[P.n_total + nbase + c0 + lane] += s2;
          }
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[buf]);
    }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (P.stats) {
    for (int i = threadIdx.x; i < 2 * P.n_total; i += blockDim.x) {
      double s = 0.0;
#pragma unroll
      for (int e = 0; e < Epi::EW; ++e) s += (double)s_stats[e * 2 * P.n_total + i];
      if (s != 0.0) atomicAdd(&P.stats[i], s);
    }
  }
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------
// weight gradient:  D_tap[cy(128-block), cx] += sum over 64-pixel tiles  dY^T(tile) * X_tap(tile)
// One pipeline stage = the dY tile (loaded once) + the X tiles of up to TPS taps; the accumulators of a whole
// tap group (<= 512 TMEM columns) stay resident while the CTA walks its share of the pixel tiles.
// ---------------------------------------------------------------------------------------------------------
template <int NX> struct WgB;   // B operand (X tile of one tap): MN-major, swizzle chosen by the row width
template <> struct WgB<16>  { static constexpr int BYTES = 64 * 32,  BOXES = 1, BOXC = 16, LAYOUT = 6, SBO = 256,  KSTEP = 512,  LBO = 256,  TPS = 9; };
template <> struct WgB<32>  { static constexpr int BYTES = 64 * 64,  BOXES = 1, BOXC = 32, LAYOUT = 4, SBO = 512,  KSTEP = 1024, LBO = 512,  TPS = 9; };
template <> struct WgB<64>  { static constexpr int BYTES = 64 * 128, BOXES = 1, BOXC = 64, LAYOUT = 2, SBO = 1024, KSTEP = 2048, LBO = 8192, TPS = 4; };
template <> struct WgB<128> { static constexpr int BYTES = 2 * 8192, BOXES = 2, BOXC = 64, LAYOUT = 2, SBO = 1024, KSTEP = 2048, LBO = 8192, TPS = 2; };
template <> struct WgB<256> { static constexpr int BYTES = 4 * 8192, BOXES = 4, BOXC = 64, LAYOUT = 2, SBO = 1024, KSTEP = 2048, LBO = 8192, TPS = 1; };

template <int NX, bool SMALL_> struct WgCfg {
  using B = WgB<NX>;
  static constexpr int A_BYTES = 2 * 64 * 128;         // two 64-channel column groups x 64 pixels x 128 B
  static constexpr int STAGE_BYTES = A_BYTES + B::TPS * B::BYTES;
  static constexpr int AUX_BYTES = 256;
  static constexpr int MAX_STAGES = (kSmemLimit - 1024 - AUX_BYTES) / STAGE_BYTES;
  // Small-channel (generator) layers: half of TMEM and <= ~100 KB of shared memory per CTA, so that a weight-gradient
  // CTA can share an SM with a CTA of the (independent) data-gradient / BatchNorm chain running on the other stream.
  static constexpr bool SMALL = SMALL_;
  static constexpr int TMEM_COLS = SMALL ? 256 : 512;
  static constexpr int STAGE_CAP = SMALL ? (100 * 1024 / STAGE_BYTES < 2 ? 2 : 100 * 1024 / STAGE_BYTES) : 8;
  static constexpr int STAGES = MAX_STAGES > STAGE_CAP ? STAGE_CAP : MAX_STAGES;
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + AUX_BYTES;
  static constexpr int MAX_TPG = TMEM_COLS / NX;        // taps whose accumulators fit in the TMEM allocation
};

template <int NX, bool SMALL, bool R3>
__global__ void __launch_bounds__(256, 1)
wgrad_kernel(const __grid_constant__ WgradParams P, const __grid_constant__ CUtensorMap tmY,
             const __grid_constant__ ActMaps tmX) {
  using Cfg = WgCfg<NX, SMALL>;
  using B = WgB<NX>;
  constexpr int STAGES = Cfg::STAGES;
  // producer warps: every warp but the MMA issuer for the small-channel layers (issue bound), one for the 128/256-channel
  // layers (measured: more pollers only cost issue slots there); runtime value = barrier arrival count
  const int kWgProducers = P.nprod;
  // No static shared memory in this kernel, so the dynamic window starts at the CTA's (1024-byte aligned) base; using
  // the symbol directly (instead of a manually aligned pointer) lets the compiler emit LDS/STS rather than generic
  // loads and stores for every shared-memory access of the epilogue.
  extern __shared__ __align__(1024) uint8_t smem[];
  if ((smem_u32(smem) & 1023u) != 0) __trap();
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + STAGES * Cfg::STAGE_BYTES);
  uint64_t* empty = full + STAGES;
  uint64_t* tfull = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && elect_one()) {
    prefetch_tmap(&tmY);
    prefetch_tmap(&tmX.m[0]);
  }
  if (warp == 1 && elect_one()) {
    for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], kWgProducers); mbar_init(&empty[i], 1); }
    mbar_init(tfull, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<Cfg::TMEM_COLS>(tmem_slot);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();      // PDL: the on-chip prologue above overlaps the previous kernel
  pdl_launch();

  int b = blockIdx.x;
  const int mb = b % P.m_blocks; b /= P.m_blocks;
  const int grp = b % P.ngroups; b /= P.ngroups;
  const int cxo = (b % P.cx_blocks) * NX; b /= P.cx_blocks;   // first X channel of this CTA's block
  const int split = b;
  const int tap0 = grp * P.taps_per_group;
  const int ntap = min(P.taps_per_group, P.ntaps - tap0);
  const int ptiles = P.tiles_n * (R3 ? P.tiles_d : 1) * P.tiles_h * P.tiles_w;
  const int tn_log2 = 6 - P.tw_log2 - P.th_log2 - (R3 ? P.td_log2 : 0);
  const int my_tiles = split < ptiles ? (ptiles - split + P.splits - 1) / P.splits : 0;
  // pixel tile pt -> tile origin (w0, h0, d0, n0)
  auto tile_origin = [&](int pt, int& w0, int& h0, int& d0, int& n0) {
    int t = pt;
    const int twi = t % P.tiles_w; t /= P.tiles_w;
    const int thi = t % P.tiles_h; t /= P.tiles_h;
    int tdi = 0;
    if constexpr (R3) { tdi = t % P.tiles_d; t /= P.tiles_d; }
    w0 = twi << P.tw_log2; h0 = thi << P.th_log2; d0 = tdi << P.td_log2; n0 = t << tn_log2;
  };
  // one box of a 64-pixel tile: channels [c0, c0 + box) of map m at pixel offset (dw, dh, dd) from the tile origin
  auto load_tile = [&](void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int w, int h, int d, int n) {
    if constexpr (R3) tma_load_5d(dst, m, bar, c0, w, h, d, n);
    else tma_load_4d(dst, m, bar, c0, w, h, n);
  };

  if (kWgProducers == 1) {
  if (warp == 0) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = split; pt < ptiles; pt += P.splits) {
        int w0, h0, d0, n0;
        tile_origin(pt, w0, h0, d0, n0);
        for (int tl0 = 0; tl0 < ntap; tl0 += B::TPS) {
          const int nt = min(B::TPS, ntap - tl0);
          mbar_wait(&empty[stage], phase ^ 1);
          uint8_t* sA = smem + stage * Cfg::STAGE_BYTES;
          uint8_t* sB = sA + Cfg::A_BYTES;
          mbar_expect_tx(&full[stage], Cfg::A_BYTES + nt * B::BYTES);
          load_tile(sA, &tmY, &full[stage], mb * 128, w0, h0, d0, n0);
          load_tile(sA + 8192, &tmY, &full[stage], mb * 128 + 64, w0, h0, d0, n0);
          for (int q = 0; q < nt; ++q) {
            const int tap = tap0 + tl0 + q;
            const CUtensorMap* mX = &tmX.m[P.tap_map[tap]];
#pragma unroll
            for (int i = 0; i < B::BOXES; ++i)
              load_tile(sB + q * B::BYTES + i * 8192, mX, &full[stage], cxo + i * 64, w0 + P.tap_dw[tap], h0 + P.tap_dh[tap],
                        d0 + P.tap_dd[tap], n0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  }
  } else {
  if (warp != 1) {
    // TMA producers: SEVEN warps (every warp but the MMA issuer; the epilogue warps have nothing else to do until
    // the last tile).  One issuing thread needs ~130 cycles per TMA instruction, and a stage of the 16/32-channel
    // layers is 11 of them (dY tile in two boxes + nine tap tiles of X) for only 4 MMAs -- the loads of a stage are
    // dealt round-robin to the producers, each posting its own byte count on the stage's barrier.
    const int pw = warp == 0 ? 0 : warp - 1;          // producer index 0..6
    if (pw < kWgProducers && elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int pt = split; pt < ptiles; pt += P.splits) {
        int w0, h0, d0, n0;
        tile_origin(pt, w0, h0, d0, n0);
        for (int tl0 = 0; tl0 < ntap; tl0 += B::TPS) {
          const int nt = min(B::TPS, ntap - tl0);
          const int items = 2 + nt * B::BOXES;          // item 0,1: dY boxes; 2 + q*BOXES + i: box i of tap q
          uint8_t* sA = smem + stage * Cfg::STAGE_BYTES;
          uint8_t* sB = sA + Cfg::A_BYTES;
          mbar_wait(&empty[stage], phase ^ 1);
          uint32_t bytes = 0;
          for (int it = pw; it < items; it += kWgProducers) bytes += it < 2 ? 8192u : (uint32_t)(B::BYTES / B::BOXES);
          if (bytes) mbar_expect_tx(&full[stage], bytes);
          else mbar_arrive(&full[stage]);
          for (int it = pw; it < items; it += kWgProducers) {
            if (it < 2) {
              load_tile(sA + it * 8192, &tmY, &full[stage], mb * 128 + it * 64, w0, h0, d0, n0);
            } else {
              const int q = (it - 2) / B::BOXES, i = (it - 2) % B::BOXES;
              const int tap = tap0 + tl0 + q;
              const CUtensorMap* mX = &tmX.m[P.tap_map[tap]];
              load_tile(sB + q * B::BYTES + i * 8192, mX, &full[stage], cxo + i * 64, w0 + P.tap_dw[tap], h0 + P.tap_dh[tap],
                        d0 + P.tap_dd[tap], n0);
            }
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
    __syncwarp();
  }
  }
  if (warp == 1) {
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int i = 0; i < my_tiles; ++i) {
        for (int tl0 = 0; tl0 < ntap; tl0 += B::TPS) {
          const int nt = min(B::TPS, ntap - tl0);
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::STAGE_BYTES);
          const uint32_t b_addr = a_addr + Cfg::A_BYTES;
          // The tap tiles of a stage are contiguous in shared memory and their accumulators are adjacent TMEM
          // columns, so up to 256/NX taps are ONE MMA with N = taps*NX: the cost of an MMA is dominated by the fetch
          // of its 128 A rows (the dY tile, shared by all taps), not by N.
          constexpr int TPM = (256 / NX) < B::TPS ? (256 / NX) : B::TPS;   // taps per MMA
          constexpr uint32_t LBO_N = NX >= 64 ? (uint32_t)B::LBO : (uint32_t)B::BYTES;   // stride between N atoms
          for (int q = 0; q < nt; q += TPM) {
            const int ntm = min(TPM, nt - q);
            const uint32_t idesc_q = make_idesc_bf16(128, ntm * NX, 1, 1);
            const uint32_t d_tmem = tmem_base + (uint32_t)((tl0 + q) * NX);
#pragma unroll
            for (int k = 0; k < 4; ++k) {  // 64 pixels = 4 x K16
              const uint64_t adesc = make_smem_desc(a_addr + k * 2048, 8192, 1024, 2);
              const uint64_t bdesc = make_smem_desc(b_addr + q * B::BYTES + k * B::KSTEP, LBO_N, B::SBO, B::LAYOUT);
              umma_bf16(d_tmem, adesc, bdesc, idesc_q, (i | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit(&empty[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1; }
        }
      }
      umma_commit(tfull);
    }
  } else if (warp >= 4 && my_tiles > 0) {
    const int q = warp - 4;
    const int m = mb * 128 + q * 32 + lane;
    mbar_wait(tfull, 0);
    tc_fence_after();
    for (int tl = 0; tl < ntap; ++tl) {
      const int tap = tap0 + tl;
      float* drow = P.dw + ((long long)m * P.ntaps + tap) * P.cx + cxo;
      constexpr int CH = NX >= 32 ? 32 : 16;
#pragma unroll 1
      for (int c0 = 0; c0 < NX; c0 += CH) {
        uint32_t r[32];
        const uint32_t ta = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(tl * NX + c0);
        if (CH == 32) tmem_ld_32x32(ta, r);
        else tmem_ld_32x16(ta, r);
        tmem_ld_wait();
        if (m < P.cy) {  // 16-byte vector reductions: 4x fewer L2 atomic operations than scalar atomicAdd
#pragma unroll
          for (int j = 0; j < CH; j += 4) red_add_v4(drow + c0 + j, r[j], r[j + 1], r[j + 2], r[j + 3]);
        }
      }
    }
  }
  __syncwarp();
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<Cfg::TMEM_COLS>(tmem_base);
  }
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

static CUtensorMapSwizzle swizzle_for_bytes(int inner_bytes) {
  return inner_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                            : inner_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
}

// bf16 tensor map, `rank` dims (innermost first); strides in elements for dims 1..rank-1
static int encode_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems,
                      const uint32_t* box, bool no_swizzle = false) {
  auto enc = get_encode();
  MPGAN_REQUIRE(enc != nullptr, MPGAN_ERR_CUDA, "cuTensorMapEncodeTiled entry point unavailable (no driver?)");
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i < rank - 1; ++i) gstr[i] = strides_elems[i] * 2;
  MPGAN_REQUIRE(((uintptr_t)base & 15) == 0, MPGAN_ERR_SHAPE, "tensor base not 16-byte aligned");
  for (int i = 0; i < rank - 1; ++i)
    MPGAN_REQUIRE(gstr[i] % 16 == 0, MPGAN_ERR_SHAPE, "tensor stride %d (=%llu B) not a multiple of 16 B", i,
                  (unsigned long long)gstr[i]);
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, no_swizzle ? CU_TENSOR_MAP_SWIZZLE_NONE : swizzle_for_bytes((int)box[0] * 2),
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  MPGAN_REQUIRE(r == CUDA_SUCCESS, MPGAN_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

// Convolution geometry in (depth, height, width); rank 2 = depth extent / kernel 1, depth padding 0.
struct Geom2 {
  int rank, n, xd, xh, xw, yd, yh, yw, cx, cy, kd, kh, kw, s, pd, ph, pw;
};

static int to_geom2(const MpganConvGeom* g, Geom2* o) {
  MPGAN_REQUIRE(g && (g->rank == 2 || g->rank == 3), MPGAN_ERR_UNSUPPORTED, "tcgen05 conv path is rank 2 or 3");
  MPGAN_REQUIRE(g->stride[1] == g->stride[2] && (g->stride[1] == 1 || g->stride[1] == 2), MPGAN_ERR_UNSUPPORTED,
                "tcgen05 conv path supports stride 1 or 2");
  o->rank = g->rank; o->n = g->n;
  o->xd = g->xs[0]; o->xh = g->xs[1]; o->xw = g->xs[2]; o->yd = g->ys[0]; o->yh = g->ys[1]; o->yw = g->ys[2];
  o->cx = g->cx; o->cy = g->cy; o->kd = g->k[0]; o->kh = g->k[1]; o->kw = g->k[2]; o->s = g->stride[1];
  o->pd = g->pad[0]; o->ph = g->pad[1]; o->pw = g->pad[2];
  if (g->rank == 2) {
    MPGAN_REQUIRE(o->xd == 1 && o->yd == 1 && o->kd == 1 && o->pd == 0, MPGAN_ERR_SHAPE, "rank-2 geometry with a depth extent");
  } else {
    MPGAN_REQUIRE(g->stride[0] == g->stride[1], MPGAN_ERR_UNSUPPORTED, "tcgen05 conv path needs equal strides");
    MPGAN_REQUIRE(o->yd <= (o->xd + 2 * o->pd - o->kd) / o->s + 1, MPGAN_ERR_SHAPE, "Y extent exceeds conv output size");
  }
  MPGAN_REQUIRE(o->kd * o->kh * o->kw <= MAXT, MPGAN_ERR_UNSUPPORTED, "too many taps");
  MPGAN_REQUIRE(o->cx % 16 == 0 && o->cy % 16 == 0, MPGAN_ERR_UNSUPPORTED, "channels must be multiples of 16");
  MPGAN_REQUIRE(o->yh <= (o->xh + 2 * o->ph - o->kh) / o->s + 1 && o->yw <= (o->xw + 2 * o->pw - o->kw) / o->s + 1,
                MPGAN_ERR_SHAPE, "Y extent exceeds conv output size");
  return 0;
}

static inline int floordiv(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }
static inline int ilog2(int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// choose a tw x th x td x tn = npix tile minimising padded work (td > 1 only for rank-3 tensors)
static void choose_tile(int ow, int oh, int od, int nimg, int npix, bool r3, int* tw_log2, int* th_log2, int* td_log2) {
  double best = 1e300;
  int bl = 0, bh = 0, bd = 0;
  for (int lw = 0; lw <= 5; ++lw)
    for (int lh = 0; lh <= 5; ++lh)
      for (int ld = 0; ld <= (r3 ? 4 : 0); ++ld) {
        int ln = ilog2(npix) - lw - lh - ld;
        if (ln < 0 || ln > 4) continue;
        int tw = 1 << lw, th = 1 << lh, td = 1 << ld, tn = 1 << ln;
        double work = (double)((ow + tw - 1) / tw * tw) * ((oh + th - 1) / th * th) * ((od + td - 1) / td * td) *
                      ((nimg + tn - 1) / tn * tn);
        work *= 1.0 + 0.02 * ln + 0.01 * (5 - lw) + 0.005 * ld;  // mild preference for wide single-image, single-slice tiles
        if (work < best) { best = work; bl = lw; bh = lh; bd = ld; }
      }
  *tw_log2 = bl;
  *th_log2 = bh;
  *td_log2 = bd;
}

// tensor maps over the gathered activation tensor (spatial d x h x w, channels c, pixel stride ld):
// stride 1 -> one map; stride 2 -> one map per parity class, index (pd * 2 + ph) * 2 + pw (pd = 0 for rank 2).
// box: {channels, tw, th, [td,] tn}
static int make_act_maps(ActMaps* maps, const void* base, bool r3, int nimg, int d, int h, int w, int c, int64_t ld, int s,
                         const uint32_t* box) {
  const bf16* b = (const bf16*)base;
  const int rank = r3 ? 5 : 4;
  memset(maps, 0, sizeof(*maps));
  for (int pd = 0; pd < (r3 && s == 2 ? 2 : 1); ++pd)
    for (int ph = 0; ph < s; ++ph)
      for (int pw = 0; pw < s; ++pw) {
        int dd = (d - pd + s - 1) / s, hh = (h - ph + s - 1) / s, ww = (w - pw + s - 1) / s;
        if (!r3) dd = 1;
        if (dd < 1) dd = 1;
        if (hh < 1) hh = 1;
        if (ww < 1) ww = 1;
        const bf16* origin = b + (((int64_t)pd * h + ph) * w + pw) * ld;
        int rc;
        if (r3) {
          uint64_t dims[5] = {(uint64_t)c, (uint64_t)ww, (uint64_t)hh, (uint64_t)dd, (uint64_t)nimg};
          uint64_t str[4] = {(uint64_t)ld * s, (uint64_t)ld * w * s, (uint64_t)ld * w * h * s, (uint64_t)ld * w * h * d};
          rc = encode_map(&maps->m[(pd * 2 + ph) * 2 + pw], origin, rank, dims, str, box);
        } else {
          uint64_t dims[4] = {(uint64_t)c, (uint64_t)ww, (uint64_t)hh, (uint64_t)nimg};
          uint64_t str[3] = {(uint64_t)ld * s, (uint64_t)ld * w * s, (uint64_t)ld * w * h};
          rc = encode_map(&maps->m[ph * 2 + pw], origin, rank, dims, str, box);
        }
        if (rc) return rc;
      }
  if (s == 1)
    for (int i = 1; i < 8; ++i) maps->m[i] = maps->m[0];
  return 0;
}

template <int BN, int KC, int MT, bool R3>
static int launch_tapgemm_t(const TapGemmParams& P, const ActMaps& mA, const CUtensorMap& mB, cudaStream_t s) {
  using Cfg = TapCfg<BN, KC, MT>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(tapgemm_kernel<BN, KC, MT, R3>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         Cfg::SMEM_BYTES);
    MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaFuncSetAttribute(tapgemm): %s", cudaGetErrorString(e));
    attr_done = true;
  }
  const long long total = (long long)P.ncls * P.tiles_n * P.tiles_d * P.tiles_h * P.tiles_w * P.n_tiles;
  int grid = (int)(total < num_sms() ? total : num_sms());
  int max_taps = 0;
  for (int c = 0; c < P.ncls; ++c) max_taps = std::max(max_taps, P.cls_tap_begin[c + 1] - P.cls_tap_begin[c]);
  TapGemmParams Q = P;
  {
    // stride-2 data gradients sweep dY once per parity class; with equal tap counts (4x4 kernels) the four classes of a
    // spatial tile are made consecutive so that the dY region is re-read from L2 instead of HBM (D3: dY is 256 MB)
    bool equal = P.ncls > 1;
    for (int c = 1; c < P.ncls; ++c)
      equal = equal && (P.cls_tap_begin[c + 1] - P.cls_tap_begin[c] == P.cls_tap_begin[1] - P.cls_tap_begin[0]);
    static int off = -1;
    if (off < 0) { const char* e = getenv("MPGAN_NO_CLS_MINOR"); off = (e && e[0] == '1') ? 1 : 0; }
    Q.cls_minor = (equal && !off) ? 1 : 0;
  }
  Q.lane_parallel = (max_taps * P.nkc <= Cfg::STAGES && max_taps <= 32) ? 1 : 0;
  launch_k(tapgemm_kernel<BN, KC, MT, R3>, grid, EpiCfg<BN>::THREADS, Cfg::SMEM_BYTES, s, Q, mA, mB);
  MPGAN_CHECK_LAUNCH("tapgemm_kernel");
  return 0;
}

template <int KC, bool R3>
static int launch_tapgemm_kc(int bn, const TapGemmParams& P, const ActMaps& mA, const CUtensorMap& mB, cudaStream_t s) {
  switch (bn) {
    case 16: return launch_tapgemm_t<16, KC, 1, R3>(P, mA, mB, s);
    case 32: return launch_tapgemm_t<32, KC, 1, R3>(P, mA, mB, s);
    case 64: return launch_tapgemm_t<64, KC, 1, R3>(P, mA, mB, s);
    case 128:
      if constexpr (KC == 64) {
        if (P.mt == 2) return launch_tapgemm_t<128, KC, 2, R3>(P, mA, mB, s);
      }
      return launch_tapgemm_t<128, KC, 1, R3>(P, mA, mB, s);
    case 256: return launch_tapgemm_t<256, KC, 1, R3>(P, mA, mB, s);
  }
  set_error("bad BN %d", bn);
  return MPGAN_ERR_UNSUPPORTED;
}

static int pick_bn(int n) {
  const int cands[5] = {256, 128, 64, 32, 16};
  for (int i = 0; i < 5; ++i)
    if (n % cands[i] == 0) return cands[i];
  return 0;
}

}  // namespace tc
}  // namespace mpgan
// stride-1 3x3 layers with resident weights and one halo load per tile (halo3x3_run returns 1 = not covered)
#include "conv_halo.cuh"
// one-input-channel forward convolutions (im2col tile built in shared memory, one MMA per tile)
#include "conv_c1mma.cuh"
// stride-2 3x3 layers (down-sampling convolutions, transposed convolutions and their data gradients)
#include "conv_s2.cuh"
// weight gradients of the 16 / 32-input-channel 3x3 layers (one X halo box per tile)
#include "conv_wgrad_halo.cuh"
namespace mpgan {
namespace tc {

static bool halo_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("MPGAN_NO_HALO"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}

// common driver for fprop (dir 0) and bprop (dir 1)
static int run_tapgemm(const Geom2& g, int dir, const void* in, int64_t ldi, const void* w, const float* bias, void* out,
                       int64_t ldo, double* stats, cudaStream_t s, const void* res = nullptr, int64_t ldres = 0,
                       const float* slope = nullptr) {
  const bool r3 = g.rank == 3;
  const int C = dir == 0 ? g.cx : g.cy;  // reduced channels
  const int N = dir == 0 ? g.cy : g.cx;  // produced channels
  const int id = dir == 0 ? g.xd : g.yd, ih = dir == 0 ? g.xh : g.yh, iw = dir == 0 ? g.xw : g.yw;
  const int od = dir == 0 ? g.yd : g.xd, oh = dir == 0 ? g.yh : g.xh, ow = dir == 0 ? g.yw : g.xw;
  if (!r3 && g.s == 1 && g.kh == 3 && g.kw == 3 && g.ph == g.pw && g.ph <= 1 && halo_enabled()) {
    int rc = halo3x3_run(dir, g.n, ih, iw, oh, ow, C, N, g.ph, in, ldi, w, bias, out, ldo, stats, res, ldres, s, 0, slope);
    if (rc != 1) return rc;
  }
  if (!r3 && g.s == 2 && g.kh == 3 && g.kw == 3 && g.ph == 1 && g.pw == 1) {
    int rc = halo_s2_run(dir, g.n, g.xh, g.xw, g.yh, g.yw, C, N, in, ldi, w, bias, out, ldo, stats, res, ldres, s, slope);
    if (rc != 1) return rc;
  }
  const int KC = C % 64 == 0 ? 64 : (C % 32 == 0 ? 32 : 16);
  const int BN = pick_bn(N);
  MPGAN_REQUIRE(BN > 0, MPGAN_ERR_UNSUPPORTED, "N=%d not tileable", N);
  MPGAN_REQUIRE(ldi % 8 == 0 && ldo % 8 == 0, MPGAN_ERR_SHAPE, "pixel strides must be multiples of 8 elements");
  MPGAN_REQUIRE(((uintptr_t)out & 15) == 0, MPGAN_ERR_SHAPE, "output not 16-byte aligned");

  TapGemmParams P;
  memset(&P, 0, sizeof(P));
  P.nkc = C / KC;
  P.nimg = g.n;
  P.n_total = N;
  P.n_tiles = N / BN;
  P.out = (bf16*)out;
  P.bias = bias;
  P.stats = stats;
  P.wide = (ldo % 16 == 0 && ((uintptr_t)out & 31) == 0) ? 1 : 0;
  P.slope = slope;
  P.res = (const bf16*)res;
  MPGAN_REQUIRE(!res || (ldres % 8 == 0 && ((uintptr_t)res & 15) == 0), MPGAN_ERR_SHAPE, "residual tensor misaligned");
  MPGAN_REQUIRE(N <= 512 || (!bias && !stats), MPGAN_ERR_UNSUPPORTED, "N > 512 is supported without bias / statistics only");

  const int sd = r3 ? g.s : 1;            // stride along depth (rank 2: a single depth slice)
  int ntap = 0;
  int lod, loh, low;  // logical output grid the tiles cover
  if (dir == 0) {  // gather X: xpos = ypos*s - pad + r
    P.ncls = 1;
    P.cls_tap_begin[0] = 0;
    for (int rd = 0; rd < g.kd; ++rd)
      for (int rh = 0; rh < g.kh; ++rh)
        for (int rw = 0; rw < g.kw; ++rw) {
          int qd = rd - g.pd, qh = rh - g.ph, qw = rw - g.pw;
          int pd = sd == 2 ? ((qd % 2) + 2) % 2 : 0;
          int ph = g.s == 2 ? ((qh % 2) + 2) % 2 : 0, pw = g.s == 2 ? ((qw % 2) + 2) % 2 : 0;
          // a parity plane the input does not have (extent 1 along a stride-2 axis): every read of this tap is
          // padding.  make_act_maps clamps that plane's map to one element, which would read the next image: skip it.
          if ((sd == 2 && (id - pd + 1) / 2 < 1) || (g.s == 2 && ((ih - ph + 1) / 2 < 1 || (iw - pw + 1) / 2 < 1))) continue;
          P.tap_map[ntap] = (signed char)((pd * 2 + ph) * 2 + pw);
          P.tap_dd[ntap] = (short)(sd == 2 ? floordiv(qd - pd, 2) : qd);
          P.tap_dh[ntap] = (short)(g.s == 2 ? floordiv(qh - ph, 2) : qh);
          P.tap_dw[ntap] = (short)(g.s == 2 ? floordiv(qw - pw, 2) : qw);
          P.tap_slab[ntap] = (short)((rd * g.kh + rh) * g.kw + rw);
          ++ntap;
        }
    P.cls_tap_begin[1] = ntap;
    P.cls_od[0] = od; P.cls_oh[0] = oh; P.cls_ow[0] = ow; P.cls_out_off[0] = 0; P.cls_res_off[0] = 0;
    P.out_sn = (long long)od * oh * ow * ldo; P.out_sd = (long long)oh * ow * ldo; P.out_sh = (long long)ow * ldo; P.out_sw = ldo;
    P.res_sn = (long long)od * oh * ow * ldres; P.res_sd = (long long)oh * ow * ldres; P.res_sh = (long long)ow * ldres; P.res_sw = ldres;
    lod = od; loh = oh; low = ow;
  } else {  // gather Y: ypos = (xpos + pad - r)/s
    P.ncls = sd * g.s * g.s;
    for (int cpd = 0; cpd < sd; ++cpd)
      for (int cph = 0; cph < g.s; ++cph)
        for (int cpw = 0; cpw < g.s; ++cpw) {
          int cls = (cpd * g.s + cph) * g.s + cpw;
          P.cls_tap_begin[cls] = ntap;
          for (int rd = 0; rd < g.kd; ++rd)
            for (int rh = 0; rh < g.kh; ++rh)
              for (int rw = 0; rw < g.kw; ++rw) {
                int ad = cpd + g.pd - rd, ah = cph + g.ph - rh, aw = cpw + g.pw - rw;
                if (g.s == 2 && ((ah & 1) || (aw & 1))) continue;
                if (sd == 2 && (ad & 1)) continue;
                P.tap_map[ntap] = 0;
                P.tap_dd[ntap] = (short)(sd == 2 ? ad / 2 : ad);   // even here, exact
                P.tap_dh[ntap] = (short)(g.s == 2 ? ah / 2 : ah);
                P.tap_dw[ntap] = (short)(g.s == 2 ? aw / 2 : aw);
                P.tap_slab[ntap] = (short)((rd * g.kh + rh) * g.kw + rw);
                ++ntap;
              }
          MPGAN_REQUIRE(ntap > P.cls_tap_begin[cls], MPGAN_ERR_UNSUPPORTED, "empty tap class (k < stride)");
          P.cls_od[cls] = (od - cpd + sd - 1) / sd;
          P.cls_oh[cls] = (oh - cph + g.s - 1) / g.s;
          P.cls_ow[cls] = (ow - cpw + g.s - 1) / g.s;
          P.cls_out_off[cls] = (((long long)cpd * oh + cph) * ow + cpw) * ldo;
          P.cls_res_off[cls] = (((long long)cpd * oh + cph) * ow + cpw) * ldres;
        }
    P.cls_tap_begin[P.ncls] = ntap;
    P.out_sn = (long long)od * oh * ow * ldo; P.out_sd = (long long)oh * ow * ldo * sd;
    P.out_sh = (long long)ow * ldo * g.s; P.out_sw = ldo * g.s;
    P.res_sn = (long long)od * oh * ow * ldres; P.res_sd = (long long)oh * ow * ldres * sd;
    P.res_sh = (long long)ow * ldres * g.s; P.res_sw = ldres * g.s;
    lod = (od + sd - 1) / sd; loh = (oh + g.s - 1) / g.s; low = (ow + g.s - 1) / g.s;
  }
  choose_tile(low, loh, lod, g.n, 128, r3, &P.tw_log2, &P.th_log2, &P.td_log2);
  const int tw = 1 << P.tw_log2, th = 1 << P.th_log2, td = 1 << P.td_log2, tn = 128 / (tw * th * td);
  P.tiles_w = (low + tw - 1) / tw; P.tiles_h = (loh + th - 1) / th; P.tiles_d = (lod + td - 1) / td;
  P.tiles_n = (g.n + tn - 1) / tn;
  // two tiles per weight stage only when the layer still has several supertiles per SM (D layer 3 data gradient)
  P.mt = (BN == 128 && KC == 64 &&
          (long long)P.ncls * P.tiles_w * P.tiles_h * P.tiles_d * P.tiles_n * P.n_tiles >= 8LL * num_sms()) ? 2 : 1;
  P.tiles_w = (P.tiles_w + P.mt - 1) / P.mt;

  ActMaps mA;
  CUtensorMap mB;
  uint32_t boxA[5] = {(uint32_t)KC, (uint32_t)tw, (uint32_t)th, (uint32_t)(r3 ? td : tn), (uint32_t)tn};
  int rc = make_act_maps(&mA, in, r3, g.n, id, ih, iw, C, ldi, dir == 0 ? g.s : 1, boxA);
  if (rc) return rc;
  {
    const int T = g.kd * g.kh * g.kw;
    uint64_t dims[3] = {(uint64_t)C, (uint64_t)T, (uint64_t)N};
    uint64_t str[2] = {(uint64_t)C, (uint64_t)C * T};
    uint32_t box[3] = {(uint32_t)KC, 1u, (uint32_t)BN};
    rc = encode_map(&mB, w, 3, dims, str, box);
    if (rc) return rc;
  }
  if (r3) {
    switch (KC) {
      case 64: return launch_tapgemm_kc<64, true>(BN, P, mA, mB, s);
      case 32: return launch_tapgemm_kc<32, true>(BN, P, mA, mB, s);
      default: return launch_tapgemm_kc<16, true>(BN, P, mA, mB, s);
    }
  }
  switch (KC) {
    case 64: return launch_tapgemm_kc<64, false>(BN, P, mA, mB, s);
    case 32: return launch_tapgemm_kc<32, false>(BN, P, mA, mB, s);
    default: return launch_tapgemm_kc<16, false>(BN, P, mA, mB, s);
  }
}

template <int NX, bool SMALL, bool R3>
static int launch_wgrad_t(const WgradParams& P, const CUtensorMap& mY, const ActMaps& mX, cudaStream_t s) {
  using Cfg = WgCfg<NX, SMALL>;
  static bool attr_done = false;
  if (!attr_done) {
    cudaError_t e = cudaFuncSetAttribute(wgrad_kernel<NX, SMALL, R3>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES);
    MPGAN_REQUIRE(e == cudaSuccess, MPGAN_ERR_CUDA, "cudaFuncSetAttribute(wgrad): %s", cudaGetErrorString(e));
    attr_done = true;
  }
  int grid = P.m_blocks * P.ngroups * P.cx_blocks * P.splits;
  launch_k(wgrad_kernel<NX, SMALL, R3>, grid, 256, Cfg::SMEM_BYTES, s, P, mY, mX);
  MPGAN_CHECK_LAUNCH("wgrad_kernel");
  return 0;
}

template <bool R3>
static int dispatch_wgrad(int cx, bool small, const WgradParams& P, const CUtensorMap& mY, const ActMaps& mX, cudaStream_t s) {
  switch (cx) {
    case 16: return small ? launch_wgrad_t<16, true, R3>(P, mY, mX, s) : launch_wgrad_t<16, false, R3>(P, mY, mX, s);
    case 32: return small ? launch_wgrad_t<32, true, R3>(P, mY, mX, s) : launch_wgrad_t<32, false, R3>(P, mY, mX, s);
    case 64: return small ? launch_wgrad_t<64, true, R3>(P, mY, mX, s) : launch_wgrad_t<64, false, R3>(P, mY, mX, s);
    case 128: return launch_wgrad_t<128, false, R3>(P, mY, mX, s);
    default: return launch_wgrad_t<256, false, R3>(P, mY, mX, s);
  }
}

static int run_wgrad(const Geom2& g, const void* x, int64_t ldx, const void* y, int64_t ldy, float* dw, cudaStream_t s) {
  MPGAN_REQUIRE(g.cx == 16 || g.cx == 32 || g.cx == 64 || g.cx == 128 || (g.cx >= 256 && g.cx % 256 == 0), MPGAN_ERR_UNSUPPORTED,
                "tc wgrad needs cx in {16,32,64,128} or a multiple of 256");
  MPGAN_REQUIRE(ldx % 8 == 0 && ldy % 8 == 0, MPGAN_ERR_SHAPE, "pixel strides must be multiples of 8 elements");
  const bool r3 = g.rank == 3;
  const int sd = r3 ? g.s : 1;
  if (!r3 && g.kh == 3 && g.kw == 3 && g.ph == g.pw) {
    int rc = wgrad_halo_run(g.s, g.ph, g.n, g.xh, g.xw, g.yh, g.yw, g.cx, g.cy, x, ldx, y, ldy, dw, s);
    if (rc != 1) return rc;
  }
  WgradParams P;
  memset(&P, 0, sizeof(P));
  P.cx = g.cx; P.cy = g.cy; P.dw = dw;
  const int nx = g.cx > 256 ? 256 : g.cx;       // X channels per CTA
  P.cx_blocks = g.cx / nx;
  {
    static int forced = -1;
    if (forced < 0) { const char* e = getenv("MPGAN_WG_NPROD"); forced = e ? atoi(e) : 0; }
    P.nprod = g.cx <= 64 ? 7 : 1;
    if (forced >= 1 && forced <= 7) P.nprod = forced;
  }
  int ntap = 0;
  for (int rd = 0; rd < g.kd; ++rd)
    for (int rh = 0; rh < g.kh; ++rh)
      for (int rw = 0; rw < g.kw; ++rw) {
        int qd = rd - g.pd, qh = rh - g.ph, qw = rw - g.pw;
        int pd = sd == 2 ? ((qd % 2) + 2) % 2 : 0;
        int ph = g.s == 2 ? ((qh % 2) + 2) % 2 : 0, pw = g.s == 2 ? ((qw % 2) + 2) % 2 : 0;
        P.tap_map[ntap] = (signed char)((pd * 2 + ph) * 2 + pw);
        P.tap_dd[ntap] = (short)(sd == 2 ? floordiv(qd - pd, 2) : qd);
        P.tap_dh[ntap] = (short)(g.s == 2 ? floordiv(qh - ph, 2) : qh);
        P.tap_dw[ntap] = (short)(g.s == 2 ? floordiv(qw - pw, 2) : qw);
        ++ntap;
      }
  P.ntaps = ntap;
  // "small" = generator-sized layer (<= 1M output pixels): half of TMEM / ~100 KB of shared memory per CTA so that a
  // CTA of the concurrent data-gradient chain fits on the same SM; large layers (D) take the whole SM
  const bool small = g.cx <= 64 && (long long)g.n * g.yd * g.yh * g.yw <= (1LL << 20);
  const int max_tpg = (small ? 256 : 512) / nx;
  P.ngroups = (ntap + max_tpg - 1) / max_tpg;
  // EQUAL groups when a slightly finer split allows it: the CTAs of the different groups of one pixel range walk the same
  // dY / X tiles side by side; with 5 + 4 taps (D layer 2: 9 taps, 8 accumulators fit) the lighter group ran ahead by more
  // than the L2 holds and every tile came from DRAM twice (ncu: 1461 MB read for 785 MB of operands)
  for (int gcount = P.ngroups; gcount <= P.ngroups + 2 && gcount <= ntap; ++gcount)
    if (ntap % gcount == 0) { P.ngroups = gcount; break; }
  P.taps_per_group = (ntap + P.ngroups - 1) / P.ngroups;   // balanced groups
  P.m_blocks = (g.cy + 127) / 128;
  choose_tile(g.yw, g.yh, g.yd, g.n, 64, r3, &P.tw_log2, &P.th_log2, &P.td_log2);
  const int tw = 1 << P.tw_log2, th = 1 << P.th_log2, td = 1 << P.td_log2, tn = 64 / (tw * th * td);
  P.tiles_w = (g.yw + tw - 1) / tw; P.tiles_h = (g.yh + th - 1) / th; P.tiles_d = (g.yd + td - 1) / td;
  P.tiles_n = (g.n + tn - 1) / tn;
  const int ptiles = P.tiles_w * P.tiles_h * P.tiles_d * P.tiles_n;
  const int items = P.m_blocks * P.ngroups * P.cx_blocks;
  // one CTA per SM for the large-channel configurations (~200 KB of shared memory each): the grid must not exceed the
  // SM count or the few extra CTAs run as a second wave and double the kernel time (152 CTAs did, on 148 SMs)
  int splits = !small ? num_sms() / items : (num_sms() + items - 1) / items;
  if (splits > ptiles) splits = ptiles;
  if (splits < 1) splits = 1;
  P.splits = splits;

  CUtensorMap mY;
  ActMaps mX;
  if (r3) {
    uint64_t dims[5] = {(uint64_t)g.cy, (uint64_t)g.yw, (uint64_t)g.yh, (uint64_t)g.yd, (uint64_t)g.n};
    uint64_t str[4] = {(uint64_t)ldy, (uint64_t)ldy * g.yw, (uint64_t)ldy * g.yw * g.yh, (uint64_t)ldy * g.yw * g.yh * g.yd};
    uint32_t box[5] = {64u, (uint32_t)tw, (uint32_t)th, (uint32_t)td, (uint32_t)tn};
    int rc = encode_map(&mY, y, 5, dims, str, box);
    if (rc) return rc;
  } else {
    uint64_t dims[4] = {(uint64_t)g.cy, (uint64_t)g.yw, (uint64_t)g.yh, (uint64_t)g.n};
    uint64_t str[3] = {(uint64_t)ldy, (uint64_t)ldy * g.yw, (uint64_t)ldy * g.yw * g.yh};
    uint32_t box[4] = {64u, (uint32_t)tw, (uint32_t)th, (uint32_t)tn};
    int rc = encode_map(&mY, y, 4, dims, str, box);
    if (rc) return rc;
  }
  uint32_t boxX[5] = {(uint32_t)(g.cx < 64 ? g.cx : 64), (uint32_t)tw, (uint32_t)th, (uint32_t)(r3 ? td : tn), (uint32_t)tn};
  int rc = make_act_maps(&mX, x, r3, g.n, g.xd, g.xh, g.xw, g.cx, ldx, g.s, boxX);
  if (rc) return rc;
  return r3 ? dispatch_wgrad<true>(nx, small, P, mY, mX, s) : dispatch_wgrad<false>(nx, small, P, mY, mX, s);
}

}  // namespace tc
}  // namespace mpgan

using namespace mpgan;
using namespace mpgan::tc;

extern "C" int mpgan_tc_supported(const MpganConvGeom* g, int direction) {
  Geom2 g2;
  if (to_geom2(g, &g2) != 0) return 0;
  if (direction == 2) return (g2.cx == 16 || g2.cx == 32 || g2.cx == 64 || g2.cx == 128 || (g2.cx >= 256 && g2.cx % 256 == 0)) ? 1 : 0;
  const int N = direction == 0 ? g2.cy : g2.cx;
  if (pick_bn(N) == 0 || N > 512) return 0;   // (wider layers run without bias / statistics only: callers ask explicitly)
  if (direction == 1 && g2.s == 2 && (g2.kh < 2 || g2.kw < 2 || (g2.rank == 3 && g2.kd < 2))) return 0;
  return 1;
}

extern "C" int mpgan_tc_conv_fprop(const MpganConvGeom* g, const void* x, int64_t ldx, const void* w_f,
                                   const float* bias, void* y, int64_t ldy, double* stats, void* stream) {
  Geom2 g2;
  int rc = to_geom2(g, &g2);
  if (rc) return rc;
  return run_tapgemm(g2, 0, x, ldx, w_f, bias, y, ldy, stats, (cudaStream_t)stream);
}

extern "C" int mpgan_tc_conv_bprop(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w_b,
                                   const float* bias, void* x, int64_t ldx, double* stats, void* stream) {
  Geom2 g2;
  int rc = to_geom2(g, &g2);
  if (rc) return rc;
  return run_tapgemm(g2, 1, y, ldy, w_b, bias, x, ldx, stats, (cudaStream_t)stream);
}

extern "C" int mpgan_tc_conv_bprop_res(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w_b,
                                       const float* bias, void* x, int64_t ldx, const void* res, int64_t ldres,
                                       double* stats, void* stream) {
  Geom2 g2;
  int rc = to_geom2(g, &g2);
  if (rc) return rc;
  return run_tapgemm(g2, 1, y, ldy, w_b, bias, x, ldx, stats, (cudaStream_t)stream, res, ldres);
}

// Inference-mode fused layer: y = prelu(conv(x, w_folded) + bias_folded) + res, BatchNorm folded into w / bias by the
// caller (MONAI Convolution / ResidualUnit in eval mode); direction 0 = convolution, 1 = transposed convolution.
extern "C" int mpgan_tc_conv_act(const MpganConvGeom* g, int direction, const void* in, int64_t ldi, const void* w,
                                 const float* bias, const float* slope, const void* res, int64_t ldres, void* out,
                                 int64_t ldo, void* stream) {
  Geom2 g2;
  int rc = to_geom2(g, &g2);
  if (rc) return rc;
  MPGAN_REQUIRE(direction == 0 || direction == 1, MPGAN_ERR_SHAPE, "conv_act: direction 0 (conv) or 1 (transposed conv)");
  return run_tapgemm(g2, direction, in, ldi, w, bias, out, ldo, nullptr, (cudaStream_t)stream, res, ldres, slope);
}

// Data gradient of a ONE-input-channel stride-1 3x3 convolution (D layer 1: dY has 64 channels, dX one): the
// halo-resident kernel with the transposed weights zero-padded to N = 16 output columns, of which only column 0 is
// stored.  w_b16: bf16 [16][9][cy] (row 0 = the layer's transposed weights, rows 1..15 zero).
extern "C" int mpgan_tc_conv_bprop_c1out(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w_b16,
                                         void* x, int64_t ldx, const void* res, int64_t ldres, void* stream) {
  MPGAN_REQUIRE(g && g->rank == 2 && g->cx == 1, MPGAN_ERR_UNSUPPORTED, "bprop_c1out: rank-2 layer with one input channel");
  MPGAN_REQUIRE(g->k[1] == 3 && g->k[2] == 3 && g->stride[1] == 1 && g->stride[2] == 1 && g->pad[1] == g->pad[2] &&
                    g->pad[1] >= 0 && g->pad[1] <= 1,
                MPGAN_ERR_UNSUPPORTED, "bprop_c1out: 3x3, stride 1, pad 0 or 1");
  MPGAN_REQUIRE(g->cy == 16 || g->cy == 32 || g->cy == 64 || g->cy == 128, MPGAN_ERR_UNSUPPORTED,
                "bprop_c1out: cy in {16, 32, 64, 128}");
  MPGAN_REQUIRE(y && w_b16 && x && ldx >= 1, MPGAN_ERR_SHAPE, "bprop_c1out: bad arguments");
  int rc = halo3x3_run(1, g->n, g->ys[1], g->ys[2], g->xs[1], g->xs[2], g->cy, 16, g->pad[1], y, ldy, w_b16, nullptr, x, ldx,
                       nullptr, res, ldres, (cudaStream_t)stream, 1);
  MPGAN_REQUIRE(rc != 1, MPGAN_ERR_UNSUPPORTED, "bprop_c1out: layer not covered by the halo kernel (alignment / size)");
  return rc;
}

// ConvTranspose(C -> 1, k3 s2 p1 op1) forward == data gradient of a one-input-channel stride-2 3x3 convolution: the
// halo kernel in its pixel-shuffle mode (conv_halo.cuh, n_store == 4).  w: the layer's bf16 [C][9] weight;
// x: (n, 2*yh, 2*yw) one channel contiguous; stats (optional): fp64 {sum, sum of squares} of the stored values.
extern "C" int mpgan_tc_convt_to1(const MpganConvGeom* g, const void* y, int64_t ldy, const void* w, const float* bias,
                                  void* x, double* stats, void* stream) {
  MPGAN_REQUIRE(g && g->rank == 2 && g->cx == 1, MPGAN_ERR_UNSUPPORTED, "convt_to1: rank-2 layer with one X channel");
  MPGAN_REQUIRE(g->k[1] == 3 && g->k[2] == 3 && g->stride[1] == 2 && g->stride[2] == 2 && g->pad[1] == 1 && g->pad[2] == 1,
                MPGAN_ERR_UNSUPPORTED, "convt_to1: 3x3, stride 2, pad 1");
  MPGAN_REQUIRE(g->xs[1] == 2 * g->ys[1] && g->xs[2] == 2 * g->ys[2], MPGAN_ERR_UNSUPPORTED, "convt_to1: X = 2 Y only");
  MPGAN_REQUIRE(g->cy == 16 || g->cy == 32 || g->cy == 64, MPGAN_ERR_UNSUPPORTED, "convt_to1: cy in {16, 32, 64}");
  MPGAN_REQUIRE(y && w && x && ((uintptr_t)x & 3) == 0, MPGAN_ERR_SHAPE, "convt_to1: bad arguments");
  // out strides describe the one-channel OUTPUT image (row pitch 2*yw); the tile grid is the Y grid
  int rc = halo3x3_run(0, g->n, g->ys[1], g->ys[2], g->ys[1], g->ys[2], g->cy, 16, 1, y, ldy, w, bias, x,
                       /*ldo, patched below*/ 1, stats, nullptr, 0, (cudaStream_t)stream, 4);
  MPGAN_REQUIRE(rc != 1, MPGAN_ERR_UNSUPPORTED, "convt_to1: layer not covered by the halo kernel (alignment / size)");
  return rc;
}

extern "C" size_t mpgan_tc_conv_wgrad_workspace(const MpganConvGeom* g) {
  (void)g;
  return 0;  // split partials are reduced with fp32 atomics straight into dw
}

extern "C" int mpgan_tc_conv_wgrad(const MpganConvGeom* g, const void* x, int64_t ldx, const void* y, int64_t ldy,
                                   float* dw, void* workspace, size_t workspace_bytes, void* stream) {
  (void)workspace; (void)workspace_bytes;
  Geom2 g2;
  int rc = to_geom2(g, &g2);
  if (rc) return rc;
  return run_wgrad(g2, x, ldx, y, ldy, dw, (cudaStream_t)stream);
}

