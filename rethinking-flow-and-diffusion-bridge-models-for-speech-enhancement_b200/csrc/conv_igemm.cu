// Implicit-GEMM convolution for the NCSN++ backbone on Blackwell tensor cores.
//
//   out[b,t,f,n] = scale * ( sum_{dt,df,c} W[n,c,df,dt] * act(in1)[b,t+dt-1,f+df-1,c]   (3x3 or 1x1; act = GroupNorm(+SiLU) on load)
//                            (+ sum_c W2[n,c] * in2[b,t,f,c])                             (fused 1x1 shortcut)
//                            + bias[n] (+ bias_b[b,n]) (+ residual[b,t,f,n]) )
//
// GEMM view: M = pixels, N = Cout, K = taps*C1 (+ C2).  Replaces nn.Conv2d / NIN of
// fdbm/backbones/ncsnpp_utils/layers.py:100-124,546-555 and the adds of layerspp.py:263,270-274.
//
// Design (B200, sm_100a):
//   * activations are 16-bit [B,T,F,C]; one M-tile = 16 frames x 8 bins = 128 pixels = one UMMA M.
//   * per 64-channel K-block ONE TMA box of 18 x 10 pixels (tile + halo, zero-filled outside the
//     image = the convolution's zero padding) lands in shared memory with the 128-byte swizzle; all
//     nine taps are fed from it by shifting the UMMA descriptor start address by (dt*10 + df) pixels
//     (row pitch 10 pixels -> stride-byte-offset 1280).  Validated on hardware by tools/umma_probe.cu.
//     1-tap (shortcut) segments load the 16 x 8 tile without halo.  The K-blocks of up to three segments are
//     walked through a per-launch schedule table.
//   * a CTA owns 2 M-tiles x 128 output channels: every weight tile (128 x 64, TMA, 3-deep ring; 24 slots of
//     16 rows for the narrow C -> 4 convolutions) is used by two MMAs; accumulators live in TMEM
//     (2 stages x 2 tiles x 128 columns = 512).
//   * warp-specialised, persistent, 512 threads: warp0 = A producer, warp1 = B producer, warp2 = MMA issuer,
//     warp3 = TMEM owner, warps4-7 = epilogue of M-tile 0, warps8-11 = operand transform (GroupNorm+SiLU applied to
//     the landed tile in shared memory), warps12-15 = epilogue of M-tile 1.  Epilogue: tcgen05.ld -> smem transpose ->
//     bias / FiLM / 16-bit identity shortcut / scale -> coalesced 16-bit stores + per-channel sum / sum-of-squares for
//     the next GroupNorm, overlapping the next item's main loop through the second accumulator stage.
//     setmaxnreg splits the register file 56 / 120 / 168 / 168 per thread between the four warpgroups.
#include <cuda.h>
#include <mutex>
#include <type_traits>
#include "common.cuh"
#include "tc05.cuh"

namespace fdbm {
int make_act_tile_map(CUtensorMap* map, const op_t* ptr, int B, int T, int F, int C, int box_f, int box_t);
namespace {

using namespace tc05;

constexpr int MT = 2;                       // M-tiles per CTA tile
constexpr int TILE_T = 16, TILE_F = 8;
constexpr int HALO_T = TILE_T + 2, HALO_F = TILE_F + 2;
constexpr int A_TILE_BYTES = HALO_T * HALO_F * 128;          // 23040 bytes landed per TMA box
constexpr int A_TILE_STRIDE = 23552;                         // rounded up to 1024
constexpr int A_STAGES = 3;
constexpr int B_STAGES = 3;
constexpr int BN = 128;
constexpr int B_TILE_BYTES = BN * 128;
constexpr int A_SBO = HALO_F * 128;                          // 1280: distance between 8-pixel row groups
// warps 0-3 pipeline (TMA A, TMA B, MMA issue, TMEM owner), warps 4-7 epilogue of M-tile 0, warps 8-11 operand
// transform, warps 12-15 epilogue of M-tile 1.  One epilogue warpgroup for both tiles was the bottleneck of every
// K <= 1408 layer (13 us of epilogue per 8 us of MMA per item); each tile now has the whole item time.
constexpr int NUM_THREADS = 512;
constexpr int EPI_GROUPS = 2;
constexpr int MAX_SEG = 3;
constexpr int MAX_KB = 16;                                     // K-blocks (64 channels of one segment) per convolution
constexpr int A_TILE1_BYTES = TILE_T * TILE_F * 128;           // 1-tap segments load the tile without halo
// 512 threads start at 128 registers each; setmaxnreg moves registers from the pipeline and transform
// warpgroups to the two epilogue warpgroups (128 * (56 + 120 + 2 * 168) = 65536)
constexpr int PIPE_REGS = 56, EPI_REGS = 168, XFORM_REGS = 120;
constexpr int STAGE_BYTES = EPI_GROUPS * 4 * 32 * 32 * 4;       // epilogue transposition tiles, one per warp
constexpr int STAT_SLOTS = 2;                                  // n-blocks whose statistics a CTA keeps in flight
constexpr int STAT_BYTES = EPI_GROUPS * 4 * BN * 8;            // per-warp channel (sum, sum of squares) partials
// no alignment slack: the dynamic segment is declared __align__(1024) and the kernel traps if it is not
// narrow-N (16 output channels) convolutions cut the same weight ring into 2 KB slots: their MMAs per tap are ~10x shorter,
// so three weight loads in flight made them TMA-latency-bound
constexpr int B_STAGES_NARROW = B_STAGES * B_TILE_BYTES / (16 * 128);
constexpr int SMEM_BYTES = A_STAGES * MT * A_TILE_STRIDE + B_STAGES * B_TILE_BYTES + STAGE_BYTES + STAT_BYTES + 512;

// One K segment = one activation tensor contributing C channels (kb = C/64 K-blocks) with 9 taps or 1.
// norm != 0: GroupNorm (+SiLU when act != 0) is applied to the tile in shared memory between the TMA
// landing and the MMA ("normalise on load"); tab[b * tab_stride + c] = (scale, shift) of channel c.
struct SegParams {
  int taps, norm, act, tab_stride;
  int halo;                                // tile loaded with its 1-pixel halo (9 taps, or normalise-on-load which works on the halo box)
  const float2* tab;
};

struct ConvParams {
  int B, T, F, Cout;
  int n_seg, n_kb;
  SegParams seg[MAX_SEG];
  // K-block schedule: entry i = segment | channel block << 4 | first weight tile (kt) << 16
  uint32_t ksched[MAX_KB];
  int tiles_t, tiles_f, n_mtiles, n_nblocks, n_items;
  // ceil(2^32 / d) of the three divisors the persistent loops divide by (every role decodes item -> tile -> (b, t0, f0) per item;
  // the compiler's 32-bit division is ~35 instructions each: 16 % of the epilogue's instructions went there)
  uint32_t mg_tiles_t, mg_tiles_f, mg_nblocks;
  int bn;                                  // MMA N = output channels per item: 128, or 16 for the C -> 4 pyramid convolutions
  // side ring (fused 1x1 shortcut operands): ksched[0 .. n_main) are the main-ring K-blocks, the rest 1-tap blocks without halo
  // that travel through A stage A_STAGES - 1 on their own (the main ring then has A_STAGES - 1 stages); in MMA order one of
  // them follows every side_gap main taps.  n_steps = weight tiles per item.
  int side_ring, n_main, side_gap, n_steps;
  const float* bias;
  const float* bias_b;
  int bias_b_stride;
  const float* residual;
  const op_t* residual_h16;
  float scale;
  float* out_f32;
  op_t* out_h16;
  double* sums;
  float* pyr_out;
  const float* pyr_prev;
  int pyr_C;
  const float* comb_pyr;
  const float* comb_w;
  const float* comb_b;
  int comb_C;
};

struct TileCoord { int b, t0, f0; bool valid; };

// n / d for n * d < 2^32 (host-checked) with mg = ceil(2^32 / d): one IMAD.HI; d == 1 has no 32-bit multiplier
__device__ __forceinline__ int fast_div(int n, int d, uint32_t mg) { return d == 1 ? n : static_cast<int>(__umulhi(static_cast<uint32_t>(n), mg)); }
__device__ __forceinline__ int item_tile(const ConvParams& p, int item) { return fast_div(item, p.n_nblocks, p.mg_nblocks); }
__device__ __forceinline__ int item_nblk(const ConvParams& p, int item) { return item - item_tile(p, item) * p.n_nblocks; }

__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int mi) {
  TileCoord c;
  c.valid = mi < p.n_mtiles;
  const int rest = fast_div(mi, p.tiles_t, p.mg_tiles_t);
  const int tt = mi - rest * p.tiles_t;
  c.t0 = tt * TILE_T;
  c.b = fast_div(rest, p.tiles_f, p.mg_tiles_f);
  c.f0 = (rest - c.b * p.tiles_f) * TILE_F;
  return c;
}

// MMA-order walk over the weight tiles (= steps) of one item when the 1-tap blocks run on the side ring: the main K-blocks tap
// by tap, a side block after every side_gap main taps, what is left of them at the end.  f(side, ksched index, tap, taps of the block).
template <typename F>
__device__ __forceinline__ void walk_steps(const ConvParams& p, F&& f) {
  const int n_side = p.n_kb - p.n_main;
  int sd = 0, cnt = 0;
  for (int m = 0; m < p.n_main; ++m) {
    const int ntaps = p.seg[p.ksched[m] & 15].taps;
    for (int tap = 0; tap < ntaps; ++tap) {
      f(false, m, tap, ntaps);
      if (++cnt == p.side_gap && sd < n_side) { f(true, p.n_main + sd, 0, 1); ++sd; cnt = 0; }
    }
  }
  for (; sd < n_side; ++sd) f(true, p.n_main + sd, 0, 1);
}

// COMB: the epilogue also applies the Combine 1x1 convolution of the input pyramid (kept out of the standard
// instantiation: even as a not-taken branch it doubled the epilogue's time).
// RES16: the identity-shortcut operand is the 16-bit copy of the residual stream (inference plans)
template <bool COMB, bool RES16>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap map_a0, const __grid_constant__ CUtensorMap map_a1,
                  const __grid_constant__ CUtensorMap map_a2, const __grid_constant__ CUtensorMap map_b,
                  const ConvParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  // (offset arithmetic on the __shared__ array itself, so the compiler keeps the shared address space: LDS/STS, not generic LD/ST)
  uint8_t* smem = smem_raw;
  if (smem_u32(smem_raw) & 1023u) __trap();
  uint8_t* sA = smem;
  uint8_t* sB = smem + A_STAGES * MT * A_TILE_STRIDE;
  uint8_t* s_stage = sB + B_STAGES * B_TILE_BYTES;
  uint8_t* s_stat = s_stage + STAGE_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_stage + STAGE_BYTES + STAT_BYTES);
  uint64_t* a_full = bars;
  uint64_t* a_empty = a_full + A_STAGES;
  uint64_t* b_full = a_empty + A_STAGES;
  uint64_t* b_empty = b_full + B_STAGES_NARROW;
  uint64_t* acc_full = b_empty + B_STAGES_NARROW;
  const int b_stages = p.bn == 16 ? B_STAGES_NARROW : B_STAGES;
  const int b_stride = p.bn * 128;                        // bytes per weight slot
  uint64_t* acc_empty = acc_full + 2;
  uint64_t* a_ready = acc_empty + 2;                   // A stage transformed (or passed through) -> MMA may read it
  uint64_t* side_full = a_ready + A_STAGES;            // side ring (one slot = both tiles of a 1-tap K-block)
  uint64_t* side_empty = side_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(side_empty + 1);
  static_assert((3 * A_STAGES + 2 * B_STAGES_NARROW + 4 + 2) * 8 + 4 <= 512, "barrier region");
  const int a_stages = p.side_ring ? A_STAGES - 1 : A_STAGES;      // main-ring depth
  const int n_main = p.side_ring ? p.n_main : p.n_kb;

  // warp index through a shuffle: the compiler then knows it is warp-uniform, keeps the role branches and everything
  // derived from them on the uniform datapath (no per-access R2UR of the memory descriptor in the epilogue)
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int n_kb = p.n_kb;

  if (threadIdx.x == 0) {
    for (int i = 0; i < A_STAGES; ++i) { mbar_init(a_full + i, 1); mbar_init(a_empty + i, 1); mbar_init(a_ready + i, 128); }
    for (int i = 0; i < B_STAGES_NARROW; ++i) { mbar_init(b_full + i, 1); mbar_init(b_empty + i, 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(acc_full + i, 1); mbar_init(acc_empty + i, 4 * EPI_GROUPS); }
    mbar_init(side_full, 1); mbar_init(side_empty, 1);
    fence_barrier_init();
  }
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a0);
    tma_prefetch_desc(&map_b);
    if (p.n_seg > 1) tma_prefetch_desc(&map_a1);
    if (p.n_seg > 2) tma_prefetch_desc(&map_a2);
  }
  if (warp == 3) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // programmatic dependent launch: everything above (barrier init, descriptor prefetch, TMEM allocation) may overlap the tail of
  // the previous kernel in the stream; its results are only touched after this point.  The next kernel may start launching now.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  if (warp < 4) {
  reg_dec<PIPE_REGS>();
  if (warp == 0) {
    // ------------------------------------------------------------------ A producer
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int ct = item_tile(p, item);
        TileCoord tc[MT];
        int n_valid = 0;
        for (int j = 0; j < MT; ++j) { tc[j] = decode_tile(p, ct * MT + j); n_valid += tc[j].valid; }
        for (int i = 0; i < n_main; ++i) {
          const uint32_t e = p.ksched[i];
          const int sgi = e & 15, c0 = ((e >> 4) & 0xFFF) * 64;
          const int halo = p.seg[sgi].halo;
          mbar_wait_relaxed<256>(a_empty + stage, phase ^ 1);   // a stage frees every ~3 us: ncu counted 19 k polls per launch at 40 ns
          mbar_expect_tx(a_full + stage, n_valid * (halo ? A_TILE_BYTES : A_TILE1_BYTES));
          const CUtensorMap* map = sgi == 0 ? &map_a0 : (sgi == 1 ? &map_a1 : &map_a2);
          for (int j = 0; j < MT; ++j) {
            if (!tc[j].valid) continue;
            tma_load_4d(sA + (stage * MT + j) * A_TILE_STRIDE, map, a_full + stage, c0, tc[j].f0 - halo, tc[j].t0 - halo,
                        tc[j].b);
          }
          if (++stage == a_stages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 3) {
    // ------------------------------------------------------------------ side-ring producer (fused 1x1 shortcut operands)
    // A 1-tap K-block is 0.35 us of MMA work behind ~1.2 us of TMA latency: in the main ring four of them in a row starved the
    // MMA warp and kept the next item's first 9-tap block from being requested (5 us of a 14 us item).  Here they have their own
    // slot (the third A stage), are requested as soon as the previous one is consumed and are consumed between the 9-tap taps.
    if (lane == 0 && p.side_ring) {
      uint32_t phase = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int ct = item_tile(p, item);
        TileCoord tc[MT];
        int n_valid = 0;
        for (int j = 0; j < MT; ++j) { tc[j] = decode_tile(p, ct * MT + j); n_valid += tc[j].valid; }
        for (int i = n_main; i < n_kb; ++i) {
          const uint32_t e = p.ksched[i];
          const int sgi = e & 15, c0 = ((e >> 4) & 0xFFF) * 64;
          mbar_wait_relaxed<128>(side_empty, phase ^ 1);
          mbar_expect_tx(side_full, n_valid * A_TILE1_BYTES);
          const CUtensorMap* map = sgi == 0 ? &map_a0 : (sgi == 1 ? &map_a1 : &map_a2);
          for (int j = 0; j < MT; ++j) {
            if (!tc[j].valid) continue;
            tma_load_4d(sA + ((A_STAGES - 1) * MT + j) * A_TILE_STRIDE, map, side_full, c0, tc[j].f0, tc[j].t0, tc[j].b);
          }
          phase ^= 1;
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------------------------------------------ B (weight) producer
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
        const int n0 = item_nblk(p, item) * BN;
        if (p.side_ring) {                                   // weight tiles in MMA order
          walk_steps(p, [&](bool, int idx, int tap, int) {
            const int kt = static_cast<int>(p.ksched[idx] >> 16) + tap;
            mbar_wait_relaxed<128>(b_empty + stage, phase ^ 1);
            mbar_expect_tx(b_full + stage, b_stride);
            tma_load_2d(sB + stage * b_stride, &map_b, b_full + stage, 0, kt * p.Cout + n0);
            if (++stage == b_stages) { stage = 0; phase ^= 1; }
          });
          continue;
        }
        for (int i = 0; i < n_kb; ++i) {
          const uint32_t e = p.ksched[i];
          const int ntaps = p.seg[e & 15].taps;
          int kt = e >> 16;
          for (int tap = 0; tap < ntaps; ++tap, ++kt) {
            mbar_wait_relaxed<128>(b_empty + stage, phase ^ 1);
            mbar_expect_tx(b_full + stage, b_stride);
            tma_load_2d(sB + stage * b_stride, &map_b, b_full + stage, 0, kt * p.Cout + n0);
            if (++stage == b_stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 2) {
    // ------------------------------------------------------------------ MMA issuer
    // The whole warp walks the pipeline (so every operand is provably warp-uniform and the compiler emits
    // no per-thread "waterfall" around the uniform-datapath UTCHMMA); one elected lane issues.  Descriptors
    // are built once: only the 14-bit start-address field changes, by a plain add per MMA.
    const uint32_t idesc = make_idesc_f16(128, p.bn, kOperandIsBf16);
    const uint64_t a_hi9 = make_desc_sw128(0, A_SBO) & 0xFFFFFFFF00000000ull;
    const uint64_t a_hi1 = make_desc_sw128(0, TILE_F * 128) & 0xFFFFFFFF00000000ull;   // tile without halo: dense rows
    const uint64_t b_hi = make_desc_sw128(0, 1024) & 0xFFFFFFFF00000000ull;
    const uint32_t lo_const = 1u << 16;                                   // LBO field (unused by swizzled K-major)
    const uint32_t sA_lo = (smem_u32(sA) & 0x3FFFF) >> 4, sB_lo = (smem_u32(sB) & 0x3FFFF) >> 4;
    uint32_t sa = 0, pa = 0, sb = 0, pb = 0, as = 0, pacc = 0, ps = 0;
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const int ct = item_tile(p, item);
      const bool valid1 = (ct * MT + 1) < p.n_mtiles;                    // M-tile 0 of an item is always valid
      mbar_wait(acc_empty + as, pacc ^ 1);
      fence_after_sync();
      uint32_t accumulate = 0;
      const uint32_t d0 = tmem_base + (as * MT) * BN, d1 = d0 + BN;
      // launches without a side ring keep the plain loop below (and so does the weight producer): walk_steps issues the same
      // MMAs in the same order, but driving them through it too was measured slower on a B200 at 1000 W (two-segment 3x3
      // GroupNorm-on-load launches +11-14 %, C -> 4 pyramid launches up to +19 %, 256 x 4 s headline 1320-1326 -> 1278-1292 audio-s/s)
      if (p.side_ring) {
        int step = 0;
        walk_steps(p, [&](bool side, int idx, int tap, int ntaps) {
          const SegParams& sg = p.seg[p.ksched[idx] & 15];
          uint32_t a_base0, a_off = 0;
          if (side) {
            mbar_wait(side_full, ps);
            fence_after_sync();
            a_base0 = sA_lo + (((A_STAGES - 1) * MT) * A_TILE_STRIDE >> 4);
          } else {
            if (tap == 0) {
              mbar_wait(sg.norm ? a_ready + sa : a_full + sa, pa);
              fence_after_sync();
            }
            a_base0 = sA_lo + ((sa * MT) * A_TILE_STRIDE >> 4);
            const int df = ntaps == 9 ? tap / 3 : sg.halo, dt = ntaps == 9 ? tap - 3 * (tap / 3) : sg.halo;
            a_off = ((dt * HALO_F + df) * 128) >> 4;
          }
          const uint64_t a_hi = sg.halo ? a_hi9 : a_hi1;
          mbar_wait(b_full + sb, pb);
          fence_after_sync();
          const uint32_t b_lo = (sB_lo + (sb * b_stride >> 4)) | lo_const;
          const uint32_t a_lo0 = (a_base0 + a_off) | lo_const, a_lo1 = (a_base0 + (A_TILE_STRIDE >> 4) + a_off) | lo_const;
          const bool last_tap = tap == ntaps - 1;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              mma_f16(d0, a_hi | (a_lo0 + 2 * k), b_hi | (b_lo + 2 * k), idesc, k == 0 ? accumulate : 1u);
            if (valid1) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                mma_f16(d1, a_hi | (a_lo1 + 2 * k), b_hi | (b_lo + 2 * k), idesc, k == 0 ? accumulate : 1u);
            }
            mma_commit(b_empty + sb);
            if (side) mma_commit(side_empty);
            else if (last_tap) mma_commit(a_empty + sa);
            if (step == p.n_steps - 1) mma_commit(acc_full + as);
          }
          __syncwarp();
          accumulate = 1;
          ++step;
          if (++sb == b_stages) { sb = 0; pb ^= 1; }
          if (side) ps ^= 1;
          else if (last_tap && ++sa == a_stages) { sa = 0; pa ^= 1; }
        });
        if (++as == 2) { as = 0; pacc ^= 1; }
        continue;
      }
      for (int i = 0; i < n_kb; ++i) {
        const SegParams& sg = p.seg[p.ksched[i] & 15];
        const int ntaps = sg.taps;
        const uint64_t a_hi = sg.halo ? a_hi9 : a_hi1;
        mbar_wait(sg.norm ? a_ready + sa : a_full + sa, pa);   // normalised-on-load stages are released by the transform warps
        fence_after_sync();
        const uint32_t a_base0 = sA_lo + ((sa * MT) * A_TILE_STRIDE >> 4), a_base1 = a_base0 + (A_TILE_STRIDE >> 4);
        int df = ntaps == 9 ? 0 : sg.halo, dt = df;                     // tap -> (df, dt); a 1-tap segment reads the box centre
        for (int tap = 0; tap < ntaps; ++tap) {
          mbar_wait(b_full + sb, pb);
          fence_after_sync();
          const uint32_t a_off = ((dt * HALO_F + df) * 128) >> 4;
          const uint32_t b_lo = (sB_lo + (sb * b_stride >> 4)) | lo_const;
          const uint32_t a_lo0 = (a_base0 + a_off) | lo_const, a_lo1 = (a_base1 + a_off) | lo_const;
          if (elect_one()) {
#pragma unroll
            for (int k = 0; k < 4; ++k)
              mma_f16(d0, a_hi | (a_lo0 + 2 * k), b_hi | (b_lo + 2 * k), idesc, k == 0 ? accumulate : 1u);
            if (valid1) {
#pragma unroll
              for (int k = 0; k < 4; ++k)
                mma_f16(d1, a_hi | (a_lo1 + 2 * k), b_hi | (b_lo + 2 * k), idesc, k == 0 ? accumulate : 1u);
            }
            mma_commit(b_empty + sb);
            if (tap == ntaps - 1) mma_commit(a_empty + sa);
            if (tap == ntaps - 1 && i == n_kb - 1) mma_commit(acc_full + as);
          }
          __syncwarp();
          accumulate = 1;
          if (++dt == 3) { dt = 0; ++df; }                                 // tap = df * 3 + dt
          if (++sb == b_stages) { sb = 0; pb ^= 1; }
        }
        if (++sa == A_STAGES) { sa = 0; pa ^= 1; }
      }
      if (++as == 2) { as = 0; pacc ^= 1; }
    }
  }
  } else if (warp >= 8 && warp < 12) {
    reg_dec<XFORM_REGS>();
    // ------------------------------------------------------------------ operand transform (4 warps)
    // GroupNorm (+SiLU) on load: when a segment is flagged `norm`, the raw 16-bit tile that TMA just
    // landed is rewritten in place as act(x * scale[b,c] + shift[b,c]) before the MMA reads it, which
    // removes the stand-alone normalisation pass (one read + one write of the tensor) from HBM.
    // Thread -> fixed 8-channel group g (its scale/shift live in registers) and a lane of pixels; the
    // physical 16-byte slot of group g in pixel row p is g ^ (p & 7) (TMA 128-byte swizzle).  Halo pixels
    // outside the image stay zero: the convolution pads the *normalised* tensor with zeros.
    // Arithmetic: the affine part in fp32 (an all-16-bit HFMA2 variant was 5% faster but doubled the backbone's
    // error), SiLU(y) = h + h * tanh(h) with h = y/2 (the 1/2 is folded into scale/shift) in packed 16-bit: one
    // MUFU.TANH per TWO elements (an fp32 ex2/rcp SiLU took ~2x the transform time).
    // The transform shares each SM sub-partition with an epilogue warp and has ~4600 cycles per K-block; the
    // (scale, shift) entries are fetched BEFORE waiting for the tile so that their latency is off the critical path.
    const int tt = threadIdx.x - 256;
    const int g = tt & 7, p_lane = tt >> 3;              // 16 pixel lanes
    uint32_t stage = 0, phase = 0;
    const bool any_norm = (p.seg[0].norm | p.seg[1].norm | p.seg[2].norm) != 0;   // else: the MMA warp never waits on a_ready
    for (int item = blockIdx.x; any_norm && item < p.n_items; item += gridDim.x) {
      const int ct = item_tile(p, item);
      TileCoord tc[MT];
      for (int j = 0; j < MT; ++j) tc[j] = decode_tile(p, ct * MT + j);
      for (int i = 0; i < n_main; ++i) {
        const uint32_t e = p.ksched[i];
        const SegParams& sg = p.seg[e & 15];
        float2 sc[MT][4], sh[MT][4];                      // (scale, shift) of channel pairs: packed fp32x2 affine
        if (sg.norm) {
          const int c0 = ((e >> 4) & 0xFFF) * 64 + g * 8;
          const float pre = sg.act ? 0.5f : 1.0f;
#pragma unroll
          for (int j = 0; j < MT; ++j) {
            const float4* tp = reinterpret_cast<const float4*>(sg.tab + static_cast<int64_t>(tc[j].valid ? tc[j].b : 0) * sg.tab_stride + c0);
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float4 e = __ldg(tp + u);
              sc[j][u] = make_float2(pre * e.x, pre * e.z); sh[j][u] = make_float2(pre * e.y, pre * e.w);
            }
          }
        }
        mbar_wait_relaxed(a_full + stage, phase);
        if (sg.norm) {
#pragma unroll
          for (int j = 0; j < MT; ++j) {
            if (!tc[j].valid) continue;
            // halo rows / columns that lie inside the image (the rest is the convolution's zero padding)
            const int r_lo = tc[j].t0 == 0 ? 1 : 0, r_hi = min(HALO_T, p.T - tc[j].t0 + 1);
            const int c_lo = tc[j].f0 == 0 ? 1 : 0, c_hi = min(HALO_F, p.F - tc[j].f0 + 1);
            const bool interior = r_lo == 0 && c_lo == 0 && r_hi == HALO_T && c_hi == HALO_F;   // warp-uniform
            uint8_t* tile = sA + (stage * MT + j) * A_TILE_STRIDE;
            // four pixel slots per pass: all four 16-byte loads are in flight before the first is consumed, and the
            // pass has no branches (a slot-at-a-time loop was one long dependent chain: ~200 cycles per slot)
            constexpr int N_PASS = (HALO_T * HALO_F + 63) / 64;
            auto xform = [&](uint4& rawv, auto act_tag) {
              constexpr bool ACT = decltype(act_tag)::value;
              op2_t* h2 = reinterpret_cast<op2_t*>(&rawv);
#pragma unroll
              for (int w = 0; w < 4; ++w) {
                const float2 y = __ffma2_rn(op22f2(h2[w]), sc[j][w], sh[j][w]);
                if (ACT) {
                  const op2_t h = f2op2(y.x, y.y);
                  h2[w] = __hfma2(h, op2_tanh(h), h);
                } else {
                  h2[w] = f2op2(y.x, y.y);
                }
              }
            };
            // tile interior to the image (the common case): the 12 slots of a thread are fixed offsets from one base
            // address (px & 7 does not depend on the pass), only the last one is conditional (180 = 11 * 16 + 4 pixels)
            auto run_interior = [&](auto act_tag) {
              uint8_t* base = tile + p_lane * 128 + ((g ^ (p_lane & 7)) << 4);
#pragma unroll
              for (int pass = 0; pass < N_PASS; ++pass) {
                uint4 raw[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const int i = pass * 4 + u;
                  if (i < 11 || p_lane < 4) raw[u] = *reinterpret_cast<uint4*>(base + i * 2048);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) xform(raw[u], act_tag);
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const int i = pass * 4 + u;
                  if (i < 11 || p_lane < 4) *reinterpret_cast<uint4*>(base + i * 2048) = raw[u];
                }
              }
            };
            auto run_border = [&](auto act_tag) {
#pragma unroll 1
              for (int pass = 0; pass < N_PASS; ++pass) {
                uint4 raw[4];
                uint4* slot[4];
                bool on[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                  const int px = p_lane + 16 * (pass * 4 + u);
                  const int hr = px / HALO_F, hc = px - hr * HALO_F;
                  on[u] = px < HALO_T * HALO_F && hr >= r_lo && hr < r_hi && hc >= c_lo && hc < c_hi;
                  slot[u] = reinterpret_cast<uint4*>(tile + px * 128 + ((g ^ (px & 7)) << 4));
                  raw[u] = on[u] ? *slot[u] : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < 4; ++u) xform(raw[u], act_tag);
#pragma unroll
                for (int u = 0; u < 4; ++u)
                  if (on[u]) *slot[u] = raw[u];
              }
            };
            if (interior) { if (sg.act) run_interior(std::true_type{}); else run_interior(std::false_type{}); }
            else { if (sg.act) run_border(std::true_type{}); else run_border(std::false_type{}); }
          }
          fence_proxy_async();                            // generic-proxy writes -> visible to the tensor core's async proxy
        }
        mbar_arrive(a_ready + stage);
        if (++stage == a_stages) { stage = 0; phase ^= 1; }
      }
    }
  } else {
    // ------------------------------------------------------------------ epilogue (4 warps = 128 TMEM lanes)
    // tcgen05.ld hands every thread one pixel row (32 consecutive channels).  Writing that straight to
    // global memory would touch 32 different 128-byte lines per store instruction, so each warp first
    // transposes its 32x32 block through a swizzled shared-memory tile; afterwards 8 lanes cover the
    // 128 contiguous bytes of one pixel and every global access (bias, residual, outputs) is coalesced.
    reg_inc<EPI_REGS>();
    const int q = warp & 3;                              // TMEM lane quadrant of this warp
    const int eg = warp >= 12 ? 1 : 0;                   // epilogue group = M-tile of the item this warpgroup drains
    float4* stage = reinterpret_cast<float4*>(s_stage) + (eg * 4 + q) * (32 * 8);   // [32 pixels][8 float4], XOR-swizzled
    const int cc = lane & 7;                             // channel quad inside the 32-channel chunk (transposed phase)
    const int rsub = lane >> 3;                          // pixel sub-row (transposed phase)
    const int et = (threadIdx.x & 127);                  // 0..127 inside the epilogue group
    uint32_t as = 0, pacc = 0;
    const bool do_stats = p.sums != nullptr;             // host guarantees n_nblocks <= STAT_SLOTS when sums are requested
    // GroupNorm statistics: every warp leaves its 32-pixel partial sums (fp32, fixed summation order) in its
    // own shared-memory slot; after each M-tile thread c adds the four warps' partials of channel c into
    // DOUBLE registers that live across the CTA's items, and only those go to global memory (double atomics).
    // E[x^2] - mean^2 amplifies rounding noise in these sums ~1000x on some layers, so no fp32 atomics here.
    float2* wstat = reinterpret_cast<float2*>(s_stat) + eg * 4 * BN;   // [4 warps][BN channels] (sum, sum of squares)
    double acc_s[STAT_SLOTS], acc_q[STAT_SLOTS];
#pragma unroll
    for (int u = 0; u < STAT_SLOTS; ++u) { acc_s[u] = 0.0; acc_q[u] = 0.0; }
    int stat_b = -1;                                     // utterance the register statistics currently belong to
    auto flush_stats = [&]() {
#pragma unroll
      for (int u = 0; u < STAT_SLOTS; ++u) {
        if (u < p.n_nblocks) {
          if (et < p.bn) {                              // bn = 64 (C_out = 64 layers): half of the group's threads own a channel
            double* dst = p.sums + (static_cast<int64_t>(stat_b) * p.Cout + u * BN + et) * 2;
            atomicAdd(dst, acc_s[u]);
            atomicAdd(dst + 1, acc_q[u]);
          }
        }
        acc_s[u] = 0.0; acc_q[u] = 0.0;
      }
    };
    for (int item = blockIdx.x; item < p.n_items; item += gridDim.x) {
      const int ct = item_tile(p, item);
      const int nblk = item - ct * p.n_nblocks;
      const int n0 = nblk * BN;
      mbar_wait_relaxed(acc_full + as, pacc);
      fence_after_sync();
      for (int j = eg; j <= eg; ++j) {
        const TileCoord tc = decode_tile(p, ct * MT + j);
        if (!tc.valid) continue;                          // warp-uniform
        if (do_stats && stat_b != tc.b) {
          if (stat_b >= 0) flush_stats();
          stat_b = tc.b;
        }
        if (p.pyr_out) {
          // progressive-output epilogue: the first pyr_C accumulator columns are the image-space residual;
          // thread = pixel, add bias and the FIR-upsampled coarser pyramid level, write fp32 [B,T,F,pyr_C]
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + ((q * 32u) << 16) + (as * MT + j) * BN, v);
          tmem_ld_wait();
          const int m = q * 32 + lane;
          const int t = tc.t0 + (m >> 3), f = tc.f0 + (m & 7);
          if (t < p.T && f < p.F) {
            float o[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) o[c] = c < p.pyr_C ? __uint_as_float(v[c]) + __ldg(p.bias + c) : 0.f;
            if (p.pyr_prev) {
              const int Tp = p.T >> 1, Fp = p.F >> 1;
              const int t_a = (t & 1) ? (t >> 1) : (t >> 1) - 1, f_a = (f & 1) ? (f >> 1) : (f >> 1) - 1;
              const float wt_a = (t & 1) ? 0.75f : 0.25f, wf_a = (f & 1) ? 0.75f : 0.25f;
              const float* pb = p.pyr_prev + static_cast<int64_t>(tc.b) * Tp * Fp * p.pyr_C;
              if (p.pyr_C == 4) {
                // the four taps as four independent 16-byte loads (a scalar loop over channels serialised 16 L2 latencies
                // per pixel and made this epilogue, not the MMA, the bound of the C -> 4 convolutions)
                float4 tap[4];
                float wg[4];
#pragma unroll
                for (int u = 0; u < 2; ++u)
#pragma unroll
                  for (int w = 0; w < 2; ++w) {
                    const int tt = t_a + u, ff = f_a + w;
                    const bool ok = tt >= 0 && tt < Tp && ff >= 0 && ff < Fp;
                    wg[u * 2 + w] = ok ? (u ? 1.0f - wt_a : wt_a) * (w ? 1.0f - wf_a : wf_a) : 0.f;
                    tap[u * 2 + w] = ok ? __ldg(reinterpret_cast<const float4*>(pb + (static_cast<int64_t>(tt) * Fp + ff) * 4))
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
                  }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                  o[0] = fmaf(wg[k], tap[k].x, o[0]); o[1] = fmaf(wg[k], tap[k].y, o[1]);
                  o[2] = fmaf(wg[k], tap[k].z, o[2]); o[3] = fmaf(wg[k], tap[k].w, o[3]);
                }
              } else {
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                  const int tt = t_a + u;
                  if (tt < 0 || tt >= Tp) continue;
                  const float wt = u ? 1.0f - wt_a : wt_a;
#pragma unroll
                  for (int w = 0; w < 2; ++w) {
                    const int ff = f_a + w;
                    if (ff < 0 || ff >= Fp) continue;
                    const float wgt = wt * (w ? 1.0f - wf_a : wf_a);
                    const float* src = pb + (static_cast<int64_t>(tt) * Fp + ff) * p.pyr_C;
                    for (int c = 0; c < p.pyr_C; ++c) o[c] = fmaf(wgt, __ldg(src + c), o[c]);
                  }
                }
              }
            }
            float* dst = p.pyr_out + ((static_cast<int64_t>(tc.b) * p.T + t) * p.F + f) * p.pyr_C;
            if (p.pyr_C == 4) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
            else for (int c = 0; c < p.pyr_C; ++c) dst[c] = o[c];
          }
          continue;
        }
        // pixel rows of this lane in the transposed phase: 64-bit tile base + 32-bit row offsets
        const bool full = tc.t0 + TILE_T <= p.T && tc.f0 + TILE_F <= p.F;       // warp-uniform
        const int64_t tile_base = ((static_cast<int64_t>(tc.b) * p.T + tc.t0) * p.F + tc.f0) * p.Cout + n0 + cc * 4;
        // row `it` of this lane is pixel m = q*32 + it*4 + rsub of the tile: frame q*4 + (it >> 1), bin (it & 1)*4 + rsub
        const int roff0 = ((q * 4) * p.F + rsub) * p.Cout, roff_t = p.F * p.Cout, roff_f = 4 * p.Cout;
        auto roff = [&](int it) { return roff0 + (it >> 1) * roff_t + (it & 1) * roff_f; };
        uint32_t okmask = 0;
#pragma unroll
        for (int it = 0; it < 8; ++it) {
          const int m = q * 32 + it * 4 + rsub;
          const bool ok = tc.t0 + (m >> 3) < p.T && tc.f0 + (m & 7) < p.F;
          okmask |= ok ? (1u << it) : 0u;
        }
        const float* res_p = !RES16 && p.residual ? p.residual + tile_base : nullptr;
        const op_t* res16_p = RES16 ? p.residual_h16 + tile_base : nullptr;
        float* of_p = p.out_f32 ? p.out_f32 + tile_base : nullptr;
        op_t* oh_p = p.out_h16 ? p.out_h16 + tile_base : nullptr;
        if (RES16 || res_p) {
          // pull the NEXT tile's residual rows (512 or 256 B per pixel) into L2 now: by the time its epilogue runs,
          // the register loads below see L2 latency instead of HBM latency
          const int nitem = item + gridDim.x;
          const int nct = item_tile(p, nitem);
          const int nmi = nitem < p.n_items ? nct * MT + j : p.n_mtiles;
          const int nblk_n = nitem - nct * p.n_nblocks;
          const TileCoord nt = decode_tile(p, nmi);
          const int t = nt.t0 + (et >> 3), f = nt.f0 + (et & 7);
          if (nt.valid && t < p.T && f < p.F) {
            const int64_t po = ((static_cast<int64_t>(nt.b) * p.T + t) * p.F + f) * p.Cout + nblk_n * BN;
            if (RES16) {
#pragma unroll
              for (int u = 0; u < 2; ++u) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.residual_h16 + po + u * 64));
            } else {
#pragma unroll
              for (int u = 0; u < 4; ++u) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.residual + po + u * 32));
            }
          }
        }
        const float2 sc2 = make_float2(p.scale, p.scale);
        // bias (+ per-utterance FiLM bias): the L1 left beside 227 KB of shared memory does not keep these lines, so the
        // loads of chunk ch + 1 are issued while chunk ch is processed
        const float* bias_p = p.bias + n0 + cc * 4;
        const float* biasb_p = p.bias_b ? p.bias_b + static_cast<int64_t>(tc.b) * p.bias_b_stride + n0 + cc * 4 : nullptr;
        float4 bv = __ldg(reinterpret_cast<const float4*>(bias_p));
        float4 bvb = biasb_p ? __ldg(reinterpret_cast<const float4*>(biasb_p)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 res[8];
        // two register buffers for the 16-bit shortcut rows: chunk ch + 1 is requested BEFORE chunk ch's accumulators are read, a
        // whole chunk ahead of its use (with one buffer the compiler hoisted the fp16 -> fp32 conversions of the freshly requested
        // rows to the top of the next chunk, in front of the TMEM read and the transposition: the warp sat on the L2 latency there,
        // and Conv_1 was 10 % slower)
        uint2 res16_buf[2][8];
        auto load_res16 = [&](int ch) {
          uint2 (&dst)[8] = res16_buf[ch & 1];
          if (full) {
#pragma unroll
            for (int it = 0; it < 8; ++it) dst[it] = __ldg(reinterpret_cast<const uint2*>(res16_p + roff(it) + ch * 32));
          } else {
#pragma unroll
            for (int it = 0; it < 8; ++it)
              dst[it] = ((okmask >> it) & 1) ? __ldg(reinterpret_cast<const uint2*>(res16_p + roff(it) + ch * 32)) : make_uint2(0u, 0u);
          }
        };
        if (RES16) load_res16(0);
        auto load_res = [&](float4 (&r)[8], int ch) {
          if (full) {
#pragma unroll
            for (int it = 0; it < 8; ++it) r[it] = __ldg(reinterpret_cast<const float4*>(res_p + roff(it) + ch * 32));
          } else {
#pragma unroll
            for (int it = 0; it < 8; ++it)
              r[it] = ((okmask >> it) & 1) ? __ldg(reinterpret_cast<const float4*>(res_p + roff(it) + ch * 32))
                                           : make_float4(0.f, 0.f, 0.f, 0.f);
          }
        };
        const int n_chunks = p.bn >> 5;                   // 4, or 2 for the 64-channel layers of the nf = 64 variant
#pragma unroll
        for (int ch = 0; ch < BN / 32; ++ch) {
          if (ch >= n_chunks) break;                        // warp-uniform
          float4 cw[4], cbias = make_float4(0.f, 0.f, 0.f, 0.f);
          if constexpr (COMB) {                               // Combine: 1x1 conv of the <=4-channel input pyramid
            const int c = n0 + ch * 32 + cc * 4;
            cbias = __ldg(reinterpret_cast<const float4*>(p.comb_b + c));
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const float* wr = p.comb_w + (c + u) * p.comb_C;
              cw[u] = make_float4(__ldg(wr), p.comb_C > 1 ? __ldg(wr + 1) : 0.f, p.comb_C > 2 ? __ldg(wr + 2) : 0.f,
                                  p.comb_C > 3 ? __ldg(wr + 3) : 0.f);
            }
          }
          float4 bvn = bv, bvbn = bvb;
          if (ch + 1 < n_chunks) {
            bvn = __ldg(reinterpret_cast<const float4*>(bias_p + (ch + 1) * 32));
            if (biasb_p) bvbn = __ldg(reinterpret_cast<const float4*>(biasb_p + (ch + 1) * 32));
          }
          uint32_t v[32];
          tmem_ld_32x32(tmem_base + ((q * 32u) << 16) + (as * MT + j) * BN + ch * 32, v);
          // (also requesting chunk 0 of the warpgroup's NEXT tile during the last chunk was measured: spills, 5 % slower)
          if (RES16) { if (ch + 1 < n_chunks) load_res16(ch + 1); }
          else if (res_p) load_res(res, ch);
          tmem_ld_wait();
#pragma unroll
          for (int g = 0; g < 8; ++g)
            stage[lane * 8 + (g ^ (lane & 7))] = make_float4(__uint_as_float(v[4 * g]), __uint_as_float(v[4 * g + 1]),
                                                             __uint_as_float(v[4 * g + 2]), __uint_as_float(v[4 * g + 3]));
          __syncwarp();
          // packed fp32x2 arithmetic (FFMA2 / FADD2): the single epilogue warp of an SM sub-partition is bound by
          // its own instruction latencies, so halving the instruction count is what speeds it up.
          // out = acc * scale + (bias * scale) (+ residual * scale)
          const float2 bs_lo = __fmul2_rn(make_float2(bv.x + bvb.x, bv.y + bvb.y), sc2), bs_hi = __fmul2_rn(make_float2(bv.z + bvb.z, bv.w + bvb.w), sc2);
          float2 o_lo[8], o_hi[8];
#pragma unroll
          for (int it = 0; it < 8; ++it) {                  // eight independent shared-memory reads in flight
            const int rr = it * 4 + rsub;                   // pixel row inside this warp's quadrant
            const float4 a = stage[rr * 8 + (cc ^ (rr & 7))];
            o_lo[it] = make_float2(a.x, a.y); o_hi[it] = make_float2(a.z, a.w);
          }
#pragma unroll
          for (int it = 0; it < 8; ++it) {
            o_lo[it] = __ffma2_rn(o_lo[it], sc2, bs_lo); o_hi[it] = __ffma2_rn(o_hi[it], sc2, bs_hi);
            if (RES16) {
              const op2_t* r2 = reinterpret_cast<const op2_t*>(&res16_buf[ch & 1][it]);
              o_lo[it] = __ffma2_rn(op22f2(r2[0]), sc2, o_lo[it]);
              o_hi[it] = __ffma2_rn(op22f2(r2[1]), sc2, o_hi[it]);
            } else if (res_p) {
              o_lo[it] = __ffma2_rn(make_float2(res[it].x, res[it].y), sc2, o_lo[it]);
              o_hi[it] = __ffma2_rn(make_float2(res[it].z, res[it].w), sc2, o_hi[it]);
            }
            if (COMB && (full || ((okmask >> it) & 1))) {
              const int m = q * 32 + it * 4 + rsub;
              const float* pq = p.comb_pyr + ((static_cast<int64_t>(tc.b) * p.T + tc.t0 + (m >> 3)) * p.F + tc.f0 + (m & 7)) * p.comb_C;
              const float p0 = __ldg(pq), p1 = p.comb_C > 1 ? __ldg(pq + 1) : 0.f, p2 = p.comb_C > 2 ? __ldg(pq + 2) : 0.f,
                          p3 = p.comb_C > 3 ? __ldg(pq + 3) : 0.f;
              o_lo[it].x += cbias.x + cw[0].x * p0 + cw[0].y * p1 + cw[0].z * p2 + cw[0].w * p3;
              o_lo[it].y += cbias.y + cw[1].x * p0 + cw[1].y * p1 + cw[1].z * p2 + cw[1].w * p3;
              o_hi[it].x += cbias.z + cw[2].x * p0 + cw[2].y * p1 + cw[2].z * p2 + cw[2].w * p3;
              o_hi[it].y += cbias.w + cw[3].x * p0 + cw[3].y * p1 + cw[3].z * p2 + cw[3].w * p3;
            }
          }
          float2 ssum_lo = make_float2(0.f, 0.f), ssum_hi = ssum_lo, ssq_lo = ssum_lo, ssq_hi = ssum_lo;
          if (full) {                                       // whole tile inside the image: no per-row predicates
            if (of_p) {
#pragma unroll
              for (int it = 0; it < 8; ++it)
                *reinterpret_cast<float4*>(of_p + roff(it) + ch * 32) = make_float4(o_lo[it].x, o_lo[it].y, o_hi[it].x, o_hi[it].y);
            }
            if (oh_p) {
#pragma unroll
              for (int it = 0; it < 8; ++it)
                *reinterpret_cast<uint2*>(oh_p + roff(it) + ch * 32) = make_uint2(pack_op2(o_lo[it].x, o_lo[it].y), pack_op2(o_hi[it].x, o_hi[it].y));
            }
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              ssum_lo = __fadd2_rn(ssum_lo, o_lo[it]); ssum_hi = __fadd2_rn(ssum_hi, o_hi[it]);
              ssq_lo = __ffma2_rn(o_lo[it], o_lo[it], ssq_lo); ssq_hi = __ffma2_rn(o_hi[it], o_hi[it], ssq_hi);
            }
          } else {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
              if ((okmask >> it) & 1) {
                if (of_p) *reinterpret_cast<float4*>(of_p + roff(it) + ch * 32) = make_float4(o_lo[it].x, o_lo[it].y, o_hi[it].x, o_hi[it].y);
                if (oh_p) *reinterpret_cast<uint2*>(oh_p + roff(it) + ch * 32) = make_uint2(pack_op2(o_lo[it].x, o_lo[it].y), pack_op2(o_hi[it].x, o_hi[it].y));
                ssum_lo = __fadd2_rn(ssum_lo, o_lo[it]); ssum_hi = __fadd2_rn(ssum_hi, o_hi[it]);
                ssq_lo = __ffma2_rn(o_lo[it], o_lo[it], ssq_lo); ssq_hi = __ffma2_rn(o_hi[it], o_hi[it], ssq_hi);
              }
            }
          }
          float4 ssum = make_float4(ssum_lo.x, ssum_lo.y, ssum_hi.x, ssum_hi.y), ssq = make_float4(ssq_lo.x, ssq_lo.y, ssq_hi.x, ssq_hi.y);
          if (do_stats) {
#pragma unroll
            for (int sft = 8; sft <= 16; sft <<= 1) {
              ssum.x += __shfl_xor_sync(0xffffffffu, ssum.x, sft); ssum.y += __shfl_xor_sync(0xffffffffu, ssum.y, sft);
              ssum.z += __shfl_xor_sync(0xffffffffu, ssum.z, sft); ssum.w += __shfl_xor_sync(0xffffffffu, ssum.w, sft);
              ssq.x += __shfl_xor_sync(0xffffffffu, ssq.x, sft); ssq.y += __shfl_xor_sync(0xffffffffu, ssq.y, sft);
              ssq.z += __shfl_xor_sync(0xffffffffu, ssq.z, sft); ssq.w += __shfl_xor_sync(0xffffffffu, ssq.w, sft);
            }
            if (rsub == 0) {
              float4* d = reinterpret_cast<float4*>(wstat + q * BN + ch * 32 + cc * 4);
              d[0] = make_float4(ssum.x, ssq.x, ssum.y, ssq.y);
              d[1] = make_float4(ssum.z, ssq.z, ssum.w, ssq.w);
            }
          }
          __syncwarp();                                   // staging tile is rewritten by the next chunk
          bv = bvn; bvb = bvbn;
        }
        // (deferring this cross-warp reduction to the start of the warpgroup's next tile -- mbarrier arrive / wait pairs instead
        // of the two bar.sync -- was measured: Conv_1 launches 25 % SLOWER; the barriers keep the four warps of a tile in step)
        if (do_stats) {                                   // block-uniform
          asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
          double s = 0.0, sq = 0.0;
#pragma unroll
          for (int w = 0; w < 4; ++w) { const float2 e = et < p.bn ? wstat[w * BN + et] : make_float2(0.f, 0.f); s += e.x; sq += e.y; }
#pragma unroll
          for (int u = 0; u < STAT_SLOTS; ++u) if (u == nblk) { acc_s[u] += s; acc_q[u] += sq; }
          asm volatile("bar.sync %0, 128;" ::"r"(1 + eg) : "memory");
        }
      }
      // all TMEM reads of this accumulator stage are done: hand it back to the MMA warp
      fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty + as);
      if (++as == 2) { as = 0; pacc ^= 1; }
    }
    if (do_stats && stat_b >= 0) flush_stats();
  }

  fence_before_sync();
  __syncthreads();
  if (warp == 3) tmem_dealloc(tmem_base, 512);
}

// weight packing: fp32 (OIHW, or [in][out] for NIN) -> 16-bit [kt][rows_total][64]
__device__ __forceinline__ void pack_fwd_element(const PackDesc& d, int64_t i) {
  const int C1 = d.C1, C2 = d.C2, Cout = d.Cout, ksize = d.ksize, io_layout = d.io;
  const int taps = ksize * ksize;
  const int j = static_cast<int>(i % 64);
  const int co = static_cast<int>((i / 64) % Cout);
  const int kt = static_cast<int>(i / (64ll * Cout));
  float v;
  if (io_layout == 2) {                           // first conv: k = tap * C1 + ci, zero beyond 9 * C1
    const int tap = j / C1, ci = j % C1;
    v = tap < 9 ? d.w1[((static_cast<int64_t>(co) * C1 + ci) * 3 + tap / 3) * 3 + tap % 3] : 0.f;
  } else if (kt < (C1 / 64) * taps) {
    const int kb = kt / taps, tap = kt % taps;
    const int ci = kb * 64 + j;
    if (io_layout) v = d.w1[static_cast<int64_t>(ci) * Cout + co];
    else {
      const int kf = ksize == 3 ? tap / 3 : 0, ktm = ksize == 3 ? tap % 3 : 0;
      v = d.w1[((static_cast<int64_t>(co) * C1 + ci) * ksize + kf) * ksize + ktm];
    }
  } else {
    const int ci = (kt - (C1 / 64) * taps) * 64 + j;
    v = d.w2[static_cast<int64_t>(co) * C2 + ci];
  }
  d.out[(static_cast<int64_t>(kt) * d.rows_total + d.row_offset + co) * 64 + j] = f2op(v);
}

// dgrad packing: the input gradient of a convolution is itself a convolution of dY with the weights transposed
// (in <-> out) and flipped (tap (df,dt) -> (2-df,2-dt)):  W'[ci][co][df'][dt'] = W[co][ci][2-df'][2-dt'].
// Output rows = Cin of the forward conv, K = Cout of the forward conv.
__device__ __forceinline__ void pack_dgrad_element(const PackDesc& d, int64_t i) {
  const int Cin = d.C1, Cin_total = d.C2, Cout = d.Cout, ksize = d.ksize, ci_off = d.row_offset;
  const int taps = ksize * ksize;
  const int j = static_cast<int>(i % 64);
  const int ci = static_cast<int>((i / 64) % Cin);
  const int kt = static_cast<int>(i / (64ll * Cin));
  const int kb = kt / taps, tap = kt % taps;
  const int co = kb * 64 + j;
  float v;
  if (d.io) v = d.w1[static_cast<int64_t>(ci_off + ci) * Cout + co];          // NIN [in][out]
  else {
    const int kf = ksize == 3 ? 2 - tap / 3 : 0, ktm = ksize == 3 ? 2 - tap % 3 : 0;
    v = d.w1[((static_cast<int64_t>(co) * Cin_total + ci_off + ci) * ksize + kf) * ksize + ktm];
  }
  d.out[i] = f2op(v);
}

__global__ void __launch_bounds__(256)
pack_batch_kernel(const PackDesc* __restrict__ descs, int n) {
  __shared__ PackDesc d;
  if (threadIdx.x == 0) {
    int lo = 0, hi = n - 1;                                   // last descriptor whose first_block <= blockIdx.x
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (descs[mid].first_block <= static_cast<long long>(blockIdx.x)) lo = mid; else hi = mid - 1; }
    d = descs[lo];
  }
  __syncthreads();
  const int64_t i0 = (static_cast<int64_t>(blockIdx.x) - d.first_block) * kPackChunk;
#pragma unroll 1
  for (int u = 0; u < kPackChunk / 256; ++u) {
    const int64_t i = i0 + u * 256 + threadIdx.x;
    if (i < d.total) { if (d.kind == 0) pack_fwd_element(d, i); else pack_dgrad_element(d, i); }
  }
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeFn get_encode() {
  static EncodeFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  });
  return fn;
}

int make_act_map(CUtensorMap* map, const op_t* ptr, int B, int T, int F, int C) {
  return make_act_tile_map(map, ptr, B, T, F, C, HALO_F, HALO_T);
}

int make_weight_map(CUtensorMap* map, const op_t* ptr, int64_t rows, int bn) {
  EncodeFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return FDBM_ECUDA; }
  cuuint64_t dims[2] = {64, (cuuint64_t)rows};
  cuuint64_t strides[1] = {128};
  cuuint32_t box[2] = {64, (cuuint32_t)bn};
  cuuint32_t es[2] = {1, 1};
  CUresult r = enc(map, (kOperandIsBf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16), 2, const_cast<op_t*>(ptr), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(weights, %lld rows) failed: %d", (long long)rows, (int)r); return FDBM_ECUDA; }
  return FDBM_OK;
}

}  // namespace

// TMA map of a 16-bit activation tensor [B,T,F,C] with a box of 64 channels x box_f bins x box_t frames, 128-byte swizzle
int make_act_tile_map(CUtensorMap* map, const op_t* ptr, int B, int T, int F, int C, int box_f, int box_t) {
  EncodeFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return FDBM_ECUDA; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)F, (cuuint64_t)T, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 2, (cuuint64_t)C * 2 * F, (cuuint64_t)C * 2 * F * T};
  cuuint32_t box[4] = {64, (cuuint32_t)box_f, (cuuint32_t)box_t, 1};
  cuuint32_t es[4] = {1, 1, 1, 1};
  CUresult r = enc(map, (kOperandIsBf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16), 4, const_cast<op_t*>(ptr), dims, strides, box, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(activation [%d,%d,%d,%d]) failed: %d", B, T, F, C, (int)r); return FDBM_ECUDA; }
  return FDBM_OK;
}

int64_t conv_wpack_bytes(int C1, int ksize, int C2, int Cout) {
  return (static_cast<int64_t>(C1 / 64) * ksize * ksize + C2 / 64) * Cout * 64 * 2;
}

PackDesc pack_desc_fwd(const float* w1, int C1, int ksize, const float* w2, int C2, int Cout, int n_rows_total, int row_offset, op_t* wpack) {
  const int io = ksize == -1 ? 1 : (ksize == -2 ? 2 : 0);   // -1: NIN [in][out];  -2: first conv as one im2col K-block
  const int k = io ? 1 : ksize;
  PackDesc d{};
  d.w1 = w1; d.w2 = w2; d.out = wpack; d.kind = 0; d.C1 = C1; d.ksize = k; d.io = io; d.C2 = C2; d.Cout = Cout;
  d.rows_total = n_rows_total; d.row_offset = row_offset;
  d.total = io == 2 ? static_cast<long long>(Cout) * 64 : (static_cast<long long>(C1 / 64) * k * k + C2 / 64) * Cout * 64;
  return d;
}
PackDesc pack_desc_dgrad(const float* w, int Cout, int Cin, int ksize, op_t* wpack, int Cin_total, int ci_off) {
  const int k = ksize == -1 ? 1 : ksize;
  PackDesc d{};
  d.w1 = w; d.w2 = nullptr; d.out = wpack; d.kind = 1; d.C1 = Cin; d.ksize = k; d.io = ksize == -1; d.C2 = Cin_total ? Cin_total : Cin; d.Cout = Cout;
  d.rows_total = 0; d.row_offset = ci_off;
  d.total = static_cast<long long>(Cout / 64) * k * k * Cin * 64;
  return d;
}
int launch_pack_batch(const PackDesc* descs_dev, int n_descs, long long n_blocks, cudaStream_t s) {
  if (n_descs <= 0 || n_blocks <= 0) return FDBM_OK;
  pack_batch_kernel<<<static_cast<unsigned>(n_blocks), 256, 0, s>>>(descs_dev, n_descs);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

// single packs (tests, one-off packs): a one-descriptor batch through a small device staging copy is not worth it -- these build
// the descriptor on the host and pass it by value
__global__ void __launch_bounds__(256) pack_one_kernel(const PackDesc d) {
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < d.total; i += 256ll * gridDim.x) {
    if (d.kind == 0) pack_fwd_element(d, i); else pack_dgrad_element(d, i);
  }
}

int launch_pack_conv_weights(const float* w1, int C1, int ksize, const float* w2, int C2, int Cout, int n_rows_total,
                             int row_offset, op_t* wpack, cudaStream_t s) {
  FDBM_REQUIRE((ksize == -2 && C1 <= 4 && C2 == 0) ||
               (C1 % 64 == 0 && C2 % 64 == 0 && (ksize == 1 || ksize == 3 || ksize == -1)),
               "pack_conv_weights: channels must be multiples of 64, ksize 1 or 3");
  const PackDesc d = pack_desc_fwd(w1, C1, ksize, w2, C2, Cout, n_rows_total, row_offset, wpack);
  pack_one_kernel<<<static_cast<int>(std::min<int64_t>(ceil_div64(d.total, 256), 4096)), 256, 0, s>>>(d);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

// packs W (OIHW [Cout,Cin,k,k], or NIN [Cin][Cout] when ksize == -1) for the dgrad convolution dX = conv(dY, W'):
// use with launch_conv_igemm(seg = {dY, C = Cout, taps}, Cout' = Cin)
// (Cin_total, ci_off): W has Cin_total input channels and only the slice ci_off.. +Cin is packed (concatenated inputs)
int launch_pack_conv_weights_dgrad(const float* w, int Cout, int Cin, int ksize, op_t* wpack, cudaStream_t s, int Cin_total, int ci_off) {
  FDBM_REQUIRE(Cout % 64 == 0 && Cin % 64 == 0 && (ksize == 1 || ksize == 3 || ksize == -1),
               "pack_conv_weights_dgrad: channels must be multiples of 64, ksize 1, 3 or -1 (NIN)");
  const PackDesc d = pack_desc_dgrad(w, Cout, Cin, ksize, wpack, Cin_total, ci_off);
  pack_one_kernel<<<static_cast<int>(std::min<int64_t>(ceil_div64(d.total, 256), 4096)), 256, 0, s>>>(d);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_conv_igemm(const ConvArgs& a, cudaStream_t s) {
  FDBM_REQUIRE(a.n_seg >= 1 && a.n_seg <= MAX_SEG, "conv_igemm: 1..%d K segments", MAX_SEG);
  const int bn = a.narrow_n ? 16 : (a.Cout == 64 ? 64 : BN);      // MMA N: 128; 64 for the C_out = 64 layers of ncsnpp_v2_16M; 16 for C -> 4
  FDBM_REQUIRE(a.Cout % bn == 0 && (!a.narrow_n || (a.Cout == 16 && a.pyr_out)), "conv_igemm: Cout must be a multiple of %d (got %d)", bn, a.Cout);
  FDBM_REQUIRE(a.out_f32 || a.out_h16 || a.pyr_out, "conv_igemm: no output");
  FDBM_REQUIRE(!a.pyr_out || (a.pyr_C >= 1 && a.pyr_C <= 4 && a.Cout == bn && !a.sums), "conv_igemm: bad pyramid epilogue arguments");
  FDBM_REQUIRE(!a.pyr_prev || (a.T % 2 == 0 && a.F % 2 == 0), "conv_igemm: pyramid level with odd size");
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device())) {
    FDBM_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    FDBM_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    FDBM_CUDA(cudaFuncSetAttribute(conv_igemm_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
  }
  FDBM_REQUIRE(!a.comb_pyr || (a.comb_w && a.comb_b && a.comb_C >= 1 && a.comb_C <= 4 && !a.pyr_out), "conv_igemm: bad Combine epilogue arguments");
  CUtensorMap map_a[MAX_SEG], map_b;
  ConvParams p;
  p.B = a.B; p.T = a.T; p.F = a.F; p.Cout = a.Cout;
  p.n_seg = a.n_seg;
  int kb = 0, n_kt = 0;
  for (int i = 0; i < MAX_SEG; ++i) {
    if (i < a.n_seg) {
      const ConvSeg& sg = a.seg[i];
      FDBM_REQUIRE(sg.in && sg.C > 0 && sg.C % 64 == 0 && (sg.taps == 9 || sg.taps == 1),
                   "conv_igemm: segment %d needs a tensor, C %% 64 == 0 and 9 or 1 taps (C=%d, taps=%d)", i, sg.C, sg.taps);
      const int halo = sg.taps == 9 || sg.norm_tab != nullptr;
      if (int rc = halo ? make_act_map(&map_a[i], sg.in, a.B, a.T, a.F, sg.C)
                        : make_act_tile_map(&map_a[i], sg.in, a.B, a.T, a.F, sg.C, TILE_F, TILE_T)) return rc;
      p.seg[i].halo = halo;
      kb += sg.C / 64; p.seg[i].taps = sg.taps;
      p.seg[i].norm = sg.norm_tab != nullptr; p.seg[i].act = sg.act; p.seg[i].tab = sg.norm_tab;
      p.seg[i].tab_stride = sg.tab_stride;
      n_kt += (sg.C / 64) * sg.taps;
    } else {
      map_a[i] = map_a[0];
      p.seg[i] = SegParams{1, 0, 0, 0, 0, nullptr};
    }
  }
  p.n_kb = kb;
  FDBM_REQUIRE(kb <= MAX_KB, "conv_igemm: at most %d K-blocks (got %d)", MAX_KB, kb);
  {
    // schedule: 9-tap blocks in order, the 1-tap blocks spread evenly between them
    uint32_t nine[MAX_KB], one[MAX_KB];
    int n9 = 0, n1 = 0, kt = 0;
    for (int i = 0; i < a.n_seg; ++i)
      for (int cb = 0; cb < a.seg[i].C / 64; ++cb) {
        const uint32_t e = static_cast<uint32_t>(i) | (static_cast<uint32_t>(cb) << 4) | (static_cast<uint32_t>(kt) << 16);
        if (a.seg[i].taps == 9) nine[n9++] = e; else one[n1++] = e;
        kt += a.seg[i].taps;
      }
    // 9-tap blocks first, back to back: the load + transform of each one hides behind the nine taps of the previous
    // one.  (Interleaving the 1-tap blocks between them IN THE SAME RING was measured 5 % slower: the next 9-tap block then
    // has only two short blocks of MMA work to hide behind.  The side ring below interleaves them without that cost.)
    int n = 0;
    for (int i = 0; i < n9; ++i) p.ksched[n++] = nine[i];
    for (int i = 0; i < n1; ++i) p.ksched[n++] = one[i];
    for (; n < MAX_KB; ++n) p.ksched[n] = 0;
    // side ring: every 1-tap block is a raw operand without halo (the fused 1x1 shortcut) and there is 9-tap work to hide behind
    bool side_ok = n1 > 0 && n9 > 0;
    for (int i = 0; i < a.n_seg; ++i) side_ok = side_ok && (a.seg[i].taps == 9 || !p.seg[i].halo);
    p.side_ring = side_ok ? 1 : 0;
    p.n_main = p.side_ring ? n9 : kb;
    p.side_gap = p.side_ring ? std::max(3, ceil_div(9 * n9, n1)) : 0;
    p.n_steps = n_kt;
  }
  if (int rc = make_weight_map(&map_b, a.wpack, static_cast<int64_t>(n_kt) * a.Cout, bn)) return rc;
  p.bn = bn;
  p.tiles_t = ceil_div(a.T, TILE_T); p.tiles_f = ceil_div(a.F, TILE_F);
  p.n_mtiles = a.B * p.tiles_t * p.tiles_f;
  p.n_nblocks = a.Cout / bn;
  p.n_items = ceil_div(p.n_mtiles, MT) * p.n_nblocks;
  {
    auto magic = [](int d) { return static_cast<uint32_t>((0x100000000ull + d - 1) / static_cast<uint64_t>(d)); };   // d == 1: unused
    p.mg_tiles_t = magic(p.tiles_t); p.mg_tiles_f = magic(p.tiles_f); p.mg_nblocks = magic(p.n_nblocks);
    const int64_t dmax = std::max(std::max(p.tiles_t, p.tiles_f), p.n_nblocks);
    FDBM_REQUIRE((2 * (static_cast<int64_t>(p.n_items) + num_sms()) + 2) * dmax < 0x100000000ll, "conv_igemm: %d items exceed the range of the index arithmetic", p.n_items);
  }
  p.bias = a.bias; p.bias_b = a.bias_b; p.bias_b_stride = a.bias_b_stride; p.residual = a.residual; p.scale = a.scale;
  p.residual_h16 = a.residual_h16;
  FDBM_REQUIRE(!(a.residual && a.residual_h16) && !(a.residual_h16 && (a.comb_pyr || a.pyr_out)), "conv_igemm: bad residual arguments");
  p.out_f32 = a.out_f32; p.out_h16 = a.out_h16; p.sums = a.sums;
  p.pyr_out = a.pyr_out; p.pyr_prev = a.pyr_prev; p.pyr_C = a.pyr_C;
  p.comb_pyr = a.comb_pyr; p.comb_w = a.comb_w; p.comb_b = a.comb_b; p.comb_C = a.comb_C;
  if (a.sums) {
    FDBM_REQUIRE(p.n_nblocks <= STAT_SLOTS, "conv_igemm: channel sums support Cout <= %d", STAT_SLOTS * BN);
    if (!a.sums_prezeroed) FDBM_CUDA(cudaMemsetAsync(a.sums, 0, sizeof(double) * 2 * a.B * a.Cout, s));
  }
  const int grid = std::min(p.n_items, num_sms());
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NUM_THREADS); cfg.dynamicSmemBytes = SMEM_BYTES; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  // measured: 256 x 4 s utterances 1321-1323 -> 1307 audio-s/s WITH the attribute, one utterance 18.78 -> 18.28 ms: it pays where the
  // launches are short (launch-bound small batches), so it is only requested there
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() && a.B <= pdl_batch_limit() ? 1 : 0;
  if (a.comb_pyr) FDBM_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<true, false>, map_a[0], map_a[1], map_a[2], map_b, p));
  else if (a.residual_h16) FDBM_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<false, true>, map_a[0], map_a[1], map_a[2], map_b, p));
  else FDBM_CUDA(cudaLaunchKernelEx(&cfg, conv_igemm_kernel<false, false>, map_a[0], map_a[1], map_a[2], map_b, p));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

}  // namespace fdbm

using namespace fdbm;

extern "C" int fdbm_pack_conv_weights(const float* w1, int C1, int ksize, const float* w2, int C2, int Cout,
                                      void* wpack, int64_t* bytes, void* stream) {
  const int k = ksize == -1 ? 1 : ksize;
  // ksize -2: the 3x3 input convolution (C1 <= 7 channels) as ONE 64-wide K-block over fdbm_im2col_input's columns
  if (bytes) *bytes = ksize == -2 ? static_cast<int64_t>(Cout) * 64 * 2 : conv_wpack_bytes(C1, k, C2, Cout);
  if (!wpack) return FDBM_OK;
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(w1 && ((C2 == 0) == (w2 == nullptr)), "fdbm_pack_conv_weights: null pointer");
  FDBM_REQUIRE(ksize != -2 || (C1 >= 1 && 9 * C1 <= 64 && C2 == 0), "fdbm_pack_conv_weights: ksize -2 needs 9 * C1 <= 64 and no second operand");
  return launch_pack_conv_weights(w1, C1, ksize, w2, C2, Cout, Cout, 0, reinterpret_cast<op_t*>(wpack),
                                  as_stream(stream));
}

extern "C" int fdbm_pack_conv_weights_dgrad(const float* w, int Cout, int Cin, int ksize, void* wpack, int64_t* bytes,
                                            void* stream) {
  const int k = ksize == -1 ? 1 : ksize;
  if (bytes) *bytes = conv_wpack_bytes(Cout, k, 0, Cin);
  if (!wpack) return FDBM_OK;
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(w, "fdbm_pack_conv_weights_dgrad: null weights");
  return launch_pack_conv_weights_dgrad(w, Cout, Cin, ksize, reinterpret_cast<op_t*>(wpack), as_stream(stream));
}

extern "C" int fdbm_conv_igemm(const void* in1, int C1, int ksize, const void* in2, int C2, const void* wpack,
                               const float* bias, const float* bias_b, const float* residual, float scale, int batch,
                               int T, int F, int Cout, float* out_f32, void* out_h16, double* sums, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(in1 && wpack && bias && batch > 0 && T > 0 && F > 0, "fdbm_conv_igemm: bad arguments");
  FDBM_REQUIRE(ksize == 1 || ksize == 3, "fdbm_conv_igemm: ksize must be 1 or 3");
  FDBM_REQUIRE((C2 == 0) == (in2 == nullptr), "fdbm_conv_igemm: in2 / C2 mismatch");
  ConvArgs a;
  a.seg[0].in = reinterpret_cast<const op_t*>(in1); a.seg[0].C = C1; a.seg[0].taps = ksize * ksize;
  a.n_seg = 1;
  if (in2) { a.seg[1].in = reinterpret_cast<const op_t*>(in2); a.seg[1].C = C2; a.seg[1].taps = 1; a.n_seg = 2; }
  a.wpack = reinterpret_cast<const op_t*>(wpack);
  a.bias = bias; a.bias_b = bias_b; a.bias_b_stride = Cout; a.residual = residual; a.scale = scale;
  a.B = batch; a.T = T; a.F = F; a.Cout = Cout;
  a.out_f32 = out_f32; a.out_h16 = reinterpret_cast<op_t*>(out_h16); a.sums = sums;
  return launch_conv_igemm(a, as_stream(stream));
}

// The plans' launch arguments from the C descriptor, field for field: callers reach exactly the launches a plan makes
extern "C" int fdbm_conv_igemm_ex(const fdbm_conv_desc* d, void* stream) {
  // first: a caller whose struct layout differs gets a message here, not a misread pointer on the device
  FDBM_REQUIRE(d && d->struct_bytes == static_cast<int>(sizeof(fdbm_conv_desc)),
               "fdbm_conv_igemm_ex: struct_bytes %d != sizeof(fdbm_conv_desc) %d: the caller's descriptor layout is out of date",
               d ? d->struct_bytes : 0, static_cast<int>(sizeof(fdbm_conv_desc)));
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(d->wpack && d->bias && d->B > 0 && d->T > 0 && d->F > 0, "fdbm_conv_igemm_ex: bad arguments");
  ConvArgs a;
  for (int i = 0; i < MAX_SEG; ++i) {
    const fdbm_conv_seg& s = d->seg[i];
    a.seg[i].in = reinterpret_cast<const op_t*>(s.in); a.seg[i].C = s.C; a.seg[i].taps = s.taps;
    a.seg[i].norm_tab = reinterpret_cast<const float2*>(s.norm_tab); a.seg[i].tab_stride = s.tab_stride; a.seg[i].act = s.act;
  }
  a.n_seg = d->n_seg;
  a.wpack = reinterpret_cast<const op_t*>(d->wpack);
  a.bias = d->bias; a.bias_b = d->bias_b; a.bias_b_stride = d->bias_b_stride; a.residual = d->residual;
  a.residual_h16 = reinterpret_cast<const op_t*>(d->residual_h16);
  a.scale = d->scale; a.B = d->B; a.T = d->T; a.F = d->F; a.Cout = d->Cout;
  a.out_f32 = d->out_f32; a.out_h16 = reinterpret_cast<op_t*>(d->out_h16);
  a.sums = d->sums; a.sums_prezeroed = d->sums_prezeroed != 0;
  a.pyr_out = d->pyr_out; a.pyr_prev = d->pyr_prev; a.pyr_C = d->pyr_C; a.narrow_n = d->narrow_n != 0;
  a.comb_pyr = d->comb_pyr; a.comb_w = d->comb_w; a.comb_b = d->comb_b; a.comb_C = d->comb_C;
  return launch_conv_igemm(a, as_stream(stream));
}
