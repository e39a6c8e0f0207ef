// TF-GridNet BiLSTM sweep on tcgen05 / TMEM: LayerNorm-ed input -> unfold 4 -> LSTM (both directions) -> ConvTranspose1d with its
// four taps already overlap-added (tfgridnet.py:335-350, :360-375).
//
// The recurrence is latency-bound: step s needs h_{s-1} of every unit.  (The first generation, mma.sync with the gate matrix
// re-read from shared memory by every warp every step, measured 15 us per step; profiles/r02_lstm_mma_sync_ncu_details.txt.)
//
//   * a CLUSTER of two CTAs owns 128 sequences of one direction for all steps.  The gate matrix does not fit one SM next to the
//     operands (4 x 112 x 241 fp16 = 211 KB), so each CTA holds the gate columns of 56 of the 112 (padded) hidden units
//     (N = 224, 105 KB) and both hold the full A operand [u_s | h_{s-1}]: every step a CTA computes its 56 units' gates
//     (UMMA M = 128, N = 224, K = 128 + 128), updates their cell state and writes the 56 new hidden values of every sequence
//     into its OWN h tile and ships them to its PEER's: the h tile's K-block r (64 columns) holds exactly CTA r's units, so the
//     exchange is four 4 KB cp.async.bulk shared::cta -> shared::cluster copies per step (one per 32 rows, issued by the warp
//     pair that wrote them) completing on the peer's `h_ready` barrier -- no generic remote stores, no cluster-scope fences.
//   * per-step hand-shake, no cluster barrier: tcgen05.commit is MULTICAST to both CTAs' `mma_done` / `y_done` barriers
//     (count 2), so h is overwritten only when both tensor cores are done reading it.  The MMA lane issues the K-block it
//     owns as soon as its 4 row groups have arrived (`h_local`) and the peer's when its 16 KB have landed (`h_peer`); the gate
//     columns are committed in two slices so the first half of the point-wise warps starts while the second slice computes.
//   * u_s (the unfolded input, 4 taps x 32 channels) is a ring of six single-position tiles [128 seq x 32 ch] (64-byte rows,
//     SWIZZLE_64B) filled by TMA one position per step; the four taps of a step are four K = 32 UMMA pairs on ring slots.  They
//     do not depend on h, so step i + 1's are issued right behind step i's commit into the second gate accumulator.
//   * the bias rides in the GEMM: column 120 of the h tile is the constant 1, that row of W_hh holds b_ih + b_hh.  The rows of
//     the i, f, o gates are pre-scaled by 1/2 (exact): sigmoid(x) = 0.5 tanh(x / 2) + 0.5 costs one MUFU and no multiply.
//   * ConvTranspose1d: y_{s-1} = h_{s-1} W_lin is issued together with the gates of step s (both read h_{s-1}); a point-wise
//     thread owns 8 output channels x 4 taps (one 32-column TMEM load) and overlap-adds them in registers over four consecutive
//     steps, so each output position is written once (fp16 [seq][L + 3][32] per direction) instead of once per tap.
//   * accumulators: gates 2 x 224 + y 64 TMEM columns.  Warp 0: TMA + MMA issue (one elected lane), warp 1: TMEM owner,
//     warps 2-9: point-wise update (thread = sequence x half of the CTA's units), cell state in registers.
#include <cuda.h>
#include "common.cuh"
#include "tc05.cuh"

namespace fdbm {
namespace {

using namespace tc05;

constexpr int UPC = 56;                    // hidden-unit slots per CTA (2 x 56 = 112 = 7 k16 steps)
constexpr int NG = 4 * UPC;                // 224 gate columns per CTA: [7 chunks][i f g o][8 units]
constexpr int NY = 64;                     // ConvTranspose1d columns per CTA: taps 2r, 2r+1
constexpr int RING = 6;
constexpr int TC_THREADS = 320;              // warp 0 TMA + MMA, warp 1 TMEM owner, warps 2-9 point-wise
// shared-memory image (bytes); every tile base is 1024-byte aligned
constexpr int OFF_WU = 0;                                  // 4 taps x [224 x 64 B]   SWIZZLE_64B
constexpr int WU_TILE = NG * 64;                           // 14336
constexpr int OFF_WH = OFF_WU + 4 * WU_TILE;               // 2 K-blocks x [224 x 128 B] SWIZZLE_128B
constexpr int WH_TILE = NG * 128;                          // 28672
constexpr int OFF_WL = OFF_WH + 2 * WH_TILE;               // 2 K-blocks x [64 x 128 B]
constexpr int WL_TILE = NY * 128;                          // 8192
constexpr int W_IMAGE_BYTES = OFF_WL + 2 * WL_TILE;        // 131072: what fdbm_tfg_lstm_pack produces per (direction, cta rank)
constexpr int OFF_U = W_IMAGE_BYTES;                       // ring of 5 x [128 x 64 B] SWIZZLE_64B
constexpr int U_TILE = 128 * 64;                           // 8192
constexpr int OFF_H = OFF_U + RING * U_TILE;               // 2 K-blocks x [128 x 128 B] SWIZZLE_128B
constexpr int H_TILE = 128 * 128;                          // 16384
constexpr int OFF_BAR = OFF_H + 2 * H_TILE;
constexpr int TC_SMEM = OFF_BAR + 256;
static_assert(OFF_WH % 1024 == 0 && OFF_WL % 1024 == 0 && OFF_U % 1024 == 0 && OFF_H % 1024 == 0, "tile alignment");
static_assert(TC_SMEM <= 232448, "shared memory");

__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(layout_type) << 61;           // 2 = SWIZZLE_128B, 4 = SWIZZLE_64B
  return d;
}
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ uint32_t map_to_peer(uint32_t local_addr, uint32_t rank) {
  uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank)); return r;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
// 4 KB of this CTA's shared memory -> the same offset in the peer's, completing on the peer's mbarrier (async proxy on both sides)
__device__ __forceinline__ void bulk_copy_to_peer(uint32_t dst_cluster, uint32_t src_cta, uint32_t bytes, uint32_t bar_cluster) {
  asm volatile("cp.async.bulk.shared::cluster.shared::cta.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_cluster), "r"(src_cta), "r"(bytes),
               "r"(bar_cluster) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory"); }
__device__ __forceinline__ void mma_commit_pair(uint64_t* bar) {                    // arrive on this barrier in BOTH CTAs of the cluster
  const uint16_t mask = 3;
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask)
               : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ float tanh_fast(float x) { float r; asm("tanh.approx.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ uint32_t pack_h2(float a, float b) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }

// byte offset of (row, 16-byte chunk) inside a K-major tile with 64-byte rows (SWIZZLE_64B) / 128-byte rows (SWIZZLE_128B)
__host__ __device__ inline int sw64_off(int row, int chunk) { return row * 64 + ((chunk ^ ((row >> 1) & 3)) << 4); }
__host__ __device__ inline int sw128_off(int row, int chunk) { return row * 128 + ((chunk ^ (row & 7)) << 4); }

// column of the h tile (K index of the recurrent GEMM) that holds hidden unit u: K-block r = the 56 units CTA r computes (+ 8 pad
// columns), so each 16 KB K-block is written by ONE CTA and travels to the peer as plain bulk copies; u = 112: the constant 1
__host__ __device__ inline int h_col(int u) { return u == 112 ? 120 : 64 * (u / UPC) + u % UPC; }

// ---- weight image: reference layout -> the shared-memory image of one (direction, cta rank) ----------------------------------
// gate column n = chunk * 32 + gate * 8 + j  <->  unit = 56 rank + 8 chunk + j, PyTorch row gate * H + unit (i, f, g, o)
__global__ void pack_lstm_tc_kernel(const float* __restrict__ w_ih, const float* __restrict__ w_hh, const float* __restrict__ b_ih,
                                    const float* __restrict__ b_hh, const float* __restrict__ w_lin, int H, int dir, int rank,
                                    uint8_t* __restrict__ img) {
  // (the image was zeroed by the caller: pad rows / columns stay 0)
  // one thread per (n, k) of the gate matrix, k in 0..239 (+ the bias row k = 240 -> h column 120)
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < NG * 241; e += gridDim.x * blockDim.x) {
    const int n = e / 241, k = e % 241;
    const int chunk = n >> 5, gate = (n >> 3) & 3, j = n & 7;
    const int unit = UPC * rank + 8 * chunk + j;
    float v = 0.f;
    int off;
    if (k < 128) {                                   // input feature tap * 32 + c  <- weight_ih[row][c * 4 + tap]
      const int tap = k >> 5, c = k & 31;
      if (unit < H) v = w_ih[(gate * H + unit) * 128 + c * 4 + tap];
      off = OFF_WU + tap * WU_TILE + sw64_off(n, c >> 3) + (c & 7) * 2;
    } else {
      const int hu = k - 128;                        // hidden unit 0..111, or 112 = the bias row
      if (unit < H) v = hu < H ? w_hh[(gate * H + unit) * H + hu] : (hu == 112 ? b_ih[gate * H + unit] + b_hh[gate * H + unit] : 0.f);
      const int hk = h_col(hu);
      off = OFF_WH + (hk >> 6) * WH_TILE + sw128_off(n, (hk & 63) >> 3) + (hk & 7) * 2;
    }
    if (gate != 2) v *= 0.5f;                        // i, f, o: the kernel evaluates sigmoid(x) as 0.5 tanh(x / 2) + 0.5
    *reinterpret_cast<__half*>(img + off) = __float2half_rn(v);
  }
  // ConvTranspose1d [2H, C, ks]: rows dir * H + unit; this CTA's columns n = half * 32 + tap * 8 + j for channels
  // c = 8 (2 rank + half) + j: one 32-column TMEM load = the four taps of 8 channels
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < NY * 112; e += gridDim.x * blockDim.x) {
    const int n = e / 112, hu = e % 112, hk = h_col(hu);
    const int tap = (n >> 3) & 3, c = 8 * (2 * rank + (n >> 5)) + (n & 7);
    const float v = hu < H ? w_lin[((dir * H + hu) * 32 + c) * 4 + tap] : 0.f;
    *reinterpret_cast<__half*>(img + OFF_WL + (hk >> 6) * WL_TILE + sw128_off(n, (hk & 63) >> 3) + (hk & 7) * 2) = __float2half_rn(v);
  }
}

struct TcArgs {
  int n_seq, L;
  const uint8_t* img[2][2];            // [direction][cta rank]
  __half* y[2];                        // [direction]: [n_seq][L + 3][32], ConvTranspose1d taps overlap-added
};

// The input half of step i + 1's gates (which does not depend on h_i) is issued right behind step i's commit into the
// second gate accumulator, so it runs under step i's point-wise update.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1)
lstm_sweep_tc_kernel(const __grid_constant__ CUtensorMap map_x, const TcArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  if (smem_u32(smem) & 1023u) __trap();
  const uint32_t rank = cluster_rank();
  const int dir = blockIdx.y, tile = blockIdx.x >> 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + OFF_BAR);
  uint64_t* u_full = bars;                         // [RING]  TMA -> MMA lane
  uint64_t* mma_done = bars + RING;                // [2] both CTAs' gate MMAs of a step are complete, per column slice -> point-wise warps
  uint64_t* y_done = bars + RING + 2;              // both CTAs' ConvTranspose1d MMAs (the last readers of h_{i-1}) are complete
  uint64_t* h_local = bars + RING + 3;             // this CTA's K-block of h_i is stored (4 row groups) -> MMA lane
  uint64_t* h_peer = bars + RING + 4;              // the peer's K-block of h_i has arrived (16 KB of bulk copies) -> MMA lane
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + RING + 5);
  const int L = a.L, n_loads = L + 3;
  const bool rev = dir == 1;

  // ---- one-time setup: weight image -> shared memory, h tile = 0 with the constant-1 column, barriers, TMEM
  {
    const uint4* src = reinterpret_cast<const uint4*>(a.img[dir][rank]);
    uint4* dst = reinterpret_cast<uint4*>(smem);
    for (int i = threadIdx.x; i < W_IMAGE_BYTES / 16; i += TC_THREADS) dst[i] = __ldg(src + i);
    uint4* hz = reinterpret_cast<uint4*>(smem + OFF_H);
    for (int i = threadIdx.x; i < 2 * H_TILE / 16; i += TC_THREADS) hz[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  if (threadIdx.x < 128) {                         // h column 120 (K-block 1, chunk 7, element 0) = 1.0 for every row
    const int r = threadIdx.x;
    *reinterpret_cast<__half*>(smem + OFF_H + H_TILE + sw128_off(r, 7)) = __float2half(1.0f);
  }
  if (threadIdx.x == 0) {
    for (int i = 0; i < RING; ++i) mbar_init(u_full + i, 1);
    mbar_init(mma_done, 2);
    mbar_init(mma_done + 1, 2);
    mbar_init(y_done, 2);
    mbar_init(h_local, 4);
    mbar_init(h_peer, 1);                          // the arming arrive; the data counts as transaction bytes
    fence_barrier_init();
    mbar_expect_tx(h_peer, H_TILE);                // phase 0: the peer's K-block arrives as 4 x 4 KB bulk copies
    tma_prefetch_desc(&map_x);
  }
  if (warp == 1) { tmem_alloc(tmem_slot, 512); tmem_relinquish(); }
  fence_proxy_all();                               // generic-proxy writes of the tiles -> visible to the tensor core
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  cluster_sync_all();                              // both CTAs initialised before anyone touches the peer's h tile / barriers

  const uint32_t s_base = smem_u32(smem);
  const int seq0 = tile * 128;
  // position of load number q (see the sweep order): forward q, reverse (L + 2) - q
  auto pos_of = [&](int q) { return rev ? (L + 2) - q : q; };
  auto gate_acc = [&](int i) { return tmem_base + (i & 1) * NG; };
  const uint32_t tmem_y = tmem_base + 2 * NG;

  if (warp == 0) {
    // ------------------------------------------------------------------ TMA producer + MMA issuer (whole warp walks, one lane issues)
    // gate columns in two slices (chunks 0..3 / 4..6 = the two point-wise warp sets), each with its own commit: the first
    // set starts on its columns while the tensor core still computes the second's
    constexpr int N0 = 128, N1 = NG - N0;
    constexpr uint32_t idesc_g = make_idesc_f16(128, NG, 0), idesc_y = make_idesc_f16(128, NY, 0);
    constexpr uint32_t idesc_s[2] = {make_idesc_f16(128, N0, 0), make_idesc_f16(128, N1, 0)};
    auto load_u = [&](int q) {
      if (q < n_loads) {
        mbar_expect_tx(u_full + q % RING, U_TILE);
        tma_load_3d(smem + OFF_U + (q % RING) * U_TILE, &map_x, u_full + q % RING, 0, pos_of(q), seq0);
      }
    };
    auto wait_u = [&](int q) { mbar_wait(u_full + q % RING, (q / RING) & 1); };
    auto issue_u_part = [&](int i) {               // gates(i) = sum over taps u_{s + tap} W_tap: first write of the accumulator
      uint32_t acc = 0;
#pragma unroll
      for (int tap = 0; tap < 4; ++tap) {
        const int q = rev ? i + 3 - tap : i + tap;                 // load number holding position s + tap
        const uint32_t a_addr = s_base + OFF_U + (q % RING) * U_TILE, b_addr = s_base + OFF_WU + tap * WU_TILE;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          mma_f16(gate_acc(i), make_desc(a_addr + 32 * k, 512, 4), make_desc(b_addr + 32 * k, 512, 4), idesc_g, acc);
          acc = 1;
        }
      }
    };
    auto issue_h_part = [&](int i, int kb, int slice) {      // columns of `slice` += K-block kb of [h_{i-1} | 1] [W_hh ; b]
#pragma unroll
      for (int k = 0; k < 4; ++k)
        mma_f16(gate_acc(i) + slice * N0, make_desc(s_base + OFF_H + kb * H_TILE + 32 * k, 1024, 2),
                make_desc(s_base + OFF_WH + kb * WH_TILE + slice * N0 * 128 + 32 * k, 1024, 2), idesc_s[slice], 1u);
    };
    auto issue_y = [&]() {                         // y = h W_lin
#pragma unroll
      for (int kk = 0; kk < 8; ++kk) {
        const int kb = kk >> 2, k = kk & 3;
        mma_f16(tmem_y, make_desc(s_base + OFF_H + kb * H_TILE + 32 * k, 1024, 2), make_desc(s_base + OFF_WL + kb * WL_TILE + 32 * k, 1024, 2),
                idesc_y, kk > 0 ? 1u : 0u);
      }
    };
    constexpr int ahead = 5;                       // loads in flight / resident beyond step i's first position
    if (elect_one()) for (int q = 0; q < ahead; ++q) load_u(q);
    __syncwarp();
    for (int q = 0; q < 4; ++q) wait_u(q);
    fence_after_sync();
    if (elect_one()) issue_u_part(0);
    __syncwarp();
    for (int i = 0; i < L; ++i) {
      const int mine = static_cast<int>(rank), theirs = mine ^ 1;
      // this CTA's own K-block of h_{i-1} is complete first (no transfer): its MMAs run while the peer's K-block is in flight.
      // (h_local also says this CTA's point-wise warps have read their accumulators of step i - 1.)
      if (i > 0) mbar_wait(h_local, (i - 1) & 1);
      fence_after_sync();
      if (elect_one()) {
        issue_h_part(i, mine, 0);
        issue_h_part(i, mine, 1);
      }
      __syncwarp();
      if (i > 0) {
        mbar_wait(h_peer, (i - 1) & 1);
        // the ring slot of load i - 1 + ahead was last read by input MMAs that completed before the commit the point-wise warps waited on
        if (elect_one()) { mbar_expect_tx(h_peer, H_TILE); load_u(i - 1 + ahead); }
        __syncwarp();
      }
      fence_after_sync();
      if (elect_one()) {
        issue_h_part(i, theirs, 0);
        mma_commit_pair(mma_done);
        issue_h_part(i, theirs, 1);
        mma_commit_pair(mma_done + 1);
        if (i > 0) issue_y();                                     // y_{i-1}: behind the gates, off the recurrence
        mma_commit_pair(y_done);                                  // = every reader of h_{i-1} (both slices, y) is done
      }
      __syncwarp();
      if (i + 1 < L) {
        wait_u(i + 4);
        fence_after_sync();
        if (elect_one()) issue_u_part(i + 1);
        __syncwarp();
      }
    }
    mbar_wait(h_local, (L - 1) & 1);
    mbar_wait(h_peer, (L - 1) & 1);
    fence_after_sync();
    if (elect_one()) { issue_y(); mma_commit_pair(y_done); }      // tail: y_{L-1}
    __syncwarp();
  } else if (warp >= 2) {
    // ------------------------------------------------------------------ point-wise update: thread = (sequence row, half of the units)
    const int qd = warp & 3;                       // TMEM lane quadrant this warp may access
    const int half = (warp - 2) >> 2;              // chunks 0..3 / 4..6 of the CTA's seven 8-unit chunks; output channels 8 (2 rank + half) ..
    const int row = qd * 32 + lane;
    const int seq = seq0 + row;
    const bool ok = seq < a.n_seq;
    const uint32_t lane_sel = (static_cast<uint32_t>(qd) * 32u) << 16;
    // this CTA's K-block of the h tile, the 4 KB of this warp pair's 32 rows in it, and the same place in the peer
    const uint32_t h_mine = s_base + OFF_H + rank * H_TILE;
    const uint32_t h_rows = h_mine + qd * 4096, h_rows_peer = map_to_peer(h_rows, rank ^ 1);
    const uint32_t ready_peer = map_to_peer(smem_u32(h_peer), rank ^ 1);
    float c[32];
#pragma unroll
    for (int u = 0; u < 32; ++u) c[u] = 0.f;
    // ConvTranspose1d overlap-add: position p = s + tap.  part[k] = what has arrived so far for the k-th next position to complete.
    float part[3][8];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int j = 0; j < 8; ++j) part[k][j] = 0.f;
    __half* yrow = a.y[dir] + (static_cast<int64_t>(ok ? seq : 0) * (L + 3)) * 32 + 8 * (2 * static_cast<int>(rank) + half);
    auto put = [&](int pos, const float (&o)[8]) {
      if (ok) *reinterpret_cast<uint4*>(yrow + static_cast<int64_t>(pos) * 32) =
          make_uint4(pack_h2(o[0], o[1]), pack_h2(o[2], o[3]), pack_h2(o[4], o[5]), pack_h2(o[6], o[7]));
    };
    auto emit = [&](int i_prev, const uint32_t (&v)[32]) {        // v = y of step i_prev: [tap][8 channels]
      const int s = rev ? L - 1 - i_prev : i_prev;
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        // forward: position s is complete with tap 0; reverse: position s + 3 with tap 3
        const float t0 = __uint_as_float(rev ? v[24 + j] : v[j]), t1 = __uint_as_float(rev ? v[16 + j] : v[8 + j]);
        const float t2 = __uint_as_float(rev ? v[8 + j] : v[16 + j]), t3 = __uint_as_float(rev ? v[j] : v[24 + j]);
        o[j] = part[0][j] + t0;
        part[0][j] = part[1][j] + t1;
        part[1][j] = part[2][j] + t2;
        part[2][j] = t3;
      }
      put(rev ? s + 3 : s, o);
    };
    uint32_t yv[32];
    for (int i = 0; i < L; ++i) {
      mbar_wait(mma_done + half, i & 1);
      fence_after_sync();
      const uint32_t t_g = gate_acc(i) + lane_sel;
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        const int ch = 4 * half + c4;
        if (ch < 7) {
          uint32_t v[32];
          tmem_ld_32x32(t_g + 32 * ch, v);
          tmem_ld_wait();
          float hv[8];
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            // i, f, o arrive pre-halved: sigmoid(x) = 0.5 tanh(x / 2) + 0.5
            const float ig = fmaf(tanh_fast(__uint_as_float(v[j])), 0.5f, 0.5f), fg = fmaf(tanh_fast(__uint_as_float(v[8 + j])), 0.5f, 0.5f);
            const float gg = tanh_fast(__uint_as_float(v[16 + j])), og = fmaf(tanh_fast(__uint_as_float(v[24 + j])), 0.5f, 0.5f);
            const float cn = fmaf(fg, c[8 * c4 + j], ig * gg);
            c[8 * c4 + j] = cn;
            hv[j] = og * tanh_fast(cn);
          }
          const uint4 pk = make_uint4(pack_h2(hv[0], hv[1]), pack_h2(hv[2], hv[3]), pack_h2(hv[4], hv[5]), pack_h2(hv[6], hv[7]));
          // h_{i-1} may be overwritten once both CTAs' MMAs of this step (the other slice, y_{i-1}) are done with it
          if (c4 == 0) { mbar_wait(y_done, i & 1); fence_after_sync(); }
          st_shared_v4(h_mine + sw128_off(row, ch), pk);          // hidden units 56 rank + 8 ch .. + 7 = chunk ch of this CTA's K-block
        }
      }
      if (i > 0) { tmem_ld_32x32(tmem_y + lane_sel + 32 * half, yv); tmem_ld_wait(); }
      fence_before_sync();                         // TMEM reads done before the next MMAs overwrite the accumulators
      fence_proxy_async();                         // h stores (generic proxy) -> visible to the async proxy (UMMA, bulk copy)
      named_bar_sync(1 + qd, 64);                  // both warps of this row group
      if (half == 0 && lane == 0) {
        bulk_copy_to_peer(h_rows_peer, h_rows, 4096, ready_peer);
        mbar_arrive(h_local);
      }
      if (i > 0) emit(i - 1, yv);                  // the global store sits behind the hand-off: its latency is off the recurrence
    }
    mbar_wait(y_done, L & 1);
    fence_after_sync();
    tmem_ld_32x32(tmem_y + lane_sel + 32 * half, yv);
    tmem_ld_wait();
    fence_before_sync();
    emit(L - 1, yv);
    // the three edge positions that never complete: forward L .. L + 2, reverse 2 .. 0
#pragma unroll
    for (int k = 0; k < 3; ++k) put(rev ? 2 - k : L + k, part[k]);
  }
  __syncthreads();
  cluster_sync_all();                              // nobody exits while the peer may still write into its shared memory
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                             const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeFn get_encode_tc() {
  static EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeFn>(p);
  }
  return fn;
}

}  // namespace
}  // namespace fdbm

using namespace fdbm;

extern "C" int64_t fdbm_tfg_lstm_pack_bytes(void) { return 4ll * W_IMAGE_BYTES; }        // [direction][cta rank]

// Both directions of one nn.LSTM + its ConvTranspose1d -> the four shared-memory images of the tcgen05 sweep.
extern "C" int fdbm_tfg_lstm_pack(const float* const* w /* fw: w_ih w_hh b_ih b_hh | bw: ... (8 device pointers) */, const float* w_lin, int hidden,
                                     void* packed, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(w && w_lin && packed && hidden >= 8 && hidden <= 112, "fdbm_tfg_lstm_pack: bad arguments (hidden units 8..112)");
  FDBM_CUDA(cudaMemsetAsync(packed, 0, 4ull * W_IMAGE_BYTES, as_stream(stream)));
  for (int d = 0; d < 2; ++d)
    for (int r = 0; r < 2; ++r) {
      pack_lstm_tc_kernel<<<64, 256, 0, as_stream(stream)>>>(w[4 * d], w[4 * d + 1], w[4 * d + 2], w[4 * d + 3], w_lin, hidden, d, r,
                                                             reinterpret_cast<uint8_t*>(packed) + static_cast<int64_t>(2 * d + r) * W_IMAGE_BYTES);
      FDBM_LAUNCH_CHECK();
    }
  return FDBM_OK;
}

// One bidirectional sweep.  xn: fp16 [n_seq][n_pos = L + 3][32] contiguous; y_fw / y_bw: fp16 [n_seq][L + 3][32] (taps overlap-added).
extern "C" int fdbm_tfg_lstm_sweep(const void* xn, int n_seq, int L, const void* packed, void* y_fw, void* y_bw, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(xn && packed && y_fw && y_bw && n_seq > 0 && L > 0, "fdbm_tfg_lstm_sweep: bad arguments");
  EncodeFn enc = get_encode_tc();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return FDBM_ECUDA; }
  CUtensorMap map;
  cuuint64_t dims[3] = {32, static_cast<cuuint64_t>(L + 3), static_cast<cuuint64_t>(n_seq)};
  cuuint64_t strides[2] = {64, static_cast<cuuint64_t>(L + 3) * 64};
  cuuint32_t box[3] = {32, 1, 128};
  cuuint32_t es[3] = {1, 1, 1};
  CUresult r = enc(&map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(xn), dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled(lstm input [%d,%d,32]) failed: %d", n_seq, L + 3, (int)r); return FDBM_ECUDA; }
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device()))
    FDBM_CUDA(cudaFuncSetAttribute(lstm_sweep_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM));
  TcArgs a;
  a.n_seq = n_seq; a.L = L;
  for (int d = 0; d < 2; ++d)
    for (int rk = 0; rk < 2; ++rk) a.img[d][rk] = reinterpret_cast<const uint8_t*>(packed) + static_cast<int64_t>(2 * d + rk) * W_IMAGE_BYTES;
  a.y[0] = reinterpret_cast<__half*>(y_fw); a.y[1] = reinterpret_cast<__half*>(y_bw);
  dim3 grid(2 * ceil_div(n_seq, 128), 2);
  lstm_sweep_tc_kernel<<<grid, TC_THREADS, TC_SMEM, as_stream(stream)>>>(map, a);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}
