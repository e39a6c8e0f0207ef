// Fast STFT + compression (+ pad_spec, + peak normalisation) and de-compression + iSTFT kernels for n_fft = 512.
// Same arithmetic as spectral.cu (fdbm/data_module.py:173-229, fdbm/util/other.py:76-90) restructured for the
// instruction budget: the first version was issue-bound (ncu: DRAM bytes = algorithmic bytes, issue slots 61-65 % busy,
// 2.2 / 1.3 TB/s), i.e. these kernels only reach the HBM roofline if one frame costs < ~400 warp-instructions.
//
//   * one warp transforms FOUR real frames as TWO 512-point complex FFTs (frames a, a+1 -> FFT A re/im; a+2, a+3 -> FFT
//     B), held as structure-of-arrays pairs (re_A, re_B), (im_A, im_B): every butterfly and twiddle product is one packed
//     fp32x2 instruction (FADD2 / FMUL2 / FFMA2) for both transforms, complex products need no swizzles;
//   * consecutive frames overlap by n_fft - hop samples: the 4 frames of a warp are framed from 16 + 3 hop/32 sample
//     loads per lane instead of 64;
//   * the radix-2 combine of the last stage is done by the consumer on read (no shuffles);
//   * spectra leave / enter through a shared-memory tile [257 bins][16 frames] so that every global access of the
//     [B,1,257,T] layout is a full 128-byte line (the direct version issued 16-byte pieces of 32 different lines per
//     store instruction);
//   * twiddles come from a compile-time table (tw512.inc, rounded from double), not from sincospif per block;
//   * peak normalisation (infer_single.py:83-87: y / max|y|) is folded into the compression scale -- the STFT is linear,
//     spec(y / n) = spec(y) / n -- and the inverse kernel applies the `* norm` rescale and records max|x_hat| per
//     utterance for the clip rule (infer_folder.py:119-120), so `enhance` needs no elementwise ATen pass.
//   * iSTFT: overlap-add in registers (three of a warp's four hop segments never leave it; the fourth takes the
//     previous warp's trailing half-frame through 1 KB of shared memory).
#include "common.cuh"

namespace fdbm {
namespace {

constexpr int NFFT = 512;
constexpr int NBIN = NFFT / 2 + 1;
// Warps per block.  A block stages [257 bins][4 * FWARPS frames] and moves it with 32 * FWARPS contiguous bytes per bin.
// Measured (256 x 4 s, B200): 2 / 4 / 8 / 16 warps -> STFT 89 / 88 / 102-118 / 133 us, iSTFT 162 / 136-155 / 157-178 / 145 us.  The
// kernels issue 2.5 x / 4 x fewer instructions than the first generation (ncu: 25.9 M vs 64 M warp instructions for the STFT)
// but are now latency-bound: ~100 registers per thread allow 16-20 warps per SM, issue slots are 20 % busy, a warp issues
// every 20 cycles, 37 % of the stall cycles are the block barriers around the staging tile -- larger blocks make that worse,
// more resident blocks (a launch-bounds minimum of 5 or 6 per SM) change nothing or spill.  Dropping the staging tile and its two block barriers
// (every lane writing the 32 contiguous bytes = 4 frames of its bins straight from registers) was measured too: 1.79 TB/s
// instead of 2.16 (96 registers), 1.53 with 80 registers / 6 blocks, 1.69 / 1.76 with 8 / 2 warps -- 16-byte pieces of 32
// different lines per store instruction cost more than the barriers they remove.
constexpr int FWARPS = 4;
constexpr int MIN_BLOCKS = 5;             // resident blocks per SM the register allocation must allow
constexpr int FPW = 4;                    // frames per warp
constexpr int FRB = FWARPS * FPW;         // frames per block
constexpr int LPL = FRB / 2;              // lanes (16-byte pieces = 2 frames) per bin line; 32 * FWARPS / LPL = 16 bins per pass
constexpr int WPITCH = 34;                // exchange buffer: 16 rows of 32 + 2 (float4 units)
constexpr int G1_OFF = 260;               // second-stage layout: g0[idx] at idx, g1[idx] at 260 + idx (conflict-free both ways)
constexpr int TILE_PITCH = FRB + 2;       // staging tile [257][18] float2: 144-byte rows -> conflict-free 16-byte accesses
constexpr int WORK_F4 = 16 * WPITCH;      // 544 float4 per warp
constexpr int UNION_BYTES = NBIN * TILE_PITCH * 8 > FWARPS * WORK_F4 * 16 ? NBIN * TILE_PITCH * 8 : FWARPS * WORK_F4 * 16;

__device__ const float2 kTw512[NFFT] = {
#include "tw512.inc"
};

// packed-pair twiddles (c, c, s, s) of exp(-+2 pi i m / 512), [0] forward, [1] inverse (filled once per device; read from
// global memory, L1-resident, 9 KB):  [32 k1 + lane] = W_512^(lane k1) (inter-stage, one row per k1 so that a lane's 15 reads
// are immediate offsets from one address);  [512 + 16 h + K] = h ? W_32^K : 1 (radix-2 split of the last stage);
// [544 + M] = W_32^M (the 16-point transform's constants)
__device__ float4 g_tw_packed[2][NFFT + 64];

struct FastSmem {
  union {
    float4 work[FWARPS][WORK_F4];
    float2 tile[NBIN][TILE_PITCH];
    uint8_t raw[UNION_BYTES];
  } u;
  float tail[FWARPS][NFFT / 2];           // iSTFT: trailing half-frame of every warp
  float red[FWARPS];
};

// two complex numbers (one of FFT A, one of FFT B) as structure of arrays
struct PC { float2 re, im; };

#define DI __device__ __forceinline__
DI float2 f2(float a, float b) { return make_float2(a, b); }
// MUFU.RSQ, 2^-22.4 relative error (`__frsqrt_rn` is the correctly rounded form: ~20 instructions)
DI float rsqrt_fast(float x) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
DI PC padd(const PC& a, const PC& b) { return PC{__fadd2_rn(a.re, b.re), __fadd2_rn(a.im, b.im)}; }
DI PC psub(const PC& a, const PC& b) { return PC{__ffma2_rn(b.re, f2(-1.f, -1.f), a.re), __ffma2_rn(b.im, f2(-1.f, -1.f), a.im)}; }
DI PC p_sub_i(const PC& a, const PC& b) { return PC{__fadd2_rn(a.re, b.im), __ffma2_rn(b.re, f2(-1.f, -1.f), a.im)}; }   // a - i b
DI PC p_add_i(const PC& a, const PC& b) { return PC{__ffma2_rn(b.im, f2(-1.f, -1.f), a.re), __fadd2_rn(a.im, b.re)}; }   // a + i b
DI PC pmul(const PC& v, float c, float s) {                                                                             // v (c + i s)
  return PC{__ffma2_rn(v.im, f2(-s, -s), __fmul2_rn(v.re, f2(c, c))), __ffma2_rn(v.im, f2(c, c), __fmul2_rn(v.re, f2(s, s)))};
}
DI PC pmul4(const PC& v, const float4& w) {                                                                             // w = (c, c, s, s)
  return PC{__ffma2_rn(v.im, f2(-w.z, -w.w), __fmul2_rn(v.re, f2(w.x, w.y))), __ffma2_rn(v.im, f2(w.x, w.y), __fmul2_rn(v.re, f2(w.z, w.w)))};
}

__host__ __device__ constexpr double cq(int m) {
  return m == 0 ? 1.0 : m == 1 ? 0.98078528040323044913 : m == 2 ? 0.92387953251128675613 : m == 3 ? 0.83146961230254523708
       : m == 4 ? 0.70710678118654752440 : m == 5 ? 0.55557023301960222474 : m == 6 ? 0.38268343236508977173
       : m == 7 ? 0.19509032201612826785 : 0.0;
}
__host__ __device__ constexpr double c32(int m) {
  m = ((m % 32) + 32) % 32;
  return m <= 8 ? cq(m) : m <= 16 ? -cq(16 - m) : m <= 24 ? -cq(m - 16) : cq(32 - m);
}
__host__ __device__ constexpr double s32(int m) { return c32(m - 8); }

// times W_32^M = exp(-+2 pi i M / 32) = tw[16 M]: the packed (c, c, s, s) entry comes from the twiddle table -- with
// immediate constants the compiler falls back to scalar FMUL / FFMA (8 instructions per product pair instead of 4 + 1 load)
template <bool INV, int M>
DI PC mul_w32(const PC& v, const float4* tw) {
  if (M % 32 == 0) return v;
  return pmul4(v, tw[NFFT + 32 + (((M % 32) + 32) % 32)]);
}

template <bool INV>
DI void fft4(PC& x0, PC& x1, PC& x2, PC& x3) {
  const PC a = padd(x0, x2), b = psub(x0, x2), c = padd(x1, x3), d = psub(x1, x3);
  x0 = padd(a, c);
  x2 = psub(a, c);
  if (!INV) { x1 = p_sub_i(b, d); x3 = p_add_i(b, d); }
  else      { x1 = p_add_i(b, d); x3 = p_sub_i(b, d); }
}

__host__ __device__ constexpr int pos16(int k) { return 4 * (k & 3) + (k >> 2); }
// 16-point DFT, natural-order input, X[k] left in v[pos16(k)]
template <bool INV>
DI void fft16(PC (&v)[16], const float4* tw) {
#pragma unroll
  for (int n2 = 0; n2 < 4; ++n2) fft4<INV>(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);
  const float4* t32 = tw + NFFT + 32;                 // W_32^M, M = 0..31
  const float4 w2 = t32[2], w4 = t32[4], w6 = t32[6], w12 = t32[12];
  v[5] = pmul4(v[5], w2);   v[6] = pmul4(v[6], w4);    v[7] = pmul4(v[7], w6);
  v[9] = pmul4(v[9], w4);
  // W_32^8 = -+ i
  v[10] = INV ? PC{__ffma2_rn(v[10].im, f2(-1.f, -1.f), f2(0.f, 0.f)), v[10].re} : PC{v[10].im, __ffma2_rn(v[10].re, f2(-1.f, -1.f), f2(0.f, 0.f))};
  v[11] = pmul4(v[11], w12);
  v[13] = pmul4(v[13], w6); v[14] = pmul4(v[14], w12); v[15] = mul_w32<INV, 18>(v[15], tw);
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1) fft4<INV>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
}

template <bool INV, int K>
DI void w32_row(PC (&v)[16], const float4* tw_odd) {     // odd lanes: v[pos16(K)] *= W_32^K, K = 1..15; even lanes read 1
  if constexpr (K < 16) {
    v[pos16(K)] = pmul4(v[pos16(K)], tw_odd[K]);
    w32_row<INV, K + 1>(v, tw_odd);
  }
}

// Two 512-point complex DFTs per warp.  In: lane holds u[32 j + lane] in v[j].  Out (in `work`, 544 float4 of this warp):
//   g0[idx] at work[idx], g1[idx] at work[260 + idx], idx = 0..255, with U[idx] = g0 + g1 and U[256 + idx] = g0 - g1.
// n = 32 n1 + n2, k = k1 + 16 k2; the 32-point transform over n2 is split radix-2 (even / odd n2 in lane pairs).
template <bool INV>
DI void fft512_pair(PC (&v)[16], float4* work, const float4* tw, int lane) {
  fft16<INV>(v, tw);
#pragma unroll
  for (int k1 = 0; k1 < 16; ++k1) {
    const PC t = k1 == 0 ? v[pos16(0)] : pmul4(v[pos16(k1)], tw[32 * k1 + lane]);      // table row k1: W_512^(lane k1)
    work[k1 * WPITCH + lane] = make_float4(t.re.x, t.re.y, t.im.x, t.im.y);
  }
  __syncwarp();
  const int k1 = lane >> 1, h = lane & 1;
#pragma unroll
  for (int m = 0; m < 16; ++m) {
    const float4 e = work[k1 * WPITCH + h + 2 * m];
    v[m] = PC{f2(e.x, e.y), f2(e.z, e.w)};
  }
  __syncwarp();
  fft16<INV>(v, tw);
  w32_row<INV, 1>(v, tw + NFFT + h * 16);          // rows 512.. of the table: [0..15] = 1 (even lanes), [16..31] = W_32^K (odd lanes)
  float4* dst = work + h * G1_OFF + k1;
#pragma unroll
  for (int k2 = 0; k2 < 16; ++k2) {
    const PC& f = v[pos16(k2)];
    dst[16 * k2] = make_float4(f.re.x, f.re.y, f.im.x, f.im.y);
  }
  __syncwarp();
}

__global__ void fill_tw_global_kernel() {
  for (int m = threadIdx.x; m < NFFT + 64; m += blockDim.x) {
    int idx;
    if (m < NFFT) idx = ((m & 31) * (m >> 5)) & 511;                       // lane * k1
    else if (m < NFFT + 32) idx = m < NFFT + 16 ? 0 : 16 * (m - NFFT - 16);  // 1 (even lanes) | W_32^K (odd lanes)
    else idx = 16 * (m - NFFT - 32);                                        // W_32^M
    const float2 w = kTw512[idx];
    g_tw_packed[0][m] = make_float4(w.x, w.x, w.y, w.y);
    g_tw_packed[1][m] = make_float4(w.x, w.x, -w.y, -w.y);
  }
}

DI int pad_source(int t, int M, int pad_mode) {
  if (t < M) return t;
  if (pad_mode == FDBM_PAD_REFLECTION) return 2 * (M - 1) - t;
  if (pad_mode == FDBM_PAD_REPLICATION) return M - 1;
  return -1;
}

// scale applied to a spectrum value z (|z|^2 = m2) by spec_fwd: the returned factor times z is the compressed value.
// `pre` multiplies z first (1/2 of the Hermitian separation and 1/norm of the peak normalisation).
// MODE 0: no transform, 1: exponent 1 (factor only), 2: the default |z|^0.5 compression, 3: anything else (out of line)
__device__ __noinline__ float compress_scale_generic(float m2, int transform, float factor, float expo, float pre) {
  const float mag = sqrtf(m2) * pre;
  if (transform == FDBM_TRANSFORM_EXPONENT) return mag > 0.f ? powf(mag, expo) / mag * factor * pre : 0.f;
  return mag > 0.f ? log1pf(mag) / mag * factor * pre : 0.f;
}
template <int MODE>
DI float compress_scale(float m2, int transform, float factor, float expo, float pre, float k_half) {
  if (MODE == 0) return pre;
  if (MODE == 1) return pre * factor;
  if (MODE == 2) {
    // factor (pre |z|)^0.5 / |z| = factor sqrt(pre) m2^(-1/4): two MUFU ops, z = 0 stays 0 (0 * finite)
    const float r = rsqrt_fast(fmaxf(m2, 1e-30f));        // 1 / |z|
    return k_half * (r * rsqrt_fast(r));                  // sqrt(1 / |z|)
  }
  return compress_scale_generic(m2, transform, factor, expo, pre);
}

// ------------------------------------------------------------------------------------------------------------------
// STFT + compression.  HS = hop / 32 (8 for hop 256, 4 for hop 128).
// ------------------------------------------------------------------------------------------------------------------
template <int HS, int MODE>
__global__ void __launch_bounds__(FWARPS * 32, MIN_BLOCKS)
stft_fast_kernel(const float* __restrict__ wave, int n_samples, const int* __restrict__ lengths, int64_t wave_stride,
                 const float* __restrict__ window, const float* __restrict__ norm, int transform, float factor, float expo,
                 int pad_mode, int M, int n_frames_out, float2* __restrict__ spec) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  FastSmem& sm = *reinterpret_cast<FastSmem*>(smem_raw);
  constexpr int hop = HS * 32;
  constexpr int NRAW = 16 + (FPW - 1) * HS;
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * FRB;
  const float* x = wave + static_cast<int64_t>(b) * wave_stride;
  if (lengths) { n_samples = __ldg(lengths + b); M = 1 + n_samples / hop; }
  const int ta = t0 + FPW * warp;
  int src[FPW];
  bool any = false, plain = true;
#pragma unroll
  for (int f = 0; f < FPW; ++f) {
    src[f] = ta + f < n_frames_out ? pad_source(ta + f, M, pad_mode) : -1;
    any |= src[f] >= 0;
    plain &= src[f] == ta + f;
  }
  const int p0 = ta * hop - NFFT / 2;
  plain = plain && p0 >= 0 && p0 + NFFT + (FPW - 1) * hop <= n_samples;     // warp-uniform
  PC v[16];
  if (any) {
    float w[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) w[j] = __ldg(window + 32 * j + lane);
    if (plain) {
      float raw[NRAW];
      const float* xp = x + p0 + lane;
#pragma unroll
      for (int r = 0; r < NRAW; ++r) raw[r] = __ldg(xp + 32 * r);
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        v[j].re = __fmul2_rn(f2(raw[j], raw[j + 2 * HS]), f2(w[j], w[j]));
        v[j].im = __fmul2_rn(f2(raw[j + HS], raw[j + 3 * HS]), f2(w[j], w[j]));
      }
    } else {                                   // first / last frames (reflect padding) and pad_spec's extra frames:
      // a rolled loop through this warp's exchange buffer (3 of the 64 warps of a 4 s utterance come here; unrolled, this
      // path was 8000 instructions of address arithmetic in the instruction cache)
      float* stage = reinterpret_cast<float*>(sm.u.work[warp]);                // [4 frames][512]
#pragma unroll 1
      for (int f = 0; f < FPW; ++f) {
        const int sf = f == 0 ? src[0] : (f == 1 ? src[1] : (f == 2 ? src[2] : src[3]));
#pragma unroll 1
        for (int j = 0; j < 16; ++j) {
          float val = 0.f;
          if (sf >= 0) {
            int p = sf * hop - NFFT / 2 + 32 * j + lane;
            if (p < 0) p = -p;
            if (p >= n_samples) p = 2 * (n_samples - 1) - p;
            val = __ldg(x + p);
          }
          stage[f * NFFT + 32 * j + lane] = val;
        }
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int n = 32 * j + lane;
        v[j].re = __fmul2_rn(f2(stage[n], stage[2 * NFFT + n]), f2(w[j], w[j]));
        v[j].im = __fmul2_rn(f2(stage[NFFT + n], stage[3 * NFFT + n]), f2(w[j], w[j]));
      }
      __syncwarp();
    }
  }
  const float4* twp = g_tw_packed[0];
  float4* work = sm.u.work[warp];
  if (any) fft512_pair<false>(v, work, twp, lane);
  // Hermitian separation + compression, results kept in registers until every warp has finished reading its exchange buffer
  // (the staging tile aliases those buffers).  With Z = (frame0 + i frame1): F0[k] = (Z[k] + conj Z[N-k]) / 2,
  // F1[k] = (Z[k] - conj Z[N-k]) / (2i); the 1/2 goes into the compression scale.
  const float inv_norm = norm ? 1.0f / __ldg(norm + b) : 1.0f;
  const float pre = 0.5f * inv_norm;
  const float k_half = factor * sqrtf(pre);
  // frames that pad_spec fills with zeros must come out as EXACT zeros: the two frames of one complex FFT leak ~1e-7 of
  // each other through rounding, which the square-root compression would blow up to ~1e-4
  const float k0 = src[0] >= 0 ? 1.f : 0.f, k1m = src[1] >= 0 ? 1.f : 0.f, k2m = src[2] >= 0 ? 1.f : 0.f, k3m = src[3] >= 0 ? 1.f : 0.f;
  float4 outA[9], outB[9];                      // (F0.re, F0.im, F1.re, F1.im) of FFT A (frames ta, ta+1) and B (ta+2, ta+3)
  // one bin: p = U[k] = g0[ip] + sp g1[ip], q = U[N - k] = g0[iq] + sq g1[iq]
  auto bin = [&](const float4& a0, const float4& a1, const float4& b0, const float4& b1, float sp, float sq, float4& oA, float4& oB) {
    const float2 p_re = __ffma2_rn(f2(a1.x, a1.y), f2(sp, sp), f2(a0.x, a0.y)), p_im = __ffma2_rn(f2(a1.z, a1.w), f2(sp, sp), f2(a0.z, a0.w));
    const float2 q_re = __ffma2_rn(f2(b1.x, b1.y), f2(sq, sq), f2(b0.x, b0.y)), q_im = __ffma2_rn(f2(b1.z, b1.w), f2(sq, sq), f2(b0.z, b0.w));
    // 2 F0 = (p.re + q.re, p.im - q.im);  2 F1 = (p.im + q.im, q.re - p.re)
    const float2 f0re = __fadd2_rn(p_re, q_re), f0im = __ffma2_rn(q_im, f2(-1.f, -1.f), p_im);
    const float2 f1re = __fadd2_rn(p_im, q_im), f1im = __ffma2_rn(p_re, f2(-1.f, -1.f), q_re);
    const float2 m0 = __ffma2_rn(f0im, f0im, __fmul2_rn(f0re, f0re)), m1 = __ffma2_rn(f1im, f1im, __fmul2_rn(f1re, f1re));
    const float s0a = compress_scale<MODE>(m0.x, transform, factor, expo, pre, k_half) * k0, s0b = compress_scale<MODE>(m0.y, transform, factor, expo, pre, k_half) * k2m;
    const float s1a = compress_scale<MODE>(m1.x, transform, factor, expo, pre, k_half) * k1m, s1b = compress_scale<MODE>(m1.y, transform, factor, expo, pre, k_half) * k3m;
    oA = make_float4(f0re.x * s0a, f0im.x * s0a, f1re.x * s1a, f1im.x * s1a);
    oB = make_float4(f0re.y * s0b, f0im.y * s0b, f1re.y * s1b, f1im.y * s1b);
  };
  if (any) {
    // bins k = lane + 32 i, i < 8: g(k) and g(256 - k) are immediate offsets from two per-lane addresses; only k = 0 (lane 0,
    // i = 0: q = U[0] = g0 + g1 at index 0) and k = 256 (lane 0 alone: p = q = U[256] = g0[0] - g1[0]) are special
    const float4* gp = work + lane;
    const float4* gq = work + (lane == 0 ? 0 : 256 - lane);
    {
      const float sq0 = lane == 0 ? 1.f : -1.f;
      bin(gp[0], gp[G1_OFF], gq[0], gq[G1_OFF], 1.f, sq0, outA[0], outB[0]);
    }
    const float4* gq2 = work + 256 - lane;
#pragma unroll
    for (int i = 1; i < 8; ++i) bin(gp[32 * i], gp[G1_OFF + 32 * i], gq2[-32 * i], gq2[G1_OFF - 32 * i], 1.f, -1.f, outA[i], outB[i]);
    outA[8] = make_float4(0.f, 0.f, 0.f, 0.f); outB[8] = outA[8];
    if (lane == 0) bin(work[0], work[G1_OFF], work[0], work[G1_OFF], -1.f, -1.f, outA[8], outB[8]);
  } else {
#pragma unroll
    for (int i = 0; i < 9; ++i) { outA[i] = make_float4(0.f, 0.f, 0.f, 0.f); outB[i] = outA[i]; }
  }
  __syncthreads();                              // all exchange buffers consumed: the tile may overwrite them
  {
    float4* row = reinterpret_cast<float4*>(&sm.u.tile[lane][FPW * warp]);
    constexpr int STEP = 32 * TILE_PITCH / 2;   // 32 bins further, in float4 units
#pragma unroll
    for (int i = 0; i < 8; ++i) { row[i * STEP] = outA[i]; row[i * STEP + 1] = outB[i]; }
    if (lane == 0) { row[8 * STEP] = outA[8]; row[8 * STEP + 1] = outB[8]; }
  }
  __syncthreads();
  // write-out: 128 contiguous bytes per bin (16 frames); 8 lanes of 16 bytes per line, 16 bins per pass of the block
  const int n_valid = min(FRB, n_frames_out - t0);             // frames of this block inside the output
  float2* out = spec + static_cast<int64_t>(b) * NBIN * n_frames_out + t0;
  if ((n_frames_out & 1) == 0) {
    const int c = (threadIdx.x % LPL) * 2, kb = threadIdx.x / LPL;
    if (c < n_valid) {                                         // n_valid is even here
      const float4* tp = reinterpret_cast<const float4*>(&sm.u.tile[kb][c]);
      float4* gp = reinterpret_cast<float4*>(out + static_cast<int64_t>(kb) * n_frames_out + c);
      const int64_t gstep = static_cast<int64_t>(8) * n_frames_out;      // 16 bins further, in float4 units
#pragma unroll 4
      for (int it = 0; it < 16; ++it) gp[it * gstep] = tp[it * (16 * TILE_PITCH / 2)];
      if (kb == 0) gp[16 * gstep] = tp[16 * (16 * TILE_PITCH / 2)];       // bin 256
    }
  } else {
    for (int e = threadIdx.x; e < NBIN * FRB; e += FWARPS * 32) {
      const int k = e / FRB, c = e % FRB;
      if (c < n_valid) out[static_cast<int64_t>(k) * n_frames_out + c] = sm.u.tile[k][c];
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------
// de-compression + iSTFT for hop = n_fft / 2 (two frames per output sample).  A block inverts 16 consecutive frames
// m0 .. m0 + 15 and completes the 15 hop segments between them (segment s = second half of frame s - 1 + first half of
// frame s); consecutive blocks overlap by one frame.
// ------------------------------------------------------------------------------------------------------------------
__device__ __noinline__ float2 decompress_generic(float2 z, int transform, float factor, float expo) {
  z.x = z.x / factor; z.y = z.y / factor;
  const float mag = sqrtf(z.x * z.x + z.y * z.y);
  float s;
  if (transform == FDBM_TRANSFORM_EXPONENT) s = mag > 0.f ? powf(mag, 1.0f / expo) / mag : 0.f;
  else s = mag > 0.f ? expm1f(mag) / mag : 0.f;
  return make_float2(z.x * s, z.y * s);
}
template <int MODE>
DI float2 decompress1(float2 z, float inv, int transform, float factor, float expo) {
  if (MODE == 0) return z;
  if (MODE <= 2) {
    z.x *= inv; z.y *= inv;
    if (MODE == 2) {                              // |z|^2 e^{j angle z} = z |z|
      const float m2 = fmaf(z.x, z.x, z.y * z.y);
      const float mag = m2 * rsqrt_fast(fmaxf(m2, 1e-30f));
      z.x *= mag; z.y *= mag;
    }
    return z;
  }
  return decompress_generic(z, transform, factor, expo);
}

template <int MODE>
__global__ void __launch_bounds__(FWARPS * 32, MIN_BLOCKS)
istft_fast_kernel(const float2* __restrict__ spec, int M, const float* __restrict__ window, int transform, float factor, float expo,
                  int64_t length, const int* __restrict__ lengths, int64_t wave_stride, const float* __restrict__ norm,
                  float* __restrict__ peak, float* __restrict__ wave) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  FastSmem& sm = *reinterpret_cast<FastSmem*>(smem_raw);
  constexpr int hop = NFFT / 2;
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  if (lengths) length = __ldg(lengths + b);
  const int m0 = blockIdx.x * (FRB - 1) - 1;      // first frame of the block (frame -1 does not exist: zeros)
  const float2* in = spec + static_cast<int64_t>(b) * NBIN * M;
  const float inv = 1.0f / factor;
  // ---- spectra tile [257][16 frames], de-compressed on the way in (each value once; the Hermitian extension below reads
  //      every bin twice), imaginary parts of DC / Nyquist dropped (irfft semantics)
  auto prep = [&](float2 z, int k) {
    z = decompress1<MODE>(z, inv, transform, factor, expo);
    if (k == 0 || k == NFFT / 2) z.y = 0.f;
    return z;
  };
  if ((M & 1) == 0) {
    // 16-byte loads of frame pairs (m, m + 1), m even; blocks with an odd first frame start one frame early (9 pairs per bin)
    const int shift = m0 & 1, ncol = LPL + shift;
    for (int e = threadIdx.x; e < NBIN * ncol; e += FWARPS * 32) {
      const int k = shift ? e / (LPL + 1) : e / LPL, c = (e - k * ncol) * 2 - shift, m = m0 + c;
      float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
      if (m >= 0 && m + 1 < M) val = __ldg(reinterpret_cast<const float4*>(in + static_cast<int64_t>(k) * M + m));
      if (c >= 0) sm.u.tile[k][c] = prep(make_float2(val.x, val.y), k);
      if (c + 1 < FRB) sm.u.tile[k][c + 1] = prep(make_float2(val.z, val.w), k);
    }
  } else {
    for (int e = threadIdx.x; e < NBIN * FRB; e += FWARPS * 32) {
      const int k = e / FRB, c = e % FRB, m = m0 + c;
      sm.u.tile[k][c] = (m >= 0 && m < M) ? prep(__ldg(in + static_cast<int64_t>(k) * M + m), k) : make_float2(0.f, 0.f);
    }
  }
  const float4* twp = g_tw_packed[1];
  __syncthreads();
  // ---- Z_A = F0 + i F1, Z_B = F2 + i F3 with Hermitian extension: bins k > 256 are the conjugates of bin 512 - k
  PC v[16];
  {
    const float4* lo_row = reinterpret_cast<const float4*>(&sm.u.tile[lane][FPW * warp]);            // bin 32 j + lane, j < 8
    const float4* hi_row = reinterpret_cast<const float4*>(&sm.u.tile[256 - lane][FPW * warp]);      // bin 512 - (256 + 32 j + lane)
    constexpr int STEP = 32 * TILE_PITCH / 2;
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float4 e0 = j < 8 ? lo_row[j * STEP] : hi_row[-(j - 8) * STEP], e1 = j < 8 ? lo_row[j * STEP + 1] : hi_row[-(j - 8) * STEP + 1];
      // e = (F0.re, F0.im, F1.re, F1.im | F2.re, F2.im, F3.re, F3.im);  Z = F_even + i F_odd  (conjugated for j >= 8)
      if (j < 8) {
        v[j].re = f2(e0.x - e0.w, e1.x - e1.w);
        v[j].im = f2(e0.y + e0.z, e1.y + e1.z);
      } else {
        v[j].re = f2(e0.x + e0.w, e1.x + e1.w);
        v[j].im = f2(e0.z - e0.y, e1.z - e1.y);
      }
    }
  }
  __syncthreads();                                // tile consumed by every warp: the exchange buffers may overwrite it
  float4* work = sm.u.work[warp];
  fft512_pair<true>(v, work, twp, lane);
  // ---- time samples n = 32 j + lane (j < 8) and n + 256 of the four frames, windowed, 1/N
  float w[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) w[j] = __ldg(window + 32 * j + lane);
  float lo[FPW][8], hi[FPW][8];                   // first / second half of frames 4 warp + f
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 g0 = work[32 * j + lane], g1 = work[G1_OFF + 32 * j + lane];
    const float wl = w[j] * (1.0f / NFFT), wh = w[j + 8] * (1.0f / NFFT);
    lo[0][j] = (g0.x + g1.x) * wl; lo[2][j] = (g0.y + g1.y) * wl; lo[1][j] = (g0.z + g1.z) * wl; lo[3][j] = (g0.w + g1.w) * wl;
    hi[0][j] = (g0.x - g1.x) * wh; hi[2][j] = (g0.y - g1.y) * wh; hi[1][j] = (g0.z - g1.z) * wh; hi[3][j] = (g0.w - g1.w) * wh;
  }
  // frames outside [0, M) contribute nothing (their spectra were loaded as zeros -> lo / hi are zero already)
#pragma unroll
  for (int j = 0; j < 8; ++j) sm.tail[warp][32 * j + lane] = hi[3][j];
  __syncthreads();
  const float scale_out = norm ? __ldg(norm + b) : 1.0f;
  float* out = wave + static_cast<int64_t>(b) * wave_stride;
  float pk = 0.f;
#pragma unroll
  for (int f = 0; f < FPW; ++f) {
    const int fb = FPW * warp + f;                 // block-relative frame whose FIRST half ends this segment
    if (fb == 0) continue;                         // its predecessor belongs to the previous block (warp-uniform)
    const int m = m0 + fb;                         // absolute frame: segment covers samples (m - 1) * hop + [0, hop) of the un-padded signal
    const bool has_cur = m >= 0 && m < M, has_prev = m - 1 >= 0 && m - 1 < M;
    if (!has_cur && !has_prev) continue;
    const int64_t n0 = static_cast<int64_t>(m) * hop - NFFT / 2;
    const float e_prev = has_prev ? 1.f : 0.f, e_cur = has_cur ? 1.f : 0.f;
    const bool inside = n0 >= 0 && n0 + hop <= length;       // warp-uniform: the whole segment is stored
    float* op = out + n0 + lane;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float prev = f == 0 ? sm.tail[warp == 0 ? 0 : warp - 1][32 * j + lane] : hi[f == 0 ? 0 : f - 1][j];
      const float acc = prev + lo[f][j];           // oldest frame first (fold order of torch.istft)
      const float env = fmaf(e_prev * w[j + 8], w[j + 8], e_cur * w[j] * w[j]);     // window envelope of the frames that exist
      // torch.istft divides by the envelope; MUFU.RCP + multiply is within 2 ulp of that quotient
      const float val = env > 1e-11f ? __fdividef(acc, env) * scale_out : 0.f;
      if (inside) {
        op[32 * j] = val;
        pk = fmaxf(pk, fabsf(val));
      } else {
        const int64_t n = n0 + 32 * j + lane;
        if (n >= 0 && n < length) { op[32 * j] = val; pk = fmaxf(pk, fabsf(val)); }
      }
    }
  }
  if (peak) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) pk = fmaxf(pk, __shfl_xor_sync(0xffffffffu, pk, o));
    if (lane == 0 && pk > 0.f) atomicMax(reinterpret_cast<int*>(peak + b), __float_as_int(pk));   // non-negative floats order like ints
  }
}

// max |x| per utterance (peak normalisation, infer_single.py:83-87); `out` must be zeroed
__global__ void __launch_bounds__(256)
absmax_kernel(const float* __restrict__ wave, int64_t n_samples, const int* __restrict__ lengths, int64_t stride, float* __restrict__ out) {
  const int b = blockIdx.y;
  const int64_t n = lengths ? __ldg(lengths + b) : n_samples;
  const float* x = wave + static_cast<int64_t>(b) * stride;
  float m = 0.f;
  const bool vec = (stride & 3) == 0 && (reinterpret_cast<uintptr_t>(wave) & 15) == 0;
  if (vec) {
    const int64_t n4 = n >> 2;
    for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n4; i += 256ll * gridDim.x) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(x) + i);
      m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    }
    for (int64_t i = (n4 << 2) + blockIdx.x * 256ll + threadIdx.x; i < n; i += 256ll * gridDim.x) m = fmaxf(m, fabsf(__ldg(x + i)));
  } else {
    for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += 256ll * gridDim.x) m = fmaxf(m, fabsf(__ldg(x + i)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(reinterpret_cast<int*>(out + b), __float_as_int(m));
}

// clip rule of the infer scripts (infer_single.py:95-97 with 0.5, infer_folder.py:119-120 with 0.95):
// if max|x| > 1: x <- x / max|x| * rescale.  Blocks of utterances that do not clip return after one 4-byte read.
__global__ void __launch_bounds__(256)
clip_rescale_kernel(float* __restrict__ wave, int64_t n_samples, const int* __restrict__ lengths, int64_t stride,
                    const float* __restrict__ peak, float rescale) {
  const int b = blockIdx.y;
  const float pk = __ldg(peak + b);
  if (!(pk > 1.0f)) return;
  const int64_t n = lengths ? __ldg(lengths + b) : n_samples;
  float* x = wave + static_cast<int64_t>(b) * stride;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += 256ll * gridDim.x) x[i] = x[i] / pk * rescale;
}

}  // namespace

bool spectral_fast_supported(int n_fft, int hop, bool inverse) {
  if (n_fft != NFFT) return false;
  return inverse ? hop == NFFT / 2 : (hop == 256 || hop == 128);
}

static int ensure_tw_table(cudaStream_t s) {
  static PerDeviceOnce once;
  if (once.first(current_device())) {
    fill_tw_global_kernel<<<1, 256, 0, s>>>();
    FDBM_LAUNCH_CHECK();
  }
  return FDBM_OK;
}

static int transform_mode(int transform, float expo) {
  return transform == FDBM_TRANSFORM_NONE ? 0 : (transform == FDBM_TRANSFORM_EXPONENT ? (expo == 1.0f ? 1 : (expo == 0.5f ? 2 : 3)) : 3);
}

template <int HS, int MODE>
static int stft_fast_launch(dim3 grid, cudaStream_t s, const float* wave, int n_samples, const int* lengths, int64_t wave_stride,
                            const float* window, const float* norm, int transform, float factor, float expo, int pad_mode, int M,
                            int n_frames_out, float2* spec) {
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device()))
    FDBM_CUDA(cudaFuncSetAttribute(stft_fast_kernel<HS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastSmem)));
  stft_fast_kernel<HS, MODE><<<grid, FWARPS * 32, sizeof(FastSmem), s>>>(wave, n_samples, lengths, wave_stride, window, norm, transform, factor,
                                                                         expo, pad_mode, M, n_frames_out, spec);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_stft_fast(const float* wave, int batch, int64_t max_samples, const int* lengths, int64_t wave_stride, const float* window,
                     const float* norm, int hop, int transform, float factor, float expo, int pad_mode, int M, int n_frames_out,
                     float* spec, cudaStream_t s) {
  dim3 grid(ceil_div(n_frames_out, FRB), batch);
  if (int rc = ensure_tw_table(s)) return rc;
  const int mode = transform_mode(transform, expo), ns = static_cast<int>(max_samples);
  float2* out = reinterpret_cast<float2*>(spec);
#define FDBM_STFT_CASE(HS_, MODE_)                                                                                                     \
  if (hop == 32 * HS_ && mode == MODE_)                                                                                                \
    return stft_fast_launch<HS_, MODE_>(grid, s, wave, ns, lengths, wave_stride, window, norm, transform, factor, expo, pad_mode, M, n_frames_out, out);
  FDBM_STFT_CASE(8, 2) FDBM_STFT_CASE(8, 0) FDBM_STFT_CASE(8, 1) FDBM_STFT_CASE(8, 3)
  FDBM_STFT_CASE(4, 2) FDBM_STFT_CASE(4, 0) FDBM_STFT_CASE(4, 1) FDBM_STFT_CASE(4, 3)
#undef FDBM_STFT_CASE
  set_error("stft_fast: unsupported hop %d", hop);
  return FDBM_EINVAL;
}

template <int MODE>
static int istft_fast_launch(dim3 grid, cudaStream_t s, const float2* spec, int n_frames, const float* window, int transform, float factor,
                             float expo, int64_t length, const int* lengths, int64_t wave_stride, const float* norm, float* peak, float* wave) {
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device()))
    FDBM_CUDA(cudaFuncSetAttribute(istft_fast_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FastSmem)));
  istft_fast_kernel<MODE><<<grid, FWARPS * 32, sizeof(FastSmem), s>>>(spec, n_frames, window, transform, factor, expo, length, lengths, wave_stride,
                                                                      norm, peak, wave);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_istft_fast(const float* spec, int batch, int n_frames, const float* window, int transform, float factor, float expo,
                      int64_t length, const int* lengths, int64_t wave_stride, const float* norm, float* peak, float* wave, cudaStream_t s) {
  // segments 1 .. ceil((length + n_fft/2) / hop) of the padded timeline; block x completes segments 15 x .. 15 x + 14
  const int64_t n_seg = ceil_div64(length + NFFT / 2, NFFT / 2);
  dim3 grid(static_cast<unsigned>(ceil_div64(n_seg + 1, FRB - 1)), batch);
  if (peak) FDBM_CUDA(cudaMemsetAsync(peak, 0, sizeof(float) * batch, s));
  if (int rc = ensure_tw_table(s)) return rc;
  const float2* in = reinterpret_cast<const float2*>(spec);
  switch (transform_mode(transform, expo)) {
    case 0: return istft_fast_launch<0>(grid, s, in, n_frames, window, transform, factor, expo, length, lengths, wave_stride, norm, peak, wave);
    case 1: return istft_fast_launch<1>(grid, s, in, n_frames, window, transform, factor, expo, length, lengths, wave_stride, norm, peak, wave);
    case 2: return istft_fast_launch<2>(grid, s, in, n_frames, window, transform, factor, expo, length, lengths, wave_stride, norm, peak, wave);
    default: return istft_fast_launch<3>(grid, s, in, n_frames, window, transform, factor, expo, length, lengths, wave_stride, norm, peak, wave);
  }
}

int launch_absmax(const float* wave, int batch, int64_t n_samples, const int* lengths, int64_t stride, float* out, cudaStream_t s) {
  FDBM_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * batch, s));
  const int bx = std::max(1, std::min<int>(static_cast<int>(ceil_div64(n_samples, 256 * 16)), std::max(1, num_sms() * 8 / batch)));
  absmax_kernel<<<dim3(bx, batch), 256, 0, s>>>(wave, n_samples, lengths, stride, out);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_clip_rescale(float* wave, int batch, int64_t n_samples, const int* lengths, int64_t stride, const float* peak, float rescale,
                        cudaStream_t s) {
  const int bx = std::max(1, std::min<int>(static_cast<int>(ceil_div64(n_samples, 256 * 8)), std::max(1, num_sms() * 8 / batch)));
  clip_rescale_kernel<<<dim3(bx, batch), 256, 0, s>>>(wave, n_samples, lengths, stride, peak, rescale);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

}  // namespace fdbm
