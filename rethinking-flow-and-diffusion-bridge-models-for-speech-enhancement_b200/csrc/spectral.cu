// Fused STFT + amplitude compression (+ pad_spec) and its inverse (de-compression + iSTFT
// overlap-add).  Replaces fdbm/data_module.py:173-229 and fdbm/util/other.py:76-90.
//
// One warp transforms TWO real frames as one 512-point complex FFT (frame a -> re, frame b -> im,
// separated afterwards by Hermitian symmetry).  The FFT lives in registers: 512 = 16 x 32, every lane
// holds 16 complex values; a 16-point transform in registers (radix 4 x 4, compile-time twiddles), one
// padded shared-memory transposition, a second 16-point transform, and a radix-2 combine with the
// neighbouring lane by shuffle.  A block of 8 warps covers 16 consecutive frames; every warp writes its two
// frames as 16-byte pieces of the (contiguous) frame axis of the reference layout [B,1,257,T] and the eight
// warps of the block complete each 128-byte line in L2.  HBM-bound: 4 B/sample read, 8 B/bin written.
#include "common.cuh"

namespace fdbm {
bool spectral_fast_supported(int n_fft, int hop, bool inverse);
int launch_stft_fast(const float* wave, int batch, int64_t max_samples, const int* lengths, int64_t wave_stride, const float* window,
                     const float* norm, int hop, int transform, float factor, float expo, int pad_mode, int M, int n_frames_out,
                     float* spec, cudaStream_t s);
int launch_istft_fast(const float* spec, int batch, int n_frames, const float* window, int transform, float factor, float expo,
                      int64_t length, const int* lengths, int64_t wave_stride, const float* norm, float* peak, float* wave, cudaStream_t s);
int launch_absmax(const float* wave, int batch, int64_t n_samples, const int* lengths, int64_t stride, float* out, cudaStream_t s);
int launch_clip_rescale(float* wave, int batch, int64_t n_samples, const int* lengths, int64_t stride, const float* peak, float rescale,
                        cudaStream_t s);
namespace {

// The first-generation kernels below serve the hops the fast kernels (spectral_fast.cu) do not cover.

constexpr int NFFT = 512;
constexpr int NBIN = NFFT / 2 + 1;
constexpr int FR = 16;            // frames per block (two per warp)
constexpr int WARPS = 8;
constexpr int MAXR = 4;           // n_fft / hop <= 4
constexpr int WORK = 16 * 34;     // per-warp exchange buffer (float2): 16 rows of 32 + 2 padding; also 512 in natural order

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
  return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }

// cos(2 pi m / 32), sin(2 pi m / 32), m = 0..8 (first quadrant); the rest by symmetry at compile time
__host__ __device__ constexpr double cos32q(int m) {
  return m == 0 ? 1.0 : m == 1 ? 0.98078528040323044913 : m == 2 ? 0.92387953251128675613 : m == 3 ? 0.83146961230254523708
       : m == 4 ? 0.70710678118654752440 : m == 5 ? 0.55557023301960222474 : m == 6 ? 0.38268343236508977173
       : m == 7 ? 0.19509032201612826785 : 0.0;
}
__host__ __device__ constexpr double cos32(int m) {          // any m
  m = ((m % 32) + 32) % 32;
  return m <= 8 ? cos32q(m) : m <= 16 ? -cos32q(16 - m) : m <= 24 ? -cos32q(m - 16) : cos32q(32 - m);
}
__host__ __device__ constexpr double sin32(int m) { return cos32(m - 8); }
// W_32^m = exp(-2 pi i m / 32) (forward) or its conjugate (inverse)
template <bool INV, int M>
__device__ __forceinline__ float2 mul_w32(float2 v) {
  constexpr float c = static_cast<float>(cos32(M)), s = static_cast<float>(INV ? sin32(M) : -sin32(M));
  if (M % 32 == 0) return v;
  return make_float2(v.x * c - v.y * s, v.x * s + v.y * c);
}

template <bool INV>
__device__ __forceinline__ void fft4(float2& x0, float2& x1, float2& x2, float2& x3) {
  const float2 a = cadd(x0, x2), b = csub(x0, x2), c = cadd(x1, x3), d = csub(x1, x3);
  x0 = cadd(a, c);
  x2 = csub(a, c);
  if (!INV) { x1 = make_float2(b.x + d.y, b.y - d.x); x3 = make_float2(b.x - d.y, b.y + d.x); }   // b -+ i d
  else      { x1 = make_float2(b.x - d.y, b.y + d.x); x3 = make_float2(b.x + d.y, b.y - d.x); }
}

// 16-point DFT in registers, n = 4 n1 + n2, k = k1 + 4 k2.  Input natural order; output X[k] is left in
// v[4 * (k & 3) + (k >> 2)] (use fft16_pos).
__host__ __device__ constexpr int fft16_pos(int k) { return 4 * (k & 3) + (k >> 2); }
template <bool INV>
__device__ __forceinline__ void fft16(float2 (&v)[16]) {
#pragma unroll
  for (int n2 = 0; n2 < 4; ++n2) fft4<INV>(v[n2], v[4 + n2], v[8 + n2], v[12 + n2]);
  // v[4 k1 + n2] *= W_16^(n2 k1) = W_32^(2 n2 k1)
  v[5] = mul_w32<INV, 2>(v[5]);  v[6] = mul_w32<INV, 4>(v[6]);   v[7] = mul_w32<INV, 6>(v[7]);
  v[9] = mul_w32<INV, 4>(v[9]);  v[10] = mul_w32<INV, 8>(v[10]); v[11] = mul_w32<INV, 12>(v[11]);
  v[13] = mul_w32<INV, 6>(v[13]); v[14] = mul_w32<INV, 12>(v[14]); v[15] = mul_w32<INV, 18>(v[15]);
#pragma unroll
  for (int k1 = 0; k1 < 4; ++k1) fft4<INV>(v[4 * k1], v[4 * k1 + 1], v[4 * k1 + 2], v[4 * k1 + 3]);
}

template <bool INV, int K>
__device__ __forceinline__ void w32_row(float2 (&v)[16], bool odd) {   // odd lanes: v[pos(k)] *= W_32^k for k = K..15
  if constexpr (K < 16) {                                              // (select, no branch: shuffles follow)
    constexpr float c = static_cast<float>(cos32(K)), s = static_cast<float>(INV ? sin32(K) : -sin32(K));
    const float cc = odd ? c : 1.0f, ss = odd ? s : 0.0f;
    const float2 x = v[fft16_pos(K)];
    v[fft16_pos(K)] = make_float2(x.x * cc - x.y * ss, x.x * ss + x.y * cc);
    w32_row<INV, K + 1>(v, odd);
  }
}

// 512-point complex DFT of a warp.  In: lane holds u[32 j + lane] in v[j], j = 0..15.  Out: `work` (WORK float2
// of shared memory owned by the warp) holds U[k] in natural order, k = 0..511.  tw[m] = exp(-2 pi i m / 512).
//   n = 32 n1 + n2, k = k1 + 16 k2:  U[k] = sum_{n2} W_512^(n2 k1) W_32^(n2 k2) sum_{n1} u[32 n1 + n2] W_16^(n1 k1)
//   the 32-point transform over n2 is split n2 = h + 2 m, k2 = k2' + 16 c: a 16-point transform per (k1, h) lane and
//   a radix-2 combine with lane ^ 1.
template <bool INV>
__device__ __forceinline__ void fft512_warp(float2 (&v)[16], float2* work, const float2* tw, int lane) {
  fft16<INV>(v);
#pragma unroll
  for (int k1 = 0; k1 < 16; ++k1) {
    float2 w = tw[(lane * k1) & 511];
    if (INV) w.y = -w.y;
    work[k1 * 34 + lane] = k1 == 0 ? v[fft16_pos(0)] : cmul(v[fft16_pos(k1)], w);
  }
  __syncwarp();
  const int k1 = lane >> 1, h = lane & 1;
#pragma unroll
  for (int m = 0; m < 16; ++m) v[m] = work[k1 * 34 + h + 2 * m];
  __syncwarp();
  fft16<INV>(v);
  w32_row<INV, 1>(v, h != 0);                        // odd half: times W_32^(k2')
#pragma unroll
  for (int k2 = 0; k2 < 16; ++k2) {
    const float2 f = v[fft16_pos(k2)];
    float2 pr;
    pr.x = __shfl_xor_sync(0xffffffffu, f.x, 1);
    pr.y = __shfl_xor_sync(0xffffffffu, f.y, 1);
    work[k1 + 16 * k2 + 256 * h] = h ? csub(pr, f) : cadd(f, pr);
  }
  __syncwarp();
}

__device__ __forceinline__ float2 compress(float2 z, int transform, float factor, float expo) {
  if (transform == FDBM_TRANSFORM_NONE) return z;
  const float mag = sqrtf(z.x * z.x + z.y * z.y);
  float s;
  if (transform == FDBM_TRANSFORM_EXPONENT) {
    if (expo == 1.0f) s = factor;
    else if (mag > 0.f) s = (expo == 0.5f ? rsqrtf(mag) : powf(mag, expo) / mag) * factor;
    else s = 0.f;
  } else {  // log
    s = mag > 0.f ? log1pf(mag) / mag * factor : 0.f;
  }
  return make_float2(z.x * s, z.y * s);
}

__device__ __forceinline__ float2 decompress(float2 z, int transform, float factor, float expo) {
  if (transform == FDBM_TRANSFORM_NONE) return z;
  z.x = z.x / factor;
  z.y = z.y / factor;
  const float mag = sqrtf(z.x * z.x + z.y * z.y);
  float s;
  if (transform == FDBM_TRANSFORM_EXPONENT) {
    if (expo == 1.0f) s = 1.f;
    else if (mag > 0.f) s = (expo == 0.5f ? mag : powf(mag, 1.0f / expo) / mag);
    else s = 0.f;
  } else {
    s = mag > 0.f ? expm1f(mag) / mag : 0.f;
  }
  return make_float2(z.x * s, z.y * s);
}

// frame index a padded output frame copies from (pad_spec, other.py:76-90); -1 = zeros
__device__ __forceinline__ int pad_source(int t, int M, int pad_mode) {
  if (t < M) return t;
  if (pad_mode == FDBM_PAD_REFLECTION) return 2 * (M - 1) - t;
  if (pad_mode == FDBM_PAD_REPLICATION) return M - 1;
  return -1;
}

struct SpecSmem {
  float2 tw[NFFT];
  float2 work[WARPS][WORK];
};

__device__ __forceinline__ void fill_twiddles(float2* tw) {
  for (int m = threadIdx.x; m < NFFT; m += WARPS * 32) {
    float s, c;
    sincospif(static_cast<float>(m) / 256.0f, &s, &c);
    tw[m] = make_float2(c, -s);
  }
}

__global__ void __launch_bounds__(WARPS * 32)
stft_compress_kernel(const float* __restrict__ wave, int n_samples, const int* __restrict__ lengths, int64_t wave_stride,
                     const float* __restrict__ window, int hop, int transform, float factor, float expo,
                     int pad_mode, int M, int n_frames_out, float2* __restrict__ spec) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  SpecSmem& sm = *reinterpret_cast<SpecSmem*>(smem_raw);
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  const int b = blockIdx.y;
  const int t0 = blockIdx.x * FR;
  const float* x = wave + static_cast<int64_t>(b) * wave_stride;
  if (lengths) {                                        // variable-length batch: this utterance's own sample / frame count
    n_samples = __ldg(lengths + b);
    M = 1 + n_samples / hop;
  }

  float2* z = sm.work[warp];
  const int ta = t0 + 2 * warp, tb = ta + 1;
  const int sa = ta < n_frames_out ? pad_source(ta, M, pad_mode) : -1;
  const int sb = tb < n_frames_out ? pad_source(tb, M, pad_mode) : -1;
  const bool any = sa >= 0 || sb >= 0;                 // warp-uniform
  float2 v[16];
  if (any) {
    const int pa0 = sa * hop - NFFT / 2, pb0 = sb * hop - NFFT / 2;     // centred framing
    if (sa >= 0 && sb >= 0 && min(pa0, pb0) >= 0 && max(pa0, pb0) + NFFT <= n_samples) {
      const float* xa = x + pa0 + lane;                 // both frames inside the signal: plain coalesced loads
      const float* xb = x + pb0 + lane;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float w = __ldg(window + 32 * j + lane);
        v[j] = make_float2(__ldg(xa + 32 * j) * w, __ldg(xb + 32 * j) * w);
      }
    } else {                                            // first / last frames: reflect padding
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const int n = 32 * j + lane;
        const float w = __ldg(window + n);
        float va = 0.f, vb = 0.f;
        if (sa >= 0) {
          int p = pa0 + n;
          if (p < 0) p = -p;
          if (p >= n_samples) p = 2 * (n_samples - 1) - p;
          va = __ldg(x + p) * w;
        }
        if (sb >= 0) {
          int p = pb0 + n;
          if (p < 0) p = -p;
          if (p >= n_samples) p = 2 * (n_samples - 1) - p;
          vb = __ldg(x + p) * w;
        }
        v[j] = make_float2(va, vb);
      }
    }
  }
  fill_twiddles(sm.tw);                                 // (after the loads are in flight)
  __syncthreads();
  if (any) fft512_warp<false>(v, z, sm.tw, lane);
  if (ta >= n_frames_out) return;
  // Hermitian separation of the two spectra, compression, 16-byte stores (frames ta, ta+1 of bin k)
  float2* out = spec + static_cast<int64_t>(b) * NBIN * n_frames_out + ta;
  const bool pair = tb < n_frames_out && (n_frames_out & 1) == 0;      // 16-byte aligned pair store
#pragma unroll 1
  for (int k = lane; k < NBIN; k += 32) {
    float2 A = make_float2(0.f, 0.f), Bv = A;
    if (any) {
      const float2 p = z[k];
      const float2 q = z[(NFFT - k) & (NFFT - 1)];
      A = make_float2(0.5f * (p.x + q.x), 0.5f * (p.y - q.y));
      Bv = make_float2(0.5f * (p.y + q.y), -0.5f * (p.x - q.x));
      A = sa >= 0 ? compress(A, transform, factor, expo) : make_float2(0.f, 0.f);     // zero-padded frames stay exact zeros
      Bv = sb >= 0 ? compress(Bv, transform, factor, expo) : make_float2(0.f, 0.f);
    }
    float2* o = out + static_cast<int64_t>(k) * n_frames_out;
    if (pair) *reinterpret_cast<float4*>(o) = make_float4(A.x, A.y, Bv.x, Bv.y);
    else { o[0] = A; if (tb < n_frames_out) o[1] = Bv; }
  }
}

// iSTFT: a block reconstructs FRB = 16 - (R - 1) hop segments from the 16 frames that overlap them (R = n_fft / hop).
// Every warp loads the two spectra it inverts itself (16-byte pieces; the block's eight warps share each line in L1),
// mirrors them through its exchange buffer for the Hermitian extension, and leaves the two windowed time-domain
// frames in that buffer for the block's overlap-add.
__global__ void __launch_bounds__(WARPS * 32)
decompress_istft_kernel(const float2* __restrict__ spec, int M, const float* __restrict__ window, int hop,
                        int transform, float factor, float expo, int64_t length, const int* __restrict__ lengths,
                        int64_t wave_stride, float* __restrict__ wave) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  SpecSmem& sm = *reinterpret_cast<SpecSmem*>(smem_raw);
  const int warp = __shfl_sync(0xffffffffu, static_cast<int>(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;   // warp-uniform for the compiler
  const int b = blockIdx.y;
  if (lengths) length = __ldg(lengths + b);    // variable-length batch: samples beyond this utterance's length are not written
  const int R = NFFT / hop;
  constexpr int NF = 2 * WARPS;                // frames per block
  const int FRB = NF - (R - 1);                // hop segments (padded timeline) completed by this block
  const int s0 = blockIdx.x * FRB;
  const int m0 = s0 - R + 1;                   // first frame touched

  const float2* in = spec + static_cast<int64_t>(b) * NBIN * M;
  float2* z = sm.work[warp];
  float4* z4 = reinterpret_cast<float4*>(z);
  const int ma = m0 + 2 * warp, mb = ma + 1;
  const bool oka = ma >= 0 && ma < M, okb = mb >= 0 && mb < M;        // warp-uniform
  const bool pair = oka && okb && (M & 1) == 0 && (ma & 1) == 0;      // 16-byte aligned pair load
  // de-compression modes: 0 none, 1 divide by the factor only (exponent 1), 2 the default |z|^0.5 compression
  // (z/f * |z/f|), 3 anything else (generic powf / expm1f path, kept out of the unrolled loop)
  const int mode = transform == FDBM_TRANSFORM_NONE ? 0
                   : (transform == FDBM_TRANSFORM_EXPONENT ? (expo == 1.0f ? 1 : (expo == 0.5f ? 2 : 3)) : 3);
  const float inv = 1.0f / factor;
  auto load_pair = [&](int k, float2& A, float2& Bv) {
    A = make_float2(0.f, 0.f); Bv = A;
    const float2* p = in + static_cast<int64_t>(k) * M + ma;
    if (pair) { const float4 t = __ldg(reinterpret_cast<const float4*>(p)); A = make_float2(t.x, t.y); Bv = make_float2(t.z, t.w); }
    else { if (oka) A = __ldg(p); if (okb) Bv = __ldg(p + 1); }
  };
  if (mode <= 2) {
#pragma unroll
    for (int j = 0; j < 9; ++j) {
      const int k = 32 * j + lane;
      if (k < NBIN) {
        float2 A, Bv;
        load_pair(k, A, Bv);
        if (mode >= 1) { A.x *= inv; A.y *= inv; Bv.x *= inv; Bv.y *= inv; }
        if (mode == 2) {
          const float ma2 = sqrtf(A.x * A.x + A.y * A.y), mb2 = sqrtf(Bv.x * Bv.x + Bv.y * Bv.y);
          A.x *= ma2; A.y *= ma2; Bv.x *= mb2; Bv.y *= mb2;
        }
        if (k == 0 || k == NFFT / 2) { A.y = 0.f; Bv.y = 0.f; }       // irfft semantics: imaginary parts of DC and Nyquist are ignored
        z4[k] = make_float4(A.x, A.y, Bv.x, Bv.y);
      }
    }
  } else {
#pragma unroll 1
    for (int k = lane; k < NBIN; k += 32) {
      float2 A, Bv;
      load_pair(k, A, Bv);
      A = decompress(A, transform, factor, expo);
      Bv = decompress(Bv, transform, factor, expo);
      if (k == 0 || k == NFFT / 2) { A.y = 0.f; Bv.y = 0.f; }
      z4[k] = make_float4(A.x, A.y, Bv.x, Bv.y);
    }
  }
  fill_twiddles(sm.tw);
  __syncthreads();                             // (also orders every warp's z4 writes before its mirrored reads)
  {
    // Hermitian extension of both spectra, Z = A + iB
    float2 v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int k = 32 * j + lane;
      float4 e;
      if (k <= NFFT / 2) e = z4[k];
      else { e = z4[NFFT - k]; e.y = -e.y; e.w = -e.w; }
      v[j] = make_float2(e.x - e.w, e.y + e.z);
    }
    __syncwarp();
    fft512_warp<true>(v, z, sm.tw, lane);
    // window and 1/N; frame a <- re, frame b <- im, stored as two float[512] in the same buffer
#pragma unroll
    for (int j = 0; j < 16; ++j) v[j] = z[32 * j + lane];
    __syncwarp();
    float* fr = reinterpret_cast<float*>(z);
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int n = 32 * j + lane;
      const float w = __ldg(window + n) * (1.0f / NFFT);
      fr[n] = v[j].x * w;
      fr[NFFT + n] = v[j].y * w;
    }
  }
  __syncthreads();

  float* out = wave + static_cast<int64_t>(b) * wave_stride;
  for (int seg = 0; seg < FRB; ++seg) {
    const int64_t n0 = static_cast<int64_t>(s0 + seg) * hop - NFFT / 2;
    for (int j = threadIdx.x; j < hop; j += WARPS * 32) {
      const int64_t n = n0 + j;
      if (n < 0 || n >= length) continue;
      float acc = 0.f, env = 0.f;
      for (int r = R - 1; r >= 0; --r) {         // oldest frame first (fold order)
        const int m = s0 + seg - r;
        if (m < 0 || m >= M) continue;
        const float w = __ldg(window + j + r * hop);
        const int fi = m - m0;
        acc += reinterpret_cast<const float*>(sm.work[fi >> 1])[(fi & 1) * NFFT + j + r * hop];
        env += w * w;
      }
      out[n] = env > 1e-11f ? acc / env : 0.f;
    }
  }
}

// stand-alone spec_fwd / spec_back (data_module.py:173-199) and pad_spec (other.py:76-90) for callers
// that use the reference's unfused API
__global__ void __launch_bounds__(256)
spec_transform_kernel(const float2* __restrict__ in, float2* __restrict__ out, int64_t n, int transform, float factor,
                      float expo, int inverse) {
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += 256ll * gridDim.x)
    out[i] = inverse ? decompress(in[i], transform, factor, expo) : compress(in[i], transform, factor, expo);
}

__global__ void __launch_bounds__(256)
pad_spec_kernel(const float2* __restrict__ in, float2* __restrict__ out, int64_t rows, int T, int T_out, int pad_mode) {
  const int64_t total = rows * T_out;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < total; i += 256ll * gridDim.x) {
    const int t = static_cast<int>(i % T_out);
    const int64_t r = i / T_out;
    const int src = pad_source(t, T, pad_mode);
    out[i] = src >= 0 ? in[r * T + src] : make_float2(0.f, 0.f);
  }
}

}  // namespace

}  // namespace fdbm

using namespace fdbm;

extern "C" int fdbm_spec_transform(const float* in, float* out, int64_t n_complex, int transform_type, float spec_factor,
                                   float abs_exponent, int inverse, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(in && out && n_complex > 0, "fdbm_spec_transform: bad arguments");
  FDBM_REQUIRE(transform_type >= 0 && transform_type <= 2, "fdbm_spec_transform: bad transform");
  const int grid = static_cast<int>(std::min<int64_t>(ceil_div64(n_complex, 256), static_cast<int64_t>(num_sms()) * 16));
  spec_transform_kernel<<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float2*>(in), reinterpret_cast<float2*>(out),
                                                              n_complex, transform_type, spec_factor, abs_exponent, inverse);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

extern "C" int fdbm_pad_spec(const float* in, int64_t rows, int n_frames, int pad_mode, int n_frames_out, float* out,
                             void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(in && out && rows > 0 && n_frames > 0 && n_frames_out >= n_frames, "fdbm_pad_spec: bad arguments");
  FDBM_REQUIRE(pad_mode >= 0 && pad_mode <= 2, "fdbm_pad_spec: bad pad mode");
  FDBM_REQUIRE(pad_mode != FDBM_PAD_REFLECTION || n_frames_out - n_frames < n_frames, "fdbm_pad_spec: reflection pad wider than the input");
  const int64_t total = rows * n_frames_out;
  const int grid = static_cast<int>(std::min<int64_t>(ceil_div64(total, 256), static_cast<int64_t>(num_sms()) * 16));
  pad_spec_kernel<<<grid, 256, 0, as_stream(stream)>>>(reinterpret_cast<const float2*>(in), reinterpret_cast<float2*>(out),
                                                        rows, n_frames, n_frames_out, pad_mode);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

static int stft_launch(const char* who, const float* wave, int batch, int64_t max_samples, int64_t min_samples, const int* lengths,
                       int64_t wave_stride, const float* window, int n_fft, int hop, int transform_type, float spec_factor,
                       float abs_exponent, int pad_mode, int n_frames_out, float* spec, void* stream, const float* norm = nullptr) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(n_fft == NFFT, "%s: n_fft must be 512 (got %d)", who, n_fft);
  FDBM_REQUIRE(hop > 0 && NFFT % hop == 0 && NFFT / hop <= MAXR && NFFT / hop >= 1, "%s: hop %d unsupported", who, hop);
  FDBM_REQUIRE(batch > 0 && min_samples > NFFT / 2 && max_samples >= min_samples && max_samples < (1ll << 30),
               "%s: need batch > 0 and n_fft/2 < n_samples < 2^30", who);
  FDBM_REQUIRE(transform_type >= 0 && transform_type <= 2 && pad_mode >= 0 && pad_mode <= 2, "%s: bad enum", who);
  const int M = 1 + static_cast<int>(max_samples / hop), M_min = 1 + static_cast<int>(min_samples / hop);
  FDBM_REQUIRE(n_frames_out >= M, "%s: n_frames_out %d < frame count %d", who, n_frames_out, M);
  FDBM_REQUIRE(pad_mode != FDBM_PAD_REFLECTION || n_frames_out - M_min < M_min, "%s: reflection pad wider than the input", who);
  FDBM_REQUIRE(wave && window && spec && wave_stride >= max_samples, "%s: null pointer or bad stride", who);
  if (spectral_fast_supported(n_fft, hop, false))
    return launch_stft_fast(wave, batch, max_samples, lengths, wave_stride, window, norm, hop, transform_type, spec_factor, abs_exponent,
                            pad_mode, M, n_frames_out, spec, as_stream(stream));
  FDBM_REQUIRE(!norm, "%s: the fused peak normalisation needs hop 128 or 256", who);
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device()))
    FDBM_CUDA(cudaFuncSetAttribute(stft_compress_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SpecSmem)));
  dim3 grid(ceil_div(n_frames_out, FR), batch);
  stft_compress_kernel<<<grid, WARPS * 32, sizeof(SpecSmem), as_stream(stream)>>>(
      wave, static_cast<int>(max_samples), lengths, wave_stride, window, hop, transform_type, spec_factor, abs_exponent, pad_mode, M,
      n_frames_out, reinterpret_cast<float2*>(spec));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

extern "C" int fdbm_stft_compress(const float* wave, int batch, int64_t n_samples, int64_t wave_stride,
                                  const float* window, int n_fft, int hop, int transform_type, float spec_factor,
                                  float abs_exponent, int pad_mode, int n_frames_out, float* spec, void* stream) {
  return stft_launch("fdbm_stft_compress", wave, batch, n_samples, n_samples, nullptr, wave_stride, window, n_fft, hop, transform_type,
                     spec_factor, abs_exponent, pad_mode, n_frames_out, spec, stream);
}

extern "C" int fdbm_stft_compress_var(const float* wave, int batch, const int* lengths, int64_t min_samples, int64_t max_samples,
                                      int64_t wave_stride, const float* window, int n_fft, int hop, int transform_type,
                                      float spec_factor, float abs_exponent, int pad_mode, int n_frames_out, float* spec,
                                      void* stream) {
  FDBM_REQUIRE(lengths, "fdbm_stft_compress_var: null lengths");
  return stft_launch("fdbm_stft_compress_var", wave, batch, max_samples, min_samples, lengths, wave_stride, window, n_fft, hop,
                     transform_type, spec_factor, abs_exponent, pad_mode, n_frames_out, spec, stream);
}

static int istft_launch(const char* who, const float* spec, int batch, int n_frames, const float* window, int n_fft, int hop,
                        int transform_type, float spec_factor, float abs_exponent, int64_t length, const int* lengths,
                        int64_t wave_stride, float* wave, void* stream, const float* norm = nullptr, float* peak = nullptr) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(n_fft == NFFT, "%s: n_fft must be 512 (got %d)", who, n_fft);
  FDBM_REQUIRE(hop > 0 && NFFT % hop == 0 && NFFT / hop <= MAXR, "%s: hop %d unsupported", who, hop);
  FDBM_REQUIRE(batch > 0 && n_frames > 0 && length > 0 && wave_stride >= length, "%s: bad sizes", who);
  FDBM_REQUIRE(transform_type >= 0 && transform_type <= 2, "%s: bad transform", who);
  FDBM_REQUIRE(spec && window && wave, "%s: null pointer", who);
  if (spectral_fast_supported(n_fft, hop, true))
    return launch_istft_fast(spec, batch, n_frames, window, transform_type, spec_factor, abs_exponent, length, lengths, wave_stride, norm,
                             peak, wave, as_stream(stream));
  FDBM_REQUIRE(!norm && !peak, "%s: the fused rescale / peak tracking needs hop = n_fft / 2", who);
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device()))
    FDBM_CUDA(cudaFuncSetAttribute(decompress_istft_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(SpecSmem)));
  const int64_t n_seg = ceil_div64(length + NFFT / 2, hop);      // hop segments covering [0, length + n_fft/2)
  const int frb = 2 * WARPS - (NFFT / hop - 1);                  // hop segments completed per block
  dim3 grid(static_cast<unsigned>(ceil_div64(n_seg, frb)), batch);
  decompress_istft_kernel<<<grid, WARPS * 32, sizeof(SpecSmem), as_stream(stream)>>>(
      reinterpret_cast<const float2*>(spec), n_frames, window, hop, transform_type, spec_factor, abs_exponent, length, lengths,
      wave_stride, wave);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

extern "C" int fdbm_decompress_istft(const float* spec, int batch, int n_frames, const float* window, int n_fft, int hop,
                                     int transform_type, float spec_factor, float abs_exponent, int64_t length,
                                     int64_t wave_stride, float* wave, void* stream) {
  return istft_launch("fdbm_decompress_istft", spec, batch, n_frames, window, n_fft, hop, transform_type, spec_factor, abs_exponent,
                      length, nullptr, wave_stride, wave, stream);
}

extern "C" int fdbm_decompress_istft_var(const float* spec, int batch, int n_frames, const float* window, int n_fft, int hop,
                                         int transform_type, float spec_factor, float abs_exponent, const int* lengths,
                                         int64_t max_length, int64_t wave_stride, float* wave, void* stream) {
  FDBM_REQUIRE(lengths, "fdbm_decompress_istft_var: null lengths");
  return istft_launch("fdbm_decompress_istft_var", spec, batch, n_frames, window, n_fft, hop, transform_type, spec_factor,
                      abs_exponent, max_length, lengths, wave_stride, wave, stream);
}

// ---- fused glue of `enhance` (fdbm/model.py:391-406, infer_single.py:80-99, infer_folder.py:100-121) ------------------------
extern "C" int fdbm_wave_absmax(const float* wave, int batch, int64_t n_samples, const int* lengths, int64_t wave_stride, float* out,
                                void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(wave && out && batch > 0 && n_samples > 0 && wave_stride >= n_samples, "fdbm_wave_absmax: bad arguments");
  return launch_absmax(wave, batch, n_samples, lengths, wave_stride, out, as_stream(stream));
}

extern "C" int fdbm_stft_compress_ex(const float* wave, int batch, const int* lengths, int64_t min_samples, int64_t max_samples,
                                     int64_t wave_stride, const float* window, const float* norm, int n_fft, int hop,
                                     int transform_type, float spec_factor, float abs_exponent, int pad_mode, int n_frames_out,
                                     float* spec, void* stream) {
  return stft_launch("fdbm_stft_compress_ex", wave, batch, max_samples, min_samples, lengths, wave_stride, window, n_fft, hop,
                     transform_type, spec_factor, abs_exponent, pad_mode, n_frames_out, spec, stream, norm);
}

extern "C" int fdbm_decompress_istft_ex(const float* spec, int batch, int n_frames, const float* window, int n_fft, int hop,
                                        int transform_type, float spec_factor, float abs_exponent, const int* lengths,
                                        int64_t max_length, int64_t wave_stride, const float* norm, float* peak, float* wave,
                                        void* stream) {
  return istft_launch("fdbm_decompress_istft_ex", spec, batch, n_frames, window, n_fft, hop, transform_type, spec_factor,
                      abs_exponent, max_length, lengths, wave_stride, wave, stream, norm, peak);
}

extern "C" int fdbm_clip_rescale(float* wave, int batch, int64_t n_samples, const int* lengths, int64_t wave_stride, const float* peak,
                                 float rescale, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(wave && peak && batch > 0 && n_samples > 0 && wave_stride >= n_samples, "fdbm_clip_rescale: bad arguments");
  return launch_clip_rescale(wave, batch, n_samples, lengths, wave_stride, peak, rescale, as_stream(stream));
}
