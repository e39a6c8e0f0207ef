// HBM-bound passes around the convolutions, all on [B,T,F,C] (channels-innermost) activations:
//   - fir_resample      : upfirdn2d with the [1,3,3,1] kernel, x2 down / x2 up
//                         (up_or_down_sampling.py:195-257, op/upfirdn2d_kernel.cu:107-207)
//   - channel_stats     : per-(b,channel) sum / sum of squares (feeds GroupNorm)
//   - groupnorm_act     : GroupNorm(eps 1e-6) [+SiLU] [+FIR up/down] of the channel concatenation of
//                         up to two fp32 sources -> bf16 GEMM operand(s)  (layerspp.py:242-257)
#include "common.cuh"

namespace fdbm {
namespace {

// ------------------------------------------------------------------------------------------------
// Resampling taps.  Down x2 (pad 1,1): o[i] = (x[2i-1] + 3x[2i] + 3x[2i+1] + x[2i+2]) / 8.
// Up x2 (zero insertion, pad 2,1, gain 4): o[2i] = (x[i-1] + 3x[i]) / 4, o[2i+1] = (3x[i] + x[i+1]) / 4.
// Samples outside the image are zero.
// ------------------------------------------------------------------------------------------------
struct Taps1D {
  int n;          // number of taps
  int pos[4];     // input positions
  float w[4];
};

__device__ __forceinline__ Taps1D taps_for(int o, int mode) {
  Taps1D t;
  if (mode == 1) {            // down
    t.n = 4;
    t.pos[0] = 2 * o - 1; t.pos[1] = 2 * o; t.pos[2] = 2 * o + 1; t.pos[3] = 2 * o + 2;
    t.w[0] = 0.125f; t.w[1] = 0.375f; t.w[2] = 0.375f; t.w[3] = 0.125f;
  } else if (mode == 2) {     // up
    const int i = o >> 1;
    t.n = 2;
    if (o & 1) { t.pos[0] = i; t.pos[1] = i + 1; t.w[0] = 0.75f; t.w[1] = 0.25f; }
    else       { t.pos[0] = i - 1; t.pos[1] = i; t.w[0] = 0.25f; t.w[1] = 0.75f; }
    t.pos[2] = t.pos[3] = -1; t.w[2] = t.w[3] = 0.f;
  } else {
    t.n = 1; t.pos[0] = o; t.w[0] = 1.f;
    t.pos[1] = t.pos[2] = t.pos[3] = -1; t.w[1] = t.w[2] = t.w[3] = 0.f;
  }
  return t;
}

__host__ __device__ inline int out_dim(int n, int mode) { return mode == 1 ? n / 2 : (mode == 2 ? n * 2 : n); }

__global__ void __launch_bounds__(256)
fir_resample_kernel(const float* __restrict__ in, int B, int T, int F, int C, int mode, float scale, float* __restrict__ out) {
  const int To = out_dim(T, mode), Fo = out_dim(F, mode);
  const int64_t total = static_cast<int64_t>(B) * To * Fo * C;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < total; i += 256ll * gridDim.x) {
    const int c = static_cast<int>(i % C);
    int64_t p = i / C;
    const int fo = static_cast<int>(p % Fo); p /= Fo;
    const int to = static_cast<int>(p % To);
    const int b = static_cast<int>(p / To);
    const Taps1D tt = taps_for(to, mode), tf = taps_for(fo, mode);
    float acc = 0.f;
    for (int a = 0; a < tt.n; ++a) {
      if (tt.pos[a] < 0 || tt.pos[a] >= T) continue;
      for (int q = 0; q < tf.n; ++q) {
        if (tf.pos[q] < 0 || tf.pos[q] >= F) continue;
        acc += tt.w[a] * tf.w[q] * in[((static_cast<int64_t>(b) * T + tt.pos[a]) * F + tf.pos[q]) * C + c];
      }
    }
    out[i] = acc * scale;
  }
}

// ------------------------------------------------------------------------------------------------
// channel_stats: block = 256 threads = (pixel lanes) x (C/4 float4 lanes); each block reduces a
// contiguous run of pixels of one batch item, then adds its partial to sums[b][c][0..1] (double).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
channel_stats_kernel(const float* __restrict__ in, int64_t P, int C, int64_t px_per_block, double* __restrict__ sums) {
  __shared__ float4 red_s[256], red_q[256];
  const int cg = C / 4;
  const int pl = 256 / cg;
  const int ci = threadIdx.x % cg, pi = threadIdx.x / cg;
  const int b = blockIdx.y;
  const int64_t p0 = blockIdx.x * px_per_block;
  const int64_t p1 = min(P, p0 + px_per_block);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), q = s;
  if (pi < pl) {
    const float4* base = reinterpret_cast<const float4*>(in + static_cast<int64_t>(b) * P * C) + ci;
    for (int64_t p = p0 + pi; p < p1; p += pl) {
      const float4 v = base[p * cg];
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
      q.x += v.x * v.x; q.y += v.y * v.y; q.z += v.z * v.z; q.w += v.w * v.w;
    }
  }
  red_s[threadIdx.x] = s;
  red_q[threadIdx.x] = q;
  __syncthreads();
  if (threadIdx.x < cg) {
    double ds[4] = {0, 0, 0, 0}, dq[4] = {0, 0, 0, 0};
    for (int j = 0; j < pl; ++j) {
      const float4 a = red_s[j * cg + threadIdx.x], c2 = red_q[j * cg + threadIdx.x];
      ds[0] += a.x; ds[1] += a.y; ds[2] += a.z; ds[3] += a.w;
      dq[0] += c2.x; dq[1] += c2.y; dq[2] += c2.z; dq[3] += c2.w;
    }
    double* o = sums + (static_cast<int64_t>(b) * C + threadIdx.x * 4) * 2;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      atomicAdd(o + 2 * j, ds[j]);
      atomicAdd(o + 2 * j + 1, dq[j]);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// groupnorm_act
// ------------------------------------------------------------------------------------------------
constexpr int GN_MAXC = 512;


template <int MODE, bool SRC16>
__global__ void __launch_bounds__(256)
groupnorm_act_kernel(const void* __restrict__ src1, const double* __restrict__ sums1, int C1,
                     const void* __restrict__ src2, const double* __restrict__ sums2, int C2,
                     const float* __restrict__ gamma, const float* __restrict__ beta, int T, int F, int silu,
                     int px_per_block, uint4* __restrict__ act_out, uint4* __restrict__ raw_out) {
  pdl_wait_then_trigger();
  __shared__ float sA[GN_MAXC], sB[GN_MAXC];
  __shared__ float s_mean[32], s_rstd[32];
  const int C = C1 + C2;
  const int b = blockIdx.y;
  const int G = min(C / 4, 32);
  const int cpg = C / G;
  if (threadIdx.x < G) {
    double s = 0, q = 0;
    for (int j = 0; j < cpg; ++j) {
      const int c = threadIdx.x * cpg + j;
      const double* e = c < C1 ? sums1 + (static_cast<int64_t>(b) * C1 + c) * 2
                               : sums2 + (static_cast<int64_t>(b) * C2 + (c - C1)) * 2;
      s += e[0];
      q += e[1];
    }
    const double cnt = static_cast<double>(cpg) * T * F;
    const double mean = s / cnt;
    double var = q / cnt - mean * mean;
    if (var < 0) var = 0;
    s_mean[threadIdx.x] = static_cast<float>(mean);
    s_rstd[threadIdx.x] = static_cast<float>(1.0 / sqrt(var + 1e-6));
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {
    const int g = c / cpg;
    const float a = gamma[c] * s_rstd[g];
    sA[c] = a;
    sB[c] = beta[c] - s_mean[g] * a;
  }
  __syncthreads();

  // thread -> fixed group of 8 channels, a lane of pixels: scale/shift live in registers for the whole loop
  const int cg8 = C / 8;
  const int npl = 256 / cg8;                           // pixel lanes per block (idle threads when 256 % cg8 != 0)
  const int g8 = threadIdx.x % cg8, pl = threadIdx.x / cg8;
  if (pl >= npl) return;
  const int c0 = g8 * 8;
  float a[8], bb[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { a[j] = sA[c0 + j]; bb[j] = sB[c0 + j]; }
  const bool from2 = c0 >= C1;
  const int Cs = from2 ? C2 : C1, cs = from2 ? c0 - C1 : c0;
  // SRC16: both sources are 16-bit tensors; otherwise both are fp32
  const float* sf = from2 ? reinterpret_cast<const float*>(src2) + (SRC16 ? 0 : static_cast<int64_t>(b) * T * F * C2)
                          : reinterpret_cast<const float*>(src1) + (SRC16 ? 0 : static_cast<int64_t>(b) * T * F * C1);
  const op_t* sh = from2 ? reinterpret_cast<const op_t*>(src2) + static_cast<int64_t>(b) * T * F * C2
                         : reinterpret_cast<const op_t*>(src1) + static_cast<int64_t>(b) * T * F * C1;

  const int To = out_dim(T, MODE), Fo = out_dim(F, MODE);
  const int n_px = To * Fo;
  const int p0 = blockIdx.x * px_per_block;
  const int p1 = min(n_px, p0 + px_per_block);
  constexpr int NT = MODE == 1 ? 4 : (MODE == 2 ? 2 : 1);
  for (int p = p0 + pl; p < p1; p += npl) {
    const int fo = p % Fo, to = p / Fo;
    float acc[8], raw[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { acc[j] = 0.f; raw[j] = 0.f; }
    const Taps1D tt = taps_for(to, MODE), tf = taps_for(fo, MODE);
#pragma unroll
    for (int u = 0; u < NT; ++u) {
      if (tt.pos[u] < 0 || tt.pos[u] >= T) continue;
#pragma unroll
      for (int v = 0; v < NT; ++v) {
        if (tf.pos[v] < 0 || tf.pos[v] >= F) continue;
        const float w = tt.w[u] * tf.w[v];
        const int64_t off = (static_cast<int64_t>(tt.pos[u]) * F + tf.pos[v]) * Cs + cs;
        float x[8];
        if (SRC16) {
          const uint4 rawv = *reinterpret_cast<const uint4*>(sh + off);
          const op2_t* h2 = reinterpret_cast<const op2_t*>(&rawv);
#pragma unroll
          for (int j = 0; j < 4; ++j) { const float2 f2 = op22f2(h2[j]); x[2 * j] = f2.x; x[2 * j + 1] = f2.y; }
        } else {
          const float4 x0 = *reinterpret_cast<const float4*>(sf + off), x1 = *reinterpret_cast<const float4*>(sf + off + 4);
          x[0] = x0.x; x[1] = x0.y; x[2] = x0.z; x[3] = x0.w; x[4] = x1.x; x[5] = x1.y; x[6] = x1.z; x[7] = x1.w;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float y = fmaf(x[j], a[j], bb[j]);
          if (silu) {                                     // y sigmoid(y), sigmoid(y) = 1/2 + tanh(y/2)/2: one MUFU instead of EX2 + RCP
            float th;
            asm("tanh.approx.f32 %0, %1;" : "=f"(th) : "f"(0.5f * y));
            y *= fmaf(th, 0.5f, 0.5f);
          }
          acc[j] = fmaf(w, y, acc[j]);
          raw[j] = fmaf(w, x[j], raw[j]);
        }
      }
    }
    const int64_t o = (static_cast<int64_t>(b) * n_px + p) * cg8 + g8;
    act_out[o] = make_uint4(pack_op2(acc[0], acc[1]), pack_op2(acc[2], acc[3]), pack_op2(acc[4], acc[5]),
                            pack_op2(acc[6], acc[7]));
    if (raw_out)
      raw_out[o] = make_uint4(pack_op2(raw[0], raw[1]), pack_op2(raw[2], raw[3]), pack_op2(raw[4], raw[5]),
                              pack_op2(raw[6], raw[7]));
  }
}

// ------------------------------------------------------------------------------------------------
// gn_resample16: the resampling ResnetBlocks' input pass (layerspp.py:242-257 with up/down):
//   act_out = FIR(SiLU(GroupNorm(cat(src1, src2)))),  raw_out = FIR(cat(src1, src2))   (x2 down or x2 up)
// from the 16-bit copies of the residual stream and the (scale, shift) table of gn_finalize.
// A thread owns 4 channels and a 2-column strip and walks down the frame axis keeping the horizontally
// filtered rows it still needs in registers, so every input pixel is fetched (and activated) by 1.5 (down)
// or 2 (up) threads instead of 16 / 4 and the pass is bound by its HBM bytes.  SiLU(y) = h + h tanh(h),
// h = y/2, in packed 16-bit (one MUFU per element) -- the same arithmetic as the convolution's
// normalise-on-load path.
// ------------------------------------------------------------------------------------------------
constexpr int RS_ROWS = 16;       // output rows (down) / input rows (up) per thread

template <int MODE>
__global__ void __launch_bounds__(256, 2)
gn_resample16_kernel(const op_t* __restrict__ src1, int C1, const op_t* __restrict__ src2, int C2,
                     const float2* __restrict__ tab, int B, int T, int F, op_t* __restrict__ act_out,
                     op_t* __restrict__ raw_out) {
  const int C = C1 + C2, C4 = C / 4;
  const int To = MODE == 1 ? T / 2 : T * 2, Fo = MODE == 1 ? F / 2 : F * 2;
  const int nstrip = MODE == 1 ? (Fo + 1) / 2 : (F + 1) / 2;
  const int nrows = MODE == 1 ? To : T;
  const int nchunk = (nrows + RS_ROWS - 1) / RS_ROWS;
  int64_t idx = blockIdx.x * 256ll + threadIdx.x;
  if (idx >= static_cast<int64_t>(B) * nchunk * nstrip * C4) return;
  const int cg = static_cast<int>(idx % C4); idx /= C4;
  const int strip = static_cast<int>(idx % nstrip); idx /= nstrip;
  const int chunk = static_cast<int>(idx % nchunk);
  const int b = static_cast<int>(idx / nchunk);
  const int c0 = cg * 4;
  const bool from2 = c0 >= C1;
  const int Cs = from2 ? C2 : C1;
  const op_t* sp = (from2 ? src2 : src1) + static_cast<int64_t>(b) * T * F * Cs + (from2 ? c0 - C1 : c0);
  // packed fp32x2 arithmetic throughout (FFMA2): the pass is instruction-bound otherwise
  float2 sc[2], sh[2];
  {
    const float4* tp = reinterpret_cast<const float4*>(tab + static_cast<int64_t>(b) * C + c0);
    const float4 e0 = __ldg(tp), e1 = __ldg(tp + 1);
    sc[0] = make_float2(0.5f * e0.x, 0.5f * e0.z); sh[0] = make_float2(0.5f * e0.y, 0.5f * e0.w);
    sc[1] = make_float2(0.5f * e1.x, 0.5f * e1.z); sh[1] = make_float2(0.5f * e1.y, 0.5f * e1.w);
  }
  // one pixel: raw values and SiLU(GroupNorm(.)) of this thread's 4 channels (two float2 each)
  auto px_act = [&](const uint2 rawv, float2 (&a)[2], float2 (&r)[2]) {
    const op2_t* h2 = reinterpret_cast<const op2_t*>(&rawv);
#pragma unroll
    for (int w = 0; w < 2; ++w) {
      r[w] = op22f2(h2[w]);
      const float2 y = __ffma2_rn(r[w], sc[w], sh[w]);
      const op2_t h = f2op2(y.x, y.y);
      a[w] = op22f2(__hfma2(h, op2_tanh(h), h));
    }
  };
  auto store_px = [&](int to, int fo, const float2 (&a)[2], const float2 (&r)[2]) {
    if (fo >= Fo) return;
    const int64_t o = ((static_cast<int64_t>(b) * To + to) * Fo + fo) * C + c0;
    *reinterpret_cast<uint2*>(act_out + o) = make_uint2(pack_op2(a[0].x, a[0].y), pack_op2(a[1].x, a[1].y));
    *reinterpret_cast<uint2*>(raw_out + o) = make_uint2(pack_op2(r[0].x, r[0].y), pack_op2(r[1].x, r[1].y));
  };
  const float2 zero2 = make_float2(0.f, 0.f);

  if (MODE == 1) {
    // down: o[i] = (x[2i-1] + 3 x[2i] + 3 x[2i+1] + x[2i+2]) / 8 per axis; output columns fo0, fo0 + 1 from input
    // columns fi0 .. fi0 + 5 (zeros outside the image)
    const int fo0 = 2 * strip, fi0 = 2 * fo0 - 1;
    uint32_t okf = 0;
#pragma unroll
    for (int k = 0; k < 6; ++k) okf |= (fi0 + k >= 0 && fi0 + k < F) ? (1u << k) : 0u;
    const float2 w1 = make_float2(0.125f, 0.125f), w3 = make_float2(0.375f, 0.375f);
    // the six input pixels of row t (zeros outside the image): loads only, so that a whole output row's twelve loads -- and the
    // next output row's -- are in flight before the first is consumed (the rolled loop was one dependent load -> compute chain per
    // input row: 16 warps per SM x 6 x 8 bytes in flight, latency-bound at 38 % of the HBM peak)
    auto load_row = [&](int t, uint2 (&raw)[6]) {
      const bool in = t >= 0 && t < T;
      const op_t* rp = sp + (static_cast<int64_t>(in ? t : 0) * F + fi0) * Cs;
#pragma unroll
      for (int k = 0; k < 6; ++k) raw[k] = (in && ((okf >> k) & 1)) ? __ldg(reinterpret_cast<const uint2*>(rp + k * Cs)) : make_uint2(0u, 0u);
    };
    // horizontally filtered row t -> ha/hr[2 output columns][2 float2]
    auto hrow = [&](int t, const uint2 (&raw)[6], float2 (&ha)[2][2], float2 (&hr)[2][2]) {
#pragma unroll
      for (int j = 0; j < 2; ++j) { ha[j][0] = zero2; ha[j][1] = zero2; hr[j][0] = zero2; hr[j][1] = zero2; }
      if (t < 0 || t >= T) return;
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        float2 a[2], r[2];
        px_act(raw[k], a, r);
        if (!((okf >> k) & 1)) { a[0] = zero2; a[1] = zero2; }           // the activation of a padding zero is not zero
        if (k < 4) {
          const float2 w = (k == 0 || k == 3) ? w1 : w3;
#pragma unroll
          for (int c = 0; c < 2; ++c) { ha[0][c] = __ffma2_rn(w, a[c], ha[0][c]); hr[0][c] = __ffma2_rn(w, r[c], hr[0][c]); }
        }
        if (k >= 2) {
          const float2 w = (k == 2 || k == 5) ? w1 : w3;
#pragma unroll
          for (int c = 0; c < 2; ++c) { ha[1][c] = __ffma2_rn(w, a[c], ha[1][c]); hr[1][c] = __ffma2_rn(w, r[c], hr[1][c]); }
        }
      }
    };
    const int to0 = chunk * RS_ROWS, to1 = min(To, to0 + RS_ROWS);
    float2 ca[2][2], cr[2][2], na[2][2], nr[2][2], ha[2][2], hr[2][2];
    uint2 ra[6], rb[6], qa[6], qb[6];
    load_row(2 * to0 - 1, ra); load_row(2 * to0, rb);
    load_row(2 * to0 + 1, qa); load_row(2 * to0 + 2, qb);
    hrow(2 * to0 - 1, ra, ha, hr);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int c = 0; c < 2; ++c) { ca[j][c] = __fmul2_rn(w1, ha[j][c]); cr[j][c] = __fmul2_rn(w1, hr[j][c]); }
    hrow(2 * to0, rb, ha, hr);
#pragma unroll
    for (int j = 0; j < 2; ++j)
#pragma unroll
      for (int c = 0; c < 2; ++c) { ca[j][c] = __ffma2_rn(w3, ha[j][c], ca[j][c]); cr[j][c] = __ffma2_rn(w3, hr[j][c], cr[j][c]); }
#pragma unroll 1
    for (int to = to0; to < to1; ++to) {
      // this output row's two new input rows are in qa / qb; request the next output row's before consuming them
#pragma unroll
      for (int k = 0; k < 6; ++k) { ra[k] = qa[k]; rb[k] = qb[k]; }
      if (to + 1 < to1) { load_row(2 * to + 3, qa); load_row(2 * to + 4, qb); }
      hrow(2 * to + 1, ra, ha, hr);
#pragma unroll
      for (int j = 0; j < 2; ++j)
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          ca[j][c] = __ffma2_rn(w3, ha[j][c], ca[j][c]); cr[j][c] = __ffma2_rn(w3, hr[j][c], cr[j][c]);
          na[j][c] = __fmul2_rn(w1, ha[j][c]); nr[j][c] = __fmul2_rn(w1, hr[j][c]);
        }
      hrow(2 * to + 2, rb, ha, hr);
#pragma unroll
      for (int j = 0; j < 2; ++j) {
#pragma unroll
        for (int c = 0; c < 2; ++c) {
          ca[j][c] = __ffma2_rn(w1, ha[j][c], ca[j][c]); cr[j][c] = __ffma2_rn(w1, hr[j][c], cr[j][c]);
          na[j][c] = __ffma2_rn(w3, ha[j][c], na[j][c]); nr[j][c] = __ffma2_rn(w3, hr[j][c], nr[j][c]);
        }
        store_px(to, fo0 + j, ca[j], cr[j]);
#pragma unroll
        for (int c = 0; c < 2; ++c) { ca[j][c] = na[j][c]; cr[j][c] = nr[j][c]; }
      }
    }
  } else {
    // up: o[2i] = (x[i-1] + 3 x[i]) / 4, o[2i+1] = (3 x[i] + x[i+1]) / 4 per axis; input columns f0 - 1 .. f0 + 2 ->
    // output columns 2 f0 .. 2 f0 + 3
    const int f0 = 2 * strip;
    uint32_t okf = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) okf |= (f0 - 1 + k >= 0 && f0 - 1 + k < F) ? (1u << k) : 0u;
    const float2 q1 = make_float2(0.25f, 0.25f), q3 = make_float2(0.75f, 0.75f);
    auto hrow = [&](int t, float2 (&ha)[4][2], float2 (&hr)[4][2]) {
      float2 a[4][2], r[4][2];
      if (t < 0 || t >= T) {
#pragma unroll
        for (int k = 0; k < 4; ++k) { ha[k][0] = zero2; ha[k][1] = zero2; hr[k][0] = zero2; hr[k][1] = zero2; }
        return;
      }
      const op_t* rp = sp + (static_cast<int64_t>(t) * F + f0 - 1) * Cs;
      uint2 raw[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) raw[k] = ((okf >> k) & 1) ? __ldg(reinterpret_cast<const uint2*>(rp + k * Cs)) : make_uint2(0u, 0u);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        px_act(raw[k], a[k], r[k]);
        if (!((okf >> k) & 1)) { a[k][0] = zero2; a[k][1] = zero2; }
      }
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        ha[0][c] = __ffma2_rn(q1, a[0][c], __fmul2_rn(q3, a[1][c])); hr[0][c] = __ffma2_rn(q1, r[0][c], __fmul2_rn(q3, r[1][c]));
        ha[1][c] = __ffma2_rn(q3, a[1][c], __fmul2_rn(q1, a[2][c])); hr[1][c] = __ffma2_rn(q3, r[1][c], __fmul2_rn(q1, r[2][c]));
        ha[2][c] = __ffma2_rn(q1, a[1][c], __fmul2_rn(q3, a[2][c])); hr[2][c] = __ffma2_rn(q1, r[1][c], __fmul2_rn(q3, r[2][c]));
        ha[3][c] = __ffma2_rn(q3, a[2][c], __fmul2_rn(q1, a[3][c])); hr[3][c] = __ffma2_rn(q3, r[2][c], __fmul2_rn(q1, r[3][c]));
      }
    };
    const int i0 = chunk * RS_ROWS, i1 = min(T, i0 + RS_ROWS);
    float2 pa[4][2], pr[4][2], qa[4][2], qr[4][2];
    hrow(i0 - 1, pa, pr);
#pragma unroll 1
    for (int i = i0; i <= i1; ++i) {
      hrow(i, qa, qr);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float2 oa[2], orr[2];
        if (i > i0) {                                    // odd output row of the previous input row
#pragma unroll
          for (int c = 0; c < 2; ++c) { oa[c] = __ffma2_rn(q3, pa[k][c], __fmul2_rn(q1, qa[k][c])); orr[c] = __ffma2_rn(q3, pr[k][c], __fmul2_rn(q1, qr[k][c])); }
          store_px(2 * i - 1, 2 * f0 + k, oa, orr);
        }
        if (i < i1) {                                    // even output row of this input row
#pragma unroll
          for (int c = 0; c < 2; ++c) { oa[c] = __ffma2_rn(q1, pa[k][c], __fmul2_rn(q3, qa[k][c])); orr[c] = __ffma2_rn(q1, pr[k][c], __fmul2_rn(q3, qr[k][c])); }
          store_px(2 * i, 2 * f0 + k, oa, orr);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) { pa[k][c] = qa[k][c]; pr[k][c] = qr[k][c]; }
      }
    }
  }
}

// (scale, shift) per (utterance, channel) of a GroupNorm over the concatenation of up to two tensors:
// scale = gamma * rstd(group), shift = beta - mean(group) * scale.  Consumed by the convolution's
// normalise-on-load stage.  One block per utterance.
// blk_real != 0 (fdbm_arch.channel_block_real): every 128-channel block holds blk_real real channels followed by zero
// channels; groups and counts follow the real channel index r = (c / 128) * blk_real + c % 128, padding gets (0, 0).
__global__ void __launch_bounds__(256)
gn_finalize_kernel(const double* __restrict__ sums1, int C1, const double* __restrict__ sums2, int C2,
                   const float* __restrict__ gamma, const float* __restrict__ beta, double pixels,
                   float2* __restrict__ table, int blk_real, float2* __restrict__ stats) {
  __shared__ double2 s_sq[GN_MAXC];
  __shared__ float s_mean[32], s_rstd[32];
  asm volatile("griddepcontrol.wait;" ::: "memory");            // programmatic dependent launch: the producer's sums are final from here
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int C = C1 + C2, b = blockIdx.x;
  const int Cr = blk_real ? C / 128 * blk_real : C;
  const int G = min(Cr / 4, 32), cpg = Cr / G;
  // all (sum, sum of squares) entries in one round of independent 16-byte loads (the launch is latency-bound)
  float gam[GN_MAXC / 256], bet[GN_MAXC / 256];
#pragma unroll
  for (int u = 0; u < GN_MAXC / 256; ++u) {
    const int c = threadIdx.x + u * 256;
    if (c < C) {
      const double* e = c < C1 ? sums1 + (static_cast<int64_t>(b) * C1 + c) * 2
                               : sums2 + (static_cast<int64_t>(b) * C2 + (c - C1)) * 2;
      s_sq[c] = *reinterpret_cast<const double2*>(e);
      gam[u] = __ldg(gamma + c); bet[u] = __ldg(beta + c);
    }
  }
  __syncthreads();
  if (threadIdx.x < G) {
    double s = 0, q = 0;
    for (int j = 0; j < cpg; ++j) {
      const int r = threadIdx.x * cpg + j;
      const double2 e = s_sq[blk_real ? r / blk_real * 128 + r % blk_real : r];
      s += e.x; q += e.y;
    }
    const double cnt = cpg * pixels;
    const double mean = s / cnt;
    double var = q / cnt - mean * mean;
    if (var < 0) var = 0;
    s_mean[threadIdx.x] = static_cast<float>(mean);
    s_rstd[threadIdx.x] = static_cast<float>(1.0 / sqrt(var + 1e-6));
    // training plans: the backward's per-group (mean, rstd), formerly a launch of its own per GroupNorm (gn_stats_kernel)
    if (stats) stats[static_cast<int64_t>(b) * G + threadIdx.x] = make_float2(s_mean[threadIdx.x], s_rstd[threadIdx.x]);
  }
  __syncthreads();
#pragma unroll
  for (int u = 0; u < GN_MAXC / 256; ++u) {
    const int c = threadIdx.x + u * 256;
    if (c < C) {
      if (blk_real && (c & 127) >= blk_real) { table[static_cast<int64_t>(b) * C + c] = make_float2(0.f, 0.f); continue; }
      const int g = (blk_real ? (c >> 7) * blk_real + (c & 127) : c) / cpg;
      const float a = gam[u] * s_rstd[g];
      table[static_cast<int64_t>(b) * C + c] = make_float2(a, bet[u] - s_mean[g] * a);
    }
  }
}

}  // namespace

int launch_gn_finalize(const double* sums1, int C1, const double* sums2, int C2, const float* gamma, const float* beta,
                       int B, int64_t pixels, float2* table, cudaStream_t s, int blk_real, float2* stats) {
  const int C = C1 + C2;
  FDBM_REQUIRE(blk_real == 0 || (blk_real > 0 && blk_real < 128 && blk_real % 4 == 0 && C1 % 128 == 0 && C2 % 128 == 0),
               "gn_finalize: channel_block_real %d needs 128-channel blocks (%d+%d)", blk_real, C1, C2);
  const int Cr = blk_real ? C / 128 * blk_real : C;
  FDBM_REQUIRE(Cr % std::min(Cr / 4, 32) == 0 && C >= 4 && C <= GN_MAXC, "gn_finalize: unsupported channels %d+%d", C1, C2);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(B); cfg.blockDim = dim3(256); cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl_enabled() && B <= pdl_batch_limit() ? 1 : 0;      // small batches only, see launch_conv_igemm
  FDBM_CUDA(cudaLaunchKernelEx(&cfg, gn_finalize_kernel, sums1, C1, sums2, C2, gamma, beta, static_cast<double>(pixels), table, blk_real, stats));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_gn_resample16(const op_t* src1, int C1, const op_t* src2, int C2, const float2* tab, int B, int T, int F,
                         int mode, op_t* act_out, op_t* raw_out, cudaStream_t s) {
  const int C = C1 + C2;
  FDBM_REQUIRE(src1 && tab && act_out && raw_out && C1 % 4 == 0 && C2 % 4 == 0 && (C2 == 0) == (src2 == nullptr),
               "gn_resample16: bad arguments (channels %d+%d)", C1, C2);
  FDBM_REQUIRE(mode == 1 || mode == 2, "gn_resample16: mode must be 1 (down) or 2 (up)");
  FDBM_REQUIRE(mode != 1 || (T % 2 == 0 && F % 2 == 0), "gn_resample16: down-sampling needs even T, F");
  const int nstrip = mode == 1 ? (F / 2 + 1) / 2 : (F + 1) / 2;
  const int nrows = mode == 1 ? T / 2 : T;
  const int64_t total = static_cast<int64_t>(B) * ceil_div(nrows, RS_ROWS) * nstrip * (C / 4);
  const unsigned grid = static_cast<unsigned>(ceil_div64(total, 256));
  if (mode == 1) gn_resample16_kernel<1><<<grid, 256, 0, s>>>(src1, C1, src2, C2, tab, B, T, F, act_out, raw_out);
  else gn_resample16_kernel<2><<<grid, 256, 0, s>>>(src1, C1, src2, C2, tab, B, T, F, act_out, raw_out);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_fir_resample(const float* in, int B, int T, int F, int C, int mode, float* out, cudaStream_t s) {
  return launch_fir_resample_scaled(in, B, T, F, C, mode, 1.0f, out, s);
}

int launch_fir_resample_scaled(const float* in, int B, int T, int F, int C, int mode, float scale, float* out, cudaStream_t s) {
  const int64_t total = static_cast<int64_t>(B) * out_dim(T, mode) * out_dim(F, mode) * C;
  const int grid = static_cast<int>(std::min<int64_t>(ceil_div64(total, 256), static_cast<int64_t>(num_sms()) * 16));
  fir_resample_kernel<<<grid, 256, 0, s>>>(in, B, T, F, C, mode, scale, out);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_channel_stats(const float* in, int B, int T, int F, int C, double* sums, cudaStream_t s) {
  FDBM_REQUIRE(C % 4 == 0 && C / 4 <= 256 && 256 % (C / 4) == 0, "channel_stats: unsupported channel count %d", C);
  FDBM_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * 2 * B * C, s));
  const int64_t P = static_cast<int64_t>(T) * F;
  const int pl = 256 / (C / 4);
  // ~4 waves of blocks over the batch, at least 8 pixels per pixel-lane
  int64_t blocks_x = std::max<int64_t>(1, (static_cast<int64_t>(num_sms()) * 8) / B);
  blocks_x = std::min<int64_t>(blocks_x, std::max<int64_t>(1, P / (pl * 8)));
  const int64_t ppb = ceil_div64(P, blocks_x);
  dim3 grid(static_cast<unsigned>(ceil_div64(P, ppb)), B);
  channel_stats_kernel<<<grid, 256, 0, s>>>(in, P, C, ppb, sums);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_groupnorm_act(const void* src1, int src1_h16, const double* sums1, int C1, const void* src2,
                         const double* sums2, int C2, const float* gamma, const float* beta, int B, int T, int F,
                         int silu, int mode, op_t* act_out, op_t* raw_out, cudaStream_t s) {
  const int C = C1 + C2;
  FDBM_REQUIRE(C <= GN_MAXC && C1 % 8 == 0 && C2 % 8 == 0 && C % std::min(C / 4, 32) == 0 && C / 8 <= 256,
               "groupnorm_act: unsupported channels %d+%d", C1, C2);
  FDBM_REQUIRE(mode >= 0 && mode <= 2, "groupnorm_act: bad mode %d", mode);
  FDBM_REQUIRE(mode != 1 || (T % 2 == 0 && F % 2 == 0), "groupnorm_act: down-sampling needs even T, F");
  const int n_px = out_dim(T, mode) * out_dim(F, mode);
  const int npl = 256 / (C / 8);
  // ~8 resident blocks per SM over the batch; every pixel lane gets at least 4 pixels
  int blocks_x = std::max(1, (num_sms() * 8) / B);
  blocks_x = std::min(blocks_x, std::max(1, n_px / (npl * 4)));
  const int ppb = ceil_div(ceil_div(n_px, blocks_x), npl) * npl;
  dim3 grid(ceil_div(n_px, ppb), B);
  uint4* ao = reinterpret_cast<uint4*>(act_out);
  uint4* ro = reinterpret_cast<uint4*>(raw_out);
#define FDBM_GN_LAUNCH(M, H) \
  FDBM_CUDA(launch_maybe_pdl(groupnorm_act_kernel<M, H>, grid, dim3(256), 0, s, pdl_enabled() && B <= pdl_batch_limit(), src1, sums1, C1, src2, sums2, C2, \
                             gamma, beta, T, F, silu, ppb, ao, ro))
  if (src1_h16) {
    if (mode == 0) FDBM_GN_LAUNCH(0, true); else if (mode == 1) FDBM_GN_LAUNCH(1, true); else FDBM_GN_LAUNCH(2, true);
  } else {
    if (mode == 0) FDBM_GN_LAUNCH(0, false); else if (mode == 1) FDBM_GN_LAUNCH(1, false); else FDBM_GN_LAUNCH(2, false);
  }
#undef FDBM_GN_LAUNCH
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

}  // namespace fdbm

using namespace fdbm;

extern "C" int fdbm_fir_resample(const float* in, int batch, int T, int F, int C, int mode, float* out, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(in && out && batch > 0 && T > 0 && F > 0 && C > 0, "fdbm_fir_resample: bad arguments");
  FDBM_REQUIRE(mode == 1 || mode == 2, "fdbm_fir_resample: mode must be 1 (down) or 2 (up)");
  FDBM_REQUIRE(mode != 1 || (T % 2 == 0 && F % 2 == 0), "fdbm_fir_resample: down-sampling needs even T, F");
  return launch_fir_resample(in, batch, T, F, C, mode, out, as_stream(stream));
}

extern "C" int fdbm_channel_stats(const float* in, int batch, int T, int F, int C, double* sums, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(in && sums && batch > 0 && T > 0 && F > 0, "fdbm_channel_stats: bad arguments");
  return launch_channel_stats(in, batch, T, F, C, sums, as_stream(stream));
}

extern "C" int fdbm_groupnorm_act(const float* src1, const double* sums1, int C1, const float* src2,
                                  const double* sums2, int C2, const float* gamma, const float* beta, int batch, int T,
                                  int F, int silu, int mode, void* act_out, void* raw_out, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(src1 && sums1 && gamma && beta && act_out && batch > 0, "fdbm_groupnorm_act: null pointer");
  FDBM_REQUIRE((C2 == 0) == (src2 == nullptr) && (C2 == 0 || sums2), "fdbm_groupnorm_act: src2/C2 mismatch");
  return launch_groupnorm_act(src1, 0, sums1, C1, src2, sums2, C2, gamma, beta, batch, T, F, silu, mode,
                              reinterpret_cast<op_t*>(act_out), reinterpret_cast<op_t*>(raw_out),
                              as_stream(stream));
}

// the table exactly as the plans build it for a normalise-on-load convolution (norm_table() in plan.cu)
extern "C" int fdbm_gn_table(const double* sums1, int C1, const double* sums2, int C2, const float* gamma, const float* beta,
                             int blk_real, int batch, int64_t pixels, float* table, float* stats, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(sums1 && gamma && beta && table && batch > 0 && pixels > 0, "fdbm_gn_table: bad arguments");
  FDBM_REQUIRE((C2 == 0) == (sums2 == nullptr), "fdbm_gn_table: sums2/C2 mismatch");
  return launch_gn_finalize(sums1, C1, sums2, C2, gamma, beta, batch, pixels, reinterpret_cast<float2*>(table), as_stream(stream),
                            blk_real, reinterpret_cast<float2*>(stats));
}

extern "C" int fdbm_gn_resample_h16(const void* src1, const double* sums1, int C1, const void* src2, const double* sums2,
                                    int C2, const float* gamma, const float* beta, float* table, int batch, int T, int F,
                                    int mode, void* act_out, void* raw_out, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(src1 && sums1 && gamma && beta && table && act_out && raw_out && batch > 0, "fdbm_gn_resample_h16: null pointer");
  FDBM_REQUIRE((C2 == 0) == (src2 == nullptr) && (C2 == 0 || sums2), "fdbm_gn_resample_h16: src2/C2 mismatch");
  float2* tab = reinterpret_cast<float2*>(table);
  if (int rc = launch_gn_finalize(sums1, C1, sums2, C2, gamma, beta, batch, static_cast<int64_t>(T) * F, tab, as_stream(stream)))
    return rc;
  return launch_gn_resample16(reinterpret_cast<const op_t*>(src1), C1, reinterpret_cast<const op_t*>(src2), C2, tab, batch, T, F,
                              mode, reinterpret_cast<op_t*>(act_out), reinterpret_cast<op_t*>(raw_out), as_stream(stream));
}
