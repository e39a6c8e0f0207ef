// HBM-bound backward passes of the training step (SURVEY.md section 8 A10): everything between the tensor-core
// dgrad / wgrad kernels.  Gradients of activations travel as 16-bit GEMM operands (loss-scaled by the caller) with
// fp32 accumulation buffers on the residual stream; parameter gradients are fp32 and un-scaled on the way out.
//
//   grad_prepare     g16 = scale * g (fp32 -> 16-bit) [+ dst += scale * g] + per-(b,c) sums         (layerspp.py:270-274)
//   gn_bwd_reduce    per-(b,c) sums of g_y and g_y * xhat for GroupNorm(+SiLU) backward                (layerspp.py:242-246)
//   gn_bwd_apply     g_x = rstd * (gamma * g_y - mean_g(gamma g_y) - xhat * mean_g(gamma g_y xhat))
//   gn_param_grad    dgamma, dbeta from the reduce sums
//   fir_resample16   FIR up/down of a 16-bit tensor (adjoints of up_or_down_sampling.py:195-257)
//   col_sums_to      bias / FiLM gradients from per-(b,c) sums
//   attention_bwd    softmax-attention backward (layerspp.py:82-86)
//   adam_ema         Adam + gradient clipping + EMA on the flat parameter buffer (model.py:101,129-132)
#include "common.cuh"

namespace fdbm {
namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}

// ------------------------------------------------------------------------------------------------
// grad_prepare: block = (C/4 float4 lanes) x pixel lanes over a run of pixels of one utterance
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
grad_prepare_kernel(const float* __restrict__ g, int64_t P, int C, int64_t px_per_block, float scale,
                    op_t* __restrict__ g16, float* __restrict__ acc_dst, double* __restrict__ sums, int acc_first) {
  pdl_wait_then_trigger();
  __shared__ float4 red[256];
  const int cg = C / 4, pl = 256 / cg;
  const int ci = threadIdx.x % cg, pi = threadIdx.x / cg;
  const int b = blockIdx.y;
  const int64_t p0 = blockIdx.x * px_per_block, p1 = min(P, p0 + px_per_block);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (pi < pl) {
    const int64_t base = static_cast<int64_t>(b) * P * cg + ci;
#pragma unroll 4
    for (int64_t p = p0 + pi; p < p1; p += pl) {
      float4 v = reinterpret_cast<const float4*>(g)[base + p * cg];
      v.x *= scale; v.y *= scale; v.z *= scale; v.w *= scale;
      if (g16) reinterpret_cast<uint2*>(g16)[base + p * cg] = make_uint2(pack_op2(v.x, v.y), pack_op2(v.z, v.w));
      if (acc_dst) {
        float4 d = v;
        if (!acc_first) { const float4 o = reinterpret_cast<float4*>(acc_dst)[base + p * cg]; d.x += o.x; d.y += o.y; d.z += o.z; d.w += o.w; }
        reinterpret_cast<float4*>(acc_dst)[base + p * cg] = d;
      }
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  }
  if (!sums) return;
  red[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x < cg) {
    double d[4] = {0, 0, 0, 0};
    for (int j = 0; j < pl; ++j) {
      const float4 a = red[j * cg + threadIdx.x];
      d[0] += a.x; d[1] += a.y; d[2] += a.z; d[3] += a.w;
    }
    double* o = sums + static_cast<int64_t>(b) * C + threadIdx.x * 4;
#pragma unroll
    for (int j = 0; j < 4; ++j) atomicAdd(o + j, d[j]);
  }
}

// ------------------------------------------------------------------------------------------------
// GroupNorm (+SiLU) backward.  y = x * sc + sh (table), a = act(y); given g_a:
//   g_y = g_a * act'(y),  xhat = (x - mean_g) * rstd_g
//   S1[b,c] = sum_px g_y,  S2[b,c] = sum_px g_y * xhat                                   (reduce)
//   g_x = rstd_g * (gamma_c g_y - m1_g - xhat m2_g),  m{1,2}_g = mean over the group of gamma_c * S{1,2}   (apply)
// The normalised tensor may be the channel concatenation of two sources: the kernels work on ONE source whose
// channels sit at offset c_off of the concatenation (C_tot channels); g_a has row stride g_ld.
// Thread -> 8 consecutive channels and a lane of pixels.
// ------------------------------------------------------------------------------------------------
struct GnBwdArgs {
  const op_t* g_a; int g_ld; int g_coff;       // gradient w.r.t. the activation output [B,P,g_ld], channels g_coff..
  const void* x; int x16;                      // source [B,P,C] fp32 or 16-bit
  int C, C_tot, c_off;
  const float2* tab;                           // [B,C_tot] (scale, shift)
  const float2* stats;                         // [B,G] (mean, rstd)
  const float* gamma;                          // [C_tot]
  int act;
  int64_t P;
  double* S;                                   // [B,C_tot,2]
  // apply outputs
  float* acc_dst;                              // fp32 [B,P,C]: += g_x   (or nullptr)
  int acc_first;                               // ... = g_x: the first contribution of this backward pass to that buffer
  op_t* out16;                                 // 16-bit [B,P,C] = g_x   (or nullptr)
  double* out_sums;                            // [B,C]: += sum_px g_x   (with out16; or nullptr)
  double inv_count;                            // 1 / (channels per group * P)
};

__device__ __forceinline__ void load8(const GnBwdArgs& a, int64_t idx8, float (&x)[8]) {
  if (a.x16) {
    const uint4 raw = reinterpret_cast<const uint4*>(a.x)[idx8];
    const op2_t* h2 = reinterpret_cast<const op2_t*>(&raw);
#pragma unroll
    for (int j = 0; j < 4; ++j) { const float2 f2 = op22f2(h2[j]); x[2 * j] = f2.x; x[2 * j + 1] = f2.y; }
  } else {
    const float4 x0 = reinterpret_cast<const float4*>(a.x)[idx8 * 2], x1 = reinterpret_cast<const float4*>(a.x)[idx8 * 2 + 1];
    x[0] = x0.x; x[1] = x0.y; x[2] = x0.z; x[3] = x0.w; x[4] = x1.x; x[5] = x1.y; x[6] = x1.z; x[7] = x1.w;
  }
}
// d SiLU / dy = sg + y sg (1 - sg), sg = sigmoid(y) = 1/2 + tanh(y/2)/2: one MUFU.TANH instead of EX2 + an IEEE division
// (these passes were instruction-bound, not HBM-bound: the division alone was a third of their instructions)
constexpr int GNBWD_BLOCKS = 4;      // resident blocks per SM the register allocation must allow
constexpr int GNBWD_UNROLL = 2;      // pixels of a thread's lane in flight per loop trip (measured, norm + elementwise part of a 16-crop backward: 1 -> 24.45 ms, 2 -> 24.00; with 3 or 2 blocks per SM and 80 - 96 registers 25.5 - 26.0)
template <bool APPLY>
__global__ void __launch_bounds__(256, GNBWD_BLOCKS)
gn_bwd_kernel(const GnBwdArgs a, int px_per_block) {
  pdl_wait_then_trigger();
  __shared__ float s_m1[32], s_m2[32];
  __shared__ float s_red[256 * 16];
  const int b = blockIdx.y;
  const int G = min(a.C_tot / 4, 32), cpg = a.C_tot / G;
  if (APPLY) {
    if (threadIdx.x < G) {
      double m1 = 0, m2 = 0;
      for (int j = 0; j < cpg; ++j) {
        const int c = threadIdx.x * cpg + j;
        const double* e = a.S + (static_cast<int64_t>(b) * a.C_tot + c) * 2;
        m1 += a.gamma[c] * e[0];
        m2 += a.gamma[c] * e[1];
      }
      s_m1[threadIdx.x] = static_cast<float>(m1 * a.inv_count);
      s_m2[threadIdx.x] = static_cast<float>(m2 * a.inv_count);
    }
    __syncthreads();
  }
  const int cg8 = a.C / 8, npl = 256 / cg8;
  const int g8 = threadIdx.x % cg8, pl = threadIdx.x / cg8;
  const int c0 = g8 * 8;                                   // channel inside this source
  // packed fp32x2 arithmetic (channel pairs).  Per-channel constants: (scale, shift) of y = GN(x); the rest is per GROUP, and a
  // group has a multiple of 4 channels, so channels c0..c0+3 and c0+4..c0+7 each share one set (register diet: 4 blocks per SM)
  float2 sc[4], sh[4];
  float ar[2], br[2], k2[2], k3[2];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int c = a.c_off + c0 + 2 * j;
    const float2 t0 = a.tab[static_cast<int64_t>(b) * a.C_tot + c], t1 = a.tab[static_cast<int64_t>(b) * a.C_tot + c + 1];
    sc[j] = make_float2(t0.x, t1.x); sh[j] = make_float2(t0.y, t1.y);    // scale = gamma * rstd: also the k1 of the apply pass
  }
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    const int g = (a.c_off + c0 + 4 * hf) / cpg;
    const float2 st = a.stats[static_cast<int64_t>(b) * G + g];
    ar[hf] = st.y; br[hf] = -st.x * st.y;                  // xhat = x * rstd - mean * rstd
    k2[hf] = APPLY ? -st.y * s_m1[g] : 0.f;
    k3[hf] = APPLY ? -st.y * s_m2[g] : 0.f;
  }
  const float2 half2v = make_float2(0.5f, 0.5f), one2 = make_float2(1.0f, 1.0f), mone2 = make_float2(-1.0f, -1.0f);
  float2 s1[4], s2[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { s1[j] = make_float2(0.f, 0.f); s2[j] = make_float2(0.f, 0.f); }
  const int64_t p0 = static_cast<int64_t>(blockIdx.x) * px_per_block, p1 = min(a.P, p0 + px_per_block);
  if (pl < npl) {
#pragma unroll GNBWD_UNROLL
    for (int64_t p = p0 + pl; p < p1; p += npl) {
      const int64_t row = static_cast<int64_t>(b) * a.P + p;
      float xs[8];
      load8(a, row * cg8 + g8, xs);
      const uint4 raw = *reinterpret_cast<const uint4*>(a.g_a + row * a.g_ld + a.g_coff + c0);
      const op2_t* h2 = reinterpret_cast<const op2_t*>(&raw);
      float2 gx[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 x = make_float2(xs[2 * j], xs[2 * j + 1]);
        float2 gy = op22f2(h2[j]);
        if (a.act) {                                       // d SiLU / dy = sg + y sg (1 - sg), sg = 1/2 + tanh(y/2)/2
          const float2 y = __ffma2_rn(x, sc[j], sh[j]);
          const float2 hy = __fmul2_rn(y, half2v);
          float2 th;
          asm("tanh.approx.f32 %0, %1;" : "=f"(th.x) : "f"(hy.x));
          asm("tanh.approx.f32 %0, %1;" : "=f"(th.y) : "f"(hy.y));
          const float2 sg = __ffma2_rn(th, half2v, half2v);
          const float2 d = __ffma2_rn(__fmul2_rn(y, sg), __ffma2_rn(sg, mone2, one2), sg);
          gy = __fmul2_rn(gy, d);
        }
        const int hf = j >> 1;
        const float2 xh = __ffma2_rn(x, make_float2(ar[hf], ar[hf]), make_float2(br[hf], br[hf]));
        if (APPLY) {
          // gamma rstd gy - rstd m1 - rstd m2 xh (signs folded in)
          gx[j] = __ffma2_rn(make_float2(k3[hf], k3[hf]), xh, __ffma2_rn(sc[j], gy, make_float2(k2[hf], k2[hf])));
          s1[j] = __fadd2_rn(s1[j], gx[j]);
        } else {
          s1[j] = __fadd2_rn(s1[j], gy);
          s2[j] = __ffma2_rn(gy, xh, s2[j]);
        }
      }
      if (APPLY) {
        if (a.acc_dst) {
          float4* d = reinterpret_cast<float4*>(a.acc_dst) + (row * cg8 + g8) * 2;
          float4 d0 = make_float4(gx[0].x, gx[0].y, gx[1].x, gx[1].y), d1 = make_float4(gx[2].x, gx[2].y, gx[3].x, gx[3].y);
          if (!a.acc_first) {
            const float4 o0 = d[0], o1 = d[1];
            d0.x += o0.x; d0.y += o0.y; d0.z += o0.z; d0.w += o0.w;
            d1.x += o1.x; d1.y += o1.y; d1.z += o1.z; d1.w += o1.w;
          }
          d[0] = d0; d[1] = d1;
        }
        if (a.out16)
          reinterpret_cast<uint4*>(a.out16)[row * cg8 + g8] =
              make_uint4(pack_op2(gx[0].x, gx[0].y), pack_op2(gx[1].x, gx[1].y), pack_op2(gx[2].x, gx[2].y), pack_op2(gx[3].x, gx[3].y));
      }
    }
  }
  if (APPLY && !a.out_sums) return;
  // block reduction over the pixel lanes, then one double atomic per channel and block
  float* red = s_red;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[threadIdx.x * 16 + 2 * j] = s1[j].x; red[threadIdx.x * 16 + 2 * j + 1] = s1[j].y;
    red[threadIdx.x * 16 + 8 + 2 * j] = s2[j].x; red[threadIdx.x * 16 + 8 + 2 * j + 1] = s2[j].y;
  }
  __syncthreads();
  if (threadIdx.x < cg8 * 8) {
    const int gg = threadIdx.x / 8, j = threadIdx.x % 8;
    double d1 = 0, d2 = 0;
    for (int l = 0; l < npl; ++l) {
      d1 += red[(l * cg8 + gg) * 16 + j];
      d2 += red[(l * cg8 + gg) * 16 + 8 + j];
    }
    if (APPLY) {
      atomicAdd(a.out_sums + static_cast<int64_t>(b) * a.C + gg * 8 + j, d1);
    } else {
      double* o = a.S + (static_cast<int64_t>(b) * a.C_tot + a.c_off + gg * 8 + j) * 2;
      atomicAdd(o, d1);
      atomicAdd(o + 1, d2);
    }
  }
}

// dgamma[c] += inv_scale * sum_b S[b,c,1],  dbeta[c] += inv_scale * sum_b S[b,c,0]
__global__ void gn_param_grad_kernel(const double* __restrict__ S, int B, int C, float inv_scale, float* __restrict__ dgamma,
                                     float* __restrict__ dbeta) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  double s1 = 0, s2 = 0;
  for (int b = 0; b < B; ++b) { s1 += S[(static_cast<int64_t>(b) * C + c) * 2]; s2 += S[(static_cast<int64_t>(b) * C + c) * 2 + 1]; }
  dbeta[c] += inv_scale * static_cast<float>(s1);
  dgamma[c] += inv_scale * static_cast<float>(s2);
}

// (mean, rstd) per (utterance, group) of a GroupNorm over the concatenation of up to two tensors
__global__ void gn_stats_kernel(const double* __restrict__ sums1, int C1, const double* __restrict__ sums2, int C2, double pixels,
                                float2* __restrict__ stats) {
  const int C = C1 + C2, b = blockIdx.x;
  const int G = min(C / 4, 32), cpg = C / G;
  if (threadIdx.x >= G) return;
  double s = 0, q = 0;
  for (int j = 0; j < cpg; ++j) {
    const int c = threadIdx.x * cpg + j;
    const double* e = c < C1 ? sums1 + (static_cast<int64_t>(b) * C1 + c) * 2 : sums2 + (static_cast<int64_t>(b) * C2 + (c - C1)) * 2;
    s += e[0]; q += e[1];
  }
  const double cnt = cpg * pixels, mean = s / cnt;
  double var = q / cnt - mean * mean;
  if (var < 0) var = 0;
  stats[static_cast<int64_t>(b) * G + threadIdx.x] = make_float2(static_cast<float>(mean), static_cast<float>(1.0 / sqrt(var + 1e-6)));
}

// ------------------------------------------------------------------------------------------------
// FIR x2 up / down of a 16-bit tensor with a scale: the adjoints of the forward resampling are
//   adjoint(down) = up / 4,  adjoint(up) = 4 * down   (2-D).  Output 16-bit and/or fp32 accumulate.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void taps1d(int o, int mode, int (&pos)[4], float (&w)[4], int& n) {
  if (mode == 1) {
    n = 4; pos[0] = 2 * o - 1; pos[1] = 2 * o; pos[2] = 2 * o + 1; pos[3] = 2 * o + 2;
    w[0] = 0.125f; w[1] = 0.375f; w[2] = 0.375f; w[3] = 0.125f;
  } else {
    const int i = o >> 1;
    n = 2;
    if (o & 1) { pos[0] = i; pos[1] = i + 1; w[0] = 0.75f; w[1] = 0.25f; }
    else { pos[0] = i - 1; pos[1] = i; w[0] = 0.25f; w[1] = 0.75f; }
    pos[2] = pos[3] = -1; w[2] = w[3] = 0.f;
  }
}

__global__ void __launch_bounds__(256)
fir_resample16_kernel(const op_t* __restrict__ in, int in_ld, int in_coff, int B, int T, int F, int C, int mode, float scale,
                      op_t* __restrict__ out16, float* __restrict__ acc_dst) {
  pdl_wait_then_trigger();
  const int To = mode == 1 ? T / 2 : T * 2, Fo = mode == 1 ? F / 2 : F * 2;
  const int cg8 = C / 8;
  const int64_t total = static_cast<int64_t>(B) * To * Fo * cg8;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < total; i += 256ll * gridDim.x) {
    const int g8 = static_cast<int>(i % cg8);
    int64_t p = i / cg8;
    const int fo = static_cast<int>(p % Fo); p /= Fo;
    const int to = static_cast<int>(p % To);
    const int b = static_cast<int>(p / To);
    int tp[4], fp[4], nt, nf; float tw[4], fw[4];
    taps1d(to, mode, tp, tw, nt);
    taps1d(fo, mode, fp, fw, nf);
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    for (int u = 0; u < nt; ++u) {
      if (tp[u] < 0 || tp[u] >= T) continue;
      for (int v = 0; v < nf; ++v) {
        if (fp[v] < 0 || fp[v] >= F) continue;
        const float w = tw[u] * fw[v] * scale;
        const uint4 raw = *reinterpret_cast<const uint4*>(in + ((static_cast<int64_t>(b) * T + tp[u]) * F + fp[v]) * in_ld + in_coff + g8 * 8);
        const op2_t* h2 = reinterpret_cast<const op2_t*>(&raw);
#pragma unroll
        for (int j = 0; j < 4; ++j) { const float2 f2 = op22f2(h2[j]); acc[2 * j] = fmaf(w, f2.x, acc[2 * j]); acc[2 * j + 1] = fmaf(w, f2.y, acc[2 * j + 1]); }
      }
    }
    if (out16)
      reinterpret_cast<uint4*>(out16)[i] = make_uint4(pack_op2(acc[0], acc[1]), pack_op2(acc[2], acc[3]), pack_op2(acc[4], acc[5]), pack_op2(acc[6], acc[7]));
    if (acc_dst) {
      float4* d = reinterpret_cast<float4*>(acc_dst) + i * 2;
      float4 d0 = d[0], d1 = d[1];
      d0.x += acc[0]; d0.y += acc[1]; d0.z += acc[2]; d0.w += acc[3];
      d1.x += acc[4]; d1.y += acc[5]; d1.z += acc[6]; d1.w += acc[7];
      d[0] = d0; d[1] = d1;
    }
  }
}

// per-(b,c) sums of a 16-bit tensor [B,P,ld] (channels c_off..c_off+C): sums[b*C + c] +=
__global__ void __launch_bounds__(256)
col_sums16_kernel(const op_t* __restrict__ in, int ld, int c_off, int64_t P, int C, int64_t px_per_block, double* __restrict__ sums) {
  __shared__ float red[256 * 8];
  const int cg8 = C / 8, npl = 256 / cg8;
  const int g8 = threadIdx.x % cg8, pl = threadIdx.x / cg8;
  const int b = blockIdx.y;
  float s[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = 0.f;
  const int64_t p0 = blockIdx.x * px_per_block, p1 = min(P, p0 + px_per_block);
  if (pl < npl)
    for (int64_t p = p0 + pl; p < p1; p += npl) {
      const uint4 raw = *reinterpret_cast<const uint4*>(in + (static_cast<int64_t>(b) * P + p) * ld + c_off + g8 * 8);
      const op2_t* h2 = reinterpret_cast<const op2_t*>(&raw);
#pragma unroll
      for (int j = 0; j < 4; ++j) { const float2 f2 = op22f2(h2[j]); s[2 * j] += f2.x; s[2 * j + 1] += f2.y; }
    }
#pragma unroll
  for (int j = 0; j < 8; ++j) red[threadIdx.x * 8 + j] = s[j];
  __syncthreads();
  if (threadIdx.x < cg8 * 8) {
    const int gg = threadIdx.x / 8, j = threadIdx.x % 8;
    double d = 0;
    for (int l = 0; l < npl; ++l) d += red[(l * cg8 + gg) * 8 + j];
    atomicAdd(sums + static_cast<int64_t>(b) * C + gg * 8 + j, d);
  }
}

// dst[c] += inv_scale * sum_b sums[b*C + c];  per_b[b*ld + c] = inv_scale * sums[b*C + c] (optional, FiLM gradient)
__global__ void col_sums_to_kernel(const double* __restrict__ sums, int B, int C, float inv_scale, float* __restrict__ dst,
                                   float* __restrict__ per_b, int per_b_ld) {
  const int c = blockIdx.x * 256 + threadIdx.x;
  if (c >= C) return;
  double s = 0;
  for (int b = 0; b < B; ++b) {
    const double v = sums[static_cast<int64_t>(b) * C + c];
    s += v;
    if (per_b) per_b[static_cast<int64_t>(b) * per_b_ld + c] = inv_scale * static_cast<float>(v);
  }
  if (dst) dst[c] += inv_scale * static_cast<float>(s);
}

// ------------------------------------------------------------------------------------------------
// Attention backward.  S = scale * q k^T, P = softmax(S), o = P v.
//   kernel A (warp per query i): recompute P_i, dP_ij = dO_i . v_j, D_i = sum_j P_ij dP_ij, dS_ij = P_ij (dP_ij - D_i),
//                                dq_i = scale * sum_j dS_ij k_j;  stores P_i and dS_i rows to scratch [B,L,L]
//   kernel B (warp per key j):   dv_j = sum_i P_ij dO_i,  dk_j = scale * sum_i dS_ij q_i
// ------------------------------------------------------------------------------------------------
constexpr int ATT_WARPS = 8;

__device__ __forceinline__ float dot_row(const op_t* row, const float* vec, int C) {
  const uint4* kr = reinterpret_cast<const uint4*>(row);
  float acc = 0.f;
  for (int c8 = 0; c8 < C / 8; ++c8) {
    const uint4 raw = kr[c8];
    const op2_t* h2 = reinterpret_cast<const op2_t*>(&raw);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float2 f2 = op22f2(h2[u]);
      acc = fmaf(f2.x, vec[c8 * 8 + 2 * u], acc);
      acc = fmaf(f2.y, vec[c8 * 8 + 2 * u + 1], acc);
    }
  }
  return acc;
}

__global__ void __launch_bounds__(ATT_WARPS * 32)
attention_bwd_q_kernel(const op_t* __restrict__ q, const op_t* __restrict__ k, const op_t* __restrict__ v, int ld,
                       const op_t* __restrict__ d_o, int ldo, int L, int C, float scale, float* __restrict__ Pm,
                       float* __restrict__ dSm, op_t* __restrict__ dq, int ldg) {
  extern __shared__ float sm[];                       // per warp: q[C] | do[C] | p[L] | ds[L]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int qi = blockIdx.x * ATT_WARPS + warp;
  if (qi >= L) return;
  float* sq = sm + warp * (2 * C + 2 * L);
  float* sdo = sq + C;
  float* sp = sdo + C;
  float* sds = sp + L;
  const int64_t base = static_cast<int64_t>(b) * L;
  for (int c = lane; c < C; c += 32) {
    sq[c] = op2f(q[(base + qi) * ld + c]) * scale;
    sdo[c] = op2f(d_o[(base + qi) * ldo + c]);
  }
  __syncwarp();
  float mx = -INFINITY;
  for (int j = lane; j < L; j += 32) {
    const float sc = dot_row(k + (base + j) * ld, sq, C);
    sp[j] = sc;
    sds[j] = dot_row(v + (base + j) * ld, sdo, C);   // dP_ij
    mx = fmaxf(mx, sc);
  }
#pragma unroll
  for (int s = 16; s >= 1; s >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, s));
  float sum = 0.f;
  for (int j = lane; j < L; j += 32) { const float e = __expf(sp[j] - mx); sp[j] = e; sum += e; }
  sum = warp_sum(sum);
  const float inv = 1.0f / sum;
  float dsum = 0.f;
  for (int j = lane; j < L; j += 32) { const float pj = sp[j] * inv; sp[j] = pj; dsum = fmaf(pj, sds[j], dsum); }
  dsum = warp_sum(dsum);
  float* Prow = Pm + (base + qi) * L;
  float* dSrow = dSm + (base + qi) * L;
  for (int j = lane; j < L; j += 32) {
    const float ds = sp[j] * (sds[j] - dsum);
    sds[j] = ds;
    Prow[j] = sp[j];
    dSrow[j] = ds;
  }
  __syncwarp();
  for (int c0 = lane * 8; c0 < C; c0 += 256) {
    float acc[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) acc[u] = 0.f;
    for (int j = 0; j < L; ++j) {
      const float w = sds[j];
      const uint4 raw = *reinterpret_cast<const uint4*>(k + (base + j) * ld + c0);
      const op2_t* h2 = reinterpret_cast<const op2_t*>(&raw);
#pragma unroll
      for (int u = 0; u < 4; ++u) { const float2 f2 = op22f2(h2[u]); acc[2 * u] = fmaf(w, f2.x, acc[2 * u]); acc[2 * u + 1] = fmaf(w, f2.y, acc[2 * u + 1]); }
    }
    op2_t ov[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) ov[u] = f2op2(acc[2 * u] * scale, acc[2 * u + 1] * scale);
    *reinterpret_cast<uint4*>(dq + (base + qi) * ldg + c0) = *reinterpret_cast<uint4*>(ov);
  }
}

__global__ void __launch_bounds__(ATT_WARPS * 32)
attention_bwd_kv_kernel(const op_t* __restrict__ q, int ld, const op_t* __restrict__ d_o, int ldo, int L, int C, float scale,
                        const float* __restrict__ Pm, const float* __restrict__ dSm, op_t* __restrict__ dk,
                        op_t* __restrict__ dv, int ldg) {
  extern __shared__ float sm[];                       // per warp: p_col[L] | ds_col[L]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int b = blockIdx.y;
  const int kj = blockIdx.x * ATT_WARPS + warp;
  if (kj >= L) return;
  float* sp = sm + warp * 2 * L;
  float* sds = sp + L;
  const int64_t base = static_cast<int64_t>(b) * L;
  for (int i = lane; i < L; i += 32) { sp[i] = Pm[(base + i) * L + kj]; sds[i] = dSm[(base + i) * L + kj]; }
  __syncwarp();
  for (int c0 = lane * 8; c0 < C; c0 += 256) {
    float av[8], ak[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) { av[u] = 0.f; ak[u] = 0.f; }
    for (int i = 0; i < L; ++i) {
      const float wp = sp[i], wd = sds[i];
      const uint4 r1 = *reinterpret_cast<const uint4*>(d_o + (base + i) * ldo + c0);
      const uint4 r2 = *reinterpret_cast<const uint4*>(q + (base + i) * ld + c0);
      const op2_t* h1 = reinterpret_cast<const op2_t*>(&r1);
      const op2_t* h2 = reinterpret_cast<const op2_t*>(&r2);
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float2 f1 = op22f2(h1[u]), f2 = op22f2(h2[u]);
        av[2 * u] = fmaf(wp, f1.x, av[2 * u]); av[2 * u + 1] = fmaf(wp, f1.y, av[2 * u + 1]);
        ak[2 * u] = fmaf(wd, f2.x, ak[2 * u]); ak[2 * u + 1] = fmaf(wd, f2.y, ak[2 * u + 1]);
      }
    }
    op2_t ov[4], ok[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { ov[u] = f2op2(av[2 * u], av[2 * u + 1]); ok[u] = f2op2(ak[2 * u] * scale, ak[2 * u + 1] * scale); }
    *reinterpret_cast<uint4*>(dv + (base + kj) * ldg + c0) = *reinterpret_cast<uint4*>(ov);
    *reinterpret_cast<uint4*>(dk + (base + kj) * ldg + c0) = *reinterpret_cast<uint4*>(ok);
  }
}

// ------------------------------------------------------------------------------------------------
// Optimiser: total squared gradient norm (double), then Adam with clipping and EMA on flat buffers.
// ------------------------------------------------------------------------------------------------
// deterministic (fixed grid, fixed summation order): every DDP rank must derive bit-identical clipping coefficients
// from the bit-identical all-reduced gradients, or the replicas drift apart
constexpr int SUMSQ_BLOCKS = 1024;
__global__ void __launch_bounds__(256)
sumsq_kernel(const float* __restrict__ g, int64_t n, double* __restrict__ partial) {
  __shared__ double red[256];
  double s = 0;
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += 256ll * gridDim.x) { const double v = g[i]; s += v * v; }
  red[threadIdx.x] = s;
  __syncthreads();
  for (int k = 128; k > 0; k >>= 1) { if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k]; __syncthreads(); }
  if (threadIdx.x == 0) partial[1 + blockIdx.x] = red[0];
}
// state (optional, device): {applied updates, skipped steps, last gradient norm (un-scaled), reserved}.  A step whose
// gradient norm is not finite (fp16 overflow of a loss-scaled activation gradient) is SKIPPED: it advances neither Adam's
// bias correction nor torch_ema's num_updates, and is counted so that the host can back the loss scale off.
__global__ void __launch_bounds__(256)
sumsq_final_kernel(double* __restrict__ partial, int n_blocks, double* __restrict__ state, float grad_div) {
  __shared__ double red[256];
  double s = 0;
  for (int i = threadIdx.x; i < n_blocks; i += 256) s += partial[1 + i];
  red[threadIdx.x] = s;
  __syncthreads();
  for (int k = 128; k > 0; k >>= 1) { if (threadIdx.x < k) red[threadIdx.x] += red[threadIdx.x + k]; __syncthreads(); }
  if (threadIdx.x == 0) {
    partial[0] = red[0];
    if (state) {
      const double norm = sqrt(red[0]) / grad_div;
      state[2] = norm;
      if (isfinite(norm)) state[0] += 1.0; else state[1] += 1.0;
    }
  }
}

__global__ void __launch_bounds__(256)
adam_ema_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                float* __restrict__ ema, const unsigned char* __restrict__ trainable, int64_t n, const double* __restrict__ sumsq,
                float grad_div, float clip, float lr, float beta1, float beta2, float eps, int step_host, const double* __restrict__ state,
                float ema_decay, int ema_warmup) {
  // torch.nn.utils.clip_grad_norm_: coef = clip / (norm + 1e-6), applied when < 1
  const double norm = sqrt(*sumsq) / grad_div;
  if (!isfinite(norm)) return;                        // overflowed step (loss scale too large): skip, as GradScaler does
  // update count: the host's when given, else the device-side count of APPLIED steps (already incremented for this one)
  const double n_upd = step_host > 0 ? static_cast<double>(step_host) : state[0];
  const float bc1 = static_cast<float>(1.0 - pow(static_cast<double>(beta1), n_upd));
  const float bc2 = static_cast<float>(1.0 - pow(static_cast<double>(beta2), n_upd));
  // torch_ema.ExponentialMovingAverage.update (use_num_updates=True, the default the reference constructs it with,
  // fdbm/model.py:56): decay = min(decay, (1 + n) / (10 + n)); shadow -= (1 - decay) * (shadow - param)
  float omd = 1.0f - ema_decay;
  if (ema_warmup) omd = static_cast<float>(1.0 - fmin(static_cast<double>(ema_decay), (1.0 + n_upd) / (10.0 + n_upd)));
  float coef = 1.0f / grad_div;
  if (clip > 0.f) { const double c = clip / (norm + 1e-6); if (c < 1.0) coef *= static_cast<float>(c); }
  for (int64_t i = blockIdx.x * 256ll + threadIdx.x; i < n; i += 256ll * gridDim.x) {
    if (trainable && !trainable[i]) continue;
    const float gi = g[i] * coef;
    const float mi = beta1 * m[i] + (1.0f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.0f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float pi = p[i] - lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
    p[i] = pi;
    if (ema) { const float e = ema[i]; ema[i] = e - omd * (e - pi); }
  }
}

int grid_for(int64_t n) { return static_cast<int>(std::min<int64_t>(ceil_div64(n, 256), static_cast<int64_t>(num_sms()) * 16)); }

}  // namespace

int launch_grad_prepare(const float* g, int B, int64_t P, int C, float scale, op_t* g16, float* acc_dst, double* sums, cudaStream_t s,
                        bool acc_first, bool sums_prezeroed) {
  FDBM_REQUIRE(C % 4 == 0 && C / 4 <= 256 && 256 % (C / 4) == 0, "grad_prepare: unsupported channel count %d", C);
  if (sums && !sums_prezeroed) FDBM_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * B * C, s));
  const int pl = 256 / (C / 4);
  int64_t blocks_x = std::max<int64_t>(1, (static_cast<int64_t>(num_sms()) * 8) / B);
  blocks_x = std::min<int64_t>(blocks_x, std::max<int64_t>(1, P / (pl * 8)));
  const int64_t ppb = ceil_div64(P, blocks_x);
  dim3 grid(static_cast<unsigned>(ceil_div64(P, ppb)), B);
  FDBM_CUDA(launch_maybe_pdl(grad_prepare_kernel, grid, dim3(256), 0, s, pdl_enabled() && B <= pdl_batch_limit(), g, P, C, ppb, scale, g16, acc_dst, sums,
                             acc_first ? 1 : 0));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

static int gn_bwd_grid(const GnBwdArgs& a, int B, dim3* grid, int* ppb) {
  FDBM_REQUIRE(a.C % 8 == 0 && a.C <= 256 && 256 % (a.C / 8) == 0 && a.C_tot % std::min(a.C_tot / 4, 32) == 0 && a.g_ld % 8 == 0 && a.g_coff % 8 == 0,
               "gn_bwd: unsupported channels %d of %d", a.C, a.C_tot);
  const int npl = 256 / (a.C / 8);
  int64_t bx = std::max<int64_t>(1, (static_cast<int64_t>(num_sms()) * 4) / B);
  bx = std::min<int64_t>(bx, std::max<int64_t>(1, a.P / (npl * 4)));
  *ppb = static_cast<int>(ceil_div64(ceil_div64(a.P, bx), npl) * npl);
  *grid = dim3(static_cast<unsigned>(ceil_div64(a.P, *ppb)), B);
  return FDBM_OK;
}

// one source tensor of a (possibly concatenated) GroupNorm: reduce pass.  S must have been zeroed by the caller.
int launch_gn_bwd_reduce(const op_t* g_a, int g_ld, int g_coff, const void* x, int x16, int C, int C_tot, int c_off,
                         const float2* tab, const float2* stats, int act, int B, int64_t P, double* S, cudaStream_t s) {
  GnBwdArgs a{};
  a.g_a = g_a; a.g_ld = g_ld; a.g_coff = g_coff; a.x = x; a.x16 = x16; a.C = C; a.C_tot = C_tot; a.c_off = c_off;
  a.tab = tab; a.stats = stats; a.gamma = nullptr; a.act = act; a.P = P; a.S = S;
  dim3 grid; int ppb;
  if (int rc = gn_bwd_grid(a, B, &grid, &ppb)) return rc;
  FDBM_CUDA(launch_maybe_pdl(gn_bwd_kernel<false>, grid, dim3(256), 0, s, pdl_enabled() && B <= pdl_batch_limit(), a, ppb));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_gn_bwd_apply(const op_t* g_a, int g_ld, int g_coff, const void* x, int x16, int C, int C_tot, int c_off,
                        const float2* tab, const float2* stats, const float* gamma, int act, int B, int64_t P, const double* S,
                        float* acc_dst, op_t* out16, double* out_sums, cudaStream_t s, bool acc_first, bool sums_prezeroed) {
  GnBwdArgs a{};
  a.g_a = g_a; a.g_ld = g_ld; a.g_coff = g_coff; a.x = x; a.x16 = x16; a.C = C; a.C_tot = C_tot; a.c_off = c_off;
  a.tab = tab; a.stats = stats; a.gamma = gamma; a.act = act; a.P = P; a.S = const_cast<double*>(S);
  a.acc_dst = acc_dst; a.out16 = out16; a.out_sums = out_sums; a.acc_first = acc_first ? 1 : 0;
  const int G = std::min(C_tot / 4, 32);
  a.inv_count = 1.0 / (static_cast<double>(C_tot / G) * static_cast<double>(P));
  if (out_sums && !sums_prezeroed) FDBM_CUDA(cudaMemsetAsync(out_sums, 0, sizeof(double) * B * C, s));
  dim3 grid; int ppb;
  if (int rc = gn_bwd_grid(a, B, &grid, &ppb)) return rc;
  FDBM_CUDA(launch_maybe_pdl(gn_bwd_kernel<true>, grid, dim3(256), 0, s, pdl_enabled() && B <= pdl_batch_limit(), a, ppb));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_gn_param_grad(const double* S, int B, int C, float inv_scale, float* dgamma, float* dbeta, cudaStream_t s) {
  gn_param_grad_kernel<<<ceil_div(C, 256), 256, 0, s>>>(S, B, C, inv_scale, dgamma, dbeta);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_gn_stats(const double* sums1, int C1, const double* sums2, int C2, int B, int64_t pixels, float2* stats, cudaStream_t s) {
  gn_stats_kernel<<<B, 32, 0, s>>>(sums1, C1, sums2, C2, static_cast<double>(pixels), stats);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_fir_resample16(const op_t* in, int in_ld, int in_coff, int B, int T, int F, int C, int mode, float scale,
                          op_t* out16, float* acc_dst, cudaStream_t s) {
  FDBM_REQUIRE(C % 8 == 0 && in_ld % 8 == 0 && in_coff % 8 == 0 && (mode == 1 || mode == 2), "fir_resample16: bad arguments");
  FDBM_REQUIRE(mode != 1 || (T % 2 == 0 && F % 2 == 0), "fir_resample16: down-sampling needs even T, F");
  const int To = mode == 1 ? T / 2 : T * 2, Fo = mode == 1 ? F / 2 : F * 2;
  FDBM_CUDA(launch_maybe_pdl(fir_resample16_kernel, dim3(grid_for(static_cast<int64_t>(B) * To * Fo * (C / 8))), dim3(256), 0, s,
                             pdl_enabled() && B <= pdl_batch_limit(), in, in_ld, in_coff, B, T, F, C, mode, scale, out16, acc_dst));
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_col_sums16(const op_t* in, int ld, int c_off, int B, int64_t P, int C, double* sums, cudaStream_t s, bool sums_prezeroed) {
  FDBM_REQUIRE(C % 8 == 0 && C / 8 <= 256, "col_sums16: unsupported channel count %d", C);
  if (!sums_prezeroed) FDBM_CUDA(cudaMemsetAsync(sums, 0, sizeof(double) * B * C, s));
  const int npl = 256 / (C / 8);
  int64_t bx = std::max<int64_t>(1, (static_cast<int64_t>(num_sms()) * 4) / B);
  bx = std::min<int64_t>(bx, std::max<int64_t>(1, P / (npl * 4)));
  const int64_t ppb = ceil_div64(P, bx);
  dim3 grid(static_cast<unsigned>(ceil_div64(P, ppb)), B);
  col_sums16_kernel<<<grid, 256, 0, s>>>(in, ld, c_off, P, C, ppb, sums);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

// every deferred reduction of a backward pass in one launch: block = one descriptor (same arithmetic as col_sums_to_kernel /
// gn_param_grad_kernel: double sum over the utterances, one float conversion, scaled add into the gradient buffer)
__global__ void __launch_bounds__(256) deferred_sums_kernel(const DeferDesc* __restrict__ descs, float inv_scale) {
  const DeferDesc d = descs[blockIdx.x];
  for (int c = threadIdx.x; c < d.C; c += 256) {
    if (d.kind == 0) {
      double s = 0;
      for (int b = 0; b < d.B; ++b) {
        const double v = d.src[static_cast<int64_t>(b) * d.C + c];
        s += v;
        if (d.per_b) d.per_b[static_cast<int64_t>(b) * d.per_b_ld + c] = inv_scale * static_cast<float>(v);
      }
      if (d.dst0) atomicAdd(d.dst0 + c, inv_scale * static_cast<float>(s));
    } else {
      double s1 = 0, s2 = 0;
      for (int b = 0; b < d.B; ++b) { s1 += d.src[(static_cast<int64_t>(b) * d.C + c) * 2]; s2 += d.src[(static_cast<int64_t>(b) * d.C + c) * 2 + 1]; }
      atomicAdd(d.dst1 + c, inv_scale * static_cast<float>(s1));
      atomicAdd(d.dst0 + c, inv_scale * static_cast<float>(s2));
    }
  }
}
int launch_deferred_sums(const DeferDesc* descs_dev, int n_descs, float inv_scale, cudaStream_t s) {
  if (n_descs <= 0) return FDBM_OK;
  deferred_sums_kernel<<<n_descs, 256, 0, s>>>(descs_dev, inv_scale);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_col_sums_to(const double* sums, int B, int C, float inv_scale, float* dst, float* per_b, int per_b_ld, cudaStream_t s) {
  col_sums_to_kernel<<<ceil_div(C, 256), 256, 0, s>>>(sums, B, C, inv_scale, dst, per_b, per_b_ld);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

// g_qkv [B,L,3C] (q | k | v gradients) from d_o [B,L,C];  scratch: 2 * B * L * L floats
int launch_attention_bwd(const op_t* qkv, int B, int L, int C, const op_t* d_o, float* scratch, op_t* g_qkv, cudaStream_t s) {
  FDBM_REQUIRE(C % 8 == 0, "attention_bwd: channels must be a multiple of 8");
  const size_t smem_a = sizeof(float) * ATT_WARPS * (2 * C + 2 * L), smem_b = sizeof(float) * ATT_WARPS * 2 * L;
  FDBM_REQUIRE(smem_a <= 200 * 1024, "attention_bwd: sequence length %d too long", L);
  static PerDeviceOnce attr_once;
  if (attr_once.first(current_device())) {
    FDBM_CUDA(cudaFuncSetAttribute(attention_bwd_q_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    FDBM_CUDA(cudaFuncSetAttribute(attention_bwd_kv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  }
  const float scale = 1.0f / sqrtf(static_cast<float>(C));
  float* Pm = scratch;
  float* dSm = scratch + static_cast<int64_t>(B) * L * L;
  dim3 grid(ceil_div(L, ATT_WARPS), B);
  attention_bwd_q_kernel<<<grid, ATT_WARPS * 32, smem_a, s>>>(qkv, qkv + C, qkv + 2 * C, 3 * C, d_o, C, L, C, scale, Pm, dSm, g_qkv, 3 * C);
  FDBM_LAUNCH_CHECK();
  attention_bwd_kv_kernel<<<grid, ATT_WARPS * 32, smem_b, s>>>(qkv, 3 * C, d_o, C, L, C, scale, Pm, dSm, g_qkv + C, g_qkv + 2 * C, 3 * C);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

int launch_adam_ema(float* p, const float* g, float* m, float* v, float* ema, const unsigned char* trainable, int64_t n,
                    double* sumsq_scratch, float grad_div, float clip, float lr, float beta1, float beta2, float eps, int step,
                    float ema_decay, int ema_warmup, double* state, cudaStream_t s) {
  FDBM_REQUIRE(step > 0 || state, "adam_ema: step == 0 needs the device-side state block");
  sumsq_kernel<<<SUMSQ_BLOCKS, 256, 0, s>>>(g, n, sumsq_scratch);
  FDBM_LAUNCH_CHECK();
  sumsq_final_kernel<<<1, 256, 0, s>>>(sumsq_scratch, SUMSQ_BLOCKS, state, grad_div);
  FDBM_LAUNCH_CHECK();
  adam_ema_kernel<<<grid_for(n), 256, 0, s>>>(p, g, m, v, ema, trainable, n, sumsq_scratch, grad_div, clip, lr, beta1, beta2, eps, step, state,
                                              ema_decay, ema_warmup);
  FDBM_LAUNCH_CHECK();
  return FDBM_OK;
}

}  // namespace fdbm

using namespace fdbm;

// ---- C ABI of the individual backward kernels (tests/test_gpu_train.py checks each against torch autograd) ----
extern "C" int fdbm_groupnorm_act_bwd(const void* g_a, const void* x, int x_is_h16, const double* sums, const float* gamma,
                                      const float* beta, int silu, int batch, int T, int F, int C, float* table, double* S,
                                      float* g_x_acc, void* g_x_h16, float* dgamma, float* dbeta, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(g_a && x && sums && gamma && beta && table && S && batch > 0, "fdbm_groupnorm_act_bwd: null pointer");
  cudaStream_t s = as_stream(stream);
  const int64_t P = static_cast<int64_t>(T) * F;
  const int G = std::min(C / 4, 32);
  float2* tab = reinterpret_cast<float2*>(table);
  float2* stats = tab + static_cast<int64_t>(batch) * C;          // table: B*C*2 + B*G*2 floats
  if (int rc = launch_gn_finalize(sums, C, nullptr, 0, gamma, beta, batch, P, tab, s)) return rc;
  if (int rc = launch_gn_stats(sums, C, nullptr, 0, batch, P, stats, s)) return rc;
  (void)G;
  FDBM_CUDA(cudaMemsetAsync(S, 0, sizeof(double) * 2 * batch * C, s));
  if (int rc = launch_gn_bwd_reduce(reinterpret_cast<const op_t*>(g_a), C, 0, x, x_is_h16, C, C, 0, tab, stats, silu, batch, P, S, s)) return rc;
  if (int rc = launch_gn_bwd_apply(reinterpret_cast<const op_t*>(g_a), C, 0, x, x_is_h16, C, C, 0, tab, stats, gamma, silu, batch, P, S,
                                   g_x_acc, reinterpret_cast<op_t*>(g_x_h16), nullptr, s)) return rc;
  if (dgamma && dbeta) return launch_gn_param_grad(S, batch, C, 1.0f, dgamma, dbeta, s);
  return FDBM_OK;
}

extern "C" int fdbm_fir_resample_h16(const void* in, int batch, int T, int F, int C, int mode, float scale, void* out, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(in && out && batch > 0, "fdbm_fir_resample_h16: null pointer");
  return launch_fir_resample16(reinterpret_cast<const op_t*>(in), C, 0, batch, T, F, C, mode, scale, reinterpret_cast<op_t*>(out), nullptr,
                               as_stream(stream));
}

extern "C" int fdbm_attention_bwd(const void* qkv, int batch, int L, int C, const void* d_o, float* scratch, void* g_qkv, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(qkv && d_o && scratch && g_qkv && batch > 0 && L > 0, "fdbm_attention_bwd: bad arguments");
  return launch_attention_bwd(reinterpret_cast<const op_t*>(qkv), batch, L, C, reinterpret_cast<const op_t*>(d_o), scratch,
                              reinterpret_cast<op_t*>(g_qkv), as_stream(stream));
}

extern "C" int fdbm_adam_ema_step(float* params, const float* grads, float* m, float* v, float* ema, int64_t n, double* scratch,
                                  float grad_div, float clip_norm, float lr, float beta1, float beta2, float eps, int step,
                                  float ema_decay, int ema_warmup, double* state, void* stream) {
  if (int rc = require_sm100()) return rc;
  FDBM_REQUIRE(params && grads && m && v && scratch && n > 0 && (step >= 1 || (step == 0 && state)), "fdbm_adam_ema_step: bad arguments");
  return launch_adam_ema(params, grads, m, v, ema, nullptr, n, scratch, grad_div, clip_norm, lr, beta1, beta2, eps, step, ema_decay,
                         ema_warmup, state, as_stream(stream));
}
