// Shared host/device helpers for libfdbm_b200: error reporting, launch checks, small math.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <stdio.h>
#include <string>
#include <algorithm>
#include "../../include/fdbm_b200.h"

namespace fdbm {

// thread-local message behind fdbm_last_error()
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what, const char* file, int line);

#define FDBM_CUDA(expr)                                                          \
  do {                                                                           \
    cudaError_t _e = (expr);                                                     \
    if (_e != cudaSuccess) return ::fdbm::cuda_fail(_e, #expr, __FILE__, __LINE__); \
  } while (0)

#define FDBM_REQUIRE(cond, ...)                \
  do {                                         \
    if (!(cond)) {                             \
      ::fdbm::set_error(__VA_ARGS__);          \
      return FDBM_EINVAL;                      \
    }                                          \
  } while (0)

// Every launch is followed by this: catches bad launch configurations immediately.
#define FDBM_LAUNCH_CHECK() FDBM_CUDA(cudaGetLastError())

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

int require_sm100();   // FDBM_OK or FDBM_EARCH (cached per device)
// Kernels that may be launched with programmatic stream serialisation call this FIRST: nothing of the previous kernel in the
// stream is read or overwritten before it has completed, and the kernel behind this one may become resident (it waits the same way).
__device__ __forceinline__ void pdl_wait_then_trigger() {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
// launch `kernel` with the programmatic-stream-serialisation attribute when `pdl` (short launches: the launch latency and block
// ramp-up overlap the previous kernel's tail), plainly otherwise.  The kernel must start with pdl_wait_then_trigger().
template <typename... KArgs, typename... Args>
inline cudaError_t launch_maybe_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, bool pdl, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
int pdl_batch_limit();   // see api.cu
struct PdlBatchScope { int prev; explicit PdlBatchScope(int limit); ~PdlBatchScope(); PdlBatchScope(const PdlBatchScope&) = delete; };
bool pdl_enabled();    // programmatic dependent launch of the convolution / GroupNorm-table kernels (FDBM_PDL=0 in the environment disables it)
int num_sms();
int current_device();  // cudaGetDevice, -1 on failure

// "done once per device" flag for cudaFuncSetAttribute opt-ins: function attributes are per device, so a process that
// drives several GPUs (infer_folder.py:70-74 spawns workers with .to(f'cuda:{gpu_id}')) must set them on each one.
struct PerDeviceOnce {
  bool done[64] = {};
  // true exactly once per device index (races between host threads only repeat the idempotent attribute call)
  bool first(int dev) { if (dev < 0 || dev >= 64) return true; if (done[dev]) return false; done[dev] = true; return true; }
};

__host__ __device__ constexpr int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ constexpr int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

__device__ __forceinline__ float silu_f(float v) { return v / (1.0f + __expf(-v)); }

// 16-bit GEMM operand format.  Default IEEE fp16: same tcgen05 kind::f16 rate as bf16 but an 11-bit
// significand (TF32's precision) -- GEMM operands here are GroupNorm-ed activations and weights, far
// inside fp16's range; conversions saturate.  Build with -DFDBM_OPERAND_BF16 for bfloat16.
#ifdef FDBM_OPERAND_BF16
typedef __nv_bfloat16 op_t;
typedef __nv_bfloat162 op2_t;
constexpr int kOperandIsBf16 = 1;
__device__ __forceinline__ op_t f2op(float v) { return __float2bfloat16(v); }
__device__ __forceinline__ float op2f(op_t v) { return __bfloat162float(v); }
__device__ __forceinline__ op2_t f2op2(float a, float b) { return __floats2bfloat162_rn(a, b); }
__device__ __forceinline__ float2 op22f2(op2_t v) { return __bfloat1622float2(v); }
__device__ __forceinline__ op2_t op2_tanh(op2_t v) {
  uint32_t r; asm("tanh.approx.bf16x2 %0, %1;" : "=r"(r) : "r"(*reinterpret_cast<uint32_t*>(&v)));
  return *reinterpret_cast<op2_t*>(&r);
}
#else
typedef __half op_t;
typedef __half2 op2_t;
constexpr int kOperandIsBf16 = 0;
__device__ __forceinline__ float sat16(float v) { return fminf(fmaxf(v, -65504.0f), 65504.0f); }
__device__ __forceinline__ op_t f2op(float v) { return __float2half_rn(sat16(v)); }
__device__ __forceinline__ float op2f(op_t v) { return __half2float(v); }
__device__ __forceinline__ op2_t f2op2(float a, float b) {     // one F2FP.SATFINITE: round to nearest, clamp to +-65504
  uint32_t r; asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(b), "f"(a));
  return *reinterpret_cast<op2_t*>(&r);
}
__device__ __forceinline__ float2 op22f2(op2_t v) { return __half22float2(v); }
__device__ __forceinline__ op2_t op2_tanh(op2_t v) {          // MUFU.TANH on both halves, max abs error ~2^-11
  uint32_t r; asm("tanh.approx.f16x2 %0, %1;" : "=r"(r) : "r"(*reinterpret_cast<uint32_t*>(&v)));
  return *reinterpret_cast<op2_t*>(&r);
}
#endif
__device__ __forceinline__ uint32_t pack_op2(float a, float b) {
  op2_t v = f2op2(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}

// --------------------------------------------------------------------------------------------
// Internal launchers (device pointers, no argument validation beyond what kernels need).
// The C ABI in api.cu validates and forwards; the backbone plan calls these directly.
// --------------------------------------------------------------------------------------------
int launch_fir_resample(const float* in, int B, int T, int F, int C, int mode, float* out, cudaStream_t s);
int launch_fir_resample_scaled(const float* in, int B, int T, int F, int C, int mode, float scale, float* out, cudaStream_t s);
int launch_channel_stats(const float* in, int B, int T, int F, int C, double* sums, cudaStream_t s);
int launch_groupnorm_act(const void* src1, int src1_h16 /* both sources 16-bit */, const double* sums1, int C1, const void* src2,
                         const double* sums2, int C2, const float* gamma, const float* beta, int B, int T, int F,
                         int silu, int mode, op_t* act_out, op_t* raw_out, cudaStream_t s);
int launch_pack_input(const float* x, const float* y, int B, int T, int F_in, int F, int Cin, float* out,
                      cudaStream_t s);
int launch_im2col_input(const float* in, int Cin, int B, int T, int F, op_t* out, cudaStream_t s);
int launch_combine(float* h, const float* pyr, int Cp, const float* w, const float* bias, int B, int T, int F,
                   int C, cudaStream_t s);
int launch_output_layer(const float* pyr, int Cp, const float* w, const float* bias, int B, int T, int F,
                        int F_out, float* out, cudaStream_t s);
int launch_temb(const float* t, const float* fourier_w, int nf, const float* w1, const float* b1, const float* w2,
                const float* b2, int B, int t_stride, float* temb_act, cudaStream_t s);
int launch_dense_all(const float* temb_act, const float* w, const float* bias, int B, int K, int rows, float* out,
                     cudaStream_t s);
int launch_gn_resample16(const op_t* src1, int C1, const op_t* src2, int C2, const float2* tab, int B, int T, int F,
                         int mode, op_t* act_out, op_t* raw_out, cudaStream_t s);
int launch_gn_finalize(const double* sums1, int C1, const double* sums2, int C2, const float* gamma, const float* beta,
                       int B, int64_t pixels, float2* table, cudaStream_t s, int blk_real = 0, float2* stats = nullptr);   // stats: also [B,G] (mean, rstd)
int launch_attention(const op_t* q, const op_t* k, const op_t* v, int ld, int B, int L,
                     int C, op_t* o, int ldo, cudaStream_t s, int fp32_probs = 0);   // fp32_probs: CUDA-core kernel with fp32 soft-max weights (training plans: matches attention_bwd)

// One K segment of the implicit GEMM: an activation tensor [B,T,F,C] (16-bit) read with 9 taps (3x3) or 1.
// norm_tab != nullptr: GroupNorm (+SiLU if act) is applied on load, norm_tab[b * tab_stride + c] = (scale, shift).
struct ConvSeg {
  const op_t* in = nullptr; int C = 0; int taps = 9;
  const float2* norm_tab = nullptr; int tab_stride = 0; int act = 0;
};
struct ConvArgs {
  ConvSeg seg[3]; int n_seg = 0;
  const op_t* wpack = nullptr;
  const float* bias = nullptr; const float* bias_b = nullptr; int bias_b_stride = 0; const float* residual = nullptr;
  const op_t* residual_h16 = nullptr;      // identity shortcut read from the 16-bit copy of the stream (instead of `residual`)
  float scale = 1.0f; int B = 0, T = 0, F = 0, Cout = 0;
  float* out_f32 = nullptr; op_t* out_h16 = nullptr;
  double* sums = nullptr;
  bool sums_prezeroed = false;             // the caller zeroes `sums` itself (plans: one memset per forward)
  // pyramid epilogue (ncsnpp_v2.py:338-359): out = conv(...)[:, :pyr_C] + bias + FIR-up x2(pyr_prev); fp32 [B,T,F,pyr_C]
  float* pyr_out = nullptr; const float* pyr_prev = nullptr; int pyr_C = 0;
  bool narrow_n = false;                   // pyramid convolutions: MMA N = 16 (Cout = 16 zero-padded weight rows) instead of 128
  // Combine epilogue (layerspp.py:52-59): out += comb_b[n] + sum_k comb_w[n][k] * comb_pyr[b,t,f,k], applied after
  // `scale`; comb_pyr is the fp32 input pyramid [B,T,F,comb_C] at the output resolution
  const float* comb_pyr = nullptr; const float* comb_w = nullptr; const float* comb_b = nullptr; int comb_C = 0;
};
int launch_conv_igemm(const ConvArgs& a, cudaStream_t s);
int launch_pack_conv_weights_dgrad(const float* w, int Cout, int Cin, int ksize, op_t* wpack, cudaStream_t s, int Cin_total = 0,
                                   int ci_off = 0);
int64_t conv_wgrad_workspace_bytes(int Cout, int Cin, int ksize, int B, int T, int F);
int launch_conv_wgrad(const op_t* dy, int Cout, const op_t* x, int Cin, int ksize, int B, int T, int F, float scale,
                      int io_layout, float* dw, float* workspace, cudaStream_t s);
// ---- training-step passes (train_kernels.cu)
int launch_grad_prepare(const float* g, int B, int64_t P, int C, float scale, op_t* g16, float* acc_dst, double* sums, cudaStream_t s,
                        bool acc_first = false, bool sums_prezeroed = false);   // acc_first: acc_dst = value instead of +=
int launch_gn_bwd_reduce(const op_t* g_a, int g_ld, int g_coff, const void* x, int x16, int C, int C_tot, int c_off,
                         const float2* tab, const float2* stats, int act, int B, int64_t P, double* S, cudaStream_t s);
int launch_gn_bwd_apply(const op_t* g_a, int g_ld, int g_coff, const void* x, int x16, int C, int C_tot, int c_off,
                        const float2* tab, const float2* stats, const float* gamma, int act, int B, int64_t P, const double* S,
                        float* acc_dst, op_t* out16, double* out_sums, cudaStream_t s, bool acc_first = false,
                        bool sums_prezeroed = false);
int launch_gn_param_grad(const double* S, int B, int C, float inv_scale, float* dgamma, float* dbeta, cudaStream_t s);
int launch_gn_stats(const double* sums1, int C1, const double* sums2, int C2, int B, int64_t pixels, float2* stats, cudaStream_t s);
int launch_fir_resample16(const op_t* in, int in_ld, int in_coff, int B, int T, int F, int C, int mode, float scale,
                          op_t* out16, float* acc_dst, cudaStream_t s);
int launch_col_sums16(const op_t* in, int ld, int c_off, int B, int64_t P, int C, double* sums, cudaStream_t s, bool sums_prezeroed = false);
int launch_col_sums_to(const double* sums, int B, int C, float inv_scale, float* dst, float* per_b, int per_b_ld, cudaStream_t s);
int launch_attention_bwd(const op_t* qkv, int B, int L, int C, const op_t* d_o, float* scratch, op_t* g_qkv, cudaStream_t s);
int launch_adam_ema(float* p, const float* g, float* m, float* v, float* ema, const unsigned char* trainable, int64_t n,
                    double* sumsq_scratch, float grad_div, float clip, float lr, float beta1, float beta2, float eps, int step,
                    float ema_decay, int ema_warmup, double* state, cudaStream_t s);
struct WgradCall {
  const op_t* dy = nullptr; int dy_ld = 0, dy_coff = 0, Cout = 0;
  const op_t* x = nullptr; int x_ld = 0, x_coff = 0, Cin = 0;
  int ksize = 3, B = 0, T = 0, F = 0;
  float scale = 1.0f;
  int layout = 0, Cin_total = 0, ci_off = 0, aux = 0;
  float* dw = nullptr; float* workspace = nullptr;
};
int launch_conv_wgrad_ex(const WgradCall& c, cudaStream_t s);
int launch_output_layer_bwd(const float* g_out, const float* pyr, int Cp, const float* w, int B, int T, int F, int F_out, float inv,
                            float* g_pyr, float* dw, float* db, cudaStream_t s);
int launch_small_col_sums(const float* g, int64_t n_px, int Cp, float inv, float* db, cudaStream_t s);
int launch_combine_bwd(const float* g, const float* pyr, int Cp, int64_t n_px, int C, float inv, float* dw, float* db, cudaStream_t s);
int launch_pack_pyr_dgrad(const float* w, int C, int Cp, op_t* out, cudaStream_t s);
int launch_dense_temb_bwd(const float* d, const float* act, const float* w, int B, int K, int rows, float* dw, float* db, float* g_act,
                          const float* t, const float* fw, int nf, const float* w1, const float* b1, const float* w2, const float* b2,
                          int t_stride, float* dw1, float* db1, float* dw2, float* db2, cudaStream_t s);
int make_act_tile_map(CUtensorMap* map, const op_t* ptr, int B, int T, int F, int C, int box_f, int box_t);
int64_t conv_wpack_bytes(int C1, int ksize, int C2, int Cout);
// ksize 3 / 1: OIHW; -1: NIN matrix [in][out]; -2: first conv, OIHW [Cout][C1<=4][3][3] as one im2col K-block of 64
int launch_pack_conv_weights(const float* w1, int C1, int ksize, const float* w2, int C2, int Cout, int n_rows_total,
                             int row_offset, op_t* wpack, cudaStream_t s);
// All weight packs of a plan in ONE launch (a training step re-packs ~300 weight tensors after Adam; one launch each was 1.9 ms
// of launch latency): a descriptor per pack, blocks of kPackChunk consecutive output elements, the block looks its descriptor up.
struct PackDesc {
  const float* w1; const float* w2; op_t* out;
  int kind;                                  // 0: forward pack (launch_pack_conv_weights), 1: dgrad pack (launch_pack_conv_weights_dgrad)
  int C1, ksize, io, C2, Cout, rows_total, row_offset;      // kind 1: C1 = Cin, C2 = Cin_total, row_offset = ci_off
  long long total;                           // elements this pack writes
  long long first_block;                     // filled by the plan: first block of the batched launch that belongs to this pack
};
// Deferred per-channel gradient sums of a training backward: every site leaves its per-(utterance, channel) double sums in its own
// slice of one pool (zeroed by ONE memset at the start of the backward) and the ~390 tiny reductions into the parameter-gradient
// buffer (conv / NIN biases, FiLM rows, GroupNorm gamma / beta) run as ONE launch at the end instead of one 4-7 us launch each
// between the big kernels.  kind 0: src [B,C] -> dst0[c] += inv * sum_b, per_b[b*ld + c] = inv * src[b,c] (optional);
// kind 1: src [B,C,2] (GroupNorm backward S) -> dst0 = dgamma[c] += inv * sum_b S[b,c,1], dst1 = dbeta[c] += inv * sum_b S[b,c,0]
struct DeferDesc {
  const double* src; int B, C, kind;
  float* dst0; float* dst1; float* per_b; int per_b_ld;
};
int launch_deferred_sums(const DeferDesc* descs_dev, int n_descs, float inv_scale, cudaStream_t s);
constexpr int kPackChunk = 2048;
PackDesc pack_desc_fwd(const float* w1, int C1, int ksize, const float* w2, int C2, int Cout, int n_rows_total, int row_offset, op_t* wpack);
PackDesc pack_desc_dgrad(const float* w, int Cout, int Cin, int ksize, op_t* wpack, int Cin_total, int ci_off);
int launch_pack_batch(const PackDesc* descs_dev, int n_descs, long long n_blocks, cudaStream_t s);

}  // namespace fdbm
