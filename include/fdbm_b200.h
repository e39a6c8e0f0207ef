/* fdbm_b200 -- C ABI of the B200-native enhancement hot path.
 *
 * Drop-in boundary for the reference's Python seams (SURVEY.md section 8(b)).  The reference
 * (Dahan-Wang/Rethinking-Flow-and-Diffusion-Bridge-Models-for-Speech-Enhancement) has no C ABI
 * of its own for this path -- it is PyTorch calls -- so every entry point below names the
 * reference function (file:line, relative to the reference root) whose arithmetic it replaces.
 *
 * Conventions
 *   - every function returns 0 on success, a negative FDBM_E* code on failure; the message is
 *     available from fdbm_last_error() (thread-local).  Nothing aborts.
 *   - all data pointers are DEVICE pointers owned by the caller; calls are stream-ordered on
 *     `stream` (a cudaStream_t passed as void*), never synchronise, never allocate -- except
 *     fdbm_plan_create / fdbm_plan_destroy, which own the packed weights and the workspace.
 *   - spectrograms use the reference layout: complex64 [B, 1, F=257, T] with T contiguous,
 *     passed as float* (interleaved re, im).  Waveforms are fp32 [B, n_samples].
 *   - sm_100a only.  There is no fallback: on any other device fdbm_* returns FDBM_EARCH.
 */
#ifndef FDBM_B200_H
#define FDBM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDBM_OK        0
#define FDBM_EINVAL   -1   /* bad argument (shape, alignment, enum)            */
#define FDBM_ECUDA    -2   /* CUDA runtime / driver error                      */
#define FDBM_EARCH    -3   /* device is not sm_100                             */
#define FDBM_ESTATE   -4   /* handle used in the wrong state                   */

/* pad_spec modes, fdbm/util/other.py:76-90 */
#define FDBM_PAD_ZERO        0
#define FDBM_PAD_REFLECTION  1
#define FDBM_PAD_REPLICATION 2
/* transform_type, fdbm/data_module.py:173-199 */
#define FDBM_TRANSFORM_EXPONENT 0
#define FDBM_TRANSFORM_LOG      1
#define FDBM_TRANSFORM_NONE     2
/* sampler update kind, fdbm/bridge.py:83 (ODE) and :109 (SDE) */
#define FDBM_STEP_ODE 0
#define FDBM_STEP_SDE 1

const char* fdbm_last_error(void);
int fdbm_version(void);
/* 0 when the current device is sm_100 (B200); FDBM_EARCH otherwise. */
int fdbm_check_device(void);
/* 16-bit GEMM operand format of this build: 0 = IEEE fp16 (default), 1 = bfloat16.  Both feed the
 * same tcgen05 kind::f16 tensor-core path at the same rate; "h16" below means this format. */
int fdbm_operand_is_bf16(void);

/* ---------------------------------------------------------------------------------------------
 * Spectral front end.  Replaces SpecsDataModule.stft (fdbm/data_module.py:223-225) +
 * spec_fwd (:173-186) + pad_spec (fdbm/util/other.py:76-90) in one kernel:
 * reflect-pad n_fft/2, frame (n_fft, hop), window, rFFT, amplitude compression
 * |z|^e * exp(j angle z) * factor, right-pad the frame axis to `n_frames_out`.
 *   wave    fp32  [B, n_samples]           (row stride = wave_stride elements)
 *   window  fp32  [n_fft]                  (the reference's window tensor, data_module.py:13-19)
 *   spec    cplx  [B, 1, n_fft/2+1, n_frames_out]
 * n_fft must be 512; hop must divide n_fft (256 or 128); n_frames_out >= 1 + n_samples/hop.
 * --------------------------------------------------------------------------------------------- */
int fdbm_stft_compress(const float* wave, int batch, int64_t n_samples, int64_t wave_stride,
                       const float* window, int n_fft, int hop,
                       int transform_type, float spec_factor, float abs_exponent,
                       int pad_mode, int n_frames_out, float* spec, void* stream);

/* Variable-length batch (the callers' side of infer_folder.py:91-121: every file has its own length): `lengths`
 * is a DEVICE int32 [B] of per-utterance sample counts, min/max_samples their host-side bounds; utterance b is framed,
 * reflect-padded and frame-padded (pad_spec) from ITS OWN length, so each row equals the single-utterance call. */
int fdbm_stft_compress_var(const float* wave, int batch, const int* lengths, int64_t min_samples, int64_t max_samples,
                           int64_t wave_stride, const float* window, int n_fft, int hop,
                           int transform_type, float spec_factor, float abs_exponent,
                           int pad_mode, int n_frames_out, float* spec, void* stream);

/* Spectral back end.  Replaces BridgeModel.to_audio (fdbm/model.py:376-377) = spec_back
 * (fdbm/data_module.py:188-199) + torch.istft (:227-229): de-compress, irFFT, window,
 * overlap-add, divide by the window-square envelope, drop n_fft/2 samples, cut to `length`.
 *   spec  cplx [B, 1, n_fft/2+1, n_frames];   wave fp32 [B, length] (row stride wave_stride) */
int fdbm_decompress_istft(const float* spec, int batch, int n_frames,
                          const float* window, int n_fft, int hop,
                          int transform_type, float spec_factor, float abs_exponent,
                          int64_t length, int64_t wave_stride, float* wave, void* stream);

/* Variable-length batch: utterance b is cut to lengths[b] (device int32 [B]); samples beyond it are not written. */
int fdbm_decompress_istft_var(const float* spec, int batch, int n_frames,
                              const float* window, int n_fft, int hop,
                              int transform_type, float spec_factor, float abs_exponent,
                              const int* lengths, int64_t max_length, int64_t wave_stride, float* wave, void* stream);

/* The same two kernels with the elementwise glue of `enhance` folded in (fdbm/model.py:391-406, infer_single.py:80-99,
 * infer_folder.py:100-121), so that no PyTorch elementwise pass is left on the path:
 *   fdbm_wave_absmax          out[b] = max_n |wave[b, n]|  (norm_factor = y.abs().max(), infer_single.py:83-84)
 *   fdbm_stft_compress_ex     spec = pad_spec(spec_fwd(stft(wave / norm[b])));  norm NULL = no normalisation; lengths NULL =
 *                             all rows max_samples long.  The division is applied to the spectrum (the STFT is linear):
 *                             results agree with dividing the waveform first to rounding (~1e-7 relative).
 *   fdbm_decompress_istft_ex  wave = istft(spec_back(spec)) * norm[b]  (x_hat * norm_factor, infer_single.py:94) and, when
 *                             `peak` is given, peak[b] = max |wave[b]| for the clip rule; norm / peak / lengths may be NULL.
 *   fdbm_clip_rescale         if peak[b] > 1: wave[b] = wave[b] / peak[b] * rescale   (infer_single.py:95-97 with 0.5,
 *                             infer_folder.py:119-120 with 0.95)
 * norm / peak: fp32 [B] device. */
int fdbm_wave_absmax(const float* wave, int batch, int64_t n_samples, const int* lengths, int64_t wave_stride, float* out,
                     void* stream);
int fdbm_stft_compress_ex(const float* wave, int batch, const int* lengths, int64_t min_samples, int64_t max_samples,
                          int64_t wave_stride, const float* window, const float* norm, int n_fft, int hop, int transform_type,
                          float spec_factor, float abs_exponent, int pad_mode, int n_frames_out, float* spec, void* stream);
int fdbm_decompress_istft_ex(const float* spec, int batch, int n_frames, const float* window, int n_fft, int hop,
                             int transform_type, float spec_factor, float abs_exponent, const int* lengths, int64_t max_length,
                             int64_t wave_stride, const float* norm, float* peak, float* wave, void* stream);
int fdbm_clip_rescale(float* wave, int batch, int64_t n_samples, const int* lengths, int64_t wave_stride, const float* peak,
                      float rescale, void* stream);

/* Unfused pieces of the same front/back end, for callers that keep the reference's call sequence:
 * spec_fwd / spec_back (fdbm/data_module.py:173-199; inverse = 0 / 1) over n_complex elements, and
 * pad_spec (fdbm/util/other.py:76-90) over `rows` = B*1*F rows of n_frames -> n_frames_out frames. */
int fdbm_spec_transform(const float* in, float* out, int64_t n_complex, int transform_type, float spec_factor,
                        float abs_exponent, int inverse, void* stream);
int fdbm_pad_spec(const float* in, int64_t rows, int n_frames, int pad_mode, int n_frames_out, float* out,
                  void* stream);

/* ---------------------------------------------------------------------------------------------
 * Bridge sampler arithmetic.
 * fdbm_prior_sample: Bridge.prior_sampling (fdbm/bridge.py:45-49)  x0 = b*y + sigma*z.
 *   z == NULL and sigma != 0 draws z in-kernel (Philox4x32-10 keyed by seed, offset, element);
 *   n_complex = number of complex elements.
 * fdbm_bridge_step: loop body of ode_sampler_ei / sde_sampler_ei (fdbm/bridge.py:83, :109)
 *   ODE: x <- (wx*x + ws*d) + wy*y          SDE: x <- (wx*x + ws*d) + wz*z
 *   `coef` is a DEVICE pointer to the 3 fp32 weights of this step (row of the [N,3] table
 *   built on the host with the reference's own op sequence, bridge.py:308-337,373-385), so a
 *   captured CUDA graph can replay the step.  Evaluated without FMA contraction: bit-identical
 *   to the reference's three multiplies and two adds.  In-place on x.
 * --------------------------------------------------------------------------------------------- */
int fdbm_prior_sample(const float* y, const float* z, float b, float sigma, uint64_t seed, uint64_t offset,
                      int64_t n_complex, float* x, void* stream);
/* Predictor-corrector sampler arithmetic (Bridge.pc_sampler fdbm/bridge.py:142-166; EulerMaruyamaPredictor
 * util/predictors.py:39-51; LangevinCorrector / AnnealedLangevinDynamics util/correctors.py:36-81).  Every update of that
 * sampler has the form   x_mean = c0*x + c1*d + c2*y ;  x = x_mean + c3*z   with per-step scalars:
 *   coef        DEVICE fp32[4] = (c0, c1, c2, c3)
 *   z           noise cplx like x, or NULL = in-kernel Philox keyed by (seed, offset, element)
 *   x_mean_out  optional: the noise-free state (`denoise=True` returns it after the last step)
 * fdbm_langevin_coef computes coef for the Langevin corrector, whose step size depends on the data
 * (correctors.py:47-50): step = 2 (snr * mean_b |z_b| / (mean_b |grad_b| + 1e-8))^2, grad = -(x - a d - b y) / (sigma^2 + 1e-8),
 * a, b, sigma = path_param(t); the norms are per utterance (batch x n_per_utt complex elements), z as above with the SAME
 * (seed, offset) the following fdbm_bridge_update4 call uses; scratch = 2*batch doubles. */
int fdbm_bridge_update4(float* x, const float* d, const float* y, const float* z, const float* coef, uint64_t seed,
                        uint64_t offset, int64_t n_complex, float* x_mean_out, void* stream);
int fdbm_langevin_coef(const float* x, const float* d, const float* y, const float* z, float a, float b, float sigma,
                       float snr, uint64_t seed, uint64_t offset, int batch, int64_t n_per_utt, double* scratch,
                       float* coef_out, void* stream);
/* Adaptive ODE sampler (Bridge.ode_sampler_int fdbm/bridge.py:115-140 -> scipy.integrate.solve_ivp RK45, whose stage
 * arithmetic the reference runs on the host over the flattened state): out = sum_k coefs[k] * srcs[k] over n_floats
 * fp32 elements (srcs: HOST array of n_terms <= 8 device pointers, coefs: HOST), and the controller's error measure
 * *out_sumsq = sum_i |sum_k coefs[k] srcs[k][i]|^2 / (atol + rtol max(|y_i|, |y_new_i|))^2 over n_complex complex
 * elements (device double; scipy's error_norm = sqrt(out_sumsq / n_complex)). */
int fdbm_lincomb(float* out, const float* const* srcs, const float* coefs, int n_terms, int64_t n_floats, void* stream);
int fdbm_rk_error_norm(const float* const* srcs, const float* coefs, int n_terms, const float* y, const float* y_new,
                       float rtol, float atol, int64_t n_complex, double* out_sumsq, void* stream);
int fdbm_bridge_step(float* x, const float* d, const float* y_or_z, const float* coef, int kind,
                     uint64_t seed, uint64_t offset, int64_t n_complex, void* stream);

/* ---------------------------------------------------------------------------------------------
 * NCSN++ backbone.  Replaces NCSNpp_v2.forward (fdbm/backbones/ncsnpp_v2.py:241-401) and
 * NCSNpp_v2_predictive.forward (ncsnpp_v2_predictive.py:222-362) with all their building blocks
 * (ncsnpp_utils/layerspp.py:32-91,212-274; layers.py:100-124,546-555; up_or_down_sampling.py
 * :195-257 and the reference's only native op, op/upfirdn2d_kernel.cu:107-207).
 *
 * A plan is built for one (architecture, batch, n_frames) shape.  Weights are passed as an array
 * of host-visible descriptors {name, device pointer, numel} using the reference's state_dict
 * names (all_modules.<i>.<Layer>.weight ..., output_layer.*); the plan packs them (h16, tap-major)
 * into its own buffer.  Re-pack with fdbm_plan_load_weights after parameters change (EMA swap,
 * fdbm/model.py:146-160; optimizer step).
 * --------------------------------------------------------------------------------------------- */
typedef struct fdbm_plan fdbm_plan;

typedef struct fdbm_tensor_ref {
  const char* name;     /* state_dict key                                   */
  const float* data;    /* device pointer, fp32, contiguous                 */
  int64_t numel;
} fdbm_tensor_ref;

typedef struct fdbm_arch {
  int nf;                 /* 128                                             */
  int n_levels;           /* len(ch_mult) = 7                                */
  int ch_mult[8];         /* 1,1,2,2,2,2,2                                   */
  int num_res_blocks;     /* 2                                               */
  int attn_resolution;    /* 16 (0 = none)                                   */
  int predictive;         /* 0: forward(x,y,t), 4 input ch;  1: forward(y)   */
  int image_size;         /* 256 (frequency bins seen by the backbone)       */
  int channel_block_real; /* 0: every channel is real.  96: the nf = 96 size variants (ncsnpp_v2.py:404-415, 436-448) run as
                           * nf = 128 with every 128-channel block = 96 real channels followed by 32 zero channels; the host
                           * zero-pads the weights (fdbm_b200/backbones.py), the only arithmetic that depends on it is the
                           * GroupNorm group structure (groups and counts follow the REAL channel index).  Inference plans only. */
} fdbm_arch;

int fdbm_plan_create(const fdbm_arch* arch, int batch, int n_frames, fdbm_plan** out);
int fdbm_plan_destroy(fdbm_plan* plan);
int fdbm_plan_load_weights(fdbm_plan* plan, const fdbm_tensor_ref* tensors, int n_tensors, void* stream);
/* bytes of device memory the plan holds (weights + activations workspace) */
int64_t fdbm_plan_device_bytes(const fdbm_plan* plan);
/* number of kernel launches one forward issues (for bench.py's gpu_launches) */
int fdbm_plan_num_launches(const fdbm_plan* plan);

/* One backbone forward: out = D(x, y, t).  x, y, out: cplx [B,1,257,T]; t: fp32 [B] device.
 * Predictive plans ignore y and t (pass NULL). */
int fdbm_ncsnpp_forward(fdbm_plan* plan, const float* x, const float* y, const float* t, float* out,
                        void* stream);

/* Whole sampler: Bridge.ode_sampler_ei / sde_sampler_ei (fdbm/bridge.py:66-113) for n_steps steps.
 *   y     cplx [B,1,257,T]   conditioning (noisy compressed spectrogram)
 *   x     cplx [B,1,257,T]   in: x_start (prior sample), out: final sample
 *   times fp32 [n_steps]     HOST; t_prev of every step (time_steps[:-1]) -- what the backbone sees
 *   coef  fp32 [n_steps,3]   HOST; coefficient table
 *   noise cplx [n_steps, B,1,257,T] device, or NULL (SDE only; NULL = in-kernel Philox with `seed`)
 * y and x are staged into buffers fdbm_plan_create allocated, and times / coef / seed travel through a plan-owned ring of
 * pinned host slots, so the call never allocates and the N-step loop is captured ONCE per (plan, n_steps, kind, noise
 * address) as a CUDA graph and replayed for every later call.  n_steps <= 1024.  `stream` must not be capturing
 * (FDBM_ESTATE): the sampler owns its graph.  A plan serves one host thread at a time and only on the device it was
 * created on (FDBM_ESTATE if another device is current). */
int fdbm_sampler_run(fdbm_plan* plan, const float* y, float* x, const float* times, const float* coef,
                     int n_steps, int kind, const float* noise, uint64_t seed, void* stream);

/* ---- training step (SURVEY section 8 A10: model.py:258-275 `_step`, configure_optimizers :101, EMA :129-132) ----
 * A TRAINING plan keeps every forward tensor (nothing in its arena is reused) and records the backward launch list:
 * per residual block  grad_prepare -> [1x1 dgrad/wgrad of the shortcut] -> GroupNorm_1 recompute -> Conv_1 wgrad, dgrad
 * -> GroupNorm_1 backward -> Conv_0 wgrad, dgrad -> [FIR adjoint] -> GroupNorm_0 backward, plus attention, progressive
 * input/output, Combine and time-embedding backward.  fdbm_ncsnpp_forward on such a plan is the training forward.
 *   fdbm_ncsnpp_backward: g_out = loss_scale * dL/dD, cplx [B,1,257,T] (activation gradients are h16 operands, hence the
 *   scale); parameter gradients land UN-scaled in the flat fp32 buffer (accumulate != 0 adds to it).
 *   fdbm_plan_buffers: the flat fp32 parameter / gradient / EMA buffers (same layout; fdbm_plan_param_info gives the
 *   element offset of a tensor by its reference name) -- the caller all-reduces `grads` across ranks (DDP).
 *   fdbm_plan_optimizer_step: Adam + clip_grad_norm_ + EMA on the flat buffers, then re-packs the 16-bit weights. */
int fdbm_plan_create_train(const fdbm_arch* arch, int batch, int n_frames, fdbm_plan** out);
int fdbm_ncsnpp_backward(fdbm_plan* plan, const float* g_out, float loss_scale, int accumulate, void* stream);
int fdbm_plan_param_info(const fdbm_plan* plan, const char* name, int64_t* offset, int64_t* numel);
int fdbm_plan_buffers(fdbm_plan* plan, float** params, float** grads, float** ema, int64_t* numel);
/* rebuild the packed 16-bit weights after the caller wrote the flat parameter buffer (DDP broadcast, checkpoint restore) */
int fdbm_plan_repack_weights(fdbm_plan* plan, void* stream);
int fdbm_plan_num_backward_launches(const fdbm_plan* plan);
/* measurement aid: backward of the last forward with a CUDA event pair around every recorded op; returns the op count */
int fdbm_plan_profile_backward(fdbm_plan* plan, const float* g_out, float loss_scale, float* ms, int* kinds, int max_ops,
                               void* stream);
/* `step` and `ema_warmup` as in fdbm_adam_ema_step (step 0 = device-side count of applied steps, the normal mode). */
int fdbm_plan_optimizer_step(fdbm_plan* plan, float grad_div, float clip_norm, float lr, float beta1, float beta2,
                             float eps, int step, float ema_decay, int ema_warmup, void* stream);
/* Adam moments <- 0, EMA <- current parameters (what torch_ema does at construction), counters <- 0. */
int fdbm_plan_reset_optimizer(fdbm_plan* plan, void* stream);
/* {applied updates, skipped steps, last gradient norm, reserved} copied to the HOST array `out`.  This call
 * synchronises `stream` (it is how the host learns about skipped steps to back the loss scale off). */
int fdbm_plan_optimizer_state(fdbm_plan* plan, double* out, void* stream);
/* Overwrite the device-side counters (checkpoint restore: torch_ema's num_updates, Adam's step). */
int fdbm_plan_set_optimizer_state(fdbm_plan* plan, double applied, double skipped, void* stream);
/* EMA evaluation swap (model.py:146-160 store / copy_to / restore): to_ema != 0 saves the current parameters in a
 * plan-owned backup and loads the EMA into the live parameters; to_ema == 0 restores the backup.  Packed weights are
 * rebuilt either way.  FDBM_ESTATE if restore is called without a preceding swap. */
int fdbm_plan_swap_ema(fdbm_plan* plan, int to_ema, void* stream);

/* Loss head of the training step: BridgeModel._loss, "data_prediction_hybrid" (fdbm/model.py:187-218, pesq_weight 0):
 *   L = 70 mean((|X|^0.3 - |X^|^0.3)^2) + 30 sum |X/|X|^0.7 - X^/|X^|^0.7|^2 / N - mean_b log10 SI-SNR(istft X, istft X^)
 * with X = spec_back(x), X^ = spec_back(x_hat).  Forward and gradient in one call (no autograd):
 *   x_hat, x  cplx [B,1,n_fft/2+1,T];  *loss fp32 (device);  g_out = loss_scale * dL/dx_hat, cplx like x_hat
 * n_fft == 2*hop (sqrt-Hann, overlap-add envelope 1), exponent transform.  workspace: fdbm_hybrid_loss_workspace_bytes. */
int64_t fdbm_hybrid_loss_workspace_bytes(int batch, int n_frames, int n_fft, int hop);
int fdbm_hybrid_loss(const float* x_hat, const float* x, int batch, int n_frames, const float* window, int n_fft, int hop,
                     int transform_type, float spec_factor, float abs_exponent, float loss_scale, void* workspace,
                     float* loss, float* g_out, void* stream);
/* "data_prediction" (fdbm/model.py:163-185, the reference's argparse default, pesq_weight 0):
 *   L = mean_b 0.5 sum_{f,t} |x_hat - x|^2 / (F T)  +  l1_weight * mean_b 0.5 sum_n |istft X^ - istft X| / target_len,
 * target_len = (T - 1) * hop; the first term on the COMPRESSED spectrograms, the second on the waveforms of the de-compressed
 * ones.  Same conventions, constraints and workspace as fdbm_hybrid_loss. */
int fdbm_data_prediction_loss(const float* x_hat, const float* x, int batch, int n_frames, const float* window, int n_fft, int hop,
                              int transform_type, float spec_factor, float abs_exponent, float l1_weight, float loss_scale,
                              void* workspace, float* loss, float* g_out, void* stream);
/* "data_prediction_mel" (fdbm/model.py:220-233) and, with_phase != 0, "data_prediction_melphase" (:235-251):
 *   L = 0.5 mean |x_hat - x|^2 + 0.1 MelSpectrogramLoss(istft X^, istft X) (+ 0.01 PhaseLoss(x_hat, x))
 * MelSpectrogramLoss as BridgeModel builds it (model.py:77-92, fdbm/loss.py:213-289): seven resolutions n_fft = 32..2048 (Hann,
 * hop n_fft/4, centred, reflection), n_mels = 5,10,20,40,80,160,210, L1 of log10(clamp(mel, 1e-5)^2), mag_weight 0; PhaseLoss =
 * loss.py:9-33 (instantaneous phase, group delay, phase time difference, anti-wrapped L1).  Forward and gradient in one call.
 * `tables`: fdbm_mel_tables_bytes() bytes of device memory the caller owns, filled once by fdbm_mel_tables_init (windows,
 * twiddles, the librosa-convention Slaney filterbanks of `sample_rate`; the call synchronises `stream`).  Same conventions and
 * constraints as fdbm_hybrid_loss; additionally target_len = (T - 1) * hop > 1024.  workspace: fdbm_mel_loss_workspace_bytes
 * (256-byte aligned). */
int64_t fdbm_mel_tables_bytes(void);
int fdbm_mel_tables_init(void* tables, int sample_rate, void* stream);
int64_t fdbm_mel_loss_workspace_bytes(int batch, int n_frames, int n_fft, int hop);
int fdbm_mel_loss(const float* x_hat, const float* x, int batch, int n_frames, const float* window, int n_fft, int hop,
                  int transform_type, float spec_factor, float abs_exponent, int with_phase, float loss_scale,
                  const void* tables, void* workspace, float* loss, float* g_out, void* stream);

/* The skinny layers of NCSN++ (SURVEY 8 A7e / A7f), exported for kernel-level parity tests and other hosts.  Activations are
 * [B,T,F,C] (channels innermost), spectrograms cplx [B,1,f_in,T].
 *   fdbm_pack_input      ncsnpp_v2.py:247-250  x (, y) cplx -> fp32 [B,T,f_used,c_in] = (Re x, Im x (, Re y, Im y)), rows >= f_used dropped
 *   fdbm_im2col_input    ncsnpp_v2.py:278      [B,T,F,c_in] fp32 -> 16-bit [B,T,F,64], k = (kf*3 + kt)*c_in + ci: the 3x3 input convolution as
 *                                              one K-block of fdbm_conv_igemm (ksize 1 with weights packed by fdbm_pack_conv_weights ksize -2)
 *   fdbm_time_embedding  layerspp.py:32-41, ncsnpp_v2.py:252-270   t [B] -> SiLU(temb) [B,4 nf]
 *   fdbm_film_rows       layerspp.py:263       all Dense_0 layers at once: out [B,rows] = act [B,k] . weight[rows,k]^T + bias
 *   fdbm_combine         layerspp.py:52-59     h += conv1x1(c_pyr -> C)(pyramid) (progressive_combine 'sum'); weight [C,c_pyr]
 *   fdbm_output_layer    ncsnpp_v2.py:392-399  conv1x1(c_pyr -> 2) -> cplx [B,1,f_out,T], rows >= n_freq zero (the Nyquist row) */
int fdbm_pack_input(const float* x, const float* y, int batch, int n_frames, int f_in, int f_used, int c_in, float* out, void* stream);
int fdbm_im2col_input(const float* in, int c_in, int batch, int n_frames, int n_freq, void* out_h16, void* stream);
int fdbm_time_embedding(const float* t, const float* fourier_w, int nf, const float* w1, const float* b1, const float* w2,
                        const float* b2, int batch, float* out, void* stream);
int fdbm_film_rows(const float* temb_act, const float* weight, const float* bias, int batch, int k, int rows, float* out, void* stream);
int fdbm_combine(float* h, const float* pyramid, int c_pyr, const float* weight, const float* bias, int batch, int n_frames, int n_freq,
                 int channels, void* stream);
int fdbm_output_layer(const float* pyramid, int c_pyr, const float* weight, const float* bias, int batch, int n_frames, int n_freq,
                      int f_out, float* out, void* stream);

/* Measurement aid for bench.py: run one forward launch by launch with a CUDA event pair around every
 * kernel.  ms[i] = device time, kinds[i] = FDBM_OP_*, flops[i] = algorithmic FLOPs (2*MAC, convolutions
 * only) of launch i.  Returns the number of launches (<= max_ops) or a negative error.  Synchronises. */
#define FDBM_OP_CONV   0   /* tcgen05 implicit-GEMM convolution           */
#define FDBM_OP_NORM   1   /* GroupNorm (+SiLU, +FIR) operand pass        */
#define FDBM_OP_STATS  2   /* per-channel statistics                      */
#define FDBM_OP_SKINNY 3   /* K or N <= 4 layers, FIR, packing            */
#define FDBM_OP_ATTN   4   /* attention core                              */
#define FDBM_OP_SMALL  5   /* time embedding, Dense_0 table               */
#define FDBM_OP_WGRAD  6   /* tcgen05 weight-gradient kernel (training)   */
int fdbm_plan_profile_forward(fdbm_plan* plan, const float* x, const float* y, const float* t, float* out,
                              float* ms, int* kinds, double* flops, int max_ops, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Building blocks, exported for the parity tests (tests/ call them one by one through ctypes).
 * Layout of activations inside the backbone: [B, T, F, C] ("NTFC": channels innermost, then
 * frequency, then frames) -- fp32 for the residual stream, h16 for GEMM operands.
 * --------------------------------------------------------------------------------------------- */

/* upfirdn2d replacement (op/upfirdn2d.cpp:12-23 restricted to the two modes the model uses,
 * up_or_down_sampling.py:195-257): separable [1,3,3,1] FIR, mode 1 = down x2, mode 2 = up x2.
 * in fp32 [B,T,F,C] -> out fp32 [B,T',F',C]. */
int fdbm_fir_resample(const float* in, int batch, int T, int F, int C, int mode, float* out, void* stream);

/* per-(b,channel) sum / sum-of-squares of an fp32 NTFC tensor -> double [B, C, 2] (zeroed inside). */
int fdbm_channel_stats(const float* in, int batch, int T, int F, int C, double* sums, void* stream);

/* GroupNorm(min(C/4,32) groups, eps 1e-6) [+SiLU] [+FIR up/down] over the channel concatenation of
 * up to two fp32 NTFC sources -> h16 NTFC operand(s).  Replaces nn.GroupNorm + nn.SiLU +
 * upsample_2d/downsample_2d + torch.cat in ResnetBlockBigGANpp.forward (layerspp.py:242-257).
 *   act_out  h16 [B,T',F',C1+C2]  = FIR(SiLU(GN(cat(src1,src2))))       (silu: 0/1)
 *   raw_out  h16 [B,T',F',C1+C2]  = FIR(cat(src1,src2)) or NULL          (operand of Conv_2) */
int fdbm_groupnorm_act(const float* src1, const double* sums1, int C1,
                       const float* src2, const double* sums2, int C2,
                       const float* gamma, const float* beta, int batch, int T, int F,
                       int silu, int mode, void* act_out, void* raw_out, void* stream);

/* The same pass for the resampling blocks (mode 1 = down x2, 2 = up x2) from the 16-bit copies of the residual
 * stream: act_out = FIR(SiLU(GN(cat(src1,src2)))), raw_out = FIR(cat(src1,src2)), both h16 [B,T',F',C1+C2].
 * src1/src2 h16 NTFC, sums double [B,C,2] of the sources, `table` scratch of 2*B*(C1+C2) floats. */
int fdbm_gn_resample_h16(const void* src1, const double* sums1, int C1, const void* src2, const double* sums2, int C2,
                         const float* gamma, const float* beta, float* table, int batch, int T, int F, int mode,
                         void* act_out, void* raw_out, void* stream);

/* Implicit-GEMM convolution on tcgen05 tensor cores (TMA-fed, TMEM accumulators):
 *   out[b,t,f,:] = scale * ( sum_taps W_tap . in1[b,t+dt,f+df,:]  (+ W2 . in2[b,t,f,:])
 *                            + bias (+ bias_b[b,:]) (+ residual[b,t,f,:]) )
 * Replaces nn.Conv2d 3x3 / 1x1 and NIN (layers.py:100-124, 546-555) together with the bias,
 * time-embedding FiLM add (layerspp.py:263), shortcut add and 1/sqrt(2) rescale (:270-274).
 *   in1   h16 [B,T,F,C1], ksize 3 or 1;  in2 h16 [B,T,F,C2] (1x1) or NULL
 *   wpack h16 packed by fdbm_pack_conv_weights;  bias fp32 [Cout];  bias_b fp32 [B,Cout] or NULL
 *   residual fp32 [B,T,F,Cout] or NULL;  out_f32 fp32 and/or out_h16 h16 [B,T,F,Cout] (either may be NULL)
 *   sums double [B,Cout,2] or NULL: receives the per-channel sum / sum of squares of the fp32 result. */
int fdbm_conv_igemm(const void* in1, int C1, int ksize, const void* in2, int C2,
                    const void* wpack, const float* bias, const float* bias_b, const float* residual,
                    float scale, int batch, int T, int F, int Cout,
                    float* out_f32, void* out_h16, double* sums, void* stream);
/* The full convolution launch the backbone plans make, as a descriptor: up to three K segments, each optionally
 * normalised on load, and every epilogue the plans use.  fdbm_conv_igemm_ex copies the descriptor field for field into
 * the plans' own launch arguments and launches the same kernel, so a caller reaches exactly the code paths a plan does.
 *
 *   out[b,t,f,n] = scale * ( sum_segments sum_taps W . act(seg.in)[b,t+dt-1,f+df-1,:]
 *                            + bias[n] + bias_b[b * bias_b_stride + n] + residual[b,t,f,n] )  (+ Combine term)
 *
 * One K segment (fdbm_conv_seg):
 *   in          h16 [B,T,F,C] activation tensor
 *   C           channels, a multiple of 64 (one K-block = 64 channels)
 *   taps        9 (3x3, zero padding outside the image) or 1 (1x1)
 *   norm_tab    NULL = raw operand.  Otherwise fp32 pairs (scale, shift): channel c of utterance b is transformed on load
 *               to x * scale + shift, then SiLU when act != 0, with entry b * tab_stride + c.  Pixels outside the image
 *               stay zero: the padding is applied to the transformed tensor.  A 1-tap normalised segment is loaded with its
 *               halo and read at the centre.  fdbm_gn_table builds such a table; two segments may share one table at
 *               offsets (tab, tab + 2 * C1 floats) with tab_stride = C1 + C2.
 *   tab_stride  (scale, shift) pairs per utterance row of norm_tab
 *   act         0 or 1 (SiLU after the transform; ignored for raw segments)
 *
 * fdbm_conv_desc:
 *   struct_bytes    must be sizeof(fdbm_conv_desc); checked before anything else, so a caller with a stale layout gets
 *                   FDBM_EINVAL and a message instead of a misread pointer
 *   seg, n_seg      1..3 segments; unused entries are ignored
 *   wpack           h16 weights packed by fdbm_pack_conv_weights, K-blocks in segment order: w1 covers the leading
 *                   segments (their channels concatenated), w2 the concatenation of the trailing raw 1-tap segments
 *   bias            fp32 [Cout], never NULL
 *   bias_b          fp32 FiLM rows or NULL; row b starts at b * bias_b_stride (stride 0: every utterance uses row 0)
 *   residual        fp32 [B,T,F,Cout] or NULL
 *   residual_h16    h16 [B,T,F,Cout] or NULL; not together with residual, comb_pyr or pyr_out
 *   scale           applied to everything but the Combine term
 *   B, T, F, Cout   Cout a multiple of the MMA N: 128, or 64 when Cout == 64, or 16 with narrow_n
 *   out_f32         fp32 [B,T,F,Cout] or NULL;  out_h16 h16 [B,T,F,Cout] or NULL;  at least one output (or pyr_out)
 *   sums            double [B,Cout,2] or NULL: per-channel (sum, sum of squares) of the fp32 result; Cout <= 256.
 *                   Zeroed by the call unless sums_prezeroed != 0, in which case the statistics are added to it
 *   narrow_n        != 0: MMA N = 16, requires Cout == 16 and pyr_out
 *   pyr_out         fp32 [B,T,F,pyr_C] or NULL: pyramid output = result[..., :pyr_C] + bias[:pyr_C] + FIR-up x2(pyr_prev)
 *                   (1 <= pyr_C <= 4, Cout == MMA N, no sums, scale not applied)
 *   pyr_prev        fp32 [B,T/2,F/2,pyr_C] or NULL; requires even T and F
 *   comb_pyr        fp32 [B,T,F,comb_C] or NULL: out += comb_b[n] + sum_k comb_w[n * comb_C + k] * comb_pyr[b,t,f,k] after
 *                   `scale` (Combine, layerspp.py:52-59); needs comb_w [Cout,comb_C], comb_b [Cout], 1 <= comb_C <= 4
 * At most 16 K-blocks in all.  Violations are refused on the host (FDBM_EINVAL, message in fdbm_last_error()) before any
 * launch. */
typedef struct fdbm_conv_seg {
  const void* in;
  int C;
  int taps;
  const float* norm_tab;
  int tab_stride;
  int act;
} fdbm_conv_seg;

typedef struct fdbm_conv_desc {
  int struct_bytes;
  fdbm_conv_seg seg[3];
  int n_seg;
  const void* wpack;
  const float* bias;
  const float* bias_b;
  int bias_b_stride;
  const float* residual;
  const void* residual_h16;
  float scale;
  int B, T, F, Cout;
  float* out_f32;
  void* out_h16;
  double* sums;
  int sums_prezeroed;
  int narrow_n;
  float* pyr_out;
  const float* pyr_prev;
  int pyr_C;
  const float* comb_pyr;
  const float* comb_w;
  const float* comb_b;
  int comb_C;
} fdbm_conv_desc;

int fdbm_conv_igemm_ex(const fdbm_conv_desc* desc, void* stream);

/* (scale, shift) table of GroupNorm(min(Cr/4, 32) groups, eps 1e-6) over the channel concatenation of two tensors, as
 * the plans build it for normalise-on-load segments (layerspp.py:242-246): scale = gamma * rstd(group),
 * shift = beta - mean(group) * scale.
 *   sums1 double [B,C1,2], sums2 double [B,C2,2] or NULL (C2 = 0): per-channel (sum, sum of squares) over `pixels` pixels
 *   gamma, beta fp32 [C1+C2]
 *   blk_real    0, or the real channels of every 128-channel block (fdbm_arch.channel_block_real, e.g. 96): groups and
 *               counts follow the real channel index, padded channels get (0, 0); C1 and C2 multiples of 128.  Cr is the
 *               number of real channels
 *   table       fp32 [B, C1+C2, 2]
 *   stats       fp32 [B, G, 2] per-group (mean, rstd), G = min(Cr/4, 32), or NULL
 * C1 + C2 <= 512, and Cr divisible into G groups. */
int fdbm_gn_table(const double* sums1, int C1, const double* sums2, int C2, const float* gamma, const float* beta,
                  int blk_real, int batch, int64_t pixels, float* table, float* stats, void* stream);
/* ---- training step (SURVEY section 8 A10): gradients of the convolutions -------------------------------------
 * dgrad: dX = conv(dY, W') with W'[ci][co][df][dt] = W[co][ci][2-df][2-dt] -- pack W with
 * fdbm_pack_conv_weights_dgrad (w fp32 OIHW [Cout,Cin,k,k]; ksize -1: NIN matrix [Cin][Cout]) and call
 * fdbm_conv_igemm(in1 = dY, C1 = Cout, ksize, ..., Cout = Cin): the same tcgen05 kernel, epilogue included
 * (`residual` = the gradient already accumulated for that tensor).  Replaces the autograd of nn.Conv2d / NIN
 * (layers.py:100-124,546-555).  *bytes receives the packed size; wpack == NULL only queries it. */
int fdbm_pack_conv_weights_dgrad(const float* w, int Cout, int Cin, int ksize, void* wpack, int64_t* bytes,
                                 void* stream);
/* wgrad: dw[n,c,df,dt] += scale * sum_{b,t,f} dY[b,t,f,n] * X[b,t+dt-1,f+df-1,c]   (fp32 OIHW, accumulated)
 *   dy h16 [B,T,F,Cout] (Cout % 128 == 0), x h16 [B,T,F,Cin] (Cin % 64 == 0), ksize 3 or 1.
 * tcgen05 kernel with MN-major operands (pixels are the GEMM K), split over pixels; the fp32 partials of the
 * splits go through `workspace` (fdbm_conv_wgrad_workspace_bytes) and are summed in a fixed order. */
int64_t fdbm_conv_wgrad_workspace_bytes(int Cout, int Cin, int ksize, int batch, int T, int F);
int fdbm_conv_wgrad(const void* dy, int Cout, const void* x, int Cin, int ksize, int batch, int T, int F,
                    float scale, float* dw, float* workspace, void* stream);

/* GroupNorm(32 groups, eps 1e-6) (+ SiLU) backward (autograd of layerspp.py:242-246): a = act(GroupNorm(x)).
 *   g_a h16 [B,T,F,C] gradient w.r.t. a;  x the normalised tensor, fp32 or h16 (x_is_h16);  sums double [B,C,2] of x
 *   table: scratch of 2*B*C + 2*B*32 floats;  S: scratch of 2*B*C doubles
 *   outputs: g_x_acc fp32 [B,T,F,C] (+=, may be NULL), g_x_h16 (=, may be NULL), dgamma / dbeta fp32 [C] (+=, may be NULL) */
int fdbm_groupnorm_act_bwd(const void* g_a, const void* x, int x_is_h16, const double* sums, const float* gamma,
                           const float* beta, int silu, int batch, int T, int F, int C, float* table, double* S,
                           float* g_x_acc, void* g_x_h16, float* dgamma, float* dbeta, void* stream);
/* FIR x2 resampling of a h16 tensor with a scale: out = scale * upfirdn(in); mode 1 down, 2 up.  The adjoints of
 * upsample_2d / downsample_2d (up_or_down_sampling.py:195-257) are adjoint(down) = up / 4, adjoint(up) = 4 * down. */
int fdbm_fir_resample_h16(const void* in, int batch, int T, int F, int C, int mode, float scale, void* out, void* stream);
/* Backward of the attention core (layerspp.py:82-86): qkv h16 [B,L,3C] as produced by the forward, d_o h16 [B,L,C]
 * -> g_qkv h16 [B,L,3C].  scratch: 2*B*L*L floats. */
int fdbm_attention_bwd(const void* qkv, int batch, int L, int C, const void* d_o, float* scratch, void* g_qkv, void* stream);
/* Adam (model.py:101 configure_optimizers) with clip_grad_norm_ (gradient_clip_val) and the EMA update
 * (model.py:129-132, torch_ema.ExponentialMovingAverage.update) on flat fp32 buffers.  grads carry a factor grad_div
 * (loss scale x world size) that is divided out.  scratch: 1025 doubles (the squared norm is reduced in a fixed order so
 * that every DDP rank derives the same clipping coefficient).
 *   step        >= 1: the update count (Adam bias correction, EMA warm-up) given by the host;
 *               0: counted on the device in state[0] -- only APPLIED steps count
 *   ema_warmup  1: decay = min(ema_decay, (1 + n) / (10 + n)), torch_ema's use_num_updates=True default, which is what the
 *               reference constructs (model.py:56); 0: constant ema_decay
 *   state       device double[4] or NULL (required when step == 0): {applied updates, skipped steps, last gradient norm,
 *               reserved}.  A non-finite gradient norm SKIPS the step (GradScaler semantics): parameters, moments, EMA
 *               and state[0] stay as they are, state[1] is incremented. */
int fdbm_adam_ema_step(float* params, const float* grads, float* m, float* v, float* ema, int64_t n, double* scratch,
                       float grad_div, float clip_norm, float lr, float beta1, float beta2, float eps, int step,
                       float ema_decay, int ema_warmup, double* state, void* stream);

/* w1 fp32 OIHW [Cout,C1,k,k] (H = frequency, W = frames as in the reference), w2 fp32 [Cout,C2,1,1] or NULL
 * -> h16 [ (k*k*C1 + C2)/64 ][Cout][64] K-blocked, tap-major (ksize -1: w1 is a NIN matrix [C1][Cout]; ksize -2: the 3x3 input
 * convolution with 9 * C1 <= 64 as ONE K-block, k = tap * C1 + ci, for fdbm_im2col_input's columns).  Returns bytes via *bytes when wpack==NULL. */
int fdbm_pack_conv_weights(const float* w1, int C1, int ksize, const float* w2, int C2, int Cout,
                           void* wpack, int64_t* bytes, void* stream);

/* Single-head attention over all T*F positions (AttnBlockpp core, layerspp.py:82-86):
 * q,k,v h16 [B, L, C] (L = T*F) -> o h16 [B, L, C], scale C^-0.5. */
int fdbm_attention(const void* q, const void* k, const void* v, int batch, int L, int C, void* o, void* stream);

/* ---------------------------------------------------------------------------------------------
 * TF-GridNet backbones (fdbm/backbones/tfgridnet.py:126-229 TFGridNet.forward, :236-427 GridNetV3Block, :430-484 the
 * normalisation layers; tfgridnet_predictive.py): tfgridnet_5l32c100 is the backbone config.yaml selects.  Geometry:
 * emb_dim 32, emb_ks 4, emb_hs 1, 4 heads, E = 2, hidden <= 112.  Activations are fp32 [B, T, Q, 32] (Q = 257 bins, channels
 * innermost); "padded" tensors are [B, T+6, Q+6, 32] (tfgridnet.py:329-334).  One block of the network is
 *   fdbm_tfg_pad_add_norm -> fdbm_tfg_lstm_sweep (intra) -> fdbm_tfg_sweep_post(mode 0) -> fdbm_tfg_lstm_sweep (inter)
 *   -> fdbm_tfg_sweep_post(mode 1) -> fdbm_tfg_attention.
 *   fdbm_tfg_lstm_pack   both directions of an nn.LSTM layer (weight_ih [4H,128], weight_hh [4H,H], biases, PyTorch gate order
 *                        i,f,g,o; w = 8 device pointers, forward w_ih w_hh b_ih b_hh then reverse, as a HOST array) + the
 *                        ConvTranspose1d weight [2H,32,4] (tfgridnet.py:257-259) -> the four shared-memory images
 *                        [direction][cta rank] of the sweep, fdbm_tfg_lstm_pack_bytes() bytes; hidden <= 112
 *   fdbm_tfg_lstm_sweep  the bidirectional LSTM over n_seq sequences of L steps whose input at step s is the 4 x 32 window
 *                        xn[pos s .. s+3] of the LayerNorm-ed fp16 tensor (F.unfold, tfgridnet.py:337-341), xn contiguous
 *                        [n_seq][L+3][32].  tcgen05: a cluster of two CTAs owns 128 sequences of one direction, each holds the
 *                        gate columns of 56 of the 112 padded hidden units in shared memory, the gate GEMM of a step is UMMA
 *                        M=128 N=224 K=256 into TMEM, the new hidden state is exchanged through distributed shared memory.
 *                        Output per direction: fp16 [n_seq][L+3][32] = ConvTranspose1d(h) with its four taps overlap-added
 *                        (bias not included).
 *   fdbm_tfg_sweep_post  both directions' outputs + bias + residual (tfgridnet.py:346-350, :371-375); mode 0 (after intra):
 *                        full padded tensor out_full + its LayerNorm xn (fp16) for the inter sweep, written [B,Q+6,T+6,32] when
 *                        xn_transposed (the inter sweep's sequences contiguous), else [B,T+6,Q+6,32]; mode 1 (after inter):
 *                        the crop [B,T,Q,32] (tfgridnet.py:381)
 *   fdbm_tfg_pad_add_norm  xp = pad(h + emb[b, :]) (tfgridnet.py:217, :334), xn = fp16 LayerNorm(xp) (intra_norm); emb may be NULL
 *   fdbm_tfg_input       Conv2d(Cin -> 32, 3x3) + GroupNorm(1, 32) on complex [B,1,Q,T] inputs (tfgridnet.py:152-155, 201-214);
 *                        Cin = 4 (x.re, x.im, y.re, y.im) or 2 (predictive: pass the input as x, y = NULL); sums: 2*B doubles
 *   fdbm_tfg_time_embedding  Fourier features of log t -> Linear/SiLU x2 -> one Linear per block (tfgridnet.py:177-192, 203-219):
 *                        emb fp32 [n_layers][B][32]; w_blocks [n_layers][32][128], b_blocks [n_layers][32]
 *   fdbm_tfg_attention   full-band self-attention of a block (tfgridnet.py:383-427).  params: 20 DEVICE pointers in the order
 *                        conv_Q.w conv_Q.b conv_K.w conv_K.b conv_V.w conv_V.b | norm_Q.act norm_K.act norm_V.act |
 *                        norm_Q.gamma .beta norm_K.gamma .beta norm_V.gamma .beta | proj.0.w proj.0.b proj.1.w proj.2.gamma .beta
 *                        (a HOST array).  workspace: fdbm_tfg_attention_workspace_bytes(), 256-byte aligned.
 *   fdbm_tfg_output      ConvTranspose2d(32 -> 2, 3x3, padding 1) -> complex [B,1,Q,T] (tfgridnet.py:175, 221-226) */
int64_t fdbm_tfg_lstm_pack_bytes(void);
int fdbm_tfg_lstm_pack(const float* const* w, const float* w_lin, int hidden, void* packed, void* stream);
int fdbm_tfg_lstm_sweep(const void* xn, int n_seq, int L, const void* packed, void* y_fw, void* y_bw, void* stream);
int fdbm_tfg_pad_add_norm(const float* h, const float* emb, const float* gamma, const float* beta, int batch, int T, int Q, float eps,
                          float* xp, void* xn, void* stream);
int fdbm_tfg_sweep_post(const void* y_fw, const void* y_bw, const float* lin_bias, const float* resid, int batch, int T, int Q, int mode,
                        const float* gamma, const float* beta, float eps, float* out_full, void* xn, float* out_crop, int xn_transposed,
                        void* stream);
int fdbm_tfg_input(const float* x, const float* y, const float* w, const float* bias, const float* gn_w, const float* gn_b, int batch,
                   int T, int Q, int Cin, float eps, double* sums, float* out, void* stream);
int fdbm_tfg_time_embedding(const float* t, int t_stride, const float* fourier_w, const float* w1, const float* b1, const float* w2,
                            const float* b2, const float* w_blocks, const float* b_blocks, int n_layers, int batch, float* emb,
                            void* stream);
int64_t fdbm_tfg_attention_workspace_bytes(int batch, int T, int Q);
int fdbm_tfg_attention(const float* z, const float* const* params, int batch, int T, int Q, float eps, void* workspace, float* out,
                       void* stream);
int fdbm_tfg_output(const float* h, const float* w, const float* bias, int batch, int T, int Q, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FDBM_B200_H */
