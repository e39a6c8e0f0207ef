"""ctypes binding of libfdbm_b200.so (the C ABI declared in include/fdbm_b200.h).

There is no fallback: if the shared library is missing or a call fails, a RuntimeError is raised
(mirrors the TORCH_CHECK behaviour of the reference's only native op, op/upfirdn2d.cpp:8-16).
"""
from __future__ import annotations

import ctypes as C
import functools
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FDBM_B200_LIB") or os.path.join(_HERE, "libfdbm_b200.so")   # env override: developer A/B builds

FDBM_PAD = {"zero_pad": 0, "reflection": 1, "replication": 2}
FDBM_TRANSFORM = {"exponent": 0, "log": 1, "none": 2}
FDBM_STEP = {"ode_ei": 0, "sde_ei": 1}

# every symbol include/fdbm_b200.h declares; tests/test_abi.py checks the library exports all of them
EXPORTS = [
    "fdbm_last_error", "fdbm_version", "fdbm_check_device", "fdbm_operand_is_bf16",
    "fdbm_stft_compress", "fdbm_stft_compress_var", "fdbm_decompress_istft", "fdbm_decompress_istft_var",
    "fdbm_spec_transform", "fdbm_pad_spec",
    "fdbm_wave_absmax", "fdbm_stft_compress_ex", "fdbm_decompress_istft_ex", "fdbm_clip_rescale",
    "fdbm_prior_sample", "fdbm_bridge_step", "fdbm_bridge_update4", "fdbm_langevin_coef",
    "fdbm_lincomb", "fdbm_rk_error_norm",
    "fdbm_plan_create", "fdbm_plan_destroy", "fdbm_plan_load_weights", "fdbm_plan_device_bytes",
    "fdbm_plan_num_launches", "fdbm_ncsnpp_forward", "fdbm_sampler_run", "fdbm_plan_profile_forward",
    "fdbm_fir_resample", "fdbm_channel_stats", "fdbm_groupnorm_act", "fdbm_gn_resample_h16", "fdbm_conv_igemm", "fdbm_conv_igemm_ex",
    "fdbm_gn_table", "fdbm_pack_conv_weights", "fdbm_attention",
    "fdbm_pack_conv_weights_dgrad", "fdbm_conv_wgrad_workspace_bytes", "fdbm_conv_wgrad",
    "fdbm_groupnorm_act_bwd", "fdbm_fir_resample_h16", "fdbm_attention_bwd", "fdbm_adam_ema_step",
    "fdbm_plan_create_train", "fdbm_ncsnpp_backward", "fdbm_plan_param_info", "fdbm_plan_buffers",
    "fdbm_plan_num_backward_launches", "fdbm_plan_optimizer_step", "fdbm_plan_profile_backward", "fdbm_plan_repack_weights",
    "fdbm_plan_reset_optimizer", "fdbm_plan_optimizer_state", "fdbm_plan_set_optimizer_state", "fdbm_plan_swap_ema",
    "fdbm_hybrid_loss_workspace_bytes", "fdbm_hybrid_loss", "fdbm_data_prediction_loss",
    "fdbm_pack_input", "fdbm_im2col_input", "fdbm_time_embedding", "fdbm_film_rows", "fdbm_combine", "fdbm_output_layer",
    "fdbm_mel_tables_bytes", "fdbm_mel_tables_init", "fdbm_mel_loss_workspace_bytes", "fdbm_mel_loss",
    "fdbm_tfg_lstm_pack_bytes", "fdbm_tfg_lstm_pack", "fdbm_tfg_lstm_sweep", "fdbm_tfg_pad_add_norm", "fdbm_tfg_sweep_post",
    "fdbm_tfg_input", "fdbm_tfg_time_embedding", "fdbm_tfg_attention_workspace_bytes", "fdbm_tfg_attention", "fdbm_tfg_output",
]


class TensorRef(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("numel", C.c_int64)]


class Arch(C.Structure):
    _fields_ = [("nf", C.c_int), ("n_levels", C.c_int), ("ch_mult", C.c_int * 8), ("num_res_blocks", C.c_int),
                ("attn_resolution", C.c_int), ("predictive", C.c_int), ("image_size", C.c_int), ("channel_block_real", C.c_int)]


class ConvSeg(C.Structure):
    # `in` of the C struct is a Python keyword: the field is `in_` here (same offset and type)
    _fields_ = [("in_", C.c_void_p), ("C", C.c_int), ("taps", C.c_int), ("norm_tab", C.c_void_p), ("tab_stride", C.c_int),
                ("act", C.c_int)]


class ConvDesc(C.Structure):
    """fdbm_conv_desc: one convolution launch as the plans make it (fields documented in include/fdbm_b200.h)."""
    _fields_ = [("struct_bytes", C.c_int), ("seg", ConvSeg * 3), ("n_seg", C.c_int), ("wpack", C.c_void_p),
                ("bias", C.c_void_p), ("bias_b", C.c_void_p), ("bias_b_stride", C.c_int), ("residual", C.c_void_p),
                ("residual_h16", C.c_void_p), ("scale", C.c_float), ("B", C.c_int), ("T", C.c_int), ("F", C.c_int),
                ("Cout", C.c_int), ("out_f32", C.c_void_p), ("out_h16", C.c_void_p), ("sums", C.c_void_p),
                ("sums_prezeroed", C.c_int), ("narrow_n", C.c_int), ("pyr_out", C.c_void_p), ("pyr_prev", C.c_void_p),
                ("pyr_C", C.c_int), ("comb_pyr", C.c_void_p), ("comb_w", C.c_void_p), ("comb_b", C.c_void_p),
                ("comb_C", C.c_int)]

    def __init__(self, **kw):
        kw.setdefault("struct_bytes", C.sizeof(ConvDesc))
        kw.setdefault("scale", 1.0)
        super().__init__(**kw)


_lib = None


def load() -> C.CDLL:
    """Load the shared library once.  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C <package>/csrc`).  fdbm_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    p, i, i64, f, u64, d = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_double
    sig = {
        "fdbm_last_error": (C.c_char_p, []),
        "fdbm_version": (i, []),
        "fdbm_check_device": (i, []),
        "fdbm_operand_is_bf16": (i, []),
        "fdbm_stft_compress": (i, [p, i, i64, i64, p, i, i, i, f, f, i, i, p, p]),
        "fdbm_decompress_istft": (i, [p, i, i, p, i, i, i, f, f, i64, i64, p, p]),
        "fdbm_stft_compress_var": (i, [p, i, p, i64, i64, i64, p, i, i, i, f, f, i, i, p, p]),
        "fdbm_decompress_istft_var": (i, [p, i, i, p, i, i, i, f, f, p, i64, i64, p, p]),
        "fdbm_spec_transform": (i, [p, p, i64, i, f, f, i, p]),
        "fdbm_wave_absmax": (i, [p, i, i64, p, i64, p, p]),
        "fdbm_stft_compress_ex": (i, [p, i, p, i64, i64, i64, p, p, i, i, i, f, f, i, i, p, p]),
        "fdbm_decompress_istft_ex": (i, [p, i, i, p, i, i, i, f, f, p, i64, i64, p, p, p, p]),
        "fdbm_clip_rescale": (i, [p, i, i64, p, i64, p, f, p]),
        "fdbm_pad_spec": (i, [p, i64, i, i, i, p, p]),
        "fdbm_prior_sample": (i, [p, p, f, f, u64, u64, i64, p, p]),
        "fdbm_bridge_step": (i, [p, p, p, p, i, u64, u64, i64, p]),
        "fdbm_bridge_update4": (i, [p, p, p, p, p, u64, u64, i64, p, p]),
        "fdbm_langevin_coef": (i, [p, p, p, p, f, f, f, f, u64, u64, i, i64, p, p, p]),
        "fdbm_lincomb": (i, [p, C.POINTER(p), C.POINTER(f), i, i64, p]),
        "fdbm_rk_error_norm": (i, [C.POINTER(p), C.POINTER(f), i, p, p, f, f, i64, p, p]),
        "fdbm_plan_create": (i, [C.POINTER(Arch), i, i, C.POINTER(p)]),
        "fdbm_plan_destroy": (i, [p]),
        "fdbm_plan_load_weights": (i, [p, C.POINTER(TensorRef), i, p]),
        "fdbm_plan_device_bytes": (i64, [p]),
        "fdbm_plan_num_launches": (i, [p]),
        "fdbm_ncsnpp_forward": (i, [p, p, p, p, p, p]),
        "fdbm_sampler_run": (i, [p, p, p, p, p, i, i, p, u64, p]),
        "fdbm_plan_profile_forward": (i, [p, p, p, p, p, p, p, p, i, p]),
        "fdbm_fir_resample": (i, [p, i, i, i, i, i, p, p]),
        "fdbm_channel_stats": (i, [p, i, i, i, i, p, p]),
        "fdbm_groupnorm_act": (i, [p, p, i, p, p, i, p, p, i, i, i, i, i, p, p, p]),
        "fdbm_gn_resample_h16": (i, [p, p, i, p, p, i, p, p, p, i, i, i, i, p, p, p]),
        "fdbm_conv_igemm": (i, [p, i, i, p, i, p, p, p, p, f, i, i, i, i, p, p, p, p]),
        "fdbm_conv_igemm_ex": (i, [C.POINTER(ConvDesc), p]),
        "fdbm_gn_table": (i, [p, i, p, i, p, p, i, i, i64, p, p, p]),
        "fdbm_pack_conv_weights": (i, [p, i, i, p, i, i, p, C.POINTER(i64), p]),
        "fdbm_pack_conv_weights_dgrad": (i, [p, i, i, i, p, C.POINTER(i64), p]),
        "fdbm_conv_wgrad_workspace_bytes": (i64, [i, i, i, i, i, i]),
        "fdbm_conv_wgrad": (i, [p, i, p, i, i, i, i, i, f, p, p, p]),
        "fdbm_groupnorm_act_bwd": (i, [p, p, i, p, p, p, i, i, i, i, i, p, p, p, p, p, p, p]),
        "fdbm_fir_resample_h16": (i, [p, i, i, i, i, i, f, p, p]),
        "fdbm_attention_bwd": (i, [p, i, i, i, p, p, p, p]),
        "fdbm_adam_ema_step": (i, [p, p, p, p, p, i64, p, f, f, f, f, f, f, i, f, i, p, p]),
        "fdbm_plan_create_train": (i, [C.POINTER(Arch), i, i, C.POINTER(p)]),
        "fdbm_ncsnpp_backward": (i, [p, p, f, i, p]),
        "fdbm_plan_param_info": (i, [p, C.c_char_p, C.POINTER(i64), C.POINTER(i64)]),
        "fdbm_plan_buffers": (i, [p, C.POINTER(p), C.POINTER(p), C.POINTER(p), C.POINTER(i64)]),
        "fdbm_plan_num_backward_launches": (i, [p]),
        "fdbm_plan_repack_weights": (i, [p, p]),
        "fdbm_hybrid_loss_workspace_bytes": (i64, [i, i, i, i]),
        "fdbm_hybrid_loss": (i, [p, p, i, i, p, i, i, i, f, f, f, p, p, p, p]),
        "fdbm_data_prediction_loss": (i, [p, p, i, i, p, i, i, i, f, f, f, f, p, p, p, p]),
        "fdbm_pack_input": (i, [p, p, i, i, i, i, i, p, p]),
        "fdbm_im2col_input": (i, [p, i, i, i, i, p, p]),
        "fdbm_time_embedding": (i, [p, p, i, p, p, p, p, i, p, p]),
        "fdbm_film_rows": (i, [p, p, p, i, i, i, p, p]),
        "fdbm_combine": (i, [p, p, i, p, p, i, i, i, i, p]),
        "fdbm_output_layer": (i, [p, i, p, p, i, i, i, i, p, p]),
        "fdbm_mel_tables_bytes": (i64, []),
        "fdbm_mel_tables_init": (i, [p, i, p]),
        "fdbm_mel_loss_workspace_bytes": (i64, [i, i, i, i]),
        "fdbm_mel_loss": (i, [p, p, i, i, p, i, i, i, f, f, i, f, p, p, p, p, p]),
        "fdbm_plan_profile_backward": (i, [p, p, f, p, p, i, p]),
        "fdbm_plan_optimizer_step": (i, [p, f, f, f, f, f, f, i, f, i, p]),
        "fdbm_plan_reset_optimizer": (i, [p, p]),
        "fdbm_plan_optimizer_state": (i, [p, C.POINTER(d), p]),
        "fdbm_plan_set_optimizer_state": (i, [p, d, d, p]),
        "fdbm_plan_swap_ema": (i, [p, i, p]),
        "fdbm_attention": (i, [p, p, p, i, i, i, p, p]),
        "fdbm_tfg_lstm_pack_bytes": (i64, []),
        "fdbm_tfg_lstm_pack": (i, [p, p, i, p, p]),
        "fdbm_tfg_lstm_sweep": (i, [p, i, i, p, p, p, p]),
        "fdbm_tfg_pad_add_norm": (i, [p, p, p, p, i, i, i, f, p, p, p]),
        "fdbm_tfg_sweep_post": (i, [p, p, p, p, i, i, i, i, p, p, f, p, p, p, i, p]),
        "fdbm_tfg_input": (i, [p, p, p, p, p, p, i, i, i, i, f, p, p, p]),
        "fdbm_tfg_time_embedding": (i, [p, i, p, p, p, p, p, p, p, i, i, p, p]),
        "fdbm_tfg_attention_workspace_bytes": (i64, [i, i, i]),
        "fdbm_tfg_attention": (i, [p, C.POINTER(p), i, i, i, f, p, p, p]),
        "fdbm_tfg_output": (i, [p, p, p, i, i, i, p, p]),
    }
    for name, (res, args) in sig.items():
        if not hasattr(lib, name) and os.environ.get("FDBM_B200_LIB"):
            continue                      # developer A/B build of an older revision
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "fdbm") -> None:
    if rc != 0:
        msg = load().fdbm_last_error()
        raise RuntimeError(f"{what} failed (code {rc}): {msg.decode() if msg else 'unknown error'}")


def operand_dtype():
    """torch dtype of the library's 16-bit GEMM operands (fp16 unless built with -DFDBM_OPERAND_BF16)."""
    import torch
    return torch.bfloat16 if load().fdbm_operand_is_bf16() else torch.float16


def ptr(t) -> int:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream() -> int:
    """The CURRENT device's current stream; callers select the tensors' device first (`on_device`)."""
    import torch
    return torch.cuda.current_stream().cuda_stream


def on_device(fn):
    """Run `fn` with the CUDA device of its first CUDA-tensor argument selected.  The library allocates, launches and
    takes streams on the *current* device, while the reference's multi-GPU workers only move tensors with
    `.to(f'cuda:{gpu_id}')` and never call `torch.cuda.set_device` (infer_folder.py:70-74,110).  All CUDA tensor
    arguments must live on one device."""
    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        import torch
        dev = None
        for a in list(args) + list(kwargs.values()):
            if isinstance(a, torch.Tensor) and a.is_cuda:
                if dev is None:
                    dev = a.device
                elif a.device != dev:
                    raise RuntimeError(f"{fn.__qualname__}: tensors on different devices ({dev} and {a.device})")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper
