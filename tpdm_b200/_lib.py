"""ctypes binding of libtpdm_b200.so (include/tpdm_b200.h).  There is no fallback: if the shared library is missing
or a call fails, an exception is raised."""
from __future__ import annotations

import ctypes as C
import math
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TPDM_B200_LIB", os.path.join(HERE, "libtpdm_b200.so"))

c_float_p = C.POINTER(C.c_float)
vp = C.c_void_p

TPDM_OK, TPDM_ERR_ARG, TPDM_ERR_SHAPE, TPDM_ERR_CUDA, TPDM_ERR_STATE, TPDM_ERR_NOMEM = 0, -1, -2, -3, -4, -5


class TpdmConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "num_layers", "num_heads", "head_dim", "joint_attention_dim", "pooled_projection_dim", "in_channels",
        "out_channels", "patch_size", "pos_embed_max_size", "qk_norm", "tpm_channels", "prediction_type", "relative")
    ] + [("min_sigma", C.c_float), ("epsilon", C.c_float), ("tpm_epsilon", C.c_float), ("dual_attention_mask", C.c_uint64)]


BLOCK_FIELDS = ("qkv_w", "qkv_b", "cqkv_w", "cqkv_b", "out_w", "out_b", "cout_w", "cout_b", "ff1_w", "ff1_b", "ff2_w",
                "ff2_b", "cff1_w", "cff1_b", "cff2_w", "cff2_b", "norm_q", "norm_k", "norm_added_q", "norm_added_k",
                "qkv2_w", "qkv2_b", "out2_w", "out2_b", "norm_q2", "norm_k2")


class TpdmBlockWeights(C.Structure):
    _fields_ = [(n, vp) for n in BLOCK_FIELDS]


FP8_BLOCK_FIELDS = ("qkv_w", "qkv_s", "cqkv_w", "cqkv_s", "ff1_w", "ff1_s", "cff1_w", "cff1_s")


class TpdmFp8BlockWeights(C.Structure):
    _fields_ = [(n, vp) for n in FP8_BLOCK_FIELDS]


GLOBAL_FIELDS_A = ("patch_w", "patch_b", "pos_table", "t_w1", "t_b1", "t_w2", "t_b2", "p_w1", "p_b1", "p_w2", "p_b2",
                   "ctx_w", "ctx_b", "adaln_w", "adaln_b", "proj_w", "proj_b")
GLOBAL_FIELDS_B = ("tpm_conv1_w", "tpm_conv1_b", "tpm_lin_w", "tpm_lin_b", "tpm_gn_w", "tpm_gn_b", "tpm_conv2_w",
                   "tpm_conv2_b", "tpm_fc1_w", "tpm_fc1_b", "tpm_fc2_w", "tpm_fc2_b")


class TpdmWeights(C.Structure):
    _fields_ = [(n, vp) for n in GLOBAL_FIELDS_A] + [("blocks", C.POINTER(TpdmBlockWeights))] + [(n, vp) for n in GLOBAL_FIELDS_B]


class TpdmVaeConfig(C.Structure):
    _fields_ = [("latent_channels", C.c_int32), ("out_channels", C.c_int32), ("num_levels", C.c_int32),
                ("block_out_channels", C.c_int32 * 8), ("layers_per_block", C.c_int32), ("norm_num_groups", C.c_int32),
                ("scaling_factor", C.c_float), ("shift_factor", C.c_float)]


VAE_RESNET_FIELDS = ("norm1_w", "norm1_b", "conv1_w", "conv1_b", "norm2_w", "norm2_b", "conv2_w", "conv2_b", "short_w", "short_b")


class TpdmVaeResnet(C.Structure):
    _fields_ = [(n, vp) for n in VAE_RESNET_FIELDS]


class TpdmVaeWeights(C.Structure):
    _fields_ = ([("conv_in_w", vp), ("conv_in_b", vp), ("resnets", C.POINTER(TpdmVaeResnet)), ("n_resnets", C.c_int32)] +
                [(n, vp) for n in ("attn_norm_w", "attn_norm_b", "attn_q_w", "attn_k_w", "attn_v_w", "attn_o_w",
                                   "attn_q_b", "attn_k_b", "attn_v_b", "attn_o_b")] +
                [("up_conv_w", C.POINTER(vp)), ("up_conv_b", C.POINTER(vp)), ("n_upsamplers", C.c_int32)] +
                [(n, vp) for n in ("norm_out_w", "norm_out_b", "conv_out_w", "conv_out_b")])


class TpdmSampleState(C.Structure):
    _fields_ = [(n, vp) for n in ("latents", "velocity", "sigma_hist", "alphas", "betas", "logprobs", "prob_masks",
                                  "all_done", "tembs", "tpm_input", "history_latents")]


class TpdmGemmOpDesc(C.Structure):
    _fields_ = ([("A", vp), ("a_row_stride", C.c_int64), ("a_batch_stride", C.c_int64), ("W", vp), ("out", vp),
                 ("out_batch_stride", C.c_int64)] + [(n, vp) for n in ("bias", "gate", "a_scale", "w_scale")] +
                [(n, C.c_int32) for n in ("rows", "batch", "K", "N", "epi", "ldo", "gate_stride", "ksplit")])


class TpdmRequestOptions(C.Structure):
    _fields_ = [("guidance_scale", C.c_float), ("max_steps", C.c_int32), ("predict", C.c_int32), ("reserved", C.c_int32),
                ("seed", C.c_uint64)]


EXPORTS = {
    "tpdm_last_error": (C.c_char_p, []),
    "tpdm_abi_version": (C.c_int, []),
    "tpdm_create": (C.c_int, [C.POINTER(TpdmConfig), C.POINTER(vp)]),
    "tpdm_destroy": (C.c_int, [vp]),
    "tpdm_set_weights": (C.c_int, [vp, C.POINTER(TpdmWeights)]),
    "tpdm_set_fp8_weights": (C.c_int, [vp, C.POINTER(TpdmFp8BlockWeights)]),
    "tpdm_plan_workspace_bytes": (C.c_size_t, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "tpdm_plan_create": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, C.POINTER(vp)]),
    "tpdm_plan_destroy": (C.c_int, [vp]),
    "tpdm_mmdit_forward": (C.c_int, [vp] + [vp] * 8 + [vp]),
    "tpdm_tpm_forward": (C.c_int, [vp, vp, vp, vp, vp]),
    "tpdm_euler_step": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_longlong, vp]),
    "tpdm_sample_begin": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_float, C.c_int, vp, C.c_ulonglong, vp]),
    "tpdm_sample_step": (C.c_int, [vp, C.c_int, vp]),
    "tpdm_sample_step_graph": (C.c_int, [vp, C.c_int, vp]),
    "tpdm_sample_state_get": (C.c_int, [vp, C.POINTER(TpdmSampleState)]),
    "tpdm_tpm_param_offsets": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_longlong)]),
    "tpdm_tpm_trainer_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "tpdm_tpm_trainer_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, vp, C.c_size_t, C.POINTER(vp)]),
    "tpdm_tpm_trainer_destroy": (C.c_int, [vp]),
    "tpdm_tpm_trainer_bind": (C.c_int, [vp, vp, vp, vp]),
    "tpdm_tpm_train_forward": (C.c_int, [vp, vp, vp, C.c_int, vp, vp]),
    "tpdm_tpm_train_backward": (C.c_int, [vp, vp, vp]),
    "tpdm_queue_workspace_bytes": (C.c_size_t, [vp, C.c_int]),
    "tpdm_queue_begin": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, C.c_float, vp, C.c_size_t, vp, vp, vp, vp, vp, C.c_int, vp, C.c_int, vp]),
    "tpdm_queue_set_rollout": (C.c_int, [vp, C.c_ulonglong, vp, vp, vp, vp, vp, vp]),
    "tpdm_queue_step": (C.c_int, [vp, vp]),
    "tpdm_queue_step_graph": (C.c_int, [vp, vp]),
    "tpdm_queue_status": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp)]),
    "tpdm_stream_workspace_bytes": (C.c_size_t, [vp, C.c_int]),
    "tpdm_stream_open": (C.c_int, [vp, C.c_int, C.c_float, vp, C.c_size_t, vp]),
    "tpdm_stream_submit": (C.c_int, [vp, C.c_int, C.POINTER(C.c_int), vp, vp, vp, vp, vp, vp]),
    "tpdm_stream_submit_options": (C.c_int, [vp, C.c_int, C.POINTER(C.c_int), vp, vp, vp, vp, vp, C.POINTER(TpdmRequestOptions), vp]),
    "tpdm_stream_records": (C.c_int, [vp] + [C.POINTER(vp)] * 3),
    "tpdm_stream_status": (C.c_int, [vp] + [C.POINTER(vp)] * 5),
    "tpdm_stream_close": (C.c_int, [vp]),
    "tpdm_vae_create": (C.c_int, [C.POINTER(TpdmVaeConfig), C.POINTER(vp)]),
    "tpdm_vae_destroy": (C.c_int, [vp]),
    "tpdm_vae_num_resnets": (C.c_int, [vp]),
    "tpdm_vae_set_weights": (C.c_int, [vp, C.POINTER(TpdmVaeWeights)]),
    "tpdm_vae_workspace_bytes": (C.c_size_t, [vp, C.c_int, C.c_int]),
    "tpdm_vae_decode": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_size_t, vp, vp, vp]),
    "tpdm_rollout_shaping": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int,
                                       vp, vp, vp, vp, vp]),
    "tpdm_ppo_clip_loss": (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_float, C.c_float, vp, vp, vp,
                                     vp, vp]),
    "tpdm_beta_logprob": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_int, C.c_int, C.c_float, vp, vp, vp]),
    "tpdm_adamw_step": (C.c_int, [vp, vp, vp, vp, C.c_longlong, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int,
                                  C.c_float, vp, vp, C.c_longlong, vp, vp]),
    "tpdm_launch_count": (C.c_longlong, [C.c_int]),
    "tpdm_profile_start": (C.c_int, [C.c_int]),
    "tpdm_profile_dropped": (C.c_longlong, []),
    "tpdm_profile_stop": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.c_int]),
    "tpdm_gemm_bf16": (C.c_int, [vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_joint_attention": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_attention_redo_count": (C.c_int, []),
    "tpdm_attention_redo_total": (C.c_longlong, []),
    "tpdm_conv3x3_nhwc": (C.c_int, [vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_conv3x3_wgrad": (C.c_int, [vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_ln_modulate": (C.c_int, [vp, vp, vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_ln_modulate_pair": (C.c_int, [vp, vp, vp, vp, C.c_int, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_quantize_fp8_rows": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp]),
    "tpdm_ln_modulate_fp8": (C.c_int, [vp, vp, vp, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_gemm_fp8": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp]),
    "tpdm_set_launch_guards": (C.c_int, [vp, vp, C.c_int]),
    "tpdm_gemm_ops": (C.c_int, [C.POINTER(TpdmGemmOpDesc), C.c_int, vp]),
}

_lib = None


def load() -> C.CDLL:
    """Load the C-ABI library; raises RuntimeError if it has not been built (python -m tpdm_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -m tpdm_b200.build` "
                               "(tpdm_b200 has no CPU / PyTorch fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in EXPORTS.items():
            fn = getattr(lib, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if lib.tpdm_abi_version() != 3:
            raise RuntimeError("libtpdm_b200.so ABI version mismatch")
        _lib = lib
    return _lib


def check(status: int) -> None:
    if status == TPDM_OK:
        return
    msg = load().tpdm_last_error().decode("utf-8", "replace")
    if status in (TPDM_ERR_ARG, TPDM_ERR_SHAPE):
        raise ValueError(msg)
    raise RuntimeError(f"libtpdm_b200 error {status}: {msg}")


def ptr(t) -> int:
    """Device pointer of a torch tensor (None -> NULL).  The tensor must be CUDA and contiguous."""
    if t is None:
        return None
    if not t.is_cuda:
        raise ValueError("tpdm_b200 needs CUDA tensors (there is no CPU path)")
    if not t.is_contiguous():
        raise ValueError("tpdm_b200 needs contiguous tensors")
    return t.data_ptr()


def stream_ptr() -> int:
    import torch

    return torch.cuda.current_stream().cuda_stream


def aligned_workspace(nbytes: int, device):
    """A device byte tensor holding ``nbytes`` bytes from a 1 KiB-aligned address on, as the library's workspaces need:
    (tensor, that address)."""
    import torch

    ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=device)
    return ws, (ws.data_ptr() + 1023) // 1024 * 1024


def view_at(ws, ptr: int, dtype, shape):
    """Typed view of the buffer the library placed at device address ``ptr`` inside the workspace tensor ``ws``."""
    off = ptr - ws.data_ptr()
    n = math.prod(shape) * dtype.itemsize
    return ws[off: off + n].view(dtype).view(shape)
