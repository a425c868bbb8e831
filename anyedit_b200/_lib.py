"""ctypes binding of ``libanysd_b200.so`` (C ABI declared in include/anysd_b200.h).

The library is the product; there is no Python/CPU fallback.  If the shared object is missing
or a call fails, this module raises -- it never silently degrades to eager PyTorch.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libanysd_b200.so")

F32, F16, I64 = 0, 1, 2
EINVAL, ECUDA, EUNSUPPORTED = -1, -2, -3


class GemmParams(C.Structure):
    _fields_ = [
        ("A", C.c_void_p), ("W", C.c_void_p), ("bias", C.c_void_p), ("rowadd", C.c_void_p),
        ("residual", C.c_void_p), ("out", C.c_void_p),
        ("M", C.c_int), ("N", C.c_int), ("K", C.c_int),
        ("lda", C.c_int), ("ldw", C.c_int), ("ldo", C.c_int), ("ldr", C.c_int), ("ld_rowadd", C.c_int),
        ("rows_per_batch", C.c_int), ("act", C.c_int), ("out_dtype", C.c_int), ("conv", C.c_int),
        ("Nimg", C.c_int), ("H", C.c_int), ("Wd", C.c_int), ("Cin", C.c_int),
        ("stride", C.c_int), ("upsample", C.c_int),
        ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
        ("conv_pad", C.c_int),
        ("stats", C.c_void_p), ("stats_images", C.c_int),
        ("splitk_workspace", C.c_void_p), ("splitk_workspace_bytes", C.c_size_t),
        ("splitk_counters", C.c_void_p), ("splitk_counters_bytes", C.c_size_t),
        ("row_stats", C.c_void_p), ("ln_stats", C.c_void_p), ("ln_colsum", C.c_void_p), ("ln_eps", C.c_float),
    ]


class AttnParams(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p),
        ("q_batch_stride", C.c_longlong), ("k_batch_stride", C.c_longlong),
        ("v_batch_stride", C.c_longlong), ("o_batch_stride", C.c_longlong),
        ("ld_q", C.c_int), ("ld_k", C.c_int), ("ld_v", C.c_int), ("ld_o", C.c_int),
        ("B", C.c_int), ("heads", C.c_int), ("n_q", C.c_int), ("n_kv", C.c_int), ("d", C.c_int),
        ("scale", C.c_float), ("gate", C.c_void_p), ("gate_stride", C.c_int), ("accumulate", C.c_int),
        ("head_stride", C.c_int),
        ("aux_cols", C.c_int),
        ("lse", C.c_void_p),
    ]


class AttnBwdParams(C.Structure):          # mirrors anysd_attn_bwd_params field for field
    _fields_ = [("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("d_out", C.c_void_p),
                ("dq", C.c_void_p), ("dk", C.c_void_p), ("dv", C.c_void_p),
                ("q_batch_stride", C.c_longlong), ("k_batch_stride", C.c_longlong), ("v_batch_stride", C.c_longlong),
                ("do_batch_stride", C.c_longlong), ("dq_batch_stride", C.c_longlong), ("dk_batch_stride", C.c_longlong),
                ("dv_batch_stride", C.c_longlong),
                ("ld_q", C.c_int), ("ld_k", C.c_int), ("ld_v", C.c_int), ("ld_do", C.c_int), ("ld_dq", C.c_int),
                ("ld_dk", C.c_int), ("ld_dv", C.c_int),
                ("B", C.c_int), ("heads", C.c_int), ("n_q", C.c_int), ("n_kv", C.c_int), ("d", C.c_int),
                ("head_stride", C.c_int), ("qk_scale", C.c_float),
                ("gate", C.c_void_p), ("gate_stride", C.c_int), ("d_gate", C.c_void_p),
                ("accumulate_dq", C.c_int), ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t),
                ("out", C.c_void_p), ("o_batch_stride", C.c_longlong), ("ld_o", C.c_int),
                ("lse", C.c_void_p), ("dout_padded", C.c_void_p)]


class ExpertAttnParams(C.Structure):       # mirrors anysd_expert_attn_params field for field
    _fields_ = [("q", C.c_void_p), ("kv", C.c_void_p), ("out", C.c_void_p),
                ("ld_q", C.c_int), ("ld_kv", C.c_int), ("ld_o", C.c_int),
                ("B", C.c_int), ("heads", C.c_int), ("n_q", C.c_int), ("n_kv", C.c_int), ("d", C.c_int),
                ("head_stride", C.c_int), ("E", C.c_int), ("set_stride", C.c_int), ("v_offset", C.c_int),
                ("qk_scale", C.c_float), ("gates", C.c_void_p), ("gate_b_stride", C.c_int)]


# name -> (restype, argtypes); mirrors include/anysd_b200.h one to one
_VP, _I, _LL, _F, _SZ = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_size_t
SIGNATURES = {
    "anysd_last_error": (C.c_char_p, []),
    "anysd_version": (_I, []),
    "anysd_device_info": (_I, [C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "anysd_nchw_to_nhwc_f16": (_I, [_VP, _I, _VP, _I, _I, _I, _I, _I, _I, _VP]),
    "anysd_add_nchw_into_nhwc_f16": (_I, [_VP, _I, _VP, _I, _I, _I, _I, _VP]),
    "anysd_nhwc_to_nchw": (_I, [_VP, _I, _I, _VP, _I, _I, _I, _I, _I, _VP]),
    "anysd_concat_channels_f16": (_I, [_VP, _I, _VP, _I, _VP, _LL, _VP]),
    "anysd_cast_f32_to_f16": (_I, [_VP, _VP, _LL, _VP]),
    "anysd_timestep_embedding_f16": (_I, [_VP, _I, _VP, _I, _I, _F, _VP]),
    "anysd_emb_finalize": (_I, [_VP, _VP, _VP, _I, _VP, _VP, _I, _I, _VP]),
    "anysd_router_gate_f32": (_I, [_VP, _VP, _I, _VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "anysd_groupnorm_workspace_bytes": (_SZ, [_I, _I, _I]),
    "anysd_groupnorm_resident": (_I, [_I, _I, _I, _I]),
    "anysd_groupnorm_nhwc_f16": (_I, [_VP, _I, _VP, _I, _VP, _VP, _VP, _I, _I, _I, _F, _I, _VP, _SZ, _VP]),
    "anysd_layernorm_f16": (_I, [_VP, _VP, _VP, _VP, _LL, _I, _F, _VP]),
    "anysd_gemm_f16": (_I, [C.POINTER(GemmParams), _VP]),
    "anysd_gemm_stats_slabs": (_I, [C.POINTER(GemmParams)]),
    "anysd_gemm_splitk_workspace_bytes": (_SZ, [C.POINTER(GemmParams)]),
    "anysd_gemm_schedule": (_I, [C.POINTER(GemmParams)] + [C.POINTER(C.c_int)] * 6),
    "anysd_groupnorm_apply_nhwc_f16": (_I, [_VP, _I, _VP, _I, _VP, _I, _VP, _VP, _VP, _I, _I, _I, _F, _I, _VP, _SZ, _VP]),
    "anysd_attention_f16": (_I, [C.POINTER(AttnParams), _VP]),
    "anysd_cfg_ddim_step_f32": (_I, [_VP, _VP, _VP, _VP, _F, _I, _I, _VP, _VP, _LL, _I, _VP]),
    "anysd_cfg3_ddim_step_f32": (_I, [_VP, _VP, _VP, _VP, _F, _F, _VP, _VP, _LL, _I, _VP]),
    "anysd_cfg_plms_step_f32": (_I, [_VP, _VP, _VP, _F, _I, _VP, _VP, _VP, _LL, _I, _VP]),
    "anysd_cfg_dpmpp_step_f32": (_I, [_VP, _VP, _VP, _F, _I, _VP, _VP, _VP, _LL, _I, _VP]),
    "anysd_softmax_rows_f32": (_I, [_VP, _LL, _VP, _LL, _I, _I, _F, _VP]),
    "anysd_gaussian_posterior_f32": (_I, [_VP, _VP, _VP, _VP, _F, _I, _LL, _VP]),
    "anysd_embed_tokens_f16": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I, _I, _VP]),
    "anysd_attention_small_f16": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I, _I, _I, _I, _I, _I, _I, _F, _I, _VP]),
    # ---- training step ----
    "anysd_q_sample_f32": (_I, [_VP, _VP, _VP, _VP, _VP, _VP, _I, _LL, _VP]),
    "anysd_mse_workspace_bytes": (_SZ, []),
    "anysd_mse_loss_f32": (_I, [_VP, _VP, _I, _I, _I, _I, _F, _VP, _VP, _VP, _VP, _SZ, _VP]),
    "anysd_geglu_f16": (_I, [_VP, _VP, _LL, _I, _VP]),
    "anysd_geglu_bwd_f16": (_I, [_VP, _VP, _VP, _LL, _I, _VP]),
    "anysd_silu_bwd_f32": (_I, [_VP, _VP, _VP, _LL, _VP]),
    "anysd_groupnorm_bwd_nhwc_f16": (_I, [_VP, _I, _VP, _I, _VP, _VP, _VP, _VP, _I, _I, _I, _F, _I, _VP]),
    "anysd_layernorm_bwd_f16": (_I, [_VP, _VP, _VP, _VP, _LL, _I, _F, _VP]),
    "anysd_attention_bwd_workspace_bytes": (_SZ, [_I, _I, _I]),
    "anysd_attention_bwd_f16": (_I, [C.POINTER(AttnBwdParams), _VP]),
    "anysd_expert_attention_f16": (_I, [C.POINTER(ExpertAttnParams), _VP]),
    "anysd_expert_attention_bwd_workspace_bytes": (_SZ, [_I, _I, _I, _I]),
    "anysd_expert_attention_bwd_f16": (_I, [C.POINTER(ExpertAttnParams), _VP, _I, _VP, _I, _VP, _VP, _VP, _SZ, _VP]),
    "anysd_colsum_f16": (_I, [_VP, _VP, _I, _I, _I, _I, _I, _VP]),
    "anysd_add_f16": (_I, [_VP, _VP, _LL, _VP]),
    "anysd_split_channels_f16": (_I, [_VP, _VP, _I, _VP, _I, _LL, _VP]),
    "anysd_zero_insert2x_f16": (_I, [_VP, _VP, _I, _I, _I, _I, _VP]),
    "anysd_sumpool2x_f16": (_I, [_VP, _VP, _I, _I, _I, _I, _VP]),
    "anysd_gemm_tn_f32": (_I, [_VP, _I, _I, _I, _I, _I, _VP, _I, _VP, _I, _I, _I, _I, _F, _I, _VP]),
    "anysd_gather_transpose_f16": (_I, [_VP, _I, _I, _I, _I, _I, _VP, _I, _I, _I, _VP]),
    "anysd_router_bwd_f32": (_I, [_VP, _VP, _VP, _VP, _I, _I, _I, _I, _F, _VP, _VP, _VP, _VP]),
    "anysd_scatter_add_rows_f32": (_I, [_VP, _VP, _I, _I, _I, _F, _VP, _VP]),
    "anysd_adamw_f32": (_I, [_VP, _VP, _VP, _VP, _LL, _F, _F, _F, _F, _F, _I, _F, _VP]),
    "anysd_grad_check_f32": (_I, [_VP, _LL, _VP, _VP]),
    "anysd_adamw_scaled_f32": (_I, [_VP, _VP, _VP, _VP, _LL, _F, _F, _F, _F, _F, _F, _VP, _VP]),
    "anysd_loss_scale_update_f32": (_I, [_VP, _F, _F, _I, _VP]),
}

_lib = None


class AnysdError(RuntimeError):
    pass


def load():
    """Load (once) and return the ctypes handle; raises if the CUDA library is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AnysdError(
            f"{LIB_PATH} is missing: build it with `python -m anyedit_b200.build` "
            "(or __graft_entry__.build()). anyedit_b200 has no CPU / eager fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc == 0:
        return
    msg = load().anysd_last_error().decode(errors="replace")
    if rc in (EINVAL, EUNSUPPORTED):
        raise ValueError(f"anysd_b200 {what}: {msg}")
    raise AnysdError(f"anysd_b200 {what}: {msg} (code {rc})")
