"""ctypes binding of libdmn_b200.so (include/dmn_b200.h).

The library is the product: if it is missing or fails to load this module raises -- there is no
PyTorch/CPU fallback anywhere in the package.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DMN_LIB_PATH") or os.path.join(_HERE, "libdmn_b200.so")   # override: A/B builds in tools/

ACT_F32, ACT_BF16 = 0, 1
CONV_SIMT, CONV_TCGEN05 = 0, 1
LOOP_DDPM, LOOP_LEARNED, LOOP_DDIM, LOOP_PC, LOOP_BPD, LOOP_DPMPP = 0, 1, 2, 3, 4, 5
COEF_STRIDE = 8


class UnetCfg(C.Structure):
    _fields_ = [
        ("dim", C.c_int32), ("n_mults", C.c_int32), ("dim_mults", C.c_int32 * 8), ("channels", C.c_int32),
        ("out_dim", C.c_int32), ("groups", C.c_int32), ("with_time_emb", C.c_int32), ("num_classes", C.c_int32),
        ("image_size", C.c_int32), ("max_batch", C.c_int32), ("act_dtype", C.c_int32), ("conv_engine", C.c_int32),
        ("max_time_rows", C.c_int32), ("film", C.c_int32), ("plain_tail", C.c_int32), ("reserved", C.c_int32 * 1),
    ]


class Rng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("stream_id", C.c_uint64)]


class LoopDesc(C.Structure):
    _fields_ = [
        ("kind", C.c_int32), ("n_steps", C.c_int32), ("batch", C.c_int32), ("n_corr", C.c_int32),
        ("snr", C.c_float), ("denoise", C.c_int32), ("use_graph", C.c_int32), ("corr_kind", C.c_int32),
        ("coef_dev", C.c_void_p), ("coef2_dev", C.c_void_p), ("classes_dev", C.c_void_p), ("noise_dev", C.c_void_p),
        ("rng", Rng), ("state_dev", C.c_void_p), ("aux_dev", C.c_void_p), ("scratch_dev", C.c_void_p),
        ("scratch_bytes", C.c_size_t), ("traj_dev", C.c_void_p), ("traj_every", C.c_int32), ("cfg_scale", C.c_float),
        ("cfg_on", C.c_int32), ("state_elems", C.c_int64),
    ]


class InpaintDesc(C.Structure):
    _fields_ = [("known_dev", C.c_void_p), ("mask_dev", C.c_void_p), ("prep_coef_dev", C.c_void_p)]


SDE_VP, SDE_VE = 0, 1
ODE_RUNNING, ODE_DONE, ODE_TOO_SMALL_STEP, ODE_LIMIT = 0, 1, -1, -2


class OdeResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("nfev", C.c_int32), ("n_accepted", C.c_int32), ("n_rejected", C.c_int32),
                ("t_final", C.c_double)]


class OdeDesc(C.Structure):
    _fields_ = [
        ("sde_kind", C.c_int32), ("N", C.c_int32), ("beta_0", C.c_double), ("beta_1", C.c_double), ("sigma_min", C.c_double),
        ("sigma_max", C.c_double), ("t0", C.c_double), ("t1", C.c_double), ("rtol", C.c_double), ("atol", C.c_double),
        ("max_nfe", C.c_int32), ("batch", C.c_int32), ("use_graph", C.c_int32), ("reserved", C.c_int32),
        ("classes_dev", C.c_void_p), ("state_dev", C.c_void_p), ("state_elems", C.c_int64), ("work_dev", C.c_void_p),
        ("work_bytes", C.c_size_t), ("result_dev", C.c_void_p),
    ]


HUTCH_RADEMACHER, HUTCH_GAUSSIAN = 0, 1


class OdeLikelihoodDesc(C.Structure):
    _fields_ = [
        ("sde_kind", C.c_int32), ("N", C.c_int32), ("beta_0", C.c_double), ("beta_1", C.c_double), ("sigma_min", C.c_double),
        ("sigma_max", C.c_double), ("t0", C.c_double), ("t1", C.c_double), ("rtol", C.c_double), ("atol", C.c_double),
        ("max_nfe", C.c_int32), ("batch", C.c_int32), ("use_graph", C.c_int32), ("hutchinson", C.c_int32), ("rng", Rng),
        ("noise_dev", C.c_void_p), ("classes_dev", C.c_void_p), ("state_dev", C.c_void_p), ("state_elems", C.c_int64),
        ("work_dev", C.c_void_p), ("work_bytes", C.c_size_t), ("result_dev", C.c_void_p),
    ]


class ConvArgs(C.Structure):
    _fields_ = [
        ("mode", C.c_int32), ("ksize", C.c_int32), ("batch", C.c_int32), ("cin", C.c_int32), ("cout", C.c_int32),
        ("hin", C.c_int32), ("win", C.c_int32), ("gn_groups", C.c_int32), ("silu", C.c_int32), ("out_groups", C.c_int32),
        ("act", C.c_int32), ("engine", C.c_int32),
        ("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("gn_gamma", C.c_void_p), ("gn_beta", C.c_void_p),
        ("temb", C.c_void_p), ("y", C.c_void_p), ("out_stats", C.c_void_p), ("scratch_dev", C.c_void_p),
        ("scratch_bytes", C.c_size_t),
    ]


class AttnBlockArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("dim", C.c_int32), ("n_tokens", C.c_int32), ("softmax", C.c_int32),
        ("x", C.c_void_p), ("norm_w", C.c_void_p), ("norm_b", C.c_void_p), ("w_qkv", C.c_void_p), ("w_out", C.c_void_p),
        ("b_out", C.c_void_p), ("out_norm_w", C.c_void_p), ("out_norm_b", C.c_void_p), ("y", C.c_void_p),
        ("scratch_dev", C.c_void_p), ("scratch_bytes", C.c_size_t),
    ]


class InitConvArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("cin", C.c_int32), ("size", C.c_int32), ("cout", C.c_int32), ("act", C.c_int32),
        ("engine", C.c_int32), ("pad_class", C.c_int32),
        ("x", C.c_void_p), ("w", C.c_void_p), ("bias", C.c_void_p), ("cls_w", C.c_void_p), ("classes", C.c_void_p),
        ("y", C.c_void_p), ("scratch_dev", C.c_void_p), ("scratch_bytes", C.c_size_t),
    ]


class GnFinalizeArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("channels", C.c_int32), ("hw", C.c_int32), ("groups", C.c_int32), ("ogroups", C.c_int32),
        ("silu", C.c_int32), ("act", C.c_int32),
        ("raw", C.c_void_p), ("res", C.c_void_p), ("stats", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
        ("y", C.c_void_p), ("out_stats", C.c_void_p), ("scratch_dev", C.c_void_p), ("scratch_bytes", C.c_size_t),
    ]


class FinalProjArgs(C.Structure):
    _fields_ = [
        ("batch", C.c_int32), ("channels", C.c_int32), ("hw", C.c_int32), ("cout", C.c_int32), ("groups", C.c_int32),
        ("plain", C.c_int32), ("act", C.c_int32),
        ("y", C.c_void_p), ("stats", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p), ("w", C.c_void_p),
        ("bias", C.c_void_p), ("eps", C.c_void_p), ("x", C.c_void_p), ("coef", C.c_void_p), ("z", C.c_void_p),
        ("step", C.c_int32), ("rng", Rng), ("x_out", C.c_void_p), ("scratch_dev", C.c_void_p), ("scratch_bytes", C.c_size_t),
    ]


# every symbol include/dmn_b200.h declares: (restype, argtypes)
_P, _I, _L, _F = C.c_void_p, C.c_int, C.c_int64, C.c_float
SYMBOLS = {
    "dmn_last_error": (C.c_char_p, []),
    "dmn_abi_version": (_I, []),
    "dmn_plan_create": (_I, [C.POINTER(UnetCfg), C.POINTER(_P)]),
    "dmn_plan_destroy": (None, [_P]),
    "dmn_plan_weights_bytes": (C.c_size_t, [_P]),
    "dmn_plan_workspace_bytes": (C.c_size_t, [_P]),
    "dmn_plan_bind": (_I, [_P, _P, C.c_size_t, _P, C.c_size_t]),
    "dmn_plan_num_params": (_I, [_P]),
    "dmn_plan_param_name": (C.c_char_p, [_P, _I]),
    "dmn_plan_param_shape": (_I, [_P, _I, C.POINTER(C.c_int64 * 4)]),
    "dmn_plan_load_param": (_I, [_P, C.c_char_p, _P, _L, _P]),
    "dmn_plan_load_freqs": (_I, [_P, _P, _I, _P]),
    "dmn_plan_ready": (_I, [_P]),
    "dmn_plan_film_layout": (_I, [_P, _P, _I]),
    "dmn_time_table": (_I, [_P, _P, _I, _I, _P]),
    "dmn_plan_time_table_info": (_I, [_P, C.POINTER(C.c_size_t), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dmn_plan_param_time_col": (_I, [_P, _I]),
    "dmn_plan_film_col": (_I, [_P, _I]),
    "dmn_unet_forward": (_I, [_P, _P, _P, _P, _P, _I, _P]),
    "dmn_unet_jvp": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, C.c_size_t, _I, _P]),
    "dmn_unet_jvp_work_bytes": (C.c_size_t, [_P, _I]),
    "dmn_plan_launches_per_forward": (_I, [_P]),
    "dmn_plan_num_ops": (_I, [_P]),
    "dmn_plan_op_info": (_I, [_P, _I, C.c_char_p, _I, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_double),
                              C.POINTER(C.c_double)]),
    "dmn_plan_profile_forward": (_I, [_P, _P, _P, _P, _P, _I, _P, _P, _I]),
    "dmn_plan_profile_forward_graph": (_I, [_P, _P, _P, _P, _P, _I, _P, _P, _I]),
    "dmn_ddpm_step": (_I, [_P, _P, _P, _P, _L, _P, _P, _I, Rng, _P]),
    "dmn_learned_step": (_I, [_P, _P, _P, _P, _I, _L, _P, _P, _I, Rng, _P]),
    "dmn_ddim_step": (_I, [_P, _P, _P, _P, _L, _P, _P, _I, Rng, _P]),
    "dmn_dpmpp_step": (_I, [_P, _P, _P, _P, _I, _L, _L, _P, _P, _I, _P]),
    "dmn_affine_noise_step": (_I, [_P, _P, _P, _P, _P, _L, _P, _P, _I, Rng, _P]),
    "dmn_langevin_step": (_I, [_P, _P, _P, _P, _P, _I, _L, _F, _P, _P, _I, _P, Rng, _P]),
    "dmn_bpd_qsample": (_I, [_P, _P, _P, _L, _P, _P, _I, Rng, _P]),
    "dmn_bpd_term": (_I, [_P, _P, _P, _P, _I, _L, _I, _I, _I, _P, _P, _P, _I, _P]),
    "dmn_unnormalize": (_I, [_P, _P, _L, _P]),
    "dmn_randn": (_I, [_P, _L, Rng, _I, _P]),
    "dmn_axpby": (_I, [_P, _P, _F, _F, _P, _L, _P]),
    "dmn_sample_loop": (_I, [_P, C.POINTER(LoopDesc), _P]),
    "dmn_loop_scratch_bytes": (C.c_size_t, [_P, C.POINTER(LoopDesc)]),
    "dmn_loop_launches_per_step": (_I, [_P, C.POINTER(LoopDesc)]),
    "dmn_inpaint_prepare": (_I, [_P, _P, _P, _P, _L, _P, _P, _I, Rng, _P]),
    "dmn_sample_loop_inpaint": (_I, [_P, C.POINTER(LoopDesc), C.POINTER(InpaintDesc), _P]),
    "dmn_ode_sample": (_I, [_P, C.POINTER(OdeDesc), _P]),
    "dmn_ode_work_bytes": (C.c_size_t, [_P, _I]),
    "dmn_ode_likelihood": (_I, [_P, C.POINTER(OdeLikelihoodDesc), _P]),
    "dmn_ode_likelihood_work_bytes": (C.c_size_t, [_P, _I]),
    "dmn_conv_forward": (_I, [C.POINTER(ConvArgs), _P]),
    "dmn_conv_scratch_bytes": (C.c_size_t, [C.POINTER(ConvArgs)]),
    "dmn_conv_forward_cat": (_I, [C.POINTER(ConvArgs), _P, C.c_int32, _P]),
    "dmn_linear_attention_core": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, C.c_size_t, _P]),
    "dmn_attention_core": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, C.c_size_t, _P]),
    "dmn_selftest_umma_gemm": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "dmn_selftest_tma_sw128_gemm": (_I, [_P, _P, _P, _I, _I, _I, _P]),
    "dmn_linear_attention_block": (_I, [C.POINTER(AttnBlockArgs), _P]),
    "dmn_linear_attention_block_scratch_bytes": (C.c_size_t, [C.POINTER(AttnBlockArgs)]),
    "dmn_init_conv_forward": (_I, [C.POINTER(InitConvArgs), _P]),
    "dmn_init_conv_scratch_bytes": (C.c_size_t, [C.POINTER(InitConvArgs)]),
    "dmn_gn_finalize_forward": (_I, [C.POINTER(GnFinalizeArgs), _P]),
    "dmn_gn_finalize_scratch_bytes": (C.c_size_t, [C.POINTER(GnFinalizeArgs)]),
    "dmn_final_proj_forward": (_I, [C.POINTER(FinalProjArgs), _P]),
    "dmn_final_proj_scratch_bytes": (C.c_size_t, [C.POINTER(FinalProjArgs)]),
}

_lib = None


class DmnError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raises if the native library is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DmnError(
                f"{LIB_PATH} is missing: build it with `python -m diffusion_model_nemo_b200._build` "
                "(nvcc, sm_100a).  There is no CPU / PyTorch fallback."
            )
        h = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(h, name)
            fn.restype = res
            fn.argtypes = args
        if h.dmn_abi_version() != 1:
            raise DmnError("libdmn_b200.so ABI version mismatch")
        _lib = h
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().dmn_last_error().decode("utf-8", "replace")
        exc = {-1: ValueError, -2: NotImplementedError}.get(rc, DmnError)
        raise exc(f"{what or 'libdmn_b200'} failed (rc={rc}): {msg}")


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device=None):
    import torch

    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)
