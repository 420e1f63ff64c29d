"""ctypes binding of libtcs.so (include/tcs.h).  There is NO fallback: if the shared library is
missing or no B200 is present, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtcs.so")

TCS_OK, ERR_BAD_ARGUMENT, ERR_UNSUPPORTED, ERR_CUDA, ERR_STATE = 0, -1, -2, -3, -4
FP32, BF16 = 0, 1
ENGINE_AUTO, ENGINE_SIMT, ENGINE_TCGEN05 = 0, 1, 2
SAMPLER_ODE, SAMPLER_SDE, SAMPLER_DPMPP_2M = 0, 1, 2


class TcsConfig(C.Structure):
    _fields_ = [("n_types", C.c_int32), ("y_cont_dim", C.c_int32), ("base_ch", C.c_int32), ("emb_dim", C.c_int32),
                ("cond_ch", C.c_int32), ("time_ch", C.c_int32), ("beta_min", C.c_double), ("beta_max", C.c_double),
                ("precision", C.c_int32), ("engine", C.c_int32), ("device", C.c_int32), ("chunk", C.c_int32),
                ("use_graph", C.c_int32), ("fuse_gn", C.c_int32)]


class TcsSampleArgs(C.Structure):
    _fields_ = [("sampler", C.c_int32), ("n", C.c_int32), ("steps", C.c_int32), ("guidance", C.c_float),
                ("t_end", C.c_double), ("y_cat", C.c_void_p), ("y_cont", C.c_void_p), ("x_init", C.c_void_p),
                ("noise", C.c_void_p), ("seed", C.c_uint64), ("global_index_offset", C.c_uint64),
                ("x_out", C.c_void_p), ("trace_eps", C.c_void_p), ("trace_x", C.c_void_p), ("x0_hat", C.c_void_p),
                ("beta_min", C.c_double), ("beta_max", C.c_double)]


class TcsPriorConfig(C.Structure):
    _fields_ = [("z_dim", C.c_int32), ("n_types", C.c_int32), ("y_cont_dim", C.c_int32), ("t_emb_dim", C.c_int32),
                ("width", C.c_int32), ("n_blocks", C.c_int32), ("y_cat_emb_dim", C.c_int32), ("T", C.c_int32),
                ("beta_start", C.c_double), ("beta_end", C.c_double), ("precision", C.c_int32), ("device", C.c_int32),
                ("use_graph", C.c_int32)]


class TcsDdimArgs(C.Structure):
    _fields_ = [("n", C.c_int32), ("n_steps", C.c_int32), ("y_cat", C.c_void_p), ("y_cont", C.c_void_p),
                ("z_init", C.c_void_p), ("seed", C.c_uint64), ("global_index_offset", C.c_uint64),
                ("z0_out", C.c_void_p), ("trace_eps", C.c_void_p), ("trace_z", C.c_void_p)]


class TcsVaeConfig(C.Structure):
    _fields_ = [("z_dim", C.c_int32), ("n_types", C.c_int32), ("y_cont_dim", C.c_int32), ("device", C.c_int32),
                ("precision", C.c_int32)]


# every symbol include/tcs.h and include/tcs_prior.h declare: name -> (restype, argtypes)
SIGNATURES = {
    "tcs_default_config": (None, [C.POINTER(TcsConfig)]),
    "tcs_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(TcsConfig)]),
    "tcs_destroy": (None, [C.c_void_p]),
    "tcs_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "tcs_finalize_weights": (C.c_int, [C.c_void_p]),
    "tcs_score": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                            C.c_void_p, C.c_void_p]),
    "tcs_sample": (C.c_int, [C.c_void_p, C.POINTER(TcsSampleArgs), C.c_void_p]),
    "tcs_nfe": (C.c_int32, [C.c_int32, C.c_int32]),
    "tcs_condition_grid": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_float, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "tcs_sde_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float, C.c_float,
                                 C.c_uint64, C.c_uint64, C.c_int32, C.c_void_p]),
    "tcs_ode_update": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                 C.c_float, C.c_float, C.c_void_p]),
    "tcs_dpm_update": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32] + [C.c_float] * 6
                       + [C.c_void_p]),
    "tcs_time_grid_host": (C.c_int, [C.c_int32, C.c_double, C.POINTER(C.c_float)]),
    "tcs_dpm_schedule_host": (C.c_int, [C.c_int32, C.c_double, C.c_double, C.c_double, C.POINTER(C.c_float),
                                        C.POINTER(C.c_float)]),
    "tcs_schedule_host": (C.c_int, [C.c_double, C.c_double, C.c_float, C.POINTER(C.c_float), C.POINTER(C.c_float),
                                    C.POINTER(C.c_float)]),
    "tcs_launch_count": (C.c_int64, [C.c_void_p]),
    "tcs_check": (C.c_int32, [C.c_void_p]),
    "tcs_launch_mode": (C.c_int32, [C.c_void_p]),
    "tcs_build_info": (C.c_char_p, []),
    "tcs_last_error": (C.c_char_p, []),
    "tcs_debug_layer": (C.c_int64, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                    C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]),
    "tcs_score_profiled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_float,
                                     C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_float), C.c_void_p]),
    # ---- include/tcs_prior.h ----
    "tcs_prior_default_config": (None, [C.POINTER(TcsPriorConfig)]),
    "tcs_prior_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(TcsPriorConfig)]),
    "tcs_prior_destroy": (None, [C.c_void_p]),
    "tcs_prior_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "tcs_prior_finalize_weights": (C.c_int, [C.c_void_p]),
    "tcs_prior_eps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                C.c_void_p]),
    "tcs_prior_ddim_sample": (C.c_int, [C.c_void_p, C.POINTER(TcsDdimArgs), C.c_void_p]),
    "tcs_prior_schedule_host": (C.c_int, [C.c_int32, C.c_double, C.c_double, C.POINTER(C.c_float)]),
    "tcs_prior_timesteps_host": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "tcs_prior_launch_count": (C.c_int64, [C.c_void_p]),
    "tcs_vae_create": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(TcsVaeConfig)]),
    "tcs_vae_destroy": (None, [C.c_void_p]),
    "tcs_vae_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "tcs_vae_finalize_weights": (C.c_int, [C.c_void_p]),
    "tcs_vae_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    "tcs_vae_launch_count": (C.c_int64, [C.c_void_p]),
    "tcs_prior_profile": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    "tcs_debug_linear": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "tcs_debug_conv": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "tcs_debug_attn_block": (C.c_int, [C.c_int32] + [C.c_void_p] * 10),
    "tcs_debug_conv_ups": (C.c_int, [C.c_int32] * 5 + [C.c_void_p] * 5),
    "tcs_debug_attn_pack": (C.c_int64, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
}

_lib: Optional[C.CDLL] = None


class TcsError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load libtcs.so (once).  Raises if it was not built — run __graft_entry__.build()."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise TcsError(f"{LIB_PATH} is missing: build it with `python __graft_entry__.py build` "
                           "(toycrystals_b200 has no CPU or PyTorch fallback)")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError here == header/library mismatch
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def last_error() -> str:
    return (lib().tcs_last_error() or b"").decode()


def check(status: int) -> None:
    """Map tcs_status to the exceptions the reference raises at the same places."""
    if status == TCS_OK:
        return
    msg = last_error()
    if status == ERR_BAD_ARGUMENT:
        raise ValueError(msg)
    if status == ERR_UNSUPPORTED:
        raise NotImplementedError(msg)
    raise TcsError(f"libtcs error {status}: {msg}")
