"""ctypes binding of libdtraj.so (include/dtraj.h).

There is deliberately NO fallback: if the CUDA library is missing or a call fails the
caller gets an exception.  The library is built in-tree by
``python -m distillation_trajectories_b200.build`` (or ``__graft_entry__.build()``).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# DTRAJ_LIB=<path>: load that build of the library instead (A/B timing of two builds inside one GPU job, tools/ab.sh; the driver's
# "which .so was loaded" record then shows that file)
LIB_PATH = os.environ.get("DTRAJ_LIB") or os.path.join(_HERE, "csrc", "libdtraj.so")

PREC_FP32, PREC_TF32, PREC_TF32X3, PREC_F16 = 0, 1, 2, 3
VAR_NONE, VAR_COND0, VAR_COND1 = 0, 1, 2
RULE_S1, RULE_S2, RULE_S3 = 1, 2, 3
METRIC_Q = 6
METRIC_Q_RAGGED = 8

PRECISIONS = {"fp32": PREC_FP32, "tf32": PREC_TF32, "tf32x3": PREC_TF32X3, "f16": PREC_F16}


class DtrajError(RuntimeError):
    pass


class UNetDesc(C.Structure):
    _fields_ = [("channels", C.c_int32), ("image_size", C.c_int32), ("dims", C.c_int32 * 4),
                ("temb_dim", C.c_int32), ("n_timesteps", C.c_int32), ("precision", C.c_int32)]


class SamplerDesc(C.Structure):
    _fields_ = [("rule", C.c_int32), ("n_samples", C.c_int32), ("n_rows", C.c_int32),
                ("n_updates", C.c_int32), ("copy_last", C.c_int32), ("n_frames", C.c_int32),
                ("use_graph", C.c_int32), ("n_rows0", C.c_int32),
                ("step_timestep", C.c_void_p), ("step_coef", C.c_void_p),
                ("row_sample", C.c_void_p), ("row_variant", C.c_void_p),
                ("sample_row_u", C.c_void_p), ("sample_row_c", C.c_void_p),
                ("guidance", C.c_void_p), ("z_bank", C.c_void_p), ("z_index", C.c_void_p),
                ("traj", C.c_void_p), ("workspace", C.c_void_p), ("workspace_bytes", C.c_int64),
                ("row_sample0", C.c_void_p), ("row_variant0", C.c_void_p),
                ("sample_row_u0", C.c_void_p), ("sample_row_c0", C.c_void_p)]


# every symbol include/dtraj.h declares: name -> (restype, argtypes)
_P, _I32, _I64 = C.c_void_p, C.c_int32, C.c_int64
SIGNATURES = {
    "dtraj_last_error": (C.c_char_p, []),
    "dtraj_version": (C.c_int, []),
    "dtraj_unet_create": (C.c_int, [C.POINTER(UNetDesc), C.POINTER(C.c_char_p), C.POINTER(_P),
                                    C.POINTER(_I64), _I32, C.POINTER(_P)]),
    "dtraj_unet_destroy": (C.c_int, [_P]),
    "dtraj_unet_workspace_bytes": (_I64, [_P, _I64]),
    "dtraj_unet_time_bias": (C.c_int, [_P, _I32, _I32, _I32, _P, _I32]),
    "dtraj_unet_forward": (C.c_int, [_P, _P, _I64, _I32, _P, _P, _P, _I64, _P]),
    "dtraj_step_fused": (C.c_int, [_I32, _P, _P, _P, _P, _P, _I64, _P, _I64, _P, _I64, _I64, _I64, _P]),
    "dtraj_sampler_create": (C.c_int, [_P, C.POINTER(SamplerDesc), C.POINTER(_P)]),
    "dtraj_sampler_run": (C.c_int, [_P, _P]),
    "dtraj_sampler_destroy": (C.c_int, [_P]),
    "dtraj_sampler_launches": (_I64, [_P]),
    "dtraj_sampler_profile": (C.c_int, [_P, _P, C.POINTER(C.c_double), C.POINTER(_I64), C.POINTER(C.c_double)]),
    "dtraj_metrics_pairs": (C.c_int, [_P, _P, _I64, _I32, _I32, _P, _P]),
    "dtraj_wasserstein": (C.c_int, [_P, _P, _I64, _I32, _I32, _P, _P, _I32, _P, _P]),
    "dtraj_metrics_pairs_ragged": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P, _P, _P, _P]),
    "dtraj_wasserstein_ragged": (C.c_int, [_P, _P, _I64, _I32, _I32, _I32, _P, _P, _I32, _P, _P]),
    "dtraj_unet_forward_rows":(C.c_int, [_P, _P, _I64, _P, _P, _P, _I64, _P]),
    "dtraj_numpy_choice_sets": (C.c_int, [_P, _I32, _I32, _I32, _I32, _P, _P]),
    "dtraj_project": (C.c_int, [_P, _I64, _I32, _P, _P, _I32, _P, _P]),
    "dtraj_sampler_flops": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "dtraj_sampler_profile_text": (C.c_int, [_P, _P, _I32, C.c_char_p, _I64]),
    "dtraj_unet_check_errors": (C.c_int, [_P]),
    "dtraj_unet_error_flag_async": (C.c_int, [_P, _P, _P]),
    "dtraj_check_errors": (C.c_int, []),
    "dtraj_error_flag_async": (C.c_int, [_P, _P]),
    "dtraj_bench_conv": (C.c_int, [_I32, _I32, _I32, _I32, _I64, _I32, _I32, _I32, _I32, _I32, C.POINTER(C.c_float)]),
    "dtraj_debug_umma_error": (C.c_uint, []),
    "dtraj_test_conv": (C.c_int, [_I32, _P, _I32, _P, _I32, _I64, _I32, _I32, _P, _P, _I32, _I32, _I32,
                                  _P, _P, _P]),
}

_lib = None


def load():
    """Load libdtraj.so (never builds implicitly, never falls back)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DtrajError(
            f"{LIB_PATH} not found: the CUDA library has not been built. Run "
            "`python -m distillation_trajectories_b200.build` (needs nvcc); there is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)       # AttributeError if the .so is stale / incomplete
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().dtraj_last_error()
        raise DtrajError(f"libdtraj error {rc}: {msg.decode() if msg else '?'}")


def ptr(t):
    """data_ptr of a torch tensor (or None) as c_void_p."""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
