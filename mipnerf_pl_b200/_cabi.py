"""ctypes binding of libmipnerf_b200.so (include/mipnerf_b200.h).

The library is the product; this file only marshals pointers.  If the shared
object is missing the import of the ops fails loudly — there is no CPU or
PyTorch fallback behind it.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_NAME = "libmipnerf_b200.so"
LIB_PATH = os.environ.get("MIPNERF_B200_LIB") or os.path.join(_HERE, LIB_NAME)  # env: experiment builds

ABI_VERSION = 4
OK, EINVAL, EUNSUPPORTED, ECUDA, EWORKSPACE = 0, -1, -2, -3, -4
FP32, BF16, FP16, FP16X3, BF16X3 = 0, 1, 2, 3, 4
PRECISIONS = {"fp32": FP32, "bf16": BF16, "fp16": FP16, "fp16x3": FP16X3, "bf16x3": BF16X3}

_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)


class Linear(C.Structure):
    _fields_ = [("weight", C.c_void_p), ("bias", C.c_void_p),
                ("in_features", C.c_int32), ("out_features", C.c_int32)]


class Config(C.Structure):
    _fields_ = [("num_samples", C.c_int32), ("num_levels", C.c_int32),
                ("min_deg_point", C.c_int32), ("max_deg_point", C.c_int32), ("deg_view", C.c_int32),
                ("use_viewdirs", C.c_int32), ("disparity", C.c_int32), ("disable_integration", C.c_int32),
                ("resample_padding", C.c_float), ("density_bias", C.c_float), ("rgb_padding", C.c_float),
                ("net_depth", C.c_int32), ("net_width", C.c_int32), ("net_depth_condition", C.c_int32),
                ("net_width_condition", C.c_int32), ("skip_index", C.c_int32),
                ("num_rgb_channels", C.c_int32), ("num_density_channels", C.c_int32),
                ("density_noise", C.c_float)]


class Weights(C.Structure):
    _fields_ = [("linears", C.POINTER(Linear)), ("num_linears", C.c_int32),
                ("packed_precision", C.c_int32), ("packed", C.c_void_p), ("packed_bytes", C.c_size_t)]


class RaysStruct(C.Structure):
    _fields_ = [("origins", C.c_void_p), ("directions", C.c_void_p), ("viewdirs", C.c_void_p),
                ("radii", C.c_void_p), ("near", C.c_void_p), ("far", C.c_void_p), ("num_rays", C.c_int64)]


class LevelOut(C.Structure):
    _fields_ = [("comp_rgb", C.c_void_p), ("distance", C.c_void_p), ("acc", C.c_void_p),
                ("weights", C.c_void_p), ("t_samples", C.c_void_p), ("inds", C.c_void_p),
                ("density_normal", C.c_void_p)]  # INPUT: [B,N] normals of the density noise (models/mip_nerf.py:233)


class Rng(C.Structure):
    _fields_ = [("seed", C.c_uint64), ("offset", C.c_uint64)]


class LinearGrad(C.Structure):
    _fields_ = [("weight_grad", C.c_void_p), ("bias_grad", C.c_void_p)]


class Loss(C.Structure):
    _fields_ = [("target_rgb", C.c_void_p), ("lossmult", C.c_void_p), ("mask_sum", C.c_void_p),
                ("dist_scale", C.c_float), ("level_mse_mult", C.POINTER(C.c_float)),
                ("level_dist_mult", C.POINTER(C.c_float)), ("per_ray_sqerr", C.c_void_p),
                ("per_ray_distloss", C.c_void_p)]


# name -> (restype, argtypes); every symbol include/mipnerf_b200.h declares.
_V = C.c_void_p
_SIGNATURES = {
    "mipnerf_b200_last_error": (C.c_char_p, []),
    "mipnerf_b200_abi_version": (C.c_int, []),
    "mipnerf_b200_workspace_bytes": (C.c_size_t, [C.POINTER(Config), C.c_int64, C.c_int]),
    "mipnerf_b200_packed_weights_bytes": (C.c_size_t, [C.POINTER(Config), C.c_int]),
    "mipnerf_b200_pack_weights": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), C.c_int, _V, C.c_size_t, _V]),
    "mipnerf_b200_forward": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), C.POINTER(RaysStruct), C.c_int,
                                       _V, _V, C.c_int, C.c_int, C.POINTER(LevelOut), _V, C.c_size_t, _V]),
    "mipnerf_b200_forward_rng": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), C.POINTER(RaysStruct), C.POINTER(Rng),
                                           C.c_int, C.c_int, C.POINTER(LevelOut), _V, C.c_size_t, _V]),
    "mipnerf_b200_philox_uniform": (C.c_int, [C.POINTER(Rng), C.c_int, C.c_int64, C.c_int, _V, _V]),
    "mipnerf_b200_philox_normal": (C.c_int, [C.POINTER(Rng), C.c_int, C.c_int64, C.c_int, _V, _V]),
    "mipnerf_b200_distloss": (C.c_int, [_V, _V, C.c_int64, C.c_int, _V, _V]),
    "mipnerf_b200_train_workspace_bytes": (C.c_size_t, [C.POINTER(Config), C.c_int64]),
    "mipnerf_b200_forward_backward": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), C.POINTER(RaysStruct), C.c_int,
                                                _V, _V, C.c_int, C.c_int, C.POINTER(Loss), C.POINTER(LevelOut),
                                                C.POINTER(LinearGrad), C.c_int, C.c_int, _V, C.c_size_t, _V]),
    "mipnerf_b200_forward_backward_rng": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), C.POINTER(RaysStruct),
                                                    C.POINTER(Rng), C.c_int, C.c_int, C.POINTER(Loss), C.POINTER(LevelOut),
                                                    C.POINTER(LinearGrad), C.c_int, C.c_int, _V, C.c_size_t, _V]),
    "mipnerf_b200_forward_backward_rng_state": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), C.POINTER(RaysStruct),
                                                          _V, C.c_int, C.c_int, C.POINTER(Loss), C.POINTER(LevelOut),
                                                          C.POINTER(LinearGrad), C.c_int, C.c_int, _V, C.c_size_t, _V]),
    "mipnerf_b200_linear_tc": (C.c_int, [_V, _V, _V, _V, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, _V, C.c_size_t, _V]),
    "mipnerf_b200_wgrad_tc_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "mipnerf_b200_wgrad_tc": (C.c_int, [_V, C.c_int, _V, C.c_int, _V, C.c_int, C.c_int, C.c_int64, _V, _V, C.c_int, _V,
                                        C.c_size_t, _V]),
    "mipnerf_b200_adam_step": (C.c_int, [_V, _V, _V, _V, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double,
                                         C.c_int64, C.c_double, _V]),
    "mipnerf_b200_adam_step_multi": (C.c_int, [C.c_int, _V, _V, _V, _V, _V, C.c_double, C.c_double, C.c_double,
                                               C.c_double, C.c_int64, C.c_double, _V]),
    "mipnerf_b200_adam_step_multi_table": (C.c_int, [C.c_int, _V, _V, _V, _V, _V, _V, _V, C.c_int64, _V, C.c_double,
                                                     C.c_double, C.c_double, C.c_double, _V]),
    "mipnerf_b200_train_step_advance": (C.c_int, [_V, _V, _V, _V, _V, C.c_int, _V]),
    "mipnerf_b200_generate_rays": (C.c_int, [_f32p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int,
                                             _V, _V, _V, _V, _V, _V, _V]),
    "mipnerf_b200_image_metrics_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "mipnerf_b200_image_metrics": (C.c_int, [_V, _V, C.c_int, C.c_int, C.c_int, _V, C.c_size_t, _V, _V]),
    "mipnerf_b200_rays_from_pixels": (C.c_int, [_V, _V, _V, C.c_int, _V, C.c_int64, _V, _V, _V, _V, _V, _V, _V, _V, _V, _V]),
    "mipnerf_b200_sample_pixels": (C.c_int, [_V, _V, _V, C.c_int, C.c_int64, _V, C.c_int64, C.c_int64, _V, _V, _V, _V,
                                             _V, _V, _V, _V, _V, _V, _V]),
    "mipnerf_b200_sample_along_rays": (C.c_int, [C.POINTER(RaysStruct), C.c_int, C.c_int, C.c_int, _V, _V, _V, _V, _V]),
    "mipnerf_b200_cast_rays": (C.c_int, [C.POINTER(RaysStruct), _V, C.c_int, _V, _V, _V]),
    "mipnerf_b200_integrated_pos_enc": (C.c_int, [_V, _V, C.c_int64, C.c_int, C.c_int, _V, _V]),
    "mipnerf_b200_pos_enc": (C.c_int, [_V, C.c_int64, C.c_int, C.c_int, C.c_int, _V, _V]),
    "mipnerf_b200_mlp_forward": (C.c_int, [C.POINTER(Config), C.POINTER(Weights), _V, _V, C.c_int64, C.c_int,
                                           C.c_int, _V, _V, _V, C.c_size_t, _V]),
    "mipnerf_b200_mlp_workspace_bytes": (C.c_size_t, [C.POINTER(Config), C.c_int64, C.c_int, C.c_int]),
    "mipnerf_b200_volumetric_rendering": (C.c_int, [_V, _V, _V, _V, C.c_int64, C.c_int, C.c_int, _V, _V, _V, _V, _V]),
    "mipnerf_b200_sorted_piecewise_constant_pdf": (C.c_int, [_V, _V, C.c_int64, C.c_int, C.c_int, C.c_int, _V, _V, _V, _V]),
    "mipnerf_b200_resample_along_rays": (C.c_int, [C.POINTER(RaysStruct), _V, _V, C.c_int, C.c_int, _V, C.c_float,
                                                   _V, _V, _V, _V, _V]),
    "mipnerf_b200_selftest_umma": (C.c_int, [_V, _V, _V, C.c_int, C.c_int, C.c_int, C.c_int, _V, C.c_size_t, _V]),
    "mipnerf_b200_selftest_umma_rate": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _V, _V]),
    "mipnerf_b200_selftest_umma_rate_pair": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _V, _V]),
    "mipnerf_b200_profile_enable": (C.c_int, [C.c_int]),
    "mipnerf_b200_profile_num_kernels": (C.c_int, []),
    "mipnerf_b200_profile_kernel_name": (C.c_char_p, [C.c_int]),
    "mipnerf_b200_profile_read": (C.c_int, [C.c_int, _i64p, C.POINTER(C.c_double), _i64p, C.c_int]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib: Optional[C.CDLL] = None


class NativeLibraryMissing(ImportError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the shared library; raise if it is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} is not built. Run `python -c 'import __graft_entry__ as g; g.build()'` "
                f"(or `python -m mipnerf_pl_b200.build`). There is no CPU fallback for this path.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if handle.mipnerf_b200_abi_version() != ABI_VERSION:
            raise ImportError("libmipnerf_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def last_error() -> str:
    return lib().mipnerf_b200_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    """Turn a C-ABI status into the exception the reference would raise."""
    if rc == OK:
        return
    msg = f"{what}: {last_error()}"
    if rc == EUNSUPPORTED:
        raise NotImplementedError(msg)  # reference raises NotImplementedError for unsupported modes
    if rc == EINVAL:
        raise ValueError(msg)
    raise RuntimeError(msg)


def profile_snapshot(reset: bool = False) -> dict:
    """{kernel name: (launches, timed_ms, timed_launches)} from the library's launch accounting."""
    l = lib()
    out = {}
    for k in range(l.mipnerf_b200_profile_num_kernels()):
        n, ms, tn = C.c_int64(0), C.c_double(0.0), C.c_int64(0)
        l.mipnerf_b200_profile_read(k, C.byref(n), C.byref(ms), C.byref(tn), int(reset))
        out[l.mipnerf_b200_profile_kernel_name(k).decode()] = (n.value, ms.value, tn.value)
    return out
