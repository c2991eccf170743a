"""ctypes binding of the C-ABI in include/skyrim_b200.h (libskyrim_b200.so, built in-tree by
``__graft_entry__.build()`` / ``make -C skyrim_b200/csrc``).

There is deliberately no fallback: if the shared library is missing or no sm_100 device is
visible, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "libskyrim_b200.so"
# development build (-DSKY_EXPERIMENTS: CUDA-core reference GEMM, single-CTA kernel variants, timing-experiment
# switches).  Never loaded unless a test asks for it with lib("dev") / SKYRIM_B200_LIB=dev.
DEV_LIB_PATH = Path(__file__).resolve().parent / "libskyrim_b200_dev.so"

SKY_MODEL_PANGU6 = 1
SKY_MODEL_SFNO73 = 2
SKY_MODEL_GRAPHCAST = 3
SKY_MODEL_AFNO26 = 4


class SkyError(RuntimeError):
    pass


class PanguConfigC(C.Structure):
    _fields_ = [("nlat", C.c_int32), ("nlon", C.c_int32), ("n_levels", C.c_int32), ("dim", C.c_int32),
                ("depths", C.c_int32 * 4), ("heads", C.c_int32 * 4), ("ln_eps", C.c_float),
                ("mask_value", C.c_float)]


class SFNOConfigC(C.Structure):
    _fields_ = [("nlat", C.c_int32), ("nlon", C.c_int32), ("n_channels", C.c_int32), ("embed", C.c_int32),
                ("layers", C.c_int32), ("scale_factor", C.c_int32), ("mlp_ratio", C.c_int32),
                ("eps", C.c_float)]


class GraphCastConfigC(C.Structure):
    _fields_ = [("nlat", C.c_int32), ("nlon", C.c_int32), ("n_mesh", C.c_int32), ("n_mesh_edges", C.c_int32),
                ("n_g2m_edges", C.c_int32), ("latent", C.c_int32), ("layers", C.c_int32), ("n_state", C.c_int32),
                ("n_prog", C.c_int32), ("n_static", C.c_int32), ("dt_hours", C.c_int32), ("ln_eps", C.c_float)]


class AFNOConfigC(C.Structure):
    _fields_ = [("nlat", C.c_int32), ("nlon", C.c_int32), ("n_channels", C.c_int32), ("patch", C.c_int32),
                ("embed", C.c_int32), ("depth", C.c_int32), ("num_blocks", C.c_int32), ("mlp_ratio", C.c_int32),
                ("sparsity", C.c_float), ("hard_thresholding_fraction", C.c_float), ("ln_eps", C.c_float)]


class ParamDesc(C.Structure):
    _fields_ = [("name", C.c_char * 96), ("offset", C.c_uint64), ("count", C.c_uint64)]


EXPORTS = {
    "sky_abi_version": (C.c_int, []),
    "sky_last_error": (C.c_char_p, []),
    "sky_model_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_void_p, C.c_size_t, C.c_int]),
    "sky_model_load_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.POINTER(ParamDesc), C.c_int32,
                                         C.c_int32, C.c_void_p]),
    "sky_model_workspace_bytes": (C.c_size_t, [C.c_void_p, C.c_int32]),
    "sky_model_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t,
                                 C.c_void_p]),
    "sky_model_set_clock": (C.c_int, [C.c_void_p, C.c_double, C.c_void_p]),
    "sky_toa_radiation": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_void_p]),
    "sky_model_debug_copy": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_int32,
                                       C.c_void_p]),
    "sky_model_debug_set": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "sky_perturb_ic": (C.c_int, [C.c_void_p, C.c_void_p, C.c_float, C.c_uint64, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int64, C.c_void_p]),
    "sky_model_profile_begin": (C.c_int, [C.c_void_p, C.c_uint64]),
    "sky_model_profile_end": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int32]),
    "sky_profile_tag_count": (C.c_int, []),
    "sky_profile_tag_name": (C.c_char_p, [C.c_int32]),
    "sky_launch_count": (C.c_uint64, []),
    "sky_model_destroy": (C.c_int, [C.c_void_p]),
}

_libs = {}


def lib(variant: str | None = None) -> C.CDLL:
    """The product library (default) or, for tests that bisect against the reference kernels, the dev build."""
    variant = variant or os.environ.get("SKYRIM_B200_LIB", "prod")
    if variant not in _libs:
        path = DEV_LIB_PATH if variant == "dev" else LIB_PATH
        if not path.exists():
            raise SkyError(f"{path} not found — build it with `python -c 'import __graft_entry__ as g; "
                           f"g.build()'` (there is no CPU fallback)")
        L = C.CDLL(os.fspath(path))
        for name, (res, args) in EXPORTS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _libs[variant] = L
    return _libs[variant]


def check(rc: int, what: str = "", L=None):
    if rc != 0:
        msg = (L or lib()).sky_last_error()
        raise SkyError(f"{what} failed (rc={rc}): {msg.decode() if msg else '?'}")
