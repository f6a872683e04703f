"""ctypes binding of libmarigold_b200.so (the C ABI in include/marigold_b200.h).

The product path has no CPU fallback: if the shared library is missing and cannot be built, or a
call returns a non-zero status, this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
_LIB_PATH = _PKG / "libmarigold_b200.so"
_lib = None


class MgbError(RuntimeError):
    pass


class mgb_config(C.Structure):
    _fields_ = [
        ("unet_in_channels", C.c_int32),
        ("unet_out_channels", C.c_int32),
        ("unet_block_channels", C.c_int32 * 4),
        ("unet_layers_per_block", C.c_int32),
        ("unet_cross_dim", C.c_int32),
        ("vae_block_channels", C.c_int32 * 4),
        ("vae_layers_per_block", C.c_int32),
        ("vae_latent_channels", C.c_int32),
        ("norm_groups", C.c_int32),
        ("latent_scale", C.c_float),
    ]


# epilogue flags (kernels.h)
EPI_GEGLU, EPI_SCHED, EPI_DEPTH, EPI_NORMALS, EPI_NCHW, EPI_SILU, EPI_SCALE, EPI_UNIT = 1, 2, 4, 8, 16, 32, 64, 128

_vp, _i32, _i64, _f32, _f64 = C.c_void_p, C.c_int32, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); every symbol include/marigold_b200.h declares
SIGNATURES = {
    "mgb_create": (_i32, [C.POINTER(mgb_config), C.POINTER(_vp)]),
    "mgb_destroy": (None, [_vp]),
    "mgb_last_error": (C.c_char_p, []),
    "mgb_build_info": (C.c_char_p, []),
    "mgb_load_tensor": (_i32, [_vp, C.c_char_p, _vp, C.POINTER(_i64), _i32, _i32]),
    "mgb_finalize_weights": (_i32, [_vp]),
    "mgb_set_text_embedding": (_i32, [_vp, _vp, _i32]),
    "mgb_set_schedule": (_i32, [_vp, _i32, _vp, _vp, _vp, _vp]),
    "mgb_encode": (_i32, [_vp, _vp, _i32, _i32, _i32, _vp, _vp]),
    "mgb_unet_step": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "mgb_denoise": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _vp]),
    "mgb_denoise_range": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "mgb_decode": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "mgb_ens_depth_cost": (_i32, [_vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _f64, C.POINTER(_f64), _vp]),
    "mgb_ens_depth_cost_batch": (_i32, [_vp, _vp, _vp, _i32, _i32, _i64, _i32, _i32, _i32, _f64, _vp, _vp]),
    "mgb_ens_depth_cost_fd": (_i32, [_vp, _vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _f64, _vp, _vp]),
    "mgb_ens_max_members": (_i32, []),
    "mgb_ens_minmax": (_i32, [_vp, _vp, _i32, _i64, _vp, _vp, _vp]),
    "mgb_ens_depth_reduce": (_i32, [_vp, _vp, _vp, _i32, _i64, _i32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "mgb_ens_iid": (_i32, [_vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp]),
    "mgb_ens_normals": (_i32, [_vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp]),
    "mgb_resize": (_i32, [_vp, _i32, _i32, _i32, _i32, _vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "mgb_colorize": (_i32, [_vp, _i64, _f32, _f32, _vp, _vp, _vp]),
    "mgb_eval_ws_bytes": (C.c_size_t, []),
    "mgb_eval_depth": (_i32, [_vp, _vp, _vp, _i64, _i32, _f32, _f32, _vp, _vp, _vp, _vp]),
    "mgb_eval_normals": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    "mgb_eval_iid": (_i32, [_vp, _vp, _vp, _i64, _i32, _i32, _vp, _vp, _vp]),
    "mgb_workspace_bytes": (C.c_size_t, [_vp, _i32, _i32, _i32]),
    "mgb_launch_count": (_i64, []),
    "mgb_op_linear": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "mgb_op_conv2d": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32,
                              _i32, _vp, _vp]),
    "mgb_op_flash_attn64": (_i32, [_vp, _vp, _i32, _i32, _i32, _f32, _vp]),
    "mgb_op_groupnorm_ws_bytes": (C.c_size_t, [_i32, _i32, _i32, _i32]),
    "mgb_op_xattn2": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f32, _f32, _vp]),
    "mgb_op_groupnorm": (_i32, [_vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _f32, _i32, _vp]),
    "mgb_op_layernorm": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _f32, _vp]),
    "mgb_op_space_to_depth": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "mgb_op_upsample2x": (_i32, [_vp, _vp, _i32, _i32, _i32, _i32, _vp]),
}


def _stale() -> bool:
    try:
        t = _LIB_PATH.stat().st_mtime
        srcs = list((_PKG / "csrc").glob("*.cu")) + list((_PKG / "csrc").glob("*.h")) + list((_PKG / "csrc").glob("*.cuh"))
        return any(p.stat().st_mtime > t for p in srcs)
    except OSError:
        return False


def lib_path() -> Path:
    return _LIB_PATH


def load(build_if_missing: bool = True):
    """Load (building first if needed). Raises MgbError when the library is unavailable."""
    global _lib
    if _lib is not None:
        return _lib
    if not _LIB_PATH.exists():
        if not build_if_missing:
            raise MgbError(f"{_LIB_PATH} is missing; run `python -m marigold_b200.build` (no CPU fallback exists)")
        from . import build as _build

        _build.build()
    elif _stale():
        # sources newer than the library (a checkout moved on). Not rebuilt implicitly: several ranks may be starting at
        # once and file times do not survive every copy; MGB_REBUILD_STALE=1 opts in.
        if os.environ.get("MGB_REBUILD_STALE") == "1" and build_if_missing:
            from . import build as _build

            _build.build()
        else:
            import warnings

            warnings.warn(f"{_LIB_PATH.name} is older than its sources under csrc/; run `python -m marigold_b200.build`",
                          RuntimeWarning, stacklevel=2)
    lib = C.CDLL(str(_LIB_PATH), mode=os.RTLD_GLOBAL if hasattr(os, "RTLD_GLOBAL") else C.DEFAULT_MODE)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # header and library out of sync
            raise MgbError(f"libmarigold_b200.so does not export {name}") from e
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().mgb_last_error().decode("utf-8", "replace")
        raise MgbError(f"{what or 'libmarigold_b200'} failed with status {status}: {msg}")


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "tensor must be contiguous"
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch

    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
