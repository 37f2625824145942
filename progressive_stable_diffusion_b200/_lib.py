"""ctypes binding of ``libdadd_b200.so`` (the C ABI declared in ``include/dadd_b200.h``).

There is no CPU fallback: if the library is missing ``load()`` raises, and every wrapper in ``ops.py`` goes through it.
"""

from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_int64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DADD_B200_LIB") or os.path.join(HERE, "libdadd_b200.so")      # (override: A/B builds of a kernel)

_P, _I, _L, _F = c_void_p, c_int, c_int64, c_float

ABI_VERSION = 15         # == DADD_ABI_VERSION of include/dadd_b200.h that SIGNATURES below was written against

# name -> argtypes; mirrors include/dadd_b200.h one to one (tests/test_abi.py checks header <-> table <-> .so)
SIGNATURES = {
    "dadd_ddim_step": [_P, _P, _P, _I, _F, _F, _F, _F, _F, _F, _P, _F, _I, _L, _P],
    "dadd_ddim_step_table": [_P, _P, _P, _I, _F, _P, _P, _I, _P, _F, _L, _P],
    "dadd_step_begin": [_P, _P, _P, _L, _I, _P],
    "dadd_groupnorm_workspace_bytes": [_I, _I, _I, _I, _I],
    "dadd_groupnorm_fwd": [_P, _P, _P, _P, _L, _P, _I, _I, _I, _I, _F, _I, _I, _I, _P, _L, _P],
    "dadd_groupnorm_cat_supported": [_I, _I, _I, _I, _I, _I],
    "dadd_groupnorm_select": [_I],
    "dadd_groupnorm_cat_fwd": [_P, _I, _P, _I, _P, _P, _P, _L, _P, _I, _I, _I, _F, _I, _I, _P, _L, _P],
    "dadd_layernorm_fwd": [_P, _P, _P, _P, _L, _I, _F, _I, _P],
    "dadd_add_layernorm_fwd": [_P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P],
    "dadd_bias_residual_fwd": [_P, _P, _P, _P, _L, _I, _I, _P],
    "dadd_upsample_nearest2x_fwd": [_P, _P, _I, _I, _I, _I, _I, _P],
    "dadd_linear_supported": [_L, _I, _I],
    "dadd_linear_fwd": [_P, _P, _P, _P, _P, _L, _I, _I, _I, _P],
    "dadd_ff_geglu_fwd": [_P, _P, _P, _P, _L, _I, _I, _I, _P],
    "dadd_quick_gelu_fwd": [_P, _P, _L, _I, _P],
    "dadd_geglu_fwd": [_P, _P, _L, _I, _I, _P],
    "dadd_cross_attn_fwd": [_P, _L, _P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _P, _F, _I, _I, _P],
    "dadd_self_attn_fwd": [_P, _P, _P, _L, _L, _L, _P, _L, _I, _I, _I, _I, _F, _I, _I, _P],
    "dadd_purifier_attn_fwd": [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P],
    "dadd_purifier_gate_ln_fwd": [_P, _P, _P, _P, _P, _P, _L, _I, _F, _P],
    "dadd_aoe_interp_fwd": [_P, _P, _P, _P, _I, _I, _I, _P],
    "dadd_image_post_fwd": [_P, _P, _L, _I, _P],
    # training step
    "dadd_layernorm_bwd_workspace_bytes": [_I],
    "dadd_layernorm_bwd": [_P, _P, _P, _P, _P, _P, _P, _L, _I, _F, _I, _P],
    "dadd_geglu_bwd": [_P, _P, _P, _L, _I, _I, _P],
    "dadd_groupnorm_bwd_workspace_bytes": [_I, _I, _I, _I],
    "dadd_groupnorm_bwd": [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _F, _I, _I, _P],
    "dadd_cross_attn_bwd_workspace_bytes": [_I, _I, _I, _I, _I],
    "dadd_cross_attn_bwd": [_P, _L, _P, _P, _P, _P, _L, _P, _L, _P, _P, _P, _I, _I, _I, _I, _I, _I, _F, _I, _P],
    "dadd_minsnr_mse_workspace_bytes": [_I],
    "dadd_minsnr_mse": [_P, _P, _P, _P, _P, _P, _I, _L, _F, _P],
    "dadd_sumsq": [_P, _L, _P, _I, _P],
    "dadd_clip_coef": [_P, _I, _F, _F, _P, _P],
    "dadd_adamw_step": [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _F, _F, _P, _P],
    "dadd_adamw_step_dev": [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _P, _P, _P],
    "dadd_ema_update": [_P, _P, _L, _F, _I, _P],
    # evaluation metrics
    "dadd_pairwise_workspace_bytes": [_L, _L, _I, _I, _I, _I],
    "dadd_pairwise": [_P, _P, _L, _L, _I, _I, _I, _I, _F, _P, _P, _P, _L, _P],
}

_lib = None


class DaddError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load the library (building is ``__graft_entry__.build()`` / ``python -m progressive_stable_diffusion_b200.build``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DaddError(
            f"{LIB_PATH} is missing: the sm_100a kernels are the only implementation of this package "
            "(no CPU / eager fallback). Build them with `python -m progressive_stable_diffusion_b200.build`."
        )
    lib = ctypes.CDLL(LIB_PATH)
    lib.dadd_abi_version.restype = c_int
    have = int(lib.dadd_abi_version())
    if have != ABI_VERSION:      # the .so is git-ignored and survives checkouts: never call it through mismatched signatures
        raise DaddError(f"{LIB_PATH} has ABI version {have}, this binding needs {ABI_VERSION}: rebuild it with "
                        "`python -m progressive_stable_diffusion_b200.build --force`")
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = c_int64 if name.endswith("_bytes") else c_int
    lib.dadd_last_error.restype = c_char_p
    lib.dadd_launch_count.restype = c_int64
    lib.dadd_reset_launch_count.restype = None
    _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().dadd_last_error().decode("utf-8", "replace")
        raise DaddError(f"{what} failed (rc={rc}): {msg}")


def launch_count() -> int:
    return int(load().dadd_launch_count())


def reset_launch_count() -> None:
    load().dadd_reset_launch_count()
