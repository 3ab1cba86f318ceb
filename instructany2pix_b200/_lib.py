"""ctypes binding of ``libia2p_sm100a.so`` (C ABI declared in ``include/ia2p.h``).

The shared library is built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``.  There is no
fallback: if the library is missing, or the device is not sm_100, every op raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IA2P_LIB_OVERRIDE") or os.path.join(_HERE, "libia2p_sm100a.so")   # override: A/B experiment builds only

F32, BF16, F16 = 0, 1, 2
EPI_NONE, EPI_GEGLU, EPI_GELU, EPI_QUICK_GELU = 0, 1, 2, 3
ACT_NONE, ACT_GELU_NEW, ACT_SILU = 0, 1, 2

_p, _i, _l, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float

# name -> argtypes; must list every symbol declared in include/ia2p.h (tests/test_abi.py checks both directions)
SIGNATURES = {
    "ia2p_version": ([], _i),
    "ia2p_last_error": ([], C.c_char_p),
    "ia2p_device_check": ([_i], _i),
    "ia2p_set_pdl": ([_i], _i),
    "ia2p_cfg_ddim_step": ([_p, _i, _p, _p, _i, _p, _i, _l, _l, _f, _f, _f, _p], _i),
    "ia2p_cfg_ddim_step_rows": ([_p, _i, _p, _p, _i, _p, _i, _l, _l, _p, _f, _f, _p], _i),
    "ia2p_cfg_step_coef_rows": ([_p, _i, _p, _p, _i, _p, _i, _l, _l, _p, _p, _p, _p, _p], _i),
    "ia2p_rowbias_gather": ([_p, _p, _p, _p, _p, _l, _l, _p, _l, _l, _p], _i),
    "ia2p_axpby": ([_p, _i, _p, _p, _i, _l, _f, _f, _p], _i),
    "ia2p_inpaint_blend": ([_p, _p, _p, _p, _p, _l, _l, _l, _f, _f, _p], _i),
    "ia2p_polar_workspace_bytes": ([], _l),
    "ia2p_polar_interpolate": ([_p, _p, _p, _l, _f, _p, _p], _i),
    "ia2p_prior_cfg_ddpm_step": ([_p, _p, _p, _p, _l, _f, _f, _f, _f, _f, _f, _p], _i),
    "ia2p_timestep_embedding": ([_p, _l, _i, _i, _f, _p, _i, _p], _i),
    "ia2p_upsample2x_nhwc": ([_p, _i, _p, _l, _l, _l, _l, _p], _i),
    "ia2p_cast_to_bf16": ([_p, _i, _p, _l, _p], _i),
    "ia2p_groupnorm_nhwc": ([_p, _l, _p, _l, _i, _p, _p, _p, _p, _l, _l, _i, _f, _i, _p, _l, _p, _l, _p, _p], _i),
    "ia2p_groupnorm_workspace_bytes": ([_l, _i], _l),
    "ia2p_layernorm": ([_p, _i, _p, _p, _p, _i, _l, _l, _f, _p], _i),
    "ia2p_clip_embed": ([_p, _l, _l, _p, _l, _p, _l, _l, _p, _p, _p, _p], _i),
    "ia2p_gemm_bf16": ([_p, _l, _l, _p, _l, _l, _p, _p, _l, _l, _l, _p, _p, _l, _p, _l, _i, _i, _i, _p], _i),
    "ia2p_gemm_ln_bf16": ([_p, _l, _l, _p, _l, _l, _p, _p, _l, _l, _l, _p, _p, _l, _p, _l, _i, _i, _i,
                           _p, _l, _p, _p, _p, _l, _p, _f, _p], _i),
    "ia2p_gemm_ln_parts": ([_l, _l, _l], _l),
    "ia2p_tc_workspace_bytes": ([], _l),
    "ia2p_tc_features": ([], _i),
    "ia2p_set_tc_workspace": ([_p, _l], _i),
    "ia2p_conv_colstats_tiles": ([_l, _l, _l], _l),
    "ia2p_tc_prefetch_hint": ([_p, _l], _i),
    "ia2p_conv3x3_nhwc_bf16": ([_p, _l, _l, _l, _l, _i, _p, _p, _l, _p, _l, _p, _i, _l, _p, _p, _p, _i, _p, _p], _i),
    "ia2p_conv_up2x_nhwc_bf16": ([_p, _l, _l, _l, _l, _p, _p, _l, _p, _p, _p], _i),
    "ia2p_conv3x3_s2_padend_nhwc_bf16": ([_p, _l, _l, _l, _l, _p, _p, _i, _l, _p, _p], _i),
    "ia2p_gaussian_sample": ([_p, _p, _p, _l, _l, _l, _f, _p], _i),
    "ia2p_conv_in_nchw": ([_p, _i, _l, _l, _l, _l, _l, _p, _p, _p, _i, _l, _p], _i),
    "ia2p_conv_out_nhwc": ([_p, _l, _l, _l, _l, _p, _p, _p, _i, _l, _p], _i),
    "ia2p_nhwc_prefix_to_nchw": ([_p, _l, _p, _l, _l, _l, _p], _i),
    "ia2p_conv1x1_nchw_small": ([_p, _p, _p, _p, _l, _l, _l, _l, _f, _p], _i),
    "ia2p_softmax_rows_f32_bf16": ([_p, _l, _p, _l, _l, _l, _f, _p], _i),
    "ia2p_flash_self_attn_bf16": ([_p, _p, _p, _l, _p, _l, _l, _l, _i, _f, _p], _i),
    "ia2p_causal_self_attn_bf16": ([_p, _p, _p, _l, _p, _l, _l, _l, _i, _f, _p], _i),
    "ia2p_decoupled_cross_attn_bf16": ([_p, _l, _p, _p, _l, _i, _p, _p, _l, _i, _f, _p, _l, _l, _l, _i, _f, _p], _i),
    "ia2p_decoupled_cross_attn_rows_bf16": ([_p, _l, _p, _p, _l, _i, _p, _p, _l, _i, _p, _p, _l, _l, _l, _i, _f, _p], _i),
    "ia2p_gemm_smallm": ([_p, _l, _p, _p, _p, _l, _p, _l, _l, _l, _l, _i, _i, _p], _i),
    "ia2p_causal_attn_small_f32": ([_p, _p, _l, _l, _i, _p], _i),
    "ia2p_prior_trunk_workspace_bytes": ([_l], _l),
    "ia2p_prior_trunk": ([_p, _p, _p, _i, _p, _p, _l, _l, _l, _i, _p, _l, _p, _p], _i),
}

_lib = None


class IA2PError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IA2PError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(nvcc, sm_100a).  instructany2pix_b200 has no CPU / PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (argtypes, restype) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = restype
    _lib = lib
    return lib


def check(status: int, what: str):
    if status != 0:
        msg = load().ia2p_last_error().decode(errors="replace")
        raise IA2PError(f"{what} failed with status {status}: {msg}")
