"""ctypes binding of ``librdvc_corr.so`` -- exactly the symbols ``include/rdvc_corr.h`` declares.

There is no fallback: if the library has not been built (``_build.build()`` /
``__graft_entry__.build()``), importing a compute entry point raises.
"""
from __future__ import annotations

import ctypes
import os

from . import _build

RDVC_DT_BF16, RDVC_DT_F32, RDVC_DT_F16 = 0, 1, 2
RDVC_LAYOUT_ROWMAJOR, RDVC_LAYOUT_TILED = 0, 1
RDVC_OUT_NCHW, RDVC_OUT_KMAJOR = 0, 1
RDVC_ACT_NONE, RDVC_ACT_RELU = 0, 1
RDVC_GRU_HORIZONTAL, RDVC_GRU_VERTICAL = 0, 1
RDVC_UC_CONVCORR2, RDVC_UC_CONVFLOW1, RDVC_UC_CONVFLOW2, RDVC_UC_CONV, RDVC_UC_FH_CONV1, RDVC_UC_FH_CONV2 = range(6)
RDVC_MASK_OUT_UPSAMPLED, RDVC_MASK_OUT_MASK = 0, 1
RDVC_CE_OUT_RAW, RDVC_CE_OUT_SPLIT = 0, 1
RDVC_FE_OUT_FEATURES, RDVC_FE_OUT_TRUNK = 0, 1

RDVC_E = {
    -1: "RDVC_E_NULL", -2: "RDVC_E_SHAPE", -3: "RDVC_E_TOO_SMALL", -4: "RDVC_E_DTYPE",
    -5: "RDVC_E_UNSUPPORTED", -6: "RDVC_E_WORKSPACE", -7: "RDVC_E_ALIGN", -8: "RDVC_E_DRIVER",
}

# every symbol of include/rdvc_corr.h: name -> (restype, argtypes)
_c = ctypes
SYMBOLS = {
    "rdvc_corr_version": (_c.c_int, []),
    "rdvc_corr_last_error": (_c.c_char_p, []),
    "rdvc_corr_build_info": (_c.c_char_p, []),
    "rdvc_corr_pyramid_bytes": (_c.c_size_t, [_c.c_int] * 6),
    "rdvc_corr_level_offset_bytes": (_c.c_size_t, [_c.c_int] * 6),
    "rdvc_corr_level_image_elems": (_c.c_size_t, [_c.c_int] * 5),
    "rdvc_corr_tile_shape": (_c.c_int, [_c.c_int, _c.POINTER(_c.c_int), _c.POINTER(_c.c_int)]),
    "rdvc_corr_workspace_bytes": (_c.c_size_t, [_c.c_int] * 4),
    "rdvc_corr_build": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_int,
                                   _c.c_int, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p,
                                   _c.c_size_t, _c.c_void_p]),
    "rdvc_corr_lookup": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int,
                                    _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p]),
    "rdvc_corr_lookup_ex": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int,
                                       _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_corr_feat_pitch": (_c.c_size_t, [_c.c_int, _c.c_int]),
    "rdvc_corr_feat_rows": (_c.c_size_t, [_c.c_int] * 3),
    "rdvc_corr_feat_bytes": (_c.c_size_t, [_c.c_int] * 5),
    "rdvc_conv1x1_packed_weight_bytes": (_c.c_size_t, [_c.c_int] * 3),
    "rdvc_conv1x1_pack_weights": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_conv1x1": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p] + [_c.c_int] * 7 +
                     [_c.c_void_p, _c.c_int, _c.c_void_p]),
    "rdvc_corr_lookup_conv1x1": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p] + [_c.c_int] * 5 +
                                 [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_size_t,
                                  _c.c_void_p, _c.c_int, _c.c_void_p]),
    "rdvc_corr_pair_host_submit_ex": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p] +
                                      [_c.c_int] * 10),
    "rdvc_corr_plan_cache_hits": (_c.c_ulonglong, []),
    "rdvc_corr_pack": (_c.c_int, [_c.c_void_p, _c.c_void_p] + [_c.c_int] * 8 + [_c.c_void_p, _c.c_size_t, _c.c_void_p]),
    "rdvc_linear_packed_weight_bytes": (_c.c_size_t, [_c.c_int, _c.c_int]),
    "rdvc_linear_pack_weights": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_corr_encoder_tail": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_int, _c.c_void_p, _c.c_void_p] + [_c.c_int] * 8 +
                               [_c.c_void_p, _c.c_size_t, _c.c_void_p]),
    "rdvc_corr_build_packed": (_c.c_int, [_c.c_int] * 5 + [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p,
                                          _c.c_size_t, _c.c_void_p]),
    "rdvc_ec_max_encoded_bytes": (_c.c_size_t, [_c.c_size_t]),
    "rdvc_ec_encode_with_indexes": (_c.c_size_t, [_c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p,
                                                  _c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_size_t]),
    "rdvc_ec_decode_with_indexes": (_c.c_int, [_c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_size_t, _c.c_void_p,
                                               _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_corr_pair_host": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p] +
                            [_c.c_int] * 8),
    "rdvc_motion_warp": (_c.c_int, [_c.c_void_p, _c.c_void_p] + [_c.c_int] * 6 + [_c.c_void_p, _c.c_void_p, _c.c_void_p]),
    "rdvc_preprocess_frame": (_c.c_int, [_c.c_void_p] + [_c.c_int] * 3 + [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_mcn_plane_bytes": (_c.c_size_t, [_c.c_int] * 3),
    "rdvc_mcn_workspace_bytes": (_c.c_size_t, [_c.c_int] * 3),
    "rdvc_mcn_packed_weight_bytes": (_c.c_size_t, [_c.c_int] * 2),
    "rdvc_mcn_pack_weights": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p,
                                         _c.POINTER(_c.c_ulonglong)]),
    "rdvc_mcn_pack_input": (_c.c_int, [_c.c_void_p] * 3 + [_c.c_int] * 6 + [_c.c_void_p, _c.c_void_p]),
    "rdvc_mcn_conv": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_ulonglong, _c.c_void_p, _c.c_int, _c.c_int,
                                 _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_mcn_conv_out": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_ulonglong, _c.c_void_p, _c.c_int, _c.c_int,
                                     _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p]),
    "rdvc_mcn_forward": (_c.c_int, [_c.c_void_p] * 3 + [_c.c_int] * 4 + [_c.c_void_p, _c.c_void_p, _c.c_void_p,
                                    _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p]),
    "rdvc_corr_convgru_packed_weight_bytes": (_c.c_size_t, []),
    "rdvc_corr_convgru_pack_weights": (_c.c_int, [_c.c_void_p] * 3 + [_c.c_int, _c.c_void_p]),
    "rdvc_corr_convgru_workspace_bytes": (_c.c_size_t, [_c.c_int] * 4),
    "rdvc_corr_convgru": (_c.c_int, [_c.c_void_p, _c.c_longlong] * 3 + [_c.c_int] * 6 +
                     [_c.c_void_p] * 5 + [_c.c_size_t, _c.c_void_p, _c.c_void_p]),
    "rdvc_conv1x1_ex": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p] + [_c.c_int] * 7 +
                        [_c.c_void_p, _c.c_int, _c.c_longlong, _c.c_void_p]),
    "rdvc_corr_lookup_conv1x1_ex": (_c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p] + [_c.c_int] * 5 +
                                    [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_size_t,
                                     _c.c_void_p, _c.c_int, _c.c_longlong, _c.c_void_p]),
    "rdvc_corr_update_conv_packed_weight_bytes": (_c.c_size_t, [_c.c_int]),
    "rdvc_corr_update_conv_pack_weights": (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_int, _c.c_void_p]),
    "rdvc_corr_update_conv": (_c.c_int, [_c.c_int, _c.c_void_p, _c.c_longlong, _c.c_void_p, _c.c_void_p] + [_c.c_int] * 4 +
                         [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_longlong, _c.c_int, _c.c_void_p]),
    "rdvc_corr_motion_encoder_workspace_bytes": (_c.c_size_t, [_c.c_int] * 3),
    "rdvc_corr_motion_encoder": (_c.c_int, [_c.c_void_p, _c.c_longlong, _c.c_void_p, _c.c_void_p] + [_c.c_int] * 4 +
                            [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_longlong, _c.c_int,
                             _c.c_void_p]),
    "rdvc_corr_flow_head_workspace_bytes": (_c.c_size_t, [_c.c_int] * 4),
    "rdvc_corr_flow_head": (_c.c_int, [_c.c_void_p, _c.c_longlong] + [_c.c_int] * 5 +
                       [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_size_t, _c.c_void_p, _c.c_void_p]),
    "rdvc_corr_mask_conv_packed_weight_bytes": (_c.c_size_t, []),
    "rdvc_corr_mask_conv_pack_weights": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p]),
    "rdvc_corr_mask_predictor_workspace_bytes": (_c.c_size_t, [_c.c_int] * 4),
    "rdvc_corr_mask_predictor": (_c.c_int, [_c.c_void_p, _c.c_longlong] + [_c.c_int] * 5 +
                                 [_c.c_void_p, _c.c_void_p, _c.c_float, _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p,
                                  _c.c_size_t, _c.c_void_p, _c.c_void_p]),
    "rdvc_corr_context_encoder_packed_weight_bytes": (_c.c_size_t, []),
    "rdvc_corr_context_encoder_packed_bias_bytes": (_c.c_size_t, []),
    "rdvc_corr_context_encoder_pack_weights": (_c.c_int, [_c.c_void_p] * 7 + [_c.c_int, _c.c_void_p, _c.c_void_p]),
    "rdvc_corr_context_encoder_workspace_bytes": (_c.c_size_t, [_c.c_int] * 4),
    "rdvc_corr_context_encoder": (_c.c_int, [_c.c_void_p, _c.c_void_p] + [_c.c_int] * 5 +
                                  [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_size_t, _c.c_void_p,
                                   _c.c_longlong, _c.c_int, _c.c_void_p]),
    "rdvc_corr_feature_encoder_workspace_bytes": (_c.c_size_t, [_c.c_int] * 4),
    "rdvc_corr_feature_encoder": (_c.c_int, [_c.c_void_p, _c.c_void_p] + [_c.c_int] * 5 +
                                  [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_size_t,
                                   _c.c_void_p, _c.c_longlong, _c.c_int, _c.c_void_p]),
    "rdvc_corr_pair_host_submit": (_c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p] +
                                   [_c.c_int] * 9),
    "rdvc_corr_pair_host_wait": (_c.c_int, [_c.c_int]),
    "rdvc_corr_release": (None, []),
    "rdvc_corr_launch_count": (_c.c_ulonglong, []),
    "rdvc_corr_set_option": (_c.c_int, [_c.c_int, _c.c_int]),
    "rdvc_corr_set_profile_events": (None, [_c.c_void_p, _c.c_void_p]),
}

_lib = None


def lib_path() -> str:
    # RDVC_CORR_LIB: developer override to A/B-test an alternative build of the same ABI
    return os.environ.get("RDVC_CORR_LIB") or _build.LIB_PATH


def load():
    """Load the shared library (never builds it implicitly on a GPU box: a
    missing library is an error, not a reason to fall back)."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} is missing: the CUDA library has not been built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "There is no CPU or PyTorch fallback for this path."
        )
    # the library must have been built from exactly the sources in this tree (content hash compiled into it):
    # a stale binary that happens to sit next to newer sources is an error, not something to run
    built_from, tree = _build.embedded_hash(path), _build.source_hash()
    if built_from != tree and not os.environ.get("RDVC_CORR_ALLOW_STALE"):
        raise RuntimeError(
            f"{path} was built from other sources (library {str(built_from)[:12]}, tree {tree[:12]}): rebuild with "
            "`python -c 'import __graft_entry__ as g; g.build()'`."
        )
    L = ctypes.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def has_experiments() -> bool:
    """True if the loaded library was compiled with -DRDVC_EXPERIMENTS (never the product build)."""
    return b"experiments=1" in load().rdvc_corr_build_info()


def last_error() -> str:
    return load().rdvc_corr_last_error().decode("utf-8", "replace")


def check(rc: int, what: str):
    """0 -> ok; negative RDVC_E_* -> ValueError (argument problems, mirrors the
    ValueErrors of TV:raft.py:368-383); positive cudaError_t -> RuntimeError."""
    if rc == 0:
        return
    msg = last_error()
    if rc < 0:
        raise ValueError(f"{what}: {RDVC_E.get(rc, rc)}: {msg}")
    raise RuntimeError(f"{what}: CUDA error {rc}: {msg}")


def forward_only(what: str, *tensors) -> None:
    """The kernels are forward-only (the reference runs this path under ``torch.no_grad()``,
    R:codec_processing.py:1436): refuse tensors that would carry a gradient instead of silently cutting the graph."""
    import torch
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise RuntimeError(
            f"{what}: rdvc_corr_b200 is forward-only; an input requires grad and gradients cannot flow through these "
            "kernels. Call it under torch.no_grad() (as the reference does) or detach the inputs."
        )
