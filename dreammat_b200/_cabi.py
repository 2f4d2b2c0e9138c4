"""ctypes binding of include/dreammat_b200.h.

The product path has no CPU fallback: if the shared object is missing or a call fails the
caller gets an exception, never a silently different code path.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libdreammat_b200.so")

_lib = None


class DmError(RuntimeError):
    pass


class HashGridCfg(C.Structure):
    _fields_ = [("n_levels", C.c_int32), ("n_features", C.c_int32), ("log2_hashmap", C.c_int32),
                ("base_resolution", C.c_int32), ("per_level_scale", C.c_float), ("bbox_min", C.c_float),
                ("bbox_max", C.c_float), ("n_hidden", C.c_int32), ("n_out", C.c_int32)]


class MaterialCfg(C.Structure):
    _fields_ = [("min_metallic", C.c_float), ("max_metallic", C.c_float), ("min_roughness", C.c_float),
                ("max_roughness", C.c_float), ("n_diffuse", C.c_int32), ("n_specular", C.c_int32)]


P = C.c_void_p
I64 = C.c_int64
I32 = C.c_int32
F = C.c_float

# name -> (restype, argtypes); kept in one table so tests can check that every symbol the
# header declares is exported by the shared object.
SIGNATURES = {
    "dm_last_error": (C.c_char_p, []),
    "dm_version": (C.c_int, []),
    "dm_launch_count": (C.c_longlong, []),
    "dm_tune": (C.c_int, [C.c_char_p, C.c_int]),
    "dm_tune_gemm": (C.c_int, [C.c_int]),
    "dm_gemm_plan": (C.c_int, [I64, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "dm_gemm_workspace_bytes": (C.c_size_t, []),
    "dm_gemm_set_workspace": (C.c_int, [P, C.c_size_t]),
    "dm_tune_attention": (C.c_int, [C.c_int]),
    "dm_device_check": (C.c_int, [C.c_int]),
    "dm_hashgrid_layout": (I64, [P, P]),
    "dm_hashgrid_mlp_fwd": (C.c_int, [P, P, I64, P, P, P, P, P]),
    "dm_hashgrid_mlp_bwd": (C.c_int, [P, P, I64, P, P, P, P, P, P, P, P]),
    "dm_hashgrid_encode": (C.c_int, [P, P, I64, P, P, P]),
    "dm_jitter_positions": (C.c_int, [P, P, P, P, I64, P, P]),
    "dm_bvh_build": (C.c_int, [P, I64, P, I64, P]),
    "dm_bvh_free": (None, [P]),
    "dm_bvh_num_nodes": (I64, [P]),
    "dm_bvh_trace": (C.c_int, [P, P, P, I64, P, P, P, P]),
    "dm_raster_gbuffer": (C.c_int, [P] * 8 + [C.c_int] * 3 + [P] * 6),
    "dm_compact_mask": (C.c_int, [P, I64, P, P, P]),
    "dm_gather_rows": (C.c_int, [P, P, I64, C.c_int, P, P]),
    "dm_depth_normalize": (C.c_int, [P, P, I64, P, P, P]),
    "dm_shade_mc_fwd": (C.c_int, [P, P, P, C.c_int, C.c_int] + [P] * 9 + [I64] + [P] * 13),
    "dm_shade_splitsum_fwd": (C.c_int, [P, P, C.c_int, P, C.c_int, P, C.c_int, C.c_int] + [P] * 4 + [I64] + [P] * 11),
    "dm_shade_bwd": (C.c_int, [P, P, P, P, P, F, F, I64, P, P, P]),
    "dm_envmap_pack": (C.c_int, [P, I64, P, P]),
    "dm_scatter_canvas": (C.c_int, [P, P, I64, C.c_int, P, P]),
    "dm_fill": (C.c_int, [P, I64, F, P]),
    "dm_gather_canvas_grad": (C.c_int, [P, P, I64, C.c_int, P, P]),
    "dm_antialias_fwd": (C.c_int, [P, P, P, P, I64, I64, C.c_int, P, P]),
    "dm_antialias_bwd": (C.c_int, [P, P, P, P, I64, I64, C.c_int, P, P]),
    "dm_resize_bilinear": (C.c_int, [P] + [C.c_int] * 6 + [P, C.c_int, P]),
    "dm_adam_step": (C.c_int, [P, P, P, P, I64, F, F, F, F, I32, F, P]),
    "dm_sds_grad": (C.c_int, [P, P, P, C.c_int, I64, F, F, F, F, P, P, P, P]),
    "dm_gemm": (C.c_int, [C.c_int, P, I64, I64, P, I64, I64, P, I64, I64, C.c_int, C.c_int, C.c_int, C.c_int, P,
                          C.c_int, P]),
    "dm_groupnorm": (C.c_int, [C.c_int, P] + [C.c_int] * 5 + [P, P, F, C.c_int, P, C.c_int, P, P]),
    "dm_groupnorm_bwd": (C.c_int, [C.c_int, P, P] + [C.c_int] * 4 + [P, P, F, C.c_int, P, P, P, P, P]),
    "dm_layernorm": (C.c_int, [C.c_int, P, I64, C.c_int, P, P, F, P, P]),
    "dm_geglu": (C.c_int, [C.c_int, P, I64, C.c_int, P, P]),
    "dm_upsample2x": (C.c_int, [C.c_int, P] + [C.c_int] * 5 + [P, P]),
    "dm_axpby2d": (C.c_int, [C.c_int, P, I64, F, P, I64, F, I64, C.c_int, P, I64, P]),
    "dm_transpose": (C.c_int, [C.c_int, P, C.c_int, C.c_int, C.c_int, I64, I64, P, I64, I64, P]),
    "dm_softmax_rows": (C.c_int, [C.c_int, P, I64, C.c_int, I64, F, P, P]),
    "dm_softmax_bwd": (C.c_int, [C.c_int, P, P, I64, C.c_int, I64, F, P, P]),
    "dm_pad_convert": (C.c_int, [C.c_int, P, I64, C.c_int, C.c_int, F, F, P, P]),
    "dm_unpad_convert": (C.c_int, [C.c_int, P, I64, C.c_int, C.c_int, F, P, P]),
    "dm_nhwc_to_nchw_f32": (C.c_int, [C.c_int, P] + [C.c_int] * 4 + [P, P]),
    "dm_vae_sample": (C.c_int, [C.c_int, P, C.c_int, C.c_int, C.c_int, P, F, P, P]),
    "dm_vae_sample_bwd": (C.c_int, [C.c_int, P, C.c_int, C.c_int, C.c_int, P, F, P, P, P]),
    "dm_add_noise": (C.c_int, [C.c_int, P, P, P, P] + [C.c_int] * 4 + [P, P]),
    "dm_timestep_embedding": (C.c_int, [C.c_int, P, C.c_int, C.c_int, P, P]),
    "dm_silu": (C.c_int, [C.c_int, P, I64, P, P]),
    "dm_attention": (C.c_int, [C.c_int, P, I64, I64, P, P, I64, I64, P, I64, I64] + [C.c_int] * 5 + [F, P]),
    "dm_cond_gather": (C.c_int, [C.c_int, P, P, P, C.c_int, I64, P, P, C.c_int, C.c_int, P, P]),
    "dm_envlight_latlong_to_cube": (C.c_int, [P, C.c_int, C.c_int, F, C.c_int, P, P]),
    "dm_envlight_downsample": (C.c_int, [P, C.c_int, P, P]),
    "dm_envlight_filter": (C.c_int, [P, C.c_int, C.c_int, F, F, P, P]),
    "dm_conv2d_csd": (C.c_int, [C.c_int, P, C.c_int, C.c_int, C.c_int, C.c_int, P, P, P, P]),
    "dm_hp_split": (C.c_int, [P, I64, C.c_int, I64, C.c_int, P, P]),
    "dm_hp_epilogue": (C.c_int, [P, I64, C.c_int, I64, P, P, I64, I64, P]),
    "dm_conv2d": (C.c_int, [C.c_int, P] + [C.c_int] * 4 + [P] + [C.c_int] * 7 + [P, I64, P, C.c_int, P]),
    "dm_uv_raster": (C.c_int, [P, P, I64, C.c_int, P, P, P, P]),
    "dm_texel_positions": (C.c_int, [P, I64, P, P, P, P, P, P]),
    "dm_material_export": (C.c_int, [P, P, I64, P, P, P, P, P, P]),
    "dm_seam_fill": (C.c_int, [P, C.c_int] + [P] * 9),
}


def lib():
    """Load the C-ABI library; raises DmError (never falls back) when it is absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DmError(f"{LIB_PATH} not found: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(dreammat_b200 has no CPU fallback)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().dm_last_error()
        raise DmError(f"{what} failed (rc={rc}): {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a contiguous torch tensor (or None)."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise DmError("non-contiguous tensor passed to the C-ABI")
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
