"""ctypes binding of libnerfpp_b200.so (include/nerfpp_b200.h).

Plumbing only: torch supplies device memory and the current CUDA stream, every computation happens in the
hand-written sm_100a kernels behind the C ABI.  There is no fallback of any kind: if the library is missing it is
built with nvcc, and if that fails, or a call returns a non-zero status, this module raises.
"""
from __future__ import annotations

import ctypes as C
from ctypes import POINTER, Structure, c_float, c_int32, c_int64, c_void_p, c_char_p, c_uint8

import torch

from . import build as _build

NRF_MAX_LEVELS = 32
ENC_F32, ENC_F16 = 0, 1
GRAD_F32, GRAD_BF16 = 0, 1
MLP_IN_ENC16_RAYDIRS, MLP_IN_F32_CAT, MLP_IN_ENC16_RAYBIAS = 0, 1, 2


class NrfError(RuntimeError):
    pass


class HashGrid(Structure):
    """struct nrf_hash_grid"""
    _fields_ = [
        ("n_levels", c_int32), ("n_features", c_int32), ("n_volumes", c_int32),
        ("base_resolution", c_int32), ("finest_resolution", c_int32),
        ("box_min", c_float * 3), ("box_max", c_float * 3),
        ("primes", c_void_p), ("biases", c_void_p), ("feat_local_idx", c_void_p),
        ("feat_local_size", c_void_p), ("level_scale", c_void_p),
        ("table_scalars", c_int64),
    ]


class MlpSmallShape(Structure):
    """struct nrf_mlp_small_shape"""
    _fields_ = [
        ("input_ch", c_int32), ("input_ch_views", c_int32), ("hidden_dim", c_int32), ("geo_feat_dim", c_int32),
        ("hidden_dim_color", c_int32), ("num_layers", c_int32), ("num_layers_color", c_int32),
    ]


class MlpNerfShape(Structure):
    """struct nrf_mlp_nerf_shape"""
    _fields_ = [("depth", c_int32), ("width", c_int32), ("input_ch", c_int32), ("input_ch_views", c_int32), ("skip_layer", c_int32),
                ("use_viewdirs", c_int32)]


class MlpNerfWeights(Structure):
    """struct nrf_mlp_nerf_weights"""
    _fields_ = [("pts_w", c_void_p * 8), ("pts_b", c_void_p * 8), ("feature_w", c_void_p), ("feature_b", c_void_p), ("alpha_w", c_void_p),
                ("alpha_b", c_void_p), ("views_w", c_void_p), ("views_b", c_void_p), ("rgb_w", c_void_p), ("rgb_b", c_void_p)]


class LerfShape(Structure):
    """struct nrf_lerf_shape"""
    _fields_ = [("geo_feat_dim", c_int32), ("num_layers", c_int32), ("hidden_dim", c_int32), ("lang_embed_dim", c_int32), ("input_ch", c_int32)]


class LerfWeights(Structure):
    """struct nrf_lerf_weights"""
    _fields_ = [("sigma_w0", c_void_p), ("sigma_w1", c_void_p), ("le_w0", c_void_p), ("le_w1", c_void_p)]


class RenderConfig(Structure):
    """struct nrf_render_config"""
    _fields_ = [("n_samples", c_int32), ("n_importance", c_int32), ("white_bkgr", c_int32), ("lin_disp", c_int32), ("sh_degree", c_int32),
                ("near_plane", c_float), ("bbox", c_float * 6)]


class PointJitter(Structure):
    """struct nrf_point_jitter"""
    _fields_ = [("cone_angle", c_void_p), ("cone_stride", c_int32), ("rand_r", c_void_p), ("rand_theta", c_void_p), ("clamp_to_box", c_int32),
                ("sp_noise", c_void_p), ("sp_alpha", c_void_p)]


NRF_MAX_PEERS = 8


class PeerGroup(Structure):
    """struct nrf_peer_group"""
    _fields_ = [("world", c_int32), ("rank", c_int32), ("grads", c_void_p * NRF_MAX_PEERS), ("shadow_f16", c_void_p * NRF_MAX_PEERS),
                ("flags", c_void_p * NRF_MAX_PEERS), ("grads_mc", c_void_p), ("shadow_f16_mc", c_void_p)]


# name -> (restype, argtypes); must list every symbol include/nerfpp_b200.h declares (tests/test_abi.py checks)
_P = c_void_p
SIGNATURES = {
    "nrf_abi_version": (c_int32, []),
    "nrf_last_error": (c_char_p, []),
    "nrf_launch_count": (c_int64, []),
    "nrf_hash_level_scales": (c_int32, [c_int32, c_int32, c_int32, _P, _P]),
    "nrf_table_to_half": (c_int32, [_P, _P, c_int64, _P]),
    "nrf_hash_cells": (c_int32, [POINTER(HashGrid), _P, c_int64, c_int32, _P, _P, _P]),
    "nrf_hash_encode_fwd": (c_int32, [POINTER(HashGrid), _P, _P, c_int64, c_int32, _P, _P, c_int32, _P]),
    "nrf_hash_encode_bwd": (c_int32, [POINTER(HashGrid), _P, c_int64, c_int32, _P, c_int32, _P, _P]),
    "nrf_hash_encode_rays_fwd": (c_int32, [POINTER(HashGrid), _P, _P, c_int32, _P, c_int64, c_int32, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, _P]),
    "nrf_hash_encode_rays_fwd_grouped": (c_int32, [POINTER(HashGrid), _P, _P, c_int32, _P, c_int64, c_int32, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32,
                                                   c_int32, _P]),
    "nrf_hash_encode_rays_bwd": (c_int32, [POINTER(HashGrid), _P, c_int32, _P, c_int64, c_int32, c_int32, _P, c_int32, _P, _P]),
    "nrf_hash_encode_rays_jitter_fwd": (c_int32, [POINTER(HashGrid), _P, _P, c_int32, _P, c_int64, c_int32, c_int32, _P, _P, c_int32,
                                                  POINTER(PointJitter), _P]),
    "nrf_hash_encode_rays_jitter_bwd": (c_int32, [POINTER(HashGrid), _P, c_int32, _P, c_int64, c_int32, c_int32, _P, c_int32, _P,
                                                  POINTER(PointJitter), _P]),
    "nrf_sample_pdf_merge_perm": (c_int32, [_P, _P, _P, c_int32, c_int64, c_int32, c_int32, _P, _P, _P, _P]),
    "nrf_sample_pdf_merge_rows": (c_int32, [_P, _P, _P, c_int32, c_int64, c_int32, c_int32, _P, _P, _P, _P, _P, _P]),
    "nrf_sh_encode_fwd": (c_int32, [_P, c_int32, c_int64, c_int32, _P, _P]),
    "nrf_posenc_fwd": (c_int32, [_P, c_int64, c_int32, c_int32, POINTER(c_float), c_int32, _P, _P]),
    "nrf_mlp_small_packed_bytes": (c_int64, [POINTER(MlpSmallShape)]),
    "nrf_mlp_small_param_count": (c_int64, [POINTER(MlpSmallShape)]),
    "nrf_mlp_small_pack": (c_int32, [POINTER(MlpSmallShape), _P, _P, _P]),
    "nrf_mlp_small_fwd": (c_int32, [POINTER(MlpSmallShape), _P, c_int32, _P, _P, c_int32, _P, c_int64, _P, _P]),
    "nrf_mlp_small_fwd_importance": (c_int32, [POINTER(MlpSmallShape), _P, c_int32, _P, _P, _P, _P, c_int64, c_int32, c_int32, _P, _P]),
    "nrf_mlp_small_view_bias_fwd": (c_int32, [POINTER(MlpSmallShape), _P, _P, c_int64, _P, _P, _P]),
    "nrf_mlp_small_view_bias_bwd": (c_int32, [POINTER(MlpSmallShape), _P, _P, c_int64, _P, _P]),
    "nrf_mlp_small_bwd_raybias": (c_int32, [POINTER(MlpSmallShape), _P, c_int32, _P, _P, c_int32, _P, c_int64, _P, _P, _P, _P, _P]),
    "nrf_mlp_small_bwd": (c_int32, [POINTER(MlpSmallShape), _P, c_int32, _P, _P, c_int32, _P, c_int64, _P, _P, _P, _P]),
    "nrf_composite_fwd": (c_int32, [_P, c_int32, _P, _P, _P, c_float, c_int32, c_int64, c_int32, _P, _P, _P, _P, _P, _P]),
    "nrf_composite_bwd": (c_int32, [_P, c_int32, _P, _P, _P, c_float, c_int32, c_int64, c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "nrf_composite_huber_bwd": (c_int32, [_P, c_int32, _P, _P, _P, c_float, c_int32, c_int64, c_int32, _P, c_float, c_float, _P, _P, _P, _P]),
    "nrf_sample_pdf": (c_int32, [_P, _P, c_int32, _P, c_int32, c_int64, c_int32, _P, _P]),
    "nrf_sample_pdf_merge": (c_int32, [_P, _P, _P, c_int32, c_int64, c_int32, c_int32, _P, _P, _P]),
    "nrf_get_rays": (c_int32, [c_int32, c_int32, POINTER(c_float), POINTER(c_float), c_int32, c_int32, _P, _P, _P]),
    "nrf_rays_prepare": (c_int32, [_P, _P, c_int64, POINTER(c_float), c_float, c_int32, _P, _P]),
    "nrf_ray_setup": (c_int32, [_P, _P, c_int64, POINTER(c_float), c_float, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P]),
    "nrf_ray_batch": (c_int32, [_P, c_int64, POINTER(c_float), POINTER(c_float), _P, c_int32, c_int32, c_int32, _P, _P, _P, POINTER(c_float), _P]),
    "nrf_ray_setup_pixels": (c_int32, [_P, c_int64, POINTER(c_float), POINTER(c_float), _P, c_int32, c_int32, c_int32, POINTER(c_float), c_float, _P, c_int32,
                                       c_int32, c_int32, _P, _P, _P, _P, _P, _P, _P, _P]),
    "nrf_z_sample": (c_int32, [_P, c_int32, _P, c_int64, c_int32, c_int32, _P, _P]),
    "nrf_sample_points": (c_int32, [_P, c_int32, _P, c_int64, c_int32, _P, _P]),
    "nrf_precondition_points": (c_int32, [_P, _P, c_float, POINTER(c_float), c_int64, _P]),
    "nrf_tangent_scatter": (c_int32, [_P, _P, _P, c_int32, _P, c_int32, _P, _P, POINTER(c_float), c_int64, c_int32, _P]),
    "nrf_huber_fwd_bwd": (c_int32, [_P, _P, c_int64, c_float, c_float, _P, _P, _P]),
    "nrf_adam_step": (c_int32, [_P, _P, _P, _P, c_int64, c_float, c_float, c_float, c_float, c_int32, c_float, c_int32, _P, _P]),
    "nrf_mlp_nerf_packed_bytes": (c_int64, [POINTER(MlpNerfShape)]),
    "nrf_mlp_nerf_pack": (c_int32, [POINTER(MlpNerfShape), POINTER(MlpNerfWeights), _P, _P]),
    "nrf_mlp_nerf_fwd": (c_int32, [POINTER(MlpNerfShape), _P, _P, c_int64, _P, _P]),
    "nrf_mlp_nerf_pack_train": (c_int32, [POINTER(MlpNerfShape), POINTER(MlpNerfWeights), _P, _P]),
    "nrf_mlp_nerf_saved_bytes": (c_int64, [POINTER(MlpNerfShape), c_int64]),
    "nrf_mlp_nerf_bwd_workspace_bytes": (c_int64, [POINTER(MlpNerfShape), c_int64]),
    "nrf_mlp_nerf_fwd_train": (c_int32, [POINTER(MlpNerfShape), _P, _P, c_int64, _P, _P, _P]),
    "nrf_mlp_nerf_bwd": (c_int32, [POINTER(MlpNerfShape), _P, _P, _P, c_int64, _P, POINTER(MlpNerfWeights), _P]),
    "nrf_mlp_nerf_fwd_points": (c_int32, [POINTER(MlpNerfShape), _P, _P, _P, c_int32, POINTER(c_float), c_int32, POINTER(c_float), c_int32, c_int64, _P, _P]),
    "nrf_mlp_nerf_fwd_train_points": (c_int32, [POINTER(MlpNerfShape), _P, _P, _P, c_int32, POINTER(c_float), c_int32, POINTER(c_float), c_int32, c_int64,
                                                _P, _P, _P]),
    "nrf_render_rays_workspace_bytes": (c_int64, [POINTER(RenderConfig), POINTER(HashGrid), c_int64]),
    "nrf_render_rays_fwd": (c_int32, [POINTER(RenderConfig), POINTER(HashGrid), _P, POINTER(MlpSmallShape), _P, _P, _P, c_int64, _P, _P, _P, c_int64,
                                      _P, _P, _P, _P, _P, _P, _P]),
    "nrf_render_tile_fwd": (c_int32, [POINTER(RenderConfig), POINTER(HashGrid), _P, POINTER(MlpSmallShape), _P, POINTER(c_float), POINTER(c_float), c_int32,
                                      c_int64, c_int64, _P, _P, _P, c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "nrf_render_raybatch_fwd": (c_int32, [POINTER(RenderConfig), POINTER(HashGrid), _P, POINTER(MlpSmallShape), _P, _P, c_int32, c_int64, _P, _P, _P, c_int64,
                                          _P, _P, _P, _P, _P, _P, _P]),
    "nrf_ray_setup_prepared": (c_int32, [_P, c_int32, c_int64, _P, c_int32, c_int32, c_int32, _P, _P, _P, _P, _P]),
    "nrf_ray_setup_tile": (c_int32, [POINTER(c_float), POINTER(c_float), c_int32, c_int64, c_int64, POINTER(c_float), c_float, _P, c_int32, c_int32, c_int32,
                                     _P, _P, _P, _P, _P, _P]),
    "nrf_lerf_packed_bytes": (c_int64, [POINTER(LerfShape)]),
    "nrf_lerf_hidden_bytes": (c_int64, [POINTER(LerfShape), c_int64]),
    "nrf_lerf_pack": (c_int32, [POINTER(LerfShape), POINTER(LerfWeights), _P, _P]),
    "nrf_lerf_fwd": (c_int32, [POINTER(LerfShape), _P, _P, _P, c_int64, _P, _P]),
    "nrf_lerf_sigma_fwd": (c_int32, [POINTER(LerfShape), _P, _P, _P, c_int64, _P, _P]),
    "nrf_lerf_hidden_fwd": (c_int32, [POINTER(LerfShape), _P, _P, _P, c_int64, _P, _P, _P, _P]),
    "nrf_lerf_render_embedding": (c_int32, [POINTER(LerfShape), _P, _P, _P, _P, c_int64, c_int32, _P, _P, _P]),
    "nrf_lerf_train_saved_bytes": (c_int64, [POINTER(LerfShape), c_int64]),
    "nrf_lerf_bwd_workspace_bytes": (c_int64, [POINTER(LerfShape), c_int64, c_int64]),
    "nrf_lerf_fwd_train": (c_int32, [POINTER(LerfShape), _P, _P, _P, c_int64, _P, _P, _P, _P]),
    "nrf_lerf_render_embedding_train": (c_int32, [POINTER(LerfShape), _P, _P, _P, _P, c_int64, c_int32, _P, _P, _P, _P]),
    "nrf_lerf_bwd_rays": (c_int32, [POINTER(LerfShape), POINTER(LerfWeights), _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int32, c_float, _P, _P, _P, _P, _P]),
    "nrf_lerf_bwd_rows": (c_int32, [POINTER(LerfShape), _P, POINTER(LerfWeights), _P, _P, _P, c_int64, c_int32, _P, POINTER(LerfWeights), _P, _P]),
    "nrf_peer_flags_bytes": (c_int64, [c_int32]),
    "nrf_adam_step_sharded": (c_int32, [POINTER(PeerGroup), _P, _P, _P, c_int64, c_int64, _P, c_float, c_float, c_float, c_float, _P]),
    "nrf_adam_schedule_advance": (c_int32, [_P, c_float, c_float, c_float, c_float, c_float, _P]),
    "nrf_adam_step_scheduled": (c_int32, [_P, _P, _P, _P, c_int64, _P, c_float, c_float, c_float, c_float, c_int32, _P, _P]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads (building first if needed) the C-ABI library.  Raises if it cannot be had — never falls back."""
    global _lib
    if _lib is None:
        path = _build.build()
        handle = C.CDLL(str(path))
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the export is missing
            fn.restype = res
            fn.argtypes = args
        if handle.nrf_abi_version() != 1:
            raise NrfError("libnerfpp_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(status: int) -> None:
    if status != 0:
        raise NrfError(f"nerfpp_b200 status {status}: {lib().nrf_last_error().decode()}")


def stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def ptr(t: torch.Tensor | None, dtype: torch.dtype | None = None) -> int | None:
    """Device pointer of a contiguous CUDA tensor (None stays NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NrfError("nerfpp_b200 ops need CUDA tensors (there is no CPU path)")
    if not t.is_contiguous():
        raise NrfError("tensor must be contiguous")
    if dtype is not None and t.dtype != dtype:
        raise NrfError(f"expected {dtype}, got {t.dtype}")
    return t.data_ptr()


def host_floats(values) -> C.Array:
    vals = [float(v) for v in values]
    return (c_float * len(vals))(*vals)


def launch_count() -> int:
    return int(lib().nrf_launch_count())
