"""Thin functional wrappers: torch tensors in, one C-ABI call each (include/nerfpp_b200.h), torch tensors out.

Used by tests/, bench.py and the Python pipeline (nerfpp_b200/pipeline.py).  Nothing is computed in Python/torch
here: allocation + pointer plumbing only.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import torch

from . import cabi
from .cabi import check, lib, ptr, stream

f32, f16, bf16, i32, u8 = torch.float32, torch.float16, torch.bfloat16, torch.int32, torch.uint8


class KernelTimer:
    """Optional per-kernel CUDA-event timing on the launching stream (bench.py roofline / breakdown).
    `only`: restrict to these entry names (without the nrf_ prefix) so the timed region carries two events per step."""

    def __init__(self, only=None, external=False):
        self.only = set(only) if only else None
        self.external = external      # events that may be recorded inside a CUDA-graph capture and read after a replay
        self.records: dict[str, list] = {}

    def summary(self) -> dict:
        """name -> (launches, total_ms); call after a stream synchronize."""
        return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in self.records.items()}


_timer: KernelTimer | None = None


def set_timer(t: KernelTimer | None) -> None:
    global _timer
    _timer = t


def _run(name: str, call) -> None:
    t = _timer
    if t is not None and (t.only is None or name in t.only):
        e0, e1 = torch.cuda.Event(enable_timing=True, external=t.external), torch.cuda.Event(enable_timing=True, external=t.external)
        e0.record()
        status = call()
        e1.record()
        t.records.setdefault(name, []).append((e0, e1))
    else:
        status = call()
    check(status)


@dataclass
class HashGridSpec:
    """Mirror of the public members of CuHashEmbedderImpl (reference src/CuHashEmbedder.h:12-27)."""
    bounding_box: tuple  # 6 floats
    primes: torch.Tensor           # int32 [L, V, 3]      ("<name>_primes")
    biases: torch.Tensor           # f32  [L*V, 3]        ("<name>_biases")
    feat_local_idx: torch.Tensor   # int32 [L]            ("<name>_feat_local_idx")
    feat_local_size: torch.Tensor  # int32 [L]            ("<name>_feat_local_size")
    n_levels: int = 16
    n_features: int = 2
    log2_hashmap_size: int = 19
    base_resolution: int = 16
    finest_resolution: int = 512
    n_volumes: int = 1
    level_scale: torch.Tensor | None = None

    def table_scalars(self) -> int:
        return (1 << self.log2_hashmap_size) * self.n_levels * self.n_features

    def used_scalars(self) -> int:
        """Scalars the kernels can touch: level offsets are in scalars (reference quirk), so levels overlap."""
        idx = self.feat_local_idx.cpu().tolist()
        size = self.feat_local_size.cpu().tolist()
        return max(o + s * self.n_features for o, s in zip(idx, size))

    def c_struct(self) -> cabi.HashGrid:
        if self.level_scale is None:
            self.level_scale = hash_level_scales(self.base_resolution, self.finest_resolution, self.n_levels, self.primes.device)
        g = cabi.HashGrid()
        g.n_levels, g.n_features, g.n_volumes = self.n_levels, self.n_features, self.n_volumes
        g.base_resolution, g.finest_resolution = self.base_resolution, self.finest_resolution
        for k in range(3):
            g.box_min[k] = float(self.bounding_box[k])
            g.box_max[k] = float(self.bounding_box[3 + k])
        g.primes = ptr(self.primes, i32)
        g.biases = ptr(self.biases, f32)
        g.feat_local_idx = ptr(self.feat_local_idx, i32)
        g.feat_local_size = ptr(self.feat_local_size, i32)
        g.level_scale = ptr(self.level_scale, f32)
        g.table_scalars = self.table_scalars()
        return g


def hash_level_scales(base_res: int, finest_res: int, n_levels: int, device) -> torch.Tensor:
    out = torch.empty(n_levels, dtype=f32, device=device)
    _run("hash_level_scales", lambda: lib().nrf_hash_level_scales(base_res, finest_res, n_levels, ptr(out), stream()))
    return out


def hash_cells(grid: HashGridSpec, points: torch.Tensor, clamp: bool = True):
    """(addr int64 [N,L,8], weights f32 [N,L,8]): the scalar addresses / trilinear weights the encode kernels use (inspection entry)."""
    n = points.shape[0]
    addr = torch.empty((n, grid.n_levels, 8), dtype=torch.int64, device=points.device)
    w = torch.empty((n, grid.n_levels, 8), dtype=f32, device=points.device)
    g = grid.c_struct()
    _run("hash_cells", lambda: lib().nrf_hash_cells(C.byref(g), ptr(points, f32), n, int(clamp), ptr(addr), ptr(w), stream()))
    return addr, w


def table_to_half(table: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    if out is None:
        out = torch.empty(table.shape, dtype=f16, device=table.device)
    _run("table_to_half", lambda: lib().nrf_table_to_half(ptr(table, f32), ptr(out, f16), table.numel(), stream()))
    return out


def hash_encode_fwd(grid: HashGridSpec, table_f16: torch.Tensor, points: torch.Tensor, clamp: bool = True,
                    out_f16: bool = False, want_keep: bool = True):
    n = points.shape[0]
    d = grid.n_levels * grid.n_features
    out = torch.empty((n, d), dtype=f16 if out_f16 else f32, device=points.device)
    keep = torch.empty(n, dtype=u8, device=points.device) if (clamp and want_keep) else None
    g = grid.c_struct()
    _run("hash_encode_fwd", lambda: lib().nrf_hash_encode_fwd(C.byref(g), ptr(table_f16, f16), ptr(points, f32), n, int(clamp), ptr(keep),
                                    ptr(out), cabi.ENC_F16 if out_f16 else cabi.ENC_F32, stream()))
    return out, keep


def hash_encode_bwd(grid: HashGridSpec, points: torch.Tensor, grad_enc: torch.Tensor, grad_table: torch.Tensor,
                    clamp: bool = True) -> torch.Tensor:
    n = points.shape[0]
    layout = {f32: cabi.GRAD_F32, bf16: cabi.GRAD_BF16}[grad_enc.dtype]
    g = grid.c_struct()
    _run("hash_encode_bwd", lambda: lib().nrf_hash_encode_bwd(C.byref(g), ptr(points, f32), n, int(clamp), ptr(grad_enc), layout,
                                    ptr(grad_table, f32), stream()))
    return grad_table


@dataclass
class PointJitter:
    """Per-sample perturbations of the shipped training configuration, applied inside the ray encode kernels (struct nrf_point_jitter).
    cone_angle: [1] (one scalar) or [R] device tensor, None = thin rays; rand_r / rand_theta [R,S] uniforms (TangentScatter's two torch.rand
    draws); clamp_to_box: TangentScatter's clamp into the grid's box; sp_noise [R,S,3] standard normal and sp_alpha a [1] device tensor:
    stochastic preconditioning (None = off)."""
    cone_angle: torch.Tensor | None = None
    rand_r: torch.Tensor | None = None
    rand_theta: torch.Tensor | None = None
    clamp_to_box: bool = True
    sp_noise: torch.Tensor | None = None
    sp_alpha: torch.Tensor | None = None

    def c_struct(self) -> cabi.PointJitter:
        j = cabi.PointJitter()
        j.cone_angle = ptr(self.cone_angle, f32)
        j.cone_stride = 0 if self.cone_angle is None or self.cone_angle.numel() == 1 else 1
        j.rand_r, j.rand_theta = ptr(self.rand_r, f32), ptr(self.rand_theta, f32)
        j.clamp_to_box = int(self.clamp_to_box)
        j.sp_noise, j.sp_alpha = ptr(self.sp_noise, f32), ptr(self.sp_alpha, f32)
        return j


def hash_encode_rays_fwd(grid: HashGridSpec, table_f16: torch.Tensor, ray_batch: torch.Tensor, z: torch.Tensor, clamp: bool = True,
                         out_f16: bool = True, reuse=None, ray_group: int = 1, jitter: PointJitter | None = None):
    """Fused point generation + encode.  reuse = (perm [R,S] int16, enc_prev [R*S_prev, D] | None, keep_prev [R*S_prev] | None, S_prev).
    ray_group > 1: the kernel walks the same sample of ray_group neighbouring rays together (rays of a rendered frame); same results.
    jitter: the points are perturbed in-kernel (nrf_hash_encode_rays_jitter_fwd); not combinable with reuse / ray_group."""
    r, s = z.shape
    d = grid.n_levels * grid.n_features
    out = torch.empty((r * s, d), dtype=f16 if out_f16 else f32, device=z.device)
    keep = torch.empty(r * s, dtype=u8, device=z.device) if clamp else None
    g = grid.c_struct()
    if jitter is not None:
        if reuse is not None or ray_group != 1:
            raise cabi.NrfError("jittered points take neither row reuse nor ray grouping")
        j = jitter.c_struct()
        _run("hash_encode_fwd", lambda: lib().nrf_hash_encode_rays_jitter_fwd(C.byref(g), ptr(table_f16, f16), ptr(ray_batch, f32), ray_batch.shape[1],
                                        ptr(z, f32), r, s, int(clamp), ptr(keep), ptr(out), cabi.ENC_F16 if out_f16 else cabi.ENC_F32, C.byref(j), stream()))
        return out, keep
    src, enc_prev, keep_prev, s_prev = reuse if reuse is not None else (None, None, None, 0)
    _run("hash_encode_fwd", lambda: lib().nrf_hash_encode_rays_fwd_grouped(C.byref(g), ptr(table_f16, f16), ptr(ray_batch, f32), ray_batch.shape[1], ptr(z, f32),
                                    r, s, int(clamp), ptr(keep), ptr(out), cabi.ENC_F16 if out_f16 else cabi.ENC_F32, ptr(src, torch.int16) if src is not None else None,
                                    ptr(enc_prev), ptr(keep_prev), s_prev, ray_group, stream()))
    return out, keep


def hash_encode_rays_bwd(grid: HashGridSpec, ray_batch: torch.Tensor, z: torch.Tensor, grad_enc: torch.Tensor, grad_table: torch.Tensor,
                         clamp: bool = True, jitter: PointJitter | None = None) -> torch.Tensor:
    """jitter: the forward's perturbed points, re-derived from the same variates (nrf_hash_encode_rays_jitter_bwd)."""
    r, s = z.shape
    layout = {f32: cabi.GRAD_F32, bf16: cabi.GRAD_BF16}[grad_enc.dtype]
    g = grid.c_struct()
    if jitter is not None:
        j = jitter.c_struct()
        _run("hash_encode_bwd", lambda: lib().nrf_hash_encode_rays_jitter_bwd(C.byref(g), ptr(ray_batch, f32), ray_batch.shape[1], ptr(z, f32), r, s,
                                        int(clamp), ptr(grad_enc), layout, ptr(grad_table, f32), C.byref(j), stream()))
        return grad_table
    _run("hash_encode_bwd", lambda: lib().nrf_hash_encode_rays_bwd(C.byref(g), ptr(ray_batch, f32), ray_batch.shape[1], ptr(z, f32), r, s, int(clamp),
                                    ptr(grad_enc), layout, ptr(grad_table, f32), stream()))
    return grad_table


def sh_encode(dirs: torch.Tensor, degree: int) -> torch.Tensor:
    """dirs: contiguous [N,3], or a column slice [:, a:a+3] of a contiguous [N,K] matrix (read in place, strided)."""
    n = dirs.shape[0]
    if dirs.dim() != 2 or dirs.shape[1] != 3 or dirs.stride(1) != 1 or dirs.dtype != f32 or not dirs.is_cuda:
        raise cabi.NrfError("sh_encode needs a CUDA fp32 [N,3] tensor with unit inner stride")
    out = torch.empty((n, degree * degree), dtype=f32, device=dirs.device)
    _run("sh_encode_fwd", lambda: lib().nrf_sh_encode_fwd(dirs.data_ptr(), dirs.stride(0) if n > 1 else 3, n, degree, ptr(out), stream()))
    return out


def posenc(x: torch.Tensor, freq_bands, include_input: bool = True) -> torch.Tensor:
    n, d = x.shape
    nf = len(freq_bands)
    out = torch.empty((n, d * (int(include_input) + 2 * nf)), dtype=f32, device=x.device)
    _run("posenc_fwd", lambda: lib().nrf_posenc_fwd(ptr(x, f32), n, d, nf, cabi.host_floats(freq_bands), int(include_input), ptr(out), stream()))
    return out


def mlp_shape(input_ch=32, input_ch_views=16, hidden=64, geo=15, hidden_color=64, num_layers=2, num_layers_color=3):
    return cabi.MlpSmallShape(input_ch, input_ch_views, hidden, geo, hidden_color, num_layers, num_layers_color)


def mlp_small_pack(params_flat: torch.Tensor, shape=None, out: torch.Tensor | None = None) -> torch.Tensor:
    shape = shape or mlp_shape()
    nbytes = lib().nrf_mlp_small_packed_bytes(C.byref(shape))
    if nbytes < 0:
        check(-3)
    if out is None:
        out = torch.empty(nbytes, dtype=u8, device=params_flat.device)
    _run("mlp_small_pack", lambda: lib().nrf_mlp_small_pack(C.byref(shape), ptr(params_flat, f32), ptr(out), stream()))
    return out


def mlp_small_fwd(packed: torch.Tensor, enc: torch.Tensor, ray_sh: torch.Tensor | None, samples_per_ray: int,
                  keep: torch.Tensor | None, shape=None, out: torch.Tensor | None = None, ray_bias: bool = False) -> torch.Tensor:
    """ray_bias: ray_sh is the per-ray view term [R,64] of mlp_small_view_bias_fwd (NRF_MLP_IN_ENC16_RAYBIAS: any view width 1..64)."""
    shape = shape or mlp_shape()
    n = enc.shape[0]
    kind = (cabi.MLP_IN_ENC16_RAYBIAS if ray_bias else cabi.MLP_IN_ENC16_RAYDIRS) if enc.dtype == f16 else cabi.MLP_IN_F32_CAT
    if out is None:
        out = torch.empty((n, 4), dtype=f32, device=enc.device)
    _run("mlp_small_fwd", lambda: lib().nrf_mlp_small_fwd(C.byref(shape), ptr(packed), kind, ptr(enc), ptr(ray_sh), samples_per_ray, ptr(keep),
                                  n, ptr(out, f32), stream()))
    return out


def mlp_small_fwd_importance(packed: torch.Tensor, enc_merged: torch.Tensor, ray_sh: torch.Tensor, keep_merged: torch.Tensor | None,
                             perm: torch.Tensor, n_importance: int, raw_merged: torch.Tensor, shape=None, ray_bias: bool = False) -> torch.Tensor:
    """Evaluate the importance samples only (rows perm[:, :n_importance] of the merged arrays) into raw_merged, whose coarse-sample
    rows sample_pdf_merge(raw_coarse=...) already holds.  Same bits as mlp_small_fwd over all merged rows."""
    shape = shape or mlp_shape()
    r, t = perm.shape
    assert enc_merged.dtype == f16 and enc_merged.shape[0] == r * t and raw_merged.shape[0] == r * t
    kind = cabi.MLP_IN_ENC16_RAYBIAS if ray_bias else cabi.MLP_IN_ENC16_RAYDIRS
    _run("mlp_small_fwd", lambda: lib().nrf_mlp_small_fwd_importance(C.byref(shape), ptr(packed), kind, ptr(enc_merged, f16), ptr(ray_sh, f32),
                                  ptr(keep_merged), ptr(perm, torch.int16), r, n_importance, t, ptr(raw_merged, f32), stream()))
    return raw_merged


def mlp_small_view_bias_fwd(packed: torch.Tensor, ray_sh: torch.Tensor, shape=None, out: torch.Tensor | None = None,
                            grad_bias_zero: torch.Tensor | None = None) -> torch.Tensor:
    """The view term of the colour net's first layer, once per ray: ray_sh [R,V] -> bias [R,64] fp32 (and grad_bias_zero [R,64] := 0)."""
    shape = shape or mlp_shape()
    r = ray_sh.shape[0]
    assert ray_sh.shape[1] == shape.input_ch_views
    if out is None:
        out = torch.empty((r, 64), dtype=f32, device=ray_sh.device)
    _run("mlp_small_view_bias", lambda: lib().nrf_mlp_small_view_bias_fwd(C.byref(shape), ptr(packed), ptr(ray_sh, f32), r, ptr(out, f32),
                                        ptr(grad_bias_zero, f32) if grad_bias_zero is not None else None, stream()))
    return out


def mlp_small_view_bias_bwd(ray_sh: torch.Tensor, grad_bias: torch.Tensor, grad_params: torch.Tensor, shape=None) -> None:
    """grad_params[view columns of color_net_0] += grad_bias^T ray_sh."""
    shape = shape or mlp_shape()
    _run("mlp_small_view_bias", lambda: lib().nrf_mlp_small_view_bias_bwd(C.byref(shape), ptr(ray_sh, f32), ptr(grad_bias, f32), ray_sh.shape[0],
                                        ptr(grad_params, f32), stream()))


def mlp_small_bwd(packed: torch.Tensor, enc: torch.Tensor, ray_sh: torch.Tensor | None, samples_per_ray: int,
                  keep: torch.Tensor | None, grad_raw: torch.Tensor, grad_params: torch.Tensor, want_grad_in: bool = True,
                  shape=None, grad_in: torch.Tensor | None = None, grad_bias: torch.Tensor | None = None):
    """grad_bias [R,64] (accumulated into) selects NRF_MLP_IN_ENC16_RAYBIAS: ray_sh is then the per-ray view term."""
    shape = shape or mlp_shape()
    n = enc.shape[0]
    if enc.dtype == f16:
        kind = cabi.MLP_IN_ENC16_RAYBIAS if grad_bias is not None else cabi.MLP_IN_ENC16_RAYDIRS
        if want_grad_in and grad_in is None:
            grad_in = torch.empty((n, 32), dtype=bf16, device=enc.device)
    else:
        kind = cabi.MLP_IN_F32_CAT
        if want_grad_in and grad_in is None:
            grad_in = torch.empty((n, 48), dtype=f32, device=enc.device)
    _run("mlp_small_bwd", lambda: lib().nrf_mlp_small_bwd_raybias(C.byref(shape), ptr(packed), kind, ptr(enc), ptr(ray_sh), samples_per_ray, ptr(keep), n,
                                  ptr(grad_raw, f32), ptr(grad_in) if want_grad_in else None, ptr(grad_params, f32),
                                  ptr(grad_bias, f32) if grad_bias is not None else None, stream()))
    return grad_in


def composite_fwd(raw: torch.Tensor, z: torch.Tensor, rays_d: torch.Tensor, white_bkgr: bool = False,
                  noise: torch.Tensor | None = None, raw_noise_std: float = 0.0, want_weights: bool = True):
    r, s, c = raw.shape
    dev = raw.device
    rgb = torch.empty((r, 3), dtype=f32, device=dev)
    depth = torch.empty(r, dtype=f32, device=dev)
    disp = torch.empty(r, dtype=f32, device=dev)
    acc = torch.empty(r, dtype=f32, device=dev)
    weights = torch.empty((r, s), dtype=f32, device=dev) if want_weights else None
    _run("composite_fwd", lambda: lib().nrf_composite_fwd(ptr(raw, f32), c, ptr(z, f32), ptr(rays_d, f32), ptr(noise), raw_noise_std, int(white_bkgr),
                                  r, s, ptr(rgb), ptr(depth), ptr(disp), ptr(acc), ptr(weights), stream()))
    return {"rgb": rgb, "depth": depth, "disp": disp, "acc": acc, "weights": weights}


def composite_bwd(raw, z, rays_d, white_bkgr=False, noise=None, raw_noise_std=0.0, g_rgb=None, g_depth=None, g_disp=None,
                  g_acc=None, g_weights=None, out: torch.Tensor | None = None) -> torch.Tensor:
    r, s, c = raw.shape
    if out is None:
        out = torch.empty((r, s, 4), dtype=f32, device=raw.device)
    _run("composite_bwd", lambda: lib().nrf_composite_bwd(ptr(raw, f32), c, ptr(z, f32), ptr(rays_d, f32), ptr(noise), raw_noise_std, int(white_bkgr),
                                  r, s, ptr(g_rgb), ptr(g_depth), ptr(g_disp), ptr(g_acc), ptr(g_weights), ptr(out), stream()))
    return out


def composite_huber_bwd(raw, z, rays_d, target, loss_out, white_bkgr=False, noise=None, raw_noise_std=0.0, delta=1.0, grad_scale=1.0, want_rgb=True):
    """composite_fwd + huber_fwd_bwd + composite_bwd(g_rgb) of a training step as ONE launch: returns (d_raw [R,S,4], rgb [R,3] | None)."""
    r, s, c = raw.shape
    d_raw = torch.empty((r, s, 4), dtype=f32, device=raw.device)
    rgb = torch.empty((r, 3), dtype=f32, device=raw.device) if want_rgb else None
    _run("composite_huber_bwd", lambda: lib().nrf_composite_huber_bwd(ptr(raw, f32), c, ptr(z, f32), ptr(rays_d, f32), ptr(noise), raw_noise_std, int(white_bkgr),
                                                                      r, s, ptr(target, f32), delta, grad_scale, ptr(loss_out, f32), ptr(rgb), ptr(d_raw), stream()))
    return d_raw, rgb


def sample_pdf(bins: torch.Tensor, weights: torch.Tensor, u: torch.Tensor) -> torch.Tensor:
    r, b = bins.shape
    per_ray = u.dim() == 2
    n = u.shape[-1]
    out = torch.empty((r, n), dtype=f32, device=bins.device)
    _run("sample_pdf", lambda: lib().nrf_sample_pdf(ptr(bins, f32), ptr(weights, f32), b, ptr(u, f32), int(per_ray), r, n, ptr(out), stream()))
    return out


def sample_pdf_merge(z_coarse: torch.Tensor, weights: torch.Tensor, u: torch.Tensor, want_samples: bool = False, want_perm: bool = False,
                     raw_coarse: torch.Tensor | None = None):
    """z_merged [, z_samples] [, perm] [, raw_merged].  raw_coarse [R*S, 4] (u shared by the rays): the coarse pass's raw rows are
    moved to their merged positions in raw_merged [R*(S+N), 4]; the other rows are left for mlp_small_fwd_importance."""
    r, s = z_coarse.shape
    per_ray = u.dim() == 2
    n = u.shape[-1]
    merged = torch.empty((r, s + n), dtype=f32, device=z_coarse.device)
    samples = torch.empty((r, n), dtype=f32, device=z_coarse.device) if want_samples else None
    src = torch.empty((r, s + n), dtype=torch.int16, device=z_coarse.device) if want_perm else None
    raw = torch.empty((r * (s + n), 4), dtype=f32, device=z_coarse.device) if raw_coarse is not None else None
    _run("sample_pdf_merge", lambda: lib().nrf_sample_pdf_merge_rows(ptr(z_coarse, f32), ptr(weights, f32), ptr(u, f32), int(per_ray), r, s, n, ptr(samples),
                                     ptr(merged), ptr(src), ptr(raw_coarse, f32), ptr(raw), stream()))
    out = (merged,) + ((samples,) if want_samples else ()) + ((src,) if want_perm else ()) + ((raw,) if raw is not None else ())
    return out if len(out) > 1 else merged


def get_rays(h: int, w: int, K, c2w, row_begin: int = 0, row_end: int | None = None, device="cuda"):
    row_end = h if row_end is None else row_end
    n = (row_end - row_begin) * w
    rays_o = torch.empty((n, 3), dtype=f32, device=device)
    rays_d = torch.empty((n, 3), dtype=f32, device=device)
    kh = cabi.host_floats(torch.as_tensor(K, dtype=f32).reshape(-1).tolist())
    ch = cabi.host_floats(torch.as_tensor(c2w, dtype=f32)[:3, :4].reshape(-1).tolist())
    _run("get_rays", lambda: lib().nrf_get_rays(h, w, kh, ch, row_begin, row_end, ptr(rays_o), ptr(rays_d), stream()))
    return rays_o, rays_d


def rays_prepare(rays_o: torch.Tensor, rays_d: torch.Tensor, bbox, near_plane: float = 0.0, use_viewdirs: bool = True) -> torch.Tensor:
    n = rays_o.shape[0]
    out = torch.empty((n, 11 if use_viewdirs else 8), dtype=f32, device=rays_o.device)
    _run("rays_prepare", lambda: lib().nrf_rays_prepare(ptr(rays_o, f32), ptr(rays_d, f32), n, cabi.host_floats(bbox), near_plane, int(use_viewdirs),
                                 ptr(out), stream()))
    return out


def ray_setup(rays_o: torch.Tensor, rays_d: torch.Tensor, bbox, near_plane: float, t_vals: torch.Tensor, sh_degree: int | None, lin_disp: bool = False,
              zero_scalar: torch.Tensor | None = None):
    """rays_prepare + z_sample + sh_encode(viewdirs) as one launch: (ray_batch [R,11], z [R,S], ray_sh [R,deg^2] or None)."""
    r, s = rays_o.shape[0], t_vals.shape[0]
    dev = rays_o.device
    ray_batch = torch.empty((r, 11), dtype=f32, device=dev)
    z = torch.empty((r, s), dtype=f32, device=dev)
    ray_sh = torch.empty((r, sh_degree * sh_degree), dtype=f32, device=dev) if sh_degree else None
    _run("ray_setup", lambda: lib().nrf_ray_setup(ptr(rays_o, f32), ptr(rays_d, f32), r, cabi.host_floats(bbox), near_plane, ptr(t_vals, f32), s, int(lin_disp),
                                                  sh_degree or 0, ptr(ray_batch), ptr(z), ptr(ray_sh), ptr(zero_scalar), stream()))
    return ray_batch, z, ray_sh


def _cam(K, c2w):
    return (cabi.host_floats(torch.as_tensor(K, dtype=f32).reshape(-1).tolist()), cabi.host_floats(torch.as_tensor(c2w, dtype=f32)[:3, :4].reshape(-1).tolist()))


def ray_batch(pix_hw: torch.Tensor, K, c2w, image: torch.Tensor | None = None):
    """NeRFDataset::GetRayBatch on the device: pix_hw int32 [R,2] (row, col) -> (rays_o, rays_d, target | None, cone_angle)."""
    r = pix_hw.shape[0]
    rays_o = torch.empty((r, 3), dtype=f32, device=pix_hw.device)
    rays_d = torch.empty((r, 3), dtype=f32, device=pix_hw.device)
    target = torch.empty((r, image.shape[2]), dtype=f32, device=pix_hw.device) if image is not None else None
    kh, ch = _cam(K, c2w)
    cone = C.c_float(0.0)
    h, w, c = image.shape if image is not None else (0, 0, 0)
    _run("ray_batch", lambda: lib().nrf_ray_batch(ptr(pix_hw, i32), r, kh, ch, ptr(image), h, w, c, ptr(rays_o), ptr(rays_d), ptr(target), C.byref(cone), stream()))
    return rays_o, rays_d, target, float(cone.value)


def ray_setup_pixels(pix_hw: torch.Tensor, K, c2w, image: torch.Tensor | None, bbox, near_plane: float, t_vals: torch.Tensor, sh_degree: int | None,
                     lin_disp: bool = False, zero_scalar: torch.Tensor | None = None, cam=None):
    """ray_batch + ray_setup as one launch: (rays_o, rays_d, target | None, ray_batch [R,11], z [R,S], ray_sh | None)."""
    r, s = pix_hw.shape[0], t_vals.shape[0]
    dev = pix_hw.device
    rays_o = torch.empty((r, 3), dtype=f32, device=dev)
    rays_d = torch.empty((r, 3), dtype=f32, device=dev)
    target = torch.empty((r, image.shape[2]), dtype=f32, device=dev) if image is not None else None
    rb = torch.empty((r, 11), dtype=f32, device=dev)
    z = torch.empty((r, s), dtype=f32, device=dev)
    ray_sh = torch.empty((r, sh_degree * sh_degree), dtype=f32, device=dev) if sh_degree else None
    kh, ch = cam if cam is not None else _cam(K, c2w)
    h, w, c = image.shape if image is not None else (0, 0, 0)
    _run("ray_setup", lambda: lib().nrf_ray_setup_pixels(ptr(pix_hw, i32), r, kh, ch, ptr(image), h, w, c, cabi.host_floats(bbox), near_plane, ptr(t_vals, f32), s,
                                                         int(lin_disp), sh_degree or 0, ptr(rays_o), ptr(rays_d), ptr(target), ptr(rb), ptr(z), ptr(ray_sh),
                                                         ptr(zero_scalar), stream()))
    return rays_o, rays_d, target, rb, z, ray_sh


def z_sample(ray_batch: torch.Tensor, t_vals: torch.Tensor, lin_disp: bool = False) -> torch.Tensor:
    r, stride = ray_batch.shape
    s = t_vals.shape[0]
    z = torch.empty((r, s), dtype=f32, device=ray_batch.device)
    _run("z_sample", lambda: lib().nrf_z_sample(ptr(ray_batch, f32), stride, ptr(t_vals, f32), r, s, int(lin_disp), ptr(z), stream()))
    return z


def sample_points(ray_batch: torch.Tensor, z: torch.Tensor) -> torch.Tensor:
    r, stride = ray_batch.shape
    s = z.shape[1]
    pts = torch.empty((r, s, 3), dtype=f32, device=z.device)
    _run("sample_points", lambda: lib().nrf_sample_points(ptr(ray_batch, f32), stride, ptr(z, f32), r, s, ptr(pts), stream()))
    return pts


def tangent_scatter(pts: torch.Tensor, z: torch.Tensor, cone_angle: torch.Tensor, rays_d: torch.Tensor, rand_r: torch.Tensor, rand_theta: torch.Tensor,
                    bbox=None) -> torch.Tensor:
    """TangentScatter in place on pts [R,S,3]; cone_angle: one-element tensor (shared) or [R]; rand_* [R,S] uniform variates."""
    r, s = z.shape
    stride = 0 if cone_angle.numel() == 1 else 1
    _run("tangent_scatter", lambda: lib().nrf_tangent_scatter(ptr(pts, f32), ptr(z, f32), ptr(cone_angle, f32), stride, ptr(rays_d, f32), rays_d.shape[1],
                                                              ptr(rand_r, f32), ptr(rand_theta, f32), cabi.host_floats(bbox) if bbox is not None else None, r, s, stream()))
    return pts


def precondition_points(pts: torch.Tensor, noise: torch.Tensor, alpha: float, bbox) -> torch.Tensor:
    """Stochastic preconditioning + ReflectBoundary in place on pts [..., 3]."""
    _run("precondition_points", lambda: lib().nrf_precondition_points(ptr(pts, f32), ptr(noise, f32), alpha, cabi.host_floats(bbox), pts.numel() // 3, stream()))
    return pts


def huber_fwd_bwd(pred: torch.Tensor, target: torch.Tensor, loss_out: torch.Tensor, grad: torch.Tensor | None,
                  delta: float = 1.0, grad_scale: float = 1.0) -> None:
    _run("huber_fwd_bwd", lambda: lib().nrf_huber_fwd_bwd(ptr(pred, f32), ptr(target, f32), pred.numel(), delta, grad_scale, ptr(loss_out, f32),
                                  ptr(grad), stream()))


def adam_step(param, grad, exp_avg, exp_avg_sq, lr, step, beta1=0.9, beta2=0.99, eps=1e-15, grad_scale=1.0,
              zero_grad=True, shadow_f16: torch.Tensor | None = None, n: int | None = None) -> None:
    n = param.numel() if n is None else n
    _run("adam_step", lambda: lib().nrf_adam_step(ptr(param, f32), ptr(grad, f32), ptr(exp_avg, f32), ptr(exp_avg_sq, f32), n, lr, beta1, beta2, eps,
                              step, grad_scale, int(zero_grad), ptr(shadow_f16), stream()))


def adam_schedule_advance(sched_state: torch.Tensor, lr0: float, decay_rate: float, decay_steps: float, beta1=0.9, beta2=0.99) -> None:
    """sched_state: 16-byte device record (4 x 32-bit, zero-initialised) — see nrf_adam_schedule_advance."""
    _run("adam_schedule_advance", lambda: lib().nrf_adam_schedule_advance(ptr(sched_state), lr0, decay_rate, decay_steps, beta1, beta2, stream()))


def adam_step_scheduled(param, grad, exp_avg, exp_avg_sq, sched_state: torch.Tensor, beta1=0.9, beta2=0.99, eps=1e-15, grad_scale=1.0,
                        zero_grad=True, shadow_f16: torch.Tensor | None = None) -> None:
    _run("adam_step", lambda: lib().nrf_adam_step_scheduled(ptr(param, f32), ptr(grad, f32), ptr(exp_avg, f32), ptr(exp_avg_sq, f32), param.numel(),
                              ptr(sched_state), beta1, beta2, eps, grad_scale, int(zero_grad), ptr(shadow_f16), stream()))


def render_rays_fwd(grid: HashGridSpec, table_f16, packed, rays_o, rays_d, t_vals, u, bbox, white_bkgr=False, sh_degree=4, near_plane=0.0,
                    lin_disp=False, want_weights=False, want_z=False, workspace: torch.Tensor | None = None, shape=None, tile=None, ray_batch=None):
    """RenderRays (inference) as ONE C-ABI call; returns (maps, workspace) — pass the workspace back in to reuse it.
    tile = (K, c2w, img_w, first_pixel, n_rays): the rays are pixels first_pixel .. first_pixel + n_rays of that view in GetRays order and are
    generated inside the call (nrf_render_tile_fwd); ray_batch [R, >= 11]: a prepared batch [o d near far viewdirs] (nrf_render_raybatch_fwd).
    rays_o / rays_d are ignored in both cases."""
    shape = shape or mlp_shape()
    dev = table_f16.device
    r = tile[4] if tile is not None else (ray_batch.shape[0] if ray_batch is not None else rays_o.shape[0])
    s, n = t_vals.shape[0], u.shape[0]
    cfg = cabi.RenderConfig(s, n, int(white_bkgr), int(lin_disp), sh_degree, float(near_plane))
    for k in range(6):
        cfg.bbox[k] = float(bbox[k])
    g = grid.c_struct()
    need = lib().nrf_render_rays_workspace_bytes(C.byref(cfg), C.byref(g), r)
    if need < 0:
        check(-1)
    if workspace is None or workspace.numel() < need:
        workspace = torch.empty(max(need, 256), dtype=u8, device=dev)
    rgb = torch.empty((r, 3), dtype=f32, device=dev)
    depth, disp, acc = (torch.empty(r, dtype=f32, device=dev) for _ in range(3))
    weights = torch.empty((r, s + n), dtype=f32, device=dev) if want_weights else None
    z = torch.empty((r, s + n), dtype=f32, device=dev) if want_z else None
    if ray_batch is not None:
        _run("render_rays_fwd", lambda: lib().nrf_render_raybatch_fwd(C.byref(cfg), C.byref(g), ptr(table_f16, f16), C.byref(shape), ptr(packed), ptr(ray_batch, f32),
                                        ray_batch.shape[1], r, ptr(t_vals, f32), ptr(u, f32), ptr(workspace), workspace.numel(), ptr(rgb), ptr(depth),
                                        ptr(disp), ptr(acc), ptr(weights), ptr(z), stream()))
    elif tile is not None:
        kh, ch = _cam(tile[0], tile[1])
        _run("render_rays_fwd", lambda: lib().nrf_render_tile_fwd(C.byref(cfg), C.byref(g), ptr(table_f16, f16), C.byref(shape), ptr(packed), kh, ch, int(tile[2]),
                                        int(tile[3]), r, ptr(t_vals, f32), ptr(u, f32), ptr(workspace), workspace.numel(), ptr(rgb), ptr(depth),
                                        ptr(disp), ptr(acc), ptr(weights), ptr(z), stream()))
    else:
        _run("render_rays_fwd", lambda: lib().nrf_render_rays_fwd(C.byref(cfg), C.byref(g), ptr(table_f16, f16), C.byref(shape), ptr(packed), ptr(rays_o, f32),
                                        ptr(rays_d, f32), r, ptr(t_vals, f32), ptr(u, f32), ptr(workspace), workspace.numel(), ptr(rgb), ptr(depth),
                                        ptr(disp), ptr(acc), ptr(weights), ptr(z), stream()))
    return {"rgb": rgb, "depth": depth, "disp": disp, "acc": acc, "weights": weights, "z": z}, workspace


def adam_step_sharded(peer_group, param, exp_avg, exp_avg_sq, n_sharded: int, sched_state, beta1=0.9, beta2=0.99, eps=1e-15, grad_scale=1.0) -> None:
    """reduce-scatter + Adam + fp16 shadow all-gather over peer memory (nrf_adam_step_sharded); peer_group: cabi.PeerGroup."""
    _run("adam_step", lambda: lib().nrf_adam_step_sharded(C.byref(peer_group), ptr(param, f32), ptr(exp_avg, f32), ptr(exp_avg_sq, f32), n_sharded,
                              param.numel(), ptr(sched_state), beta1, beta2, eps, grad_scale, stream()))


def mlp_nerf_shape(depth=8, width=256, input_ch=63, input_ch_views=27, skip_layer=4, use_viewdirs=True):
    return cabi.MlpNerfShape(depth, width, input_ch, input_ch_views, skip_layer, int(use_viewdirs))


def _mlp_nerf_ptrs(p: dict) -> "cabi.MlpNerfWeights":
    """nrf_mlp_nerf_weights / nrf_mlp_nerf_grads (same field layout) from the reference's registered names."""
    w = cabi.MlpNerfWeights()
    for i in range(8):
        w.pts_w[i] = ptr(p[f"model_pts_linears_{i}.weight"], f32)
        w.pts_b[i] = ptr(p[f"model_pts_linears_{i}.bias"], f32)
    for name in ("feature", "alpha", "rgb"):
        setattr(w, f"{name}_w", ptr(p[f"model_{name}_linear.weight"], f32))
        setattr(w, f"{name}_b", ptr(p[f"model_{name}_linear.bias"], f32))
    w.views_w, w.views_b = ptr(p["model_views_linears_0.weight"], f32), ptr(p["model_views_linears_0.bias"], f32)
    return w


def mlp_nerf_pack(p: dict, shape=None, out: torch.Tensor | None = None, train: bool = False) -> torch.Tensor:
    """p: the reference's registered names ('model_pts_linears_<i>.weight' ... 'model_rgb_linear.bias', src/NeRF.cpp:76-89) ->
    contiguous fp32 CUDA tensors.  Returns the packed UMMA-operand blob (+ fp32 biases): fp16 for nrf_mlp_nerf_fwd, bf16
    (train=True) for nrf_mlp_nerf_fwd_train / nrf_mlp_nerf_bwd."""
    shape = shape or mlp_nerf_shape()
    nbytes = lib().nrf_mlp_nerf_packed_bytes(C.byref(shape))
    if nbytes < 0:
        check(-3)
    w = _mlp_nerf_ptrs(p)
    if out is None:
        out = torch.empty(nbytes, dtype=u8, device=p["model_rgb_linear.bias"].device)
    fn = lib().nrf_mlp_nerf_pack_train if train else lib().nrf_mlp_nerf_pack
    _run("mlp_nerf_pack", lambda: fn(C.byref(shape), C.byref(w), ptr(out), stream()))
    return out


def mlp_nerf_fwd_train(packed_train: torch.Tensor, x: torch.Tensor, shape=None):
    """Training forward: (out [N,4], saved) — saved holds every layer's input (bf16 records) for mlp_nerf_bwd."""
    shape = shape or mlp_nerf_shape()
    n = x.shape[0]
    out = torch.empty((n, 4), dtype=f32, device=x.device)
    saved = torch.empty(max(lib().nrf_mlp_nerf_saved_bytes(C.byref(shape), n), 0), dtype=u8, device=x.device)
    _run("mlp_nerf_fwd_train", lambda: lib().nrf_mlp_nerf_fwd_train(C.byref(shape), ptr(packed_train), ptr(x, f32), n, ptr(out, f32), ptr(saved), stream()))
    return out, saved


def mlp_nerf_fwd_points(packed: torch.Tensor, points: torch.Tensor, dirs: torch.Tensor, samples_per_ray: int, freqs_pts, freqs_views, train: bool = False,
                        shape=None):
    """RunNetwork for the classic model with the positional embeddings evaluated inside the MLP kernel: points [N,3], dirs [R,3]
    (N = R * samples_per_ray) -> out [N,4] (train=True: (out, saved) as mlp_nerf_fwd_train)."""
    shape = shape or mlp_nerf_shape()
    n = points.shape[0]
    out = torch.empty((n, 4), dtype=f32, device=points.device)
    fp, fv = cabi.host_floats(freqs_pts), cabi.host_floats(freqs_views)
    if not train:
        _run("mlp_nerf_fwd", lambda: lib().nrf_mlp_nerf_fwd_points(C.byref(shape), ptr(packed), ptr(points, f32), ptr(dirs, f32), samples_per_ray, fp, len(fp), fv,
                                                                   len(fv), n, ptr(out, f32), stream()))
        return out
    saved = torch.empty(max(lib().nrf_mlp_nerf_saved_bytes(C.byref(shape), n), 0), dtype=u8, device=points.device)
    _run("mlp_nerf_fwd_train", lambda: lib().nrf_mlp_nerf_fwd_train_points(C.byref(shape), ptr(packed), ptr(points, f32), ptr(dirs, f32), samples_per_ray, fp,
                                                                           len(fp), fv, len(fv), n, ptr(out, f32), ptr(saved), stream()))
    return out, saved


def mlp_nerf_bwd(packed_train: torch.Tensor, saved: torch.Tensor, grad_out: torch.Tensor, grads: dict, shape=None, workspace: torch.Tensor | None = None):
    """Backward of NeRFImpl::forward: grad_out [N,4] fp32 -> grads (dict with the parameter names of `mlp_nerf_pack`, fp32 CUDA
    tensors of the parameters' shapes) += d loss / d parameter."""
    shape = shape or mlp_nerf_shape()
    n = grad_out.shape[0]
    if workspace is None:
        workspace = torch.empty(max(lib().nrf_mlp_nerf_bwd_workspace_bytes(C.byref(shape), n), 0), dtype=u8, device=grad_out.device)
    g = _mlp_nerf_ptrs(grads)
    _run("mlp_nerf_bwd", lambda: lib().nrf_mlp_nerf_bwd(C.byref(shape), ptr(packed_train), ptr(saved), ptr(grad_out, f32), n, ptr(workspace), C.byref(g),
                                                        stream()))
    return grads


def mlp_nerf_fwd(packed: torch.Tensor, x: torch.Tensor, shape=None, out: torch.Tensor | None = None) -> torch.Tensor:
    """NeRFImpl::forward (inference): x [N, 90] fp32 -> [N, 4] = [rgb logits, alpha]."""
    shape = shape or mlp_nerf_shape()
    n = x.shape[0]
    if out is None:
        out = torch.empty((n, 4), dtype=f32, device=x.device)
    _run("mlp_nerf_fwd", lambda: lib().nrf_mlp_nerf_fwd(C.byref(shape), ptr(packed), ptr(x, f32), n, ptr(out, f32), stream()))
    return out


# ------------------------------------------------------------------------------------------------ LeRF language head (SURVEY §8f-1)

LERF_WEIGHT_NAMES = ("sigma_le_net_0", "sigma_le_net_1", "le_net_0", "le_net_1")


def lerf_shape(geo_feat_dim=32, num_layers=2, hidden_dim=256, lang_embed_dim=512, input_ch=128):
    return cabi.LerfShape(geo_feat_dim, num_layers, hidden_dim, lang_embed_dim, input_ch)


def lerf_pack(p: dict, shape=None, out: torch.Tensor | None = None, prefix: str = "lang_model") -> torch.Tensor:
    """p: the reference's registered names ('<prefix>_sigma_le_net_<i>.weight', '<prefix>_le_net_<i>.weight', src/LeRF.cpp:17-25) ->
    contiguous fp32 CUDA tensors.  Returns the operand blob of the fused head (fp16 UMMA core matrices of the four layers and of
    G = W_e1^T W_e1, then W_e1^T in fp32)."""
    shape = shape or lerf_shape()
    nbytes = lib().nrf_lerf_packed_bytes(C.byref(shape))
    if nbytes < 0:
        check(-3)
    w = cabi.LerfWeights(*[ptr(p[f"{prefix}_{n}.weight"], f32) for n in LERF_WEIGHT_NAMES])
    if out is None:
        out = torch.empty(nbytes, dtype=u8, device=p[f"{prefix}_le_net_1.weight"].device)
    _run("lerf_pack", lambda: lib().nrf_lerf_pack(C.byref(shape), C.byref(w), ptr(out), stream()))
    return out


def lerf_fwd(packed: torch.Tensor, enc: torch.Tensor, keep: torch.Tensor | None = None, shape=None) -> torch.Tensor:
    """LeRF::forward + the keep mask of RunLENetwork: enc [N,128] fp16 -> raw_le [N,513] fp32."""
    shape = shape or lerf_shape()
    n = enc.shape[0]
    out = torch.empty((n, shape.lang_embed_dim + 1), dtype=f32, device=enc.device)
    _run("lerf_fwd", lambda: lib().nrf_lerf_fwd(C.byref(shape), ptr(packed), ptr(enc, f16), ptr(keep, u8) if keep is not None else None, n, ptr(out), stream()))
    return out


def lerf_sigma_fwd(packed: torch.Tensor, enc: torch.Tensor, keep: torch.Tensor | None = None, shape=None) -> torch.Tensor:
    """Density of the language field only: raw4 [N,4] = [0,0,0,sigma_le]."""
    shape = shape or lerf_shape()
    n = enc.shape[0]
    raw4 = torch.empty((n, 4), dtype=f32, device=enc.device)
    _run("lerf_sigma_fwd", lambda: lib().nrf_lerf_sigma_fwd(C.byref(shape), ptr(packed), ptr(enc, f16), ptr(keep, u8) if keep is not None else None, n,
                                                             ptr(raw4), stream()))
    return raw4


def lerf_hidden_fwd(packed: torch.Tensor, enc: torch.Tensor, keep: torch.Tensor | None = None, shape=None):
    """Fine pass without the [N,512] embedding: (raw4 [N,4], hidden (fp16 tile records of h2), q [N] = |e|^2)."""
    shape = shape or lerf_shape()
    n = enc.shape[0]
    raw4 = torch.empty((n, 4), dtype=f32, device=enc.device)
    hidden = torch.empty(max(lib().nrf_lerf_hidden_bytes(C.byref(shape), n), 0), dtype=u8, device=enc.device)
    q = torch.empty(n, dtype=f32, device=enc.device)
    _run("lerf_hidden_fwd", lambda: lib().nrf_lerf_hidden_fwd(C.byref(shape), ptr(packed), ptr(enc, f16), ptr(keep, u8) if keep is not None else None, n,
                                                               ptr(raw4), ptr(hidden), ptr(q), stream()))
    return raw4, hidden, q


def lerf_render_embedding(packed: torch.Tensor, weights: torch.Tensor, hidden: torch.Tensor, q: torch.Tensor, shape=None) -> torch.Tensor:
    """RenderCLIPEmbedding on the (never materialised) normalised embeddings: weights [R,S] -> rendered [R,512]."""
    shape = shape or lerf_shape()
    r, s = weights.shape
    hsum = torch.empty((r, shape.hidden_dim), dtype=f32, device=weights.device)
    out = torch.empty((r, shape.lang_embed_dim), dtype=f32, device=weights.device)
    _run("lerf_render_embedding", lambda: lib().nrf_lerf_render_embedding(C.byref(shape), ptr(packed), ptr(weights, f32), ptr(hidden), ptr(q, f32), r, s,
                                                                           ptr(hsum), ptr(out), stream()))
    return out


# ---- training of the language head (nrf_lerf_fwd_train ... nrf_lerf_bwd_rows)


def _lerf_ptrs(p: dict, prefix: str) -> "cabi.LerfWeights":
    return cabi.LerfWeights(*[ptr(p[f"{prefix}_{n}.weight"], f32) for n in LERF_WEIGHT_NAMES])


def lerf_fwd_train(packed: torch.Tensor, enc: torch.Tensor, keep: torch.Tensor | None = None, shape=None):
    """Training forward of the fine pass: (raw4 [N,4], saved (bf16 tile records of [x | geo], h1, h2 + the ReLU mask of h1), q [N] = |e|^2)."""
    shape = shape or lerf_shape()
    n = enc.shape[0]
    raw4 = torch.empty((n, 4), dtype=f32, device=enc.device)
    saved = torch.empty(max(lib().nrf_lerf_train_saved_bytes(C.byref(shape), n), 0), dtype=u8, device=enc.device)
    q = torch.empty(n, dtype=f32, device=enc.device)
    _run("lerf_fwd_train", lambda: lib().nrf_lerf_fwd_train(C.byref(shape), ptr(packed), ptr(enc, f16), ptr(keep, u8) if keep is not None else None, n,
                                                             ptr(raw4), ptr(saved), ptr(q), stream()))
    return raw4, saved, q


def lerf_render_embedding_train(packed: torch.Tensor, weights: torch.Tensor, saved: torch.Tensor, q: torch.Tensor, shape=None):
    """(rendered [R,512], hsum [R,256], enorm [R]) from the training records."""
    shape = shape or lerf_shape()
    r, s = weights.shape
    hsum = torch.empty((r, shape.hidden_dim), dtype=f32, device=weights.device)
    out = torch.empty((r, shape.lang_embed_dim), dtype=f32, device=weights.device)
    enorm = torch.empty(r, dtype=f32, device=weights.device)
    _run("lerf_render_embedding", lambda: lib().nrf_lerf_render_embedding_train(C.byref(shape), ptr(packed), ptr(weights, f32), ptr(saved), ptr(q, f32), r, s,
                                                                                 ptr(hsum), ptr(out), ptr(enorm), stream()))
    return out, hsum, enorm


def lerf_bwd_workspace(n: int, n_rays: int, device, shape=None) -> torch.Tensor:
    shape = shape or lerf_shape()
    return torch.empty(max(lib().nrf_lerf_bwd_workspace_bytes(C.byref(shape), n, n_rays), 256), dtype=u8, device=device)


def lerf_bwd_rays(weights: dict, saved, q, comp_weights, hsum, rendered, enorm, grad_le_w1, workspace, target=None, grad_rendered=None, grad_scale=1.0,
                  loss_out=None, prefix="lang_model", shape=None) -> torch.Tensor:
    """Per-ray half of the backward; returns dw [R,S] = d loss / d compositing weights (feed it to composite_bwd as g_weights)."""
    shape = shape or lerf_shape()
    r, s = comp_weights.shape
    dw = torch.empty((r, s), dtype=f32, device=comp_weights.device)
    w = _lerf_ptrs(weights, prefix)
    _run("lerf_bwd_rays", lambda: lib().nrf_lerf_bwd_rays(C.byref(shape), C.byref(w), ptr(saved), ptr(q, f32), ptr(comp_weights, f32), ptr(hsum, f32),
                                                           ptr(rendered, f32), ptr(enorm, f32), ptr(target), ptr(grad_rendered), r, s, grad_scale, ptr(loss_out),
                                                           ptr(grad_le_w1, f32), ptr(workspace), ptr(dw), stream()))
    return dw


def lerf_bwd_rows(packed, weights: dict, saved, keep, d_raw4, n_samples: int, workspace, grads: dict, prefix="lang_model", shape=None,
                  d_enc: torch.Tensor | None = None) -> torch.Tensor:
    """Per-row half: grads[<prefix>_<layer>.weight] += (fp32), returns d_enc [N,128] bf16."""
    shape = shape or lerf_shape()
    n = d_raw4.numel() // 4
    if d_enc is None:
        d_enc = torch.empty((n, shape.input_ch), dtype=bf16, device=d_raw4.device)
    w, g = _lerf_ptrs(weights, prefix), _lerf_ptrs(grads, prefix)
    _run("lerf_bwd_rows", lambda: lib().nrf_lerf_bwd_rows(C.byref(shape), ptr(packed), C.byref(w), ptr(saved), ptr(keep, u8) if keep is not None else None,
                                                           ptr(d_raw4, f32), n, n_samples, ptr(workspace), C.byref(g), ptr(d_enc), stream()))
    return d_enc
