"""HashNeRF ray-batch pipeline on the C ABI: RenderRays (inference) and one training step.

Host-side mirror, in Python, of what the reference does in NeRFRenderer::Render/RenderRays
(src/NeRFRenderer.h:366-459, 530-604) and the ~20 training lines of NeRFExecutor::Train
(src/NeRFExecutor.h:868-890, 923, 986-996) for the <CuHashEmbedder, CuSHEncoder, NeRFSmall> instantiation
(src/main.cpp:220-221).  Every arithmetic step is one call into libnerfpp_b200.so; torch only owns the buffers,
the stream and (for data-parallel training) the NCCL all-reduce.

Divergences from the reference, all deliberate (SURVEY §9):
  * Q3  the coarse pass never receives a gradient, so it runs as inference (nothing recorded);
  * Q5  table reads go through a persistent fp16 shadow refreshed by the Adam kernel, gradients accumulate in fp32;
  * Q1  sample points are kept per call (the reference back-propagates with the last forward's points);
  * the SH basis is evaluated once per ray, not once per sample.
Configuration is the parity one: ThinRay, Perturb 0, no raw noise, no stochastic preconditioning.
"""
from __future__ import annotations

import math
import os

import numpy as np
import torch

from . import ops
from .ops import HashGridSpec, f16, f32, i32

def mlp_layers(n_views: int = 16):
    """[out, in] of sigma_net_0, sigma_net_1, color_net_0 (in = views + geo 15), color_net_1, color_net_2 (src/NeRF.cpp:338-342)."""
    return [(64, 32), (16, 64), (64, n_views + 15), (64, 64), (3, 64)]


def _is_prime(x: int) -> bool:
    i = 2
    while i * i <= x:
        if x % i == 0:
            return False
        i += 1
    return True


def random_primes(n: int, rng: np.random.Generator) -> np.ndarray:
    """Rejection-sampled primes in [2^28, 2^30) (src/CuHashEmbedder.cpp:28-47)."""
    out = []
    while len(out) < n:
        v = int(rng.integers(1 << 28, 1 << 30))
        if _is_prime(v):
            out.append(v)
    return np.asarray(out, dtype=np.int32)


def make_grid(bbox, n_levels=16, n_features=2, log2_hashmap_size=19, base_resolution=16, finest_resolution=512,
              device="cuda", seed=42, primes: np.ndarray | None = None) -> HashGridSpec:
    """Buffers of CuHashEmbedderImpl's constructor (src/CuHashEmbedder.cpp:37-76); Primes are an input when given."""
    rng = np.random.default_rng(seed)
    if primes is None:
        primes = random_primes(3 * n_levels, rng)
    local = ((1 << log2_hashmap_size) >> 4) << 4
    size = torch.full((n_levels,), local, dtype=i32)
    idx = (torch.cumsum(size, 0) - local).to(i32)
    return HashGridSpec(
        bounding_box=tuple(float(v) for v in bbox),
        primes=torch.as_tensor(np.asarray(primes, dtype=np.int32).reshape(n_levels, 1, 3)).to(device),
        biases=torch.zeros((n_levels, 3), dtype=f32, device=device),
        feat_local_idx=idx.to(device), feat_local_size=size.to(device),
        n_levels=n_levels, n_features=n_features, log2_hashmap_size=log2_hashmap_size,
        base_resolution=base_resolution, finest_resolution=finest_resolution)


class FlatAdamModel:
    """One flat fp32 parameter vector [hash-table scalars (n_table) | network weights] with its gradient, Adam moments and fp16 shadow, and the
    optimiser step on it (src/NeRFExecutor.h:539 Adam(0.9, 0.99, eps 1e-15); :986-996 step + learning-rate decay) as ONE kernel launch:
    dense (nrf_adam_step[_scheduled]) or, data-parallel, the fused peer-memory kernel (parallel.PeerShardedOptimizer).  Subclasses provide
    `repack()` (operand blob of the network from the fp32 weights) and fill `params`."""

    def _init_flat(self, n_params: int, device, lr: float, lrate_decay: int):
        self.params = torch.empty(n_params, dtype=f32, device=device)
        self.grads = torch.zeros_like(self.params)
        self.exp_avg = torch.zeros_like(self.params)
        self.exp_avg_sq = torch.zeros_like(self.params)
        self.shadow = torch.empty(self.params.shape, dtype=f16, device=device)                   # fp16 copy; table part is what the gathers read
        self.lr0, self.lrate_decay, self.step = lr, lrate_decay, 0
        self.loss = torch.zeros(1, dtype=f32, device=device)
        self.peer = None          # parallel.PeerShardedOptimizer when the fused data-parallel optimiser is in use
        self.masters_synced = True  # False while the fused optimiser has stepped and the non-owned fp32 shards are stale
        self.sched = None
        self._sched_step = -1

    @property
    def table(self):
        self._require_synced("table")
        return self.params[:self.n_table]

    @property
    def table_f16(self): return self.shadow[:self.n_table]

    def _require_synced(self, what):
        if not self.masters_synced:
            raise RuntimeError(f"{type(self).__name__}.{what}: the fp32 master is sharded over the ranks (fused data-parallel optimiser) and this rank's "
                               "non-owned shards are stale — call model.peer.allgather_master(model) first (collective)")

    def state_dict(self):
        """fp32 master + Adam moments + step, valid on every rank (gathers the owners' shards first under the fused optimiser)."""
        if self.peer is not None and not self.masters_synced:
            self.peer.allgather_master(self)
        return {"params": self.params.clone(), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(), "step": self.step}

    def refresh(self):
        """Re-derive the fp16 table shadow and the packed network weights from the fp32 masters."""
        ops.table_to_half(self.table, self.table_f16)
        self.shadow[self.n_table:].copy_(self.params[self.n_table:])      # the network tail of the shadow: what the Adam kernels will keep writing
        self.repack()

    def optimizer_step(self, grad_scale=1.0):
        self.step += 1
        # src/NeRFExecutor.h:986-996: step() runs with the rate set at the END of the previous iteration,
        # lr0 * 0.1^(global_step / decay_steps) with global_step counted from 0 and incremented after the update
        lr = self.lr0 * (0.1 ** (max(self.step - 2, 0) / (self.lrate_decay * 1000)))
        ops.adam_step(self.params, self.grads, self.exp_avg, self.exp_avg_sq, lr, self.step, 0.9, 0.99, 1e-15,
                      grad_scale, True, self.shadow)
        self.repack()

    def _init_sched(self):
        if self.sched is None:
            self.sched = torch.zeros(4, dtype=i32, device=self.device)
            self._sched_step = -1

    def _sync_sched(self):
        if self._sched_step != self.step:          # eager steps ran in between: re-seed the device-side step counter
            self.sched[0:1].copy_(torch.tensor([self.step], dtype=i32), non_blocking=False)
            self._sched_step = self.step

    def _optimizer_step_sharded(self):
        """Data-parallel step without NCCL: one kernel per rank over NVLink peer memory (parallel.PeerShardedOptimizer)."""
        self.masters_synced = False
        peer = self.peer
        q4, n = self.n_table // 4 * 4, self.params.numel()
        args = (self.params, self.exp_avg, self.exp_avg_sq)
        if not peer.overlap:
            ops.adam_schedule_advance(self.sched, self.lr0, 0.1, float(self.lrate_decay * 1000))
            ops.adam_step_sharded_range(peer.pg, *args, (0, q4), (q4, n), self.sched, 0.9, 0.99, 1e-15, 1.0 / peer.world)
        else:
            # two ranges, each partitioned over the ranks on its own (ownership never changes).  The first one was already exchanged behind the
            # backward (PeerShardedOptimizer.backward_overlapped) or, when the step is taken on a finished gradient (dp_check), goes first here.
            if peer._side_pending:
                torch.cuda.current_stream(self.device).wait_stream(peer.side_stream)
                peer._side_pending = False
            else:
                ops.adam_schedule_advance(self.sched, self.lr0, 0.1, float(self.lrate_decay * 1000))
                ops.adam_step_sharded_range(peer.pg_side, *args, peer.ranges[0], (0, 0), self.sched, 0.9, 0.99, 1e-15, 1.0 / peer.world)
            ops.adam_step_sharded_range(peer.pg, *args, peer.ranges[1], (q4, n), self.sched, 0.9, 0.99, 1e-15, 1.0 / peer.world)
        self.repack()

    def flags_timeout(self) -> int:
        """1 if a peer barrier of the fused optimiser ever gave up waiting (a rank missed a step), else 0.  Synchronises."""
        return self.peer.timeout() if self.peer is not None else 0

    def optimizer_step_sharded(self):
        """Eager (non-graph) entry of the fused data-parallel optimiser step."""
        self.peer.check()
        self._init_sched()
        self._sync_sched()
        self._optimizer_step_sharded()
        self.peer.mirror_flag()
        self.step += 1
        self._sched_step = self.step

    def _optimizer_step_scheduled(self, grad_scale):
        ops.adam_schedule_advance(self.sched, self.lr0, 0.1, float(self.lrate_decay * 1000))
        ops.adam_step_scheduled(self.params, self.grads, self.exp_avg, self.exp_avg_sq, self.sched, 0.9, 0.99, 1e-15, grad_scale, True, self.shadow)
        self.repack()

    # -- the step as ONE CUDA-graph replay (launch-bound otherwise: ~20 kernels of 3..300 us behind ~20 ctypes calls)
    def capture_train_step(self, n_rays: int, world: int = 1, allreduce=None, pixels: bool = False):
        """Captures forward_backward and the optimiser for a fixed ray count.  pixels: the step's input is the int32 [n_rays,2] pixel list of the
        current training view (HashNeRF.set_camera) instead of rays + targets.  world == 1: one graph per step;
        world > 1: graph(render + loss + backward) -> allreduce(self.grads) (eager NCCL call) -> graph(Adam + repack), or, with the fused
        peer-memory optimiser, one graph.  The step count / bias corrections / decayed rate advance on the device (nrf_adam_schedule_advance)."""
        dev = self.device
        self._g_in = self._static_inputs(n_rays, pixels) if pixels else self._static_inputs(n_rays)
        self._g_world, self._g_allreduce = world, allreduce
        self._init_sched()
        # warm-up outside the capture (one-time function attributes, level scales, allocator pools); its gradient is discarded
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self.forward_backward(*self._g_in)
            self.grads.zero_()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        from . import cabi
        l0 = cabi.launch_count()
        self._g_fb = torch.cuda.CUDAGraph()
        overlap = world > 1 and self.peer is not None and getattr(self.peer, "overlap", False)
        with torch.cuda.graph(self._g_fb):
            self._g_out = self.forward_backward(*self._g_in, dp_overlap=True) if overlap else self.forward_backward(*self._g_in)
            if world == 1:
                self._optimizer_step_scheduled(1.0)
            elif self.peer is not None:
                self._optimizer_step_sharded()
        self._g_opt = None
        if world > 1 and self.peer is None:
            self._g_opt = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self._g_opt):
                self._optimizer_step_scheduled(1.0 / world)
        self.graph_kernels_per_step = cabi.launch_count() - l0
        return self

    def train_step_graph(self, *inputs):
        """Replay of the captured step.  Inputs may be device tensors or pinned host tensors (copied on the current stream)."""
        if self.peer is not None:
            self.peer.check()             # a lost peer fails loudly (pinned-host mirror of the timeout marker, no synchronisation)
        self._sync_sched()
        for dst, src in zip(self._g_in, inputs):
            dst.copy_(src, non_blocking=True)
        self._g_fb.replay()
        if self._g_opt is not None:
            self._g_allreduce(self.grads)
            self._g_opt.replay()
        elif self.peer is not None:
            self.masters_synced = False
            self.peer.mirror_flag()
        self.step += 1
        self._sched_step = self.step
        return self.loss

    @property
    def graph_outputs(self) -> dict:
        """What the captured step's forward_backward returns (its static output buffers): after a replay, that step's results."""
        return self._g_out

    def train_step(self, *inputs):
        self.forward_backward(*inputs)
        self.optimizer_step()
        return self.loss


class HashNeRF(FlatAdamModel):
    """Parameters + optimiser state of one HashNeRF replica, as flat device buffers.

    params = [table scalars the kernels can reach | NeRFSmall weights], one fp32 vector, so the data-parallel
    gradient exchange is ONE all-reduce and the optimiser is ONE kernel.  The reachable table prefix is
    (L+1) * 2^T scalars: level offsets are in scalars (reference quirk), the rest of the [L*2^T, F] parameter is
    never read or written by the reference either (its gradient is identically zero, and Adam with eps=1e-15 leaves
    a zero-gradient entry with zero moments untouched)."""

    def __init__(self, bbox=(-1.5, -1.5, -1.5, 1.5, 1.5, 1.5), n_levels=16, n_features=2, log2_hashmap_size=19,
                 base_resolution=16, finest_resolution=512, sh_degree=4, n_samples=64, n_importance=128,
                 device="cuda", seed=42, lr=1e-2, lrate_decay=250, primes=None, ray_bias=None):
        """sh_degree 4 (16 view channels): the view channels are the first k-step of the fused colour net.  Any other degree 1..8 (8 = the
        reference's shipped configuration, src/main.cpp:176): the view term of that layer is computed once per RAY and enters the fused kernels
        as a bias (ops.mlp_small_view_bias_fwd / _bwd, NRF_MLP_IN_ENC16_RAYBIAS).  ray_bias=True forces that form at degree 4 (tests)."""
        assert n_levels * n_features == 32 and 1 <= sh_degree <= 8, "the fused MLP is built for 32 encoding channels and SH degree 1..8"
        self.n_views = sh_degree * sh_degree
        self.ray_bias = (self.n_views != 16) if ray_bias is None else bool(ray_bias)
        assert self.ray_bias or self.n_views == 16
        self.mlp_shape = ops.mlp_shape(input_ch_views=self.n_views)
        self.mlp_layers = mlp_layers(self.n_views)
        self._grad_bias = None
        self.device = torch.device(device)
        self.bbox = tuple(float(v) for v in bbox)
        self.grid = make_grid(bbox, n_levels, n_features, log2_hashmap_size, base_resolution, finest_resolution, device, seed, primes)
        self.sh_degree, self.S, self.N = sh_degree, n_samples, n_importance
        self.n_table = self.grid.used_scalars()
        g = torch.Generator(device="cpu").manual_seed(seed)
        self._init_flat(self.n_table + sum(fo * fi for fo, fi in self.mlp_layers), device, lr, lrate_decay)
        self.params[:self.n_table] = (torch.rand(self.n_table, generator=g) * 1e-4).to(device)   # src/CuHashEmbedder.cpp:24
        off = self.n_table
        for fo, fi in self.mlp_layers:                                                            # Trainable.h:43 Xavier normal, gain 0.1
            std = 0.1 * math.sqrt(2.0 / (fi + fo))
            self.params[off:off + fo * fi] = (torch.randn(fo * fi, generator=g) * std).to(device)
            off += fo * fi
        self.packed = None
        self.t_vals = torch.linspace(0.0, 1.0, n_samples, dtype=f32).to(device)                  # src/NeRFRenderer.h:393
        self.u = torch.linspace(0.0, 1.0, n_importance, dtype=f32).to(device)                    # src/Sampler.h:20
        # Copy the coarse samples' encoding rows into the fine pass instead of gathering them again: the merged z list contains the
        # coarse samples bit for bit, so the rows are bit-identical (tests/test_gpu_hash.py::test_row_reuse...); ~10 % of the fine-pass encode.
        self.reuse_coarse_rows = True
        self.reuse_coarse_raw = True
        self._u_cache = {}
        self._render_ws = None
        self._cam = None
        self.refresh()

    # -- views into the flat buffers
    @property
    def mlp_params(self): return self.params[self.n_table:]

    def mlp_weights(self):
        out, off = [], 0
        for fo, fi in self.mlp_layers:
            out.append(self.mlp_params[off:off + fo * fi].view(fo, fi))
            off += fo * fi
        return out

    def mlp_grads_view(self, layer: int):
        """Gradient of NeRFSmall weight `layer` (0..4) as a [out, in] view into the flat gradient."""
        off = self.n_table + sum(fo * fi for fo, fi in self.mlp_layers[:layer])
        fo, fi = self.mlp_layers[layer]
        return self.grads[off:off + fo * fi].view(fo, fi)

    def repack(self):
        self.packed = ops.mlp_small_pack(self.mlp_params, shape=self.mlp_shape, out=self.packed)

    def _views(self, ray_sh, for_backward=False):
        """What the fused MLP kernels take as the rays' view input: the SH table itself (16 channels), or — ray_bias — the view term of the
        colour net's first layer, one [64] row per ray, shared by the coarse and the fine pass (for_backward: its gradient accumulator is
        zeroed by the same launch)."""
        if not self.ray_bias:
            return ray_sh
        gb = None
        if for_backward:
            if self._grad_bias is None or self._grad_bias.shape[0] != ray_sh.shape[0]:
                self._grad_bias = torch.empty((ray_sh.shape[0], 64), dtype=f32, device=self.device)
            gb = self._grad_bias
        return ops.mlp_small_view_bias_fwd(self.packed, ray_sh, shape=self.mlp_shape, grad_bias_zero=gb)

    def _static_inputs(self, n_rays, pixels=False):
        dev = self.device
        if pixels:
            assert self._cam is not None, "set_camera(image, K, c2w) first"
            return (torch.zeros((n_rays, 2), dtype=i32, device=dev),)
        return (torch.tensor([[0.0, 0.0, 4.0]], device=dev).repeat(n_rays, 1), torch.tensor([[0.0, 0.0, -1.0]], device=dev).repeat(n_rays, 1),
                torch.full((n_rays, 3), 0.5, dtype=f32, device=dev))

    def set_camera(self, image: torch.Tensor, K, c2w):
        """The current training view (NeRFDataset's CurrentImage / K / pose, src/NeRFDataset.cpp:149-157): image fp32 [H,W,3] on the device.  A step
        can then be fed with pixel coordinates only: GetRayBatch (:109-144) and the target gather (:156) run inside the step's first kernel."""
        assert image.is_cuda and image.dtype == f32 and image.dim() == 3 and image.is_contiguous()
        self._cam = (image, ops._cam(K, c2w))

    # -- RenderRays (src/NeRFRenderer.h:366-459)
    def _network(self, ray_batch, z, views, reuse=None):
        """RunNetwork (src/NeRFRenderer.h:164-194): points are generated inside the encode kernel (o + d z), the SH basis comes
        per ray (views: see _views), sigma is zeroed outside the box in the MLP epilogue.  reuse: see ops.hash_encode_rays_fwd."""
        s = z.shape[1]
        enc, keep = ops.hash_encode_rays_fwd(self.grid, self.table_f16, ray_batch, z, clamp=True, out_f16=True, reuse=reuse)
        raw = ops.mlp_small_fwd(self.packed, enc, views, s, keep, shape=self.mlp_shape, ray_bias=self.ray_bias)
        return enc, keep, raw.view(-1, s, 4)

    def _u(self, n_importance):
        if n_importance is None or n_importance == self.N:
            return self.u
        u = self._u_cache.get(n_importance)
        if u is None:
            u = self._u_cache[n_importance] = torch.linspace(0.0, 1.0, n_importance, dtype=f32).to(self.device)
        return u

    def render_rays_fused(self, rays_o, rays_d, white_bkgr=False, n_importance=None, want_weights=False, want_z=False):
        """Inference RenderRays as ONE C-ABI call (nrf_render_rays_fwd) into a cached workspace."""
        out, self._render_ws = ops.render_rays_fwd(self.grid, self.table_f16, self.packed, rays_o, rays_d, self.t_vals, self._u(n_importance),
                                                   self.bbox, white_bkgr, self.sh_degree, want_weights=want_weights, want_z=want_z,
                                                   workspace=self._render_ws, shape=self.mlp_shape)
        return out

    def render_rays(self, rays_o, rays_d, white_bkgr=False, keep_for_backward=False, n_importance=None, zero_scalar=None, setup=None, fine_composite=True):
        # Render prologue + coarse depths + per-ray SH (+ the caller's loss accumulator reset) in one launch (setup: already done by the caller)
        ray_batch, z, ray_sh = setup if setup is not None else ops.ray_setup(rays_o, rays_d, self.bbox, 0.0, self.t_vals, self.sh_degree, zero_scalar=zero_scalar)
        views = self._views(ray_sh, for_backward=keep_for_backward)
        enc_c, keep_c, raw = self._network(ray_batch, z, views)
        coarse = ops.composite_fwd(raw, z, rays_d, white_bkgr)
        u = self._u(n_importance)
        # the merged list contains the coarse samples bit for bit: their encoding rows are copied, not gathered again (reuse_coarse_rows), and —
        # one network for both passes (src/NeRFRenderer.h:422,447) — their raw rows are the coarse pass's own (reuse_coarse_raw): the fine
        # forward evaluates the importance samples only.  Same bits either way (tests/test_gpu_pipeline.py).
        if self.reuse_coarse_rows and self.reuse_coarse_raw:
            z_fine, perm, raw_m = ops.sample_pdf_merge(z, coarse["weights"], u, want_perm=True, raw_coarse=raw.view(-1, 4))
            enc, keep = ops.hash_encode_rays_fwd(self.grid, self.table_f16, ray_batch, z_fine, clamp=True, out_f16=True,
                                                 reuse=(perm, enc_c, keep_c, z.shape[1]))
            raw = ops.mlp_small_fwd_importance(self.packed, enc, views, keep, perm, u.shape[-1], raw_m, shape=self.mlp_shape,
                                               ray_bias=self.ray_bias).view(-1, z_fine.shape[1], 4)
        else:
            if self.reuse_coarse_rows:
                z_fine, perm = ops.sample_pdf_merge(z, coarse["weights"], u, want_perm=True)
                reuse = (perm, enc_c, keep_c, z.shape[1])
            else:
                z_fine, reuse = ops.sample_pdf_merge(z, coarse["weights"], u), None
            enc, keep, raw = self._network(ray_batch, z_fine, views, reuse)
        # fine_composite False (training): the caller composites, takes the loss and back-propagates in one launch (ops.composite_huber_bwd)
        out = ops.composite_fwd(raw, z_fine, rays_d, white_bkgr) if fine_composite else {}
        out["z"] = z_fine
        if keep_for_backward:
            out["_saved"] = (ray_batch, enc, keep, raw, views, ray_sh)
        return out

    def forward_backward_shipped(self, rays_o, rays_d, target, cone_angle: float, raw_noise_std: float, sp_alpha: float, clamp_to_box: bool = True):
        """The step with the RNG-gated stages of the reference's shipped configuration ON (src/main.cpp:187 thin_ray = false; src/NeRFExecutor.h:
        411-412 raw_noise_std and StochasticPreconditioningAlpha > 0): in-cone jitter of both passes' sample points (TangentScatter,
        src/NeRFRenderer.h:307-362), stochastic preconditioning + ReflectBoundary of the fine pass (:435-443), density noise in both RawToOutputs
        (:253-254).  The variates are torch.rand / torch.randn draws — the reference's own calls — so results are statistically, not bitwise, equal
        (SURVEY §9-Q4); everything else is the C ABI.  The jittered points are explicit [R,S,3] arrays here (the parity path never forms them).
        clamp_to_box: TangentScatter clamps the jittered points into the box (:356-360) — which also pulls the samples of rays that MISS the box
        onto its surface, where they pass the embedder's keep test; False (tests) leaves them outside."""
        dev = self.device
        r = rays_o.shape[0]
        if getattr(self, "_cone", None) is None or self._cone[0] != cone_angle:
            self._cone = (cone_angle, torch.full((1,), cone_angle, dtype=f32, device=dev))
        cone = self._cone[1]
        ray_batch, z, ray_sh = ops.ray_setup(rays_o, rays_d, self.bbox, 0.0, self.t_vals, self.sh_degree, zero_scalar=self.loss)
        views = self._views(ray_sh, for_backward=True)

        def network(zz, precondition):
            s = zz.shape[1]
            pts = ops.sample_points(ray_batch, zz)
            if precondition and sp_alpha > 0:
                ops.precondition_points(pts, torch.randn_like(pts), sp_alpha, self.bbox)
            ops.tangent_scatter(pts, zz, cone, rays_d, torch.rand((r, s), device=dev), torch.rand((r, s), device=dev), self.bbox if clamp_to_box else None)
            pts = pts.view(-1, 3)
            enc, keep = ops.hash_encode_fwd(self.grid, self.table_f16, pts, clamp=True, out_f16=True)
            raw = ops.mlp_small_fwd(self.packed, enc, views, s, keep, shape=self.mlp_shape, ray_bias=self.ray_bias).view(r, s, 4)
            noise = torch.randn((r, s), device=dev) if raw_noise_std > 0 else None
            return pts, enc, keep, raw, noise

        _, _, _, raw_c, noise_c = network(z, False)
        coarse = ops.composite_fwd(raw_c, z, rays_d, noise=noise_c, raw_noise_std=raw_noise_std)
        z_fine = ops.sample_pdf_merge(z, coarse["weights"], self.u)
        pts, enc, keep, raw, noise = network(z_fine, True)
        out = ops.composite_fwd(raw, z_fine, rays_d, noise=noise, raw_noise_std=raw_noise_std)
        g_rgb = torch.empty_like(out["rgb"])
        ops.huber_fwd_bwd(out["rgb"], target, self.loss, g_rgb, 1.0, 1.0)
        d_raw = ops.composite_bwd(raw, z_fine, rays_d, noise=noise, raw_noise_std=raw_noise_std, g_rgb=g_rgb)
        g_enc = self._mlp_backward(enc, views, ray_sh, raw.shape[1], keep, d_raw)
        ops.hash_encode_bwd(self.grid, pts, g_enc, self.grads[:self.n_table], clamp=True)
        return out

    def render_image(self, h, w, K, c2w, chunk=1 << 18, row_begin=0, row_end=None, white_bkgr=False, n_importance=None, from_camera=True):
        """Render(h,w,K,c2w) for image rows [row_begin,row_end) (src/NeRFRenderer.h:540-547, RenderPath :684).  from_camera (default): each chunk
        is ONE C-ABI call that needs only (K, c2w, first pixel, count) — GetRays runs inside its prologue kernel (nrf_render_tile_fwd, SURVEY
        §8f-3); False: nrf_get_rays + nrf_render_rays_fwd on the ray arrays.  Same bits either way."""
        row_end = h if row_end is None else row_end
        n, first = (row_end - row_begin) * w, row_begin * w
        if from_camera:
            outs = []
            for i in range(0, n, chunk):
                out, self._render_ws = ops.render_rays_fwd(self.grid, self.table_f16, self.packed, None, None, self.t_vals, self._u(n_importance), self.bbox,
                                                           white_bkgr, self.sh_degree, workspace=self._render_ws, shape=self.mlp_shape,
                                                           tile=(K, c2w, w, first + i, min(chunk, n - i)))
                outs.append(out)
        else:
            rays_o, rays_d = ops.get_rays(h, w, K, c2w, row_begin, row_end, self.device)
            outs = [self.render_rays_fused(rays_o[i:i + chunk], rays_d[i:i + chunk], white_bkgr, n_importance=n_importance) for i in range(0, n, chunk)]
        return {k: torch.cat([o[k] for o in outs], 0) for k in ("rgb", "depth", "disp", "acc")}

    def _mlp_backward(self, enc, views, ray_sh, samples_per_ray, keep, d_raw):
        """NeRFSmall backward into self.grads (weights) -> gradient of the encodings (bf16 [N,32])."""
        g_mlp = self.grads[self.n_table:]
        if not self.ray_bias:
            return ops.mlp_small_bwd(self.packed, enc, views, samples_per_ray, keep, d_raw.view(-1, 4), g_mlp, shape=self.mlp_shape)
        g_enc = ops.mlp_small_bwd(self.packed, enc, views, samples_per_ray, keep, d_raw.view(-1, 4), g_mlp, shape=self.mlp_shape, grad_bias=self._grad_bias)
        ops.mlp_small_view_bias_bwd(ray_sh, self._grad_bias, g_mlp, shape=self.mlp_shape)          # the view columns of color_net_0
        return g_enc

    # -- one optimisation step (src/NeRFExecutor.h:868-890, 923, 986-996)
    def dp_overlap_split(self):
        """(level k, scalar offset of level k in the flat table): the table gradient below that offset is complete once levels [0, k) have been
        scattered — what parallel.PeerShardedOptimizer exchanges behind the scatter of levels [k, L) (NRF_DP_OVERLAP=1)."""
        k = int(os.environ.get("NRF_DP_OVERLAP_LEVEL", "14"))
        k = min(max(k, 1), self.grid.n_levels - 1)
        return k, int(self.grid.feat_local_idx[k])

    def forward_backward(self, *inputs, grad_scale=1.0, dp_overlap=False):
        """Render + huber + backward into self.grads (accumulating).  self.loss holds the mean huber loss.  inputs: (rays_o, rays_d, target), or
        (pix_hw,) — int32 [R,2] pixel coordinates of the view given to set_camera: rays and targets are then formed on the device.
        dp_overlap (a training step under the fused data-parallel optimiser with NRF_DP_OVERLAP=1): the table gradient is scattered in two level
        ranges and the exchange of the first starts behind the second (the optimiser step that follows joins it)."""
        if len(inputs) == 1:
            image, cam = self._cam
            rays_o, rays_d, target, rb, z, sh = ops.ray_setup_pixels(inputs[0], None, None, image, self.bbox, 0.0, self.t_vals, self.sh_degree,
                                                                     zero_scalar=self.loss, cam=cam)
            out = self.render_rays(rays_o, rays_d, keep_for_backward=True, setup=(rb, z, sh), fine_composite=False)
        else:
            rays_o, rays_d, target = inputs
            out = self.render_rays(rays_o, rays_d, keep_for_backward=True, zero_scalar=self.loss, fine_composite=False)
        ray_batch, enc, keep, raw, views, ray_sh = out.pop("_saved")
        # RawToOutputs of the fine pass + huber + their backward: one launch
        d_raw, out["rgb"] = ops.composite_huber_bwd(raw, out["z"], rays_d, target, self.loss, grad_scale=grad_scale)
        g_enc = self._mlp_backward(enc, views, ray_sh, raw.shape[1], keep, d_raw)
        if dp_overlap and self.peer is not None and self.peer.overlap:
            self.peer.backward_overlapped(self, lambda levels: ops.hash_encode_rays_bwd(self.grid, ray_batch, out["z"], g_enc, self.grads[:self.n_table],
                                                                                        clamp=True, levels=levels))
        else:
            ops.hash_encode_rays_bwd(self.grid, ray_batch, out["z"], g_enc, self.grads[:self.n_table], clamp=True)
        return out


def synthetic_view(h=800, w=800, radius=4.0):
    """(K [3,3], c2w [4,4]) of the synthetic training view of BASELINE C2: pinhole with camera_angle_x = 0.6911 (src/load_blender.h:144-185) on a
    radius-4 sphere pose (pose_spherical(30, -30, 4), :43-57)."""
    focal = 0.5 * w / math.tan(0.5 * 0.6911)
    K = torch.tensor([[focal, 0, 0.5 * w], [0, focal, 0.5 * h], [0, 0, 1]], dtype=f32)
    th, ph = math.radians(30.0), math.radians(-30.0)
    rot_phi = torch.tensor([[1, 0, 0], [0, math.cos(ph), -math.sin(ph)], [0, math.sin(ph), math.cos(ph)]], dtype=f32)
    rot_th = torch.tensor([[math.cos(th), 0, -math.sin(th)], [0, 1, 0], [math.sin(th), 0, math.cos(th)]], dtype=f32)
    R = rot_th @ rot_phi
    c2w = torch.eye(4, dtype=f32)
    c2w[:3, :3] = R
    c2w[:3, 3] = R @ torch.tensor([0.0, 0.0, radius])
    return K, c2w


def synthetic_pixels(n, h=800, w=800, seed=0):
    """Pixel sampling of NeRFDataset::get_batch (src/NeRFDataset.cpp:154-155): int32 [n,2] = (row, col), host tensor."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.stack([torch.randint(0, h, (n,), generator=g), torch.randint(0, w, (n,), generator=g)], -1).to(torch.int32)


def synthetic_rays(n, h=800, w=800, device="cuda", seed=0, radius=4.0):
    """Random pixels of an h x w pinhole view on a radius-4 sphere pose (BASELINE C2): pixel sampling as
    NeRFDataset::get_batch (src/NeRFDataset.cpp:154-157), ray maths as GetRayBatch (:109-144), targets U[0,1]^3."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    focal = 0.5 * w / math.tan(0.5 * 0.6911)
    py = torch.randint(0, h, (n,), generator=g).float()
    px = torch.randint(0, w, (n,), generator=g).float()
    dirs = torch.stack([(px - 0.5 * w) / focal, -(py - 0.5 * h) / focal, -torch.ones(n)], -1)
    th, ph = math.radians(30.0), math.radians(-30.0)
    rot_phi = torch.tensor([[1, 0, 0], [0, math.cos(ph), -math.sin(ph)], [0, math.sin(ph), math.cos(ph)]], dtype=f32)
    rot_th = torch.tensor([[math.cos(th), 0, -math.sin(th)], [0, 1, 0], [math.sin(th), 0, math.cos(th)]], dtype=f32)
    R = rot_th @ rot_phi
    rays_d = dirs @ R.t()
    rays_o = (R @ torch.tensor([0.0, 0.0, radius])).expand(n, 3).contiguous()
    target = torch.rand(n, 3, generator=g)
    return rays_o.to(device), rays_d.contiguous().to(device), target.to(device)
