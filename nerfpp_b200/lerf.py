"""LeRF language field on the C ABI: LeRFRenderer::RenderRays / Render for inference (SURVEY §8f-1, BASELINE C5).

Host-side mirror, in Python, of src/LeRFRenderer.cpp:85-162 (RenderRays) and :266-331 (Render) for the instantiation the
reference trains: CuHashEmbedder("lang_embedder", bbox, 16, 8, 19, 16, 512) (src/main.cpp:203-207, src/NeRFExecutor.h:461) and
LeRF(32, 2, 256, D, 128, "lang_model") (src/NeRFExecutor.h:507-514) with D = 512 (BASELINE C5).  Every arithmetic step is one call
into libnerfpp_b200.so; torch only owns the buffers and the stream.

What is not computed, because the reference discards it: the coarse pass evaluates the language density only (its embedding,
src/LeRFRenderer.cpp:133-134, is never used), and the fine pass never forms LangEmbedding [R,S,D] — RenderedLangEmbedding comes from
the last hidden layer (nrf_lerf_hidden_fwd + nrf_lerf_render_embedding).  `return_embedding=True` evaluates the compatibility entry
(nrf_lerf_fwd) as well and returns the reference's LangEmbedding / Raw tensors.
Configuration is the parity one: ThinRay, Perturb 0, no raw noise, no stochastic preconditioning.  Relevancy (RuCLIP) is out of scope.

Training of the language field (src/NeRFExecutor.h:957-983: RenderRays on the language renderer, huber(delta 1.25).sum(-1).nanmean() against the
CLIP target, backward, Adam over {lang_embedder, lang_model}): `LeRFField.train_step` — the fine pass through nrf_lerf_fwd_train, the fused backward
(nrf_lerf_bwd_rays / nrf_composite_bwd / nrf_lerf_bwd_rows), nrf_hash_encode_bwd at F = 8 and ONE Adam launch over the flat vector
[language table | the four weight matrices].
"""
from __future__ import annotations

import math

import torch

from . import ops
from .ops import f16, f32
from .pipeline import FlatAdamModel, make_grid

LERF_LAYERS = (("sigma_le_net_0", 256, 128), ("sigma_le_net_1", 33, 256), ("le_net_0", 256, 160), ("le_net_1", 512, 256))


def head_forward_backward(packed, weights: dict, enc, keep, z, rays_d, target, grads: dict, loss_out=None, grad_scale=1.0, prefix="lang_model",
                          workspace=None):
    """The differentiated part of LeRFRenderer::RenderRays' fine pass + the language loss, forward and backward, on the fused kernels:
    enc [R*S,128] fp16 (hash encoding of the fine samples), keep [R*S] u8 | None, z [R,S], rays_d [R,3], target [R,512].
    grads[<prefix>_<layer>.weight] += d loss / d weight (fp32).  Returns (out dict with rendered / weights / depth / acc, d_enc [R*S,128] bf16)."""
    r, s = z.shape
    raw4, saved, q = ops.lerf_fwd_train(packed, enc, keep)
    comp = ops.composite_fwd(raw4.view(r, s, 4), z, rays_d)
    rendered, hsum, enorm = ops.lerf_render_embedding_train(packed, comp["weights"], saved, q)
    if workspace is None:
        workspace = ops.lerf_bwd_workspace(r * s, r, enc.device)
    dw = ops.lerf_bwd_rays(weights, saved, q, comp["weights"], hsum, rendered, enorm, grads[f"{prefix}_le_net_1.weight"], workspace, target=target,
                           grad_scale=grad_scale, loss_out=loss_out, prefix=prefix)
    d_raw4 = ops.composite_bwd(raw4.view(r, s, 4), z, rays_d, g_weights=dw)
    d_enc = ops.lerf_bwd_rows(packed, weights, saved, keep, d_raw4, s, workspace, grads, prefix=prefix)
    return {"rendered": rendered, "weights": comp["weights"], "depth": comp["depth"], "disp": comp["disp"], "acc": comp["acc"], "raw4": raw4, "q": q,
            "dw": dw, "d_raw4": d_raw4}, d_enc


class LeRFField(FlatAdamModel):
    """Language hash grid + LeRF head of one replica, and the LeRFRenderer stages on them.  Parameters live in ONE flat fp32 vector
    [reachable table scalars | sigma_le_net_0 | sigma_le_net_1 | le_net_0 | le_net_1] (`table` / `weights` are views), so that training is one
    gradient exchange and one Adam launch, as for HashNeRF."""

    def __init__(self, bbox=(-1.5, -1.5, -1.5, 1.5, 1.5, 1.5), n_levels=16, n_features=8, log2_hashmap_size=19, base_resolution=16,
                 finest_resolution=512, n_samples=64, n_importance=128, device="cuda", seed=42, primes=None, prefix="lang_model", lr=1e-2,
                 lrate_decay=250):
        assert n_levels * n_features == 128, "the fused head is built for 128 input channels (16 levels x 8 features)"
        self.device = torch.device(device)
        self.bbox = tuple(float(v) for v in bbox)
        self.prefix = prefix
        self.grid = make_grid(bbox, n_levels, n_features, log2_hashmap_size, base_resolution, finest_resolution, device, seed, primes)
        self.S, self.N = n_samples, n_importance
        self.n_table = self.grid.used_scalars()
        g = torch.Generator(device="cpu").manual_seed(seed)
        self._init_flat(self.n_table + sum(fo * fi for _, fo, fi in LERF_LAYERS), device, lr, lrate_decay)
        self.params[:self.n_table] = (torch.rand(self.n_table, generator=g) * 1e-4).to(device)    # src/CuHashEmbedder.cpp:24
        self.weights, self.weight_grads = {}, {}
        off = self.n_table
        for name, fo, fi in LERF_LAYERS:                                                          # Trainable.h:43 Xavier normal, gain 0.1
            view = self.params[off:off + fo * fi].view(fo, fi)
            view.copy_((torch.randn(fo, fi, generator=g) * 0.1 * math.sqrt(2.0 / (fi + fo))).to(device))
            self.weights[f"{prefix}_{name}.weight"] = view
            self.weight_grads[f"{prefix}_{name}.weight"] = self.grads[off:off + fo * fi].view(fo, fi)
            off += fo * fi
        self.t_vals = torch.linspace(0.0, 1.0, n_samples, dtype=f32).to(device)                   # src/LeRFRenderer.cpp:112
        self.u = torch.linspace(0.0, 1.0, n_importance, dtype=f32).to(device)                     # src/Sampler.h:20
        self.packed = None
        self._render_graph = None
        self.render_ray_group = 32           # render_image: GetRays order = adjacent pixels
        self.reuse_coarse_rows = True        # the fine pass copies the coarse samples' encoding rows instead of gathering them again (bit-identical)
        self._bwd_ws = None
        self.refresh()

    def repack(self):
        self.packed = ops.lerf_pack(self.weights, out=self.packed, prefix=self.prefix)

    def bind_peer_buffers(self):
        """After parallel.PeerShardedOptimizer re-pointed self.grads at symmetric memory: the per-layer gradient views follow."""
        off = self.n_table
        for name, fo, fi in LERF_LAYERS:
            self.weight_grads[f"{self.prefix}_{name}.weight"] = self.grads[off:off + fo * fi].view(fo, fi)
            off += fo * fi

    def _static_inputs(self, n_rays):
        dev = self.device
        tgt = torch.zeros((n_rays, 512), dtype=f32, device=dev)
        tgt[:, 0] = 1.0
        return (torch.tensor([[0.0, 0.0, 4.0]], device=dev).repeat(n_rays, 1), torch.tensor([[0.0, 0.0, -1.0]], device=dev).repeat(n_rays, 1), tgt)

    # -- one optimisation step of the language field (src/NeRFExecutor.h:957-983, 986-996)
    def forward_backward(self, rays_o, rays_d, target, grad_scale=1.0):
        """LeRFRenderer::RenderRays + the language loss + backward into self.grads (accumulating).  self.loss holds the loss.  The coarse pass is
        inference (it never receives a gradient, SURVEY §9-Q3); the fine pass runs the bf16 training program of the fused head."""
        r = rays_o.shape[0]
        ray_batch, z, _ = ops.ray_setup(rays_o, rays_d, self.bbox, 0.0, self.t_vals, None, zero_scalar=self.loss)
        enc_c, keep_c = ops.hash_encode_rays_fwd(self.grid, self.table_f16, ray_batch, z, clamp=True, out_f16=True)
        raw4 = ops.lerf_sigma_fwd(self.packed, enc_c, keep_c)
        coarse = ops.composite_fwd(raw4.view(r, self.S, 4), z, rays_d)
        if self.reuse_coarse_rows:
            z_fine, perm = ops.sample_pdf_merge(z, coarse["weights"], self.u, want_perm=True)
            reuse = (perm, enc_c, keep_c, z.shape[1])
        else:
            z_fine, reuse = ops.sample_pdf_merge(z, coarse["weights"], self.u), None
        s = z_fine.shape[1]
        enc, keep = ops.hash_encode_rays_fwd(self.grid, self.table_f16, ray_batch, z_fine, clamp=True, out_f16=True, reuse=reuse)
        if self._bwd_ws is None or self._bwd_ws[0] != (r, s):
            self._bwd_ws = ((r, s), ops.lerf_bwd_workspace(r * s, r, self.device))
        out, d_enc = head_forward_backward(self.packed, self.weights, enc, keep, z_fine, rays_d, target, self.weight_grads, loss_out=self.loss,
                                           grad_scale=grad_scale, prefix=self.prefix, workspace=self._bwd_ws[1])
        ops.hash_encode_rays_bwd(self.grid, ray_batch, z_fine, d_enc, self.grads[:self.n_table], clamp=True)
        out["z"] = z_fine
        return out

    def render_rays(self, rays_o, rays_d, return_embedding=False, return_weights=True, ray_group=1):
        """LeRFRenderer::RenderRays after Render's prologue (IntersectWithAABB, src/LeRFRenderer.cpp:296-302): LeRFRendererOutputs as a dict.
        ray_group > 1: the rays are neighbouring pixels of a frame — the encode kernels walk ray_group of them together (same results)."""
        r = rays_o.shape[0]
        ray_batch, z, _ = ops.ray_setup(rays_o, rays_d, self.bbox, 0.0, self.t_vals, None)
        # coarse pass: density only (RunLENetwork + the weights of RawToLEOutputs)
        enc_c, keep_c = ops.hash_encode_rays_fwd(self.grid, self.table_f16, ray_batch, z, clamp=True, out_f16=True, ray_group=ray_group)
        raw4 = ops.lerf_sigma_fwd(self.packed, enc_c, keep_c)
        coarse = ops.composite_fwd(raw4.view(r, self.S, 4), z, rays_d)
        if self.reuse_coarse_rows:                                                                # :143-147; the merged list holds the coarse z bit for bit
            z_fine, perm = ops.sample_pdf_merge(z, coarse["weights"], self.u, want_perm=True)
            reuse = (perm, enc_c, keep_c, z.shape[1])
        else:
            z_fine, reuse = ops.sample_pdf_merge(z, coarse["weights"], self.u), None
        s = z_fine.shape[1]
        # fine pass
        enc, keep = ops.hash_encode_rays_fwd(self.grid, self.table_f16, ray_batch, z_fine, clamp=True, out_f16=True, reuse=reuse, ray_group=ray_group)
        raw4, hidden, q = ops.lerf_hidden_fwd(self.packed, enc, keep)
        comp = ops.composite_fwd(raw4.view(r, s, 4), z_fine, rays_d)
        out = {"rendered": ops.lerf_render_embedding(self.packed, comp["weights"], hidden, q), "depth": comp["depth"], "disp": comp["disp"],
               "acc": comp["acc"], "z": z_fine}
        if return_weights:
            out["weights"] = comp["weights"]
        if return_embedding:
            out["raw"] = ops.lerf_fwd(self.packed, enc, keep).view(r, s, -1)                      # LeRFRenderResult::Raw
            out["embedding"] = out["raw"][..., :-1]                                               # LeRFRendererOutputs::LangEmbedding
        return out

    # -- the same chunk as ONE CUDA-graph replay (11 kernels of 3..110 us behind 11 ctypes calls are launch-bound otherwise)
    def capture_render(self, n_rays: int):
        dev = self.device
        self._g_in = (torch.tensor([[0.0, 0.0, 4.0]], device=dev).repeat(n_rays, 1), torch.tensor([[0.0, 0.0, -1.0]], device=dev).repeat(n_rays, 1))
        side = torch.cuda.Stream(device=dev)                      # warm-up outside the capture (function attributes, level scales, allocator pools)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self.render_rays(*self._g_in, return_weights=False)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        self._g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._g):
            self._g_out = self.render_rays(*self._g_in, return_weights=False)
        return self

    def render_rays_graph(self, rays_o, rays_d):
        """Replay of the captured chunk; inputs may be device tensors or pinned host tensors.  The returned tensors are overwritten by the next replay."""
        self._g_in[0].copy_(rays_o, non_blocking=True)
        self._g_in[1].copy_(rays_d, non_blocking=True)
        self._g.replay()
        return self._g_out

    def _chunk_graph(self, chunk):
        """render_rays of one full chunk as a CUDA graph (11 launches + their allocations replayed as one): a frame is hundreds of chunks, and the
        eager path is bound by the host (ctypes calls, allocator) rather than by the GPU.  Inputs / outputs are static buffers; weights and table are
        read through the persistent packed / shadow buffers, so a re-packed or trained field renders correctly without a new capture."""
        if self._render_graph is not None and self._render_graph[0] == (chunk, self.render_ray_group):
            return self._render_graph
        dev = self.device
        o = torch.tensor([[0.0, 0.0, 4.0]], device=dev).repeat(chunk, 1)
        d = torch.tensor([[0.0, 0.0, -1.0]], device=dev).repeat(chunk, 1)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            self.render_rays(o, d, return_weights=False, ray_group=self.render_ray_group)
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = self.render_rays(o, d, return_weights=False, ray_group=self.render_ray_group)
        self._render_graph = ((chunk, self.render_ray_group), g, o, d, out)
        return self._render_graph

    def render_image(self, h, w, K, c2w, chunk=1 << 15, row_begin=0, row_end=None, use_graph=True):
        """Render(h, w, K, c2w) for image rows [row_begin, row_end) (src/LeRFRenderer.cpp:266-331; chunking as BatchifyRays :165-263).  Full chunks
        replay one captured graph (use_graph), the ragged last chunk is launched eagerly; same kernels, same results."""
        rays_o, rays_d = ops.get_rays(h, w, K, c2w, row_begin, row_end, self.device)
        keys = ("rendered", "depth", "disp", "acc")
        n = rays_o.shape[0]
        outs = []
        for i in range(0, n, chunk):
            if use_graph and i + chunk <= n and n >= 2 * chunk:
                _, g, o, d, out = self._chunk_graph(chunk)
                o.copy_(rays_o[i:i + chunk])
                d.copy_(rays_d[i:i + chunk])
                g.replay()
                outs.append({k: out[k].clone() for k in keys})
            else:
                outs.append(self.render_rays(rays_o[i:i + chunk], rays_d[i:i + chunk], return_weights=False, ray_group=self.render_ray_group))
        return {k: torch.cat([o[k] for o in outs], 0) for k in keys}
