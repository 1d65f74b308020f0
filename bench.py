#!/usr/bin/env python
"""Headline benchmark: HashNeRF training throughput (rays/s) on the ray-batch hot path, BASELINE config C2/C3.

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's sm_100a path
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference's own LibTorch CPU path (oracle/_ref)

One step = render(4096 rays: 64 coarse + 128 importance samples, two network passes) + huber + backward + all-reduce
(N>1) + Adam, i.e. NeRFExecutor::Train's loop body (reference src/NeRFExecutor.h:868-996) in the parity configuration.
Prints ONE JSON line (rank 0).  See DESIGN.md §measurement for the definitions of every field.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
for p in (str(ROOT), str(ROOT / "oracle"), str(ROOT / "oracle" / "_ref")):
    if p not in sys.path:
        sys.path.insert(0, p)

RAYS_PER_GPU = 4096
N_SAMPLES, N_IMPORTANCE = 64, 128
BBOX = (-1.5, -1.5, -1.5, 1.5, 1.5, 1.5)
CPU_SAMPLE_RAYS = 256   # bounded sample of the 4096-ray step for the CPU arms
CPU_STEPS, CPU_WARMUP = 10, 2   # cpu_baseline inside the GPU line (the reference arm uses the driver's --steps / --warmup on the same sample)
MLP_BWD_PIPE = "mma.sync (HMMA) chain + tcgen05 dW"

# algorithmic bytes per unit (DESIGN.md §kernels; SURVEY §8d with this repo's fp16 encoding output)
BYTES_PER_POINT = {
    "hash_encode_fwd": 12 + 512 + 64 + 1,   # xyz in, 16 lvl x 8 corners x 2 feat x fp16 gathered, fp16 [32] out, keep byte
    "hash_encode_bwd": 12 + 64 + 2 * 512,   # xyz in, bf16 [32] grad in, read-modify-write of the 8x16 gathered entries
}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed regions (B200_PROFILING.md recipe): one `nvidia-smi -lms` process
    streaming a sample every 20 ms, started before the first timed region and stopped after the last."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.rows = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index), "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:  # noqa: BLE001 - sampling must never break the bench
            self.proc = None

    def stop(self) -> dict:
        if self.proc is not None:
            try:
                self.proc.terminate()
                out, _ = self.proc.communicate(timeout=10)
                self.rows = [[c.strip() for c in line.split(",")] for line in out.splitlines() if line.count(",") >= 6]
            except Exception:  # noqa: BLE001
                self.proc.kill()
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows if len(r) > 3 + i)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": float(self.rows[0][1]), "samples": len(self.rows),
                "power_w_max": max(float(r[2]) for r in self.rows), "reasons": reasons,
                "window": "resident + roofline + e2e timed regions"}


def reference_cpu_rays_per_s(steps: int, warmup: int, rays: int = CPU_SAMPLE_RAYS):
    """The reference's own implementation of the step — NeRFRenderer<HashEmbedder,SHEncoder,NeRFSmall> + huber + backward +
    torch::optim::Adam, LibTorch CPU fp32 on all host threads (BASELINE.md §2) — on a bounded `rays`-ray sample."""
    import torch
    import nerfpp_ref_cpu as R
    R.set_num_threads(os.cpu_count() or 1)
    R.manual_seed(42)
    devnull = os.open(os.devnull, os.O_WRONLY)   # the reference prints parameter names from Trainable::Initialize
    saved = os.dup(1)
    os.dup2(devnull, 1)
    try:
        pipe = R.make_hash_cpu(torch.tensor(BBOX), 16, 2, 19, 16, 512, 4, 2, 64, 15, 3, 64)
        pipe.init_model()
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    from nerfpp_b200.pipeline import synthetic_rays
    o, d, tgt = synthetic_rays(rays, device="cpu", seed=0)
    if warmup:
        pipe.train_steps(o, d, tgt, warmup, N_SAMPLES, N_IMPORTANCE, 4096, True, 1e-2, 250)
    secs, _ = pipe.train_steps(o, d, tgt, steps, N_SAMPLES, N_IMPORTANCE, 4096, True, 1e-2, 250)
    total = sum(secs)
    return rays * steps / total, total / steps, R.get_num_threads()


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    try:
        value, sec_per_step, threads = reference_cpu_rays_per_s(args.steps, args.warmup)
    except ImportError as e:
        print(json.dumps({"impl": "reference", "unavailable": f"oracle/_ref/nerfpp_ref_cpu.so not importable: {e}"}))
        return
    sample = f"{CPU_SAMPLE_RAYS}-ray sample of the {RAYS_PER_GPU}-ray step, {args.steps} steps after {args.warmup} warm-up"
    print(json.dumps({
        "impl": "reference", "metric": "train_rays_per_s", "value": value, "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "HashNeRF train step (L16 T2^19 F2 hash grid, SH4, 2x64 + 3x64 MLP), 64+128 samples/ray, "
                               f"{CPU_SAMPLE_RAYS}-ray bounded sample of the 4096-ray batch, LibTorch CPU"},
        "cpu_baseline": {"value": value, "unit": "rays/s", "cores": threads, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def _graph_timed(fn, reps: int) -> float:
    """ms per launch of `fn` (C-ABI launches on torch's current stream): `reps` launches captured in ONE CUDA graph and replayed, so
    the figure is device time of back-to-back launches, not ctypes / allocator time on the host (these kernels take 5-400 us)."""
    import torch
    fn()
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fn()
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            for _ in range(reps):
                fn()
    torch.cuda.current_stream().wait_stream(side)
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def render_ops_leg(hbm_peak: float, reps: int = 20) -> dict:
    """HBM roofline of the CustomOps / RayUtils rendering kernels (compositing forward / backward, sample_pdf + merge), each timed alone
    with a CUDA-event pair over `reps` launches at two sizes: the fine pass of one 4096-ray training step (64+128 samples) and a
    262 144-ray render tile (BASELINE C4: one GPU's share of a 1080p frame, 64+64 samples).  Algorithmic bytes per SURVEY §8(d):
    forward 24 B/sample + 44 B/ray, backward 40 B/sample + 12 B/ray of map gradients, sampler 4 B x (2S + N + S+N) per ray.
    The same buffers are re-read by every launch: the small size (19 MB) is L2-resident, as it is inside the training step; the
    large size (0.8-1.3 GB per launch) cannot be."""
    import torch
    from nerfpp_b200 import ops

    def timed(fn):
        return _graph_timed(fn, reps)

    out = {"unit": "GB/s", "peak": hbm_peak, "sizes": {}}
    g = torch.Generator().manual_seed(0)
    for tag, rays, s_c, n_imp in (("train_fine_4096x192", 4096, 64, 128), ("render_tile_262144x128", 262144, 64, 64)):
        s = s_c + n_imp
        raw = torch.randn(rays, s, 4, generator=g).cuda()
        z = (2 + torch.sort(torch.rand(rays, s, generator=g) * 4, -1).values).cuda()
        d = torch.randn(rays, 3, generator=g).cuda()
        g_rgb = torch.randn(rays, 3, generator=g).cuda()
        d_raw = torch.empty_like(raw)
        zc = z[:, :s_c].contiguous()
        w = torch.rand(rays, s_c, generator=g).cuda()
        u = torch.linspace(0, 1, n_imp).cuda()
        from nerfpp_b200.cabi import lib, ptr, stream
        maps = [torch.empty(rays, 3, device="cuda")] + [torch.empty(rays, device="cuda") for _ in range(3)] + [torch.empty(rays, s, device="cuda")]
        merged = torch.empty(rays, s, device="cuda")
        ms_f = timed(lambda: lib().nrf_composite_fwd(ptr(raw), 4, ptr(z), ptr(d), None, 0.0, 0, rays, s, *[ptr(m) for m in maps], stream()))
        ms_b = timed(lambda: lib().nrf_composite_bwd(ptr(raw), 4, ptr(z), ptr(d), None, 0.0, 0, rays, s, ptr(g_rgb), None, None, None, None, ptr(d_raw),
                                                       stream()))
        ms_s = timed(lambda: lib().nrf_sample_pdf_merge(ptr(zc), ptr(w), ptr(u), 0, rays, s_c, n_imp, None, ptr(merged), stream()))
        by_f, by_b, by_s = rays * (s * 24 + 44), rays * (s * 40 + 24), rays * 4 * (2 * s_c + n_imp + s)
        out["sizes"][tag] = {
            "composite_fwd": {"ms": ms_f, "achieved": by_f / ms_f / 1e6, "frac": by_f / ms_f / 1e6 / hbm_peak, "bytes": by_f},
            "composite_bwd": {"ms": ms_b, "achieved": by_b / ms_b / 1e6, "frac": by_b / ms_b / 1e6 / hbm_peak, "bytes": by_b},
            "sample_pdf_merge": {"ms": ms_s, "achieved": by_s / ms_s / 1e6, "frac": by_s / ms_s / 1e6 / hbm_peak, "bytes": by_s}}
        del raw, z, d_raw
    return out


def classic_nerf_leg(tf_peak: float, rows: int = 1024 * 192, reps: int = 10) -> dict:
    """BASELINE C1's network (NeRFImpl 8x256, src/NeRF.cpp:92-126) at one 1024-ray training batch of 64+128 samples (196 608 rows):
    inference forward, training forward (stores the layer inputs) and backward (gradient chain + weight gradients), each timed with
    a CUDA-event pair over `reps` launches.  1.187 MFLOP/row forward, 2x that backward (no input gradient: layer 0 has dW only)."""
    import ctypes
    import math

    import torch
    from nerfpp_b200 import ops
    g = torch.Generator().manual_seed(0)
    shapes = {f"model_pts_linears_{i}": (256, 63 if i == 0 else (319 if i == 5 else 256)) for i in range(8)}
    shapes.update({"model_feature_linear": (256, 256), "model_alpha_linear": (1, 256), "model_views_linears_0": (128, 283), "model_rgb_linear": (3, 128)})
    p = {}
    for name, (o, i) in shapes.items():
        p[name + ".weight"] = (torch.randn(o, i, generator=g) * math.sqrt(2.0 / i)).cuda()
        p[name + ".bias"] = (torch.randn(o, generator=g) * 0.1).cuda()
    x = (torch.rand(rows, 90, generator=g) * 2 - 1).cuda()
    gout = (torch.randn(rows, 4, generator=g) * 1e-3).cuda()
    packed, packed_t = ops.mlp_nerf_pack(p), ops.mlp_nerf_pack(p, train=True)
    grads = {k: torch.zeros_like(v) for k, v in p.items()}
    out, saved = ops.mlp_nerf_fwd_train(packed_t, x)
    ws = torch.empty(ops.lib().nrf_mlp_nerf_bwd_workspace_bytes(ctypes.byref(ops.mlp_nerf_shape()), rows), dtype=torch.uint8, device="cuda")

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms_inf = timed(lambda: ops.mlp_nerf_fwd(packed, x, out=out))
    ms_fwd = timed(lambda: ops.mlp_nerf_fwd_train(packed_t, x))
    ms_bwd = timed(lambda: ops.mlp_nerf_bwd(packed_t, saved, gout, grads, workspace=ws))
    fl = rows * 1.186816e6
    bwd_flop = 2 * fl - rows * 2 * (63 * 256 + 63 * 256 + 27 * 128)      # no dX for the embedded inputs
    return {"rows": rows, "config": "C1 network: 8x256 + skip + view branch, one 1024-ray batch x (64+128) samples",
            "fwd_inference": {"ms": ms_inf, "achieved": fl / ms_inf / 1e9, "frac": fl / ms_inf / 1e9 / tf_peak, "dtype": "fp16"},
            "fwd_train": {"ms": ms_fwd, "achieved": fl / ms_fwd / 1e9, "frac": fl / ms_fwd / 1e9 / tf_peak, "dtype": "bf16",
                          "saved_bytes": int(saved.numel())},
            "bwd": {"ms": ms_bwd, "achieved": bwd_flop / ms_bwd / 1e9, "frac": bwd_flop / ms_bwd / 1e9 / tf_peak, "dtype": "bf16",
                    "kernels": "mlp_nerf_bwd_chain_kernel + mlp_nerf_bwd_dw_kernel"}}


def lerf_leg(tf_peak: float, rays: int = 1024, reps: int = 10) -> dict:
    """BASELINE C5's language head (LeRF(32, 2, 256, 512, 128), src/LeRF.cpp:28-111) at one 1024-ray batch of 64 + 128 samples: the three
    stage programs of the fused tcgen05 kernel and the per-ray finish, each timed with a CUDA-event pair over `reps` launches, and the whole
    LeRFRenderer::RenderRays (inference).  FLOP counts are the REFERENCE's (the full 512-wide last layer), not the issued ones."""
    import torch
    from nerfpp_b200 import ops
    from nerfpp_b200.lerf import LeRFField
    f = LeRFField(seed=0)
    g = torch.Generator().manual_seed(0)
    for v in f.weights.values():
        v.copy_((torch.randn(v.shape, generator=g) * (2.0 / v.shape[1]) ** 0.5).cuda())
    f.table.copy_((torch.rand(f.n_table, generator=g) * 2 - 1).cuda())
    f.refresh()
    n_c, n_f = rays * 64, rays * 192
    enc_c, enc_f = torch.randn(n_c, 128, generator=g).half().cuda(), torch.randn(n_f, 128, generator=g).half().cuda()
    w = torch.rand(rays, 192, generator=g).cuda()

    def timed(fn):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    ms_sigma = timed(lambda: ops.lerf_sigma_fwd(f.packed, enc_c))
    ms_hidden = timed(lambda: ops.lerf_hidden_fwd(f.packed, enc_f))
    _, hidden, q = ops.lerf_hidden_fwd(f.packed, enc_f)
    ms_finish = timed(lambda: ops.lerf_render_embedding(f.packed, w, hidden, q))
    ms_raw = timed(lambda: ops.lerf_fwd(f.packed, enc_f))
    from nerfpp_b200.pipeline import synthetic_rays
    o, d, _ = synthetic_rays(rays, seed=3)
    ms_render = timed(lambda: f.render_rays(o, d, return_weights=False))
    # per-kernel shares of the chunk: one CUDA-event pair around every C-ABI call over `reps` eager chunks
    kt = ops.KernelTimer()
    ops.set_timer(kt)
    for _ in range(reps):
        f.render_rays(o, d, return_weights=False)
    torch.cuda.synchronize()
    ops.set_timer(None)
    kernels_ms = {k: round(ms / reps, 4) for k, (_, ms) in sorted(kt.summary().items(), key=lambda kv: -kv[1][1])}
    f.capture_render(rays)
    ms_render_graph = timed(lambda: f.render_rays_graph(o, d))
    fl_sigma, fl_full = 2 * (128 * 256 + 256 * 33), 2 * (128 * 256 + 256 * 33 + 160 * 256 + 256 * 512)

    def tf(rows, flop, ms):
        return rows * flop / ms / 1e9

    return {"rays": rays, "config": "C5 language head: LeRF(32,2,256,512,128) on a 16x8 hash grid, 1024 rays x (64 coarse + 192 fine) samples, inference",
            "sigma_program": {"rows": n_c, "ms": ms_sigma, "achieved": tf(n_c, fl_sigma, ms_sigma), "frac": tf(n_c, fl_sigma, ms_sigma) / tf_peak},
            "hidden_program_plus_finish": {"rows": n_f, "ms": ms_hidden + ms_finish, "ms_tc_kernel": ms_hidden, "ms_per_ray_finish": ms_finish,
                                           "achieved": tf(n_f, fl_full, ms_hidden + ms_finish), "frac": tf(n_f, fl_full, ms_hidden + ms_finish) / tf_peak,
                                           "note": "reference-equivalent FLOPs (512-wide last layer); issued: 303 kFLOP/row (G = W^T W norm layer)"},
            "raw_program": {"rows": n_f, "ms": ms_raw, "achieved": tf(n_f, fl_full, ms_raw), "frac": tf(n_f, fl_full, ms_raw) / tf_peak,
                            "hbm_gbs": n_f * (513 * 4 + 256) / ms_raw / 1e6, "note": "writes raw_le [N,513] fp32 (the reference's layout)"},
            "render_rays": {"ms": ms_render_graph, "rays_per_s": rays / ms_render_graph * 1e3, "ms_eager": ms_render, "kernels_ms_per_chunk": kernels_ms, "dtype": "fp16 operands, fp32 accumulate",
                            "note": "LeRFRenderer::RenderRays of one 1024-ray chunk (11 kernels) replayed as one CUDA graph; ms_eager = the same through 11 ctypes calls"}}


def graph_breakdown(model, batch, world: int, reps: int = 20) -> dict:
    """Per-launch device times INSIDE the step: the same step captured a second time with an external CUDA-event pair around every
    C-ABI call (event-record nodes in the graph), replayed `reps` times.  No host launch gaps, the L2 state each kernel sees is the
    step's own.  Returns {entry name: [ms per launch, in launch order]} (hash_encode_fwd: [coarse, fine])."""
    import torch
    from nerfpp_b200 import ops
    timer = ops.KernelTimer(external=True)
    model._init_sched()
    model._sync_sched()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            ops.set_timer(timer)
            try:
                model.forward_backward(*batch)
                if model.peer is not None:
                    model._optimizer_step_sharded()
                elif world == 1:
                    model._optimizer_step_scheduled(1.0)
                else:
                    model.grads.zero_()      # NCCL path: the all-reduce + Adam are not part of this breakdown (replicas must stay identical)
            finally:
                ops.set_timer(None)
    torch.cuda.current_stream().wait_stream(side)
    acc = {k: [0.0] * len(v) for k, v in timer.records.items()}
    for _ in range(reps):
        graph.replay()
        torch.cuda.synchronize()
        for k, v in timer.records.items():
            for j, (e0, e1) in enumerate(v):
                acc[k][j] += e0.elapsed_time(e1)
        model.step += 1
        model._sched_step = model.step
    return {k: [t / reps for t in v] for k, v in acc.items()}


def gpu_loop_leg(which: str, rays: int, steps: int) -> dict:
    """NeRFExecutor::Train's loop (Render + huber + backward + Adam, reference src/NeRFExecutor.h:868-996) in C++ on one GPU at the C2 shape:
    `reference_cuda` = the reference's own CUDA instantiation NeRFRenderer<CuHashEmbedder,CuSHEncoder,NeRFSmall> (oracle/_ref/nerfpp_ref_cuda.so,
    unmodified sources, nvcc -arch=sm_100) — the same-box GPU comparison of SURVEY §8(d); `dropin_cpp` = the SAME loop on this repo's C++
    drop-in classes (nerfpp_b200/lib/nerfpp_b200_torch.so).  Timed with CUDA events around `steps` steps after 5 warm-up steps."""
    import torch
    from nerfpp_b200.pipeline import synthetic_rays
    if which == "reference_cuda":
        import nerfpp_ref_cuda as R
    else:
        from nerfpp_b200 import build
        sys.path.insert(0, str(build.build_host().parent))
        import nerfpp_b200_torch as R
    R.manual_seed(42)
    devnull = os.open(os.devnull, os.O_WRONLY)   # the reference prints parameter names from Trainable::Initialize
    saved = os.dup(1)
    os.dup2(devnull, 1)
    try:
        pipe = R.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, 19, 16, 512, 4, 2, 64, 15, 3, 64)
        pipe.init_model()
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    fast = which == "dropin_cpp" and hasattr(pipe, "use_train_graph")
    if which == "dropin_cpp":
        pipe.use_fused_adam(True)
        if fast:
            pipe.use_train_graph(True)
    o, d, tgt = synthetic_rays(rays, device="cuda", seed=0)
    pipe.train_steps(o, d, tgt, 5, N_SAMPLES, N_IMPORTANCE, rays, True, 1e-2, 250)   # warm-up; single chunk (SURVEY §9-Q1)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    secs, losses = pipe.train_steps(o, d, tgt, steps, N_SAMPLES, N_IMPORTANCE, rays, True, 1e-2, 250)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"ms_per_step": ms, "value": rays / ms * 1e3, "unit": "rays/s", "rays": rays, "steps": steps, "loss_last": losses[-1],
            "loop": "C++: Render + huber_loss + backward + Adam per step, loss.item() every step (the reference's own loop)",
            "impl": ("reference CUDA path (CuHashEmbedder/CuSHEncoder kernels + LibTorch), unmodified, on this B200" if which == "reference_cuda" else
                     "nerfpp_b200 C++ drop-in classes (torch::Tensor boundary, FusedAdam" + (", captured train graph)" if fast else ")"))}


def cpp_render_leg(which: str) -> dict:
    """BASELINE C4 through the C++ surface: NeRFRenderer::Render(h, w, K, params, c2w) (src/NeRFRenderer.h:530-604) of one 1920x1080 frame, 64 + 64
    samples, 131072-ray chunks, NoGradGuard — `dropin_cpp`: this repo's drop-in classes (RenderRays = one C-ABI call per chunk), `dropin_cpp_staged`:
    the same classes with the one-call path switched off (stage by stage, the path training takes), `reference_cuda`: the reference's own classes
    and CUDA kernels on this B200.  Random-init weights with O(1) table values.  Two frames after one warm-up frame, CUDA events."""
    import math
    import torch
    if which == "reference_cuda":
        import nerfpp_ref_cuda as R
    else:
        from nerfpp_b200 import build
        sys.path.insert(0, str(build.build_host().parent))
        import nerfpp_b200_torch as R
    R.manual_seed(42)
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    os.dup2(devnull, 1)
    try:
        pipe = R.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, 19, 16, 512, 4, 2, 64, 15, 3, 64)
        pipe.init_model()
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    if which != "reference_cuda":
        pipe.use_fused_inference(which == "dropin_cpp")
    H, W = 1080, 1920
    focal = 0.5 * W / math.tan(0.5 * 0.6911)
    K = torch.tensor([[focal, 0, 0.5 * W], [0, focal, 0.5 * H], [0, 0, 1]]).cuda()
    c2w = torch.eye(4)
    c2w[2, 3] = 4.0
    c2w = c2w.cuda()
    frames = 2 if which != "reference_cuda" else 1
    torch.cuda.empty_cache()                        # the legs before this one leave the caching allocator fragmented: start from a clean pool
    for _ in range(2 if which != "reference_cuda" else 1):
        pipe.render_image(H, W, K, c2w, N_SAMPLES, 64, 131072, False, True)      # untimed: workspace, output maps and the cat buffers reach their sizes
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(frames):
        out = pipe.render_image(H, W, K, c2w, N_SAMPLES, 64, 131072, False, True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / frames
    assert tuple(out["rgb"].shape[:2]) == (H, W)
    return {"ms_per_frame": ms, "msamples_per_s": H * W * (N_SAMPLES + N_SAMPLES + 64) / (ms * 1e3), "frames": frames, "impl": which}


def shipped_shape_leg(dev, rays: int, steps: int = 50) -> dict:
    """The network shape src/main.cpp:176-191 ships: SH degree 8 (64 view channels into NeRFSmall), finest resolution 1024, 64 + 192 samples —
    parity configuration (thin rays, no noise), one CUDA graph.  The 64 view channels enter the fused kernels as a per-ray bias of the colour
    net's first layer (NRF_MLP_IN_ENC16_RAYBIAS): two small per-ray kernels on top of the C2 step's launches."""
    import torch
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    m = HashNeRF(BBOX, finest_resolution=1024, sh_degree=8, n_samples=N_SAMPLES, n_importance=192, device=dev, seed=42)
    batch = synthetic_rays(rays, device=dev, seed=31)
    m.capture_train_step(rays)
    for _ in range(5):
        m.train_step_graph(*batch)
    torch.cuda.synchronize(dev)
    first = float(m.loss)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        m.train_step_graph(*batch)
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {"ms_per_step": ms, "value": rays / ms * 1e3, "unit": "rays/s", "steps": steps, "kernels_per_step": m.graph_kernels_per_step,
            "loss": {"first": first, "last": float(m.loss)},
            "config": f"src/main.cpp:176-191 shape: L16 F2 T2^19 16->1024 grid, SH degree 8 (64 view channels), NeRFSmall 32->64->16 | 79->64->64->3, "
                      f"{rays} rays x (64 coarse + 192 importance) samples, parity configuration, one CUDA graph"}


def shipped_leg(dev, rays: int, steps: int = 50) -> dict:
    """BASELINE C2, second run (SURVEY §8d): the step with the RNG-gated stages of the reference's shipped configuration ON — thin_ray = false
    (in-cone jitter of both passes, src/NeRFRenderer.h:307-362), raw_noise_std 0.5 and stochastic preconditioning alpha = 0.01 x bbox diagonal
    (mid-schedule values of src/NeRFExecutor.h:411-412) — at the BASELINE shape, captured as one CUDA graph (torch's Philox generator is
    graph-safe: the offset advances per replay).  The jittered sample points are explicit arrays here, so both passes gather from a point list."""
    import torch
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    m = HashNeRF(BBOX, n_samples=N_SAMPLES, n_importance=N_IMPORTANCE, device=dev, seed=42)
    batch = synthetic_rays(rays, device=dev, seed=31)
    cone, noise_std, alpha = (1.0 / 1111.1 + 1.0 / 1111.1) / 2.0, 0.5, 0.01 * (3 * 3.0 ** 2) ** 0.5
    m._init_sched()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        m.forward_backward_shipped(*batch, cone, noise_std, alpha)
        m.grads.zero_()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.forward_backward_shipped(*batch, cone, noise_std, alpha)
        m._optimizer_step_scheduled(1.0)
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize(dev)
    first = float(m.loss)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        g.replay()
    e1.record()
    torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / steps
    return {"ms_per_step": ms, "value": rays / ms * 1e3, "unit": "rays/s", "steps": steps, "loss": {"first": first, "last": float(m.loss)},
            "config": f"C2 shape, {rays} rays, thin_ray = false (cone jitter both passes), raw_noise_std {noise_std}, stochastic preconditioning alpha "
                      f"{alpha:.4f} + ReflectBoundary; torch Philox draws (the reference's own rand / randn calls), everything else C ABI; one CUDA graph"}


def lerf_train_leg(rank: int, world: int, dev, hash_model, tf_peak: float, rays: int = 1024, steps: int = 50) -> dict | None:
    """BASELINE C5: LeRF training, 1024 rays per GPU.  One iteration of NeRFExecutor::Train with use_lerf (src/NeRFExecutor.h:868-996) = the HashNeRF
    step (render + huber + backward) AND the language step (LeRFRenderer::Render + huber(1.25).sum(-1).nanmean() + backward, :957-983), then Adam
    over both parameter sets.  Timed: the language step alone and the joint iteration (both captured graphs replayed back to back), CUDA events,
    max over ranks.  Collective: every rank calls it."""
    import torch
    from nerfpp_b200 import ops, parallel
    from nerfpp_b200.lerf import LeRFField
    from nerfpp_b200.pipeline import synthetic_rays
    out, ready, field = {}, True, None
    try:
        # same seed on every rank: identical replicas without a broadcast.  lr 5e-4: with O(1) weights the reference's 1e-2 kills the density within ~50
        # steps (relu on sigma: every weight -> 0, every gradient -> 0) and the scatter / chain kernels would be timed on the all-zero skip path
        field = LeRFField(BBOX, seed=0, device=dev, lr=5e-4)
        g = torch.Generator().manual_seed(0)
        for v in field.weights.values():                       # O(1) signals (He-scaled weights, table U(-1,1)): every ReLU / density regime is exercised
            v.copy_((torch.randn(v.shape, generator=g) * (2.0 / v.shape[1]) ** 0.5).to(dev))
        field.params[:field.n_table].copy_((torch.rand(field.n_table, generator=g) * 2 - 1).to(dev))
        field.refresh()
    except Exception as e:  # noqa: BLE001 - a secondary leg must not take the headline line down
        ready, out = False, {"error": f"{type(e).__name__}: {e}"}
    if not parallel.all_ranks_ready(ready, world, dev):
        return out or {"error": "set-up failed on another rank"}
    dp_mode, dp_check = "single", None
    if world > 1:
        dp_mode = "nccl all-reduce of the flat gradient + dense Adam"
        try:
            peer = parallel.PeerShardedOptimizer(field, rank, world)
        except Exception as e:  # noqa: BLE001
            peer, dp_mode = None, dp_mode + f" (fused path unavailable: {type(e).__name__}: {e})"
        have = torch.tensor([int(peer is not None)], dtype=torch.int32, device=dev)
        torch.distributed.all_reduce(have, op=torch.distributed.ReduceOp.MIN)
        if bool(have.item()):
            dp_check = peer.dp_check(field)
        if dp_check is not None and dp_check["ok"]:
            dp_mode = "fused peer-memory kernel (reduce-scatter + Adam + fp16 shadow all-gather over NVLink)"
        else:
            field.peer = None
    pool = 4
    batches = []
    for i in range(pool):
        o, d, _ = synthetic_rays(rays, device=dev, seed=5000 + 1000 * rank + i)
        tgt = torch.nn.functional.normalize(torch.randn(rays, 512, generator=torch.Generator().manual_seed(9000 + 1000 * rank + i)), dim=-1).to(dev)
        batches.append((o, d, tgt))
    nerf_batches = [synthetic_rays(rays, device=dev, seed=6000 + 1000 * rank + i) for i in range(pool)]
    field.capture_train_step(rays, world, lambda gr: parallel.allreduce_gradients(gr, world))
    hash_model.capture_train_step(rays, world, lambda gr: parallel.allreduce_gradients(gr, world))

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()

    def timed(fn):
        for i in range(3):
            fn(i)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        sync_all()
        return parallel.max_over_ranks(e0.elapsed_time(e1), world, dev) / steps

    losses = []
    ms_lang = timed(lambda i: losses.append(field.train_step_graph(*batches[i % pool])) if i % 10 == 0 else field.train_step_graph(*batches[i % pool]))
    loss_first, loss_last = float(field.loss), None
    ms_joint = timed(lambda i: (hash_model.train_step_graph(*nerf_batches[i % pool]), field.train_step_graph(*batches[i % pool])))
    loss_last = float(field.loss)
    per_launch = graph_breakdown(field, batches[0], world, reps=10)
    if field.peer is not None:
        field.peer.check()
    rows = rays * (N_SAMPLES + N_IMPORTANCE)
    fwd_ms, bwd_ms = per_launch.get("lerf_fwd_train", [0.0])[0], per_launch.get("lerf_bwd_rows", [0.0])[0]
    fl_fwd, fl_bwd = rows * 303104, rows * 606208
    return {"metric": "lerf_train_rays_per_s", "value": rays * world / (ms_joint * 1e-3), "unit": "rays/s", "ms_per_step": ms_joint, "steps": steps,
            "rays_per_gpu": rays, "n_gpus": world, "scaling": "weak",
            "language_step_only": {"ms_per_step": ms_lang, "value": rays * world / (ms_lang * 1e-3), "kernels_per_step": field.graph_kernels_per_step},
            "loss": {"after_language_only_leg": loss_first, "after_joint_leg": loss_last},
            "kernels_ms_per_step": {k: [round(t, 4) for t in v] for k, v in sorted(per_launch.items(), key=lambda kv: -sum(kv[1]))},
            "roofline_tensor": {"peak": tf_peak, "unit": "TFLOP/s", "rows": rows,
                                "lerf_head_fwd_train": {"ms": fwd_ms, "achieved": fl_fwd / max(fwd_ms, 1e-9) / 1e9, "frac": fl_fwd / max(fwd_ms, 1e-9) / 1e9 / tf_peak,
                                                        "flop_per_row": 303104},
                                "lerf_head_bwd": {"ms": bwd_ms, "achieved": fl_bwd / max(bwd_ms, 1e-9) / 1e9, "frac": fl_bwd / max(bwd_ms, 1e-9) / 1e9 / tf_peak,
                                                  "flop_per_row": 606208, "kernels": "lerf_bwd_chain_kernel + mlp_nerf_bwd_dw_kernel (4 units) + lerf_gram_apply_kernel"}},
            "dp_check": dp_check, "parallelism": f"ray-sharded dp{world}: {dp_mode}",
            "config": "BASELINE C5: HashNeRF (L16 F2 T2^19 + SH4 + NeRFSmall) and the language field (L16 F8 T2^19 grid + LeRF(32,2,256,512,128)) trained jointly, "
                      f"{rays} rays/GPU/step, 64 + 128 samples, random unit 512-d targets; random-init O(1) language weights"}


def dump_outputs(out_dir: str, model, step_out: dict, rank: int, max_rows: int = 8192) -> None:
    """Writes what the last timed training step computed as <out_dir>/<name>.npy, float32: the loss, the fine pass's rgb [R,3] and depths z [R,S+N]
    of rank 0's rays (a fixed, seeded sample of max_rows rays when R is larger) and the parameters after the step's Adam update (hash table +
    NeRFSmall weights, 8.9 M values at the benchmark's shape; under 64 MB in all).  Collective under the fused data-parallel optimiser."""
    import numpy as np
    import torch
    params = model.state_dict()["params"]          # gathers the owners' shards first under the fused optimiser
    if rank != 0:
        return
    rgb, z = step_out["rgb"], step_out["z"]
    if rgb.shape[0] > max_rows:
        rows = torch.randperm(rgb.shape[0], generator=torch.Generator().manual_seed(0))[:max_rows].sort().values.to(rgb.device)
        rgb, z = rgb[rows], z[rows]
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    for name, t in (("loss", model.loss), ("rgb", rgb), ("z", z), ("params", params)):
        np.save(d / f"{name}.npy", t.detach().float().cpu().numpy())


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200,
                    help="timed steps of the headline (its resident and e2e regions); the secondary legs keep their own step counts")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rays", type=int, default=RAYS_PER_GPU, help="rays per GPU per step (weak scaling, the headline)")
    ap.add_argument("--global-rays", type=int, default=8 * RAYS_PER_GPU,
                    help="global batch of the strong-scaling sub-record (BASELINE C3: 8 x 4096 rays split over the GPUs); 0 = skip")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel eagerly instead of replaying the captured step")
    ap.add_argument("--quick", action="store_true", help="headline + roofline only: skip the render / LeRF / classic / C++-loop legs")
    ap.add_argument("--dp", default="fused", choices=["fused", "nccl"],
                    help="N>1 optimiser step: one peer-memory kernel (reduce-scatter + Adam + shadow all-gather) or NCCL all-reduce + dense Adam")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the headline's timed steps, write what its last step computed (loss, fine-pass rgb and z of rank 0's rays, the "
                         "updated parameters) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of this repository's path: it does not apply to --impl reference")
    # stdout carries exactly ONE JSON line: everything native libraries print on file descriptor 1 while the job runs (NCCL's version
    # banner, for one) is sent to stderr; the line itself goes to the saved descriptor at the end
    sys.stdout.flush()
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real_stdout
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    from nerfpp_b200 import cabi, ops, parallel
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback (use --impl reference for the CPU arm)")
    rank, world, local_rank = parallel.init_from_env()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    warmup = max(args.warmup, 3)
    R = args.rays

    model = HashNeRF(BBOX, n_samples=N_SAMPLES, n_importance=N_IMPORTANCE, device=dev, seed=42)
    parallel.broadcast_parameters(model.params, world)
    model.refresh()

    dp_mode, dp_check = "single", None
    if world > 1:
        dp_mode = "nccl all-reduce of the flat gradient + dense Adam on every rank"
        if args.dp == "fused":
            why = ""
            try:
                peer = parallel.PeerShardedOptimizer(model, rank, world)
            except Exception as e:  # noqa: BLE001 - symmetric memory unavailable on this rank
                peer, why = None, f"{type(e).__name__}: {e}"
            have = torch.tensor([int(peer is not None)], dtype=torch.int32, device=dev)
            torch.distributed.all_reduce(have, op=torch.distributed.ReduceOp.MIN)      # all ranks or none
            if bool(have.item()):
                # one step on a RANDOM gradient through the fused kernel and through NCCL all-reduce + dense Adam, compared (collective)
                dp_check = peer.dp_check(model)
            if dp_check is not None and dp_check["ok"]:
                dp_mode = "fused peer-memory kernel per rank: reduce-scatter(grad) + Adam(1/N shard) + all-gather(fp16 shadow) over NVLink, no NCCL in the step"
            else:
                model.peer = None        # stay on the NCCL path (the symmetric buffers remain ordinary device memory) and say so
                dp_mode += f" (fused path unavailable: {why or 'dp_check failed: ' + json.dumps(dp_check)})"

    pool = 8  # distinct pre-generated ray batches per rank, cycled

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            torch.distributed.barrier()

    def eager_step(batch):
        model.forward_backward(*batch)
        if model.peer is not None:
            model.optimizer_step_sharded()
        else:
            scale = parallel.allreduce_gradients(model.grads, world)
            model.optimizer_step(grad_scale=scale)

    def train_leg(rays_per_gpu: int, steps: int, n_warm: int, seed0: int, with_e2e: bool, dump_dir: str | None = None):
        """Timed regions of one configuration.  What a step consumes is the list of pixels sampled for it (NeRFDataset::get_batch draws them,
        src/NeRFDataset.cpp:154-155): rays (GetRayBatch, :109-144) and targets (the image gather, :156) are formed on the device inside the step's
        first kernel from the resident training view (HashNeRF.set_camera).  value: `steps` replays of the captured step with the pixel lists
        resident in HBM; e2e: the same call with pinned HOST int32 [R,2] lists (H2D inside the timed region) and a D2H read of the loss every
        step.  CUDA events, max over ranks."""
        from nerfpp_b200.pipeline import synthetic_pixels, synthetic_view
        dev_batches = [synthetic_rays(rays_per_gpu, device=dev, seed=seed0 + 1000 * rank + i) for i in range(pool)]
        for i in range(n_warm):
            eager_step(dev_batches[i % pool])
        K_view, c2w_view = synthetic_view(800, 800)
        image = torch.rand(800, 800, 3, generator=torch.Generator().manual_seed(77)).to(dev)
        model.set_camera(image, K_view, c2w_view)
        host_pix = [synthetic_pixels(rays_per_gpu, 800, 800, seed=seed0 + 3000 + 1000 * rank + i).pin_memory() for i in range(pool)]
        dev_pix = [p.to(dev) for p in host_pix]
        use_graph = not args.no_graph
        last_out = {}
        if use_graph:
            model.capture_train_step(rays_per_gpu, world, lambda g: parallel.allreduce_gradients(g, world), pixels=True)
            step = lambda pix: model.train_step_graph(pix)   # noqa: E731 - copies the pixel list (device or pinned host) into its static input
            launches_per_step = model.graph_kernels_per_step
        else:
            stage_pix = torch.empty((rays_per_gpu, 2), dtype=torch.int32, device=dev)

            def step(pix):
                stage_pix.copy_(pix, non_blocking=True)
                fb_out = model.forward_backward(stage_pix)
                if dump_dir is not None:
                    last_out.update(fb_out)
                if model.peer is not None:
                    model.optimizer_step_sharded()
                else:
                    model.optimizer_step(grad_scale=parallel.allreduce_gradients(model.grads, world))
            l0 = cabi.launch_count()
            step(dev_pix[0])
            launches_per_step = cabi.launch_count() - l0 + 1
        for i in range(3):
            step(dev_pix[i % pool])
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(dev_pix[i % pool])
        e1.record()
        sync_all()
        out = {"ms_total": parallel.max_over_ranks(e0.elapsed_time(e1), world, dev), "loss": float(model.loss), "launches_per_step": launches_per_step,
               "dev_batches": dev_batches, "use_graph": use_graph}
        if dump_dir is not None:
            dump_outputs(dump_dir, model, model.graph_outputs if use_graph else last_out, rank)
        if with_e2e:
            for i in range(3):
                step(host_pix[i % pool])
            sync_all()
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record()
            loss_host = 0.0
            for i in range(steps):
                step(host_pix[i % pool])
                loss_host = float(model.loss)   # device -> host read of the step's result
            e3.record()
            sync_all()
            out.update(ms_e2e=parallel.max_over_ranks(e2.elapsed_time(e3), world, dev), loss_e2e=loss_host,
                       h2d=host_pix[0].numel() * host_pix[0].element_size())
        return out

    # ---- headline: weak scaling, R rays per GPU (BASELINE C2 at N=1; C3's per-GPU share at N=8)
    sampler = ClockSampler(local_rank)
    sampler.start()
    head = train_leg(R, args.steps, warmup, 0, with_e2e=True, dump_dir=args.dump_outputs)
    clocks = sampler.stop()
    ms_total, ms_e2e, use_graph, launches_per_step = head["ms_total"], head["ms_e2e"], head["use_graph"], head["launches_per_step"]
    dev_batches = head["dev_batches"]
    launches = launches_per_step * args.steps   # kernels inside the resident timed region (graph: kernel nodes per replay x replays)

    # ---- per-launch device times inside the step (second capture with external event pairs), for the roofline and the breakdown
    per_launch = graph_breakdown(model, dev_batches[0], world)
    if model.peer is not None:
        model.peer.check()
    timeout_after = model.flags_timeout() if model.peer is not None else 0
    if world > 1:
        timeout_after = int(parallel.max_over_ranks(float(timeout_after), world, dev))

    # ---- BASELINE C3 as written: a FIXED global batch of 8 x 4096 rays split over the ranks (strong scaling)
    strong = None
    if args.global_rays and args.global_rays % world == 0 and not args.no_graph:
        rs = args.global_rays // world
        if rs == R:
            strong = {"global_rays": args.global_rays, "rays_per_gpu": rs, "ms_per_step": ms_total / args.steps,
                      "value": args.global_rays * args.steps / (ms_total / 1e3), "steps": args.steps, "note": "same configuration as the headline at this N"}
        else:
            s_steps = max(10, min(args.steps, 50))
            leg = train_leg(rs, s_steps, 3, 7000, with_e2e=False)
            strong = {"global_rays": args.global_rays, "rays_per_gpu": rs, "ms_per_step": leg["ms_total"] / s_steps,
                      "value": args.global_rays * s_steps / (leg["ms_total"] / 1e3), "steps": s_steps}
        strong.update(unit="rays/s", scaling="strong",
                      config="BASELINE C3: fixed global batch of 8 x 4096 rays per step, ray-sharded over the GPUs (32768 / 16384 / 8192 / 4096 rays per GPU at "
                             "N = 1 / 2 / 4 / 8); efficiency(N) = value(N) / (N x value(1)) from the per-N records")

    quick = args.quick
    # ---- render leg (BASELINE C4): one 1920x1080 frame, image rows sharded over the ranks, 64 coarse + 64 importance samples
    # (the fine pass evaluates 128 samples/ray), no communication until the final gather of the maps to rank 0
    import math
    H, W = 1080, 1920
    focal = 0.5 * W / math.tan(0.5 * 0.6911)
    K = [[focal, 0, 0.5 * W], [0, focal, 0.5 * H], [0, 0, 1]]
    c2w = torch.eye(4)
    c2w[2, 3] = 4.0
    r0, r1 = parallel.shard_bounds(H, rank, world)
    frames = 3
    render = None
    if not quick:
        def render_frame():
            maps = model.render_image(H, W, K, c2w, chunk=131072, row_begin=r0, row_end=r1, n_importance=64)
            return parallel.gather_rows(maps["rgb"], H * W, rank, world, unit=W) if world > 1 else maps["rgb"]

        torch.cuda.empty_cache()      # the training legs leave the caching allocator fragmented: the frame's chunk buffers start from a clean pool
        render_frame()
        render_frame()
        sync_all()
        e6, e7 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e6.record()
        for _ in range(frames):
            img = render_frame()
        e7.record()
        sync_all()
        ms_render = parallel.max_over_ranks(e6.elapsed_time(e7), world, dev) / frames
        render = {"metric": "render_msamples_per_s", "value": H * W * (N_SAMPLES + N_SAMPLES + 64) / (ms_render * 1e3), "unit": "Msamples/s",
                  "frames_per_s": 1e3 / ms_render, "ms_per_frame": ms_render, "frames": frames,
                  "config": "1920x1080 frame, image rows sharded over the GPUs, 64 coarse + 64 importance samples (192 network evaluations/ray in the "
                            "reference, which is what Msamples/s counts), 131072-ray chunks, rgb gathered on rank 0; untrained (random-init) model",
                  "evaluations_per_ray": {"reference": 192, "computed": 128 if os.environ.get("NRF_RENDER_REUSE", "1") != "0" else 192,
                                          "note": "one network for both passes (src/NeRFRenderer.h:422,447): the 64 coarse samples inside the merged fine "
                                                  "pass keep the raw rows of the coarse pass; maps bit-identical to evaluating all 128 "
                                                  "(tests/test_gpu_variants.py NRF_RENDER_REUSE=0)"}}
        del img

    # ---- LeRF render leg (BASELINE C5's field, the C4 frame): RenderedLangEmbedding of one 1920x1080 frame, image rows sharded over the ranks,
    # 64 coarse + 128 importance samples (256 head evaluations per ray), no communication until the final gather of the [rows, 512] map
    render_lerf = None
    ready = False
    if not quick:
        try:
            from nerfpp_b200.lerf import LeRFField
            field = LeRFField(BBOX, seed=0)                    # same seed on every rank: identical table, primes and weights without a broadcast
            g = torch.Generator().manual_seed(0)
            for v in field.weights.values():
                v.copy_((torch.randn(v.shape, generator=g) * (2.0 / v.shape[1]) ** 0.5).to(dev))
            field.table.copy_((torch.rand(field.n_table, generator=g) * 2 - 1).to(dev))
            field.refresh()
            # warm-up on a few rows: 9 rows = two full 8192-ray chunks (the per-chunk graph is captured here, not inside the timed frame) + a ragged one
            field.render_image(H, W, K, c2w, chunk=8192, row_begin=r0, row_end=min(r0 + 9, r1))
            torch.cuda.synchronize(dev)
            ready = True
        except Exception as e:  # noqa: BLE001 - a secondary leg must not take the headline line down
            ready, render_lerf = False, {"error": f"{type(e).__name__}: {e}"}
    if not quick and parallel.all_ranks_ready(ready, world, dev):                    # else all ranks skip the leg together

        def lerf_frame():
            maps = field.render_image(H, W, K, c2w, chunk=8192, row_begin=r0, row_end=r1)
            return parallel.gather_rows(maps["rendered"], H * W, rank, world, unit=W) if world > 1 else maps["rendered"]

        lerf_frames = 2
        emb = lerf_frame()                        # untimed: allocator growth for the [rows, 512] maps
        sync_all()
        e8, e9 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e8.record()
        for _ in range(lerf_frames):
            emb = lerf_frame()
        e9.record()
        sync_all()
        ms_lerf = parallel.max_over_ranks(e8.elapsed_time(e9), world, dev) / lerf_frames
        render_lerf = {"metric": "lerf_render_rays_per_s", "value": H * W / (ms_lerf * 1e-3), "unit": "rays/s", "ms_per_frame": ms_lerf, "frames": lerf_frames,
                       "msamples_per_s": H * W * (N_SAMPLES + N_SAMPLES + N_IMPORTANCE) / (ms_lerf * 1e3),
                       "config": "1920x1080 frame of RenderedLangEmbedding [H,W,512] fp32, LeRF(32,2,256,512,128) on a 16x8 T2^19 language grid, image rows sharded "
                                 "over the GPUs, 64 coarse (density-only head) + 192 fine samples per ray, 8192-ray chunks (one captured graph per full chunk), map "
                                 "gathered on rank 0; random-init field"}
        del emb

    # ---- LeRF training leg (BASELINE C5): 1024 rays per GPU, language field trained through the fused head backward
    peaks_early = json.loads((ROOT / "MEASURED_PEAKS.json").read_text()) if (ROOT / "MEASURED_PEAKS.json").exists() else {}
    try:
        train_lerf = lerf_train_leg(rank, world, dev, model, peaks_early.get("bf16_tflops", 1590.0)) if not quick else None
    except Exception as e:  # noqa: BLE001 - after the readiness agreement a failure here is local: report it, do not hang the line
        train_lerf = {"error": f"{type(e).__name__}: {e}"}

    if rank != 0:
        return

    peaks_path = ROOT / "MEASURED_PEAKS.json"
    peaks = json.loads(peaks_path.read_text()) if peaks_path.exists() else {}
    if peaks:
        peak_gbs, peak_src = peaks["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (sustained copy)"
    else:
        peak_gbs, peak_src = 6650.0, "fallback B200_PROFILING.md"
    ms_step = ms_total / args.steps
    n_c, n_f = R * N_SAMPLES, R * (N_SAMPLES + N_IMPORTANCE)
    traffic_path = ROOT / "profiles" / "r2_ncu_traffic.json"        # dram bytes per launch out of the committed ncu --set full captures
    traffic = json.loads(traffic_path.read_text()) if traffic_path.exists() else {}

    def hbm_row(name, ms, units, bytes_per_unit, traffic_key=None, extra=None):
        by = units * bytes_per_unit
        row = {"kernel": name, "ms_per_launch": ms, "bytes_per_launch": by, "achieved": by / ms / 1e6, "frac": by / ms / 1e6 / peak_gbs,
               "share_of_step": ms / ms_step, "traffic": traffic.get(traffic_key or name)}
        if extra:
            row.update(extra)
        return row

    fwd_ms = per_launch.get("hash_encode_fwd", [0.0, 0.0])
    bwd_ms = per_launch.get("hash_encode_bwd", [0.0])
    reused = n_c if model.reuse_coarse_rows else 0
    launches_hbm = {
        "hash_encode_fwd_coarse": hbm_row("hash_fwd_kernel (coarse pass)", fwd_ms[0], n_c, BYTES_PER_POINT["hash_encode_fwd"], "hash_encode_fwd_coarse"),
        "hash_encode_fwd_fine": hbm_row("hash_fwd_kernel (fine pass)", fwd_ms[-1], n_f, BYTES_PER_POINT["hash_encode_fwd"], "hash_encode_fwd_fine",
                                        {"rows_copied_from_the_coarse_pass": reused,
                                         "achieved_counting_copied_rows_as_128B": ((n_f - reused) * BYTES_PER_POINT["hash_encode_fwd"] + reused * 129) / fwd_ms[-1] / 1e6}),
        "hash_encode_bwd": hbm_row("hash_bwd_kernel", bwd_ms[0], n_f, BYTES_PER_POINT["hash_encode_bwd"], "hash_encode_bwd"),
    }
    dom_key = max(launches_hbm, key=lambda k: launches_hbm[k]["ms_per_launch"])
    dom = launches_hbm[dom_key]
    roofline = {"bound": "hbm", "kernel": dom["kernel"], "achieved": dom["achieved"], "peak": peak_gbs, "unit": "GB/s", "frac": dom["frac"],
                "traffic": dom["traffic"], "peak_source": peak_src, "bytes_per_launch": dom["bytes_per_launch"], "ms_per_launch": dom["ms_per_launch"],
                "share_of_step": dom["share_of_step"], "launches": launches_hbm,
                "timing": "external CUDA-event pair around the launch INSIDE a second capture of the step graph, mean of 20 replays run right after the timed "
                          "regions (device time in situ: no host launch gaps, the step's own L2 state)",
                "traffic_source": "profiles/r2_ncu_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full)" if traffic else None,
                "l2_note": "the table shadow (17 MiB) is L2-resident: the kernel is bound by L1 miss sectors (forward) / L2 RED operations (backward), "
                           "not by HBM. Ceilings measured on B200 with scripts/exp/{gather,red}_bench.cu: 280 G random 4 B gathers/s, 209 G REDs/s "
                           "(any operand width) (DESIGN.md §4)"}

    # the tensor-core side of the step: fused NeRFSmall forward and backward, useful FLOPs only (18 688 FLOP/point forward over coarse +
    # fine points, 37 376 FLOP/point backward over the fine points; the backward also recomputes the forward, which is not counted)
    tf_peak = peaks.get("bf16_tflops", 1590.0)
    mf, mb = per_launch.get("mlp_small_fwd", [0.0, 0.0]), per_launch.get("mlp_small_bwd", [0.0])
    # reuse_coarse_raw: the fine forward evaluates the importance samples only (the coarse samples' raw rows are the coarse pass's own)
    n_eval = n_c + (n_f - n_c if getattr(model, "reuse_coarse_raw", False) and model.reuse_coarse_rows else n_f)
    tf_fwd = n_eval * 18688 / (sum(mf) * 1e-3) / 1e12
    tf_bwd = n_f * 37376 / (mb[0] * 1e-3) / 1e12
    roofline_tensor = {"bound": "tensor", "unit": "TFLOP/s", "peak": tf_peak,
                       "peak_source": "MEASURED_PEAKS.json bf16_tflops (cuBLAS burst)" if peaks else "fallback B200_PROFILING.md",
                       "mlp_small_fwd": {"achieved": tf_fwd, "frac": tf_fwd / tf_peak, "ms_per_step": sum(mf), "ms_per_launch": mf, "pipe": "tcgen05",
                                         "rows_evaluated_per_step": n_eval, "rows_the_reference_evaluates": n_c + n_f},
                       "mlp_small_bwd": {"achieved": tf_bwd, "frac": tf_bwd / tf_peak, "ms_per_step": mb[0], "pipe": MLP_BWD_PIPE},
                       "note": "in-graph event pairs per launch (coarse, fine); ncu per-launch figures in profiles/"}
    # TMEM -> register read rate, measured with scripts/exp/tmem_ld_bench.cu (profiles/r2_tmem_ld_bench.jsonl): 61 B/clk per WARP (a warp owns one
    # lane quarter), 228-246 B/clk/SM with 4 warps, 440-457 with 8, 470-487 with 16.  Round 1 read B300_MICROARCH's "64 B/clk" as a per-SM figure and
    # called this kernel TMEM-read-bound; it has 16 epilogue warps, so its read floor is 8x lower than its time: the kernel is bound by the latency of
    # five dependent MMA -> tcgen05.ld -> convert -> tcgen05.st round trips per tile (4 tile pipelines per SM share the 512 columns), not by bandwidth
    sm_mhz = peaks.get("sm_max_mhz", 1965.0)
    tmem_floor_ms = n_eval * 224 * 4 / (148 * 480 * sm_mhz * 1e6) * 1e3
    roofline_tensor["mlp_small_fwd"]["tmem_read"] = {"bytes_per_point": 896, "measured_peak": "480 B/clk/SM with 16 reading warps (61 B/clk per warp)",
                                                      "floor_ms_per_step": tmem_floor_ms, "frac": tmem_floor_ms / max(sum(mf), 1e-9),
                                                      "source": "profiles/r2_tmem_ld_bench.jsonl"}

    roofline_render_ops = None
    if not quick:
        roofline_tensor["mlp_nerf"] = classic_nerf_leg(tf_peak)
        try:
            roofline_tensor["lerf_head"] = lerf_leg(tf_peak)
        except Exception as e:  # noqa: BLE001 - a secondary leg must not take the headline line down
            roofline_tensor["lerf_head"] = {"error": f"{type(e).__name__}: {e}"}
        roofline_render_ops = render_ops_leg(roofline["peak"])

    shipped_shape = None
    if world == 1 and not quick:
        try:
            shipped_shape = shipped_shape_leg(dev, R)
        except Exception as e:  # noqa: BLE001 - a secondary leg must not take the headline line down
            shipped_shape = {"error": f"{type(e).__name__}: {e}"}
    as_shipped = None
    if world == 1 and not quick:
        try:
            as_shipped = shipped_leg(dev, R)
        except Exception as e:  # noqa: BLE001
            as_shipped = {"error": f"{type(e).__name__}: {e}"}

    # ---- the same step through the C++ surfaces, on this GPU (N = 1 only): the reference's own CUDA path and the C++ drop-in classes
    dropin_cpp = reference_cuda = None
    if world == 1 and not quick:
        for which in ("reference_cuda", "dropin_cpp"):
            try:
                leg = gpu_loop_leg(which, R, 30)
            except Exception as e:  # noqa: BLE001
                leg = {"error": f"{type(e).__name__}: {e}"}
            if which == "reference_cuda":
                reference_cuda = leg
            else:
                dropin_cpp = leg
        if reference_cuda and dropin_cpp and "value" in reference_cuda and "value" in dropin_cpp:
            dropin_cpp["vs_reference_cuda"] = dropin_cpp["value"] / reference_cuda["value"]
            reference_cuda["ours_vs_reference_cuda"] = (R * args.steps / (ms_total / 1e3)) / reference_cuda["value"]

    # ---- BASELINE C4 through the same C++ surfaces (N = 1 only)
    render_cpp = None
    if world == 1 and not quick:
        render_cpp = {}
        for which in ("dropin_cpp", "dropin_cpp_staged", "reference_cuda"):
            try:
                render_cpp[which] = cpp_render_leg(which)
            except Exception as e:  # noqa: BLE001
                render_cpp[which] = {"error": f"{type(e).__name__}: {e}"}
            torch.cuda.empty_cache()

    cpu_baseline = None
    if world == 1 and not args.no_cpu_baseline:
        try:
            v, sps, threads = reference_cpu_rays_per_s(steps=CPU_STEPS, warmup=CPU_WARMUP)
            cpu_baseline = {"value": v, "unit": "rays/s", "cores": threads, "kind": "reference",
                            "sample": f"{CPU_SAMPLE_RAYS}-ray sample of the {RAYS_PER_GPU}-ray step, {CPU_STEPS} steps after {CPU_WARMUP} warm-up ({sps:.2f} s/step)"}
        except ImportError as e:
            cpu_baseline = {"value": None, "unit": "rays/s", "cores": 0, "kind": "reference", "sample": f"oracle/_ref not importable: {e}"}

    rays_total = R * world * args.steps
    print(json.dumps({
        "metric": "train_rays_per_s", "value": rays_total / (ms_total / 1e3), "unit": "rays/s", "n_gpus": world, "steps": args.steps,
        "warmup": warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "C2/C3 HashNeRF training: L16 F2 T2^19 hash grid 16->512 + SH deg 4 + NeRFSmall 32->64->16 | 31->64->64->3, "
                               f"{R} rays/GPU/step of an 800x800 view, 64 coarse + 128 importance samples, huber + Adam(0.9,0.99,1e-15)",
                   "rays_per_gpu": R, "global_rays": R * world, "parallelism": f"ray-sharded dp{world}: {dp_mode}",
                   "l2": "not flushed explicitly: each step streams ~300 MB (Adam pass over 8.9M params + moments + gradient) through the 126 MB L2",
                   "precision": "fp16 hash table reads / encodings, bf16 tensor-core MLP with fp32 accumulate, fp32 everything else",
                   "feed": "a step consumes the int32 [R,2] pixel list sampled for it (src/NeRFDataset.cpp:154-155); rays (GetRayBatch) and targets (the image "
                           "gather) are formed by the step's first kernel from the resident 800x800 view.  value: lists resident in HBM (one 32 KB D2D copy "
                           "into the graph's static input per step); e2e: the same lists in pinned host memory + a loss read per step",
                   "reuse_coarse_rows": bool(model.reuse_coarse_rows),
                   "reuse_coarse_raw": bool(getattr(model, "reuse_coarse_raw", False)),
                   "reuse_note": "the merged fine pass holds the 64 coarse samples bit for bit and the reference uses ONE network for both passes "
                                 "(src/NeRFRenderer.h:422,447): their encoding rows are copied and their raw rows taken from the coarse pass, the fine "
                                 "forward gathers / evaluates the 128 importance samples only; outputs and gradients are bit-identical to evaluating all "
                                 "192 (tests/test_gpu_pipeline.py::test_coarse_reuse_leaves_the_render_unchanged); the backward covers all 192"},
        "e2e": {"value": rays_total / (ms_e2e / 1e3), "unit": "rays/s", "h2d_bytes_per_step": head["h2d"], "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps,
                "input": "pinned-host int32 [R,2] pixel coordinates of the step's batch; rays (GetRayBatch) and targets (image gather) are formed on the "
                         "device by the step's first kernel from the resident 800x800 training view",
                "note": "same captured step as `value`, run right after it on the same model (K more optimisation steps): the hash gathers / scatter are "
                        "data dependent — as the density concentrates, importance samples cluster and share cells (kernels_ms_per_step is taken after "
                        "both regions) — so e2e can come out faster than value although it adds the H2D copy and the loss read"},
        "gpu_launches": launches * world, "graph_replay": use_graph, "kernels_per_step": launches_per_step, "roofline": roofline,
        "roofline_tensor": roofline_tensor, "roofline_render_ops": roofline_render_ops, "cpu_baseline": cpu_baseline, "clocks": clocks,
        "kernels_ms_per_step": {k: [round(t, 4) for t in v] for k, v in sorted(per_launch.items(), key=lambda kv: -sum(kv[1]))},
        "kernels_ms_per_step_sum": round(sum(sum(v) for v in per_launch.values()), 4),
        "dp_check": dp_check, "flags_timeout_after_timed_regions": timeout_after, "strong": strong,
        "reference_cuda": reference_cuda, "dropin_cpp": dropin_cpp, "train_as_shipped": as_shipped, "train_shipped_shape": shipped_shape, "render_cpp": render_cpp,
        "final_loss": {"resident": head["loss"], "e2e": head["loss_e2e"]}, "render": render, "render_lerf": render_lerf, "train_lerf": train_lerf,
    }))


if __name__ == "__main__":
    main()
