"""Training step in the reference's shipped configuration (src/main.cpp:187 thin_ray = false; raw noise and stochastic preconditioning on,
src/NeRFExecutor.h:411-412), three implementations timed in ONE process with CUDA events, alternating arm by arm over several rounds:

  cpp_autograd   the C++ drop-in's autograd loop (renderer.h: Render -> huber -> backward -> FusedAdam), train_steps_shipped without the graph
  cpp_graph      HashNeRFTrainGraph (host/train_graph.h) through train_steps_shipped: jitter inside the hash kernels, one graph replay per step
  py_mirror      the Python mirror's forward_backward_shipped + scheduled Adam captured as one CUDA graph (bench.py's train_as_shipped leg)

Every arm reads the loss on the host after each step (loss.item(), as the reference's loop does).  Shapes:
  baseline  SH degree 4, finest 512, 64 + 128 samples, 4096 rays (one chunk)
  shipped   SH degree 8, finest 1024, 64 + 192 samples, 16384 rays in 4096-ray chunks (the mirror has no chunks: one 16384-ray pass)

    python scripts/exp/shipped_train_graph.py --out shipped_train_graph.jsonl
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))

BBOX = (-1.5, -1.5, -1.5, 1.5, 1.5, 1.5)
SHAPES = {
    # name: (finest resolution, SH degree, n_samples, n_importance, rays, chunk)
    "baseline": (512, 4, 64, 128, 4096, 4096),
    "shipped": (1024, 8, 64, 192, 16384, 4096),
}
CONE = (1.0 / 1111.1 + 1.0 / 1111.1) / 2.0          # bench.py shipped_leg's values: mid-schedule amplitudes
NOISE_STD = 0.5
ALPHA = 0.01 * (3 * 3.0 ** 2) ** 0.5


def device_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines()[0].split(", ") + ["?"])[:2] if q.returncode == 0 and q.stdout.strip() else (torch.cuda.get_device_name(), "?")
    return {"device": name, "power_limit": power}


def make_arms(shape: str):
    from nerfpp_b200 import build
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    sys.path.insert(0, str(build.build_host().parent))
    import nerfpp_b200_torch as H
    finest, deg, S, N, rays, chunk = SHAPES[shape]
    o, d, tgt = synthetic_rays(rays, seed=31)
    cone = torch.tensor(CONE, device="cuda")
    arms = {}
    for name, graph in (("cpp_autograd", False), ("cpp_graph", True)):
        H.manual_seed(42)
        p = H.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, 19, 16, finest, deg, 2, 64, 15, 3, 64)
        p.init_model()
        p.use_fused_adam(True)
        p.use_train_graph(graph)

        def run(k, p=p):
            return p.train_steps_shipped(o, d, tgt, cone, k, S, N, chunk, 1e-2, 250, [NOISE_STD] * k, [ALPHA] * k)[1][-1]
        arms[name] = run
    m = HashNeRF(BBOX, finest_resolution=finest, sh_degree=deg, n_samples=S, n_importance=N, seed=42)
    m._init_sched()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        m.forward_backward_shipped(o, d, tgt, CONE, NOISE_STD, ALPHA)
        m.grads.zero_()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        m.forward_backward_shipped(o, d, tgt, CONE, NOISE_STD, ALPHA)
        m._optimizer_step_scheduled(1.0)

    def run_mirror(k):
        lv = None
        for _ in range(k):
            g.replay()
            lv = float(m.loss)
        return lv
    arms["py_mirror"] = run_mirror
    return arms


def timed(fn, k: int) -> tuple[float, float]:
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    loss = fn(k)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / k, loss


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default="baseline,shipped")
    ap.add_argument("--steps", type=int, default=20, help="steps per timed block")
    ap.add_argument("--rounds", type=int, default=5, help="alternating rounds (each arm timed once per round)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this measurement needs a CUDA device"
    info = device_info()
    lines = []
    for shape in args.shapes.split(","):
        arms = make_arms(shape)
        for fn in arms.values():
            fn(args.warmup)
        per = {k: [] for k in arms}
        last = {}
        for _ in range(args.rounds):
            for name, fn in arms.items():
                ms, loss = timed(fn, args.steps)
                per[name].append(ms)
                last[name] = loss
        finest, deg, S, N, rays, chunk = SHAPES[shape]
        for name, v in per.items():
            v = sorted(v)
            line = {"shape": shape, "arm": name, "ms_per_step_median": v[len(v) // 2], "ms_per_step_min": v[0], "ms_per_step_max": v[-1],
                    "rays": rays, "chunk": chunk, "sh_degree": deg, "finest": finest, "samples": f"{S}+{N}", "steps_per_block": args.steps,
                    "rounds": args.rounds, "last_loss": last[name], **info}
            lines.append(line)
            print(json.dumps(line), flush=True)
        del arms
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(x) + "\n" for x in lines))


if __name__ == "__main__":
    main()
