"""Worker for tests/test_gpu_multi.py (one process per GPU, launched by torch.distributed.run).
Checks (1) that an N-rank step produces the 1-GPU gradient of the same global batch (SURVEY App. B, "DP training" row), (2) the fused
data-parallel optimiser (nrf_adam_step_sharded over NVLink peer memory) against the NCCL all-reduce + dense-Adam path — on a random
gradient (dp_check) and over a training trajectory, eager and graph-replayed —, (3) the fp32 master gather for checkpoints, and (4) the
row-sharded render gather."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nerfpp_b200 import parallel  # noqa: E402
from nerfpp_b200.pipeline import HashNeRF, synthetic_rays  # noqa: E402

BBOX = (-1.5, -1.5, -1.5, 1.5, 1.5, 1.5)


def main():
    rank, world, local = parallel.init_from_env("nccl")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    R = 512

    # ---- (1) gradients of an N-rank step == gradients of the 1-GPU step on the same global batch, up to reduction order
    g_model = HashNeRF(BBOX, log2_hashmap_size=15, seed=5, device=dev)
    parallel.broadcast_parameters(g_model.params, world); g_model.refresh()
    go, gd, gt = synthetic_rays(R * world, device=dev, seed=77)              # the same global batch on every rank
    b, e = parallel.shard_bounds(R * world, rank, world)
    g_model.grads.zero_()
    g_model.forward_backward(go[b:e].contiguous(), gd[b:e].contiguous(), gt[b:e].contiguous(), grad_scale=1.0 / world)   # loss = mean over the GLOBAL batch
    sharded = g_model.grads.clone()
    dist.all_reduce(sharded, op=dist.ReduceOp.SUM)
    g_model.grads.zero_()
    g_model.forward_backward(go, gd, gt)
    whole = g_model.grads.clone()
    g_model.grads.zero_()
    rel = float((sharded.double() - whole.double()).norm() / whole.double().norm())
    rel_mlp = float((sharded[g_model.n_table:].double() - whole[g_model.n_table:].double()).norm() / whole[g_model.n_table:].double().norm())
    assert float(whole.abs().max()) > 0
    assert rel <= 1e-5 and rel_mlp <= 1e-5, ("DP gradient differs from the 1-GPU gradient", rel, rel_mlp)

    batches = [synthetic_rays(R, device=dev, seed=100 * rank + i) for i in range(3)]
    # A: NCCL all-reduce + dense Adam on every rank (eager)
    a = HashNeRF(BBOX, log2_hashmap_size=15, seed=3, device=dev, lrate_decay=1)
    parallel.broadcast_parameters(a.params, world); a.refresh()
    # B: fused peer-memory optimiser (eager), C: the same inside the captured graph
    b_ = HashNeRF(BBOX, log2_hashmap_size=15, seed=3, device=dev, lrate_decay=1)
    parallel.broadcast_parameters(b_.params, world); b_.refresh()
    os.environ["NRF_DP_MULTICAST"] = "1"          # forced: the default picks multicast from 4 ranks up, and both forms of the kernel are checked here
    parallel.PeerShardedOptimizer(b_, rank, world)
    os.environ.pop("NRF_DP_MULTICAST")
    c = HashNeRF(BBOX, log2_hashmap_size=15, seed=3, device=dev, lrate_decay=1)
    parallel.broadcast_parameters(c.params, world); c.refresh()
    # ---- (2a) one step on a random gradient through both paths; everything is restored afterwards.  b_ uses the NVSwitch multicast mappings when
    # the box has them (multimem.ld_reduce / multimem.st), c the plain peer loads / stores: both forms of the kernel are checked
    os.environ["NRF_DP_MULTICAST"] = "0"
    before = c.params.clone()
    peer_c = parallel.PeerShardedOptimizer(c, rank, world)
    os.environ.pop("NRF_DP_MULTICAST")
    assert not peer_c.multicast
    chk = peer_c.dp_check(c)
    assert chk["ok"], chk
    assert c.step == 0 and torch.equal(before, c.params) and float(c.grads.abs().max()) == 0.0
    c.capture_train_step(R, world)

    la, lb, lc = [], [], []
    for i in range(6):
        batch = batches[i % 3]
        a.forward_backward(*batch)
        a.optimizer_step(grad_scale=parallel.allreduce_gradients(a.grads, world))
        la.append(float(a.loss))
        b_.forward_backward(*batch)
        b_.optimizer_step_sharded()
        lb.append(float(b_.loss))
        lc.append(float(c.train_step_graph(*batch)))
    torch.cuda.synchronize()
    for name, m, losses in (("eager", b_, lb), ("graph", c, lc)):
        assert int(m.flags_timeout()) == 0, f"{name}: peer barrier timed out"
        m.peer.check()
        # every rank holds the SAME fp16 shadow, bit for bit
        ref = m.shadow.clone()
        dist.broadcast(ref, src=0)
        assert torch.equal(ref, m.shadow), f"{name}: shadows differ between ranks"
        # the owner's fp32 master agrees with the shadow it published; the MLP tail is replicated
        lo, hi = m.peer.owned_range()
        assert torch.equal(m.params[lo:hi].half(), m.shadow[lo:hi]), f"{name}: owner shard / shadow mismatch"
        assert torch.equal(m.params[m.n_table:].half(), m.shadow[m.n_table:])
        tail = m.params[m.n_table:].clone()
        dist.broadcast(tail, src=0)
        assert torch.equal(tail, m.params[m.n_table:]), f"{name}: MLP replicas differ"
        assert float(m.grads.abs().max()) == 0.0, f"{name}: gradient not cleared"
        # against the NCCL path: same training trajectory (Adam is sign-like, so compare the bulk, see test_gpu_pipeline)
        for x, y in zip(losses, la):
            assert abs(x - y) <= 5e-3 * abs(y) + 1e-6, (name, losses, la)
        d = (a.shadow.float() - m.shadow.float()).abs()
        frac = (d > 1e-4).float().mean().item()
        assert frac < 3e-2 and d.median().item() < 1e-6, (name, frac)
        assert m.step == 6 and int(m.sched[0]) == 6

        # ---- (3) the fp32 master is sharded: refresh / table refuse to run on stale shards, allgather_master re-assembles them
        assert not m.masters_synced
        try:
            m.refresh()
            raise AssertionError("refresh() must refuse stale fp32 shards")
        except RuntimeError:
            pass
        sd = m.state_dict()                       # gathers (collective)
        assert m.masters_synced
        assert torch.equal(sd["params"][:m.n_table].half(), m.shadow[:m.n_table]), f"{name}: gathered master != shadow"
        full = sd["params"].clone()
        dist.broadcast(full, src=0)
        assert torch.equal(full, sd["params"]), f"{name}: gathered masters differ between ranks"
        for k in ("exp_avg", "exp_avg_sq"):
            t = sd[k].clone()
            dist.broadcast(t, src=0)
            assert torch.equal(t, sd[k]), f"{name}: gathered {k} differs between ranks"
        d_master = (a.params - sd["params"]).abs()
        assert (d_master > 1e-4).float().mean().item() < 3e-2 and d_master.median().item() < 1e-6
        shadow_before = m.shadow.clone()
        m.refresh()                               # now allowed, and a no-op on the shadow
        assert torch.equal(shadow_before, m.shadow)

    # row-sharded render + final gather
    H, W = 24, 32
    K = [[40.0, 0, 16.0], [0, 40.0, 12.0], [0, 0, 1]]
    c2w = torch.eye(4); c2w[2, 3] = 4.0
    r0, r1 = parallel.shard_bounds(H, rank, world)
    part = c.render_image(H, W, K, c2w, row_begin=r0, row_end=r1)["rgb"]
    full = parallel.gather_rows(part, H * W, rank, world, unit=W)
    if rank == 0:
        whole = c.render_image(H, W, K, c2w)["rgb"]
        assert torch.equal(full, whole)
        print("MULTI_GPU_WORKER_OK", world, la[-1], lb[-1], lc[-1], "dp_grad_rel", rel, rel_mlp, "multicast(b)", b_.peer.multicast, "dp_check", chk)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
