"""Multi-GPU plumbing: one process per GPU, torch.distributed (NCCL over NVLink on the box, gloo in CPU tests).

The reference has no multi-GPU code at all (SURVEY §2, §5); this is the sharding the hot path admits:
  * training  — rays are independent, so the global ray batch is split contiguously by rank, every rank runs
    forward/backward on its shard, and the ONE exchange step is an all-reduce(sum) of the flat gradient vector
    [reachable hash-table scalars | NeRFSmall weights] (34 MiB + 37 KiB fp32 at the BASELINE shape), scaled by 1/world
    inside the Adam kernel (the loss is a mean over rays, src/NeRFExecutor.h:883-886).  Replicas stay identical
    because they start identical (same seed) and apply the same reduced gradient.
  * rendering — image rows are split into contiguous tiles, no communication until a final gather of the maps.
"""
from __future__ import annotations

import os

import sys

import torch
import torch.distributed as dist


def init_from_env(backend: str | None = None) -> tuple[int, int, int]:
    """(rank, world, local_rank) from the torchrun environment; initialises the default process group if world > 1."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            dist.init_process_group(backend, device_id=torch.device("cuda", local_rank))
        else:
            dist.init_process_group(backend)
    return rank, world, local_rank


def shard_bounds(n: int, rank: int, world: int) -> tuple[int, int]:
    """Contiguous, balanced partition of n units (rays or image rows): the first n % world ranks get one extra."""
    base, extra = divmod(n, world)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def allreduce_gradients(flat_grad: torch.Tensor, world: int) -> float:
    """Sum the flat gradient over ranks in place; returns the scale (1/world) the optimiser must apply."""
    if world > 1:
        dist.all_reduce(flat_grad, op=dist.ReduceOp.SUM)
    return 1.0 / world


def broadcast_parameters(flat_params: torch.Tensor, world: int, src: int = 0) -> None:
    """Rank 0's table / primes / weights become everyone's (the reference draws them at random, SURVEY §8e)."""
    if world > 1:
        dist.broadcast(flat_params, src=src)


def gather_rows(local: torch.Tensor, n_total: int, rank: int, world: int, dst: int = 0, unit: int = 1) -> torch.Tensor | None:
    """Final gather of a row-sharded map ([rows_local, ...]) onto `dst`; shards follow shard_bounds over n_total // unit
    units of `unit` tensor rows each (unit = image width when image rows are the sharded unit)."""
    if world == 1:
        return local
    shapes = [tuple(unit * v for v in shard_bounds(n_total // unit, r, world)) for r in range(world)]
    # equal-size exchange (gloo's gather refuses ragged shards; shard sizes differ by at most one unit): pad to the largest shard, trim on dst
    biggest = max(e - b for b, e in shapes)
    local = local.contiguous()
    if local.shape[0] < biggest:
        local = torch.cat([local, local.new_zeros((biggest - local.shape[0],) + tuple(local.shape[1:]))], 0)
    if rank == dst:
        parts = [torch.empty_like(local) for _ in shapes]
        dist.gather(local, parts, dst=dst)
        return torch.cat([p[:e - b] for p, (b, e) in zip(parts, shapes)], 0)
    dist.gather(local, None, dst=dst)
    return None


def max_over_ranks(value: float, world: int, device) -> float:
    if world == 1:
        return value
    t = torch.tensor([value], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_ranks_ready(ok: bool, world: int, device) -> bool:
    """True only if EVERY rank passed ok = True (min over ranks).  Called before the first collective of an optional leg, so that a rank
    whose set-up failed makes all ranks skip it together instead of leaving the others waiting in a gather."""
    return -max_over_ranks(-(1.0 if ok else 0.0), world, device) > 0.5


class PeerShardedOptimizer:
    """Plumbing for nrf_adam_step_sharded: allocates the model's flat gradient, its fp16 shadow and a flag block in
    torch.distributed symmetric memory (peer-mapped over NVLink), exchanges the peer addresses, and re-points the model at
    those buffers.  After this, one kernel per rank performs reduce-scatter(grad) + Adam(owned shard) + all-gather(fp16 shadow);
    NCCL is not on the training path any more (it still does the one-off parameter broadcast and the final render gather)."""

    def __init__(self, model, rank: int, world: int, group=None):
        import torch.distributed._symmetric_memory as symm
        from . import cabi
        group = group or dist.group.WORLD
        dev = model.device
        n = model.params.numel()
        try:                                   # older torch releases need the group enabled explicitly
            symm.enable_symm_mem_for_group(group.group_name)
        except Exception:                      # noqa: BLE001
            pass
        self.grads = symm.empty(n, dtype=torch.float32, device=dev)
        self.shadow = symm.empty(n, dtype=torch.float16, device=dev)
        n_flags = max(int(cabi.lib().nrf_peer_flags_bytes(world)) // 4, 64)
        self.flags = symm.empty(n_flags, dtype=torch.int32, device=dev)
        self.grads.zero_()
        self.flags.zero_()
        self.shadow.copy_(model.shadow)
        handles = [symm.rendezvous(t, group.group_name) for t in (self.grads, self.shadow, self.flags)]
        pg = cabi.PeerGroup()
        pg.world, pg.rank = world, rank
        for field, h, t in zip(("grads", "shadow_f16", "flags"), handles, (self.grads, self.shadow, self.flags)):
            ptrs = list(h.buffer_ptrs)
            off = t.data_ptr() - ptrs[rank]    # offset of the tensor inside this rank's symmetric block (same on every rank)
            assert 0 <= off < (1 << 40), "symmetric-memory tensor is not inside its own block"
            for p in range(world):
                getattr(pg, field)[p] = ptrs[p] + off
        self.pg, self.handles, self.rank, self.world = pg, handles, rank, world
        # NVSwitch multicast mappings of the gradient and the shadow (multimem.ld_reduce / multimem.st): the reduction happens in the switch.
        # NRF_DP_MULTICAST=0 keeps the peer-load kernel, =1 forces multicast (A/B).  Default: multicast from 4 ranks up — with two ranks every
        # byte crosses the link once either way and multimem only adds latency (0.887 vs 0.862 ms per step at N = 2; 0.882 vs 0.901 ms at N = 8:
        # profiles/r2_bench_{2,8}gpu_{multicast,peerloads}.json).
        self.multicast = False
        want = os.environ.get("NRF_DP_MULTICAST", "auto")
        if bool(getattr(handles[0], "has_multicast_support", False)) and (want == "1" or (want != "0" and self.world >= 4)):
            mc = [int(getattr(h, "multicast_ptr", 0) or 0) for h in handles[:2]]
            if all(mc):
                pg.grads_mc = mc[0] + (self.grads.data_ptr() - list(handles[0].buffer_ptrs)[rank])
                pg.shadow_f16_mc = mc[1] + (self.shadow.data_ptr() - list(handles[1].buffer_ptrs)[rank])
                self.multicast = True
        self.n_table = model.n_table
        model.grads, model.shadow = self.grads, self.shadow
        model.peer = self
        if hasattr(model, "bind_peer_buffers"):
            model.bind_peer_buffers()          # views into the flat gradient follow it into symmetric memory
        self._flag_host = None
        torch.cuda.synchronize(dev)
        dist.barrier(group)

    def dp_check(self, model, seed: int = 1234) -> dict:
        """ONE optimiser step on a random per-rank gradient through BOTH data-parallel paths, on the model's own buffers, then everything
        is put back: (A) NCCL all-reduce(sum) + dense Adam on clones (parallel.allreduce_gradients + nrf_adam_step), (B) the fused
        peer-memory kernel.  Collective; call before training starts (model.step == 0).  Returns
          max_abs_shadow_diff               max |shadow_B - shadow_A| over the whole flat vector, max over ranks (A and B differ only in the
                                            order of the cross-rank sum: NCCL's ring vs fixed rank order), and the number of entries where
                                            it exceeds 5 % of lr (a summed gradient within rounding of zero flips the sign of the step)
          shadows_bit_identical_across_ranks   every rank holds rank 0's fp16 shadow bit for bit after (B)
          owner_master_matches_shadow       on every rank the owned fp32 shard rounds to the shadow it published
          flags_timeout                     max over ranks of the sticky barrier-timeout marker
        The first Adam step moves every parameter by ~lr * sign(g), so a wrong reduction (a missing rank, a wrong shard) shows up at
        the 1e-2 level against lr-sized differences of 0 for a correct one."""
        from . import ops
        dev, world, rank = model.device, self.world, self.rank
        assert model.step == 0, "dp_check must run before the first step"
        saved = {k: getattr(model, k).clone() for k in ("params", "exp_avg", "exp_avg_sq", "shadow")}
        g = torch.Generator(device=dev).manual_seed(seed + rank)
        grad = torch.randn(model.params.numel(), generator=g, device=dev, dtype=torch.float32) * 1e-3
        # (A) reference path on clones
        g_sum = grad.clone()
        dist.all_reduce(g_sum, op=dist.ReduceOp.SUM)
        pa, ma, va = saved["params"].clone(), saved["exp_avg"].clone(), saved["exp_avg_sq"].clone()
        shadow_a = torch.empty_like(saved["shadow"])
        ops.adam_step(pa, g_sum, ma, va, model.lr0, 1, 0.9, 0.99, 1e-15, 1.0 / world, True, shadow_a)
        # (B) fused path on the live buffers
        model.grads.copy_(grad)
        torch.cuda.synchronize(dev)
        dist.barrier()
        model.optimizer_step_sharded()
        torch.cuda.synchronize(dev)
        dist.barrier()
        d = (model.shadow.float() - shadow_a.float()).abs()
        diff = d.max()
        n_diff = (d > 0.05 * model.lr0).sum()          # sign flips of a ~zero summed gradient (the step is ~lr * sign(g)): expect 0, allow a handful
        ref = model.shadow.clone()
        dist.broadcast(ref, src=0)
        same = torch.equal(ref, model.shadow)
        lo, hi = self.owned_range()
        owner_ok = torch.equal(model.params[lo:hi].half(), model.shadow[lo:hi])
        master_diff = (model.params[lo:hi] - pa[lo:hi]).abs().max() if hi > lo else torch.zeros((), device=dev)
        cleared = float(model.grads.abs().max()) == 0.0
        stats = torch.tensor([float(diff), float(master_diff), float(not same), float(not owner_ok), float(not cleared), float(self.timeout()), float(n_diff)],
                             dtype=torch.float64, device=dev)
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        # put everything back (every rank restores its own buffers; the peers' writes into this rank's shadow are overwritten)
        dist.barrier()
        for k, v in saved.items():
            getattr(model, k).copy_(v)
        model.grads.zero_()
        model.step = 0
        model._sched_step = -1          # the check advanced the device-side counter: re-seed it on the next step
        model.repack()
        torch.cuda.synchronize(dev)
        dist.barrier()
        out = {"max_abs_shadow_diff": stats[0].item(), "max_abs_owned_master_diff": stats[1].item(),
               "shadows_bit_identical_across_ranks": stats[2].item() == 0.0, "owner_master_matches_shadow": stats[3].item() == 0.0,
               "gradient_cleared": stats[4].item() == 0.0, "flags_timeout": int(stats[5].item()), "entries_differing_by_more_than_5pct_of_lr": int(stats[6].item()),
               "entries": int(model.params.numel()), "lr": model.lr0,
               "multicast": bool(self.multicast),
               "what": "one step on a random per-rank gradient: fused peer-memory kernel vs NCCL all-reduce + dense Adam"}
        out["ok"] = bool(out["shadows_bit_identical_across_ranks"] and out["owner_master_matches_shadow"] and out["gradient_cleared"]
                         and out["flags_timeout"] == 0 and out["entries_differing_by_more_than_5pct_of_lr"] <= 8)
        return out

    def timeout(self) -> int:
        """The sticky barrier-timeout marker of this rank's flag block (synchronises the device)."""
        return int(self.flags[2 * self.world + 2])

    def check(self) -> None:
        """Raises if a peer barrier of the fused optimiser ever gave up waiting.  Reads a pinned-host mirror of the marker that
        `mirror_flag` refreshes asynchronously after every step: no device synchronisation, at most a few steps late."""
        if self._flag_host is not None and int(self._flag_host[0]) != 0:
            raise RuntimeError(f"nerfpp_b200: rank {self.rank}: a peer barrier of the fused data-parallel optimiser timed out — a rank missed a "
                               "step; parameters were left untouched from that step on (nrf_adam_step_sharded)")

    def mirror_flag(self) -> None:
        if self._flag_host is None:
            self._flag_host = torch.zeros(1, dtype=torch.int32).pin_memory()
        self._flag_host.copy_(self.flags[2 * self.world + 2: 2 * self.world + 3], non_blocking=True)

    def allgather_master(self, model) -> None:
        """Re-assemble the fp32 master and the Adam moments on every rank: under the fused optimiser a rank only updates the shard it
        owns (the forward reads the fp16 shadow), so before a checkpoint (the reference's embedder_checkpoint.pt,
        src/NeRFExecutor.h:1055-1069), HashNeRF.refresh() or a switch back to the NCCL path the owners publish their shards.
        Collective (one broadcast per rank and buffer: 3 x 35 MB in total, off the hot path)."""
        torch.cuda.synchronize(model.device)
        for r in range(self.world):
            lo, hi = self.owned_range(r)
            for buf in (model.params, model.exp_avg, model.exp_avg_sq):
                dist.broadcast(buf[lo:hi], src=r)
        model.masters_synced = True

    def owned_range(self, rank: int | None = None) -> tuple[int, int]:
        """[begin, end) scalars of the table that `rank` (default: this rank) owns: the kernel's own split (quads, the first ranks take one
        extra); the scalars past the last whole quad belong to the replicated tail."""
        b, e = shard_bounds(self.n_table // 4, self.rank if rank is None else rank, self.world)
        return 4 * b, 4 * e
