"""CPU tests of the host-side logic: grid buffers, sharding, and the N>1 exchange path on gloo (world_size 2)."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from nerfpp_b200 import parallel, pipeline


def test_grid_buffers_mirror_reference_constructor():
    g = pipeline.make_grid((-1.5,) * 3 + (1.5,) * 3, device="cpu", seed=7)
    assert g.primes.shape == (16, 1, 3) and g.primes.dtype == torch.int32
    p = g.primes.reshape(-1).tolist()
    assert all((1 << 28) <= v < (1 << 30) and pipeline._is_prime(v) for v in p)       # src/CuHashEmbedder.cpp:37-47
    assert g.feat_local_size.tolist() == [1 << 19] * 16                                # (2^19 >> 4) << 4
    assert g.feat_local_idx.tolist() == [i << 19 for i in range(16)]                   # cumsum - size: SCALAR offsets
    assert g.table_scalars() == 16 * (1 << 19) * 2
    assert g.used_scalars() == 17 * (1 << 19)                                          # levels overlap by half (F = 2)
    g8 = pipeline.make_grid((-1,) * 3 + (1,) * 3, 16, 8, 19, 16, 512, device="cpu")    # LeRF grid, F = 8
    assert g8.used_scalars() == (15 + 8) * (1 << 19)


def test_lerf_parameter_names_and_shapes_are_the_reference_modules(golden):
    """The Python mirror's parameter table (nerfpp_b200/lerf.py, ops.lerf_pack) against the names the reference's LeRF registers
    (fixture tests/golden/lerf.npz, written from oracle/_ref: src/LeRF.cpp:17-25) and the shapes of its weights."""
    from nerfpp_b200 import lerf, ops
    g = golden("lerf.npz")
    names = [f"lang_model_{n}.weight" for n, _, _ in lerf.LERF_LAYERS]
    assert names == list(g["names"]) == [f"lang_model_{n}.weight" for n in ops.LERF_WEIGHT_NAMES]
    assert [(o, i) for _, o, i in lerf.LERF_LAYERS] == [tuple(g[k].shape) for k in ("sw0", "sw1", "lw0", "lw1")]
    s = ops.lerf_shape()
    assert (s.geo_feat_dim, s.num_layers, s.hidden_dim, s.lang_embed_dim, s.input_ch) == (32, 2, 256, 512, 128)      # src/main.cpp:203-213, C5: D = 512


def test_shard_bounds_partition():
    for n, world in ((4096, 8), (1080, 8), (7, 3), (5, 8), (32768, 4)):
        spans = [parallel.shard_bounds(n, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == n
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        sizes = [e - b for b, e in spans]
        assert max(sizes) - min(sizes) <= 1


def test_owned_range_of_the_fused_optimiser_partitions_the_table():
    """PeerShardedOptimizer.owned_range mirrors the kernel's split (csrc/optim_sharded.cu: quads, the first ranks take one extra): the owners'
    slices tile the table's whole quads exactly."""
    n_table = 8912896 + 3                                   # not a multiple of 4: the leftover scalars belong to the replicated tail
    q4 = n_table // 4 * 4
    for world in (1, 2, 3, 4, 8):
        spans = []
        for rank in range(world):
            opt = object.__new__(parallel.PeerShardedOptimizer)
            opt.rank, opt.world, opt.n_table = rank, world, n_table
            spans.append(opt.owned_range())
            assert spans[-1] == opt.owned_range(rank)
        assert spans[0][0] == 0 and spans[-1][1] == q4
        assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
        assert all(b % 4 == 0 and e % 4 == 0 for b, e in spans)
        base, extra = divmod(q4 // 4, world)
        assert [(e - b) // 4 for b, e in spans] == [base + (1 if r < extra else 0) for r in range(world)]   # the kernel's formula


def test_lr_schedule_matches_reference_order():
    """src/NeRFExecutor.h:986-996: step() uses the rate set after the previous step, global_step counted from 0."""
    lr0, decay = 1e-2, 250
    ref, cur, g = [], lr0, 0
    for _ in range(5):
        ref.append(cur)
        cur = lr0 * 0.1 ** (g / (decay * 1000))
        g += 1
    ours = [lr0 * (0.1 ** (max(s - 2, 0) / (decay * 1000))) for s in range(1, 6)]
    np.testing.assert_allclose(ours, ref, rtol=1e-12)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    r, w, _ = parallel.init_from_env("gloo")
    torch.manual_seed(0)
    n_rays = 10
    per_ray = torch.arange(n_rays, dtype=torch.float32)[:, None] * torch.ones(1, 6)      # a fake per-ray gradient contribution
    b, e = parallel.shard_bounds(n_rays, r, w)
    flat = per_ray[b:e].sum(0)                                                           # local "backward"
    scale = parallel.allreduce_gradients(flat, w)
    params = torch.full((6,), float(r))
    parallel.broadcast_parameters(params, w)
    rows = parallel.gather_rows(per_ray[b:e], n_rays, r, w)
    tmax = parallel.max_over_ranks(float(r + 1), w, "cpu")
    # image rows as the sharded unit (the render / render_lerf legs): 5 rows of width 4, [rows * 4, 3] map
    img = torch.arange(5 * 4 * 3, dtype=torch.float32).reshape(20, 3)
    rb, re = parallel.shard_bounds(5, r, w)
    tiles = parallel.gather_rows(img[rb * 4:re * 4], 20, r, w, unit=4)
    ready_all = parallel.all_ranks_ready(True, w, "cpu")
    ready_one = parallel.all_ranks_ready(r == 0, w, "cpu")       # rank 1 failed its set-up: every rank must see False
    assert ready_all and not ready_one
    if r == 0:
        torch.save({"flat": flat, "scale": scale, "params": params, "rows": rows, "tmax": tmax, "tiles": tiles}, out)
    else:
        assert torch.equal(params, torch.zeros(6)) and rows is None
    dist.destroy_process_group()


def test_world_size_2_exchange_on_gloo(tmp_path):
    out = str(tmp_path / "r0.pt")
    mp.spawn(_worker, args=(2, _free_port(), out), nprocs=2, join=True)
    got = torch.load(out)
    per_ray = torch.arange(10, dtype=torch.float32)[:, None] * torch.ones(1, 6)
    assert torch.equal(got["flat"], per_ray.sum(0))            # all-reduce(sum) over ray shards == single-process sum
    assert got["scale"] == 0.5 and got["tmax"] == 2.0
    assert torch.equal(got["rows"], per_ray)                   # tile gather restores row order
    assert torch.equal(got["tiles"], torch.arange(60, dtype=torch.float32).reshape(20, 3))   # image-row shards (3 + 2 rows of width 4)
