"""GPU parity of the hash-grid kernels through the C ABI (nrf_hash_encode_fwd / _bwd) against oracle/restate.py,
the committed CUDA golden fixtures, and — when oracle/_ref/nerfpp_ref_cuda.so is loadable — the reference's own
CuHashEmbedder kernels run live on the same device."""
import numpy as np
import pytest
import torch

import restate as O

pytestmark = pytest.mark.gpu

BBOX = (-1.5, -1.5, -1.5, 1.5, 1.5, 1.5)


def _grid(L=16, F=2, T=19, base=16, finest=512, seed=1):
    from nerfpp_b200 import pipeline
    return pipeline.make_grid(BBOX, L, F, T, base, finest, "cuda", seed)


# L16 F2: the forward runs four lanes per point; L12 F2 (three 16-byte chunks per row, not a power of two): one thread per point
SHAPES = [(16, 2), (12, 2)]


def _np(grid):
    grid.c_struct()  # materialises the device-computed level scales
    return dict(box_min=BBOX[:3], box_max=BBOX[3:], scales=grid.level_scale.cpu().numpy(),
                primes=grid.primes.cpu().numpy(), biases=grid.biases.cpu().numpy(),
                offsets=grid.feat_local_idx.cpu().numpy(), sizes=grid.feat_local_size.cpu().numpy())


def _points(n, seed=0, with_edges=True):
    g = torch.Generator().manual_seed(seed)
    p = torch.rand(n, 3, generator=g) * 3 - 1.5
    if with_edges:
        p[0] = -1.5                                   # exact box_min
        p[1] = 1.5                                    # exact box_max
        p[2] = torch.tensor([0.0, 0.0, 0.0])          # cell boundary on the power-of-two levels
        p[3] = torch.tensor([1.5, -1.5, 0.75])
        p[4] = torch.tensor([1.7, 0.1, 0.2])          # outside: clamped, keep = 0
        p[5] = torch.tensor([0.1, -9.0, 0.2])
    return p.cuda()


def test_level_scales_match_expression():
    from nerfpp_b200 import ops
    s = ops.hash_level_scales(16, 512, 16, "cuda").cpu().numpy()
    assert [float(s[i]) for i in (0, 3, 6, 9, 12, 15)] == [16.0, 32.0, 64.0, 128.0, 256.0, 512.0]
    np.testing.assert_allclose(s, O.level_scales(16, 512, 16), rtol=3e-7)   # device exp2f vs numpy: <= 2 ulp
    assert np.all(np.diff(s) > 0)


def test_indices_bit_exact_at_vertices():
    """Points placed exactly on grid vertices of the power-of-two levels get weight 1 on corner 000, so the output IS
    the table entry; a table that stores bit-slices of its own scalar address reveals the hashed address exactly."""
    from nerfpp_b200 import ops
    grid = _grid()
    meta = _np(grid)
    n_sc = grid.used_scalars()
    rng = np.random.default_rng(3)
    idx = np.arange(grid.table_scalars(), dtype=np.int64)
    tables = [torch.from_numpy(((idx >> (11 * j)) & 2047).astype(np.float16)).cuda() for j in range(3)]  # 3 x 11 address bits
    for level, res in ((0, 16), (3, 32), (6, 64), (9, 128), (12, 256), (15, 512)):
        v = rng.integers(0, res + 1, size=(4096, 3))
        pts_np = (v.astype(np.float64) / res * 3.0 - 1.5).astype(np.float32)
        # keep only points whose normalised coordinate is exactly the vertex in fp32 (always true for these res)
        pos, w = O.hash_cells(pts_np, scales=meta["scales"], box_min=meta["box_min"], box_max=meta["box_max"],
                              primes=meta["primes"], biases=meta["biases"], sizes=meta["sizes"])
        assert np.all(w[:, level, 0] == 1.0)
        addr = np.zeros(len(pts_np), dtype=np.int64)
        for j in range(3):
            enc, _ = ops.hash_encode_fwd(grid, tables[j], torch.from_numpy(pts_np).cuda(), clamp=True)
            addr |= enc[:, level * 2].cpu().numpy().astype(np.int64) << (11 * j)
        expect = meta["offsets"][level].astype(np.int64) + pos[:, level, 0].astype(np.int64) * 2
        assert np.array_equal(addr, expect), f"hashed address mismatch at level {level}"
        assert expect.max() < n_sc


@pytest.mark.parametrize("F,T", [(2, 19), (8, 19), (2, 14)])
def test_every_point_level_corner_address_is_bit_exact(F, T):
    """SURVEY App. B row 1: for EVERY (point, level, corner) — all 16 levels, the ten non-power-of-two ones included, all 8 corners — the
    table address and the trilinear weight the kernels use (nrf_hash_cells runs the encode kernels' own clamp / locate code) equal the
    oracle's restatement of src/CuHashEmbedder.cu:44-90 bit for bit.  Points: uniform in the box, exact box corners, cell boundaries,
    outside points (clamped), and points within a few ulp of cell boundaries of the non-power-of-two levels."""
    from nerfpp_b200 import ops
    grid = _grid(F=F, T=T)
    meta = _np(grid)
    pts = _points(20000, seed=21).cpu().numpy()
    # points straddling cell boundaries of every level: vertex coordinate +- {0, 1, 2} ulp
    rng = np.random.default_rng(4)
    near = []
    for l, sc in enumerate(meta["scales"]):
        v = rng.integers(0, int(np.ceil(sc)) + 1, size=(400, 3)).astype(np.float64)
        p = (v / float(sc) * 3.0 - 1.5).astype(np.float32)
        for k in (-2, -1, 0, 1, 2):
            q = p.copy()
            for _ in range(abs(k)):
                q = np.nextafter(q, np.float32(np.inf if k > 0 else -np.inf), dtype=np.float32)
            near.append(q)
    pts = np.concatenate([pts] + near, 0).astype(np.float32)
    addr, w = ops.hash_cells(grid, torch.from_numpy(pts).cuda(), clamp=True)
    cl, _ = O.clamp_keep(pts, BBOX[:3], BBOX[3:])
    pos, w_ref = O.hash_cells(cl, scales=meta["scales"], box_min=meta["box_min"], box_max=meta["box_max"], primes=meta["primes"],
                              biases=meta["biases"], sizes=meta["sizes"])
    expect = meta["offsets"].astype(np.int64)[None, :, None] + pos.astype(np.int64) * F
    got = addr.cpu().numpy()
    bad = np.argwhere(got != expect)
    assert bad.size == 0, f"{len(bad)} of {got.size} (point, level, corner) addresses differ; first: {bad[:5].tolist()}"
    assert np.array_equal(w.cpu().numpy(), w_ref), "trilinear weights differ"
    assert got.max() + F <= grid.used_scalars()


@pytest.mark.parametrize("table_kind,L", [("init", 16), ("unit", 16), ("init", 12), ("unit", 12)], ids=["init", "unit", "init-L12F2", "unit-L12F2"])
def test_forward_matches_oracle(table_kind, L):
    from nerfpp_b200 import ops
    grid = _grid(L=L)
    meta = _np(grid)
    g = torch.Generator().manual_seed(5)
    n_sc = grid.table_scalars()
    table = torch.rand(n_sc, generator=g) * 1e-4 if table_kind == "init" else torch.rand(n_sc, generator=g) * 2 - 1
    t16 = ops.table_to_half(table.cuda())
    assert torch.equal(t16.cpu(), table.half())               # round-to-nearest-even like .to(kFloat16)
    pts = _points(3000)
    enc, keep = ops.hash_encode_fwd(grid, t16, pts, clamp=True)
    enc16, _ = ops.hash_encode_fwd(grid, t16, pts, clamp=True, out_f16=True)
    assert torch.equal(enc16.float(), enc)                    # both layouts carry the same fp16 values
    cl, keep_ref = O.clamp_keep(pts.cpu().numpy(), BBOX[:3], BBOX[3:])
    assert np.array_equal(keep.cpu().numpy().astype(bool), keep_ref)
    assert keep_ref[:4].all() and not keep_ref[4] and not keep_ref[5]
    ref = O.hash_encode(cl, table_f16=t16.cpu().numpy(), n_features=2, **meta)
    scale = 1e-4 if table_kind == "init" else 1.0
    # rel 1e-3 of the value plus one fp16 ulp at the table's scale (fp16 output rounding dominates, SURVEY App. B)
    np.testing.assert_allclose(enc.cpu().numpy(), ref, rtol=1e-3, atol=scale * 2 ** -10)
    exact = (enc.cpu().numpy() == ref).mean()
    assert exact > 0.9, f"only {exact:.3f} of outputs bit-equal the sequential-fp32 restatement"


def test_backward_matches_fp64_adjoint():
    from nerfpp_b200 import ops
    grid = _grid()
    meta = _np(grid)
    pts = _points(4000, seed=9)
    g = torch.Generator().manual_seed(11)
    grad = torch.randn(4000, 32, generator=g)
    grad[7] = 0.0                                             # all-zero rows take the skip path (.cu:195)
    grad[8, ::2] = 0.0
    gt = torch.zeros(grid.table_scalars(), device="cuda")
    ops.hash_encode_bwd(grid, pts, grad.cuda(), gt, clamp=True)
    cl, _ = O.clamp_keep(pts.cpu().numpy(), BBOX[:3], BBOX[3:])
    ref = O.hash_encode_bwd_f64(cl, grad_enc=grad.numpy(), n_features=2, table_scalars=grid.table_scalars(), **meta)
    got = gt.cpu().numpy().astype(np.float64)
    assert np.array_equal(got != 0, ref != 0)                 # exactly the same set of touched scalars
    assert np.all(got[grid.used_scalars():] == 0)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    assert err < 2e-6, err                                    # fp32 accumulation
    # bf16 gradient input (what nrf_mlp_small_bwd hands over)
    gt2 = torch.zeros_like(gt)
    gb = grad.cuda().bfloat16()
    ops.hash_encode_bwd(grid, pts, gb, gt2, clamp=True)
    ref2 = O.hash_encode_bwd_f64(cl, grad_enc=gb.float().cpu().numpy(), n_features=2, table_scalars=grid.table_scalars(), **meta)
    assert np.abs(gt2.cpu().numpy() - ref2).max() / np.abs(ref2).max() < 2e-6


def test_f8_grid_lerf_shape():
    """F=8 (the LeRF grid, src/main.cpp:203-207) through the same kernels."""
    from nerfpp_b200 import ops, pipeline
    grid = pipeline.make_grid(BBOX, 8, 8, 12, 8, 128, "cuda", 4)
    meta = _np(grid)
    g = torch.Generator().manual_seed(2)
    table = (torch.rand(grid.table_scalars(), generator=g) * 2 - 1).cuda()
    t16 = ops.table_to_half(table)
    pts = _points(1000, seed=4)
    enc, _ = ops.hash_encode_fwd(grid, t16, pts, clamp=True)
    cl, _ = O.clamp_keep(pts.cpu().numpy(), BBOX[:3], BBOX[3:])
    ref = O.hash_encode(cl, table_f16=t16.cpu().numpy(), n_features=8, **meta)
    np.testing.assert_allclose(enc.cpu().numpy(), ref, rtol=1e-3, atol=2 ** -10)
    grad = torch.randn(1000, 64, generator=g)
    gt = torch.zeros(grid.table_scalars(), device="cuda")
    ops.hash_encode_bwd(grid, pts, grad.cuda(), gt, clamp=True)
    refg = O.hash_encode_bwd_f64(cl, grad_enc=grad.numpy(), n_features=8, table_scalars=grid.table_scalars(), **meta)
    assert np.abs(gt.cpu().numpy() - refg).max() / np.abs(refg).max() < 2e-6


def test_empty_and_ragged():
    from nerfpp_b200 import ops
    grid = _grid()
    t16 = torch.zeros(grid.table_scalars(), dtype=torch.float16, device="cuda")
    enc, keep = ops.hash_encode_fwd(grid, t16, torch.empty(0, 3, device="cuda"))
    assert enc.shape == (0, 32) and keep.shape == (0,)
    for n in (1, 31, 257):
        enc, _ = ops.hash_encode_fwd(grid, t16, _points(n, with_edges=False))
        assert enc.shape == (n, 32) and float(enc.abs().max()) == 0.0


def test_full_size_adjoint_identity():
    """BASELINE fine-pass size (786 432 points): <enc(T), G> == <T, bwd(G)> — the forward and backward kernels are
    adjoint maps over the same hashed addresses (size-independent property; tolerance = fp16 output rounding)."""
    from nerfpp_b200 import ops
    grid = _grid()
    n = 4096 * 192
    g = torch.Generator(device="cuda").manual_seed(1)
    table = torch.rand(grid.table_scalars(), generator=g, device="cuda") * 2 - 1
    t16 = ops.table_to_half(table)
    pts = torch.rand(n, 3, generator=g, device="cuda") * 3 - 1.5
    G = torch.randn(n, 32, generator=g, device="cuda")
    enc, _ = ops.hash_encode_fwd(grid, t16, pts)
    gt = torch.zeros(grid.table_scalars(), device="cuda")
    ops.hash_encode_bwd(grid, pts, G, gt)
    lhs = (enc.double() * G.double()).sum().item()
    rhs = (t16.double() * gt.double()).sum().item()
    assert abs(lhs - rhs) / (enc.double().abs() * G.double().abs()).sum().item() < 1e-4


def _ray_ordered_points(n_rays, n_samples, seed=0):
    """Samples of a ray are consecutive rows (the order RenderRays produces): on the coarse levels neighbouring points
    share a grid cell, which is the case the warp-aggregated scatter reduces before issuing its REDs."""
    g = torch.Generator().manual_seed(seed)
    o = torch.randn(n_rays, 1, 3, generator=g)
    o = 4.0 * o / o.norm(dim=-1, keepdim=True)
    d = -o / 4.0 + 0.15 * torch.randn(n_rays, 1, 3, generator=g)
    t = torch.sort(2.0 + 4.0 * torch.rand(n_rays, n_samples, 1, generator=g), dim=1).values
    return (o + d * t).reshape(-1, 3)


@pytest.mark.parametrize("n_rays,n_samples,dtype", [(40, 100, "f32"), (33, 192, "bf16"), (7, 61, "f32")])
def test_backward_warp_aggregation_on_ray_ordered_points(n_rays, n_samples, dtype):
    """Runs of equal cells (incl. runs cut by zero-gradient rows, warp boundaries, out-of-box points and a ragged tail)
    must scatter exactly what the per-point fp64 adjoint does."""
    from nerfpp_b200 import ops
    grid = _grid()
    meta = _np(grid)
    pts = _ray_ordered_points(n_rays, n_samples, seed=n_rays)
    n = pts.shape[0]
    pts[5:9] = pts[5]                                         # identical points: one run, four members
    g = torch.Generator().manual_seed(3)
    grad = torch.randn(n, 32, generator=g)
    grad[10:14] = 0.0                                         # inactive lanes inside a run
    grad[20, 4:6] = 0.0                                       # one level of one point inactive
    grad[64:96, :8] = 0.0                                     # a whole warp inactive on the first four levels
    if dtype == "bf16":
        grad = grad.bfloat16()
    gt = torch.zeros(grid.table_scalars(), device="cuda")
    ops.hash_encode_bwd(grid, pts.cuda(), grad.cuda(), gt, clamp=True)
    cl, keep = O.clamp_keep(pts.numpy(), BBOX[:3], BBOX[3:])
    assert (~keep).any() and keep.any()
    ref = O.hash_encode_bwd_f64(cl, grad_enc=grad.float().numpy(), n_features=2, table_scalars=grid.table_scalars(), **meta)
    got = gt.cpu().numpy().astype(np.float64)
    assert np.all(got[ref == 0] == 0)                         # nothing outside the touched entries (sums may cancel to 0 inside)
    err = np.abs(got - ref).max() / np.abs(ref).max()
    assert err < 2e-6, err


def test_backward_full_size_ray_ordered_adjoint():
    """786 432 ray-ordered points (4096 rays x 192 samples): <enc(T), G> == <T, bwd(G)> with the aggregation active."""
    from nerfpp_b200 import ops
    grid = _grid()
    g = torch.Generator(device="cuda").manual_seed(5)
    table = torch.rand(grid.table_scalars(), generator=g, device="cuda") * 2 - 1
    t16 = ops.table_to_half(table)
    pts = _ray_ordered_points(4096, 192, seed=8).cuda()
    G = torch.randn(pts.shape[0], 32, generator=g, device="cuda")
    enc, _ = ops.hash_encode_fwd(grid, t16, pts)
    gt = torch.zeros(grid.table_scalars(), device="cuda")
    ops.hash_encode_bwd(grid, pts, G, gt)
    lhs = (enc.double() * G.double()).sum().item()
    rhs = (t16.double() * gt.double()).sum().item()
    assert abs(lhs - rhs) / (enc.double().abs() * G.double().abs()).sum().item() < 1e-4


def _ray_batch(n_rays, seed=0):
    from nerfpp_b200 import ops
    g = torch.Generator().manual_seed(seed)
    o = torch.randn(n_rays, 3, generator=g)
    o = (4.0 * o / o.norm(dim=-1, keepdim=True)).cuda()
    d = (-o / 4.0 + 0.2 * torch.randn(n_rays, 3, generator=g).cuda()).contiguous()
    return ops.rays_prepare(o, d, BBOX, 0.0, True)


def test_fused_point_generation_is_bit_identical():
    """nrf_hash_encode_rays_fwd/_bwd (points built in-kernel from ray_batch and z) == nrf_sample_points followed by the
    point-array entries, bit for bit (forward) / to accumulation order (backward), incl. rays that miss the box; at each of SHAPES."""
    for L, F in SHAPES:
        _fused_point_generation(L, F)


def _fused_point_generation(L, F):
    from nerfpp_b200 import ops
    grid = _grid(L=L, F=F)
    g = torch.Generator(device="cuda").manual_seed(4)
    t16 = ops.table_to_half(torch.rand(grid.table_scalars(), generator=g, device="cuda") * 2 - 1)
    rb = _ray_batch(300, seed=2)
    z = ops.z_sample(rb, torch.linspace(0, 1, 77).cuda())
    pts = ops.sample_points(rb, z)
    e0, k0 = ops.hash_encode_fwd(grid, t16, pts.view(-1, 3), clamp=True, out_f16=True)
    e1, k1 = ops.hash_encode_rays_fwd(grid, t16, rb, z, clamp=True, out_f16=True)
    assert torch.equal(e0, e1) and torch.equal(k0, k1)
    e2, _ = ops.hash_encode_rays_fwd(grid, t16, rb, z, clamp=True, out_f16=False)
    assert torch.equal(e2, ops.hash_encode_fwd(grid, t16, pts.view(-1, 3), clamp=True)[0])
    G = torch.randn(300 * 77, L * F, generator=g, device="cuda").bfloat16()
    g0 = torch.zeros(grid.table_scalars(), device="cuda")
    g1 = torch.zeros_like(g0)
    ops.hash_encode_bwd(grid, pts.view(-1, 3), G, g0)
    ops.hash_encode_rays_bwd(grid, rb, z, G, g1)
    assert torch.equal(g0 != 0, g1 != 0)
    assert (g0 - g1).abs().max().item() <= 2e-6 * g0.abs().max().item()


def test_coarse_row_reuse_is_bit_identical():
    """The fine pass copies the encoding rows of the coarse samples it contains (same z => same point): the result must
    equal a full re-encode bit for bit, perm must name only bit-identical z, and EVERY coarse sample must be found — also on the
    ray that misses the box, whose coarse depths the merge re-orders.  The raw-row scatter follows the same positions.  At each of SHAPES."""
    for L, F in SHAPES:
        _coarse_row_reuse(L, F)


def _coarse_row_reuse(L, F):
    from nerfpp_b200 import ops
    grid = _grid(L=L, F=F)
    g = torch.Generator(device="cuda").manual_seed(6)
    t16 = ops.table_to_half(torch.rand(grid.table_scalars(), generator=g, device="cuda") * 2 - 1)
    R, S, N = 257, 64, 128
    rb = _ray_batch(R, seed=5)
    rb[7, 3:6] = torch.tensor([0.0, 1.0, 0.0], device="cuda")        # a ray that misses the box: far = near + 1e-6, z not monotone in fp32
    rb[7, 0:3] = torch.tensor([9.0, 9.0, 9.0], device="cuda")
    rb2 = ops.rays_prepare(rb[:, 0:3].contiguous(), rb[:, 3:6].contiguous(), BBOX, 0.0, True)
    z = ops.z_sample(rb2, torch.linspace(0, 1, S).cuda())
    w = torch.rand(R, S, generator=g, device="cuda")
    w[3] = 0.0
    zf, perm = ops.sample_pdf_merge(z, w, torch.linspace(0, 1, N).cuda(), want_perm=True)
    assert torch.equal(zf, ops.sample_pdf_merge(z, w, torch.linspace(0, 1, N).cuda()))
    pl = perm.long()
    pos = torch.where(pl >= 0, pl, -(pl + 1))
    assert torch.equal(torch.sort(pos, dim=1).values, torch.arange(S + N, device="cuda").expand(R, -1))   # a permutation of the merged row
    claimed = pl[:, N:] >= 0
    z_at = torch.gather(zf, 1, pos[:, N:])
    assert torch.equal(z_at[claimed], z[claimed])                      # a claimed position holds the coarse z bit for bit
    assert bool((pl[:, :N] >= 0).all())
    regular = (z[:, 1:] > z[:, :-1]).all(dim=1)                        # strictly increasing coarse z (rays that really cross the box)
    assert int(regular.sum()) > R // 2 and not bool(regular.all()) and bool(claimed.all())
    # the positions against an independent formulation (torch.searchsorted): importance sample j goes behind every coarse depth <= it
    # ("coarse first on ties"), coarse sample k behind every importance depth < it — on the rays whose two lists are sorted as they stand
    _, zs = ops.sample_pdf_merge(z, w, torch.linspace(0, 1, N).cuda(), want_samples=True)
    tidy = regular & (zs[:, 1:] >= zs[:, :-1]).all(dim=1)
    assert int(tidy.sum()) > R // 2
    ar_n, ar_s = torch.arange(N, device="cuda"), torch.arange(S, device="cuda")
    assert torch.equal(pl[tidy, :N], ar_n + torch.searchsorted(z[tidy].contiguous(), zs[tidy].contiguous(), right=True))
    assert torch.equal(pl[tidy, N:], ar_s + torch.searchsorted(zs[tidy].contiguous(), z[tidy].contiguous(), right=False))
    rows = torch.randn(R * S, 4, generator=g, device="cuda")
    zf2, perm2, merged_rows = ops.sample_pdf_merge(z, w, torch.linspace(0, 1, N).cuda(), want_perm=True, raw_coarse=rows)
    assert torch.equal(zf2, zf) and torch.equal(perm2, perm)
    assert torch.equal(torch.gather(merged_rows.view(R, S + N, 4), 1, pos[:, N:, None].expand(-1, -1, 4)), rows.view(R, S, 4))
    src = perm
    enc_c, keep_c = ops.hash_encode_rays_fwd(grid, t16, rb2, z)
    full, keep_full = ops.hash_encode_rays_fwd(grid, t16, rb2, zf)
    fast, keep_fast = ops.hash_encode_rays_fwd(grid, t16, rb2, zf, reuse=(src, enc_c, keep_c, S))
    assert torch.equal(full, fast) and torch.equal(keep_full, keep_fast)


@pytest.mark.parametrize("L,feat", [(16, 2), (16, 8), (12, 2)], ids=["2", "8", "L12F2"])
def test_ray_grouped_order_changes_no_bit(L, feat):
    """nrf_hash_encode_rays_fwd_grouped walks the same sample of ray_group neighbouring rays together: rows and keep flags are those of the
    per-ray order, for a ragged ray count (not a multiple of the group), with and without row reuse, at L16 F = 2 (4 lanes / point) and F = 8
    (16), and at L12 F2 (one thread per point)."""
    from nerfpp_b200 import ops
    grid = _grid(L=L, F=feat, T=16)
    g = torch.Generator(device="cuda").manual_seed(16)
    t16 = ops.table_to_half(torch.rand(grid.table_scalars(), generator=g, device="cuda") * 2 - 1)
    R, S, N = 301, 64, 64
    rb = _ray_batch(R, seed=9)
    rb2 = ops.rays_prepare(rb[:, 0:3].contiguous(), rb[:, 3:6].contiguous(), BBOX, 0.0, True)
    z = ops.z_sample(rb2, torch.linspace(0, 1, S).cuda())
    base, keep = ops.hash_encode_rays_fwd(grid, t16, rb2, z)
    w = torch.rand(R, S, generator=g, device="cuda")
    zf, perm = ops.sample_pdf_merge(z, w, torch.linspace(0, 1, N).cuda(), want_perm=True)
    fine, keep_f = ops.hash_encode_rays_fwd(grid, t16, rb2, zf)
    for group in (8, 32, 1000):
        a, k = ops.hash_encode_rays_fwd(grid, t16, rb2, z, ray_group=group)
        assert torch.equal(a, base) and torch.equal(k, keep), group
        b, kb = ops.hash_encode_rays_fwd(grid, t16, rb2, zf, reuse=(perm, base, keep, S), ray_group=group)
        assert torch.equal(b, fine) and torch.equal(kb, keep_f), group
        # inference: no copy of the coarse rows (reuse_enc NULL) — the importance samples' rows and keep flags are all that is written
        c, kc = ops.hash_encode_rays_fwd(grid, t16, rb2, zf, reuse=(perm, None, None, S), ray_group=group)
        new = perm[:, :N].long()
        d = fine.shape[1]
        assert torch.equal(torch.gather(c.view(R, S + N, d), 1, new[:, :, None].expand(-1, -1, d)),
                           torch.gather(fine.view(R, S + N, d), 1, new[:, :, None].expand(-1, -1, d))), group
        assert torch.equal(torch.gather(kc.view(R, S + N), 1, new), torch.gather(keep_f.view(R, S + N), 1, new)), group


def test_against_reference_cuda_kernels(ref_cuda):
    """Live: the reference's CuHashEmbedder forward/backward kernels on the same table, primes and points."""
    if ref_cuda is None:
        pytest.skip("oracle/_ref/nerfpp_ref_cuda.so not loadable")
    from nerfpp_b200 import ops
    from nerfpp_b200.ops import HashGridSpec
    ref_cuda.manual_seed(42)
    # BoundingBox is a plain member of the reference module, not a buffer: ->to(device) does not move it
    pipe = ref_cuda.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, 19, 16, 512, 4, 2, 64, 15, 3, 64)
    bufs = dict(zip(pipe.embed_buffer_names(), pipe.embed_buffers()))
    table = pipe.embed_params()[0]
    with torch.no_grad():
        table.copy_(torch.rand_like(table) * 2 - 1)
    grid = HashGridSpec(BBOX, bufs["embedder_primes"].contiguous(), bufs["embedder_biases"].contiguous(),
                        bufs["embedder_feat_local_idx"].contiguous(), bufs["embedder_feat_local_size"].contiguous())
    pts = _points(20000, seed=21)
    ref_enc, ref_keep = pipe.embed(pts)
    t16 = ops.table_to_half(table.detach().reshape(-1))
    enc, keep = ops.hash_encode_fwd(grid, t16, pts)
    assert torch.equal(keep.bool(), ref_keep)
    # identical hashed cells => outputs agree to fp16 rounding of differently-ordered fp32 sums
    assert (enc - ref_enc).abs().max().item() <= 2 ** -9
    assert (enc == ref_enc).float().mean().item() > 0.95
    # gradient: ours (fp32 atomics) vs the reference's (x128 fp16 atomics), both judged against the fp64 adjoint
    gout = torch.randn(20000, 32, device="cuda") * 1e-3
    ref_enc.backward(gout)
    ref_grad = table.grad.reshape(-1).double().cpu().numpy()
    gt = torch.zeros(grid.table_scalars(), device="cuda")
    ops.hash_encode_bwd(grid, pts, gout, gt)
    meta = _np(grid)
    cl, _ = O.clamp_keep(pts.cpu().numpy(), BBOX[:3], BBOX[3:])
    exact = O.hash_encode_bwd_f64(cl, grad_enc=gout.cpu().numpy(), n_features=2, table_scalars=grid.table_scalars(), **meta)
    ours_err = np.abs(gt.double().cpu().numpy() - exact).max()
    ref_err = np.abs(ref_grad - exact).max()
    assert ours_err <= ref_err, (ours_err, ref_err)
    assert np.abs(gt.double().cpu().numpy() - ref_grad).max() <= 1e-2 * np.abs(exact).max() + 2 * ref_err


def test_against_reference_cuda_fixture(golden):
    """The committed outputs of the reference's CuHashEmbedder forward/backward kernels (tests/golden/cuhash.npz)."""
    from nerfpp_b200 import ops
    from nerfpp_b200.ops import HashGridSpec
    g = golden("cuhash.npz")
    T = lambda k: torch.from_numpy(g[k]).cuda().contiguous()   # noqa: E731
    grid = HashGridSpec(BBOX, T("primes"), T("biases"), T("feat_local_idx"), T("feat_local_size"), log2_hashmap_size=10)
    t16 = T("table_f16").reshape(-1)
    pts = T("points")
    enc, keep = ops.hash_encode_fwd(grid, t16, pts)
    assert np.array_equal(keep.cpu().numpy().astype(bool), g["keep"])
    assert (enc.cpu().numpy() == g["enc"]).mean() > 0.97                     # same cells; fp16 rounding of re-ordered fp32 sums
    np.testing.assert_allclose(enc.cpu().numpy(), g["enc"], rtol=2 ** -10, atol=2 ** -24)
    enc16, _ = ops.hash_encode_fwd(grid, t16, pts, out_f16=True)
    assert torch.equal(enc16.float(), enc)
    gt = torch.zeros(g["grad_table"].size, device="cuda")
    ops.hash_encode_bwd(grid, pts, T("grad_enc"), gt)
    meta = _np(grid)
    cl, _ = O.clamp_keep(g["points"], BBOX[:3], BBOX[3:])
    exact = O.hash_encode_bwd_f64(cl, grad_enc=g["grad_enc"], n_features=2, table_scalars=gt.numel(), **meta)
    ours_err = np.abs(gt.double().cpu().numpy() - exact).max()
    ref_err = np.abs(g["grad_table"].reshape(-1).astype(np.float64) - exact).max()
    print(f"max |dTable - fp64 adjoint|: ours {ours_err:.3e}, reference (x128 fp16 atomics) {ref_err:.3e}")
    assert ours_err <= ref_err
    assert ours_err <= 1e-5 * np.abs(exact).max()
    # the device-evaluated level scales are the fixture's
    assert np.array_equal(grid.level_scale.cpu().numpy(), golden("level_scales.npz")["s_16_512_16"])
