"""The C++ drop-in layer (nerfpp_b200/host, torch::Tensor boundary) against the reference's own C++ classes.

Both sides are driven through the SAME pybind surface — oracle/_ref/nerfpp_ref_cuda.so wraps the unmodified reference
(CuHashEmbedder, CuSHEncoder, NeRFSmall, NeRFRenderer<>; oracle/ref_bindings.cpp), nerfpp_b200/lib/nerfpp_b200_torch.so wraps
this repo's classes of the same names (nerfpp_b200/host/bindings.cpp) — so each test reads like a test of the reference."""
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
BBOX = [-1.5, -1.5, -1.5, 1.5, 1.5, 1.5]
ARGS = (16, 2, 14, 16, 512, 4, 2, 64, 15, 3, 64)   # L, F, log2T, base, finest, SH degree, sigma layers, hidden, geo, colour layers, hidden


@pytest.fixture(scope="module")
def host():
    from nerfpp_b200 import build
    sys.path.insert(0, str(build.build_host().parent))
    import nerfpp_b200_torch
    return nerfpp_b200_torch


def _pair(host, ref_cuda, seed=42, args=ARGS):
    """Same seed -> same RNG call sequence -> the two implementations draw the same table, primes and weights."""
    pipes = []
    for mod in (host, ref_cuda):
        mod.manual_seed(seed)
        torch.manual_seed(seed)
        p = mod.make_cuhash(torch.tensor(BBOX).cuda(), *args)
        p.init_model()
        pipes.append(p)
    return pipes


def _rays(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    o = torch.tensor([0.3, -0.2, 4.0]).repeat(n, 1) + 0.05 * torch.randn(n, 3, generator=g)
    d = torch.tensor([0.0, 0.0, -1.0]) + 0.25 * torch.randn(n, 3, generator=g)
    return o.cuda(), d.cuda()


def _positive_density(*pipes, value=0.3):
    """Random-init classic NeRF has sigma = 0 +- 1e-4, and RawToOutputs is DISCONTINUOUS in the sign of the last sample's sigma
    (the 1e10 interval, NeRFRenderer.h:240: acc jumps 0 -> 1), so fp16-operand vs fp32 GEMMs would be compared on a coin flip.
    Shift the density bias away from zero in every pipeline (also exercises the re-pack on a parameter change)."""
    with torch.no_grad():
        for p in pipes:
            for name, t in zip(p.model_param_names(), p.model_params()):
                if name.endswith("alpha_linear.bias"):
                    t.fill_(value)


def _need(ref_cuda):
    if ref_cuda is None:
        pytest.skip("oracle/_ref/nerfpp_ref_cuda.so not loadable")


def _fixture_pipe(host, seed, log2_t):
    """A drop-in HashNeRF pipeline built the way tests/golden/make_golden_cuda.py built the reference's for its fixtures: same seeds, same arguments."""
    host.manual_seed(seed)
    torch.manual_seed(seed)
    return host.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, log2_t, 16, 512, 4, 2, 64, 15, 3, 64)


def test_seeded_construction_and_names_match_reference(host, ref_cuda, golden):
    # the reference's seeded draws stored in tests/golden/cuhash.npz (seed 42, 2^10 table): primes, biases, level sizes / offsets bit for bit
    g = golden("cuhash.npz")
    p = _fixture_pipe(host, 42, 10)
    bufs = dict(zip(p.embed_buffer_names(), p.embed_buffers()))
    for k in ("primes", "biases", "feat_local_idx", "feat_local_size"):
        assert np.array_equal(bufs["embedder_" + k].cpu().numpy(), g[k]), k
    assert p.embed_param_names() == ["embedder_embeddings"] and tuple(p.embed_params()[0].shape) == g["table_f16"].shape
    if ref_cuda is None:
        return
    ours, ref = _pair(host, ref_cuda)
    assert ours.embed_buffer_names() == ref.embed_buffer_names()            # checkpoint compatibility (SURVEY §5)
    assert ours.model_param_names() == ref.model_param_names()
    assert ours.embed_param_names() == ["embedder_embeddings"]
    for a, b in zip(ours.embed_buffers(), ref.embed_buffers()):
        assert a.dtype == b.dtype and a.shape == b.shape and torch.equal(a, b)   # primes, biases, level sizes / offsets
    assert torch.equal(ours.embed_params()[0], ref.embed_params()[0])       # the U[0,1e-4) table, bit for bit
    for a, b in zip(ours.model_params(), ref.model_params()):
        assert torch.equal(a, b)                                            # Xavier-normal(0.1) weights
    assert ours.output_dims() == 32


def test_embedders_forward_backward_match_reference(host, ref_cuda, golden):
    # the reference's CuHashEmbedder forward / backward and CuSHEncoder outputs stored in tests/golden/cuhash.npz and cush.npz
    g = golden("cuhash.npz")
    p = _fixture_pipe(host, 42, 10)
    with torch.no_grad():
        p.embed_params()[0].copy_(torch.from_numpy(g["table_f16"]).float().cuda())
    e, k = p.embed(torch.from_numpy(g["points"]).cuda())
    assert np.array_equal(k.cpu().numpy(), g["keep"])
    ge = torch.from_numpy(g["enc"]).cuda()
    assert (e - ge).abs().max().item() <= 2 ** -9 and (e == ge).float().mean().item() > 0.95
    e.backward(torch.from_numpy(g["grad_enc"]).cuda())
    gt = p.embed_params()[0].grad.cpu().numpy()
    assert gt.shape == g["grad_table"].shape
    assert np.abs(gt - g["grad_table"]).max() <= 2e-2 * np.abs(g["grad_table"]).max()      # reference: x128 fp16 atomics
    c = golden("cush.npz")
    d = torch.from_numpy(c["dirs"]).cuda()
    for deg in range(1, 9):
        b = torch.from_numpy(c[f"sh{deg}"]).cuda()
        assert torch.allclose(host.cu_sh_encoder(d, deg), b, rtol=2e-5, atol=2e-6 * b.abs().max().item()), deg
    if ref_cuda is None:
        return
    ours, ref = _pair(host, ref_cuda)
    with torch.no_grad():
        t = torch.rand_like(ref.embed_params()[0]) * 2 - 1
        ours.embed_params()[0].copy_(t)
        ref.embed_params()[0].copy_(t)
    pts = (torch.rand(5000, 3, device="cuda") * 3.4 - 1.7).contiguous()     # some outside the box
    e1, k1 = ours.embed(pts)
    e2, k2 = ref.embed(pts)
    assert k1.dtype == torch.bool and torch.equal(k1, k2)
    assert e1.dtype == torch.float32 and (e1 - e2).abs().max().item() <= 2 ** -9 and (e1 == e2).float().mean().item() > 0.95
    g = torch.randn_like(e1) * 1e-3
    e1.backward(g)
    e2.backward(g)
    g1, g2 = ours.embed_params()[0].grad, ref.embed_params()[0].grad
    assert g1.shape == g2.shape
    assert (g1 - g2).abs().max().item() <= 2e-2 * g2.abs().max().item()     # reference: x128 fp16 atomics
    # a second forward before backward must not disturb the first one's gradient (the reference fails this, SURVEY §9-Q1)
    ours.embed_params()[0].grad = None
    ea, _ = ours.embed(pts)
    ours.embed(torch.zeros(7, 3, device="cuda"))
    ea.backward(g)
    assert torch.allclose(ours.embed_params()[0].grad, g1, rtol=1e-4, atol=1e-9)
    # the fp16 shadow follows in-place updates of the parameter (version counter), no per-forward cast
    with torch.no_grad():
        ours.embed_params()[0].mul_(0.5)
    e3, _ = ours.embed(pts)
    assert torch.allclose(e3, e1.detach() * 0.5, rtol=2e-3, atol=1e-6)
    # SH, degrees 1..8, same polynomial table
    d = torch.randn(300, 3, device="cuda")
    for deg in range(1, 9):
        a, b = host.cu_sh_encoder(d, deg), ref_cuda.cu_sh_encoder(d, deg)     # non-unit |d| up to ~4: degree-8 terms reach 1e4
        assert torch.allclose(a, b, rtol=2e-5, atol=2e-6 * b.abs().max().item())
    x = torch.rand(100, 3, device="cuda") * 2 - 1
    assert torch.allclose(host.embedder(x, 10), ref_cuda.embedder(x, 10), rtol=1e-5, atol=2e-5)


def test_model_and_render_stages_match_reference(host, ref_cuda, golden):
    # Render() of the reference's NeRFRenderer<CuHashEmbedder,CuSHEncoder,NeRFSmall> stored in tests/golden/cuhash_render.npz (single chunk, ThinRay, no
    # noise): the same seeded primes, and the maps on the fixture's table and weights
    g = golden("cuhash_render.npz")
    p = _fixture_pipe(host, 7, 12)
    bufs = dict(zip(p.embed_buffer_names(), p.embed_buffers()))
    assert np.array_equal(bufs["embedder_primes"].cpu().numpy(), g["primes"])
    with torch.no_grad():
        p.embed_params()[0].copy_(torch.from_numpy(g["table_f16"]).float().cuda())
        for i, w in enumerate(p.model_params()):
            w.copy_(torch.from_numpy(g[f"w{i}"]).cuda())
    r = p.render(torch.from_numpy(g["o"]).cuda(), torch.from_numpy(g["d"]).cuda(), 64, 128, 4096, False, True)
    assert tuple(r["weights"].shape) == g["weights"].shape == (48, 192)                  # sample count exact
    for k in ("rgb", "acc", "depth"):
        scale = max(1.0, float(np.abs(g[k]).max()))
        err = np.abs(r[k].detach().cpu().numpy() - g[k]) / scale
        assert np.median(err) < 2e-3 and err.max() < 3e-2, (k, float(np.median(err)), float(err.max()))
    if ref_cuda is None:
        return
    ours, ref = _pair(host, ref_cuda, seed=7)
    with torch.no_grad():                                                   # O(1) signal instead of the 1e-4 / 0.1-gain init
        t = (torch.rand_like(ref.embed_params()[0]) * 2 - 1).half().float()
        ours.embed_params()[0].copy_(t)
        ref.embed_params()[0].copy_(t)
        for a, b in zip(ours.model_params(), ref.model_params()):
            w = torch.randn_like(b) * (2.0 / b.shape[1]) ** 0.5
            a.copy_(w)
            b.copy_(w)
    x = torch.cat([torch.randn(777, 32, device="cuda").half().float(), torch.randn(777, 16, device="cuda")], -1)
    m1, m2 = ours.model(x), ref.model(x)
    assert (m1 - m2).abs().max().item() <= 1e-2 * m2.abs().max().item()    # bf16-class tensor-core MLP vs fp32 SGEMM
    # RawToOutputs: one fused op vs ~25 ATen launches
    raw = torch.randn(64, 192, 4, device="cuda", requires_grad=True)
    z = (2 + torch.sort(torch.rand(64, 192, device="cuda") * 4, -1).values)
    d = torch.randn(64, 3, device="cuda")
    o1 = ours.raw_to_outputs(raw, z, d, 0.0, True)
    (o1["rgb"].sum() + o1["depth"].sum() + (o1["weights"] ** 2).sum()).backward()
    g1 = raw.grad.clone()
    raw.grad = None
    o2 = ref.raw_to_outputs(raw, z, d, 0.0, True)
    (o2["rgb"].sum() + o2["depth"].sum() + (o2["weights"] ** 2).sum()).backward()
    for k in ("rgb", "depth", "disp", "acc", "weights"):
        assert torch.allclose(o1[k], o2[k], rtol=1e-3, atol=1e-6), k
    assert torch.allclose(g1, raw.grad, rtol=1e-3, atol=1e-5 * raw.grad.abs().max().item())
    # whole Render() on a ray batch, parity configuration (ThinRay, no noise), single chunk
    o, dd = _rays(96)
    r1 = ours.render(o, dd, 64, 128, 4096, False, True)
    r2 = ref.render(o, dd, 64, 128, 4096, False, True)
    assert r1["weights"].shape == r2["weights"].shape == (96, 192)          # sample count exact
    assert abs(r1["near"] - r2["near"]) < 1e-6 and abs(r1["far"] - r2["far"]) < 1e-6
    for k in ("rgb", "acc", "depth"):
        scale = max(1.0, r2[k].abs().max().item())
        err = (r1[k] - r2[k]).abs() / scale
        assert err.median().item() < 2e-3 and err.max().item() < 3e-2, (k, err.median().item(), err.max().item())
    # chunking does not change the result (and, unlike the reference, not the gradient either)
    r3 = ours.render(o, dd, 64, 128, 32, False, True)
    assert torch.allclose(r3["rgb"], r1["rgb"], rtol=1e-5, atol=1e-6)


def test_c2_size_render_matches_reference(host, ref_cuda):
    """SURVEY App. B "full RenderRays" row at the BASELINE C2 batch: 4096 rays, T = 2^19, 64 + 128 samples, ThinRay, no noise, single
    chunk, through both Render()s on the same B200 — sample count exact, maps within the bf16 class."""
    _need(ref_cuda)
    from nerfpp_b200.pipeline import synthetic_rays
    ours, ref = _pair(host, ref_cuda, seed=11, args=(16, 2, 19, 16, 512, 4, 2, 64, 15, 3, 64))
    with torch.no_grad():                                                   # O(1) signal instead of the 1e-4 / 0.1-gain init
        t = (torch.rand_like(ref.embed_params()[0]) * 2 - 1).half().float()
        ours.embed_params()[0].copy_(t)
        ref.embed_params()[0].copy_(t)
        for a, b in zip(ours.model_params(), ref.model_params()):
            w = torch.randn_like(b) * (2.0 / b.shape[1]) ** 0.5
            a.copy_(w)
            b.copy_(w)
    o, d, _ = synthetic_rays(4096, seed=12)
    r1 = ours.render(o, d, 64, 128, 4096, False, True)
    r2 = ref.render(o, d, 64, 128, 4096, False, True)
    assert r1["weights"].shape == r2["weights"].shape == (4096, 192)        # sample count = S + N_imp, exact
    assert abs(r1["near"] - r2["near"]) < 1e-6 and abs(r1["far"] - r2["far"]) < 1e-6
    assert int((r2["acc"] > 0.5).sum()) > 200                               # a real image, not an empty box
    for k in ("rgb", "acc", "depth"):
        scale = max(1.0, r2[k].abs().max().item())
        err = (r1[k] - r2[k]).abs() / scale
        print(k, "median", err.median().item(), "p99", err.flatten().kthvalue(int(0.99 * err.numel())).values.item(), "max", err.max().item())
        assert err.median().item() < 2e-3 and err.flatten().kthvalue(int(0.99 * err.numel())).values.item() < 1e-2, k
        assert err.max().item() < 1e-1, k     # a coarse-pass weight within rounding of a CDF step moves one importance sample


def test_train_steps_track_reference(host, ref_cuda):
    _need(ref_cuda)
    from nerfpp_b200.pipeline import synthetic_rays
    ours, ref = _pair(host, ref_cuda, seed=3, args=(16, 2, 15, 16, 512, 4, 2, 64, 15, 3, 64))
    o, d, tgt = synthetic_rays(1024, seed=4)
    _, l1 = ours.train_steps(o, d, tgt, 25, 64, 128, 4096, True, 1e-2, 250)
    _, l2 = ref.train_steps(o, d, tgt, 25, 64, 128, 4096, True, 1e-2, 250)
    l1, l2 = np.asarray(l1), np.asarray(l2)
    print("loss ours", l1[[0, 5, 12, 24]], "reference", l2[[0, 5, 12, 24]])
    assert abs(l1[0] - l2[0]) < 1e-4 * l2[0]                                 # identical start (same seed, same draws)
    assert np.all(np.abs(l1 - l2) < 3e-2 * l2 + 1e-5)                        # same trajectory within the bf16 class
    assert l1[-1] < 0.8 * l1[0]


def test_train_graph_tracks_the_autograd_loop(host, tmp_path):
    """HashNeRFTrainGraph (host/train_graph.h): NeRFExecutor::Train's iteration as ONE CUDA-graph replay on the C++ surface — the same kernels in
    the same order as the autograd loop issues them, on parameters that stay owned by the modules (re-pointed at one flat vector).  Same seed, same
    batch: the two loops follow the same loss trajectory, the modules end up holding the trained parameters, and checkpoints still round-trip."""
    from nerfpp_b200.pipeline import synthetic_rays
    pipes = []
    for graph in (True, False):
        host.manual_seed(3)
        torch.manual_seed(3)
        p = host.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, 15, 16, 512, 4, 2, 64, 15, 3, 64)
        p.init_model()
        p.use_fused_adam(True)
        p.use_train_graph(graph)
        pipes.append(p)
    o, d, tgt = synthetic_rays(1024, seed=4)
    before = [t.detach().clone() for t in pipes[0].model_params() + pipes[0].embed_params()]
    _, la = pipes[0].train_steps(o, d, tgt, 25, 64, 128, 4096, True, 1e-2, 250)
    _, lb = pipes[1].train_steps(o, d, tgt, 25, 64, 128, 4096, True, 1e-2, 250)
    la, lb = np.asarray(la), np.asarray(lb)
    print("graph   ", la[[0, 5, 12, 24]], "autograd", lb[[0, 5, 12, 24]])
    assert abs(la[0] - lb[0]) < 1e-5 * lb[0] + 1e-7
    assert np.all(np.abs(la - lb) < 2e-2 * lb + 1e-5)
    assert la[-1] < 0.8 * la[0]
    after = pipes[0].model_params() + pipes[0].embed_params()
    assert all(float((a - b).abs().max()) > 0 for a, b in zip(after, before))          # the MODULES' parameters moved
    assert pipes[0].model_param_names() == pipes[1].model_param_names()
    for a, b in zip(after, pipes[1].model_params() + pipes[1].embed_params()):
        diff = (a - b).abs()
        assert (diff > 1e-3).float().mean().item() < 3e-2, float((diff > 1e-3).float().mean())   # sign-like Adam: compare the bulk
    # the trained modules render (autograd-free path: fp16 shadow / packed weights re-derived from the re-pointed parameters)
    r1 = pipes[0].render(o[:96], d[:96], 64, 128, 4096, False, True)
    r2 = pipes[1].render(o[:96], d[:96], 64, 128, 4096, False, True)
    assert float((r1["rgb"] - r2["rgb"]).abs().mean()) < 2e-2
    # checkpoint round trip through torch::save / torch::load on the re-pointed parameters
    pipes[0].save_checkpoint(str(tmp_path))
    host.manual_seed(9)
    q = host.make_cuhash(torch.tensor(BBOX).cuda(), 16, 2, 15, 16, 512, 4, 2, 64, 15, 3, 64)
    q.init_model()
    q.load_checkpoint(str(tmp_path))
    r3 = q.render(o[:96], d[:96], 64, 128, 4096, False, True)
    assert torch.equal(r3["rgb"], r1["rgb"])
    # and training continues from the graph state
    _, lc = pipes[0].train_steps(o, d, tgt, 5, 64, 128, 4096, True, 1e-2, 250)
    assert lc[-1] <= la[-1] * 1.05


def test_shipped_configuration_runs(host):
    """thin_ray = false, raw noise and stochastic preconditioning on (src/main.cpp:187): the RNG-gated stages (SURVEY §9-Q4)."""
    host.manual_seed(1)
    p = host.make_cuhash(torch.tensor(BBOX).cuda(), *ARGS)
    p.init_model()
    o, d = _rays(64)
    cone = torch.tensor(1.1 / 1111.0, device="cuda")
    out = p.render_shipped(o, d, cone, 64, 128, 4096, 0.5, 0.02)
    assert out["rgb"].shape == (64, 3) and bool(torch.isfinite(out["rgb"]).all())
    # TangentScatter: offsets stay inside the cone radius and the box
    pts = torch.zeros(8, 16, 3, device="cuda")
    z = torch.linspace(2, 6, 16, device="cuda").repeat(8, 1).contiguous()
    dirs = torch.nn.functional.normalize(torch.randn(8, 3, device="cuda"), dim=-1)
    moved = host.tangent_scatter(pts, z, torch.tensor(0.01, device="cuda"), dirs, torch.tensor([-9.0] * 3 + [9.0] * 3).cuda())
    off = moved - pts
    assert bool((off.norm(dim=-1) <= 0.01 * z * 1.0001).all())
    assert float((off * dirs[:, None, :]).sum(-1).abs().max()) < 1e-5        # perpendicular to the ray
    assert float(off.norm(dim=-1).mean()) > 0.3 * 0.01 * 4                   # and actually jittered
    tv = host.total_variation_loss(p)
    assert tv.ndim == 0 and bool(torch.isfinite(tv))


def test_classic_pipeline_matches_reference(host, ref_cuda, golden):
    # Render() of the reference's NeRFRenderer<Embedder,Embedder,NeRF> stored in tests/golden/render_rays_classic.npz (width 32, the fixture's
    # weights; black and white background)
    g = golden("render_rays_classic.npz")
    host.manual_seed(5)
    torch.manual_seed(5)
    c = host.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 32, True)
    c.init_model()
    with torch.no_grad():
        for name, t in zip(c.model_param_names(), c.model_params()):
            t.copy_(torch.from_numpy(g[name.replace(".", "__")]).cuda())
    o, d = torch.from_numpy(g["o"]).cuda(), torch.from_numpy(g["d"]).cuda()
    for white, rgb_key in ((False, "rgb"), (True, "rgb_white")):
        r = c.render(o, d, 64, 128, 4096, white, True)
        assert torch.allclose(r["rgb"].cpu(), torch.from_numpy(g[rgb_key]), rtol=1e-2, atol=1e-2), white
        if not white:
            for k in ("acc", "depth"):
                assert torch.allclose(r[k].cpu(), torch.from_numpy(g[k]), rtol=1e-2, atol=1e-2), k
    if ref_cuda is None:
        return
    pipes = []
    for mod, extra in ((host, ()), (ref_cuda, (True,))):
        mod.manual_seed(5)
        torch.manual_seed(5)
        p = mod.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 256, True, *extra)
        p.init_model()
        pipes.append(p)
    ours, ref = pipes
    for a, b in zip(ours.model_params(), ref.model_params()):
        assert torch.equal(a, b)
    assert ours.model_param_names() == ref.model_param_names()
    _positive_density(ours, ref)
    o, d = _rays(32)
    r1 = ours.render(o, d, 64, 128, 4096, False, True)
    r2 = ref.render(o, d, 64, 128, 4096, False, True)
    for k in ("rgb", "acc", "depth"):
        # the coarse pass (never differentiated) runs on the fused fp16-operand forward: importance samples move by O(1e-3)
        assert torch.allclose(r1[k], r2[k], rtol=1e-2, atol=1e-2), k


def test_classic_inference_runs_on_the_fused_tcgen05_forward(host, ref_cuda):
    """Under NoGradGuard (render_image) the drop-in NeRF::forward is ONE nrf_mlp_nerf_fwd launch; the reference renders the same
    image through 11 cuBLAS SGEMMs.  fp16 operands vs fp32: maps agree to 1e-2; and the drop-in's own autograd path (torch::linear)
    agrees with its fused path.  The comparison with the reference runs where oracle/_ref/nerfpp_ref_cuda.so is loadable."""
    from nerfpp_b200 import cabi
    pipes = []
    for mod, extra in ((host, ()), (ref_cuda, (True,))):
        if mod is None:
            continue
        mod.manual_seed(9)
        torch.manual_seed(9)
        p = mod.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 256, True, *extra)
        p.init_model()
        pipes.append(p)
    ours = pipes[0]
    _positive_density(*pipes)
    K = torch.tensor([[30.0, 0, 12.0], [0, 30.0, 10.0], [0, 0, 1]])
    c2w = torch.eye(4)
    c2w[2, 3] = 4.0
    n0 = cabi.launch_count()
    a = ours.render_image(20, 24, K.cuda(), c2w.cuda(), 64, 128, 4096, False, True)
    assert cabi.launch_count() > n0
    if ref_cuda is not None:
        b = pipes[1].render_image(20, 24, K.cuda(), c2w.cuda(), 64, 128, 4096, False, True)
        for k in ("rgb", "acc", "depth"):
            assert torch.allclose(a[k], b[k], rtol=1e-2, atol=1e-2), k
    # staged inference evaluates the importance samples only (one network for both passes): the coarse samples' rows come from the coarse pass.
    # Same rows through the same row-independent kernel => the same maps bit for bit, with a third fewer network evaluations
    ours.reuse_coarse_rows(False)
    n1 = cabi.launch_count()
    full = ours.render_image(20, 24, K.cuda(), c2w.cuda(), 64, 128, 4096, False, True)
    ours.reuse_coarse_rows(True)
    for k in ("rgb", "acc", "depth", "weights"):
        assert torch.equal(a[k], full[k]), k
    assert cabi.launch_count() > n1
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ours.model(torch.rand(4, 90))                             # a CPU tensor at the built shape is refused, not routed through ATen
    x = torch.rand(300, 90).cuda()
    with torch.no_grad():
        fused = ours.model(x)
    plain = ours.model(x.requires_grad_(True))      # grad mode on: torch::linear path
    assert float((fused - plain.detach()).abs().max()) <= 1e-2 * float(plain.abs().max()) + 1e-4


def test_fused_adam_tracks_torch_adam(host):
    """FusedAdam (nrf_adam_step per parameter, same state objects) in the reference's training loop vs torch::optim::Adam."""
    pipes = []
    for fused in (False, True):
        host.manual_seed(7)
        torch.manual_seed(7)
        p = host.make_cuhash(torch.tensor(BBOX).cuda(), *ARGS)
        p.init_model()
        p.use_fused_adam(fused)
        pipes.append(p)
    o, d = _rays(512, seed=3)
    tgt = torch.rand(512, 3, generator=torch.Generator().manual_seed(1)).cuda()
    losses = [p.train_steps(o, d, tgt, 5, 64, 128, 512, True, 1e-2, 250)[1] for p in pipes]
    np.testing.assert_allclose(losses[1], losses[0], rtol=5e-3)
    for a, b in zip(pipes[0].model_params() + pipes[0].embed_params(), pipes[1].model_params() + pipes[1].embed_params()):
        diff = (a - b).abs()
        assert (diff > 1e-4).float().mean().item() < 2e-2 and diff.median().item() < 1e-6   # sign-like Adam: see test_gpu_pipeline


def test_classic_training_runs_on_the_fused_tcgen05_kernels(host):
    """NeRFExecutor::Train's loop (Render + huber + backward + Adam, src/NeRFExecutor.h:868-996) on NeRFRenderer<Embedder,Embedder,NeRF>:
    the drop-in's fused training path (nrf_mlp_nerf_fwd_train / nrf_mlp_nerf_bwd behind one autograd Function, bf16) against the same
    module on torch::linear + LibTorch autograd (fp32 cuBLAS — the reference's arithmetic).  Same seeds, reference initialisation
    (Xavier 0.1): gradients agree in direction and scale, and the loss curves track each other."""
    from nerfpp_b200 import cabi
    pipes = []
    for fused in (True, False):
        host.manual_seed(11)
        torch.manual_seed(11)
        p = host.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 256, True)
        p.init_model()
        host.classic_set_fused_training(p, fused)
        pipes.append(p)
    o, d = _rays(256, seed=5)
    tgt = torch.rand(256, 3, generator=torch.Generator().manual_seed(2)).cuda()
    # one step with lr = 0: parameters unchanged, .grad populated
    n0 = cabi.launch_count()
    pipes[0].train_steps(o, d, tgt, 1, 64, 128, 4096, True, 0.0, 250)
    assert cabi.launch_count() - n0 >= 4            # pack, fwd_train, chain, dW at least
    pipes[1].train_steps(o, d, tgt, 1, 64, 128, 4096, True, 0.0, 250)
    for name, a, b in zip(pipes[0].model_param_names(), pipes[0].model_params(), pipes[1].model_params()):
        ga, gb = a.grad.double(), b.grad.double()
        assert float(gb.norm()) > 0, name
        cos = float((ga * gb).sum() / (ga.norm() * gb.norm()))
        # Xavier(0.1): activations shrink ~14x per layer, a large share of the units sit within bf16 rounding of the ReLU kink, and the
        # bf16 forward flips them — direction check here; the element-wise 1e-2 check on the same active sets is
        # tests/test_gpu_mlp_nerf.py::test_train_forward_and_backward_match_fp64_autograd, and the O(1)-weights case follows
        assert cos >= 0.97 and 0.8 <= float(ga.norm() / gb.norm()) <= 1.25, (name, cos, float(ga.norm() / gb.norm()))
    losses = [p.train_steps(o, d, tgt, 20, 64, 128, 4096, True, 5e-4, 250)[1] for p in pipes]
    assert losses[0][-1] < losses[0][0] and losses[1][-1] < losses[1][0]
    np.testing.assert_allclose(losses[0], losses[1], rtol=5e-2)


def test_classic_training_gradients_with_order_one_weights(host):
    """The same comparison with He-initialised weights (activations O(1): few units within bf16 rounding of the ReLU kink): the fused bf16
    training path against torch::linear + LibTorch autograd in fp32, through the whole Render + huber + backward — norm-wise rel 2e-2."""
    import math
    pipes = []
    for fused in (True, False):
        host.manual_seed(13)
        torch.manual_seed(13)
        p = host.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 256, True)
        p.init_model()
        host.classic_set_fused_training(p, fused)
        pipes.append(p)
    g = torch.Generator().manual_seed(14)
    with torch.no_grad():
        for a, b in zip(pipes[0].model_params(), pipes[1].model_params()):
            w = torch.randn(a.shape, generator=g) * (math.sqrt(2.0 / a.shape[1]) if a.dim() == 2 else 0.1)
            a.copy_(w.cuda())
            b.copy_(w.cuda())
    _positive_density(*pipes)
    o, d = _rays(256, seed=6)
    tgt = torch.rand(256, 3, generator=torch.Generator().manual_seed(3)).cuda()
    for p in pipes:
        p.train_steps(o, d, tgt, 1, 64, 128, 4096, True, 0.0, 250)
    stats = {}
    for name, a, b in zip(pipes[0].model_param_names(), pipes[0].model_params(), pipes[1].model_params()):
        ga, gb = a.grad.double(), b.grad.double()
        stats[name] = (float((ga - gb).norm() / gb.norm().clamp_min(1e-300)), float((ga * gb).sum() / (ga.norm() * gb.norm()).clamp_min(1e-300)))
    print("classic training gradients, fused bf16 vs fp32 ATen, (rel, cos):", {k: (round(r, 4), round(c, 5)) for k, (r, c) in stats.items()})
    for name, (rel, cos) in stats.items():
        # the last layers see one bf16 rounding of their operands; the first layers inherit the rounding of nine layers in both directions
        tol = 2e-2 if ("rgb_linear" in name or "views_linears" in name) else 1.5e-1
        assert rel <= tol and cos >= 0.99, (name, rel, cos)


@pytest.mark.parametrize("kind", ["cuhash", "classic"])
def test_checkpoints_are_interchangeable_with_the_reference(host, ref_cuda, kind, tmp_path):
    """SURVEY §8f-4: torch::save archives written by NeRFExecutor::SaveCheckpoint (src/NeRFExecutor.h:1054-1068: embedder_checkpoint.pt,
    model_checkpoint.pt) load into the drop-in modules and vice versa — same registered parameter / buffer names and shapes — and the
    loaded model renders the same image as the one that wrote the archive."""
    _need(ref_cuda)
    make = (lambda mod, *extra: mod.make_cuhash(torch.tensor(BBOX).cuda(), *ARGS)) if kind == "cuhash" else \
        (lambda mod, *extra: mod.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 256, True, *extra))
    extra = () if kind == "cuhash" else (True,)
    o, d = _rays(300, seed=8)
    for writer, reader, w_extra, r_extra in ((ref_cuda, host, extra, ()), (host, ref_cuda, (), extra)):
        writer.manual_seed(21)
        torch.manual_seed(21)
        a = make(writer, *w_extra)
        a.init_model()
        with torch.no_grad():                # trained-looking values: the initialisation renders an all-background image on both sides
            for t in a.model_params():
                if t.dim() == 2:
                    t.mul_(12.0)
            for t in a.embed_params():
                t.copy_((torch.rand(t.shape, generator=torch.Generator().manual_seed(3)) * 2 - 1).to(t.device))
        if kind == "classic":
            _positive_density(a)
        reader.manual_seed(5)
        torch.manual_seed(5)
        b = make(reader, *r_extra)
        b.init_model()
        ckpt = tmp_path / f"{kind}_{writer.__name__}"
        ckpt.mkdir()
        a.save_checkpoint(str(ckpt))
        b.load_checkpoint(str(ckpt))
        for x, y in zip(a.model_params() + a.embed_params() + a.embed_buffers(), b.model_params() + b.embed_params() + b.embed_buffers()):
            assert torch.equal(x, y)
        with torch.no_grad():
            ra = a.render(o, d, 64, 128, 4096, False, True)
            rb = b.render(o, d, 64, 128, 4096, False, True)
        solid = rb["acc"] > 0.5                                             # depth = sum(w z) / max(acc, 1e-10) is ill-conditioned on empty rays
        for k in ("rgb", "acc", "depth"):                                   # same criterion as the render parity test above
            scale = max(1.0, rb[k].abs().max().item())
            err = (ra[k] - rb[k]).abs() / scale
            if k == "depth":
                err = err[solid]
            assert err.median().item() < 2e-3 and err.max().item() < 3e-2, (kind, k, err.median().item(), err.max().item())


def test_classic_run_network_fuses_the_embeddings(host):
    """RunNetwork for <Embedder, Embedder, NeRF> (src/NeRFRenderer.h:164-194): with the positional embeddings evaluated inside the MLP
    kernel (default) the raw outputs, rendered maps and parameter gradients equal those of embed + expand + cat + forward with separate
    kernels (FusedEmbedding = false): same operands, so inference is bit-identical; gradients differ by fp32 atomic order only."""
    pipes = []
    for fused in (True, False):
        host.manual_seed(13)
        torch.manual_seed(13)
        p = host.make_classic(torch.tensor(BBOX).cuda(), 10, 4, 8, 256, True)
        p.init_model()
        host.classic_set_fused_embedding(p, fused)
        pipes.append(p)
    a, b = pipes
    _positive_density(a, b)
    with torch.no_grad():
        for x, y in zip(a.model_params(), b.model_params()):
            if x.dim() == 2:
                x.mul_(12.0)
                y.mul_(12.0)
    g = torch.Generator().manual_seed(6)
    pts = (torch.rand(37, 50, 3, generator=g) * 3 - 1.5).cuda()
    dirs = torch.nn.functional.normalize(torch.randn(37, 3, generator=g), dim=-1).cuda()
    with torch.no_grad():
        ra, rb = a.run_network(pts, dirs), b.run_network(pts, dirs)
        assert ra.shape == (37, 50, 4) and torch.equal(ra, rb)
        o, d = _rays(300, seed=4)
        ia, ib = a.render(o, d, 64, 128, 4096, False, True), b.render(o, d, 64, 128, 4096, False, True)
        for k in ("rgb", "acc", "depth"):
            assert torch.equal(ia[k], ib[k]), k
    tgt = torch.rand(300, 3, generator=g).cuda()
    a.train_steps(o, d, tgt, 1, 64, 128, 4096, True, 0.0, 250)
    b.train_steps(o, d, tgt, 1, 64, 128, 4096, True, 0.0, 250)
    for name, x, y in zip(a.model_param_names(), a.model_params(), b.model_params()):
        assert float(y.grad.abs().max()) > 0, name
        assert torch.allclose(x.grad, y.grad, rtol=1e-3, atol=1e-6 * float(y.grad.abs().max())), name


def test_writes_behind_the_version_counter_need_invalidate_caches(host):
    """The fp16 table shadow and the packed weight blobs are keyed on (data_ptr, Tensor::_version()).  A write through an alias with its own
    version counter (`.data`, a raw kernel, an NCCL broadcast) is invisible to that key: InvalidateCaches() is the documented hand-shake."""
    host.manual_seed(7)
    pipe = host.make_cuhash(torch.tensor(BBOX).cuda(), *ARGS)
    table = pipe.embed_params()[0]
    with torch.no_grad():
        table.copy_(torch.rand_like(table) * 2 - 1)
    x = (torch.rand(257, 3, device="cuda") * 2 - 1)
    with torch.no_grad():
        a = pipe.embed(x)[0].clone()
        table.mul_(2.0)                                   # through the parameter: version bumped, the shadow follows
        b = pipe.embed(x)[0].clone()
        np.testing.assert_allclose(b.cpu().numpy(), 2 * a.cpu().numpy(), rtol=2e-3, atol=1e-4)
        table.data.mul_(0.5)                              # through .data: own version counter, the key does not move
        stale = pipe.embed(x)[0].clone()
        assert torch.equal(stale, b)
        host.invalidate_caches(pipe)
        c = pipe.embed(x)[0]
        np.testing.assert_allclose(c.cpu().numpy(), a.cpu().numpy(), rtol=2e-3, atol=1e-4)


def test_inference_render_is_one_call_and_matches_the_staged_path_and_the_reference(host, ref_cuda):
    """Render() under NoGradGuard in the parity configuration: the drop-in RenderRays is ONE C-ABI call per chunk (nrf_render_raybatch_fwd:
    importance-only fine pass, ray-grouped gathers).  Same kernels as the staged path, hence the same bits; against the reference's own
    Render on the same weights within the tensor-core tolerance.  A ragged last chunk and white background included."""
    from nerfpp_b200 import cabi
    host.manual_seed(11)
    torch.manual_seed(11)
    ours = host.make_cuhash(torch.tensor(BBOX).cuda(), *ARGS)
    ours.init_model()
    with torch.no_grad():
        t = (torch.rand_like(ours.embed_params()[0]) * 2 - 1).half().float()
        ours.embed_params()[0].copy_(t)
        ws = [torch.randn_like(b) * (2.0 / b.shape[1]) ** 0.5 for b in ours.model_params()]
        for a, w in zip(ours.model_params(), ws):
            a.copy_(w)
    K = torch.tensor([[60.0, 0, 24.0], [0, 60.0, 20.0], [0, 0, 1]])
    c2w = torch.tensor([[1.0, 0, 0, 0.2], [0, 1, 0, -0.1], [0, 0, 1, 4.0], [0, 0, 0, 1]])
    for white in (False, True):
        ours.use_fused_inference(True)
        l0 = cabi.launch_count()
        a = ours.render_image(40, 48, K.cuda(), c2w.cuda(), 64, 128, 700, white, True)       # 1920 rays: two full chunks + a ragged one
        fused_launches = cabi.launch_count() - l0
        ours.use_fused_inference(False)
        l0 = cabi.launch_count()
        b = ours.render_image(40, 48, K.cuda(), c2w.cuda(), 64, 128, 700, white, True)
        staged_launches = cabi.launch_count() - l0
        for k in ("rgb", "depth", "disp", "acc", "weights"):
            assert torch.equal(a[k], b[k]), (k, white)
        assert fused_launches < staged_launches
    if ref_cuda is not None:
        ref_cuda.manual_seed(11)
        torch.manual_seed(11)
        ref = ref_cuda.make_cuhash(torch.tensor(BBOX).cuda(), *ARGS)
        ref.init_model()
        with torch.no_grad():
            ref.embed_params()[0].copy_(t)
            for b_, w in zip(ref.model_params(), ws):
                b_.copy_(w)
        for pa, pb in zip(ours.embed_buffers(), ref.embed_buffers()):                         # same primes / offsets (same seed, same call order)
            assert torch.equal(pa.cpu(), pb.cpu())
        ours.use_fused_inference(True)
        a = ours.render_image(40, 48, K.cuda(), c2w.cuda(), 64, 128, 700, False, True)
        r = ref.render_image(40, 48, K.cuda(), c2w.cuda(), 64, 128, 700, False, True)
        for k in ("rgb", "depth", "acc"):
            x, y = a[k].float().cpu().numpy(), r[k].float().cpu().numpy()
            close = np.isclose(x, y, rtol=1e-2, atol=1e-2)
            close = close.all(axis=-1) if close.ndim > 2 else close
            assert close.mean() > 0.97, (k, close.mean())                                     # bf16-class MLP behind importance sampling: see test_gpu_pipeline
            np.testing.assert_allclose(x, y, rtol=1e-1, atol=1e-1)
