"""The C++ drop-in LeRF / LeRFRenderer (nerfpp_b200/host/lerf.{h,cpp}, torch::Tensor boundary) against the reference's own C++ classes
(src/LeRF.cpp, src/LeRFRenderer.cpp compiled unmodified into oracle/_ref/nerfpp_ref_cuda.so) on the same B200, driven through the SAME
pybind surface (LerfPipe in nerfpp_b200/host/bindings.cpp and in oracle/ref_bindings.cpp) — SURVEY §8f-1, BASELINE C5 shape.
Tolerance: fp16-operand tensor-core head vs the reference's fp32 SGEMMs, rel 1e-2 (the north star's bf16-class bound)."""
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
BBOX = [-1.5, -1.5, -1.5, 1.5, 1.5, 1.5]
ARGS = (16, 8, 14, 16, 512, 32, 2, 256, 512)   # L, F, log2T, base, finest, geo_feat_dim_le, num_layers_le, hidden_dim_le, lang_embed_dim


@pytest.fixture(scope="module")
def host():
    from nerfpp_b200 import build
    sys.path.insert(0, str(build.build_host().parent))
    import nerfpp_b200_torch
    return nerfpp_b200_torch


def _need(ref_cuda):
    if ref_cuda is None or not hasattr(ref_cuda, "make_lerf"):
        pytest.skip("oracle/_ref/nerfpp_ref_cuda.so (with the LeRF classes) not loadable")


def _trained_looking(p, seed=3):
    """O(1) table entries, He-scaled weights and a x6 density row: the Xavier(0.1) initialisation renders empty rays on both sides."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for t in p.embed_params():
            t.copy_((torch.rand(t.shape, generator=g) * 2 - 1).to(t.device))
        for name, t in zip(p.model_param_names(), p.model_params()):
            t.copy_((torch.randn(t.shape, generator=g) * (2.0 / t.shape[1]) ** 0.5).to(t.device))
            if name.endswith("sigma_le_net_1.weight"):
                t[0] *= 6.0


def _pair(host, ref_cuda, seed=42):
    pipes = []
    for mod in (host, ref_cuda):
        mod.manual_seed(seed)
        torch.manual_seed(seed)
        p = mod.make_lerf(torch.tensor(BBOX).cuda(), *ARGS)
        p.init_model()
        _trained_looking(p)
        pipes.append(p)
    return pipes


def _rays(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    o = torch.tensor([0.3, -0.2, 4.0]).repeat(n, 1) + 0.05 * torch.randn(n, 3, generator=g)
    d = torch.tensor([0.0, 0.0, -1.0]) + 0.25 * torch.randn(n, 3, generator=g)
    return o.cuda(), d.cuda()


def test_module_surface_and_forward(host, ref_cuda, golden):
    """Registered parameter names / shapes / order equal the reference's; LeRF::forward (fused, no autograd) and RunLENetwork match it.  Against the
    reference's LeRF::forward stored in tests/golden/lerf.npz always, live against oracle/_ref when it loads."""
    g = golden("lerf.npz")
    host.manual_seed(42)
    torch.manual_seed(42)
    p = host.make_lerf(torch.tensor(BBOX).cuda(), *ARGS)
    assert p.model_param_names() == [str(n) for n in g["names"]]
    with torch.no_grad():
        for t, k in zip(p.model_params(), ("sw0", "sw1", "lw0", "lw1")):
            assert tuple(t.shape) == g[k].shape
            t.copy_(torch.from_numpy(g[k]).cuda())
        f = p.model(torch.from_numpy(g["x"]).cuda())
    assert tuple(f.shape) == g["out"].shape
    assert float(np.abs(f.cpu().numpy() - g["out"]).max()) <= 1e-2 * float(np.abs(g["out"]).max())
    if ref_cuda is None or not hasattr(ref_cuda, "make_lerf"):
        return
    a, b = _pair(host, ref_cuda)
    assert a.model_param_names() == b.model_param_names() == [f"lang_model_{n}.weight" for n in ("sigma_le_net_0", "sigma_le_net_1", "le_net_0", "le_net_1")]
    assert [tuple(t.shape) for t in a.model_params()] == [tuple(t.shape) for t in b.model_params()] == [(256, 128), (33, 256), (256, 160), (512, 256)]
    for x, y in zip(a.model_params() + a.embed_params(), b.model_params() + b.embed_params()):
        assert torch.equal(x, y)
    pts = (torch.rand(7, 50, 3, generator=torch.Generator().manual_seed(1)) * 3.4 - 1.7).cuda()      # some points outside the box
    with torch.no_grad():
        ra, rb = a.run_le_network(pts), b.run_le_network(pts)
    assert ra.shape == rb.shape == (7, 50, 513)
    assert float((ra[..., :512] - rb[..., :512]).abs().max()) <= 1e-2 * float(rb[..., :512].abs().max())
    assert float((ra[..., 512] - rb[..., 512]).abs().max()) <= 1e-2 * float(rb[..., 512].abs().max())
    outside = ((pts < -1.5) | (pts > 1.5)).any(-1)
    assert bool(outside.any()) and float(ra[outside][:, 512].abs().max()) == 0.0 and float(rb[outside][:, 512].abs().max()) == 0.0
    x = torch.randn(300, 128, generator=torch.Generator().manual_seed(2)).half().float().cuda()
    with torch.no_grad():
        fa, fb = a.model(x), b.model(x)
    assert float((fa - fb).abs().max()) <= 1e-2 * float(fb.abs().max())
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        a.model(x.cpu())


def test_render_matches_the_reference_renderer(host, ref_cuda, golden):
    """LeRFRenderer::Render on a ray batch (the call of src/NeRFExecutor.h:960-962) — fused inference path vs the reference's LibTorch + CUDA path.
    Always: RawToLEOutputs against the reference's stored in tests/golden/lerf.npz (an empty ray and an opaque wall included)."""
    g = golden("lerf.npz")
    host.manual_seed(7)
    torch.manual_seed(7)
    p = host.make_lerf(torch.tensor(BBOX).cuda(), *ARGS)
    with torch.no_grad():
        res = p.raw_to_le_outputs(*(torch.from_numpy(g[k]).cuda() for k in ("raw", "z", "rays_d")))
    for k in ("rendered", "weights", "depth", "disp", "acc"):
        np.testing.assert_allclose(res[k].cpu().numpy(), g[f"le_{k}"], rtol=1e-3, atol=1e-5, err_msg=k)
    if ref_cuda is None or not hasattr(ref_cuda, "make_lerf"):
        return
    a, b = _pair(host, ref_cuda, seed=7)
    o, d = _rays(300, seed=8)
    with torch.no_grad():
        ra = a.render(o, d, 64, 128, 128, False, False)          # 3 chunks
        rb = b.render(o, d, 64, 128, 128, False, False)
    assert ra["rendered"].shape == rb["rendered"].shape == (300, 512) and ra["weights"].shape == rb["weights"].shape == (300, 192)
    assert abs(ra["near"] - rb["near"]) < 1e-5 and abs(ra["far"] - rb["far"]) < 1e-5
    hit = rb["acc"] > 0.5
    print("rays with acc > 0.5:", int(hit.sum()))
    assert int(hit.sum()) > 20
    cos = (ra["rendered"] * rb["rendered"]).sum(-1)[hit]
    print("cosine(rendered): min", float(cos.min()), "median", float(cos.median()))
    assert float(cos.median()) > 1 - 1e-4 and float(cos.min()) > 1 - 2e-2
    for k in ("acc", "depth"):
        scale = max(1.0, float(rb[k].abs().max()))
        err = ((ra[k] - rb[k]).abs() / scale)[hit]
        print(k, "median rel err", float(err.median()), "max", float(err.max()))
        assert float(err.median()) < 2e-3 and float(err.max()) < 3e-2
    assert ra["embedding"] is None                                # the fused path does not form LangEmbedding unless asked
    with torch.no_grad():
        rm = a.render(o, d, 64, 128, 512, True, True)
    assert rm["embedding"].shape == (300, 192, 512) and rm["raw"].shape == (300, 192, 513)
    assert torch.equal(rm["rendered"], ra["rendered"])            # chunking does not change a ray's result


def test_fused_training_node_matches_libtorch_autograd(host):
    """LeRFRenderer::Render under autograd: the fused fine-pass node (nrf_lerf_fwd_train / nrf_lerf_bwd_rays / nrf_lerf_bwd_rows behind ONE
    torch::autograd::Function) against the SAME drop-in classes routed through torch::linear + LibTorch autograd (fp32 cuBLAS — the
    reference's arithmetic): loss, the gradient of every Linear weight and of the language table."""
    from nerfpp_b200 import cabi
    pipes = []
    for fused in (True, False):
        host.manual_seed(21)
        torch.manual_seed(21)
        p = host.make_lerf(torch.tensor(BBOX).cuda(), *ARGS)
        p.init_model()
        _trained_looking(p)
        p.use_fused_training(fused)
        pipes.append(p)
    o, d = _rays(256, seed=22)
    tgt = torch.nn.functional.normalize(torch.randn(256, 512, generator=torch.Generator().manual_seed(23)), dim=-1).cuda()
    n0 = cabi.launch_count()
    la, ga = pipes[0].language_grads(o, d, tgt, 64, 128)
    n1 = cabi.launch_count()
    lb, gb = pipes[1].language_grads(o, d, tgt, 64, 128)
    assert n1 - n0 >= 12                     # the fused path is made of C-ABI launches (chain, dW, per-ray kernels ...)
    assert abs(la - lb) <= 1e-2 * abs(lb)
    names = ["embeddings"] + pipes[0].model_param_names()
    stats = {}
    for name, a, b in zip(names, ga, gb):
        a, b = a.double(), b.double()
        assert float(b.norm()) > 0, name
        stats[name] = (float((a - b).norm() / b.norm()), float((a * b).sum() / (a.norm() * b.norm())))
    print("fused vs LibTorch autograd (rel, cos):", {k: (round(r, 4), round(c, 5)) for k, (r, c) in stats.items()})
    for name, (rel, cos) in stats.items():
        # bf16 operands against fp32 SGEMMs, different ReLU active sets near zero (see tests/test_gpu_lerf_train.py): direction + scale
        assert cos >= 0.995 and rel <= 8e-2, (name, rel, cos)


def test_training_steps_track_the_reference(host, ref_cuda):
    """The language lines of NeRFExecutor::Train (src/NeRFExecutor.h:957-986): Render -> huber(delta 1.25).sum(-1).nanmean() -> backward -> Adam.
    The drop-in trains through the fused fine-pass node (bf16 tcgen05 forward / backward of the head, CuHashEmbedder's sm_100a kernels at F = 8)."""
    _need(ref_cuda)
    a, b = _pair(host, ref_cuda, seed=11)
    o, d = _rays(256, seed=12)
    tgt = torch.nn.functional.normalize(torch.randn(256, 512, generator=torch.Generator().manual_seed(13)), dim=-1).cuda()
    la = a.train_steps(o, d, tgt, 12, 64, 128, 1024, 3e-4)
    lb = b.train_steps(o, d, tgt, 12, 64, 128, 1024, 3e-4)
    print("drop-in  ", [round(v, 5) for v in la])
    print("reference", [round(v, 5) for v in lb])
    assert abs(la[0] - lb[0]) <= 1e-2 * abs(lb[0])
    assert la[-1] < la[0] and lb[-1] < lb[0]
    assert abs(la[-1] - lb[-1]) <= 5e-2 * abs(lb[-1])


def test_checkpoints_are_interchangeable_with_the_reference(host, ref_cuda, tmp_path):
    """lang_embedder_checkpoint.pt / lang_model_checkpoint.pt (src/NeRFExecutor.h:556-560, 1062-1066) written by either side load into the other."""
    _need(ref_cuda)
    o, d = _rays(64, seed=4)
    for writer, reader in ((ref_cuda, host), (host, ref_cuda)):
        writer.manual_seed(21)
        torch.manual_seed(21)
        a = writer.make_lerf(torch.tensor(BBOX).cuda(), *ARGS)
        a.init_model()
        _trained_looking(a, seed=9)
        reader.manual_seed(5)
        torch.manual_seed(5)
        b = reader.make_lerf(torch.tensor(BBOX).cuda(), *ARGS)
        b.init_model()
        ckpt = tmp_path / f"lerf_{writer.__name__}"
        ckpt.mkdir()
        a.save_checkpoint(str(ckpt))
        b.load_checkpoint(str(ckpt))
        for x, y in zip(a.model_params() + a.embed_params(), b.model_params() + b.embed_params()):
            assert torch.equal(x, y)
        with torch.no_grad():
            ra, rb = a.render(o, d, 64, 128, 4096, False, False), b.render(o, d, 64, 128, 4096, False, False)
        hit = rb["acc"] > 0.5
        assert float((ra["rendered"] * rb["rendered"]).sum(-1)[hit].median()) > 1 - 1e-4
