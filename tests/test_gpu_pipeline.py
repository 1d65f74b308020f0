"""End-to-end GPU parity of the HashNeRF pipeline (nerfpp_b200/pipeline.py, every stage a C-ABI call) against the
composed oracle (oracle/restate.py): RenderRays outputs, sample counts, and the gradients of one training step."""
import numpy as np
import pytest
import torch

import restate as O

pytestmark = pytest.mark.gpu
BBOX = (-1.5, -1.5, -1.5, 1.5, 1.5, 1.5)


def _model(**kw):
    from nerfpp_b200.pipeline import HashNeRF
    return HashNeRF(BBOX, log2_hashmap_size=kw.pop("T", 14), **kw)


def _meta(m):
    g = m.grid
    g.c_struct()
    return dict(box_min=BBOX[:3], box_max=BBOX[3:], scales=g.level_scale.cpu().numpy(), primes=g.primes.cpu().numpy(),
                biases=g.biases.cpu().numpy(), offsets=g.feat_local_idx.cpu().numpy(), sizes=g.feat_local_size.cpu().numpy())


def _oracle_network(m, table_f16_np, weights):
    meta = _meta(m)

    def run(pts, viewdirs):
        r, s, _ = pts.shape
        flat = pts.reshape(-1, 3).numpy()
        cl, keep = O.clamp_keep(flat, BBOX[:3], BBOX[3:])
        enc = O.hash_encode(cl, table_f16=table_f16_np, n_features=2, **meta)
        sh = O.sh_encode_closed_form(viewdirs.numpy(), m.sh_degree).astype(np.float32)
        x = torch.cat([torch.from_numpy(enc), torch.from_numpy(sh).repeat_interleave(s, 0)], -1)
        out = O.nerf_small_forward(x, (weights[:2], weights[2:]), input_ch_views=m.sh_degree ** 2)
        out = torch.cat([out[:, :3], out[:, 3:] * torch.from_numpy(keep).float()[:, None]], -1)   # NeRFRenderer.h:188
        return out.reshape(r, s, 4)
    return run


def _rays(n, seed=0):
    g = torch.Generator().manual_seed(seed)
    o = torch.tensor([0.3, -0.2, 4.0]).repeat(n, 1) + 0.05 * torch.randn(n, 3, generator=g)
    d = torch.tensor([0.0, 0.0, -1.0]) + 0.25 * torch.randn(n, 3, generator=g)
    return o, d


@pytest.mark.parametrize("degree", [4, 8])
def test_render_rays_matches_composed_oracle(degree):
    """degree 8: the reference's shipped 64 view channels (src/main.cpp:176), which the fused kernels take as a per-ray term."""
    m = _model(seed=3, sh_degree=degree)
    g = torch.Generator(device="cuda").manual_seed(1234)         # own generator: the result must not depend on which tests ran before
    with torch.no_grad():                                        # O(1) densities / colours so the test has signal
        m.params[:m.n_table] = torch.rand(m.n_table, device="cuda", generator=g) * 2 - 1
        off = m.n_table
        for fo, fi in m.mlp_layers:
            m.params[off:off + fo * fi] = torch.randn(fo * fi, device="cuda", generator=g) * (2.0 / fi) ** 0.5
            off += fo * fi
    m.refresh()
    o, d = _rays(24)
    out = m.render_rays(o.cuda(), d.cuda())
    assert out["z"].shape == (24, 64 + 128)                       # sample count exact
    ws = [w.detach().cpu().clone() for w in m.mlp_weights()]
    net = _oracle_network(m, m.table_f16.cpu().numpy(), ws)
    rb = O.ray_batch(o, d, torch.tensor(BBOX))
    ref, ref_coarse, z_ref = O.render_rays(rb, 64, 128, net)
    # BASELINE tolerance for the bf16 tensor-core class: rel 1e-2 on RGB / depth / acc.  The maps are a chain network -> weights -> importance
    # samples -> network, and with O(1) random densities a ray whose opacity sits on one sample amplifies the network's rounding: every ray
    # within 5e-2, nine in ten within 1e-2 (the network itself is held to 1e-2 row by row in test_gpu_mlp.py)
    for k in ("rgb", "depth", "acc"):
        a, b = out[k].cpu().numpy(), ref[k].numpy()
        np.testing.assert_allclose(a, b, rtol=5e-2, atol=5e-2, err_msg=k)
        close = np.isclose(a, b, rtol=1e-2, atol=1e-2)
        close = close.all(axis=-1) if close.ndim > 1 else close
        assert close.mean() >= 0.9, (k, close.mean())
    # the coarse z grid is the same floats; fine z within the sampler's tolerance of the oracle's
    assert torch.equal(torch.sort(out["z"], -1).values, out["z"])
    zd = (out["z"].cpu() - z_ref).abs()
    print("max |z_fine - oracle| =", float(zd.max()), " median =", float(zd.median()))
    assert float(zd.median()) < 1e-3


def test_render_against_reference_cuda_fixture(golden):
    """Render() of the reference's NeRFRenderer<CuHashEmbedder,CuSHEncoder,NeRFSmall> on the B200 (tests/golden/cuhash_render.npz)."""
    g = golden("cuhash_render.npz")
    m = _model(seed=0, T=12, primes=g["primes"])
    with torch.no_grad():
        m.params[:m.n_table] = torch.from_numpy(g["table_f16"]).reshape(-1)[:m.n_table].float().cuda()
        m.params[m.n_table:] = torch.cat([torch.from_numpy(g[f"w{i}"]).reshape(-1) for i in range(5)]).cuda()
    m.refresh()
    out = m.render_rays(torch.from_numpy(g["o"]).cuda(), torch.from_numpy(g["d"]).cuda())
    assert out["z"].shape == (48, 192)
    for k in ("rgb", "acc", "depth"):
        scale = max(1.0, float(np.abs(g[k]).max()))                          # rgb / acc are O(1), depth is in scene units
        err = np.abs(out[k].cpu().numpy() - g[k]) / scale
        print(k, "median rel err", float(np.median(err)), "max", float(err.max()))
        assert np.median(err) < 2e-3, k                                       # bf16-class MLP vs the reference's fp32 SGEMM
        assert err.max() < 3e-2, k                                            # a ray whose u == 1.0 sample took the other tie branch


@pytest.mark.parametrize("degree", [4, 8])
def test_train_step_gradients_match_autograd_oracle(degree):
    """One training step against fp64 autograd through the composed oracle.  degree 8 = 64 view channels, whose weight gradient takes the per-ray
    route (nrf_mlp_small_bwd_raybias -> nrf_mlp_small_view_bias_bwd)."""
    m = _model(seed=5, T=12, sh_degree=degree)
    torch.manual_seed(20261017)          # the parameters below come from the CUDA generator: do not depend on which tests ran before
    with torch.no_grad():
        m.params[:m.n_table] = torch.rand(m.n_table, device="cuda") * 2 - 1
        off = m.n_table
        for fo, fi in m.mlp_layers:
            m.params[off:off + fo * fi] = torch.randn(fo * fi, device="cuda") * (1.0 / fi) ** 0.5
            off += fo * fi
    m.refresh()
    o, d = _rays(16, seed=2)
    target = torch.rand(16, 3)
    out = m.forward_backward(o.cuda(), d.cuda(), target.cuda())
    z_fine = out["z"].cpu()                                        # z is detached in the reference (NeRFRenderer.h:429)

    meta = _meta(m)
    rb = O.ray_batch(o, d, torch.tensor(BBOX))
    pts = (rb[:, None, 0:3] + rb[:, None, 3:6] * z_fine[:, :, None]).reshape(-1, 3).numpy()
    cl, keep = O.clamp_keep(pts, BBOX[:3], BBOX[3:])
    pos, w = O.hash_cells(cl, meta["box_min"], meta["box_max"], meta["scales"], meta["primes"], meta["biases"], meta["sizes"])
    table = m.table_f16.cpu().double().requires_grad_(True)
    idx = torch.from_numpy(meta["offsets"].astype(np.int64))[None, :, None] + torch.from_numpy(pos.astype(np.int64)) * 2
    wt = torch.from_numpy(w).double()
    enc = torch.stack([(wt * table[idx + k]).sum(-1) for k in range(2)], -1).reshape(len(pts), 32)
    enc = enc + (enc.detach().half().double() - enc.detach())     # fp16 output rounding, straight-through
    sh = torch.from_numpy(O.sh_encode_closed_form(rb[:, 8:11].numpy(), degree)).repeat_interleave(192, 0)
    ws = [x.detach().cpu().double().requires_grad_(True) for x in m.mlp_weights()]
    raw = O.nerf_small_forward(torch.cat([enc, sh], -1), (ws[:2], ws[2:]), input_ch_views=degree * degree)
    raw = torch.cat([raw[:, :3], raw[:, 3:] * torch.from_numpy(keep).double()[:, None]], -1).reshape(16, 192, 4)
    res = O.raw_to_outputs(raw, z_fine.double(), rb[:, 3:6].double())
    loss = O.huber(res["rgb"], target.double())
    loss.backward()

    assert abs(float(m.loss) - float(loss.detach())) < 1e-2 * abs(float(loss.detach())) + 1e-6
    g_mlp = m.grads[m.n_table:].cpu().double()
    g_ref = torch.cat([x.grad.reshape(-1) for x in ws])
    e_mlp = float((g_mlp - g_ref).abs().max() / g_ref.abs().max())
    g_tab = m.grads[:m.n_table].cpu().double()
    e_tab = float((g_tab - table.grad).abs().max() / table.grad.abs().max())
    print(f"rel err: loss {abs(float(m.loss) - float(loss)) / float(loss):.2e}  dMLP {e_mlp:.2e}  dTable {e_tab:.2e}")
    assert e_mlp < 2e-2                                            # bf16 class (north star: rel 1e-2 bf16, on a chained backward)
    assert e_tab < 3e-2
    gv, rv = m.mlp_grads_view(2)[:, :degree * degree], ws[2].grad[:, :degree * degree]      # the view columns of color_net_0 on their own
    assert float((gv.cpu().double() - rv).abs().max() / rv.abs().max()) < 2e-2
    assert torch.equal(g_tab != 0, table.grad != 0) or float(((g_tab != 0) != (table.grad != 0)).float().mean()) < 1e-3


def test_training_reduces_loss_and_keeps_shadow_in_sync():
    from nerfpp_b200.pipeline import synthetic_rays
    m = _model(seed=1, T=15)
    o, d, tgt = synthetic_rays(1024, seed=4)
    losses = []
    for _ in range(40):
        losses.append(float(m.train_step(o, d, tgt)))
    assert np.isfinite(losses).all()
    assert losses[-1] < 0.7 * losses[0], losses[::8]
    assert torch.equal(m.table_f16, m.table.half())               # Adam refreshed the fp16 shadow
    assert float(m.grads.abs().max()) == 0.0                      # and cleared the gradient
    assert m.step == 40


def test_render_image_tiles_agree():
    m = _model(seed=2, T=14)
    K = np.array([[60.0, 0, 20], [0, 60.0, 15], [0, 0, 1]], dtype=np.float32)
    c2w = np.array([[1, 0, 0, 0.1], [0, 1, 0, -0.2], [0, 0, 1, 4.0]], dtype=np.float32)
    full = m.render_image(30, 40, K, c2w)
    top = m.render_image(30, 40, K, c2w, row_begin=0, row_end=15)
    bot = m.render_image(30, 40, K, c2w, row_begin=15, row_end=30)
    assert torch.equal(full["rgb"], torch.cat([top["rgb"], bot["rgb"]], 0))
    assert full["rgb"].shape == (1200, 3)
    # from the camera alone (nrf_render_tile_fwd: GetRays inside the prologue kernel) == nrf_get_rays + nrf_render_rays_fwd, also when a
    # chunk starts in the middle of an image row
    for chunk in (1 << 18, 333):
        rays = m.render_image(30, 40, K, c2w, chunk=chunk, row_begin=7, row_end=30, from_camera=False)
        cam = m.render_image(30, 40, K, c2w, chunk=chunk, row_begin=7, row_end=30)
        for k in ("rgb", "depth", "disp", "acc"):
            assert torch.equal(rays[k], cam[k]), (k, chunk)


def test_graph_replay_matches_eager_steps():
    """The captured step (one CUDA-graph replay, device-side Adam schedule) must train like the eagerly launched one."""
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    a = HashNeRF(BBOX, log2_hashmap_size=15, seed=3, lrate_decay=1)     # fast decay: the schedule matters within a few steps
    b = HashNeRF(BBOX, log2_hashmap_size=15, seed=3, lrate_decay=1)
    c = HashNeRF(BBOX, log2_hashmap_size=15, seed=3, lrate_decay=1)     # second eager replica: the atomic-order noise floor
    assert torch.equal(a.params, b.params)
    batches = [synthetic_rays(512, seed=20 + i) for i in range(3)]
    b.capture_train_step(512)
    assert torch.equal(a.params, b.params)                              # capture + warm-up leave the parameters untouched
    la, lb = [], []
    for i in range(6):
        la.append(float(a.train_step(*batches[i % 3])))
        lb.append(float(b.train_step_graph(*batches[i % 3])))
        c.train_step(*batches[i % 3])
    assert b.step == a.step == 6 and int(b.sched[0]) == 6
    np.testing.assert_allclose(lb, la, rtol=2e-3)
    # same arithmetic, different atomic orders.  Adam with eps = 1e-15 is sign-like, so the few entries whose gradient is a
    # cancelling sum (order-dependent sign) may move by up to 2 lr per step in either run; everything else must agree
    diff = (a.params - b.params).abs()
    noise = ((a.params - c.params).abs() > 1e-4).float().mean().item()
    frac = (diff > 1e-4).float().mean().item()
    # (two eager replicas share launch timing, so their atomic orders are correlated and `noise` is a lower bound)
    assert frac < max(4.0 * noise, 2e-2), (frac, noise)
    assert diff.median().item() < 1e-6
    assert torch.equal(b.shadow[:b.n_table], b.params[:b.n_table].half())
    # eager steps in between re-seed the device-side step counter
    a.train_step(*batches[0]); b.train_step(*batches[0])
    a.train_step(*batches[1]); b.train_step_graph(*batches[1])
    assert int(b.sched[0]) == 8 and b.step == 8
    assert ((a.params - b.params).abs() > 1e-4).float().mean().item() < max(6.0 * noise, 3e-2)


def test_scheduled_adam_matches_host_schedule():
    from nerfpp_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(0)
    n = 4099
    p0 = torch.randn(n, device="cuda", generator=g)
    pa, pb = p0.clone(), p0.clone()
    ma, va, mb, vb = (torch.zeros(n, device="cuda") for _ in range(4))
    sched = torch.zeros(4, dtype=torch.int32, device="cuda")
    for step in range(1, 6):
        grad = torch.randn(n, device="cuda", generator=g)
        lr = 1e-2 * (0.1 ** (max(step - 2, 0) / 3.0))
        ops.adam_step(pa, grad.clone(), ma, va, lr, step, 0.9, 0.99, 1e-15, 0.5, True)
        ops.adam_schedule_advance(sched, 1e-2, 0.1, 3.0)
        ops.adam_step_scheduled(pb, grad.clone(), mb, vb, sched, 0.9, 0.99, 1e-15, 0.5, True)
        assert int(sched[0]) == step
        np.testing.assert_allclose(sched[3:4].view(torch.float32).item(), lr, rtol=1e-6)
    np.testing.assert_allclose(pb.cpu().numpy(), pa.cpu().numpy(), rtol=1e-5, atol=1e-7)


def test_coarse_reuse_leaves_the_render_unchanged():
    """Copying the coarse samples' encoding rows (reuse_coarse_rows) and taking their raw rows from the coarse pass while the fine forward
    evaluates the importance samples only (reuse_coarse_raw) change no bit of the fine pass: raw rows, depths and maps — also on rays that
    miss the box, whose fp32 depths are not monotone and get re-ordered by the merge."""
    from nerfpp_b200.pipeline import synthetic_rays
    m = _model()
    o, d, _ = synthetic_rays(300, seed=4)
    o, d = o.clone(), d.clone()
    o[:7] = torch.tensor([3.0, 2.5, -4.0], device=o.device)          # outside the box, looking away: near = far - 1e-6
    d[:7] = torch.tensor([0.3, 0.8, -0.52], device=o.device)
    outs = []
    for rows, raw in ((False, False), (True, False), (True, True)):
        m.reuse_coarse_rows, m.reuse_coarse_raw = rows, raw
        outs.append(m.render_rays(o, d, keep_for_backward=True))
    a = outs[0]
    for b in outs[1:]:
        for k in ("rgb", "depth", "acc", "weights", "z"):
            assert torch.equal(a[k], b[k]), k
        for i, name in ((1, "enc"), (2, "keep"), (3, "raw")):
            assert torch.equal(a["_saved"][i], b["_saved"][i]), name


def test_per_ray_view_term_model_matches_the_view_input_model():
    """HashNeRF(ray_bias=True) at SH degree 4 == the default model (same seed): loss, maps and gradients within the bf16 class."""
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    a = HashNeRF(BBOX, log2_hashmap_size=14, seed=42)
    b = HashNeRF(BBOX, log2_hashmap_size=14, seed=42, ray_bias=True)
    assert torch.equal(a.params, b.params)
    o, d, tgt = synthetic_rays(256, seed=3)
    oa, ob = a.forward_backward(o, d, tgt), b.forward_backward(o, d, tgt)
    np.testing.assert_allclose(float(b.loss), float(a.loss), rtol=2e-3)
    np.testing.assert_allclose(ob["rgb"].cpu().numpy(), oa["rgb"].cpu().numpy(), rtol=1e-2, atol=2e-3)
    ga, gb = a.grads.double(), b.grads.double()
    assert float(ga @ gb / (ga.norm() * gb.norm())) > 0.9995
    w2 = slice(a.n_table + 3072, a.n_table + 3072 + 64 * 31)                 # color_net_0: the layer whose view columns take the other route
    np.testing.assert_allclose(gb[w2].cpu().numpy(), ga[w2].cpu().numpy(), rtol=5e-2, atol=2e-2 * float(ga[w2].abs().max()))


def test_shipped_shape_trains_and_renders():
    """The reference's shipped network shape (src/main.cpp:176-191): SH degree 8 (64 view channels), finest resolution 1024, 64 + 192
    samples.  Loss falls on the fused kernels; the one-call render entry equals the composed path bit for bit at this shape too."""
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    m = HashNeRF(BBOX, log2_hashmap_size=15, finest_resolution=1024, sh_degree=8, n_importance=192, seed=42)
    assert m.ray_bias and m.params.numel() == m.n_table + 9344 + 64 * 48
    o, d, tgt = synthetic_rays(512, seed=1)
    losses = []
    for _ in range(40):
        m.train_step(o, d, tgt)
        losses.append(float(m.loss))
    w2_before = m.mlp_weights()[2].clone()
    assert np.isfinite(losses).all() and losses[-1] < 0.9 * losses[0], (losses[0], losses[-1])
    m.train_step(o, d, tgt)
    moved = (m.mlp_weights()[2] - w2_before).abs().amax(dim=0)               # color_net_0 [64, 64 view + 15 geo columns]
    assert float(moved[:64].min()) > 0 and float(moved[64:].min()) > 0        # the view columns train through the per-ray route
    o2, d2, _ = synthetic_rays(300, seed=6)
    x = m.render_rays(o2, d2)
    y = m.render_rays_fused(o2, d2, want_weights=True, want_z=True)
    for k in ("rgb", "depth", "disp", "acc", "weights", "z"):
        assert torch.equal(x[k], y[k]), k
    m.capture_train_step(512)                                                 # the same step as one CUDA graph keeps training
    for _ in range(5):
        m.train_step_graph(o, d, tgt)
    assert np.isfinite(float(m.loss)) and float(m.loss) <= losses[-1] * 1.05, (float(m.loss), losses[-1])


def test_fused_render_entry_equals_the_composed_path():
    """nrf_render_rays_fwd (one C-ABI call) == the same kernels called one by one, bit for bit, incl. a ragged ray count."""
    from nerfpp_b200.pipeline import synthetic_rays
    m = _model()
    for n, white in ((300, False), (1, True)):
        o, d, _ = synthetic_rays(n, seed=6)
        a = m.render_rays(o, d, white_bkgr=white)
        b = m.render_rays_fused(o, d, white_bkgr=white, want_weights=True, want_z=True)
        for k in ("rgb", "depth", "disp", "acc", "weights", "z"):
            assert torch.equal(a[k], b[k]), k
    c = m.render_rays_fused(o, d, n_importance=64)
    assert c["rgb"].shape == (1, 3)
    # a prepared batch [o d near far viewdirs] (what BatchifyRays hands to RenderRays): same bits; its near / far are taken as given
    from nerfpp_b200 import ops
    o, d, _ = synthetic_rays(300, seed=8)
    rb = ops.rays_prepare(o, d, m.bbox, 0.0, True)
    a = m.render_rays_fused(o, d, want_weights=True, want_z=True)
    b, _ = ops.render_rays_fwd(m.grid, m.table_f16, m.packed, None, None, m.t_vals, m.u, m.bbox, sh_degree=m.sh_degree, want_weights=True, want_z=True,
                               shape=m.mlp_shape, ray_batch=rb)
    for k in ("rgb", "depth", "disp", "acc", "weights", "z"):
        assert torch.equal(a[k], b[k]), k
    rb2 = rb.clone()
    rb2[:, 6] += 0.25                                                           # a caller-chosen near plane
    c, _ = ops.render_rays_fwd(m.grid, m.table_f16, m.packed, None, None, m.t_vals, m.u, m.bbox, sh_degree=m.sh_degree, want_z=True, shape=m.mlp_shape, ray_batch=rb2)
    ok = rb2[:, 6] < rb2[:, 7]                                                  # (a ray whose shifted near passes its far has no ordered depths)
    assert int(ok.sum()) > 100 and torch.equal(c["z"][ok, 0], rb2[ok, 6])


def test_fp16_shadow_is_fully_initialised():
    """The Adam kernels keep the WHOLE fp16 shadow (table + MLP tail) equal to the rounded fp32 masters; refresh() must start it that
    way — the fused multi-GPU optimiser's dry self-test compares the full buffer (it once saw uninitialised memory in the tail and
    fell back to NCCL)."""
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    m = HashNeRF(BBOX, log2_hashmap_size=12, seed=5)
    assert torch.equal(m.shadow, m.params.half())
    o, d, tgt = synthetic_rays(128, seed=2)
    for _ in range(3):
        m.train_step(o, d, tgt)
    assert torch.equal(m.shadow, m.params.half())


def test_device_side_ray_batch_equals_get_rays_and_the_ray_path():
    """SURVEY §8f-3: NeRFDataset::GetRayBatch + the target gather on the device (nrf_ray_batch, nrf_ray_setup_pixels).  (a) the rays of a pixel
    list are the rows of nrf_get_rays at those pixels, bit for bit (that kernel is pinned to the reference's GetRays fixture); (b) against the
    oracle's restatement of GetRayBatch (src/NeRFDataset.cpp:109-144); (c) the fused set-up equals ray_batch + ray_setup bit for bit; (d) a
    training step fed with pixel coordinates follows the step fed with the same rays and targets."""
    import restate as O
    from nerfpp_b200 import ops
    from nerfpp_b200.pipeline import HashNeRF, synthetic_pixels, synthetic_view
    h, w = 60, 80
    K, c2w = synthetic_view(h, w)
    pix = synthetic_pixels(500, h, w, seed=3)
    pix[0] = torch.tensor([0, 0]); pix[1] = torch.tensor([h - 1, w - 1])
    image = torch.rand(h, w, 3, generator=torch.Generator().manual_seed(4)).cuda()
    rays_o, rays_d, target, cone = ops.ray_batch(pix.cuda(), K, c2w, image)
    full_o, full_d = ops.get_rays(h, w, K, c2w)
    idx = (pix[:, 0].long() * w + pix[:, 1].long()).cuda()
    assert torch.equal(rays_d, full_d[idx]) and torch.equal(rays_o, full_o[idx])
    assert torch.equal(target, image[pix[:, 0].long().cuda(), pix[:, 1].long().cuda()])
    ro, rd, ca = O.get_ray_batch(pix[:, 0], pix[:, 1], K, c2w)
    assert torch.allclose(rays_d.cpu(), rd, rtol=1e-6, atol=1e-7) and torch.equal(rays_o.cpu(), ro.expand_as(rd).contiguous())
    assert abs(cone - float(ca)) <= 1e-9
    m = HashNeRF(BBOX, log2_hashmap_size=14, seed=42)
    a = ops.ray_setup(rays_o, rays_d, m.bbox, 0.0, m.t_vals, 4)
    b = ops.ray_setup_pixels(pix.cuda(), K, c2w, image, m.bbox, 0.0, m.t_vals, 4)
    assert torch.equal(b[0], rays_o) and torch.equal(b[1], rays_d) and torch.equal(b[2], target)
    for x, y in zip(a, b[3:]):
        assert torch.equal(x, y)
    # (d) two replicas, same seed: one stepped on (rays, targets), one on pixel coordinates (eagerly and as a captured graph)
    m1, m2, m3 = (HashNeRF(BBOX, log2_hashmap_size=14, seed=42) for _ in range(3))
    for mm in (m2, m3):
        mm.set_camera(image, K, c2w)
    m3.capture_train_step(pix.shape[0], pixels=True)
    l1 = [float(m1.train_step(rays_o, rays_d, target)) for _ in range(4)]
    l2 = [float(m2.train_step(pix.cuda())) for _ in range(4)]
    l3 = [float(m3.train_step_graph(pix.pin_memory())) for _ in range(4)]
    np.testing.assert_allclose(l2, l1, rtol=1e-4)
    np.testing.assert_allclose(l3, l1, rtol=1e-4)


def test_shipped_configuration_step_statistics():
    """The RNG-gated stages of the shipped configuration (cone jitter, stochastic preconditioning + ReflectBoundary, density noise): with all
    amplitudes at 0 (and without TangentScatter's clamp, which pulls the samples of rays that miss the box onto its surface) the step equals the parity
    step; with them on it trains, the jitter stays inside the cone and the box, and the
    reflected points match the oracle's restatement of ReflectBoundary."""
    from nerfpp_b200 import ops
    from nerfpp_b200.pipeline import HashNeRF, synthetic_rays
    o, d, tgt = synthetic_rays(512, seed=5)
    a, b = HashNeRF(BBOX, log2_hashmap_size=15, seed=42), HashNeRF(BBOX, log2_hashmap_size=15, seed=42)
    a.forward_backward(o, d, tgt)
    b.forward_backward_shipped(o, d, tgt, cone_angle=0.0, raw_noise_std=0.0, sp_alpha=0.0, clamp_to_box=False)
    assert abs(float(a.loss) - float(b.loss)) <= 1e-6 * float(a.loss)
    ga, gb = a.grads.clone(), b.grads.clone()
    assert float((ga - gb).abs().max()) <= 1e-4 * float(ga.abs().max())          # same kernels on the same points; atomics order only
    a.grads.zero_(); b.grads.zero_()
    losses = []
    for _ in range(30):
        b.forward_backward_shipped(o, d, tgt, cone_angle=1.0 / 1111.0, raw_noise_std=0.5, sp_alpha=0.02 * 5.196)
        b.optimizer_step()
        losses.append(float(b.loss))
    assert all(np.isfinite(losses)) and np.mean(losses[-5:]) < np.mean(losses[:5])
    # ReflectBoundary against the oracle's restatement (src/NeRFRenderer.h:285-304)
    g = torch.Generator().manual_seed(1)
    pts = (torch.rand(4096, 3, generator=g) * 3 - 1.5)
    noise = torch.randn(4096, 3, generator=g)
    got = ops.precondition_points(pts.clone().cuda(), noise.cuda(), 0.4, BBOX).cpu()
    lo, hi = torch.tensor(BBOX[:3]), torch.tensor(BBOX[3:])
    q = torch.fmod((pts + noise * 0.4 - lo) / (hi - lo), 2.0)
    q = torch.where(q > 1.0, 2.0 - q, q)
    assert torch.allclose(got, q * (hi - lo) + lo, rtol=1e-6, atol=1e-6)
