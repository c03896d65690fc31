"""GPU parity of the assembled path (field, rendering, render_image, render_image_test) against the golden
vectors frozen from the reference's own Python (tests/golden/make_golden.py) and against the oracle.

Tolerances (BASELINE.json north_star): marcher outputs bit-exact; fp16 MLP path <= 2e-3; loss and gradient
relative error <= 1e-3 (measured as ||g - g_ref|| / ||g_ref|| per parameter tensor).
"""
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import cednerf_ref as cr  # noqa: E402
from oracle import nerfacc_ref as nf  # noqa: E402

DEV = "cuda:0"
FIELD_KW = dict(n_levels=8, log2_hashmap_size=12, dst_resolution=256, moving_step=1.0 / 256)
FLAG_SETS = {
    "plain": dict(),
    "te_ta_df": dict(use_time_embedding=True, use_time_attenuation=True, use_div_offsets=True),
    "te_after": dict(use_time_embedding=True, time_inject_before_sigma=False),
}
OPTS = dict(near_plane=0.2, render_step_size=2e-2, cone_angle=0.004, alpha_thre=1e-2)


@pytest.fixture(scope="module")
def cb():
    import cednerf_b200

    return cednerf_b200


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def gpu_scene(cb, golden):
    est = cb.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=16, levels=2).to(DEV)
    est.binaries = golden["scene.binaries"].to(DEV)
    est.occs = golden["scene.occs"].to(DEV)
    assert torch.equal(est.aabbs.cpu(), golden["scene.aabbs"])
    rays = cb.Rays(golden["scene.origins"].to(DEV), golden["scene.dirs"].to(DEV))
    return est, rays, golden["scene.timestamps"].to(DEV)


def gpu_field(cb, golden, name, extra=None):
    field = cb.DNGPradianceField(golden["scene.aabbs"][-1], **FIELD_KW, **FLAG_SETS[name], **(extra or {}))
    sd = {k[len(name) + 7:]: v for k, v in golden.items() if k.startswith(f"{name}.state.")}
    # the golden state dict has the reference's own key set (made by cednerf/model.py): nothing may be left over
    missing = field.load_state_dict(sd, strict=False)
    assert not missing.unexpected_keys and all("prediction" in k for k in missing.missing_keys)
    return field.to(DEV)


@pytest.mark.parametrize("name", list(FLAG_SETS))
def test_field_against_golden(cb, golden, name):
    field = gpu_field(cb, golden, name).train()
    to = lambda k: golden[f"{name}.field.{k}"].to(DEV)
    rgb, res = field(to("pts"), to("t"), to("dirs"))
    assert rgb.dtype == torch.float32 and res["density"].dtype == torch.float32
    torch.testing.assert_close(rgb.detach().cpu(), golden[f"{name}.field.rgb"], rtol=0, atol=2e-3)
    torch.testing.assert_close(res["density"].detach().cpu(), golden[f"{name}.field.density"], rtol=8e-3, atol=2e-3)
    bo = golden[f"{name}.field.base_mlp_out"]
    torch.testing.assert_close(res["base_mlp_out"].detach().float().cpu(), bo, rtol=2e-3, atol=2e-3 * float(bo.abs().max()))
    mv = golden[f"{name}.field.move"]
    torch.testing.assert_close(res["interal_output"]["move"].detach().cpu(), mv, rtol=2e-3, atol=2e-3 * float(mv.abs().max()))
    ((rgb * to("grgb")).sum() + (res["density"] * to("gsig")).sum()).backward()
    for k, got, want in golden.grads(f"{name}.field", field):
        assert rel(got.cpu(), want) < 1e-3, (k, rel(got.cpu(), want))


@pytest.mark.parametrize("name", list(FLAG_SETS))
def test_render_paths_against_golden(cb, golden, name):
    est, rays, ts = gpu_scene(cb, golden)
    field = gpu_field(cb, golden, name)
    bkgd = torch.tensor([0.2, 0.5, 0.8], device=DEV)
    field.train(), est.train()
    torch.manual_seed(123)
    jitter = torch.rand(rays.origins.shape[0])  # the draw the reference's sampling() made under the same seed
    # marcher alone, before visibility filtering: bit-exact against the oracle
    near = torch.full((96,), 0.2) + jitter * 2e-2
    r_ref, a_ref, b_ref, _, _ = nf.traverse_grids(golden["scene.origins"], golden["scene.dirs"], golden["scene.binaries"],
                                                  golden["scene.aabbs"], near, torch.full((96,), 1e10), 2e-2, 0.004,
                                                  packed_only=True)
    r_g, a_g, b_g, _ = est.march(rays.origins, rays.viewdirs, 0.2, 1e10, 2e-2, 0.004, True, jitter)
    assert torch.equal(r_g.cpu(), r_ref) and torch.equal(a_g.cpu(), a_ref) and torch.equal(b_g.cpu(), b_ref)

    rgb, acc, depth, n_s, extra = cb.render_image(field, est, rays, render_bkgd=bkgd, timestamps=ts, jitter=jitter,
                                                  **OPTS)
    assert n_s == int(golden[f"{name}.train.n_samples"])
    for k in ("ray_indices", "t_starts", "t_ends"):
        assert torch.equal(extra[0][k].cpu(), golden[f"{name}.train.{k}"])
    for a, k in ((rgb, "rgb"), (acc, "acc"), (depth, "depth"), (extra[0]["weights"], "weights"),
                 (extra[0]["trans"], "trans"), (extra[0]["alphas"], "alphas")):
        torch.testing.assert_close(a.detach().cpu(), golden[f"{name}.train.{k}"], rtol=0, atol=2e-3)
    # sigma = exp(logit - 1) with an fp16 logit: one fp16 ulp of a logit in [4, 8) is 2^-8 = 3.9e-3 relative
    torch.testing.assert_close(extra[0]["sigmas"].detach().cpu(), golden[f"{name}.train.sigmas"], rtol=8e-3, atol=2e-3)
    loss = torch.nn.functional.mse_loss(rgb, golden[f"{name}.train.pixels"].to(DEV))
    (loss * 1024.0).backward()
    assert abs(float(loss.detach()) - float(golden[f"{name}.train.loss"])) <= 1e-3 * float(golden[f"{name}.train.loss"])
    for k, got, want in golden.grads(f"{name}.train", field):
        # Deformation net: on this 96-ray batch ONE hidden activation of its third layer sits at 3.5e-5 (an fp16
        # subnormal); a 1-ulp fp16 difference in one of its 64 inputs (tensor-core vs CPU fp32 summation order)
        # moves the pre-activation across zero, the ReLU mask of that unit flips, and that single element is
        # 2.4e-3 of the gradient norm (measured; independent of the loss scale).  Every other tensor holds 1e-3.
        tol = 5e-3 if k.startswith("xyz_wrap") else 1e-3
        assert rel(got.cpu(), want) < tol, (k, rel(got.cpu(), want))

    field.eval(), est.eval()
    t_frame = torch.tensor([[0.5]], device=DEV)
    with torch.no_grad():
        rgb, acc, depth, n_s, _ = cb.render_image(field, est, rays, render_bkgd=bkgd, timestamps=t_frame,
                                                  test_chunk_size=40, **OPTS)
    assert n_s == int(golden[f"{name}.eval.n_samples"])
    for a, k in ((rgb, "rgb"), (acc, "acc"), (depth, "depth")):
        torch.testing.assert_close(a.cpu(), golden[f"{name}.eval.{k}"], rtol=0, atol=2e-3)
    rgb, acc, depth, n_s = cb.render_image_test(64, field, est, rays, render_bkgd=bkgd, timestamps=t_frame, **OPTS)
    assert n_s == int(golden[f"{name}.test.n_samples"])
    for a, k in ((rgb, "rgb"), (acc, "acc"), (depth, "depth")):
        torch.testing.assert_close(a.cpu(), golden[f"{name}.test.{k}"], rtol=0, atol=2e-3)


def test_predictor_flags_against_oracle(cb, golden):
    """-f / -w heads (cednerf/model.py:312-344, cednerf/render.py:101-124): no golden, compare with the oracle."""
    flags = dict(use_time_embedding=True, use_time_attenuation=True, use_div_offsets=True, use_feat_predict=True,
                 use_weight_predict=True)
    ref = cr.DNGPradianceField(golden["scene.aabbs"][-1], **FIELD_KW, **flags).train()
    with torch.no_grad():
        ref.hash_encoder.params.mul_(5000.0)
        ref.mlp_base.params.mul_(3.0)
    field = cb.DNGPradianceField(golden["scene.aabbs"][-1], **FIELD_KW, **flags)
    field.load_state_dict(ref.state_dict())
    field = field.to(DEV).train()
    est, rays, ts = gpu_scene(cb, golden)
    est.train()
    est_ref = nf.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=16, levels=2).train()
    est_ref.binaries, est_ref.occs = golden["scene.binaries"], golden["scene.occs"]
    jitter = torch.rand(96, generator=torch.Generator().manual_seed(3))
    bk = torch.tensor([0.1, 0.2, 0.3])
    rays_ref = cr.Rays(golden["scene.origins"], golden["scene.dirs"])
    out_ref = cr.render_image(ref, est_ref, rays_ref, render_bkgd=bk, timestamps=golden["scene.timestamps"],
                              jitter=jitter, **OPTS)
    out = cb.render_image(field, est, rays, render_bkgd=bk.to(DEV), timestamps=ts, jitter=jitter, **OPTS)
    assert out[3] == out_ref[3]

    def total(o):
        ex = o[4][0]
        return (o[0] ** 2).mean() + ex["latent_losses"].mean() + ex["weight_losses"].mean()

    for k in ("latent_losses", "weight_losses"):
        a, b = out[4][0][k].detach().cpu(), out_ref[4][0][k].detach()
        torch.testing.assert_close(a, b, rtol=5e-3, atol=2e-3 * float(b.abs().max()))
    (total(out_ref) * 1024).backward()
    (total(out) * 1024).backward()
    for (k, p), (_, q) in zip(field.named_parameters(), ref.named_parameters()):
        if q.grad is not None and q.numel():
            assert rel(p.grad.cpu(), q.grad) < 2e-3, (k, rel(p.grad.cpu(), q.grad))


def test_estimator_update_matches_oracle(cb, golden):
    """OccGridEstimator._update (SURVEY A.2) with shared random draws: occs close, binaries equal."""
    est_ref = nf.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=16, levels=2).train()
    est = cb.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=16, levels=2).to(DEV).train()

    def occ_fn(x):  # smooth analytic density, identical on both sides
        return torch.exp(-4.0 * (x ** 2).sum(-1, keepdim=True)) * 0.05

    for step in (0, 16, 256, 272):
        # same starting state on both sides (the rule for duplicate cells differs, see below)
        est.occs.copy_(est_ref.occs.to(DEV))
        est.binaries = est_ref.binaries.to(DEV)
        before, binaries_before = est_ref.occs.clone(), est_ref.binaries.clone()
        est_ref.update_every_n_steps(step, occ_fn, occ_thre=1e-2, rng=nf.HostRng(step))
        est.update_every_n_steps(step, occ_fn, occ_thre=1e-2, rng=nf.HostRng(step, device=DEV))
        got, want = est.occs.cpu(), est_ref.occs
        if step < 256:  # warm-up: every cell exactly once
            torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-8)
            assert int((est.binaries.cpu() != est_ref.binaries).sum()) <= 2  # threshold ties only
        else:
            # the same update with the oracle resolving duplicate cells the way the product does (largest candidate):
            # every cell agrees, as in the warm-up
            est_max = nf.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=16, levels=2).train()
            est_max.occs, est_max.binaries, est_max.duplicate_rule = before.clone(), binaries_before.clone(), "max"
            est_max.update_every_n_steps(step, occ_fn, occ_thre=1e-2, rng=nf.HostRng(step))
            torch.testing.assert_close(got, est_max.occs, rtol=1e-5, atol=1e-8)
            assert int((est.binaries.cpu() != est_max.binaries).sum()) <= 2
            # cells drawn more than once: the oracle keeps the last candidate (CPU index_put), the product the
            # largest (nerfacc on CUDA: undefined).  Both are candidates, so got >= want, and most cells agree.
            assert bool((got >= want - 1e-7).all()) and bool((got >= before * 0.95 - 1e-7).all())
            assert float(((got - want).abs() > 1e-6).float().mean()) < 0.05
    assert int(est.binaries.sum()) > 0
    # the bit field used by the marcher follows the update
    from cednerf_b200.nerfacc.grid import occupancy_bits

    assert torch.equal(occupancy_bits(est.binaries), cb.ops.pack_occupancy(est.binaries))
    sd = est.state_dict()
    assert set(sd) == {"resolution", "aabbs", "occs", "binaries"}


@pytest.mark.parametrize("name", list(FLAG_SETS))
def test_fused_field_query_matches_modular_path(cb, golden, name):
    """cednerf_field_fwd (one kernel, no autograd) against the op-by-op path on the same points and on packed samples."""
    field = gpu_field(cb, golden, name).eval()
    assert field.fused_supported()
    g = torch.Generator().manual_seed(11)
    n = 1000
    pts = ((torch.rand(n, 3, generator=g) * 2 - 1) * 1.3).to(DEV)
    tt = torch.rand(n, 1, generator=g).to(DEV)
    dd = torch.nn.functional.normalize(torch.randn(n, 3, generator=g), dim=-1).to(DEV)
    with torch.enable_grad():
        rgb_m, res_m = field(pts, tt, dd)                      # modular (autograd-capable) path
    with torch.no_grad():
        sig_f = field.query_density(pts, tt)["density"]        # fused, explicit points
        sig2, rgb_f = field.fused_query(n, points=(pts, dd), timestamps=tt.view(-1), t_stride=1, sigma_only=False)
    torch.testing.assert_close(sig_f, res_m["density"].detach(), rtol=8e-3, atol=2e-3)
    torch.testing.assert_close(sig2[:, None], sig_f, rtol=0, atol=0)
    torch.testing.assert_close(rgb_f, rgb_m.detach(), rtol=0, atol=2e-3)
    # packed-sample entry: positions are formed in the kernel exactly as cednerf/utils.py:74-104 forms them
    o = ((torch.rand(50, 3, generator=g) - 0.5)).to(DEV)
    d = torch.nn.functional.normalize(torch.randn(50, 3, generator=g), dim=-1).to(DEV)
    ridx = torch.sort(torch.randint(0, 50, (n,), generator=g))[0].to(DEV)
    t0 = torch.rand(n, generator=g).to(DEV)
    t1 = t0 + 0.01
    ts_ray = torch.rand(50, 1, generator=g).to(DEV)
    x = o[ridx] + d[ridx] * (t0 + t1)[:, None] / 2.0
    with torch.no_grad():
        s_pts, c_pts = field.fused_query(n, points=(x, d[ridx]), timestamps=ts_ray[ridx].view(-1), t_stride=1,
                                         sigma_only=False)
        s_pk, c_pk = field.fused_query(n, packed=(ridx, t0, t1, o, d), timestamps=ts_ray, t_stride=1, sigma_only=False)
        s_one, _ = field.fused_query(n, packed=(ridx, t0, t1, o, d), timestamps=ts_ray[:1], t_stride=0)
        s_ref, _ = field.fused_query(n, points=(x, None), timestamps=ts_ray[:1].expand(n, 1).contiguous().view(-1))
    assert torch.equal(s_pk, s_pts) and torch.equal(c_pk, c_pts) and torch.equal(s_one, s_ref)


@pytest.mark.parametrize("name,extra", [("plain", {}), ("te_ta_df", {}), ("te_after", {}),
                                        ("te_ta_df", {"use_feat_predict": True})])
def test_fused_training_path_matches_op_by_op_path(cb, golden, name, extra):
    """cednerf_field_train_fwd/bwd (5-7 launches) against the op-by-op autograd path on the same packed samples."""
    kw = dict(FIELD_KW)
    if extra.get("use_feat_predict"):
        kw.update(n_levels=16, log2_hashmap_size=14, dst_resolution=512)  # the predictor regresses 16 x 2 features
    field = cb.DNGPradianceField(golden["scene.aabbs"][-1], **kw, **FLAG_SETS[name], **extra)
    with torch.no_grad():
        field.hash_encoder.params.mul_(5000.0)
        field.mlp_base.params.mul_(3.0)
    field = field.to(DEV).train()
    assert field.fused_train_supported()
    g = torch.Generator().manual_seed(21)
    n_rays, n = 64, 1500
    o = (torch.tensor([0.0, 0.0, -3.0]) + (torch.rand(n_rays, 3, generator=g) - 0.5) * 0.4).to(DEV)
    d = torch.nn.functional.normalize(torch.randn(n_rays, 3, generator=g) * 0.2 + torch.tensor([0.0, 0.0, 1.0]), dim=-1).to(DEV)
    ridx = torch.sort(torch.randint(0, n_rays, (n,), generator=g))[0].to(DEV)
    t0 = (1.5 + torch.rand(n, generator=g) * 3).to(DEV)
    t1 = t0 + 0.02
    ts = torch.rand(n_rays, 1, generator=g).to(DEV)
    g_rgb, g_sig = torch.rand(n, 3, generator=g).to(DEV), torch.rand(n, 1, generator=g).to(DEV)
    g_lat = torch.rand(n, 32, generator=g).to(DEV) * 0.1

    def loss_of(rgb, res):
        l = (rgb * g_rgb).sum() + (res["density"] * g_sig).sum()
        if "latent_losses" in res["interal_output"]:
            l = l + (res["interal_output"]["latent_losses"] * g_lat).sum()
        return l * 64.0

    x = o[ridx] + d[ridx] * (t0 + t1)[:, None] / 2.0
    rgb_m, res_m = field(x, ts[ridx], d[ridx])
    field.zero_grad()
    loss_of(rgb_m, res_m).backward()
    grads_m = {k: p.grad.clone() for k, p in field.named_parameters() if p.grad is not None and p.numel()}
    rgb_f, res_f = field.fused_train(ridx, t0, t1, o, d, ts, 1)
    field.zero_grad()
    loss_of(rgb_f, res_f).backward()
    torch.testing.assert_close(rgb_f, rgb_m, rtol=0, atol=2e-3)
    torch.testing.assert_close(res_f["density"], res_m["density"], rtol=8e-3, atol=2e-3)
    mv_f, mv_m = res_f["interal_output"]["move"], res_m["interal_output"]["move"]
    torch.testing.assert_close(mv_f, mv_m, rtol=2e-3, atol=2e-3 * float(mv_m.abs().max()))
    if extra.get("use_feat_predict"):
        lf, lm = res_f["interal_output"]["latent_losses"], res_m["interal_output"]["latent_losses"]
        torch.testing.assert_close(lf, lm, rtol=1e-2, atol=2e-3 * float(lm.abs().max()))
        assert torch.equal(res_f["interal_output"]["selector"], res_m["interal_output"]["selector"])
    for k, p in field.named_parameters():
        if k in grads_m:
            assert p.grad is not None, k
            assert rel(p.grad, grads_m[k]) < 5e-3, (k, rel(p.grad, grads_m[k]))


def test_device_count_sampling_matches_the_host_count_path(cb):
    """render_image(..., device_counts=True): capacity-sized sample tensors whose live count never leaves the device must
    give the same rendering, loss and gradients as the default path (which reads the totals back, like the reference)."""
    from cednerf_b200 import workload as w

    cfg = w.TINY
    rk = w.render_kwargs(cfg)
    est, field = w.build_scene(cfg, DEV, cb, seed=42)
    est.train(), field.train()
    b = {k: v.to(DEV) for k, v in w.draw_batch(cfg, 70000, torch.Generator().manual_seed(3)).items()}
    rays = cb.Rays(b["origins"], b["viewdirs"])

    def run(device_counts):
        for p in field.parameters():
            p.grad = None
        rgb, acc, depth, n_s, extra = cb.render_image(field, est, rays, render_bkgd=b["color_bkgd"], timestamps=b["timestamps"],
                                                      jitter=b["jitter"], device_counts=device_counts, **rk)
        loss = cb.losses.training_loss(rgb, acc, b["pixels"], extra, acc_entropy_loss=True, weight_rgbper=True,
                                       use_feat_predict=True)
        (loss * 1024.0).backward()
        grads = {k: p.grad.detach().clone() for k, p in field.named_parameters() if p.grad is not None}
        return rgb.detach(), acc.detach(), depth.detach(), n_s, extra[0], float(loss), grads

    ref = run(False)
    assert isinstance(ref[3], int) and ref[3] > 50000
    first = run(True)            # no capacity known yet: falls back to the host-count path and seeds the capacities
    assert isinstance(first[3], int) and first[3] == ref[3]
    got = run(True)
    assert torch.is_tensor(got[3]) and got[3].is_cuda and int(got[3]) == ref[3] and est.dropped_samples == 0
    n = ref[3]
    ex, ex_ref = got[4], ref[4]
    assert ex["t_starts"].numel() > n                      # allocated at a capacity with headroom ...
    for k in ("ray_indices", "t_starts", "t_ends"):        # ... whose live prefix is the default path's sample set
        assert torch.equal(ex[k][:n], ex_ref[k])
    for i in range(3):
        assert torch.equal(got[i], ref[i])
    assert torch.equal(ex["weights"][:n], ex_ref["weights"]) and torch.equal(ex["rgbs"][:n], ex_ref["rgbs"])
    assert abs(got[5] - ref[5]) <= 1e-6 * abs(ref[5])
    for k, g in ref[6].items():
        assert rel(got[6][k], g) <= 2e-6, (k, rel(got[6][k], g))
    # a capacity that is too small drops the tail of the batch and says so
    est._cap_state["visible"]["last"] = n // 4
    est._cap_state["visible"]["pending"].clear()
    short = run(True)
    torch.cuda.synchronize()
    est._capacity("visible")
    assert int(short[3]) < n and est.dropped_samples > 0


def test_device_resident_render_rounds_match_the_host_driven_loop(cb, monkeypatch):
    """render_image_test with the alive list / per-round k / termination test on the device against the loop that reads
    `alive.sum()` back every round (cednerf/utils.py:231): same image, same sample total - per ray the two paths do the
    same arithmetic on the same samples, only the packing order of the rays inside a round differs.  The last input is a
    checkerboard occupancy with a run limit of 1: every ray with more than one run takes the full-march fallback fill."""
    from cednerf_b200 import ops, utils as U, workload as w

    for cfg, opengl, checker in ((w.TINY, False, False), (w.DNERF, True, False), (w.TINY, False, True)):
        rk = w.render_kwargs(cfg)
        est, field = w.build_scene(cfg, DEV, cb, seed=42)
        est.eval(), field.eval()
        if checker:
            i = torch.arange(cfg.occ_res, device=DEV)
            cells = ((i[:, None, None] + i[None, :, None] + i[None, None, :]) % 2) == 0
            est.binaries = cells[None].expand_as(est.binaries).contiguous()
            monkeypatch.setattr(ops.MarchInputs, "RUN_CAP", 1)
        pose = w.orbit_pose(4.0, 0.3) if opengl else w.spiral_poses(cfg, 8)[3]
        o, d = w.pose_rays(cfg, pose, opengl, DEV)
        if cfg is w.DNERF:   # a 96 x 128 window of the 800 x 800 frame
            sel = (torch.arange(352, 448, device=DEV)[:, None] * cfg.width + torch.arange(336, 464, device=DEV)[None, :]).reshape(-1)
            o, d = o[sel].contiguous(), d[sel].contiguous()
        rays = cb.Rays(o, d)
        t = torch.tensor([[0.37]], device=DEV)
        bk = torch.tensor([0.1, 0.6, 0.9], device=DEV)
        outs = {}
        for mode in (True, False):
            U._DEVICE_ROUNDS = mode
            try:
                outs[mode] = cb.render_image_test(1024, field, est, rays, render_bkgd=bk, timestamps=t, **rk)
            finally:
                U._DEVICE_ROUNDS = True
        assert outs[True][3] == outs[False][3] and outs[True][3] > 1000, (cfg.name, outs[True][3], outs[False][3])
        for i in range(3):   # (the lane group per ray is picked differently: shuffle-scan order, i.e. fp32 rounding, differs)
            torch.testing.assert_close(outs[True][i], outs[False][i], rtol=0, atol=2e-6)


def test_fused_occupancy_update_matches_the_op_by_op_update(cb):
    """OccGridEstimator._update with a FieldOccEval (one launch per level: cell -> jittered point -> field -> EMA-max,
    cednerf_occ_update_level) against the same update driven by a plain closure (element-wise torch glue around the
    fused density kernel), draws shared through seeded generators: bit-identical occs and binaries, in the warm-up
    (every cell once) and afterwards (uniform + occupied draws with duplicate cells)."""
    from cednerf_b200 import dp, workload as w

    cfg = w.TINY
    rk = w.render_kwargs(cfg)
    _, field = w.build_scene(cfg, DEV, cb, seed=42)
    field.eval()
    ests = [cb.OccGridEstimator(list(cfg.roi_aabb), resolution=cfg.occ_res, levels=cfg.occ_levels).to(DEV).train()
            for _ in range(2)]
    rng_a, rng_b = dp.SharedRng(99, DEV), dp.SharedRng(99, DEV)
    fused_fn = cb.utils.FieldOccEval(field, rk["render_step_size"], rng=rng_a)

    def plain_fn(x):   # what train_real.py:324-328 writes
        return field.query_density(x, rng_b.rand(x.shape[0], 1))["density"] * rk["render_step_size"]

    launches = []
    for step in (0, 16, 32, 256, 272, 288):
        l0 = cb._lib.launch_count()
        ests[0].update_every_n_steps(step, fused_fn, occ_thre=1e-2, rng=rng_a)
        launches.append(cb._lib.launch_count() - l0)
        ests[1].update_every_n_steps(step, plain_fn, occ_thre=1e-2, rng=rng_b)
        assert torch.equal(ests[0].occs, ests[1].occs), step
        assert torch.equal(ests[0].binaries, ests[1].binaries), step
    assert bool(ests[0].binaries.any()) and float(ests[0].occs.max()) > 0
    assert launches[1] == cfg.occ_levels + 1          # one fused launch per level + threshold / pack (images cached)
    # the reference's calling convention still works with the object
    x = torch.rand(100, 3, device=DEV)
    assert fused_fn(x).shape == (100, 1)


def test_interleaved_frames_match_frame_by_frame_rendering(cb):
    """render_images_test (marching rounds of several frames interleaved on separate streams) returns, frame by frame,
    what render_image_test returns."""
    from cednerf_b200 import workload as w

    cfg = w.TINY
    rk = w.render_kwargs(cfg)
    est, field = w.build_scene(cfg, DEV, cb, seed=42)
    est.eval(), field.eval()
    poses = w.spiral_poses(cfg, 5)
    K = [[cfg.focal, 0.0, cfg.width / 2], [0.0, cfg.focal, cfg.height / 2], [0.0, 0.0, 1.0]]
    bk = torch.tensor([0.2, 0.4, 0.6], device=DEV)
    ts = [torch.tensor([[k / 5.0]], device=DEV) for k in range(5)]
    want = [cb.render_image_test(1024, field, est, cb.utils.generate_rays(K, poses[k].to(DEV), cfg.width, cfg.height),
                                 render_bkgd=bk, timestamps=ts[k], **rk) for k in range(5)]
    rays = [(lambda k=k: cb.utils.generate_rays(K, poses[k].to(DEV), cfg.width, cfg.height)) for k in range(5)]
    for conc in (1, 2, 3):
        got = cb.render_images_test(1024, field, est, rays, ts, concurrency=conc, render_bkgd=bk, **rk)
        torch.cuda.synchronize()
        for k in range(5):
            assert got[k][3] == want[k][3] and got[k][3] > 0
            for i in range(3):
                assert torch.equal(got[k][i], want[k][i]), (conc, k, i)
    seen = []
    cb.render_images_test(1024, field, est, rays, ts, concurrency=2, render_bkgd=bk,
                          on_frame=lambda idx, res: seen.append((idx, res[3])), **rk)
    assert sorted(seen) == [(k, want[k][3]) for k in range(5)]


def test_spatial_bucket_order_changes_nothing_but_the_walk(cb):
    """cednerf_sample_order + the `sample_order` indirection of the fused training kernels: the same batch walked in
    spatial buckets gives bit-identical per-sample outputs (every sample is computed independently) and gradients equal up
    to fp32 summation order; the order is a permutation, deterministic, and identity on the unused tail of a
    capacity-sized array.  Both the host-count and the device-count (capacity) paths."""
    from cednerf_b200 import workload as w, ops

    cfg = w.TINY
    rk = w.render_kwargs(cfg)
    est, field = w.build_scene(cfg, DEV, cb, seed=42)
    est.train(), field.train()
    b = {k: v.to(DEV) for k, v in w.draw_batch(cfg, 70000, torch.Generator().manual_seed(5)).items()}
    rays = cb.Rays(b["origins"], b["viewdirs"])

    def run(order_min, device_counts):
        old, ops.SAMPLE_ORDER_MIN = ops.SAMPLE_ORDER_MIN, order_min
        try:
            for p in field.parameters():
                p.grad = None
            rgb, acc, depth, n_s, extra = cb.render_image(field, est, rays, render_bkgd=b["color_bkgd"],
                                                          timestamps=b["timestamps"], jitter=b["jitter"],
                                                          device_counts=device_counts, **rk)
            loss = cb.losses.training_loss(rgb, acc, b["pixels"], extra, acc_entropy_loss=True, weight_rgbper=True,
                                           use_feat_predict=True)
            (loss * 1024.0).backward()
            grads = {k: p.grad.detach().clone() for k, p in field.named_parameters() if p.grad is not None}
            return rgb.detach(), extra[0], int(n_s), float(loss), grads
        finally:
            ops.SAMPLE_ORDER_MIN = old

    plain = run(None, False)
    n = plain[2]
    assert n > 20000
    for dc in (False, True, True):   # the first device-count call seeds the capacities through the host-count path
        got = run(1, dc)
        assert got[2] == n and torch.equal(got[0], plain[0])
        for k in ("rgbs", "sigmas", "weights", "latent_losses"):
            if k in plain[1] and torch.is_tensor(plain[1][k]):
                assert torch.equal(got[1][k][:n] if got[1][k].shape[0] >= n and k != "latent_losses" else got[1][k],
                                   plain[1][k]), k
        assert abs(got[3] - plain[3]) <= 1e-6 * abs(plain[3])
        for k, g in plain[4].items():
            assert rel(got[4][k], g) <= 1e-5, (k, rel(got[4][k], g))
    again = run(1, True)
    for k, g in got[4].items():      # deterministic: the walk is a pure function of the inputs
        assert rel(again[4][k], g) <= 2e-6, (k, rel(again[4][k], g))

    # the order itself
    ex = plain[1]
    ridx, t0, t1 = ex["ray_indices"], ex["t_starts"], ex["t_ends"]
    cap = n + 1000
    ridx_p, t0_p, t1_p = (torch.cat([t, t.new_zeros(cap - n)]) for t in (ridx, t0, t1))   # bound: they outlive the launches
    o_c, d_c = rays.origins.contiguous(), rays.viewdirs.contiguous()
    n_dev = torch.tensor([n], dtype=torch.int64, device=DEV)
    lib = cb._lib.load()
    orders = []
    for _ in range(2):
        order = torch.full((cap,), -1, dtype=torch.int32, device=DEV)
        ws = torch.empty(int(lib.cednerf_sample_order_workspace_bytes(cap)), dtype=torch.uint8, device=DEV)
        cb._lib.call("cednerf_sample_order", cb._lib.ptr(ridx_p), cb._lib.ptr(t0_p), cb._lib.ptr(t1_p),
                     cb._lib.ptr(o_c), cb._lib.ptr(d_c), cap, cb._lib.ptr(n_dev),
                     -1.0, -1.0, -1.0, 1.0, 1.0, 1.0, cb._lib.ptr(ws), cb._lib.ptr(order), cb._lib.stream())
        orders.append(order.cpu().long())
    o = orders[0]
    assert torch.equal(orders[0], orders[1])
    assert torch.equal(torch.sort(o[:n])[0], torch.arange(n)) and torch.equal(o[n:], torch.arange(n, cap))
    x = (rays.origins[ridx] + rays.viewdirs[ridx] * ((t0 + t1) / 2)[:, None]).cpu()
    q = ((x + 1.0) / 2.0 * 128).clamp(0, 127).long()

    def spread(v):
        out = torch.zeros_like(v)
        for i in range(7):
            out |= ((v >> i) & 1) << (3 * i)
        return out

    key = spread(q[:, 0]) | (spread(q[:, 1]) << 1) | (spread(q[:, 2]) << 2)
    walked = key[o[:n]]
    # samples on a bucket boundary may fall either side (the kernel multiplies by 128 / extent, this check divides): the
    # walk is sorted by key except for such samples
    assert float((walked[1:] < walked[:-1]).float().mean()) < 1e-3
    same = walked[1:] == walked[:-1]
    assert bool((o[:n][1:][same] > o[:n][:-1][same]).all())      # ascending sample index inside a bucket
