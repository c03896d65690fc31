"""Oracle vs the frozen outputs of the reference's own in-tree Python (tests/golden/make_golden.py)."""
import math

import pytest
import torch

from oracle import cednerf_ref as cr
from oracle import nerfacc_ref as nf

FIELD_KW = dict(n_levels=8, log2_hashmap_size=12, dst_resolution=256, moving_step=1.0 / 256)
FLAG_SETS = {
    "plain": dict(),
    "te_ta_df": dict(use_time_embedding=True, use_time_attenuation=True, use_div_offsets=True),
    "te_after": dict(use_time_embedding=True, time_inject_before_sigma=False),
}


@pytest.fixture(autouse=True)
def golden_thread_count():
    """The CPU kernels split their float32 sums by the intra-op thread count, and gradient entries that nearly cancel move
    by more than atol under another split.  The reference ran with 8 threads, so the oracle does too, on any host."""
    n = torch.get_num_threads()
    torch.set_num_threads(8)
    yield
    torch.set_num_threads(n)


def scene(golden):
    est = nf.OccGridEstimator([-1.0, -1.0, -1.0, 1.0, 1.0, 1.0], resolution=16, levels=2)
    est.binaries, est.occs = golden["scene.binaries"], golden["scene.occs"]
    assert torch.equal(est.aabbs, golden["scene.aabbs"])
    return est, cr.Rays(golden["scene.origins"], golden["scene.dirs"]), golden["scene.timestamps"]


def load_field(golden, name):
    est, _, _ = scene(golden)
    field = cr.DNGPradianceField(est.aabbs[-1], **FIELD_KW, **FLAG_SETS[name])
    sd = {k[len(name) + 7:]: v for k, v in golden.items() if k.startswith(f"{name}.state.")}
    field.load_state_dict(sd)  # strict: the reference's exact key set
    return field


def test_time_encoders(golden):
    assert torch.equal(cr.time_embed(golden["enc.t"]), golden["enc.sin"])
    torch.testing.assert_close(cr.time_embed_attenuated(golden["enc.t"], golden["enc.move"]), golden["enc.sinexp"],
                               rtol=0, atol=1e-7)


def test_trunc_exp(golden):
    x = golden["texp.x"].clone().requires_grad_(True)
    y = cr.trunc_exp(x)
    y.backward(golden["texp.gy"])
    assert torch.equal(y.detach(), golden["texp.y"]) and torch.equal(x.grad, golden["texp.gx"])


def test_rendering_closed_form(golden):
    sig = golden["rend.sigma"].clone().requires_grad_(True)
    col = golden["rend.rgb"].clone().requires_grad_(True)
    c, o, d, ex = cr.rendering(golden["rend.t0"], golden["rend.t1"], golden["rend.ridx"], 6,
                               lambda a, b, r: (col, {"density": sig[:, None]}), torch.ones(3))
    ((c * golden["rend.gc"]).sum() + (o * golden["rend.go"]).sum() + (d * golden["rend.gd"]).sum()).backward()
    for a, b in ((c, "colors"), (o, "opac"), (d, "depth"), (ex["weights"], "weights"), (ex["trans"], "trans"),
                 (sig.grad, "gsigma"), (col.grad, "grgb")):
        torch.testing.assert_close(a.detach(), golden[f"rend.{b}"], rtol=1e-6, atol=1e-7)
    # independent closed form for ray 0
    s, dt = golden["rend.sigma"][:3].double(), 0.1
    T = torch.exp(-torch.cumsum(torch.cat([torch.zeros(1, dtype=torch.float64), s[:-1] * dt]), 0))
    w = T * (1 - torch.exp(-s * dt))
    torch.testing.assert_close(ex["weights"][:3].double().detach(), w, rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("name", list(FLAG_SETS))
def test_field_forward_backward(golden, name):
    field = load_field(golden, name).train()
    rgb, res = field(golden[f"{name}.field.pts"], golden[f"{name}.field.t"], golden[f"{name}.field.dirs"])
    assert torch.equal(rgb.detach(), golden[f"{name}.field.rgb"])
    assert torch.equal(res["density"].detach(), golden[f"{name}.field.density"])
    assert torch.equal(res["base_mlp_out"].detach(), golden[f"{name}.field.base_mlp_out"])
    assert torch.equal(res["interal_output"]["move"].detach(), golden[f"{name}.field.move"])
    ((rgb * golden[f"{name}.field.grgb"]).sum() + (res["density"] * golden[f"{name}.field.gsig"]).sum()).backward()
    for k, got, want in golden.grads(f"{name}.field", field):
        torch.testing.assert_close(got, want, rtol=1e-5, atol=1e-9)


@pytest.mark.parametrize("name", list(FLAG_SETS))
def test_render_paths(golden, name):
    est, rays, ts = scene(golden)
    field = load_field(golden, name)
    opts = dict(near_plane=0.2, render_step_size=2e-2, cone_angle=0.004, alpha_thre=1e-2)
    bkgd = torch.tensor([0.2, 0.5, 0.8])
    field.train(), est.train()
    torch.manual_seed(123)
    rgb, acc, depth, n_s, extra = cr.render_image(field, est, rays, render_bkgd=bkgd, timestamps=ts, **opts)
    assert n_s == int(golden[f"{name}.train.n_samples"]) and n_s > 200
    for k in ("ray_indices", "t_starts", "t_ends"):
        assert torch.equal(extra[0][k], golden[f"{name}.train.{k}"])
    for a, k in ((rgb, "rgb"), (acc, "acc"), (depth, "depth"), (extra[0]["weights"], "weights"),
                 (extra[0]["sigmas"], "sigmas")):
        torch.testing.assert_close(a.detach(), golden[f"{name}.train.{k}"], rtol=1e-6, atol=1e-7)
    loss = torch.nn.functional.mse_loss(rgb, golden[f"{name}.train.pixels"])
    (loss * 1024.0).backward()
    torch.testing.assert_close(loss.detach(), golden[f"{name}.train.loss"], rtol=1e-6, atol=0)
    for k, got, want in golden.grads(f"{name}.train", field):
        torch.testing.assert_close(got, want, rtol=1e-4, atol=1e-9)
    field.eval(), est.eval()
    t_frame = torch.tensor([[0.5]])
    with torch.no_grad():
        rgb, acc, depth, n_s, _ = cr.render_image(field, est, rays, render_bkgd=bkgd, timestamps=t_frame,
                                                  test_chunk_size=40, **opts)
    assert n_s == int(golden[f"{name}.eval.n_samples"])
    for a, k in ((rgb, "rgb"), (acc, "acc"), (depth, "depth")):
        torch.testing.assert_close(a, golden[f"{name}.eval.{k}"], rtol=1e-6, atol=1e-7)
    rgb, acc, depth, n_s = cr.render_image_test(64, field, est, rays, render_bkgd=bkgd, timestamps=t_frame, **opts)
    assert n_s == int(golden[f"{name}.test.n_samples"]) and n_s > 100
    for a, k in ((rgb, "rgb"), (acc, "acc"), (depth, "depth")):
        torch.testing.assert_close(a, golden[f"{name}.test.{k}"], rtol=1e-6, atol=1e-7)
    assert float(acc.max()) > 0.5  # the synthetic density really occludes


def test_distortion_restatement_against_its_definition():
    """torch_efficient_distloss is not vendored: the O(N) restatement is pinned to the loss it implements (Mip-NeRF 360
    eq. 15, the O(N^2) double sum) on random packed samples with sorted mid-points, value and gradient."""
    g = torch.Generator().manual_seed(4)
    counts = torch.randint(0, 9, (40,), generator=g)
    counts[-3:] = 0                                    # trailing empty rays: n_rays of the loss = last ray with samples + 1
    ray_ids = torch.repeat_interleave(torch.arange(40), counts)
    n = ray_ids.numel()
    dt = torch.rand(n, generator=g) * 0.1 + 0.01
    t0 = torch.zeros(n)
    for r in range(40):   # consecutive, sorted intervals inside every ray
        k = torch.nonzero(ray_ids == r).flatten()
        if k.numel():
            t0[k] = 0.3 + torch.cumsum(dt[k], 0) - dt[k]
    t1 = t0 + dt * 0.8
    w = torch.rand(n, generator=g).double().requires_grad_(True)
    a = cr.distortion(ray_ids, w, t0, t1)
    (ga,) = torch.autograd.grad(a, w)
    w2 = w.detach().clone().requires_grad_(True)
    b = cr.distortion_bruteforce(ray_ids, w2, t0, t1)
    (gb,) = torch.autograd.grad(b, w2)
    torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-14)
    torch.testing.assert_close(ga, gb, rtol=1e-10, atol=1e-13)


def test_multinomial_restatement_is_torch_multinomial():
    """oracle/dataset_ref.py states torch.multinomial(w, k) without replacement as topk(w / Exp(1) draws, k): pinned here
    to torch.multinomial ITSELF under the same generator state (ATen's implementation runs on the CPU in this container),
    and the fetch_data restatement to the reference's index arithmetic on a hand-checked case."""
    from oracle import dataset_ref as dr

    for seed, n, k in ((0, 1000, 64), (1, 50000, 4096), (2, 17, 17)):
        w = torch.rand(n, generator=torch.Generator().manual_seed(100 + seed)) ** 4
        w[::7] = 0.0 if k < n else w[::7]
        want = torch.multinomial(w, k, generator=torch.Generator().manual_seed(seed))
        noise = torch.empty_like(w).exponential_(1, generator=torch.Generator().manual_seed(seed))
        got = dr.multinomial_without_replacement(w, k, noise)
        assert torch.equal(got, want)
    # cell -> pixel expansion (dnerf_3d_video_IS.py:424-441): cell 5 of a 2-image set of 4 x 6 frames subsampled by 2
    # (hsub 2, wsub 3) is image 0, ysub 1, xsub 2 -> pixels (x, y) = (4, 2), (5, 2), (4, 3), (5, 3)
    images = torch.arange(2 * 4 * 6 * 3, dtype=torch.int64).remainder(251).to(torch.uint8).view(2, 4, 6, 3)
    c2w = torch.eye(4)[None, :3].repeat(2, 1, 1)
    K = torch.tensor([[5.0, 0, 3.0], [0, 5.0, 2.0], [0, 0, 1.0]])
    w = torch.zeros(2 * 2 * 3)
    w[5] = 1.0
    out = dr.fetch_data_train(images, c2w, K, torch.tensor([[0.25], [0.75]]), w, 2, 4, 6, 4, False, None, torch.ones(12))
    assert out["cells"].tolist() == [5] and out["idx"].tolist() == [0, 0, 0, 0]
    want_px = [(4, 2), (5, 2), (4, 3), (5, 3)]
    for j, (x, y) in enumerate(want_px):
        assert torch.equal(out["rgb"][j], images[0, y, x] / 255.0)
        d = torch.tensor([(x - 3.0 + 0.5) / 5.0, (y - 2.0 + 0.5) / 5.0, 1.0])
        torch.testing.assert_close(out["viewdirs"][j], d / d.norm(), rtol=0, atol=1e-7)
    assert torch.equal(out["timestamps"], torch.full((4, 1), 0.25))
