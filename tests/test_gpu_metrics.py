"""cednerf_b200.metrics.ms_ssim (csrc/metrics.cu) against oracle/metrics_ref.py: the fp32 torch restatement of
pytorch_msssim.ms_ssim and the fp64 restatement from the definition; pooled planes bit for bit, identity, determinism,
strided inputs, 6 launches and no host synchronisation per call, and scoring inside render_images_test's on_frame."""
import dataclasses

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import metrics_ref as mr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIZES = [(1, 1014, 1352), (1, 800, 800), (1, 960, 536), (1, 161, 333), (3, 200, 240)]
# |kernel - oracle| bound for values and per-scale means (both oracles).  Measured on a B200 over the cases below: 1.4e-6 on
# the smooth images, 2.7e-5 on uniform noise and flat images (fp32 cancellation in E[x^2] - mu^2 on coarse scales of a
# few hundred pixels).  The bounds are about 10x and 4x of that.
TOL = {"smooth": 2e-5, "noise": 1e-4, "flat": 1e-4}


@pytest.fixture(scope="module")
def cb():
    import cednerf_b200

    return cednerf_b200


@pytest.mark.parametrize("data_range", [1.0, 255.0])
@pytest.mark.parametrize("kind", ["smooth", "noise", "flat"])
@pytest.mark.parametrize("n,h,w", SIZES)
def test_values_and_scales_against_both_oracles(cb, kind, n, h, w, data_range):
    X, Y = (t * data_range for t in mr.sample_images(kind, n, h, w, seed=h + w))
    Xd, Yd = X.to(DEV), Y.to(DEV)
    val, scales = cb.metrics._ms_ssim_scales(Xd, Yd, data_range)
    mean = cb.metrics.ms_ssim(Xd, Yd, data_range=data_range)
    per_image = cb.metrics.ms_ssim(Xd, Yd, data_range=data_range, size_average=False)
    assert mean.shape == () and per_image.shape == (n,) and mean.dtype == per_image.dtype == torch.float32
    assert torch.equal(per_image, val)

    v32, sc32 = mr.ms_ssim_scales(X, Y, data_range)
    v64, sc64 = mr.ms_ssim_fp64_scales(X, Y, data_range, taps=mr.fspecial_gauss_1d().view(-1).double().numpy())
    dev32 = max(float((per_image.cpu() - v32.mean(1)).abs().max()), abs(float(mean) - float(v32.mean())))
    dev64 = max(float(np.abs(per_image.cpu().double().numpy() - v64.mean(1)).max()), abs(float(mean) - v64.mean()))
    for s, ((ss, cs, xs, ys), (ss32, cs32, _, _), (ss64, cs64, _, _)) in enumerate(zip(scales, sc32, sc64)):
        ss, cs = ss.cpu(), cs.cpu()
        dev32 = max(dev32, float((ss - ss32.double()).abs().max()), float((cs - cs32.double()).abs().max()))
        dev64 = max(dev64, float(np.abs(ss.numpy() - ss64).max()), float(np.abs(cs.numpy() - cs64).max()))
        if s + 1 < len(scales):   # the next scale's planes are F.avg_pool2d of this scale's, bit for bit
            pad = [h_ % 2 for h_ in xs.shape[2:]]
            assert torch.equal(scales[s + 1][2], F.avg_pool2d(xs, kernel_size=2, padding=pad)), s
            assert torch.equal(scales[s + 1][3], F.avg_pool2d(ys, kernel_size=2, padding=pad)), s
    print(f"ms_ssim deviation {kind} n={n} {h}x{w} data_range={data_range:g}: fp32 oracle {dev32:.2e}, fp64 {dev64:.2e}")
    assert dev32 <= TOL[kind] and dev64 <= TOL[kind], (dev32, dev64)


def test_identity_determinism_and_strided_inputs(cb):
    ms_ssim = cb.metrics.ms_ssim
    X, Y = (t.to(DEV) for t in mr.sample_images("smooth", 1, 1014, 1352, seed=5))
    assert float(ms_ssim(X, X, data_range=1.0)) == 1.0
    assert torch.equal(ms_ssim(X, X.clone(), data_range=1.0, size_average=False), torch.ones(1, device=DEV))
    a = cb.metrics._ms_ssim_scales(X, Y, 1.0)
    b = cb.metrics._ms_ssim_scales(X, Y, 1.0)
    assert torch.equal(a[0], b[0])
    for sa, sb in zip(a[1], b[1]):
        assert all(torch.equal(p, q) for p, q in zip(sa, sb))
    # the reference's call: rgb.permute(2, 0, 1)[None] of HWC frames, read in place; x and y at different strides
    hwc = X[0].permute(1, 2, 0).contiguous()
    tgt = Y[0].permute(1, 2, 0).contiguous()
    view = hwc.permute(2, 0, 1)[None]
    assert not view.is_contiguous()
    for size_average in (True, False):
        want = ms_ssim(view.contiguous(), Y, data_range=1.0, size_average=size_average)
        assert torch.equal(ms_ssim(view, Y, data_range=1.0, size_average=size_average), want)
        assert torch.equal(ms_ssim(view, tgt.permute(2, 0, 1)[None], data_range=1.0, size_average=size_average), want)
    # a batch of views: a strided slice of a larger tensor
    big = torch.rand(3, 3, 500, 500, device=DEV)
    sl = big[:, :, 7:407:2, 11:411]   # 200 x 400, every second row
    other = torch.rand(3, 3, 200, 400, device=DEV)
    assert torch.equal(ms_ssim(sl, other, 1.0, size_average=False), ms_ssim(sl.contiguous(), other, 1.0, size_average=False))


@pytest.mark.parametrize("n", [1, 4])
def test_six_launches_and_no_host_synchronisation(cb, n):
    X, Y = (torch.rand(n, 3, 240, 320, device=DEV) for _ in range(2))
    cb.metrics.ms_ssim(X, Y, 1.0)
    torch.cuda.synchronize()
    before = cb._lib.launch_count()
    torch.cuda.set_sync_debug_mode("error")
    try:
        out = cb.metrics.ms_ssim(X, Y, data_range=1.0, size_average=False)
        mean = cb.metrics.ms_ssim(X, Y, data_range=1.0)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert cb._lib.launch_count() == before + 12
    assert out.is_cuda and mean.is_cuda
    torch.testing.assert_close(mean.cpu(), mr.ms_ssim(X.cpu(), Y.cpu(), 1.0), rtol=0, atol=TOL["noise"])


@pytest.mark.parametrize("concurrency", [1, 3])
def test_scores_inside_on_frame_equal_render_then_score(cb, concurrency):
    from cednerf_b200 import workload as w

    cfg = dataclasses.replace(w.TINY, width=256, height=192, focal=160.0)
    rk = w.render_kwargs(cfg)
    est, field = w.build_scene(cfg, DEV, cb, seed=42)
    est.eval(), field.eval()
    poses = w.spiral_poses(cfg, 4)
    K = [[cfg.focal, 0.0, cfg.width / 2], [0.0, cfg.focal, cfg.height / 2], [0.0, 0.0, 1.0]]
    bk = torch.tensor([0.2, 0.4, 0.6], device=DEV)
    rays = [cb.utils.generate_rays(K, poses[k].to(DEV), cfg.width, cfg.height) for k in range(4)]
    ts = [torch.tensor([[k / 8.0]], device=DEV) for k in range(4)]
    score = lambda rgb, tgt: cb.metrics.ms_ssim(rgb.permute(2, 0, 1)[None], tgt.permute(2, 0, 1)[None],  # noqa: E731
                                                data_range=1.0)
    with torch.no_grad():
        targets = [cb.render_image_test(1024, field, est, rays[k], render_bkgd=bk, timestamps=ts[k] + 0.5, **rk)[0]
                   for k in range(4)]
        want = [score(cb.render_image_test(1024, field, est, rays[k], render_bkgd=bk, timestamps=ts[k], **rk)[0],
                      targets[k]) for k in range(4)]
        got = [None] * 4

        def on_frame(k, result):
            assert result[0].shape == (cfg.height, cfg.width, 3)
            got[k] = score(result[0], targets[k])

        cb.render_images_test(1024, field, est, rays, ts, concurrency=concurrency, on_frame=on_frame, render_bkgd=bk, **rk)
        torch.cuda.synchronize()
    for k in range(4):
        assert torch.equal(got[k], want[k]), (k, float(got[k]), float(want[k]))
    assert all(0.0 < float(v) <= 1.0 for v in want), [float(v) for v in want]
