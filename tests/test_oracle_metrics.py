"""oracle/metrics_ref.py: the torch restatement of pytorch_msssim.ms_ssim pinned to the fp64 restatement from the
definition, and cednerf_b200.metrics.ms_ssim's argument checks (all on the CPU, before any launch)."""
import numpy as np
import pytest
import torch

from oracle import metrics_ref as mr

SIZES = [(1, 1014, 1352), (1, 800, 800), (1, 960, 536), (1, 161, 333), (3, 200, 240)]
SCALE_SIDES = {(1014, 1352): [(1014, 1352), (507, 676), (254, 338), (127, 169), (64, 85)],
               (161, 333): [(161, 333), (81, 167), (41, 84), (21, 42), (11, 21)]}


def deviations(got, want):
    """max |value difference|, max |difference| of every scale's ssim and cs means"""
    (v, sc), (v64, sc64) = got, want
    per_scale = max(max(np.abs(a.double().numpy() - b).max(), np.abs(c.double().numpy() - d).max())
                    for (a, c, _, _), (b, d, _, _) in zip(sc, sc64))
    return float(np.abs(v.double().numpy() - v64).max()), float(per_scale)


@pytest.mark.parametrize("kind", ["smooth", "noise", "flat"])
@pytest.mark.parametrize("n,h,w", SIZES)
def test_torch_restatement_against_the_definition(kind, n, h, w):
    X, Y = mr.sample_images(kind, n, h, w, seed=h + w)
    # the formulation: run in fp64 with the fp64 window, op order, valid crop, H before W and the pooling rule are those
    # of the definition up to fp64 rounding
    v, sc = mr.ms_ssim_scales(X.double(), Y.double(), 1.0, taps=torch.from_numpy(mr.taps64()))
    v64, sc64 = mr.ms_ssim_fp64_scales(X, Y, 1.0)
    assert max(deviations((v, sc), (v64, sc64))) <= 1e-12
    for (_, _, x, y), (_, _, x64, y64) in zip(sc, sc64):
        assert np.abs(x.numpy() - x64).max() <= 1e-15 and np.abs(y.numpy() - y64).max() <= 1e-15
    # the package's fp32 arithmetic with its fp32 window against the definition with that window.  Measured on the CPU:
    # values <= 3.3e-7 (textured) and 7.0e-6 (flat: the fp32 cancellation in E[x^2] - mu^2), per-scale means <= 3.7e-5
    taps32 = mr.fspecial_gauss_1d().view(-1).double().numpy()
    d_val, d_scale = deviations(mr.ms_ssim_scales(X, Y, 1.0), mr.ms_ssim_fp64_scales(X, Y, 1.0, taps=taps32))
    assert d_val <= (1e-6 if kind != "flat" else 1e-4), d_val
    assert d_scale <= 1e-4, d_scale


def test_identity_scale_sides_and_constant_images():
    x = mr.sample_images("smooth", 1, 1014, 1352, seed=3)[0]
    assert float(mr.ms_ssim(x, x, 1.0)) == 1.0
    for (h, w), sides in SCALE_SIDES.items():
        _, sc = mr.ms_ssim_scales(torch.rand(1, 1, h, w), torch.rand(1, 1, h, w), 1.0)
        assert [tuple(s[2].shape[-2:]) for s in sc] == sides
    # constant images a and b: ssim = (2ab + C1) / (a^2 + b^2 + C1), cs = 1 - up to the fp32 window not summing to 1
    for a, b, dr in ((0.3, 0.7, 1.0), (10.0, 30.0, 255.0), (0.5, 0.5, 1.0)):
        c1 = (0.01 * dr) ** 2
        _, sc = mr.ms_ssim_scales(torch.full((2, 3, 170, 200), a), torch.full((2, 3, 170, 200), b), dr)
        for s, (ssim, cs, _, _) in enumerate(sc):
            if s == 0:   # the pooled borders are darker (count_include_pad): only scale 0 is constant everywhere
                torch.testing.assert_close(ssim, torch.full_like(ssim, (2 * a * b + c1) / (a * a + b * b + c1)),
                                           rtol=0, atol=1e-4)
                torch.testing.assert_close(cs, torch.ones_like(cs), rtol=0, atol=1e-4)


def test_ms_ssim_checks_its_arguments_before_any_launch():
    from cednerf_b200 import _lib, metrics

    x = torch.rand(1, 3, 170, 180)
    launches = _lib.launch_count()
    with pytest.raises(ValueError):
        metrics.ms_ssim(x, torch.rand(1, 3, 170, 181))
    with pytest.raises(AssertionError, match="Image size should be larger than 160 due to the 4 downsamplings in ms-ssim"):
        metrics.ms_ssim(torch.rand(1, 3, 160, 300), torch.rand(1, 3, 160, 300))
    with pytest.raises(NotImplementedError):
        metrics.ms_ssim(x, x, win_size=7)
    for kw in (dict(win_sigma=2.0), dict(K=(0.02, 0.03)), dict(weights=[0.2] * 5), dict(win=torch.ones(3, 1, 1, 11))):
        with pytest.raises(NotImplementedError):
            metrics.ms_ssim(x, x, **kw)
    with pytest.raises(NotImplementedError):
        metrics.ms_ssim(x.clone().requires_grad_(True), x)
    with pytest.raises(NotImplementedError):
        metrics.ms_ssim(torch.rand(1, 3, 2, 170, 180), torch.rand(1, 3, 2, 170, 180))
    with pytest.raises(RuntimeError):   # no CPU fallback
        metrics.ms_ssim(x, x)
    with pytest.raises(RuntimeError):
        metrics.ms_ssim(x, x, data_range=1.0, size_average=False, weights=list(mr.WEIGHTS))
    assert _lib.launch_count() == launches
