"""pytorch_msssim.ms_ssim (v1.0.x, 4-D inputs), the score of the reference's evaluation (train_real.py:497-499).

The package is not vendored and not installed here, so two restatements stand in for it:

* `ms_ssim` / `ms_ssim_scales`: the package's own formulation in torch fp32, op for op (grouped conv2d along H then W,
  F.avg_pool2d with padding [H % 2, W % 2]).  Runs on CPU tensors, and on CUDA tensors as the baseline the reference
  pays for.
* `ms_ssim_fp64`: straight from the definition in numpy fp64: scipy.ndimage.correlate1d along H then W cropped to the
  valid region, pooling by explicit zero padding, 2x2 sums and division by 4 (count_include_pad).

tests/test_oracle_metrics.py pins the first to the second."""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

WEIGHTS = [0.0448, 0.2856, 0.3001, 0.2363, 0.1333]


def fspecial_gauss_1d(size=11, sigma=1.5):
    coords = torch.arange(size, dtype=torch.float)
    coords -= size // 2
    g = torch.exp(-(coords ** 2) / (2 * sigma ** 2))
    g /= g.sum()
    return g.unsqueeze(0).unsqueeze(0)


def gaussian_filter(x, win):
    """Valid cross-correlation with the 1-D window along H, then along W (win [C, 1, 1, size])."""
    c = x.shape[1]
    out = x
    for i in range(2):
        out = F.conv2d(out, weight=win.transpose(2 + i, -1), stride=1, padding=0, groups=c)
    return out


def _ssim(X, Y, data_range, win, K=(0.01, 0.03)):
    K1, K2 = K
    C1 = (K1 * data_range) ** 2
    C2 = (K2 * data_range) ** 2
    win = win.to(X.device, dtype=X.dtype)
    mu1 = gaussian_filter(X, win)
    mu2 = gaussian_filter(Y, win)
    mu1_sq = mu1.pow(2)
    mu2_sq = mu2.pow(2)
    mu1_mu2 = mu1 * mu2
    sigma1_sq = gaussian_filter(X * X, win) - mu1_sq
    sigma2_sq = gaussian_filter(Y * Y, win) - mu2_sq
    sigma12 = gaussian_filter(X * Y, win) - mu1_mu2
    cs_map = (2 * sigma12 + C2) / (sigma1_sq + sigma2_sq + C2)
    ssim_map = ((2 * mu1_mu2 + C1) / (mu1_sq + mu2_sq + C1)) * cs_map
    return torch.flatten(ssim_map, 2).mean(-1), torch.flatten(cs_map, 2).mean(-1)


def ms_ssim_scales(X, Y, data_range=255, taps=None):
    """-> (value [N, C], per scale: (ssim mean [N, C], cs mean [N, C], X_s, Y_s)) in X's dtype (fp32: the package).
    taps: the 11 window taps (default: the package's fp32 ones)."""
    assert X.shape == Y.shape and X.dim() == 4
    assert min(X.shape[-2:]) > 160, "Image size should be larger than 160 due to the 4 downsamplings in ms-ssim"
    win = (fspecial_gauss_1d(11, 1.5) if taps is None else torch.as_tensor(taps).view(1, 1, -1))
    win = win.repeat([X.shape[1], 1, 1, 1])
    weights = X.new_tensor(WEIGHTS)
    mcs, scales = [], []
    for i in range(len(WEIGHTS)):
        ssim_pc, cs = _ssim(X, Y, data_range, win)
        scales.append((ssim_pc, cs, X, Y))
        if i < len(WEIGHTS) - 1:
            mcs.append(torch.relu(cs))
            padding = [s % 2 for s in X.shape[2:]]
            X = F.avg_pool2d(X, kernel_size=2, padding=padding)
            Y = F.avg_pool2d(Y, kernel_size=2, padding=padding)
    ssim_pc = torch.relu(ssim_pc)
    val = torch.prod(torch.stack(mcs + [ssim_pc], dim=0) ** weights.view(-1, 1, 1), dim=0)
    return val, scales


def ms_ssim(X, Y, data_range=255, size_average=True):
    val, _ = ms_ssim_scales(X, Y, data_range)
    return val.mean() if size_average else val.mean(1)


def sample_images(kind, n, h, w, seed):
    """Test inputs: a pair of [n, 3, h, w] images in [0, 1], "smooth" (+ noise), "noise" (uniform) or "flat" (0.5 + 1e-3
    noise: the fp32 cancellation in E[x^2] - mu^2 is largest there)."""
    g = torch.Generator().manual_seed(seed)

    def one():
        if kind == "smooth":
            yy, xx = torch.meshgrid(torch.linspace(0, 6, h), torch.linspace(0, 9, w), indexing="ij")
            base = 0.5 + 0.3 * torch.sin(xx[None, None] + torch.arange(3).view(1, 3, 1, 1)) * torch.cos(yy)
            return (base.expand(n, 3, h, w) + 0.05 * torch.randn(n, 3, h, w, generator=g)).clamp(0, 1).contiguous()
        if kind == "noise":
            return torch.rand(n, 3, h, w, generator=g)
        return 0.5 + 1e-3 * torch.randn(n, 3, h, w, generator=g)

    return one(), one()


# ------------------------------------------------------------------------------------------------ fp64, from the definition
def taps64(size=11, sigma=1.5):
    """The normalised Gaussian window in fp64 (the package forms it in fp32: its taps differ by ~1e-8 and do not sum to
    exactly 1, which moves the cs of low-variance coarse scales by up to ~1e-5)."""
    c = np.arange(size, dtype=np.float64) - size // 2
    g = np.exp(-(c ** 2) / (2 * sigma ** 2))
    return g / g.sum()


def _gf64(img, g):
    from scipy.ndimage import correlate1d

    r = len(g) // 2
    out = correlate1d(img, g, axis=0, mode="constant")[r:img.shape[0] - r]
    return correlate1d(out, g, axis=1, mode="constant")[:, r:img.shape[1] - r]


def _pool64(img):
    h, w = img.shape
    ph, pw = h % 2, w % 2
    p = np.zeros((h + 2 * ph, w + 2 * pw))
    p[ph:ph + h, pw:pw + w] = img
    ho, wo = (h + 2 * ph - 2) // 2 + 1, (w + 2 * pw - 2) // 2 + 1
    p = p[:2 * ho, :2 * wo]
    return (p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]) / 4


def ms_ssim_fp64_scales(X, Y, data_range=255, taps=None):
    """-> (value [N, C], per scale: (ssim mean [N, C], cs mean [N, C], X_s [N, C, h, w], Y_s)) as fp64 numpy arrays.
    taps: the window (default: taps64())."""
    x = np.asarray(X.detach().cpu().double().numpy())
    y = np.asarray(Y.detach().cpu().double().numpy())
    n, c = x.shape[:2]
    g = taps64() if taps is None else np.asarray(taps, dtype=np.float64).reshape(-1)
    c1, c2 = (0.01 * data_range) ** 2, (0.03 * data_range) ** 2
    scales = []
    for s in range(len(WEIGHTS)):
        ss, cs = np.zeros((n, c)), np.zeros((n, c))
        for i in range(n):
            for j in range(c):
                a, b = x[i, j], y[i, j]
                mu1, mu2 = _gf64(a, g), _gf64(b, g)
                s1 = _gf64(a * a, g) - mu1 * mu1
                s2 = _gf64(b * b, g) - mu2 * mu2
                s12 = _gf64(a * b, g) - mu1 * mu2
                cs_map = (2 * s12 + c2) / (s1 + s2 + c2)
                ssim_map = (2 * mu1 * mu2 + c1) / (mu1 * mu1 + mu2 * mu2 + c1) * cs_map
                ss[i, j], cs[i, j] = ssim_map.mean(), cs_map.mean()
        scales.append((ss, cs, x, y))
        if s < len(WEIGHTS) - 1:
            x = np.stack([np.stack([_pool64(x[i, j]) for j in range(c)]) for i in range(n)])
            y = np.stack([np.stack([_pool64(y[i, j]) for j in range(c)]) for i in range(n)])
    val = np.ones((n, c))
    for s, w in enumerate(WEIGHTS):
        m = scales[s][1] if s < len(WEIGHTS) - 1 else scales[s][0]
        val = val * np.maximum(m, 0.0) ** w
    return val, scales


def ms_ssim_fp64(X, Y, data_range=255, size_average=True, taps=None):
    val, _ = ms_ssim_fp64_scales(X, Y, data_range, taps)
    return float(val.mean()) if size_average else val.mean(1)
