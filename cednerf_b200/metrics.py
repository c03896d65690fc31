"""Image metric of the evaluation after training (train_real.py:443-520): `ms_ssim` with pytorch_msssim's signature
(v1.0, called at train_real.py:497-499), on the kernels of `csrc/metrics.cu`.

    from pytorch_msssim import ms_ssim   ->   from cednerf_b200.metrics import ms_ssim

Five scales and the final product in 6 launches on the current stream, for any batch size, with no host read; the
result is a device tensor and is the same from run to run.  The inputs are read in place at their strides, so the
reference's `rgb.permute(2, 0, 1)[None]` of an HWC frame costs no copy.  What the reference never calls is refused:
gradients, 5-D inputs, other windows, weights or K."""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from ._lib import call, stream

WIN_SIZE, WIN_SIGMA, K = 11, 1.5, (0.01, 0.03)
WEIGHTS = [0.0448, 0.2856, 0.3001, 0.2363, 0.1333]
N_SCALES = len(WEIGHTS)

_taps = None


def _gauss_taps():
    """pytorch_msssim._fspecial_gauss_1d(11, 1.5): fp32 taps formed with torch on the host."""
    global _taps
    if _taps is None:
        coords = torch.arange(WIN_SIZE, dtype=torch.float32)
        coords -= WIN_SIZE // 2
        g = torch.exp(-(coords ** 2) / (2 * WIN_SIGMA ** 2))
        g /= g.sum()
        _taps = (ctypes.c_float * WIN_SIZE)(*g.tolist())
    return _taps


def _check(X, Y, win_size, win_sigma, win, weights, K_):
    """pytorch_msssim's checks, in its order, then what this package does not support; nothing is launched."""
    if not X.shape == Y.shape:
        raise ValueError(f"Input images should have the same dimensions, but got {X.shape} and {Y.shape}.")
    if X.dim() == 5:
        raise NotImplementedError("ms_ssim: 5-D (video) inputs are not supported; the reference scores 4-D frames")
    if X.dim() != 4:
        raise ValueError(f"Input images should be 4-d or 5-d tensors, but got {X.shape}")
    if (win is not None or win_size != WIN_SIZE or win_sigma != WIN_SIGMA or tuple(K_) != K
            or (weights is not None and list(weights) != WEIGHTS)):
        raise NotImplementedError("ms_ssim: only the default window (11, 1.5), weights and K=(0.01, 0.03)")
    if X.requires_grad or Y.requires_grad:
        raise NotImplementedError("ms_ssim: no gradient (the reference only evaluates with it); pass detached tensors")
    smaller_side = min(X.shape[-2:])
    if not smaller_side > (WIN_SIZE - 1) * (2 ** 4):
        raise AssertionError("Image size should be larger than %d due to the 4 downsamplings in ms-ssim"
                             % ((WIN_SIZE - 1) * (2 ** 4)))
    if X.shape[0] < 1 or X.shape[1] < 1 or max(X.shape[-2:]) > 65536 or X.shape[0] * X.shape[1] > 65535:
        raise ValueError(f"ms_ssim: need 1 to 65535 image channels and sides up to 65536, got {X.shape}")
    if not (X.is_cuda and Y.is_cuda):
        raise RuntimeError("cednerf_b200 ops need CUDA tensors (no CPU fallback)")
    if X.device != Y.device:
        raise ValueError(f"ms_ssim: inputs on {X.device} and {Y.device}")
    if X.dtype != torch.float32 or Y.dtype != torch.float32:
        raise NotImplementedError(f"ms_ssim: fp32 inputs only, got {X.dtype} and {Y.dtype}")


def _layout(n, c, h, w):
    """Sides of every scale and the byte offsets of the pooled planes and the means in the workspace
    (include/cednerf_b200.h, cednerf_ms_ssim)."""
    sides = [(h, w)]
    for _ in range(N_SCALES - 1):
        sides.append(((sides[-1][0] + 1) // 2, (sides[-1][1] + 1) // 2))
    off, planes = 0, [None]
    for hs, ws in sides[1:]:
        size = n * c * hs * ws * 4
        planes.append((off, off + size))
        off += 2 * size
    return sides, planes, (off + 15) // 16 * 16


def _run(X, Y, data_range):
    n, c, h, w = X.shape
    lib = _lib.load()
    work = torch.empty(int(lib.cednerf_ms_ssim_workspace_bytes(n, c, h, w)), dtype=torch.uint8, device=X.device)
    out = torch.empty(n + 1, dtype=torch.float32, device=X.device)
    xs, ys = (ctypes.c_int64 * 4)(*X.stride()), (ctypes.c_int64 * 4)(*Y.stride())
    c1, c2 = (K[0] * data_range) ** 2, (K[1] * data_range) ** 2
    call("cednerf_ms_ssim", X.data_ptr(), ctypes.addressof(xs), Y.data_ptr(), ctypes.addressof(ys), n, c, h, w,
         ctypes.addressof(_gauss_taps()), c1, c2, work.data_ptr(), out.data_ptr(), stream())
    return out, work


def ms_ssim(X, Y, data_range=255, size_average=True, win_size=11, win_sigma=1.5, win=None, weights=None,
            K=(0.01, 0.03)):
    """pytorch_msssim.ms_ssim for fp32 CUDA [N, C, H, W] inputs (any strides), min(H, W) > 160.
    -> 0-dim tensor (size_average) or [N] (mean over channels per image), on X's device, computed on the current
    stream."""
    _check(X, Y, win_size, win_sigma, win, weights, K)
    out, _ = _run(X, Y, data_range)
    n = X.shape[0]
    return out[n] if size_average else out[:n]


def _ms_ssim_scales(X, Y, data_range=255):
    """For tests: (value per image [N], per scale: (ssim mean [N, C] fp64, cs mean [N, C] fp64, X_s, Y_s)), with X_s /
    Y_s the planes the kernel read at scale s (the inputs themselves at scale 0, the pooled planes after)."""
    _check(X, Y, WIN_SIZE, WIN_SIGMA, None, None, K)
    out, work = _run(X, Y, data_range)
    n, c, h, w = X.shape
    sides, planes, means_off = _layout(n, c, h, w)
    means = work[means_off:means_off + N_SCALES * n * c * 16].view(torch.float64).view(N_SCALES, n, c, 2)
    scales = []
    for s, (hs, ws) in enumerate(sides):
        if s == 0:
            xs, ys = X, Y
        else:
            size = n * c * hs * ws * 4
            xs, ys = (work[o:o + size].view(torch.float32).view(n, c, hs, ws) for o in planes[s])
        scales.append((means[s, ..., 0], means[s, ..., 1], xs, ys))
    return out[:n], scales
