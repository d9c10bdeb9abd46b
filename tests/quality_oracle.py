"""Float64 restatement of the frame quality metrics (docs/SPEC.md "Evaluation metrics", U10) — TEST INFRASTRUCTURE.

PSNR as skimage's peak_signal_noise_ratio with data_range 1, SSIM as the upstream 3DGS ssim (the mean of U9's S map,
tests/loss_oracle.py), MS-SSIM as pytorch_msssim.ms_ssim(X, Y, data_range=1, size_average=False) writes it: valid
grouped convolutions with the 11x11 window per level, 2x2 average pooling with the odd side padded in front between
levels.  Any torch device (the GPU tests run it on the GPU at full size), float64 throughout.  The fused CUDA metrics
(gsvc_b200/csrc/quality.cu) are checked against it; tests/test_quality_cpu.py checks it against an independent scipy
restatement.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from tests import loss_oracle

WEIGHTS = (0.0448, 0.2856, 0.3001, 0.2363, 0.1333)
LEVELS = len(WEIGHTS)
MIN_SIDE = 161                      # MS-SSIM is defined when min(H, W) > (11 - 1) * 2^4


def _f64(t):
    return torch.as_tensor(t).to(torch.float64)


def psnr(x, y):
    """[N,3,H,W] -> [N]: 10 log10(1 / mse) of clamp(x, 0, 1) against y, +inf where mse == 0."""
    x, y = _f64(x).clamp(0.0, 1.0), _f64(y)
    mse = ((x - y) ** 2).mean(dim=(1, 2, 3))
    return torch.where(mse == 0, torch.full_like(mse, math.inf), 10.0 * torch.log10(1.0 / mse))


def ssim(x, y):
    """[N,3,H,W] -> [N]: mean of the zero-padded S map of clamp(x, 0, 1) and y."""
    return loss_oracle.ssim_map(_f64(x).clamp(0.0, 1.0), _f64(y)).mean(dim=(1, 2, 3))


def pool(a):
    """avg_pool2d(a, 2, stride 2, padding (h % 2, w % 2), count_include_pad=True), written out: an odd side gains one
    zero row / column in front, every window divides by 4, the output side is ceil(side / 2)."""
    h, w = a.shape[-2:]
    a = F.pad(a, (w % 2, 0, h % 2, 0))
    return (a[..., 0::2, 0::2] + a[..., 0::2, 1::2] + a[..., 1::2, 0::2] + a[..., 1::2, 1::2]) / 4.0


def level_means(x, y):
    """[N,3,h,w] -> (cs, ssim) [N,3]: the means of cs_map and ssim_map over the valid window positions."""
    win = loss_oracle.create_window(dtype=torch.float64).to(x.device)
    c = lambda a: F.conv2d(a, win, groups=3)
    mx, my = c(x), c(y)
    vx, vy, cxy = c(x * x) - mx * mx, c(y * y) - my * my, c(x * y) - mx * my
    C1, C2 = loss_oracle.C1, loss_oracle.C2
    cs_map = (2 * cxy + C2) / (vx + vy + C2)
    ssim_map = (2 * mx * my + C1) / (mx * mx + my * my + C1) * cs_map
    return cs_map.mean(dim=(2, 3)), ssim_map.mean(dim=(2, 3))


def ms_ssim_args(x, y):
    """[N,3,H,W] -> [N,3,5]: the per-channel arguments a_l of relu(.)^w_l: cs of levels 0-3, ssim of level 4."""
    x, y = _f64(x).clamp(0.0, 1.0), _f64(y)
    out = []
    for l in range(LEVELS):
        cs, ss = level_means(x, y)
        out.append(cs if l < LEVELS - 1 else ss)
        if l < LEVELS - 1:
            x, y = pool(x), pool(y)
    return torch.stack(out, dim=-1)


def ms_ssim_from_args(a):
    """[N,3,5] relu arguments -> ([N] MS-SSIM, [N,3] per channel)."""
    w = torch.tensor(WEIGHTS, dtype=torch.float64, device=a.device)
    per_c = torch.prod(torch.relu(a) ** w, dim=-1)
    return per_c.mean(dim=1), per_c


def ms_ssim(x, y):
    """[N,3,H,W] -> [N]; NaN when min(H, W) <= 160."""
    N, _, H, W = x.shape
    if min(H, W) < MIN_SIDE:
        return torch.full((N,), math.nan, dtype=torch.float64, device=_f64(x).device)
    return ms_ssim_from_args(ms_ssim_args(x, y))[0]


def frame_quality(x, y):
    """[N,3,H,W] -> [N,3] float64: (psnr, ssim, ms_ssim) per image."""
    return torch.stack([psnr(x, y), ssim(x, y), ms_ssim(x, y)], dim=1)
