"""Float64 restatement of the photometric loss (docs/SPEC.md "Photometric loss", U9) — TEST INFRASTRUCTURE.

Written the way the upstream 3DGS code writes it (utils/loss_utils.py:41-72: F.conv2d with groups=3, padding=5 over
the 11x11 Gaussian window), on the CPU in float64, with the gradient from autograd.  It is the reference the fused
CUDA loss (gsvc_b200/csrc/loss.cu) is checked against; tests/test_loss_cpu.py checks it against an independent
scipy restatement and against finite differences.
"""
from __future__ import annotations

import math

import numpy as np
import torch
import torch.nn.functional as F

WINDOW = 11
SIGMA = 1.5
C1 = 0.01 ** 2
C2 = 0.03 ** 2


def gaussian(window_size=WINDOW, sigma=SIGMA, dtype=torch.float64):
    g = torch.tensor([math.exp(-(x - window_size // 2) ** 2 / float(2 * sigma ** 2)) for x in range(window_size)],
                     dtype=dtype)
    return g / g.sum()


def create_window(window_size=WINDOW, channel=3, dtype=torch.float64):
    g = gaussian(window_size, dtype=dtype).unsqueeze(1)
    w2 = g.mm(g.t()).unsqueeze(0).unsqueeze(0)
    return w2.expand(channel, 1, window_size, window_size).contiguous()


def ssim_map(img1, img2, window_size=WINDOW, window=None):
    """[N,3,H,W] -> the per-pixel S of the upstream _ssim (same expression, same order).  `window`: a prebuilt
    create_window() on the inputs' device and dtype (built per call otherwise, as upstream does)."""
    channel = img1.shape[-3]
    if window is None:
        window = create_window(window_size, channel, img1.dtype).to(img1.device)
    pad = window_size // 2
    mu1 = F.conv2d(img1, window, padding=pad, groups=channel)
    mu2 = F.conv2d(img2, window, padding=pad, groups=channel)
    mu1_sq, mu2_sq, mu1_mu2 = mu1.pow(2), mu2.pow(2), mu1 * mu2
    sigma1_sq = F.conv2d(img1 * img1, window, padding=pad, groups=channel) - mu1_sq
    sigma2_sq = F.conv2d(img2 * img2, window, padding=pad, groups=channel) - mu2_sq
    sigma12 = F.conv2d(img1 * img2, window, padding=pad, groups=channel) - mu1_mu2
    return ((2 * mu1_mu2 + C1) * (2 * sigma12 + C2)) / ((mu1_sq + mu2_sq + C1) * (sigma1_sq + sigma2_sq + C2))


def photometric_loss(x, y, lambda_dssim=0.2, window=None):
    """x, y [N,3,H,W] -> [N]: (1 - l) mean|x - y| + l (1 - mean S), means per image."""
    l1 = (x - y).abs().mean(dim=(1, 2, 3))
    s = ssim_map(x, y, window=window).mean(dim=(1, 2, 3))
    return (1.0 - lambda_dssim) * l1 + lambda_dssim * (1.0 - s)


def loss_and_grad(x, y, lambda_dssim=0.2, dL_dloss=None):
    """Float64 loss [N] and dL/dx [N,3,H,W] (numpy) for dL = sum_n dL_dloss[n] loss[n] (all ones by default)."""
    xd = torch.as_tensor(np.asarray(x), dtype=torch.float64).clone().requires_grad_(True)
    yd = torch.as_tensor(np.asarray(y), dtype=torch.float64)
    loss = photometric_loss(xd, yd, lambda_dssim)
    g = torch.ones_like(loss) if dL_dloss is None else torch.as_tensor(np.asarray(dL_dloss), dtype=torch.float64)
    (grad,) = torch.autograd.grad(loss, xd, grad_outputs=g)
    return loss.detach().numpy(), grad.numpy()
