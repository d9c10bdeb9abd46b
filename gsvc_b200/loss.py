"""Fused L1 + D-SSIM photometric training loss (docs/SPEC.md "Photometric loss", decision U9).

The reference's iteration (pipeline/train.py:407-444) computes `(1 - l) * l1_loss(image, gt) + l * (1 - ssim(image,
gt))` with the upstream 3DGS ssim (utils/loss_utils.py:41-72): five depthwise 11x11 convolutions and about twenty
element-wise ops over full-size tensors.  Here the forward is one pass over the images plus a per-image reduction and
the backward one pass (gsvc_b200/csrc/loss.cu), both deterministic and capturable in a CUDA graph:

    loss = photometric_loss(image, gt, lambda_dssim=0.2)      # [3,H,W] -> 0-dim, [N,3,H,W] -> [N]
    loss.backward()

lambda_dssim = 0 is the L1 term alone, 1 is 1 - SSIM.  The target gets no gradient (passing a target that requires
one raises).  CUDA tensors only: there is no CPU fallback.

The targets may be the source video's 8-bit frames (SPEC U12, gsvc_b200.targets): a uint8 [H,W,3] / [N,H,W,3] tensor,
or a resident [F,H,W,3] cube with a device index that picks frame index[n] for image n:

    loss = photometric_loss(image, cube, index=idx)          # [N,3,H,W] images, cube [F,H,W,3] uint8, idx [N] int
"""
from __future__ import annotations

import math

import torch

from . import _lib, targets as T8
from .rasterizer import RasterizerError, _bytes, _dev_f32, _on_device, _require_cuda, _stream_ptr


def _check_lambda(lambda_dssim) -> float:
    lam = float(lambda_dssim)
    if not math.isfinite(lam) or not 0.0 <= lam <= 1.0:
        raise RasterizerError(f"lambda_dssim must be a finite value in [0, 1], got {lambda_dssim}")
    return lam


class _PhotometricLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, images, targets, lam):
        L = _lib.lib()
        device = images.device
        N, _, H, W = images.shape
        with _on_device(device):
            x = _dev_f32(images, device, "images")
            y = _dev_f32(targets, device, "targets")
            loss = torch.empty(N, dtype=torch.float32, device=device)
            scratch = _bytes(L.gsvc_rast_loss_scratch_bytes(N, H, W), device)
            _lib.check(L.gsvc_rast_loss_forward(N, H, W, x.data_ptr(), y.data_ptr(), lam, loss.data_ptr(),
                                                scratch.data_ptr(), _stream_ptr(device)), "gsvc_rast_loss_forward")
        ctx.lam, ctx.in_dtype = lam, images.dtype
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(x, y)     # the backward recomputes the window moments from these two
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        x, y = ctx.saved_tensors
        device = x.device
        N, _, H, W = x.shape
        with _on_device(device):
            g = _dev_f32(grad_loss, device, "grad of the loss")
            dx = torch.empty_like(x)
            _lib.check(_lib.lib().gsvc_rast_loss_backward(N, H, W, x.data_ptr(), y.data_ptr(), ctx.lam, g.data_ptr(),
                                                          dx.data_ptr(), _stream_ptr(device)), "gsvc_rast_loss_backward")
        return (dx if ctx.in_dtype == torch.float32 else dx.to(ctx.in_dtype)), None, None


class _PhotometricLossRgb8(torch.autograd.Function):
    @staticmethod
    def forward(ctx, images, frames, index, lam):
        L = _lib.lib()
        device = images.device
        N, _, H, W = images.shape
        with _on_device(device):
            x = _dev_f32(images, device, "images")
            loss = torch.empty(N, dtype=torch.float32, device=device)
            scratch = _bytes(L.gsvc_rast_loss_scratch_bytes(N, H, W), device)
            _lib.check(L.gsvc_rast_loss_forward_rgb8(N, H, W, x.data_ptr(), frames.data_ptr(), frames.shape[0],
                                                     _ptr(index), lam, loss.data_ptr(), scratch.data_ptr(),
                                                     _stream_ptr(device)), "gsvc_rast_loss_forward_rgb8")
        ctx.lam, ctx.in_dtype = lam, images.dtype
        if ctx.needs_input_grad[0]:
            ctx.save_for_backward(x, frames, index)     # an in-place write of the index before backward raises
        return loss

    @staticmethod
    def backward(ctx, grad_loss):
        x, frames, index = ctx.saved_tensors
        device = x.device
        N, _, H, W = x.shape
        with _on_device(device):
            g = _dev_f32(grad_loss, device, "grad of the loss")
            dx = torch.empty_like(x)
            _lib.check(_lib.lib().gsvc_rast_loss_backward_rgb8(N, H, W, x.data_ptr(), frames.data_ptr(),
                                                               frames.shape[0], _ptr(index), ctx.lam, g.data_ptr(),
                                                               dx.data_ptr(), _stream_ptr(device)),
                       "gsvc_rast_loss_backward_rgb8")
        return (dx if ctx.in_dtype == torch.float32 else dx.to(ctx.in_dtype)), None, None, None


def _ptr(t):
    return None if t is None else t.data_ptr()


def photometric_loss(images: torch.Tensor, targets: torch.Tensor, lambda_dssim: float = 0.2,
                     index: torch.Tensor = None) -> torch.Tensor:
    """(1 - lambda_dssim) * mean|images - targets| + lambda_dssim * (1 - SSIM(images, targets)) per image.

    `images`, `targets`: [3,H,W] (returns a 0-dim tensor, the reference's scalar) or [N,3,H,W] (returns [N]) CUDA
    tensors on the same device; cast to fp32 and made contiguous as the rasterizer's inputs are.  The gradient flows
    to `images` only.

    8-bit targets (SPEC U12): `targets` uint8 [H,W,3] / [N,H,W,3] (image n against frame n), or a [F,H,W,3] cube with
    `index`, an integer [N] tensor on the device (image n against frame index[n]; an int32 index is read in place, a
    wider one converted).  The result equals the fp32 call with `gsvc_b200.targets.to_float(frames, index)` bit for bit; an
    index outside [0, F) gives that image a NaN loss and a zero gradient."""
    lam = _check_lambda(lambda_dssim)
    if T8.is_rgb8(targets):
        return _photometric_loss_rgb8(images, targets, lam, index)
    if index is not None:
        raise RasterizerError("index selects frames of a uint8 target cube; these targets are not uint8")
    for t, what in ((images, "images"), (targets, "targets")):
        if not isinstance(t, torch.Tensor):
            raise RasterizerError(f"{what} must be a tensor")
        _require_cuda(t, what)
    if targets.requires_grad:
        raise RasterizerError("targets.requires_grad is set, but the loss gives the target no gradient: detach it")
    if images.device != targets.device:
        raise RasterizerError(f"images are on {images.device}, targets on {targets.device}")
    if images.shape != targets.shape:
        raise RasterizerError(f"images {tuple(images.shape)} and targets {tuple(targets.shape)} differ in shape")
    single = images.dim() == 3
    if images.dim() not in (3, 4) or images.shape[-3] != 3 or images.numel() == 0:
        raise RasterizerError(f"expected [3,H,W] or [N,3,H,W] images with N, H, W >= 1, got {tuple(images.shape)}")
    if single:
        images, targets = images.unsqueeze(0), targets.unsqueeze(0)
    loss = _PhotometricLoss.apply(images, targets, lam)
    return loss[0] if single else loss


def _photometric_loss_rgb8(images, targets, lam, index):
    if not isinstance(images, torch.Tensor):
        raise RasterizerError("images must be a tensor")
    _require_cuda(images, "images")
    single = images.dim() == 3
    if images.dim() not in (3, 4) or images.shape[-3] != 3 or images.numel() == 0:
        raise RasterizerError(f"expected [3,H,W] or [N,3,H,W] images with N, H, W >= 1, got {tuple(images.shape)}")
    if single:
        images = images.unsqueeze(0)
    frames, _, idx = T8.check(images, targets, index, single)
    loss = _PhotometricLossRgb8.apply(images, frames, idx, lam)
    return loss[0] if single else loss
