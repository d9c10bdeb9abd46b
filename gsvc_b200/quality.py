"""Frame quality metrics on the device: PSNR, SSIM and MS-SSIM (docs/SPEC.md "Evaluation metrics", decision U10).

The reference's `evaluate()` (utils/report_utils.py:267-407) copies every rendered frame to the host for skimage's
PSNR, runs the unfused 3DGS ssim and pytorch_msssim's 5-level pyramid.  Here one call computes all three per image
(gsvc_b200/csrc/quality.cu): one pass over the full-size images, four small pyramid levels and a per-image
reduction, deterministic, without host synchronisation and capturable in a CUDA graph:

    q = frame_quality(image, gt)          # [3,H,W] -> [3]; [N,3,H,W] -> [N,3]; columns psnr, ssim, ms_ssim

`image` is clamped to [0, 1] on read (the evaluation clamp), `gt` is used as given.  MS-SSIM is NaN when
min(H, W) <= 160 (pytorch_msssim refuses such images); PSNR is +inf for identical images.  No gradient.

`gt` may be the source video's 8-bit frames (SPEC U12, gsvc_b200.targets): uint8 [H,W,3] / [N,H,W,3], or a [F,H,W,3]
cube with `index=` ([N] integer, on the device).  An index outside [0, F) gives that image a NaN row.
"""
from __future__ import annotations

import torch

from . import _lib, targets as T8
from .rasterizer import RasterizerError, _bytes, _dev_f32, _on_device, _require_cuda, _stream_ptr


def _check(images, targets):
    for t, what in ((images, "images"), (targets, "targets")):
        if not isinstance(t, torch.Tensor):
            raise RasterizerError(f"{what} must be a tensor")
        _require_cuda(t, what)
    if images.device != targets.device:
        raise RasterizerError(f"images are on {images.device}, targets on {targets.device}")
    if images.shape != targets.shape:
        raise RasterizerError(f"images {tuple(images.shape)} and targets {tuple(targets.shape)} differ in shape")
    if images.dim() not in (3, 4) or images.shape[-3] != 3 or images.numel() == 0:
        raise RasterizerError(f"expected [3,H,W] or [N,3,H,W] images with N, H, W >= 1, got {tuple(images.shape)}")


def scratch_bytes(n: int, H: int, W: int) -> int:
    return int(_lib.lib().gsvc_rast_quality_scratch_bytes(n, H, W))


def quality_into(out: torch.Tensor, images: torch.Tensor, targets: torch.Tensor, scratch: torch.Tensor) -> None:
    """Enqueue the metrics of [N,3,H,W] fp32 contiguous `images` / `targets` into `out` ([N,3] fp32 contiguous) on the
    current stream, with a caller-owned `scratch` of at least scratch_bytes(N, H, W) bytes."""
    N, _, H, W = images.shape
    _lib.check(_lib.lib().gsvc_rast_quality(N, H, W, images.data_ptr(), targets.data_ptr(), out.data_ptr(),
                                            scratch.data_ptr(), _stream_ptr(images.device)), "gsvc_rast_quality")


def quality_rgb8_into(out: torch.Tensor, images: torch.Tensor, frames: torch.Tensor, index, scratch: torch.Tensor) -> None:
    """quality_into with 8-bit targets: `frames` uint8 [F,H,W,3] contiguous, `index` int32 [N] contiguous or None
    (image n against frame n, N <= F), both on the images' device."""
    N, _, H, W = images.shape
    _lib.check(_lib.lib().gsvc_rast_quality_rgb8(N, H, W, images.data_ptr(), frames.data_ptr(), frames.shape[0],
                                                 None if index is None else index.data_ptr(), out.data_ptr(),
                                                 scratch.data_ptr(), _stream_ptr(images.device)),
               "gsvc_rast_quality_rgb8")


def frame_quality(images: torch.Tensor, targets: torch.Tensor, index: torch.Tensor = None) -> torch.Tensor:
    """(PSNR, SSIM, MS-SSIM) of each image against its target.

    `images`, `targets`: [3,H,W] (returns [3]) or [N,3,H,W] (returns [N,3]) CUDA tensors on the same device, cast to
    fp32 and made contiguous.  The result is fp32 on that device and carries no gradient.

    8-bit targets (SPEC U12): `targets` uint8 [H,W,3] / [N,H,W,3], or a [F,H,W,3] cube with `index` (integer [N] on
    the device); bit for bit the fp32 result with `gsvc_b200.targets.to_float(frames, index)`."""
    if T8.is_rgb8(targets):
        return _frame_quality_rgb8(images, targets, index)
    if index is not None:
        raise RasterizerError("index selects frames of a uint8 target cube; these targets are not uint8")
    _check(images, targets)
    single = images.dim() == 3
    device = images.device
    with torch.no_grad(), _on_device(device):
        x = _dev_f32(images.detach(), device, "images")
        y = _dev_f32(targets.detach(), device, "targets")
        if single:
            x, y = x.unsqueeze(0), y.unsqueeze(0)
        N, _, H, W = x.shape
        out = torch.empty((N, 3), dtype=torch.float32, device=device)
        quality_into(out, x, y, _bytes(scratch_bytes(N, H, W), device))
    return out[0] if single else out


def _frame_quality_rgb8(images, targets, index):
    if not isinstance(images, torch.Tensor):
        raise RasterizerError("images must be a tensor")
    _require_cuda(images, "images")
    if images.dim() not in (3, 4) or images.shape[-3] != 3 or images.numel() == 0:
        raise RasterizerError(f"expected [3,H,W] or [N,3,H,W] images with N, H, W >= 1, got {tuple(images.shape)}")
    single = images.dim() == 3
    device = images.device
    with torch.no_grad(), _on_device(device):
        x = _dev_f32(images.detach(), device, "images")
        if single:
            x = x.unsqueeze(0)
        frames, _, idx = T8.check(x, targets, index, single)
        N, _, H, W = x.shape
        out = torch.empty((N, 3), dtype=torch.float32, device=device)
        quality_rgb8_into(out, x, frames, idx, _bytes(scratch_bytes(N, H, W), device))
    return out[0] if single else out
