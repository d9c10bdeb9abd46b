"""8-bit frame export on the device (docs/SPEC.md "8-bit frame export", decision U11).

A decoded frame leaves the renderer as fp32 [3,H,W] planes; image writers (PIL, PNG encoders) take 8-bit RGB
[H,W,3].  The reference saves its renders with torchvision's save_image, whose arithmetic this conversion restates in
one kernel (gsvc_b200/csrc/export.cu): a quarter of the bytes of the fp32 frame to copy to the host, no host
synchronisation, capturable in a CUDA graph:

    rgb = frames_rgb8(image)          # [3,H,W] -> [H,W,3]; [N,3,H,W] -> [N,H,W,3]; uint8 on the images' device

Per value q = uint8(clamp(fl(fl(x * 255) + 0.5), 0, 255)), truncated, the product and the sum rounded separately;
NaN -> 0.  No gradient.  FrameStreamer.render(..., host_out=) converts and copies each decoded frame to pinned host
memory this way.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from .rasterizer import RasterizerError, _dev_f32, _on_device, _require_cuda, _stream_ptr


def rgb8_into(out: torch.Tensor, images: torch.Tensor) -> None:
    """Enqueue the conversion of [N,3,H,W] fp32 contiguous `images` into `out` (contiguous uint8, N*H*W*3 bytes) on the
    current stream."""
    N, _, H, W = images.shape
    _lib.check(_lib.lib().gsvc_rast_frames_rgb8(N, H, W, images.data_ptr(), out.data_ptr(),
                                                _stream_ptr(images.device)), "gsvc_rast_frames_rgb8")


def frames_rgb8(images: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """8-bit RGB of composed frames.

    `images`: [3,H,W] (returns [H,W,3]) or [N,3,H,W] (returns [N,H,W,3]) on a CUDA device, cast to fp32 and made
    contiguous.  `out`: an optional contiguous uint8 tensor of the result's shape on that device, written and
    returned.  The result carries no gradient."""
    if not isinstance(images, torch.Tensor):
        raise RasterizerError("images must be a tensor")
    _require_cuda(images, "images")
    if images.dim() not in (3, 4) or images.shape[-3] != 3 or images.numel() == 0:
        raise RasterizerError(f"expected [3,H,W] or [N,3,H,W] images with N, H, W >= 1, got {tuple(images.shape)}")
    device = images.device
    H, W = images.shape[-2:]
    want = (H, W, 3) if images.dim() == 3 else (images.shape[0], H, W, 3)
    if out is not None and (not isinstance(out, torch.Tensor) or out.device != device or out.dtype != torch.uint8
                            or tuple(out.shape) != want or not out.is_contiguous()):
        raise RasterizerError(f"out must be a contiguous uint8 tensor of shape {want} on {device}")
    with torch.no_grad(), _on_device(device):
        x = _dev_f32(images.detach(), device, "images")
        if out is None:
            out = torch.empty(want, dtype=torch.uint8, device=device)
        rgb8_into(out, x.reshape(-1, 3, H, W))
    return out
