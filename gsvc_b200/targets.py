"""8-bit source frames as targets of the loss and the quality metrics (docs/SPEC.md "8-bit source frames", U12).

A video's frames are bytes.  `photometric_loss`, `frame_quality`, `GraphedStep(loss_target=)` and
`FrameStreamer.render(target=)` take them as they are: a uint8 [F,H,W,3] cube (RGB interleaved, what
`np.array(PIL.Image)` and `frames_rgb8` hold) and an optional device index that picks frame index[n] for image n.
The kernels read byte q as fl(q / 255), torchvision's to_tensor, so every result equals the fp32 call with
`to_float(frames, index)` as the target, bit for bit.  An index outside [0, F) gives that image a NaN loss and quality
row and a zero gradient; it is never dereferenced.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from .rasterizer import RasterizerError


def decode_table() -> torch.Tensor:
    """The 256 fp32 values of the bytes: fl(q / 255), one correctly rounded division each (computed on the host,
    where torch divides; on CUDA, torch's division by a Python scalar multiplies by fl(1/255), which differs in 126
    of the 256 values)."""
    return torch.arange(256, dtype=torch.float32).div(255.0)


def to_float(frames: torch.Tensor, index: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The fp32 [N,3,H,W] targets the uint8 path computes with: frames[index] (or all frames), planar, decoded."""
    sel = frames if index is None else frames[index.long()]
    return decode_table().to(frames.device)[sel.long()].permute(0, 3, 1, 2).contiguous()


def is_rgb8(targets) -> bool:
    return isinstance(targets, torch.Tensor) and targets.dtype == torch.uint8


def index_i32(index: torch.Tensor, n_frames: int) -> torch.Tensor:
    """An integer index as the kernels read it: int32 contiguous.  A wider index is converted (a copy) with values
    beyond int32 clamped to -1 / n_frames, so they stay out of range instead of wrapping into it."""
    if index.dtype == torch.int32:
        return index if index.is_contiguous() else index.contiguous()
    return index.to(torch.int64).clamp(-1, n_frames).to(torch.int32)


def check(images: torch.Tensor, targets: torch.Tensor, index: Optional[torch.Tensor], single: bool,
          what: str = "targets") -> Tuple[torch.Tensor, int, Optional[torch.Tensor]]:
    """Validate a uint8 target of [N,3,H,W] `images` (`single`: the caller passed one [3,H,W] image).

    Without `index`: `targets` is [H,W,3] (single) or [N,H,W,3], image n against frame n.  With `index`: `targets`
    is a [F,H,W,3] cube and `index` an integer [N] tensor on the images' device.  Returns (frames [F,H,W,3]
    contiguous, F, index int32 [N] or None)."""
    N, _, H, W = images.shape
    if not is_rgb8(targets):
        raise RasterizerError(f"{what} must be a uint8 tensor")
    if targets.device != images.device:
        raise RasterizerError(f"images are on {images.device}, {what} on {targets.device}")
    if index is None:
        want = (H, W, 3) if single else (N, H, W, 3)
        if tuple(targets.shape) != want:
            raise RasterizerError(f"{what} must be uint8 {want} for images {tuple(images.shape[1 if single else 0:])} "
                                  f"(or a [F,{H},{W},3] cube with an index), got {tuple(targets.shape)}")
        frames = targets.unsqueeze(0) if single else targets
    else:
        if targets.dim() != 4 or tuple(targets.shape[1:]) != (H, W, 3) or targets.shape[0] < 1:
            raise RasterizerError(f"with an index, {what} must be a uint8 [F,{H},{W},3] frame cube, got "
                                  f"{tuple(targets.shape)}")
        if not isinstance(index, torch.Tensor) or index.dtype in (torch.bool,) or index.is_floating_point() \
                or index.is_complex():
            raise RasterizerError("index must be an integer tensor")
        if index.device != images.device:
            raise RasterizerError(f"index is on {index.device}, expected {images.device} (the kernels read it)")
        if tuple(index.shape) != (N,):
            raise RasterizerError(f"index must be shaped [{N}] (one frame per image), got {tuple(index.shape)}")
        if index.requires_grad:
            raise RasterizerError("index must not require a gradient")
        frames = targets
    n_frames = int(frames.shape[0])
    if n_frames >= 2 ** 31:
        raise RasterizerError(f"{what}: {n_frames} frames exceed an int32 frame index")
    frames = frames if frames.is_contiguous() else frames.contiguous()
    return frames, n_frames, None if index is None else index_i32(index, n_frames)
