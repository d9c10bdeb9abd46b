"""gsvc_b200 — B200-native (sm_100a) orthographic TSW Gaussian rasterizer for GSVC's render() hot path.

  rasterizer   GaussianRasterizationSettings / GaussianRasterizer: the reference-shaped drop-in (renderer.py:63-98)
  views        ViewBatch / rasterize_views / render_toast: a frame's front + back view (or a window) in one chain
  graphed      GraphedStep: CUDA-graph replay of forward + backward on static tensors (optionally with its own loss)
  loss         photometric_loss: the fused L1 + D-SSIM training loss (SPEC U9)
  quality      frame_quality: PSNR, SSIM and MS-SSIM of rendered frames on the device (SPEC U10)
  export       frames_rgb8: composed frames to 8-bit RGB [H,W,3] on the device, for image writers (SPEC U11)
  hostpipe     HostStepPipeline: pinned host parameters in, pinned host gradients out, copies overlapped
  sharding     frame-sharded rendering, packed [P,14] gradients, NCCL all-reduce
  frames       cube geometry and the synthetic workload generator
"""
from .rasterizer import GaussianRasterizationSettings, GaussianRasterizer, RasterizerError  # noqa: F401
from .quality import frame_quality  # noqa: F401
from .export import frames_rgb8  # noqa: F401

__all__ = ["GaussianRasterizationSettings", "GaussianRasterizer", "RasterizerError", "frame_quality", "frames_rgb8"]
