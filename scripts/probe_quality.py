"""Fused frame quality metrics (gsvc_b200.quality) against fp32 PyTorch restatements, on one GPU.

  1. per case ([1,3,1080,1920], [8,3,1080,1920], [1,3,2160,3840]): the fused frame_quality (PSNR + SSIM + MS-SSIM);
     the fused loss forward (photometric_loss, the same window pass without pyramid) for scale; SSIM as the upstream
     3DGS ssim (F.conv2d, 11x11 window, padding 5); MS-SSIM as pytorch_msssim writes it (grouped separable conv2d,
     valid, + avg_pool2d); PSNR on the device and reference-shaped (device-to-host copy of the frame, numpy in double);
  2. FrameStreamer decode alone against decode + quality= (one [F,3] result, one synchronisation), frames/s, at the
     sizes of configs 2 and 4 (1080p, 200 k and 1 M Gaussians);
  3. the largest difference of the fused metrics and of the fp32 restatements from the float64 oracle.

CUDA events, warm-up first, arms alternated window by window; the median over windows is reported.  Inputs are not
flushed from the 126 MB L2 between calls: a 1080p pair (50 MB) stays resident, 8 pairs (398 MB) and a 4K pair
(199 MB) do not.  The card's name and power limit are read (a query) in the same run.

    python scripts/probe_quality.py [--out profiles/r8_quality.json] [--windows 7]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(ROOT)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from gsvc_b200 import _lib, frame_quality  # noqa: E402
from gsvc_b200.loss import photometric_loss  # noqa: E402
from probe_loss import ab, card  # noqa: E402
from tests import loss_oracle, quality_oracle  # noqa: E402

L2_BYTES = 126 * 2 ** 20


def torch_ssim(x, y, win2d):
    return loss_oracle.ssim_map(x.clamp(0, 1), y, window=win2d).mean(dim=(1, 2, 3))


def torch_ms_ssim(x, y, g1d):
    """pytorch_msssim.ms_ssim(X, Y, data_range=1, size_average=False) restated: separable valid Gaussian filter as two
    grouped conv2d, E[x^2] - mu^2 moments, avg_pool2d with padding (h % 2, w % 2) between levels."""
    wh = g1d.view(1, 1, 1, 11).expand(3, 1, 1, 11)
    wv = g1d.view(1, 1, 11, 1).expand(3, 1, 11, 1)
    filt = lambda a: F.conv2d(F.conv2d(a, wv, groups=3), wh, groups=3)
    w = torch.tensor(quality_oracle.WEIGHTS, dtype=x.dtype, device=x.device)
    x = x.clamp(0, 1)
    mcs = []
    for l in range(5):
        mx, my = filt(x), filt(y)
        sxx, syy, sxy = filt(x * x) - mx * mx, filt(y * y) - my * my, filt(x * y) - mx * my
        cs_map = (2 * sxy + loss_oracle.C2) / (sxx + syy + loss_oracle.C2)
        ssim_map = (2 * mx * my + loss_oracle.C1) / (mx * mx + my * my + loss_oracle.C1) * cs_map
        if l < 4:
            mcs.append(torch.relu(cs_map.flatten(2).mean(-1)))
            h, wd = x.shape[-2:]
            x = F.avg_pool2d(x, 2, padding=(h % 2, wd % 2))
            y = F.avg_pool2d(y, 2, padding=(h % 2, wd % 2))
    ss = torch.relu(ssim_map.flatten(2).mean(-1))
    vals = torch.stack(mcs + [ss], dim=0)
    return torch.prod(vals ** w.view(-1, 1, 1), dim=0).mean(dim=1)


def torch_psnr_device(x, y):
    return 10 * torch.log10(1.0 / ((x.clamp(0, 1) - y) ** 2).mean(dim=(1, 2, 3)))


def psnr_host(x, y):
    """Reference-shaped: the frame is copied to the host and PSNR runs in numpy float64 (skimage's arithmetic)."""
    xh, yh = x.clamp(0, 1).cpu().numpy().astype(np.float64), y.cpu().numpy().astype(np.float64)
    return [10 * np.log10(1.0 / np.mean((a - b) ** 2)) for a, b in zip(xh, yh)]


def metrics_case(shape, dev, windows):
    g = torch.Generator().manual_seed(1)
    x = torch.rand(shape, generator=g).to(dev)
    y = (0.7 * x + 0.3 * torch.rand(shape, generator=g).to(dev)).contiguous()
    win2d = loss_oracle.create_window(dtype=torch.float32).to(dev)
    g1d = loss_oracle.gaussian(dtype=torch.float32).to(dev)
    arms = {
        "fused_frame_quality": lambda: frame_quality(x, y),
        "fused_loss_forward": lambda: photometric_loss(x, y, 0.2),
        "torch_ssim": lambda: torch_ssim(x, y, win2d),
        "torch_ms_ssim": lambda: torch_ms_ssim(x, y, g1d),
        "torch_psnr_device": lambda: torch_psnr_device(x, y),
        "psnr_host_numpy": lambda: psnr_host(x, y),
    }
    n = shape[0]
    iters = 5 if n * shape[2] * shape[3] >= 4_000_000 else 20
    with torch.no_grad():
        t = ab(arms, iters, windows)
    for k in t:
        t[k]["median_ms_per_image"] = t[k]["median_ms"] / n
    t["torch_ssim_ms_ssim_psnr_total_ms"] = (t["torch_ssim"]["median_ms"] + t["torch_ms_ssim"]["median_ms"]
                                             + t["psnr_host_numpy"]["median_ms"])
    t["fused_over_loss_forward"] = t["fused_frame_quality"]["median_ms"] / t["fused_loss_forward"]["median_ms"]
    with torch.no_grad():
        q = frame_quality(x, y).double()
        ref = quality_oracle.frame_quality(x.double(), y.double())
        t32 = torch.stack([torch_psnr_device(x, y), torch_ssim(x, y, win2d), torch_ms_ssim(x, y, g1d)], 1).double()
    acc = {f"{name}_{col}": (v[:, i] - ref[:, i]).abs().max().item()
           for name, v in (("fused_minus_float64", q), ("torch32_minus_float64", t32))
           for i, col in enumerate(("psnr_db", "ssim", "ms_ssim"))}
    acc["float64"] = ref.cpu().tolist()
    pair = 2 * x.numel() * 4
    del ref, t32
    torch.cuda.empty_cache()
    return dict(shape=list(shape), input_pair_bytes=pair, l2_resident=pair <= L2_BYTES, iters_per_window=iters,
                **t, accuracy=acc)


def streamer_case(config, dev, windows, frames=64):
    from bench import THRESHOLD, settings_for
    from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians
    from gsvc_b200.graphed import FrameStreamer
    cfg = CONFIGS[config]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    params = synthetic_gaussians(cfg["P"], geom, f0, f0 + frames - 1, threshold=THRESHOLD, seed=2, device=dev)
    sets = [(settings_for(geom, f, dev), settings_for(geom, f, dev, back=True)) for f in range(f0, f0 + frames)]
    streamer = FrameStreamer(sets[0][0], sets[0][1], params, n_streams=4)
    targets = torch.rand((frames, 3, cfg["H"], cfg["W"]), generator=torch.Generator().manual_seed(5)).to(dev)
    q = torch.empty((frames, 3), device=dev)

    def decode():
        for i, (a, b) in enumerate(sets):
            streamer.render(a.viewmatrix, b.viewmatrix)
        for s in streamer.streams:
            torch.cuda.current_stream(dev).wait_stream(s)

    def decode_eval():
        for i, (a, b) in enumerate(sets):
            streamer.render(a.viewmatrix, b.viewmatrix, target=targets[i], quality=q[i])
        for s in streamer.streams:
            torch.cuda.current_stream(dev).wait_stream(s)

    t = ab({"decode": decode, "decode_plus_quality": decode_eval}, 1, windows)
    torch.cuda.synchronize()
    out = dict(P=cfg["P"], H=cfg["H"], W=cfg["W"], frames_per_call=frames, n_streams=4,
               capacity_ok=bool(streamer.capacity_ok()))
    for k, v in t.items():
        out[k] = dict(frames_per_s=frames / (v["median_ms"] * 1e-3), ms_per_frame=v["median_ms"] / frames, **v)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r8_quality.json"))
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_quality measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    _lib.lib()
    out = dict(card=card(), windows=args.windows)
    out["1080p_x1"] = metrics_case((1, 3, 1080, 1920), dev, args.windows)
    out["1080p_x8"] = metrics_case((8, 3, 1080, 1920), dev, args.windows)
    out["4k_x1"] = metrics_case((1, 3, 2160, 3840), dev, args.windows)
    out["streamer_config2"] = streamer_case(2, dev, args.windows)
    out["streamer_config4"] = streamer_case(4, dev, args.windows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: v for k, v in out.items()}, indent=1)[:6000])


if __name__ == "__main__":
    main()
