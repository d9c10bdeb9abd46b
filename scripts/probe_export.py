"""8-bit frame export (gsvc_b200.frames_rgb8) and decode-to-host through FrameStreamer, on one GPU.

  1. per case ([1,3,1080,1920], [8,3,1080,1920], [1,3,2160,3840]): the frames_rgb8 kernel against the PyTorch
     expression it replaces (mul, add_, clamp_, permute, cast to uint8, made contiguous), ms per call and the achieved
     bytes/s of the kernel (12 bytes read + 3 written per pixel) against the 7.7 TB/s of the data sheet; the same call
     into an output 1 byte off alignment, which takes the scalar path, shows what the float4 path is worth;
  2. a bare device-to-host copy into pinned memory of one 8-bit 1080p frame (6.2 MB) and of one fp32 frame (24.9 MB):
     the link's ceiling in this run;
  3. FrameStreamer at the sizes of configs 2 and 4 (1080p, 200 k and 1 M Gaussians), 4 streams, 64 frames per
     synchronisation, frames/s of: decode alone; decode + 8-bit export to pinned host as the library does it
     (render(host_out=): conversion on the frame's stream, copy on one device-to-host stream, a ring of 2 x n_streams
     staging buffers, event-ordered); the same with the copy on the frame's own stream (the simpler alternative the
     library does not ship); decode + the fp32 frame copied to pinned host; decode + the PyTorch expression and a
     non-blocking copy.
     Pinned host buffers: a ring of 2 x n_streams frames, overwritten (nothing reads them during the timing).

CUDA events, warm-up first, arms alternated window by window; the median over windows is reported.  The kernel's input
is not flushed from the 126 MB L2 between calls: one 1080p frame (24.9 MB) and one 4K frame (99.5 MB) stay resident,
8 frames (199 MB) do not.  The card's name and power limit are read (a query) in the same run.

    python scripts/probe_export.py [--out profiles/r9_export.json] [--windows 7]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(ROOT)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from gsvc_b200 import _lib, frames_rgb8  # noqa: E402
from gsvc_b200.export import rgb8_into  # noqa: E402
from probe_loss import ab, card  # noqa: E402

L2_BYTES = 126 * 2 ** 20
HBM_BYTES_PER_S = 7.7e12


def torch_expression(x):
    return x.mul(255).add_(0.5).clamp_(0, 255).permute(0, 2, 3, 1).to(torch.uint8).contiguous()


def kernel_case(shape, dev, windows):
    x = (torch.rand(shape, generator=torch.Generator().manual_seed(1)) * 1.2 - 0.1).to(dev)
    out = torch.empty((shape[0], shape[2], shape[3], 3), dtype=torch.uint8, device=dev)
    # an output 1 byte off a 4-byte boundary sends the same call down the scalar (byte-store) path
    odd = torch.empty(out.numel() + 1, dtype=torch.uint8, device=dev)[1:].view(out.shape)
    arms = {"frames_rgb8": lambda: frames_rgb8(x, out=out), "frames_rgb8_scalar_path": lambda: frames_rgb8(x, out=odd),
            "torch_expression": lambda: torch_expression(x)}
    iters = 50 if shape[0] * shape[2] * shape[3] >= 4_000_000 else 200
    t = ab(arms, iters, windows)
    same = bool(torch.equal(frames_rgb8(x), torch_expression(x)) and torch.equal(odd, out))
    px = shape[0] * shape[2] * shape[3]
    moved = px * (12 + 3)
    k = t["frames_rgb8"]
    k["bytes_moved"] = moved
    k["achieved_bytes_per_s"] = moved / (k["median_ms"] * 1e-3)
    k["share_of_7_7_TBps"] = k["achieved_bytes_per_s"] / HBM_BYTES_PER_S
    t["torch_over_kernel"] = t["torch_expression"]["median_ms"] / k["median_ms"]
    t["scalar_path_over_vector_path"] = t["frames_rgb8_scalar_path"]["median_ms"] / k["median_ms"]
    return dict(shape=list(shape), input_bytes=px * 12, input_l2_resident=px * 12 <= L2_BYTES, iters_per_window=iters,
                equal_to_torch_expression=same, **t)


def copy_case(dev, windows):
    H, W = 1080, 1920
    arms = {}
    bufs = {}
    for name, shape, dtype in (("rgb8_6.2MB", (H, W, 3), torch.uint8), ("fp32_24.9MB", (3, H, W), torch.float32)):
        d = torch.ones(shape, dtype=dtype, device=dev)
        h = torch.empty(shape, dtype=dtype).pin_memory()
        bufs[name] = (d, h)
        arms[name] = (lambda d=d, h=h: h.copy_(d, non_blocking=True))
    t = ab(arms, 64, windows)
    for name, (d, h) in bufs.items():
        nbytes = d.numel() * d.element_size()
        t[name]["bytes"] = nbytes
        t[name]["bytes_per_s"] = nbytes / (t[name]["median_ms"] * 1e-3)
        t[name]["frames_per_s"] = 1e3 / t[name]["median_ms"]
    return t


def streamer_case(config, dev, windows, frames=64):
    from bench import THRESHOLD, settings_for
    from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians
    from gsvc_b200.graphed import FrameStreamer
    cfg = CONFIGS[config]
    H, W = cfg["H"], cfg["W"]
    geom = CubeGeometry(W, H, cfg["F"])
    f0 = cfg["F"] // 2
    params = synthetic_gaussians(cfg["P"], geom, f0, f0 + frames - 1, threshold=THRESHOLD, seed=2, device=dev)
    sets = [(settings_for(geom, f, dev), settings_for(geom, f, dev, back=True)) for f in range(f0, f0 + frames)]
    n = 4
    streamer = FrameStreamer(sets[0][0], sets[0][1], params, n_streams=n)
    ring = 2 * n
    host8 = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(ring)]
    host32 = [torch.empty((3, H, W), dtype=torch.float32).pin_memory() for _ in range(ring)]
    stage = [torch.empty((H, W, 3), dtype=torch.uint8, device=dev) for _ in range(n)]
    cur = torch.cuda.current_stream(dev)

    def join():
        for s in streamer.streams:
            cur.wait_stream(s)

    def decode():
        for a, b in sets:
            streamer.render(a.viewmatrix, b.viewmatrix)
        join()

    def host_copy_stream():                          # the library's path
        for i, (a, b) in enumerate(sets):
            streamer.render(a.viewmatrix, b.viewmatrix, host_out=host8[i % ring])
        join()
        cur.wait_stream(streamer.copy_stream)

    def host_same_stream():                          # the alternative: conversion and copy on the frame's stream
        for i, (a, b) in enumerate(sets):
            k = streamer.i % n
            img = streamer.render(a.viewmatrix, b.viewmatrix)
            with torch.cuda.stream(streamer.streams[k]):
                rgb8_into(stage[k], img.unsqueeze(0))
                host8[i % ring].copy_(stage[k], non_blocking=True)
        join()

    def host_fp32():
        for i, (a, b) in enumerate(sets):
            k = streamer.i % n
            img = streamer.render(a.viewmatrix, b.viewmatrix)
            with torch.cuda.stream(streamer.streams[k]):
                host32[i % ring].copy_(img, non_blocking=True)
        join()

    def host_torch_expression():
        for i, (a, b) in enumerate(sets):
            k = streamer.i % n
            img = streamer.render(a.viewmatrix, b.viewmatrix)
            with torch.cuda.stream(streamer.streams[k]):
                host8[i % ring].copy_(img.mul(255).add_(0.5).clamp_(0, 255).permute(1, 2, 0).to(torch.uint8),
                                      non_blocking=True)
        join()

    arms = {"decode": decode, "decode_rgb8_host_copy_stream": host_copy_stream,
            "decode_rgb8_host_same_stream": host_same_stream, "decode_fp32_host": host_fp32,
            "decode_torch_expression_host": host_torch_expression}
    t = ab(arms, 1, windows)
    torch.cuda.synchronize()
    # the last window's host frames of both 8-bit paths against frames_rgb8 of the same views (frame 63 -> slot 7)
    host_same_stream()
    torch.cuda.synchronize()
    a, b = sets[-1]
    img = streamer.render(a.viewmatrix, b.viewmatrix)
    streamer.wait()
    ref = frames_rgb8(img)
    torch.cuda.synchronize()
    ok_same = bool(torch.equal(host8[(frames - 1) % ring], ref.cpu()))
    host_copy_stream()
    torch.cuda.synchronize()
    ok_copy = bool(torch.equal(host8[(frames - 1) % ring], ref.cpu()))
    out = dict(P=cfg["P"], H=H, W=W, frames_per_call=frames, n_streams=n, host_ring=ring,
               capacity_ok=bool(streamer.capacity_ok()), host_frame_equals_frames_rgb8=dict(
                   same_stream=ok_same, copy_stream=ok_copy))
    for k, v in t.items():
        out[k] = dict(frames_per_s=frames / (v["median_ms"] * 1e-3), ms_per_frame=v["median_ms"] / frames, **v)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r9_export.json"))
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_export measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    _lib.lib()
    out = dict(card=card(), windows=args.windows)
    with torch.no_grad():
        out["kernel_1080p_x1"] = kernel_case((1, 3, 1080, 1920), dev, args.windows)
        out["kernel_1080p_x8"] = kernel_case((8, 3, 1080, 1920), dev, args.windows)
        out["kernel_4k_x1"] = kernel_case((1, 3, 2160, 3840), dev, args.windows)
        out["pinned_copy"] = copy_case(dev, args.windows)
        link8 = out["pinned_copy"]["rgb8_6.2MB"]["frames_per_s"]
        for c in (2, 4):
            s = streamer_case(c, dev, args.windows)
            dec = s["decode"]["frames_per_s"]
            s["rgb8_link_ceiling_frames_per_s"] = link8
            s["bar_90pct_of_min_decode_link"] = 0.9 * min(dec, link8)
            for arm in ("decode_rgb8_host_same_stream", "decode_rgb8_host_copy_stream"):
                s[arm]["share_of_min_decode_link"] = s[arm]["frames_per_s"] / min(dec, link8)
            out[f"streamer_config{c}"] = s
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1)[:8000])


if __name__ == "__main__":
    main()
