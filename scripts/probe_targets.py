"""8-bit source frames as targets (SPEC U12) against fp32 targets, on one GPU.

  1. the fused loss, forward + backward at [2,3,1080,1920], and the quality metrics at [8,3,1080,1920]: fp32 targets
     against a uint8 cube with a device index.  Each arm cycles through RING input sets (images and targets) so that
     its working set exceeds the 126 MB L2: the inputs are not L2-resident between calls;
  2. config 2's graphed two-frame training step (ViewBatch.toasts, GraphedStep with the fused loss): the iteration's
     two fp32 target frames gathered from a resident fp32 cube into the static target (index_select into it, 49.8 MB)
     against a resident uint8 cube whose static int32 index gets an 8-byte in-place write;
  3. decode + evaluate with FrameStreamer(n_streams=4) at configs 2 and 4, 64 frames per synchronisation, each frame
     with its own target: device-resident fp32; pinned host fp32 (uploaded by the caller on the current stream into a
     ring of device frames, the only way fp32 targets reach the streamer); pinned host uint8 (render's own upload);
     pinned host uint8 with host_out as well (both directions of the link); decode alone for reference.  And the bare
     host-to-device copy of one 8-bit and one fp32 1080p frame from pinned memory.

CUDA events, warm-up first, arms alternated window by window; the median over windows is reported.  The card's name
and power limit are read (a query) in the same run.

    python scripts/probe_targets.py [--out profiles/r11_targets.json] [--windows 7]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import torch  # noqa: E402

from gsvc_b200 import _lib, frame_quality  # noqa: E402
from gsvc_b200 import targets as T8  # noqa: E402
from gsvc_b200.loss import photometric_loss  # noqa: E402
from probe_loss import ab, card  # noqa: E402

L2_BYTES = 126 * 2 ** 20
LAM = 0.2
RING = 4


def _inputs(N, H, W, dev, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.rand((N, 3, H, W), generator=g).to(dev)
    cube = torch.randint(0, 256, (N + 2, H, W, 3), dtype=torch.uint8, generator=g).to(dev)
    index = torch.arange(N, 0, -1, dtype=torch.int32).add_(1).to(dev)          # frames N+1 .. 2
    return x, cube, index, T8.to_float(cube, index)


def kernel_case(dev, windows):
    out = {}
    N, H, W = 2, 1080, 1920
    sets = [_inputs(N, H, W, dev, s) for s in range(RING)]
    leaves = [s[0].clone().requires_grad_(True) for s in sets]
    it = {"i": 0}

    def loss_arm(rgb8):
        def run():
            k = it["i"] % RING
            it["i"] += 1
            x, cube, index, y = sets[k]
            loss = photometric_loss(leaves[k], cube, LAM, index=index) if rgb8 else photometric_loss(leaves[k], y, LAM)
            torch.autograd.grad(loss.sum(), leaves[k])
        return run
    t = ab({"fp32_target": loss_arm(False), "uint8_cube": loss_arm(True)}, 20, windows)
    ok = all(torch.equal(photometric_loss(s[0], s[1], LAM, index=s[2]), photometric_loss(s[0], s[3], LAM))
             for s in sets)
    per_set = N * 3 * H * W * 4 * 2
    out["loss_fwd_bwd_2x1080p"] = dict(shape=[N, 3, H, W], ring=RING, working_set_bytes_fp32=RING * per_set,
                                       l2_resident=RING * per_set <= L2_BYTES, loss_equal=ok,
                                       uint8_over_fp32=t["uint8_cube"]["median_ms"] / t["fp32_target"]["median_ms"],
                                       **t)
    del sets, leaves
    N = 8
    sets = [_inputs(N, H, W, dev, 10 + s) for s in range(RING)]

    def q_arm(rgb8):
        def run():
            k = it["i"] % RING
            it["i"] += 1
            x, cube, index, y = sets[k]
            frame_quality(x, cube, index=index) if rgb8 else frame_quality(x, y)
        return run
    t = ab({"fp32_target": q_arm(False), "uint8_cube": q_arm(True)}, 10, windows)
    ok = all(torch.equal(frame_quality(s[0], s[1], index=s[2]), frame_quality(s[0], s[3])) for s in sets)
    per_set = N * 3 * H * W * 4 * 2
    out["quality_8x1080p"] = dict(shape=[N, 3, H, W], ring=RING, working_set_bytes_fp32=RING * per_set,
                                  l2_resident=False, quality_equal=ok,
                                  uint8_over_fp32=t["uint8_cube"]["median_ms"] / t["fp32_target"]["median_ms"], **t)
    return out


def _scene(config, dev, frames):
    from bench import THRESHOLD, settings_for
    from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians
    cfg = CONFIGS[config]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    params = synthetic_gaussians(cfg["P"], geom, f0, f0 + frames - 1, threshold=THRESHOLD, seed=2, device=dev)
    sets = [(settings_for(geom, f, dev), settings_for(geom, f, dev, back=True)) for f in range(f0, f0 + frames)]
    return cfg, params, sets


def train_case(dev, windows, F=64, iters=20):
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.views import ViewBatch
    cfg, params, sets = _scene(2, dev, 2)
    H, W = cfg["H"], cfg["W"]
    params = {k: params[k].contiguous().clone() for k in ("means3D", "colors_precomp", "opacities", "scales",
                                                          "rotations")}
    batch = ViewBatch.toasts(sets)
    g = torch.Generator().manual_seed(5)
    cube8 = torch.randint(0, 256, (F, H, W, 3), dtype=torch.uint8, generator=g).to(dev)
    cube32 = T8.to_float(cube8)                                                # [F,3,H,W] resident fp32
    pairs = torch.randint(0, F, (iters, 2), dtype=torch.int32, generator=g).to(dev)
    pairs64 = pairs.long()
    tgt = torch.empty((2, 3, H, W), device=dev)
    index = torch.zeros(2, dtype=torch.int32, device=dev)
    step32 = GraphedStep(batch, params, None, loss_target=tgt, lambda_dssim=LAM)
    step8 = GraphedStep(batch, params, None, loss_target=cube8, loss_index=index, lambda_dssim=LAM)
    it = {"a": 0, "b": 0}

    def fp32_copy():
        i = it["a"] % iters
        it["a"] += 1
        torch.index_select(cube32, 0, pairs64[i], out=tgt)
        step32()

    def uint8_index():
        i = it["b"] % iters
        it["b"] += 1
        index.copy_(pairs[i], non_blocking=True)
        step8()
    t = ab({"fp32_cube_copy": fp32_copy, "uint8_cube_index_write": uint8_index}, iters, windows)
    torch.cuda.synchronize()
    same = True
    for i in range(3):
        torch.index_select(cube32, 0, pairs64[i], out=tgt)
        step32()
        index.copy_(pairs[i])
        step8()
        torch.cuda.synchronize()
        same = same and torch.equal(step32.loss, step8.loss)
    return dict(P=cfg["P"], H=H, W=W, resident_frames=F, fp32_cube_bytes=cube32.numel() * 4,
                uint8_cube_bytes=cube8.numel(), target_bytes_copied_per_step_fp32=2 * 3 * H * W * 4,
                loss_equal=bool(same), capacity_ok=bool(step32.capacity_ok() and step8.capacity_ok()),
                uint8_over_fp32=t["uint8_cube_index_write"]["median_ms"] / t["fp32_cube_copy"]["median_ms"], **t)


def h2d_case(windows):
    H, W = 1080, 1920
    arms, sizes = {}, {}
    for name, shape, dtype in (("rgb8_6.2MB", (H, W, 3), torch.uint8), ("fp32_24.9MB", (3, H, W), torch.float32)):
        d = torch.empty(shape, dtype=dtype, device="cuda")
        h = torch.ones(shape, dtype=dtype).pin_memory()
        sizes[name] = d.numel() * d.element_size()
        arms[name] = (lambda d=d, h=h: d.copy_(h, non_blocking=True))
    t = ab(arms, 64, windows)
    for name, n in sizes.items():
        t[name]["bytes"] = n
        t[name]["bytes_per_s"] = n / (t[name]["median_ms"] * 1e-3)
        t[name]["frames_per_s"] = 1e3 / t[name]["median_ms"]
    return t


def streamer_case(config, dev, windows, frames=64):
    from gsvc_b200.graphed import FrameStreamer
    cfg, params, sets = _scene(config, dev, frames)
    H, W = cfg["H"], cfg["W"]
    n = 4
    streamer = FrameStreamer(sets[0][0], sets[0][1], params, n_streams=n)
    ring = 2 * n
    g = torch.Generator().manual_seed(7)
    src8 = [torch.randint(0, 256, (H, W, 3), dtype=torch.uint8, generator=g) for _ in range(frames)]
    dev32 = [T8.to_float(s[None].to(dev))[0] for s in src8]                    # device-resident fp32 targets
    host8 = [s.pin_memory() for s in src8]
    host32 = [d.cpu().pin_memory() for d in dev32]
    up32 = [torch.empty((3, H, W), device=dev) for _ in range(ring)]
    up_done = [None] * ring
    outs = [torch.empty((H, W, 3), dtype=torch.uint8).pin_memory() for _ in range(ring)]
    q = torch.empty((frames, 3), device=dev)
    cur = torch.cuda.current_stream(dev)

    def join():
        for s in streamer.streams:
            cur.wait_stream(s)
        for s in (streamer.copy_stream, streamer.upload_stream):
            if s is not None:
                cur.wait_stream(s)

    def decode():
        for a, b in sets:
            streamer.render(a.viewmatrix, b.viewmatrix)
        join()

    def device_fp32():
        for i, (a, b) in enumerate(sets):
            streamer.render(a.viewmatrix, b.viewmatrix, target=dev32[i], quality=q[i])
        join()

    def host_fp32():                         # the caller uploads each fp32 frame on the current stream
        for i, (a, b) in enumerate(sets):
            j = i % ring
            if up_done[j] is not None:
                cur.wait_event(up_done[j])   # the quality pass that read this device frame
            up32[j].copy_(host32[i], non_blocking=True)
            streamer.render(a.viewmatrix, b.viewmatrix, target=up32[j], quality=q[i])
            up_done[j] = streamer.last_event()
        join()

    def host_uint8():
        for i, (a, b) in enumerate(sets):
            streamer.render(a.viewmatrix, b.viewmatrix, target=host8[i], quality=q[i])
        join()

    def host_uint8_out():
        for i, (a, b) in enumerate(sets):
            streamer.render(a.viewmatrix, b.viewmatrix, target=host8[i], quality=q[i], host_out=outs[i % ring])
        join()

    arms = {"decode": decode, "device_fp32": device_fp32, "host_fp32": host_fp32, "host_uint8": host_uint8,
            "host_uint8_host_out": host_uint8_out}
    t = ab(arms, 1, windows)
    torch.cuda.synchronize()
    rows = {}
    for name in ("device_fp32", "host_fp32", "host_uint8", "host_uint8_host_out"):
        q.fill_(-1.0)
        arms[name]()
        torch.cuda.synchronize()
        rows[name] = q.clone()
    same = all(torch.equal(rows[k], rows["device_fp32"]) for k in rows)
    out = dict(P=cfg["P"], H=H, W=W, frames_per_call=frames, n_streams=n, quality_rows_equal=bool(same),
               capacity_ok=bool(streamer.capacity_ok()))
    for k, v in t.items():
        out[k] = dict(frames_per_s=frames / (v["median_ms"] * 1e-3), ms_per_frame=v["median_ms"] / frames, **v)
    dev_rate = out["device_fp32"]["frames_per_s"]
    for k in ("host_fp32", "host_uint8", "host_uint8_host_out"):
        out[k]["share_of_device_fp32"] = out[k]["frames_per_s"] / dev_rate
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r11_targets.json"))
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_targets measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    _lib.lib()
    out = dict(card=card(), windows=args.windows)
    out.update(kernel_case(dev, args.windows))
    torch.cuda.empty_cache()
    out["train_step_config2"] = train_case(dev, args.windows)
    torch.cuda.empty_cache()
    with torch.no_grad():
        out["h2d_copy"] = h2d_case(args.windows)
        for c in (2, 4):
            out[f"streamer_config{c}"] = streamer_case(c, dev, args.windows)
            torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1)[:6000])


if __name__ == "__main__":
    main()
