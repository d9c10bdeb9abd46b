"""Fused L1 + D-SSIM loss (gsvc_b200.loss) against the fp32 PyTorch expression of upstream 3DGS, on one GPU.

  1. the loss alone, forward and forward + backward, at [2,3,1080,1920] (inputs 100 MB: they stay in the 126 MB L2
     between calls) and [1,3,2160,3840] (199 MB: they do not);
  2. config 2's two-frame training iteration (ViewBatch.toasts: render + loss + backward of the Gaussian parameters)
     with each loss, eager and captured in a CUDA graph (GraphedStep(loss_target=) for the fused loss, the same
     capture by hand for the PyTorch expression), beside today's graphed step seeded with a fixed dL;
  3. bytes and FMAs per value of the built kernels, counted from their tile shapes;
  4. the largest difference of the fused loss and gradient from the fp32 PyTorch expression and from float64.

CUDA events, warm-up first, arms alternated window by window; the median over windows is reported.  The PyTorch arm
builds its Gaussian window once (upstream rebuilds it and copies it to the GPU on every call).  The card's name and
power limit are read (a query) in the same run.

    python scripts/probe_loss.py [--out profiles/r7_loss.json] [--windows 7]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from gsvc_b200 import _lib  # noqa: E402
from gsvc_b200.loss import photometric_loss  # noqa: E402
from tests import loss_oracle  # noqa: E402

LAM = 0.2


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:        # the numbers stay valid, the card is then only what torch reports
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def ab(arms: dict, iters: int, windows: int) -> dict:
    """ms per call of each arm: `windows` rounds, each timing `iters` back-to-back calls of every arm in turn."""
    for fn in arms.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    res = {k: [] for k in arms}
    for _ in range(windows):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                fn()
            b.record()
            b.synchronize()
            res[k].append(a.elapsed_time(b) / iters)
    return {k: dict(median_ms=statistics.median(v), min_ms=min(v), max_ms=max(v)) for k, v in res.items()}


def loss_alone(shape, dev, windows):
    g = torch.Generator().manual_seed(1)
    x = torch.rand(shape, generator=g).to(dev)
    y = (0.7 * x + 0.3 * torch.rand(shape, generator=g).to(dev)).contiguous()
    win = loss_oracle.create_window(dtype=torch.float32).to(dev)
    xl = x.clone().requires_grad_(True)
    ones = torch.ones(shape[0], device=dev)

    def f_fwd():
        return photometric_loss(x, y, LAM)

    def t_fwd():
        return loss_oracle.photometric_loss(x, y, LAM, window=win)

    def f_both():
        return torch.autograd.grad(photometric_loss(xl, y, LAM), xl, grad_outputs=ones)[0]

    def t_both():
        return torch.autograd.grad(loss_oracle.photometric_loss(xl, y, LAM, window=win), xl, grad_outputs=ones)[0]

    iters = 20 if shape[0] * shape[2] * shape[3] >= 4_000_000 else 50
    with torch.no_grad():
        t1 = ab({"fused_forward": f_fwd, "torch_forward": t_fwd}, iters, windows)
    t2 = ab({"fused_forward_backward": f_both, "torch_forward_backward": t_both}, iters, windows)
    # accuracy at this size: fused and fp32 PyTorch against float64 (on the GPU)
    lf, gf = photometric_loss(xl, y, LAM), f_both()
    lt, gt = loss_oracle.photometric_loss(xl, y, LAM, window=win), t_both()
    xd = x.double().requires_grad_(True)
    ld = loss_oracle.photometric_loss(xd, y.double(), LAM)
    (gd,) = torch.autograd.grad(ld, xd, grad_outputs=ones.double())
    gmax = gd.abs().amax().item()
    acc = dict(
        loss_fused_minus_torch32=(lf - lt).abs().max().item(),
        grad_fused_minus_torch32_max=(gf - gt).abs().max().item(),
        loss_fused_minus_float64=(lf.double() - ld).abs().max().item(),
        loss_torch32_minus_float64=(lt.double() - ld).abs().max().item(),
        grad_fused_minus_float64_rel_to_max=(gf.double() - gd).abs().max().item() / gmax,
        grad_torch32_minus_float64_rel_to_max=(gt.double() - gd).abs().max().item() / gmax,
        max_abs_grad_float64=gmax)
    del xd, ld, gd
    torch.cuda.empty_cache()
    return dict(shape=list(shape), input_bytes=2 * x.numel() * 4, iters_per_window=iters, **t1, **t2, accuracy=acc)


def counts():
    """Per value (pixel x channel) of the built kernels (csrc/loss.cu: 32x32 tiles, RUN 4)."""
    T, R = 32, 5
    fwd_h = (T + 2 * R) * T * 5 * 11          # horizontal pass: 42 rows x 32 columns x 5 signals x 11 taps
    fwd_v = T * T * 5 * 11
    bw = 44
    bwd_h5 = (bw + 2 * R) * bw * 5 * 11       # moments on the 44 x 44 map region (42 x 42 used)
    bwd_v5 = bw * bw * 5 * 11
    bwd_h3 = (T + 2 * R) * T * 3 * 11         # correlation of the three maps
    bwd_v3 = T * T * 3 * 11
    px = T * T
    return dict(
        forward_window_fma_per_value=(fwd_h + fwd_v) / px,
        backward_window_fma_per_value=(bwd_h5 + bwd_v5 + bwd_h3 + bwd_v3) / px,
        forward_dram_bytes_per_value=8,        # x and y once (the halo re-reads hit L2)
        backward_dram_bytes_per_value=12,      # x and y once, dL/dx written once
        forward_staged_reads_per_value=2 * (T + 2 * R) ** 2 / px,
        backward_staged_reads_per_value=2 * (bw + 2 * R) ** 2 / px,
        torch_forward_intermediates_fp32=27)


def step_arms(dev, windows):
    from bench import build_scene, settings_for
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.sharding import GRAD_LAYOUT
    from gsvc_b200.views import ViewBatch, rasterize_views
    cfg, geom, f0, g = build_scene(2, dev)
    batch = ViewBatch.toasts([(settings_for(geom, f, dev), settings_for(geom, f, dev, back=True)) for f in (f0, f0 + 1)])
    params = {k: g[k].contiguous().clone() for k, _ in GRAD_LAYOUT}
    with torch.no_grad():
        target, _, _ = rasterize_views(batch, **{k: (v * 1.01 if k == "means3D" else v) for k, v in params.items()})
    target = target.contiguous()
    win = loss_oracle.create_window(dtype=torch.float32).to(dev)

    def eager(loss_fn):
        def run():
            leaves = {k: params[k].detach().requires_grad_(True) for k, _ in GRAD_LAYOUT}
            color, _, _ = rasterize_views(batch, **leaves)
            torch.autograd.grad(loss_fn(color).mean(), [leaves[k] for k, _ in GRAD_LAYOUT])
        return run

    fused = lambda c: photometric_loss(c, target, LAM)
    torch_loss = lambda c: loss_oracle.photometric_loss(c, target, LAM, window=win)
    step_fused = GraphedStep(batch, params, None, loss_target=target, lambda_dssim=LAM)
    dL = torch.randn(target.shape, generator=torch.Generator().manual_seed(3)).to(dev)
    step_dl = GraphedStep(batch, params, dL)
    # the PyTorch expression captured the same way (GraphedStep's loss is the fused one)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            eager(torch_loss)()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph_torch = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph_torch):
        eager(torch_loss)()
    arms = {"eager_fused_loss": eager(fused), "eager_torch_loss": eager(torch_loss),
            "graphed_fused_loss": step_fused, "graphed_torch_loss": graph_torch.replay,
            "graphed_fixed_dL_no_loss": step_dl}
    res = ab(arms, 20, windows)
    torch.cuda.synchronize()
    res["capacity_ok"] = bool(step_fused.capacity_ok() and step_dl.capacity_ok())
    res["scene"] = dict(P=cfg["P"], H=cfg["H"], W=cfg["W"], frames=2, views=4)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_loss.json"))
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_loss measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    _lib.lib()
    out = dict(card=card(), lambda_dssim=LAM, windows=args.windows, counts=counts(),
               note="1080p inputs fit the 126 MB L2 and are not flushed between calls; 4K inputs do not fit")
    out["loss_1080p_x2"] = loss_alone((2, 3, 1080, 1920), dev, args.windows)
    out["loss_4k_x1"] = loss_alone((1, 3, 2160, 3840), dev, args.windows)
    out["config2_two_frame_step"] = step_arms(dev, args.windows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
