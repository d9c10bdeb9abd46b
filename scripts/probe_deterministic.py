"""The deterministic blend backward (docs/SPEC.md U14) against the default atomic one, on one GPU.

Workloads:
  1. config 2's graphed two-view step: ViewBatch.toast of one frame, forward + backward replayed from a GraphedStep
     (one graph captured per mode: the mode is fixed at capture);
  2. the reference's 4-view training iteration with the fused loss: four views with Gaussian sets of their own
     (ragged, ViewBatch.toasts of two frames), photometric_loss, eager;
  3. config 5 per view: 2 M Gaussians at 3840x2160, forward + backward of one view, eager.
Arms: atomic; deterministic with torch.utils.deterministic.fill_uninitialized_memory on (PyTorch's default under the
flag: every torch.empty is filled with NaN); deterministic with that fill off.  For each: time per step (CUDA events,
arms alternated window by window, median), peak memory allocated by PyTorch over a few steps, and, from a separate
torch.profiler run, the device time of the deterministic blend backward and of its reducer per step.  The card's name
and power limit are read in the same run.

    python scripts/probe_deterministic.py [--out profiles/r12_deterministic.json] [--windows 7]
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
import torch.utils.deterministic as tud  # noqa: E402

from gsvc_b200 import _lib  # noqa: E402
from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians  # noqa: E402
from gsvc_b200.sharding import GRAD_LAYOUT  # noqa: E402
from probe_loss import ab, card  # noqa: E402

THRESHOLD = 0.05
ARMS = ("atomic", "deterministic_nan_fill", "deterministic_no_fill")


class mode:
    """Run inside one arm's mode: the flag and PyTorch's fill of uninitialised memory."""

    def __init__(self, arm):
        self.det = arm != "atomic"
        self.fill = arm == "deterministic_nan_fill"

    def __enter__(self):
        self.prev = (torch.are_deterministic_algorithms_enabled(), tud.fill_uninitialized_memory)
        torch.use_deterministic_algorithms(self.det)
        tud.fill_uninitialized_memory = self.fill

    def __exit__(self, *exc):
        torch.use_deterministic_algorithms(self.prev[0])
        tud.fill_uninitialized_memory = self.prev[1]
        return False


def settings_for(geom, frame_id, device, back=False):
    from gsvc_b200.rasterizer import GaussianRasterizationSettings
    fr = geom.frame(frame_id)
    vm = fr.view_matrix_s if back else fr.view_matrix
    return GaussianRasterizationSettings(
        image_height=int(fr.image_height), image_width=int(fr.image_width), x_min=fr.x_min, y_min=fr.y_min,
        scale=fr.scale, threshold=THRESHOLD, bg=torch.zeros(3, dtype=torch.float32, device=device),
        scale_modifier=1.0, viewmatrix=vm.permute(1, 0).to(device), sh_degree=0, campos=fr.cam_pos,
        prefiltered=False, debug=False)


def wrapped(arm, fn):
    def run():
        with mode(arm):
            return fn()
    return run


def peak_mb(fn, n=3):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    for _ in range(n):
        fn()
    torch.cuda.synchronize()
    return dict(peak_mb=torch.cuda.max_memory_allocated() / 2 ** 20, resident_mb=base / 2 ** 20)


def kernel_ms(fn, steps=10):
    """Device time per step of the deterministic backward's two kernels (torch.profiler, its own run)."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            fn()
        torch.cuda.synchronize()
    out = {"det_reduce_kernel": 0.0, "render_backward_kernel<true>": 0.0, "render_backward_kernel<false>": 0.0}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if "det_reduce_kernel" in e.key:
            out["det_reduce_kernel"] += t / 1e3 / steps
        elif "render_backward_kernel<true>" in e.key:
            out["render_backward_kernel<true>"] += t / 1e3 / steps
        elif "render_backward_kernel<false>" in e.key:
            out["render_backward_kernel<false>"] += t / 1e3 / steps
    return {k + "_ms": v for k, v in out.items()}


def measure(arms: dict, iters, windows):
    t = ab(arms, iters, windows)
    res = {}
    for k, fn in arms.items():
        res[k] = dict(t[k], **peak_mb(fn))
        torch.cuda.empty_cache()
    res["deterministic_nan_fill"].update(kernel_ms(arms["deterministic_nan_fill"]))
    res["atomic"].update(kernel_ms(arms["atomic"]))
    for k in ARMS[1:]:
        res[k]["time_over_atomic"] = res[k]["median_ms"] / res["atomic"]["median_ms"]
    return res


def config2_graphed(dev, windows):
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.views import ViewBatch
    cfg = CONFIGS[2]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    g = synthetic_gaussians(cfg["P"], geom, f0, f0, threshold=THRESHOLD, seed=2, device=dev)
    toast = ViewBatch.toast(settings_for(geom, f0, dev), settings_for(geom, f0, dev, back=True))
    dL = torch.randn((1, 3, cfg["H"], cfg["W"]), generator=torch.Generator().manual_seed(1)).to(dev)
    steps, captured_mb = {}, {}
    for arm in ARMS:
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        before = torch.cuda.memory_reserved()
        with mode(arm):
            steps[arm] = GraphedStep(toast, g, dL)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        captured_mb[arm] = (torch.cuda.memory_reserved() - before) / 2 ** 20
    arms = {arm: (lambda s=steps[arm]: s()) for arm in ARMS}
    res = measure(arms, 20, windows)
    for arm, s in steps.items():
        assert s.capacity_ok()
        # a replay allocates nothing: a graph holds the private memory pool its capture reserved
        res[arm]["graph_memory_mb"] = captured_mb[arm]
    R = int(steps["atomic"].num_rendered())
    return dict(workload=f"config 2: {cfg['P']} Gaussians, {cfg['W']}x{cfg['H']}, one frame as two views (toast), "
                         "forward + backward replayed from a GraphedStep", P=cfg["P"], R=R,
                partials_mb_at_R=_lib.lib().gsvc_rast_backward_partials_bytes(R) / 2 ** 20,
                note="peak_mb / resident_mb of the graphed arms include every graph's pool; graph_memory_mb is the "
                     "memory each arm's capture reserved (its graph pool and what the step keeps)", **res)


def reference_iteration(dev, windows):
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.views import ViewBatch, rasterize_views
    cfg = CONFIGS[2]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    frames = (f0, f0 + 1)
    sets = [synthetic_gaussians(cfg["P"], geom, f, f, threshold=THRESHOLD, seed=10 + i, device=dev)
            for i, f in enumerate((f0, f0, f0 + 1, f0 + 1))]
    names = [k for k, _ in GRAD_LAYOUT]
    cat = {k: torch.cat([s[k] for s in sets]) for k in names}
    counts = [cfg["P"]] * 4
    batch = ViewBatch.toasts([(settings_for(geom, f, dev), settings_for(geom, f, dev, back=True)) for f in frames])
    target = torch.rand((2, 3, cfg["H"], cfg["W"]), generator=torch.Generator().manual_seed(3)).to(dev)

    def step():
        p = {k: v.detach().requires_grad_(True) for k, v in cat.items()}
        m2d = torch.zeros((sum(counts), 3), device=dev, requires_grad=True)
        images, radii, n = rasterize_views(batch, means2D=m2d, counts=counts, **p)
        loss = photometric_loss(images, target, 0.2).mean()
        torch.autograd.grad(loss, [p[k] for k in names] + [m2d])
        return n

    arms = {arm: wrapped(arm, step) for arm in ARMS}
    R = int(step())
    res = measure(arms, 10, windows)
    return dict(workload=f"the reference's training iteration: 4 views (two frames, front + back) with {cfg['P']} "
                         f"Gaussians each of their own (ragged), {cfg['W']}x{cfg['H']}, fused L1 + D-SSIM(0.2), eager",
                R=R, **res)


def config5_view(dev, windows):
    from gsvc_b200.rasterizer import GaussianRasterizer
    c5 = CONFIGS[5]
    geom = CubeGeometry(c5["W"], c5["H"], c5["F"])
    f5 = c5["F"] // 2
    g = synthetic_gaussians(c5["P"], geom, f5, f5, threshold=THRESHOLD, seed=5, device=dev)
    rast = GaussianRasterizer(raster_settings=settings_for(geom, f5, dev))
    dL = torch.randn((3, c5["H"], c5["W"]), generator=torch.Generator().manual_seed(5)).to(dev)
    names = [k for k, _ in GRAD_LAYOUT]

    def step():
        p = {k: g[k].detach().requires_grad_(True) for k in names}
        m2 = torch.zeros_like(p["means3D"], requires_grad=True)
        color, radii, n = rast(means3D=p["means3D"], means2D=m2, shs=None, colors_precomp=p["colors_precomp"],
                               opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"],
                               cov3D_precomp=None)
        torch.autograd.grad(color, [p[k] for k in names] + [m2], grad_outputs=dL)
        return n

    arms = {arm: wrapped(arm, step) for arm in ARMS}
    R = int(step())
    res = measure(arms, 5, windows)
    return dict(workload=f"config 5: {c5['P']} Gaussians, {c5['W']}x{c5['H']}, forward + backward of one view, eager",
                P=c5["P"], R=R, **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r12_deterministic.json"))
    ap.add_argument("--windows", type=int, default=7)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("probe_deterministic measures on a GPU; none is visible")
    dev = torch.device("cuda:0")
    _lib.lib()
    out = dict(card=card(), windows=args.windows, arms=list(ARMS))
    for name, fn in (("config2_graphed_toast", config2_graphed), ("reference_iteration_ragged_loss", reference_iteration),
                     ("config5_per_view", config5_view)):
        out[name] = fn(dev, args.windows)
        torch.cuda.empty_cache()
        print(name, json.dumps(out[name])[:2000], flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
