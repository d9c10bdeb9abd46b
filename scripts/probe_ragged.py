"""Batched views over per-view Gaussian sets (rasterize_views / render_toast with `counts`) against the per-view calls
they replace, on the config 2 geometry (1920x1080, synthetic Gaussians of seed 12 as bench.py's `dropin_eager` leg).

Every iteration draws each view's P from 200 k +- 20 % (a prefix of one 240 k set, as `dropin_eager` draws it), so no
two calls have the same shape and the binning capacity comes from the density hint.
  1. training iteration, eager, 4 views (front / back of two frames), fused L1 + D-SSIM loss, backward to the per-view
     leaves: four GaussianRasterizer calls + flip / add / scale in PyTorch + photometric_loss on the two frames, against
     torch.cat of the four sets + one ragged rasterize_views(ViewBatch.toasts(...)) + photometric_loss;
  2. frame decode, forward only, 2 views: two GaussianRasterizer calls + (front + flip(back)) / 2, against torch.cat +
     one ragged render_toast;
  3. (--bench DIR) bench.py lines of the parent commit and of this tree, run alternately in the same session
     (bench_parent_*.json / bench_branch_*.json in DIR): the config 2 headline of each and their spread.

CUDA events, warm-up first, the two arms alternated window by window, medians over windows.  L2 is not flushed
between iterations: one iteration's working set (4 x ~200 k Gaussians in and out, ~4 x 1.2 M binning instances, the
images) is several times the 126 MB L2.  The card's name and power limit are read in the same run.

    python scripts/probe_ragged.py [--out profiles/r10_ragged.json] [--windows 9] [--bench DIR]
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from probe_loss import ab, card  # noqa: E402


def setup(dev):
    from bench import THRESHOLD, settings_for
    from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians
    cfg = CONFIGS[2]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    g = synthetic_gaussians(int(cfg["P"] * 1.2), geom, f0, f0 + 1, threshold=THRESHOLD, seed=12, device=dev)
    views = [settings_for(geom, f, dev, back=b) for f in (f0, f0 + 1) for b in (False, True)]
    return cfg, g, views


class Sizes:
    """Per-view P drawn per iteration from 200 k +- 20 %; every arm walks the same sequence."""

    def __init__(self, P, n_views, n=256, seed=7):
        rng = np.random.default_rng(seed)
        self.sizes = [[int(P * (0.8 + 0.4 * rng.random())) for _ in range(n_views)] for _ in range(n)]
        self.i = 0

    def next(self):
        s = self.sizes[self.i % len(self.sizes)]
        self.i += 1
        return s


def leg_train(cfg, g, views, dev, windows, iters):
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import ViewBatch, rasterize_views
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")
    H, W = cfg["H"], cfg["W"]
    targets = torch.rand((2, 3, H, W), generator=torch.Generator().manual_seed(3)).to(dev)
    rasts = [GaussianRasterizer(v) for v in views]
    batch = ViewBatch.toasts([(views[0], views[1]), (views[2], views[3])])
    sz = {"four_dropin_calls": Sizes(cfg["P"], 4), "one_ragged_chain": Sizes(cfg["P"], 4)}

    def leaves(counts):
        return [{k: g[k][:c].detach().requires_grad_(True) for k in names} for c in counts]

    def dropin():
        ps = leaves(sz["four_dropin_calls"].next())
        imgs, m2d = [], []
        for r, p in zip(rasts, ps):
            m = torch.zeros_like(p["means3D"], requires_grad=True)
            img, _, _ = r(means3D=p["means3D"], means2D=m, opacities=p["opacities"], colors_precomp=p["colors_precomp"],
                          scales=p["scales"], rotations=p["rotations"])
            imgs.append(img)
            m2d.append(m)
        images = torch.stack([(imgs[0] + imgs[1].flip(-1)) / 2, (imgs[2] + imgs[3].flip(-1)) / 2])
        loss = photometric_loss(images, targets).sum()
        return torch.autograd.grad(loss, [p[k] for p in ps for k in names] + m2d)

    def ragged():
        counts = sz["one_ragged_chain"].next()
        ps = leaves(counts)
        cat = {k: torch.cat([p[k] for p in ps]) for k in names}
        m2d = torch.zeros_like(cat["means3D"], requires_grad=True)
        images, _, _ = rasterize_views(batch, means3D=cat["means3D"], means2D=m2d, opacities=cat["opacities"],
                                       colors_precomp=cat["colors_precomp"], scales=cat["scales"],
                                       rotations=cat["rotations"], counts=counts)
        loss = photometric_loss(images, targets).sum()
        return torch.autograd.grad(loss, [p[k] for p in ps for k in names] + [m2d])

    t = ab({"four_dropin_calls": dropin, "one_ragged_chain": ragged}, iters, windows)
    t["speedup"] = t["four_dropin_calls"]["median_ms"] / t["one_ragged_chain"]["median_ms"]
    t["ms_per_view"] = {k: t[k]["median_ms"] / 4 for k in ("four_dropin_calls", "one_ragged_chain")}
    t["what"] = ("one training iteration: 4 views (front / back of 2 frames), each with its own set of P_v ~ U(160k, "
                 "240k) Gaussians, forward + fused L1/D-SSIM loss on the 2 composed frames + backward to every "
                 "view's leaves; the ragged arm includes its torch.cat of the four sets")
    return t


def leg_decode(cfg, g, views, dev, windows, iters):
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import render_toast
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")
    front, back = views[0], views[1]
    rf, rb = GaussianRasterizer(front), GaussianRasterizer(back)
    sz = {"two_dropin_calls": Sizes(cfg["P"], 2, seed=8), "one_ragged_toast": Sizes(cfg["P"], 2, seed=8)}
    z = {}

    def m2d(P):
        if P not in z:
            z[P] = torch.zeros((P, 3), device=dev)
        return z[P]

    def dropin():
        a, b = sz["two_dropin_calls"].next()
        pa, pb = ({k: g[k][:c] for k in names} for c in (a, b))
        with torch.no_grad():
            ca, _, _ = rf(means2D=m2d(a), **pa)
            cb, _, _ = rb(means2D=m2d(b), **pb)
            return (ca + cb.flip(-1)) / 2

    def ragged():
        counts = sz["one_ragged_toast"].next()
        with torch.no_grad():
            cat = {k: torch.cat([g[k][:c] for c in counts]) for k in names}
            return render_toast(front, back, counts=counts, **cat)[0]

    t = ab({"two_dropin_calls": dropin, "one_ragged_toast": ragged}, iters, windows)
    t["speedup"] = t["two_dropin_calls"]["median_ms"] / t["one_ragged_toast"]["median_ms"]
    t["what"] = ("one decoded frame: front and back view with their own sets of P_v ~ U(160k, 240k) Gaussians, "
                 "forward only, composed (front + flip(back)) / 2; the ragged arm includes its torch.cat")
    return t


def check_equal(cfg, g, views, dev):
    """The two arms of leg 1 on one draw of sizes: composed images equal, gradient rows within the atomics bound."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import ViewBatch, rasterize_views
    counts = Sizes(cfg["P"], 4, seed=99).next()
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")
    ps = [{k: g[k][:c].detach().requires_grad_(True) for k in names} for c in counts]
    imgs = [GaussianRasterizer(v)(means2D=torch.zeros((c, 3), device=dev), **p)[0]
            for v, p, c in zip(views, ps, counts)]
    ref = torch.stack([(imgs[0] + imgs[1].flip(-1)) / 2, (imgs[2] + imgs[3].flip(-1)) / 2])
    cat = {k: torch.cat([p[k] for p in ps]) for k in names}
    batch = ViewBatch.toasts([(views[0], views[1]), (views[2], views[3])])
    got = rasterize_views(batch, counts=counts, **cat)[0]
    dL = torch.randn(ref.shape, generator=torch.Generator().manual_seed(5)).to(dev)
    a = torch.autograd.grad(got, [p[k] for p in ps for k in names], grad_outputs=dL)
    b = torch.autograd.grad(ref, [p[k] for p in ps for k in names], grad_outputs=dL)
    rel = max(float((x - y).abs().max()) / max(float(y.abs().max()), 1e-30) for x, y in zip(a, b))
    return dict(counts=counts, images_equal=bool(torch.equal(got, ref)), grad_max_err_over_tensor_max=rel)


def bench_leg(d):
    def load(pattern):
        out = []
        for f in sorted(glob.glob(os.path.join(d, pattern))):
            lines = [ln for ln in open(f).read().splitlines() if ln.startswith("{")]
            if lines:
                out.append(json.loads(lines[-1])["value"])
        return out
    parent, branch = load("bench_parent_*.json"), load("bench_branch_*.json")
    res = dict(parent_iters_per_s=parent, branch_iters_per_s=branch,
               how="bench.py --gpus 1 --no-cpu-baseline --no-gpu-baseline, parent commit and this tree alternately "
                   "in the same session; value = config 2 headline (view-iters/s, 2-view step replayed from a CUDA graph)")
    if parent and branch:
        res["parent_median"], res["branch_median"] = statistics.median(parent), statistics.median(branch)
        res["parent_spread"] = [min(parent), max(parent)]
        res["branch_over_parent"] = res["branch_median"] / res["parent_median"]
        res["not_below_parent_spread"] = res["branch_median"] >= min(parent)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r10_ragged.json"))
    ap.add_argument("--windows", type=int, default=9)
    ap.add_argument("--bench", metavar="DIR", help="directory of the bench_parent_*.json / bench_branch_*.json lines")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "probe_ragged needs a GPU"
    dev = torch.device("cuda", 0)
    cfg, g, views = setup(dev)
    res = dict(card=card(), windows=args.windows, l2="not flushed (an iteration's working set is several times the "
               "126 MB L2)", timing="CUDA events around a window of back-to-back iterations per arm, arms alternated, "
               "median over windows")
    res["equality"] = check_equal(cfg, g, views, dev)
    res["train_iteration"] = leg_train(cfg, g, views, dev, args.windows, 20)
    res["frame_decode"] = leg_decode(cfg, g, views, dev, args.windows, 40)
    if args.bench:
        res["bench_regression_guard"] = bench_leg(args.bench)
    from gsvc_b200 import rasterizer as R_
    res["capacity_stats"] = dict(R_.capacity_stats)
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
