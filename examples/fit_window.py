"""Rasterizer-level stand-in for the reference's training iteration (pipeline/train.py:325-581), SURVEY.md §8f
row f3: two frames x (front + back view), L1 loss against target frames (or the fused L1 + D-SSIM loss of
train.py:409-410 with --lambda-dssim, gsvc_b200.loss), Adam on the Gaussian parameters.  The four
views of an iteration are ONE batched kernel chain (gsvc_b200.views); under torchrun each rank takes its own frame
pair and the parameter gradients are summed with one NCCL all-reduce per step (gsvc_b200.sharding).

    python examples/fit_window.py [--iters 200] [--P 20000] [--lambda-dssim 0.2]
    python -m torch.distributed.run --nproc-per-node 2 --master-addr 127.0.0.1 examples/fit_window.py
"""
from __future__ import annotations

import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch
import torch.nn.functional as F

from gsvc_b200 import sharding
from gsvc_b200.frames import CubeGeometry, synthetic_gaussians
from gsvc_b200.loss import photometric_loss
from gsvc_b200.rasterizer import GaussianRasterizationSettings
from gsvc_b200.views import ViewBatch, rasterize_views

THRESHOLD = 0.05


def settings(geom, frame_id, device, back=False):
    fr = geom.frame(frame_id)
    vm = fr.view_matrix_s if back else fr.view_matrix
    return GaussianRasterizationSettings(
        image_height=fr.image_height, image_width=fr.image_width, x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale,
        threshold=THRESHOLD, bg=torch.zeros(3, device=device), scale_modifier=1.0, viewmatrix=vm.permute(1, 0).to(device),
        sh_degree=0, campos=fr.cam_pos, prefiltered=False, debug=False)


class Gaussians(torch.nn.Module):
    """Free Gaussian parameters with the activations the reference applies (guassian.py:251-287:
    opacity in (0,1), positive scales, unit quaternions, colours in (0,1))."""

    def __init__(self, g):
        super().__init__()
        self.xyz = torch.nn.Parameter(g["means3D"].clone())
        self.log_s = torch.nn.Parameter(g["scales"].log())
        self.rot = torch.nn.Parameter(g["rotations"].clone())
        self.op = torch.nn.Parameter(torch.logit(g["opacities"].clamp(1e-3, 1 - 1e-3)))
        self.col = torch.nn.Parameter(torch.logit(g["colors_precomp"].clamp(1e-3, 1 - 1e-3)))

    def forward(self):
        return dict(means3D=self.xyz, scales=self.log_s.exp(), rotations=F.normalize(self.rot, dim=-1),
                    opacities=torch.sigmoid(self.op), colors_precomp=torch.sigmoid(self.col))


def render_frames(batch, g, means2D=None):
    images, radii, n = rasterize_views(batch, means3D=g["means3D"], opacities=g["opacities"], means2D=means2D,
                                       colors_precomp=g["colors_precomp"], scales=g["scales"], rotations=g["rotations"])
    return images, radii, n


def fit(device, iters=200, P=20000, W=320, H=192, Fr=320, rank=0, world=1, log=None, seed=0, lambda_dssim=None):
    """Returns the list of per-iteration losses (this rank's frames).  lambda_dssim None: the L1 loss; a float: the
    fused (1 - lambda) L1 + lambda (1 - SSIM), averaged over the frames."""
    geom = CubeGeometry(W, H, Fr)
    f0 = Fr // 2 + 2 * rank                                      # this rank's frame pair (frame_idx, frame_idx + 1)
    span = (Fr // 2, Fr // 2 + 2 * world - 1)
    target_g = synthetic_gaussians(P, geom, span[0], span[1], threshold=THRESHOLD, seed=100 + seed, device=device)
    init_g = synthetic_gaussians(P, geom, span[0], span[1], threshold=THRESHOLD, seed=200 + seed, device=device)
    batch = ViewBatch.toasts([(settings(geom, f, device), settings(geom, f, device, back=True)) for f in (f0, f0 + 1)])
    with torch.no_grad():
        targets, _, _ = render_frames(batch, target_g)            # [2,3,H,W]: the "video frames"
    model = Gaussians(init_g).to(device)
    opt = torch.optim.Adam([dict(params=[model.xyz], lr=2e-4), dict(params=[model.log_s], lr=5e-3),
                            dict(params=[model.rot], lr=1e-3), dict(params=[model.op], lr=5e-2),
                            dict(params=[model.col], lr=2.5e-2)])
    losses = []
    name = "L1" if lambda_dssim is None else f"L1+D-SSIM({lambda_dssim:g})"
    # the densification statistic of training_statis (scene/gaussian_model.py:1298-1314): accumulated |dL/dmeans2D|
    # and the number of views each Gaussian was drawn in, over ALL ranks' views
    stat_accum = torch.zeros((P, sharding.STATS_WIDTH), device=device)
    for it in range(iters):
        means2D = torch.zeros((batch.n_views, P, 3), device=device, requires_grad=True)   # viewspace_points, per view
        images, radii, n = render_frames(batch, model(), means2D)
        if lambda_dssim is None:
            loss = (images - targets).abs().mean()                # Ll1 of train.py:409
        else:
            loss = photometric_loss(images, targets, lambda_dssim).mean()   # train.py:409-410, per frame
        opt.zero_grad(set_to_none=True)
        loss.backward()
        stats = sharding.densify_stats(means2D.grad, radii)       # one pass for the step's 4 views
        if world > 1:
            import torch.distributed as dist
            flat = torch.cat([p.grad.reshape(-1) for p in model.parameters()] + [stats.reshape(-1) * world])
            dist.all_reduce(flat, op=dist.ReduceOp.SUM)           # one collective per step: gradients + statistic
            flat /= world
            o = 0
            for p in model.parameters():
                p.grad.copy_(flat[o:o + p.numel()].view_as(p))
                o += p.numel()
            stats = flat[o:].view_as(stats)                       # summed (not averaged) over the ranks
        stat_accum += stats
        opt.step()
        losses.append(float(loss.detach()))
        if log and (it % 50 == 0 or it == iters - 1):
            log(f"iter {it:4d}  {name} {losses[-1]:.5f}  num_rendered {n}  visible {int((radii > 0).sum())}")
    # what adjust_anchor would threshold (scene/gaussian_model.py: grads = offset_gradient_accum / offset_denom)
    seen = stat_accum[:, 1] > 0
    mean_grad = torch.where(seen, stat_accum[:, 0] / stat_accum[:, 1].clamp(min=1), torch.zeros_like(stat_accum[:, 0]))
    fit.last_densify = dict(seen=int(seen.sum()), candidates=int((mean_grad > 2e-4).sum()),
                            checksum=float(stat_accum.double().sum()))
    if log:
        log(f"densification statistic: {fit.last_densify['seen']} Gaussians drawn at least once, "
            f"{fit.last_densify['candidates']} above the 2e-4 mean screen-gradient threshold")
    return losses


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--P", type=int, default=20000)
    ap.add_argument("--lambda-dssim", type=float, default=None,
                    help="train on (1 - l) L1 + l (1 - SSIM) (the reference's lambda_dssim, upstream 0.2); default: L1")
    args = ap.parse_args()
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    device = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
    torch.cuda.set_device(device)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")   # collectives beside full-occupancy blend kernels
        dist.init_process_group("nccl", device_id=device)
    losses = fit(device, args.iters, args.P, rank=rank, world=world, log=print if rank == 0 else None,
                 lambda_dssim=args.lambda_dssim)
    if rank == 0:
        print(f"{'L1' if args.lambda_dssim is None else 'loss'} {losses[0]:.5f} -> {losses[-1]:.5f}")
    if world > 1:
        # every rank must hold the same statistic (it decides densification): compare the checksums
        mine = torch.tensor([fit.last_densify["checksum"], float(fit.last_densify["candidates"])], dtype=torch.float64,
                            device=device)
        every = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        assert all(torch.equal(e, every[0]) for e in every), every
        if rank == 0:
            print(f"densification statistic identical on all {world} ranks")
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
