"""GPU parity at BASELINE.json's full sizes (configs 2-5): direct comparison with the C oracle where it
finishes in seconds, plus size-independent properties of the domain: the sorted list is a permutation of
the emitted instances, keys ascend inside every tile, ranges partition [0, R), the per-tile counts sum to R,
the backward is linear in dL/dimage, culled Gaussians get exactly zero gradient, and the frame-sharded
gradient sum is independent of how the frames are split."""
import numpy as np
import pytest
import torch

from oracle import c_oracle
from tests import parity
from tests.scenes import stretch_gaussians
from gsvc_b200.frames import CONFIGS, CubeGeometry, synthetic_gaussians
from oracle.c_oracle import OracleSettings

pytestmark = pytest.mark.gpu

# two GPU runs of the same backward differ by the order of the float atomics: up to 4e-6 of the largest gradient in
# 300 repeats (scripts/probe_noise.py); GPU-vs-GPU comparisons get 4e-5, still 2.5x inside the 1e-4 parity bar
ATOMIC_RTOL = 4e-5
THRESHOLD = 0.05


def build(cfg_id, device, frame=None, n_frames=1, back=False, needle_mix=None):
    from gsvc_b200.rasterizer import GaussianRasterizationSettings
    cfg = CONFIGS[cfg_id]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    g = synthetic_gaussians(cfg["P"], geom, f0, f0 + n_frames - 1, threshold=THRESHOLD, seed=cfg_id)
    stretch_gaussians(g, needle_mix=needle_mix, seed=cfg_id)
    fr = geom.frame(f0 if frame is None else frame)
    vm = fr.view_matrix_s if back else fr.view_matrix
    rs = GaussianRasterizationSettings(
        image_height=cfg["H"], image_width=cfg["W"], x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale,
        threshold=THRESHOLD, bg=torch.zeros(3, device=device), scale_modifier=1.0,
        viewmatrix=vm.permute(1, 0).to(device), sh_degree=0, campos=fr.cam_pos, prefiltered=False, debug=False)
    st = OracleSettings(image_height=cfg["H"], image_width=cfg["W"], x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale,
                        threshold=THRESHOLD, bg=np.zeros(3, np.float32), viewmatrix=vm.permute(1, 0).numpy().copy(),
                        campos=fr.cam_pos.numpy())
    return cfg, g, rs, st


def oracle_forward(st, g):
    return parity.oracle_forward(st, {k: v.numpy() for k, v in g.items()})


check_forward = parity.check_forward


def check_stage_properties(state, cfg):
    keys, pl, ranges = state.export_keys()
    R = state.num_rendered
    T = ((cfg["W"] + 15) // 16) * ((cfg["H"] + 15) // 16)
    keys = keys.cpu().numpy().view(np.uint64)
    rg = ranges.cpu().numpy().view(np.uint32).astype(np.int64)
    lens = rg[:, 1] - rg[:, 0]
    assert lens.sum() == R and (lens >= 0).all()
    nz = np.nonzero(lens)[0]
    assert (rg[nz, 0] == np.cumsum(lens[nz]) - lens[nz]).all()           # ranges partition [0, R) in tile order
    assert (rg[lens == 0] == 0).all()                                      # untouched tiles keep (0, 0)
    assert (np.diff(keys.astype(np.uint64)) >= 0).all() if R else True     # globally sorted 64-bit keys
    tiles = (keys >> np.uint64(32)).astype(np.int64)
    assert (np.bincount(tiles, minlength=T) == lens).all()
    # permutation of the emitted instances: every Gaussian appears exactly tiles_touched times
    geo = state.export_geom()
    rect = geo["rect"].cpu().numpy().astype(np.int64)
    touched = (rect[:, 2] - rect[:, 0]) * (rect[:, 3] - rect[:, 1])
    assert (np.bincount(pl.cpu().numpy().view(np.uint32), minlength=cfg["P"]) == touched).all()
    assert ((state.radii.cpu().numpy() > 0) == (touched > 0)).all()


def run(rs, g, device, requires_grad):
    from gsvc_b200.rasterizer import GaussianRasterizer
    gd = {k: v.to(device).requires_grad_(requires_grad) for k, v in g.items()}
    m2d = torch.zeros_like(gd["means3D"], requires_grad=requires_grad)
    color, radii, n = GaussianRasterizer(raster_settings=rs)(
        means3D=gd["means3D"], means2D=m2d, shs=None, colors_precomp=gd["colors_precomp"], opacities=gd["opacities"],
        scales=gd["scales"], rotations=gd["rotations"], cov3D_precomp=None)
    return gd, m2d, color, radii, n


@pytest.mark.parametrize("needle_mix", [None, 0.05], ids=["generator", "with_needles"])
def test_config2_1080p_200k_forward_backward_vs_oracle(cuda_device, needle_mix):
    """BASELINE config 2 at full size against the referee oracle, every visible Gaussian compared; the second case
    turns 5 % of the Gaussians into needles (axis ratios 4:1 .. 256:1)."""
    cfg, g, rs, st = build(2, cuda_device, needle_mix=needle_mix)
    fo = oracle_forward(st, g)
    gd, m2d, color, radii, n = run(rs, g, cuda_device, True)
    assert n == fo["num_rendered"] and np.array_equal(radii.cpu().numpy(), fo["radii"])
    check_forward(fo, color, max_fragile=2e-3 if needle_mix is None else 5e-3)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(2)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    got = {k: gd[k].grad for k in parity.GRAD_NAMES}
    got["means2D"] = m2d.grad
    parity.check_grads(fo, go, got)


def test_config4_1080p_1M_forward_vs_oracle_and_stage_properties(cuda_device):
    """BASELINE config 4: with more than 160 instances per tile the sort takes its dense path (sort_tiles_kernel<true>);
    integer stages, forward and every visible Gaussian's gradient against the referee oracle behind it."""
    from gsvc_b200.rasterizer import RasterState
    cfg, g, rs, st = build(4, cuda_device)
    fo = oracle_forward(st, g)
    gd = {k: v.to(cuda_device) for k, v in g.items()}
    state = RasterState(rs, gd["means3D"], gd["opacities"], colors_precomp=gd["colors_precomp"], scales=gd["scales"],
                        rotations=gd["rotations"])
    assert state.num_rendered == fo["num_rendered"]
    assert state.num_rendered / (((cfg["W"] + 15) // 16) * ((cfg["H"] + 15) // 16)) > 160
    check_forward(fo, state.color)
    check_stage_properties(state, cfg)
    keys, pl, ranges = state.export_keys()
    assert np.array_equal(pl.cpu().numpy().view(np.uint32), fo["bin"]["point_list"])     # bit-exact order at 3M+ instances
    del state, keys, pl, ranges
    gd, m2d, color, radii, n = run(rs, g, cuda_device, True)
    assert n == fo["num_rendered"] and np.array_equal(radii.cpu().numpy(), fo["radii"])
    check_forward(fo, color)
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(4)))
    color.backward(torch.as_tensor(dL).to(cuda_device))
    go = parity.oracle_backward(fo, dL)
    got = {k: gd[k].grad for k in parity.GRAD_NAMES}
    got["means2D"] = m2d.grad
    parity.check_grads(fo, go, got)


def test_config5_4k_2M_stress(cuda_device):
    """4K, 2M Gaussians: 15-bit tile ids, multi-CTA scan (32 CTAs), scratch sized from the measured R; every visible
    Gaussian's gradient against the referee oracle."""
    from gsvc_b200.rasterizer import RasterState
    cfg, g, rs, st = build(5, cuda_device)
    fo = oracle_forward(st, g)
    gd, m2d, color, radii, n = run(rs, g, cuda_device, True)
    assert n == fo["num_rendered"] and np.array_equal(radii.cpu().numpy(), fo["radii"])
    check_forward(fo, color)
    names = ("means3D", "scales", "rotations", "opacities", "colors_precomp")
    ins = [gd[k] for k in names]
    dL = parity.masked_dL(fo, torch.randn(color.shape, generator=torch.Generator().manual_seed(55)))
    got = dict(zip(names + ("means2D",), torch.autograd.grad(color, ins + [m2d], retain_graph=True,
                                                             grad_outputs=torch.as_tensor(dL).to(cuda_device))))
    parity.check_grads(fo, parity.oracle_backward(fo, dL), got)
    # backward: linearity in dL/dimage and exact zeros for culled Gaussians
    gen = torch.Generator().manual_seed(5)
    d1 = torch.randn(color.shape, generator=gen).to(cuda_device)
    d2 = torch.randn(color.shape, generator=gen).to(cuda_device)
    ga = torch.autograd.grad(color, ins, grad_outputs=d1, retain_graph=True)
    gb = torch.autograd.grad(color, ins, grad_outputs=d2, retain_graph=True)
    gc = torch.autograd.grad(color, ins, grad_outputs=d1 + 2 * d2)
    for k, a, b, c in zip(names, ga, gb, gc):
        ref = a + 2 * b
        assert (c - ref).abs().max() <= 2e-4 * ref.abs().max(), k
        assert torch.isfinite(c).all()
    culled = radii == 0
    assert (gc[0][culled] == 0).all()
    state = RasterState(rs, *[gd[k].detach() for k in ("means3D", "opacities")],
                        colors_precomp=gd["colors_precomp"].detach(), scales=gd["scales"].detach(),
                        rotations=gd["rotations"].detach())
    check_stage_properties(state, cfg)


def test_config3_window_sharding_is_split_independent(cuda_device):
    """500k Gaussians over an 8-frame window: the summed [P,14] gradient buffer is the same whether one rank
    renders all 8 frames or G ranks render 8/G each (single-process emulation of the rank loop; the real
    NCCL all-reduce is exercised by bench.py --gpus N and, on CPU, by the gloo test)."""
    from gsvc_b200 import sharding
    from gsvc_b200.rasterizer import GaussianRasterizer
    cfg = CONFIGS[3]
    geom = CubeGeometry(cfg["W"], cfg["H"], cfg["F"])
    f0 = cfg["F"] // 2
    frames = list(range(f0, f0 + cfg["window"]))
    g = synthetic_gaussians(cfg["P"], geom, frames[0], frames[-1], threshold=THRESHOLD, seed=3, device=cuda_device)

    def view_grads(frame_id, back):
        from gsvc_b200.rasterizer import GaussianRasterizationSettings
        fr = geom.frame(frame_id)
        vm = fr.view_matrix_s if back else fr.view_matrix
        rs = GaussianRasterizationSettings(
            image_height=cfg["H"], image_width=cfg["W"], x_min=fr.x_min, y_min=fr.y_min, scale=fr.scale,
            threshold=THRESHOLD, bg=torch.zeros(3, device=cuda_device), scale_modifier=1.0,
            viewmatrix=vm.permute(1, 0).to(cuda_device), sh_degree=0, campos=fr.cam_pos, prefiltered=False, debug=False)
        p = {k: v.clone().requires_grad_(True) for k, v in g.items()}
        color, radii, n = GaussianRasterizer(raster_settings=rs)(
            means3D=p["means3D"], means2D=torch.zeros_like(p["means3D"]), shs=None, colors_precomp=p["colors_precomp"],
            opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        dL = torch.randn(color.shape, generator=torch.Generator().manual_seed(frame_id * 2 + int(back))).to(cuda_device)
        grads = torch.autograd.grad(color, [p[k] for k, _ in sharding.GRAD_LAYOUT], grad_outputs=dL)
        return {k: gr for (k, _), gr in zip(sharding.GRAD_LAYOUT, grads)}

    single = sharding.render_window_grads(frames, view_grads, rank=0, world=1)
    for world in (2, 4):
        total = None
        for r in range(world):
            part = sharding.render_window_grads(frames, view_grads, rank=r, world=world)   # no process group: local sum
            total = part if total is None else total + part
        # every backward sums its fp32 atomics in a different order: equal to rounding, not bitwise
        assert (total - single).abs().max() <= 5e-5 * single.abs().max()
    assert single.abs().max() > 0


def test_config2_toast_equals_two_calls(cuda_device):
    """BASELINE config 2 as the reference composes a frame — (front + flip(back)) / 2 — in one batched chain:
    equals the two single-view calls composed in PyTorch (forward within rounding of the final average, gradients
    up to summation order), and the frame's instance count is the sum of the views'."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import render_toast
    cfg, g, rs_f, _ = build(2, cuda_device)
    _, _, rs_b, _ = build(2, cuda_device, back=True)
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")
    p = {k: g[k].to(cuda_device).requires_grad_(True) for k in names}
    image, radii, n = render_toast(rs_f, rs_b, means3D=p["means3D"], opacities=p["opacities"],
                                   colors_precomp=p["colors_precomp"], scales=p["scales"], rotations=p["rotations"])
    dL = torch.randn((3, cfg["H"], cfg["W"]), generator=torch.Generator().manual_seed(2)).to(cuda_device)
    grads = torch.autograd.grad(image, [p[k] for k in names], grad_outputs=dL)
    outs, total = [], 0
    for rs in (rs_f, rs_b):
        m2d = torch.zeros_like(p["means3D"], requires_grad=True)
        c, r, k = GaussianRasterizer(raster_settings=rs)(
            means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"], opacities=p["opacities"],
            scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        outs.append((c, r))
        total += k
    assert n == total
    assert torch.equal(radii[0], outs[0][1]) and torch.equal(radii[1], outs[1][1])
    ref = (outs[0][0] + torch.flip(outs[1][0], dims=(-1,))) / 2          # pipeline/train.py:366-375
    assert (image - ref).abs().max() <= 2e-7
    ref_grads = torch.autograd.grad(ref, [p[k] for k in names], grad_outputs=dL)
    for k, a, b in zip(names, grads, ref_grads):
        assert (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max(), k


def test_config3_window_in_one_chain(cuda_device):
    """BASELINE config 3: the 8-frame TSW window (16 views, 500k Gaussians) as ONE batched chain; per-view images
    bit-identical to single calls for a sample of views, and the gradient of the window equals the frame-sharded
    sum (ranks = frames) the multi-GPU path computes."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import ViewBatch, rasterize_views
    cfg = CONFIGS[3]
    f0 = cfg["F"] // 2
    names = ("means3D", "colors_precomp", "opacities", "scales", "rotations")
    _, g, _, _ = build(3, cuda_device, n_frames=cfg["window"])
    p = {k: g[k].to(cuda_device).requires_grad_(True) for k in names}
    settings = []
    for f in range(f0, f0 + cfg["window"]):
        settings.append(build(3, cuda_device, frame=f, n_frames=cfg["window"])[2])
        settings.append(build(3, cuda_device, frame=f, n_frames=cfg["window"], back=True)[2])
    V = len(settings)
    images, radii, n = rasterize_views(ViewBatch(settings), means3D=p["means3D"], opacities=p["opacities"],
                                       colors_precomp=p["colors_precomp"], scales=p["scales"], rotations=p["rotations"])
    assert images.shape == (V, 3, cfg["H"], cfg["W"]) and radii.shape == (V, cfg["P"])
    dL = torch.randn((V, 3, cfg["H"], cfg["W"]), generator=torch.Generator().manual_seed(3)).to(cuda_device)
    grads = torch.autograd.grad(images, [p[k] for k in names], grad_outputs=dL)
    sums, total = None, 0
    for v, rs in enumerate(settings):
        m2d = torch.zeros_like(p["means3D"], requires_grad=True)
        c, r, k = GaussianRasterizer(raster_settings=rs)(
            means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"], opacities=p["opacities"],
            scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        total += k
        if v in (0, 5, 15):
            assert torch.equal(images[v], c) and torch.equal(radii[v], r)
        gv = torch.autograd.grad(c, [p[k] for k in names], grad_outputs=dL[v])
        sums = list(gv) if sums is None else [a + b for a, b in zip(sums, gv)]
    assert n == total
    for k, a, b in zip(names, grads, sums):
        assert (a - b).abs().max() <= 5e-5 * b.abs().max(), k
