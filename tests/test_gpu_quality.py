"""The fused frame quality metrics (gsvc_b200.quality, csrc/quality.cu) against the float64 oracle
(tests/quality_oracle.py), their determinism, batching and CUDA-graph capture, and FrameStreamer.render(quality=).

Bars: PSNR within 1e-4 dB; SSIM within 1e-6 of the oracle and of 1 - photometric_loss(clamp(x), y, 1); MS-SSIM within
mean_c(ms_c * sum_l w_l 1e-6 / a_{l,c} + 1e-7), the propagation of a 1e-6 error of each per-level mean a_{l,c} (the
oracle's relu arguments), where every a_{l,c} >= 1e-4 or a channel has some a_{l,c} <= -1e-5 (it contributes exactly 0).
Scenes whose arguments sit between the two are reported as not qualifying; the tests assert which scenes qualify."""
import math

import numpy as np
import pytest
import torch

from tests import quality_oracle

pytestmark = pytest.mark.gpu

PSNR_TOL = 1e-4
SSIM_TOL = 1e-6
LEVEL_TOL = 1e-6


def _fused(x, y):
    from gsvc_b200 import frame_quality
    return frame_quality(x, y)


def check(x, y):
    """x, y [N,3,H,W] CUDA.  Compares with the float64 oracle (run on the GPU); returns whether MS-SSIM qualified."""
    from gsvc_b200.loss import photometric_loss
    N, _, H, W = x.shape
    q = _fused(x, y).double().cpu()
    xd, yd = x.double(), y.double()
    ref = torch.stack([quality_oracle.psnr(xd, yd), quality_oracle.ssim(xd, yd)], dim=1).cpu()
    finite = torch.isfinite(ref[:, 0])
    assert torch.equal(torch.isfinite(q[:, 0]), finite), (q[:, 0], ref[:, 0])
    if finite.any():
        assert (q[finite, 0] - ref[finite, 0]).abs().max().item() <= PSNR_TOL, (q[:, 0], ref[:, 0])
    assert (q[:, 1] - ref[:, 1]).abs().max().item() <= SSIM_TOL, (q[:, 1], ref[:, 1])
    one_minus_loss = 1.0 - photometric_loss(x.float().clamp(0.0, 1.0), y.float(), 1.0).double().cpu()
    assert (q[:, 1] - one_minus_loss).abs().max().item() <= SSIM_TOL
    if min(H, W) < quality_oracle.MIN_SIDE:
        assert torch.isnan(q[:, 2]).all()
        return False
    a = quality_oracle.ms_ssim_args(xd, yd)
    ms_ref, per_c = quality_oracle.ms_ssim_from_args(a)
    a, ms_ref, per_c = a.cpu(), ms_ref.cpu(), per_c.cpu()
    w = torch.tensor(quality_oracle.WEIGHTS, dtype=torch.float64)
    zero = (a <= -1e-5).any(dim=-1)                                   # [N,3]
    regular = (a >= 1e-4).all(dim=-1)
    if not (zero | regular).all():
        return False
    bar_c = torch.where(zero, torch.zeros_like(per_c),
                        per_c * (w * LEVEL_TOL / a.clamp_min(1e-4)).sum(dim=-1) + 1e-7)
    err = (q[:, 2] - ms_ref).abs()
    assert (err <= bar_c.mean(dim=1) + 1e-12).all(), (q[:, 2], ms_ref, bar_c)
    assert (q[zero.all(dim=1), 2] == 0.0).all()
    return True


def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _noisy(x, sigma, seed):
    return (x + sigma * torch.randn(x.shape, generator=_gen(seed)).to(x.device)).contiguous()


def _render(device, P, W, H, seed, jitter=0.0):
    from gsvc_b200.rasterizer import GaussianRasterizer
    from tests.scenes import make_scene, product_settings
    scene = make_scene(P=P, W=W, H=H, F=W, seed=seed, bg=(0.0, 0.0, 0.0))
    g = {k: v.to(device) for k, v in scene["gaussians"].items()}
    if jitter:
        g["means3D"] = g["means3D"] + jitter * torch.randn(g["means3D"].shape, generator=_gen(seed + 1)).to(device)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, device))
    with torch.no_grad():
        color, _, _ = rast(means3D=g["means3D"], means2D=None, shs=None, colors_precomp=g["colors_precomp"],
                           opacities=g["opacities"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    return color.unsqueeze(0).contiguous()


def test_render_against_perturbed_gaussians(cuda_device):
    x = _render(cuda_device, 4000, 256, 192, seed=5)
    y = _render(cuda_device, 4000, 256, 192, seed=5, jitter=0.002)
    assert not torch.equal(x, y)
    assert check(x, y)


@pytest.mark.parametrize("sigma", [0.01, 0.03, 0.1])
def test_render_against_noisy_copies(cuda_device, sigma):
    x = _render(cuda_device, 4000, 256, 192, seed=6)
    assert check(x, _noisy(x, sigma, 7))


def test_exact_zero_background(cuda_device):
    """A sparse scene on black: x == y == 0 on much of the image, flat zero windows at every level."""
    x = _render(cuda_device, 150, 256, 192, seed=8)
    y = _render(cuda_device, 150, 256, 192, seed=8, jitter=0.003)
    assert ((x == 0) & (y == 0)).float().mean() > 0.2
    check(x, y)                             # MS-SSIM is compared where the oracle's arguments qualify


def test_values_outside_the_unit_range(cuda_device):
    x = _render(cuda_device, 4000, 256, 192, seed=9)
    y = _noisy(x, 0.03, 10)
    xo = (1.5 * x - 0.25).contiguous()
    assert (xo < 0).any() and (xo > 1).any() and (y < 0).any()
    assert check(xo, y)
    assert not torch.equal(_fused(xo, y), _fused(x, y))


@pytest.mark.parametrize("hw", [(161, 161), (171, 333), (1080, 1920), (2160, 3840), (96, 64), (5, 7)])
def test_sizes(cuda_device, hw):
    x = torch.rand((1, 3) + hw, generator=_gen(hw[0] + hw[1])).to(cuda_device)
    y = _noisy(x, 0.05, 11)
    assert check(x, y) == (min(hw) > 160)


def test_closed_forms(cuda_device):
    x = torch.rand((2, 3, 171, 333), generator=_gen(12)).to(cuda_device)
    q = _fused(x, x.clone()).cpu()
    assert (q[:, 0] == math.inf).all() and (q[:, 1] == 1.0).all() and (q[:, 2] == 1.0).all()
    q = _fused(x, 1.0 - x).cpu()                                       # anticorrelated: cs < 0 at level 0
    assert (q[:, 2] == 0.0).all()
    assert check(x, 1.0 - x)
    xs = x * 0.9
    for delta in (0.1, 0.01, 0.001):
        q = _fused(xs, xs + delta).double().cpu()
        np.testing.assert_allclose(q[:, 0].numpy(), -20 * math.log10(delta), rtol=0, atol=PSNR_TOL)
    assert torch.isnan(_fused(x[..., :160, :], x[..., :160, :] + 0.01)[:, 2]).all()


def test_bit_reproducible_and_batch_independent(cuda_device):
    x = torch.rand((3, 3, 171, 333), generator=_gen(13)).to(cuda_device)
    y = _noisy(x, 0.05, 14)
    a, b = _fused(x, y), _fused(x, y)
    assert torch.equal(a, b)
    for n in range(3):
        one = _fused(x[n], y[n])
        assert one.shape == (3,) and torch.equal(one, a[n])


def test_graph_replay_equals_eager(cuda_device):
    from gsvc_b200 import frame_quality
    x = torch.rand((2, 3, 200, 300), generator=_gen(15)).to(cuda_device)
    y = _noisy(x, 0.05, 16).clamp(0.0, 1.0)
    ref = frame_quality(x, y)
    xs = x.clone()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        frame_quality(xs, y)
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        q = frame_quality(xs, y)
    xs.copy_(y)
    graph.replay()
    torch.cuda.synchronize()
    assert (q[:, 0] == math.inf).all()                                 # the replay read the new input ...
    xs.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(q, ref)                                         # ... and this one the original, bit for bit


def test_layouts_dtypes_and_errors(cuda_device):
    from gsvc_b200 import frame_quality
    from gsvc_b200.rasterizer import RasterizerError
    x = torch.rand((2, 3, 170, 180), generator=_gen(17)).to(cuda_device)
    y = _noisy(x, 0.05, 18)
    ref = frame_quality(x, y)
    xc = x.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)        # channels-last storage
    yc = torch.zeros((2, 3, 170, 360), device=cuda_device)
    yc[..., ::2] = y
    assert not xc.is_contiguous() and not yc[..., ::2].is_contiguous()
    assert torch.equal(frame_quality(xc, yc[..., ::2]), ref)
    assert torch.equal(frame_quality(x.double(), y.double()), frame_quality(x.double().float(), y.double().float()))
    xg = x.clone().requires_grad_(True)
    q = frame_quality(xg, y)
    assert not q.requires_grad and torch.equal(q, ref)
    with pytest.raises(RasterizerError, match="CUDA"):
        frame_quality(x, y.cpu())
    with pytest.raises(RasterizerError, match="shape"):
        frame_quality(x, y[:, :, :-1])
    with pytest.raises(RasterizerError):
        frame_quality(x[:, :2], y[:, :2])                              # not 3 channels


def test_frame_streamer_quality(cuda_device):
    """FrameStreamer.render(target=, quality=) over 3x n_streams frames writes frame_quality(render_toast(...), target)
    of every frame, bit for bit, with one synchronisation at the end."""
    from gsvc_b200 import frame_quality
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.rasterizer import RasterizerError
    from gsvc_b200.views import render_toast
    from tests.scenes import make_scene, product_settings
    P, W, H, F = 8000, 192, 176, 192
    frames = list(range(90, 99))
    base = make_scene(P=P, W=W, H=H, F=F, frame=frames[0], seed=61, window=len(frames))
    sets = []
    for f in frames:
        for back in (False, True):
            sc = make_scene(P=P, W=W, H=H, F=F, frame=f, seed=61, back=back)
            sets.append(product_settings(sc, cuda_device))
    params = {k: v.to(cuda_device) for k, v in base["gaussians"].items()}
    with torch.no_grad():
        refs = [render_toast(sets[2 * i], sets[2 * i + 1], means3D=params["means3D"], opacities=params["opacities"],
                             colors_precomp=params["colors_precomp"], scales=params["scales"],
                             rotations=params["rotations"])[0] for i in range(len(frames))]
    targets = [_noisy(r, 0.02, 100 + i) for i, r in enumerate(refs)]
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3)
    q = torch.full((len(frames), 3), -1.0, device=cuda_device)
    with pytest.raises(RasterizerError, match="both"):
        streamer.render(sets[0].viewmatrix, sets[1].viewmatrix, target=targets[0])
    with pytest.raises(RasterizerError, match="quality"):
        streamer.render(sets[0].viewmatrix, sets[1].viewmatrix, target=targets[0], quality=q[:, 0])
    for i in range(len(frames)):
        streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix, target=targets[i], quality=q[i])
    streamer.synchronize()
    want = torch.stack([frame_quality(r, t) for r, t in zip(refs, targets)])
    assert torch.isfinite(want).all()
    assert torch.equal(q, want)
    assert streamer.capacity_ok()
