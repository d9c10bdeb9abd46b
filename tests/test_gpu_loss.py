"""The fused L1 + D-SSIM loss (gsvc_b200.loss, csrc/loss.cu) against the float64 oracle (tests/loss_oracle.py) and the
float64 error budget of the kernel's evaluation order (tests/loss_budget.py), its determinism and CUDA-graph capture,
its wiring into the rasterizer's autograd chain, and GraphedStep(loss_target=).

Bars, all of them on every case:
  * per image |loss - loss64| <= 2 B_loss and per pixel |dL/dx - g64| <= 2 B(p), B the budget's first-order bound on
    the kernel's fp32 rounding (tests/test_loss_budget_cpu.py: an fp32 emulation stays within 0.5 B);
  * the per-image bars: the loss within 1e-6 (relative above 1, where fp32 cannot resolve 1e-6), and dL/dx within 1e-4
    of the larger of max|g64| of that image and |dL/dloss| / (3HW), the gradient scale of one value of the mean (the
    second term matters only where the oracle's gradient is all but zero, x == y: SSIM is at its maximum there); not
    where 1e-4 of that scale is below the normal range, where fp32 errors are absolute;
  * NaN and infinities of the loss and the gradient exactly where float64 autograd has them."""
import math

import numpy as np
import pytest
import torch

from tests import loss_budget, loss_oracle

pytestmark = pytest.mark.gpu

LOSS_TOL = 1e-6
GRAD_REL = 1e-4


def fused(x, y, lam, dL=None):
    from gsvc_b200.loss import photometric_loss
    xl = x.detach().clone().requires_grad_(True)
    loss = photometric_loss(xl, y, lam)
    g = torch.ones_like(loss) if dL is None else dL
    (grad,) = torch.autograd.grad(loss, xl, grad_outputs=g)
    return loss.detach(), grad


def _masks_equal(a, b):
    return torch.equal(torch.isnan(a), torch.isnan(b)) and torch.equal(torch.isposinf(a), torch.isposinf(b)) \
        and torch.equal(torch.isneginf(a), torch.isneginf(b))


def check_against_oracle(x, y, lam, dL=None, oracle_device="cpu", group=None, y_float=None):
    """x, y [N,3,H,W] CUDA (y fp32, or a uint8 target with y_float its fp32 values).  Returns the worst
    (loss error / B_loss, gradient error / B) over finite values, and prints them with the name `group`."""
    N, _, H, W = x.shape
    yf = y if y_float is None else y_float
    dL = torch.linspace(0.7, -1.3, N, device=x.device) if dL is None else dL
    loss, grad = fused(x, y, lam, dL)
    loss64, bl, g64, B = loss_budget.budget(x, yf, lam, dL)
    xo = x.double().to(oracle_device)
    yo = yf.double().to(oracle_device)
    xo.requires_grad_(True)
    lo = loss_oracle.photometric_loss(xo, yo, lam)
    (go,) = torch.autograd.grad(lo, xo, grad_outputs=dL.double().to(oracle_device))
    lo, go = lo.detach().to(x.device), go.to(x.device)
    loss, grad = loss.double(), grad.double()
    # the budget's value is the oracle's (float64 rounding; tests/test_loss_budget_cpu.py), and so are the masks
    assert _masks_equal(loss64, lo) and _masks_equal(g64, go)
    fin = torch.isfinite(go)
    scale = max(go[fin].abs().max().item() if fin.any() else 0.0, dL.abs().max().item() / (3.0 * H * W))
    assert (g64 - go)[fin].abs().max().item() <= 1e-9 * scale
    assert _masks_equal(loss, lo), (loss, lo)
    assert _masks_equal(grad, go), (torch.isnan(grad).sum().item(), torch.isnan(go).sum().item())
    lf = torch.isfinite(lo)
    lr = ((loss - loss64).abs() / bl)[lf].max().item() if lf.any() else 0.0
    gr = ((grad - g64).abs() / B)[fin].max().item() if fin.any() else 0.0
    assert lr <= 2.0, (lr, loss, loss64, bl)
    if gr > 2.0:
        r = (grad - g64).abs() / B
        i = torch.nonzero(torch.where(fin, r, 0.0) == gr)[0].tolist()
        raise AssertionError(f"dL/dx at {i}: {grad[tuple(i)].item()!r} against {g64[tuple(i)].item()!r}, "
                             f"error {gr:.3g} B(p) (B = {B[tuple(i)].item():.3g})")
    # the per-image bars
    lerr = (loss - lo)[lf].abs()
    assert (lerr <= LOSS_TOL * lo[lf].abs().clamp_min(1.0)).all(), (loss, lo)
    for n in range(N):
        fn = fin[n]
        bar = GRAD_REL * max(go[n][fn].abs().max().item() if fn.any() else 0.0, abs(float(dL[n])) / (3.0 * H * W))
        if 0.0 < bar < 2.0 ** -126:
            continue
        err = (grad[n] - go[n])[fn].abs().max().item() if fn.any() else 0.0
        assert err <= bar, (n, err, bar)
    if group:
        print(f"{group}: loss err/B_loss {lr:.3f}, gradient err/B {gr:.3f}")
    return lr, gr


def _rand(shape, seed, device):
    return torch.rand(shape, generator=torch.Generator().manual_seed(seed)).to(device)


LAMBDAS = [0.0, 0.2, 1.0]


@pytest.mark.parametrize("lam", LAMBDAS)
def test_random_pairs_96x64(cuda_device, lam):
    x, y = _rand((2, 3, 64, 96), 1, cuda_device), _rand((2, 3, 64, 96), 2, cuda_device)
    check_against_oracle(x, y, lam, group="random")


# H, W in {1, 4, 10, 11, 31, 32, 33, 63, 65} crossed sparsely: one tile and its edges, the 5- and 10-pixel rings
@pytest.mark.parametrize("hw", [(1, 1), (5, 7), (11, 11), (12, 300), (33, 65), (1, 65), (65, 1), (4, 10), (10, 4),
                                (11, 63), (31, 32), (32, 33), (33, 31), (63, 65), (65, 11), (32, 32), (4, 4)])
@pytest.mark.parametrize("lam", LAMBDAS)
def test_tiny_and_ragged_sizes(cuda_device, hw, lam):
    x, y = _rand((2, 3) + hw, 3, cuda_device), _rand((2, 3) + hw, 4, cuda_device)
    check_against_oracle(x, y, lam, group="sizes")


def _render(seed, device, W=128, H=80):
    from gsvc_b200.rasterizer import GaussianRasterizer
    from tests.scenes import make_scene, product_settings
    scene = make_scene(P=150, W=W, H=H, F=W, seed=seed, bg=(0.0, 0.0, 0.0))   # sparse: background left
    g = {k: v.to(device) for k, v in scene["gaussians"].items()}
    rast = GaussianRasterizer(raster_settings=product_settings(scene, device))
    with torch.no_grad():
        color, _, _ = rast(means3D=g["means3D"], means2D=None, shs=None, colors_precomp=g["colors_precomp"],
                           opacities=g["opacities"], scales=g["scales"], rotations=g["rotations"], cov3D_precomp=None)
    return color


@pytest.mark.parametrize("lam", LAMBDAS)
def test_render_against_another_render(cuda_device, lam):
    """Exact-zero background in both images: |x - y| has its kink (x == y == 0) on many pixels."""
    x, y = _render(5, cuda_device), _render(6, cuda_device)
    assert ((x == 0) & (y == 0)).any()
    check_against_oracle(torch.stack([x, y]), torch.stack([y, x]), lam, group="renders")
    # over-bright renders: colours are clamped at 0 only, a render may reach 3
    check_against_oracle(torch.stack([3.0 * x, y]), torch.stack([y, 3.0 * x]), lam, group="renders")


@pytest.mark.parametrize("lam", LAMBDAS)
def test_flat_images_with_small_noise(cuda_device, lam):
    """sigma^2 ~ 1e-7 under mu^2 ~ 0.4: E[x^2] - mu^2 would cancel in fp32 (the kernels form centred sums)."""
    n = (torch.rand((2, 3, 150, 200), generator=torch.Generator().manual_seed(7)) - 0.5) * 2e-3
    x = (torch.tensor([0.62, 0.35]).view(2, 1, 1, 1) + n).to(cuda_device)
    y = torch.tensor([0.3, 0.71]).view(2, 1, 1, 1).expand(2, 3, 150, 200).contiguous().to(cuda_device)
    check_against_oracle(x, y, lam, group="flat")
    check_against_oracle(x, x.flip(-1).contiguous(), lam, group="flat")   # two noisy flat images at the same level
    # 0.9 +- 5e-2 against a flat 0.3: where E[x^2] - mu^2 across rows would exceed the bound
    n = (torch.rand((1, 3, 96, 96), generator=torch.Generator().manual_seed(7)) - 0.5) * 0.1
    check_against_oracle((0.9 + n).to(cuda_device), torch.full((1, 3, 96, 96), 0.3, device=cuda_device), lam,
                         group="flat")


@pytest.mark.parametrize("lam", LAMBDAS)
def test_identical_images(cuda_device, lam):
    x = _rand((2, 3, 70, 90), 8, cuda_device)
    loss, grad = fused(x, x.clone(), lam)
    np.testing.assert_allclose(loss.cpu().numpy(), 0.0, atol=1e-6)
    check_against_oracle(x, x.clone(), lam, group="identical")
    if lam == 0.0:
        assert not grad.any()                                     # torch.sign: no L1 gradient where x == y


def test_full_size_1080p(cuda_device):
    """[2,3,1080,1920], the two frames of one training iteration; the float64 oracle runs on the GPU here."""
    x = _rand((2, 3, 1080, 1920), 9, cuda_device)
    y = (0.7 * x + 0.3 * _rand((2, 3, 1080, 1920), 10, cuda_device)).contiguous()
    x[:, :, :200] = 0.0
    y[:, :, :200] = 0.0                                           # an exact-zero band in both
    for lam in (0.2, 1.0):
        check_against_oracle(x, y, lam, oracle_device=cuda_device, group="full size")


def test_full_size_4k(cuda_device):
    """One [1,3,2160,3840] frame: 3HW is above 2^24; oracle and budget on the GPU."""
    x = _rand((1, 3, 2160, 3840), 19, cuda_device)
    y = (0.6 * x + 0.4 * _rand((1, 3, 2160, 3840), 20, cuda_device)).contiguous()
    check_against_oracle(x, y, 0.2, dL=torch.tensor([1.0], device=cuda_device), oracle_device=cuda_device,
                         group="full size")


@pytest.mark.parametrize("lam", LAMBDAS)
def test_batch_of_eight_cotangents(cuda_device, lam):
    """Subnormal products in wl1 / wss (1e-38, 2^-140 over 3HW) and a zero cotangent, which gives exact zeros."""
    dL = torch.tensor([1.0, -3.5, 0.0, 1e-30, 1e-38, 2.0 ** -140, 7.0, -1e-3], device=cuda_device)
    x, y = _rand((8, 3, 40, 70), 21, cuda_device), _rand((8, 3, 40, 70), 22, cuda_device)
    check_against_oracle(x, y, lam, dL=dL, group="cotangents")
    _, grad = fused(x, y, lam, dL)
    assert not grad[2].any()


def _tile_centres(H, W):
    return [(r, c) for r in range(16, H, 32) for c in range(16, W, 32)]


@pytest.mark.parametrize("level", [1.0, 1e4])
@pytest.mark.parametrize("lam", [0.2, 1.0])
def test_bright_pixels_at_tile_centres(cuda_device, level, lam):
    """A bright pixel at every tile centre on a black image: the shift k of every CTA is 1 (clamped), the maps around
    it span orders of magnitude."""
    x = torch.zeros((2, 3, 80, 100))
    for r, c in _tile_centres(80, 100):
        x[0, :, r, c] = level
        x[1, 1, r, c] = level
    y = torch.rand((2, 3, 80, 100), generator=torch.Generator().manual_seed(23)) * 0.1
    check_against_oracle(x.to(cuda_device), y.to(cuda_device), lam, group="bright")


@pytest.mark.parametrize("lam", [0.2, 1.0])
def test_step_edges(cuda_device, lam):
    """Steps on tile boundaries (column 32, row 64) and through tile centres (column 48, row 16)."""
    x = torch.full((2, 3, 96, 100), 0.2)
    x[0, :, :, 32:] = 0.8
    x[0, :, 64:, :] += 0.1
    x[1, :, :, 48:] = 0.9
    x[1, :, 16:, :] -= 0.15
    y = torch.rand((2, 3, 96, 100), generator=torch.Generator().manual_seed(24)) * 0.02 + 0.5
    check_against_oracle(x.to(cuda_device), y.to(cuda_device), lam, group="steps")


def test_rgb8_target_per_pixel(cuda_device):
    """An 8-bit target holding all 256 byte values, through gsvc_rast_loss_*_rgb8, against the budget of its fp32
    values fl(q / 255)."""
    from gsvc_b200 import targets as T8
    g = torch.Generator().manual_seed(25)
    cube = torch.randint(0, 256, (2, 48, 70, 3), dtype=torch.uint8, generator=g)
    cube.view(-1)[:256] = torch.arange(256, dtype=torch.uint8)
    cube = cube.to(cuda_device)
    x = (torch.rand((2, 3, 48, 70), generator=g) * 1.2 - 0.1).to(cuda_device)
    for lam in LAMBDAS:
        check_against_oracle(x, cube, lam, y_float=T8.to_float(cube), group="rgb8")


# non-finite values: a tile centre, a tile corner, the image border, the stage ring of the neighbouring tile
PLACES = {"centre": (16, 48), "corner": (31, 32), "border": (0, 20), "ring": (37, 40)}


@pytest.mark.parametrize("place", list(PLACES))
@pytest.mark.parametrize("value", [math.nan, math.inf, -math.inf])
@pytest.mark.parametrize("lam", [0.0, 0.2])
def test_non_finite_x(cuda_device, place, value, lam):
    x, y = _rand((3, 3, 64, 70), 26, cuda_device), _rand((3, 3, 64, 70), 27, cuda_device)
    bad = x.clone()
    bad[1, 2][PLACES[place]] = value
    _check_non_finite(x, bad, y, y, lam)


def test_nan_in_the_target(cuda_device):
    x, y = _rand((3, 3, 64, 70), 28, cuda_device), _rand((3, 3, 64, 70), 29, cuda_device)
    bad = y.clone()
    bad[1, 0, 16, 16] = math.nan
    _check_non_finite(x, x, y, bad, 0.2)


def _check_non_finite(x, xb, y, yb, lam):
    """Image 1 of xb / yb holds the bad value: masks and bars against the oracle; only its loss is NaN; the other
    images are bit-identical to the batch without the bad value."""
    dL = torch.tensor([0.7, -1.3, 2.0], device=x.device)
    check_against_oracle(xb, yb, lam, dL=dL, group="non-finite")
    loss, grad = fused(xb, yb, lam, dL)
    l0, g0 = fused(x, y, lam, dL)
    assert torch.isnan(loss[1]) and torch.isfinite(loss[[0, 2]]).all()
    assert not torch.isfinite(grad[1]).all()
    assert torch.equal(loss[[0, 2]], l0[[0, 2]]) and torch.equal(grad[[0, 2]], g0[[0, 2]])


def test_bit_reproducible(cuda_device):
    x, y = _rand((2, 3, 540, 960), 11, cuda_device), _rand((2, 3, 540, 960), 12, cuda_device)
    l1, g1 = fused(x, y, 0.2)
    l2, g2 = fused(x, y, 0.2)
    assert torch.equal(l1, l2) and torch.equal(g1, g2)


def test_graph_replay_equals_eager(cuda_device):
    from gsvc_b200.loss import photometric_loss
    x, y = _rand((2, 3, 200, 300), 13, cuda_device), _rand((2, 3, 200, 300), 14, cuda_device)
    dL = torch.tensor([0.5, -2.0], device=cuda_device)
    l_e, g_e = fused(x, y, 0.2, dL)
    xs = x.clone().requires_grad_(True)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        photometric_loss(xs, y, 0.2)                              # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        loss = photometric_loss(xs, y, 0.2)
        (grad,) = torch.autograd.grad(loss, xs, grad_outputs=dL)
    with torch.no_grad():
        xs.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert not torch.equal(loss, l_e)                             # the replay read the zeroed input ...
    with torch.no_grad():
        xs.copy_(x)
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(loss, l_e) and torch.equal(grad, g_e)      # ... and this one the original, bit for bit


def test_layouts_batching_and_errors(cuda_device):
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.rasterizer import RasterizerError
    x, y = _rand((2, 3, 48, 80), 15, cuda_device), _rand((2, 3, 48, 80), 16, cuda_device)
    l_ref, g_ref = fused(x, y, 0.2)
    # channels-last storage (non-contiguous [N,3,H,W] views) and a strided target
    xc = x.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2)
    yc = torch.zeros((2, 3, 48, 160), device=cuda_device)
    yc[..., ::2] = y
    assert not xc.is_contiguous() and not yc[..., ::2].is_contiguous()
    l_nc, g_nc = fused(xc, yc[..., ::2], 0.2)
    assert torch.equal(l_nc, l_ref) and torch.equal(g_nc, g_ref)
    # one image at a time gives the batch's per-image values; [3,H,W] returns the 0-dim loss
    for n in range(2):
        xl = x[n].clone().requires_grad_(True)
        loss = photometric_loss(xl, y[n], 0.2)
        assert loss.dim() == 0 and torch.equal(loss.detach(), l_ref[n])
        loss.backward()
        assert torch.equal(xl.grad, g_ref[n])
    with pytest.raises(RasterizerError, match="CUDA"):
        photometric_loss(x, y.cpu())
    with pytest.raises(RasterizerError, match="shape"):
        photometric_loss(x, y[:, :, :-1])
    with pytest.raises(RasterizerError, match="requires_grad"):
        photometric_loss(x, y.clone().requires_grad_(True))
    with pytest.raises(RasterizerError):
        photometric_loss(x[:, :2], y[:, :2])                      # not 3 channels


def _toast_setup(device, P=6000, W=192, H=128, seed=0):
    from examples.fit_window import THRESHOLD, settings
    from gsvc_b200.frames import CubeGeometry, synthetic_gaussians
    from gsvc_b200.views import ViewBatch, rasterize_views
    geom = CubeGeometry(W, H, W)
    f0 = W // 2
    batch = ViewBatch.toasts([(settings(geom, f, device), settings(geom, f, device, back=True)) for f in (f0, f0 + 1)])
    params = synthetic_gaussians(P, geom, f0, f0 + 1, threshold=THRESHOLD, seed=200 + seed, device=device)
    target_g = synthetic_gaussians(P, geom, f0, f0 + 1, threshold=THRESHOLD, seed=100 + seed, device=device)
    with torch.no_grad():
        target, _, _ = rasterize_views(batch, **{k: target_g[k] for k in
                                                 ("means3D", "opacities", "colors_precomp", "scales", "rotations")})
    params = {k: params[k].contiguous().clone() for k in ("means3D", "colors_precomp", "opacities", "scales",
                                                          "rotations")}
    return batch, params, target.contiguous()


def _eager_step(batch, params, target, lam, dimage=None):
    """Rendered images, per-image losses and the GRAD_LAYOUT gradients of their mean (or of the images seeded with
    `dimage`), packed [P,14]."""
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.sharding import GRAD_LAYOUT
    from gsvc_b200.views import rasterize_views
    leaves = {k: params[k].detach().clone().requires_grad_(True) for k, _ in GRAD_LAYOUT}
    color, _, _ = rasterize_views(batch, means3D=leaves["means3D"], opacities=leaves["opacities"],
                                  colors_precomp=leaves["colors_precomp"], scales=leaves["scales"],
                                  rotations=leaves["rotations"])
    loss = photometric_loss(color, target, lam)
    if dimage is None:
        grads = torch.autograd.grad(loss.mean(), [leaves[k] for k, _ in GRAD_LAYOUT])
    else:
        grads = torch.autograd.grad(color, [leaves[k] for k, _ in GRAD_LAYOUT], grad_outputs=dimage)
    P = params["means3D"].shape[0]
    return color.detach(), loss.detach(), torch.cat([g.reshape(P, -1) for g in grads], dim=1)


def _assert_packed_close(a, b):
    from gsvc_b200.sharding import GRAD_LAYOUT
    o = 0
    for k, w in GRAD_LAYOUT:
        ra, rb = a[:, o:o + w], b[:, o:o + w]
        bar = 1e-4 * rb.abs().max().item()
        assert (ra - rb).abs().max().item() <= bar, (k, (ra - rb).abs().max().item(), bar)
        o += w


def test_rasterizer_chain_with_the_fused_loss(cuda_device):
    """rasterize_views(toasts) -> photometric_loss -> backward equals the same chain seeded with the oracle's
    dL/dimage, within the rasterizer's per-tensor bar."""
    batch, params, target = _toast_setup(cuda_device)
    lam = 0.2
    color, loss, packed = _eager_step(batch, params, target, lam)
    _, go = loss_oracle.loss_and_grad(color.double().cpu().numpy(), target.double().cpu().numpy(), lam,
                                      np.full(color.shape[0], 1.0 / color.shape[0]))
    _, _, packed_o = _eager_step(batch, params, target, lam, dimage=torch.from_numpy(go).float().to(cuda_device))
    assert torch.isfinite(packed).all() and packed.abs().max() > 0
    _assert_packed_close(packed, packed_o)


def test_graphed_step_with_loss_target(cuda_device):
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.rasterizer import RasterizerError
    lam = 0.2
    batch, params, target = _toast_setup(cuda_device)
    tgt = target.clone()
    with pytest.raises(RasterizerError, match="either dL"):
        GraphedStep(batch, params, torch.zeros_like(tgt), loss_target=tgt)
    step = GraphedStep(batch, params, None, loss_target=tgt, lambda_dssim=lam)
    for it in range(3):
        with torch.no_grad():
            params["means3D"][:, 1] += 0.002
            params["opacities"].mul_(0.97)
        color, _, packed = step()
        torch.cuda.synchronize()
        assert step.capacity_ok()
        color_e, loss_e, packed_e = _eager_step(batch, params, tgt, lam)
        assert step.loss.shape == (2,)
        assert torch.equal(color, color_e)
        assert torch.equal(step.loss, loss_e)                    # the forward is deterministic
        _assert_packed_close(packed, packed_e)                   # the blend backward accumulates with atomics
    # a new target written in place is what the next replay trains against
    before = step.loss.clone()
    tgt.copy_(target.flip(-1))
    step()
    torch.cuda.synchronize()
    _, loss_e, packed_e = _eager_step(batch, params, tgt, lam)
    assert not torch.equal(step.loss, before) and torch.equal(step.loss, loss_e)
    _assert_packed_close(step.packed, packed_e)


def test_fit_window_converges_with_the_fused_loss(cuda_device):
    from examples.fit_window import fit
    losses = fit(cuda_device, iters=150, P=6000, W=192, H=128, Fr=192, lambda_dssim=0.2)
    assert all(l == l for l in losses)                      # no NaN
    first, last = sum(losses[:5]) / 5, sum(losses[-5:]) / 5
    print(f"fit_window lambda_dssim=0.2: loss {first:.5f} -> {last:.5f} ({last / first:.3f})")
    assert last < 0.2 * first, (first, last)             # measured on a B200: 0.250 -> 0.021 (ratio 0.083)
