"""GPU parity tests of the batched-view ("toast") path, SURVEY.md §8f row f1: gsvc_b200.views against
(a) the single-view CUDA path it must reproduce exactly and (b) the CPU oracle composed the way the reference
composes a frame — (front + flip_x(back)) / 2, pipeline/train.py:353-375.
"""
import numpy as np
import pytest
import torch

from oracle import c_oracle
from tests import parity
from tests.scenes import make_scene, np_inputs, product_settings

pytestmark = pytest.mark.gpu

# two GPU runs of the same backward differ by the order of the float atomics: up to 4e-6 of the largest gradient in
# 300 repeats (scripts/probe_noise.py); GPU-vs-GPU comparisons get 4e-5, still 2.5x inside the 1e-4 parity bar
ATOMIC_RTOL = 4e-5

NAMES = ("means3D", "colors_precomp", "opacities", "scales", "rotations")


def _scenes(P, W, H, F, seed, frames):
    """Front/back scenes of several frames over ONE Gaussian set (the window of frames shares it)."""
    base = make_scene(P=P, W=W, H=H, F=F, frame=frames[0], seed=seed, window=len(frames))
    out = []
    for f in frames:
        for back in (False, True):
            sc = make_scene(P=P, W=W, H=H, F=F, frame=f, seed=seed, back=back)
            sc["gaussians"] = base["gaussians"]
            out.append(sc)
    return out


def _oracle(scene):
    return parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]))


def _leaves(scene, device):
    return {k: scene["gaussians"][k].to(device).clone().requires_grad_(True) for k in NAMES}


def _single(scene, device, p, dL):
    from gsvc_b200.rasterizer import GaussianRasterizer, _RasterizeViews
    rast = GaussianRasterizer(raster_settings=product_settings(scene, device))
    m2d = torch.zeros_like(p["means3D"], requires_grad=True)
    color, radii, n = rast(means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"],
                           opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
    # the drop-in's outputs come in upstream's shapes straight from the Function: no select / index node in between
    assert type(color.grad_fn) is _RasterizeViews._backward_cls
    assert color.shape == (3,) + tuple(dL.shape[-2:]) and radii.shape == (p["means3D"].shape[0],)
    grads = torch.autograd.grad(color, [p[k] for k in NAMES] + [m2d], grad_outputs=dL)
    assert grads[-1].shape == m2d.shape
    return color, radii, n, grads


@pytest.mark.parametrize("W,H", [(192, 128), (200, 120)])
def test_batched_views_equal_single_calls(cuda_device, W, H):
    """4 views (front/back of two frames) in one chain == 4 single calls: images and radii bit-exact,
    summed parameter gradients up to summation order, per-view means2D gradients."""
    from gsvc_b200.views import rasterize_views
    P = 12000
    scenes = _scenes(P, W, H, 192, seed=41, frames=(96, 97))
    p = _leaves(scenes[0], cuda_device)
    dL = torch.randn((4, 3, H, W), generator=torch.Generator().manual_seed(7)).to(cuda_device)
    m2d = torch.zeros((4, P, 3), device=cuda_device, requires_grad=True)
    settings = [product_settings(s, cuda_device) for s in scenes]
    images, radii, n = rasterize_views(settings, means3D=p["means3D"], opacities=p["opacities"], means2D=m2d,
                                       colors_precomp=p["colors_precomp"], scales=p["scales"], rotations=p["rotations"])
    grads = torch.autograd.grad(images, [p[k] for k in NAMES] + [m2d], grad_outputs=dL)
    assert images.shape == (4, 3, H, W) and radii.shape == (4, P)
    total, sums = 0, None
    for v, sc in enumerate(scenes):
        c1, r1, n1, g1 = _single(sc, cuda_device, p, dL[v])
        total += n1
        assert torch.equal(images[v], c1), f"view {v}"
        assert torch.equal(radii[v], r1)
        assert (grads[-1][v] - g1[-1]).abs().max() <= ATOMIC_RTOL * g1[-1].abs().max()
        sums = list(g1[:-1]) if sums is None else [a + b for a, b in zip(sums, g1[:-1])]
    assert n == total
    for k, a, b in zip(NAMES, grads[:-1], sums):
        assert (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max(), k
    # a batch of one view is the drop-in call
    m2d1 = torch.zeros((1, P, 3), device=cuda_device, requires_grad=True)
    images1, radii1, n1 = rasterize_views(settings[:1], means3D=p["means3D"], opacities=p["opacities"], means2D=m2d1,
                                          colors_precomp=p["colors_precomp"], scales=p["scales"],
                                          rotations=p["rotations"])
    grads1 = torch.autograd.grad(images1, [p[k] for k in NAMES] + [m2d1], grad_outputs=dL[:1])
    c1, r1, k1, g1 = _single(scenes[0], cuda_device, p, dL[0])
    assert torch.equal(images1[0], c1) and torch.equal(radii1[0], r1) and n1 == k1
    for k, a, b in zip(NAMES + ("means2D",), grads1, g1):
        assert (a.reshape(b.shape) - b).abs().max() <= ATOMIC_RTOL * b.abs().max(), k


@pytest.mark.parametrize("W,H", [(160, 96), (150, 90)])
def test_toast_matches_oracle(cuda_device, W, H):
    """render_toast == (oracle front + flip_x(oracle back)) / 2, forward and backward (W not a multiple of the tile
    size puts mirrored pixels in different tiles of the two views)."""
    from gsvc_b200.views import render_toast
    P = 10000
    front, back = _scenes(P, W, H, 160, seed=43, frames=(80,))
    fo_f, fo_b = _oracle(front), _oracle(back)
    p = _leaves(front, cuda_device)
    image, radii, n = render_toast(product_settings(front, cuda_device), product_settings(back, cuda_device),
                                   means3D=p["means3D"], opacities=p["opacities"], colors_precomp=p["colors_precomp"],
                                   scales=p["scales"], rotations=p["rotations"])
    assert n == fo_f["num_rendered"] + fo_b["num_rendered"]
    np.testing.assert_array_equal(radii[0].cpu().numpy(), fo_f["radii"])
    np.testing.assert_array_equal(radii[1].cpu().numpy(), fo_b["radii"])
    ref = 0.5 * (fo_f["color"] + fo_b["color"][:, :, ::-1])
    frag = fo_f["fragile"] | fo_b["fragile"][:, ::-1]          # in the composed image's pixel coordinates
    assert frag.mean() <= parity.MAX_FRAGILE
    err = np.abs(image.detach().cpu().numpy() - ref)[:, ~frag]
    assert err.max() <= 1e-5, err.max()
    # the seed gradient is zeroed where EITHER view's pixel is fragile, so every visible Gaussian is compared
    dL = parity.masked_dL(fo_f, torch.randn((3, H, W), generator=torch.Generator().manual_seed(9)), fragile_extra=frag)
    grads = torch.autograd.grad(image, [p[k] for k in NAMES], grad_outputs=torch.as_tensor(dL).to(cuda_device))
    go_f = parity.oracle_backward(fo_f, 0.5 * dL)
    go_b = parity.oracle_backward(fo_b, np.ascontiguousarray(0.5 * dL[:, :, ::-1]))
    both = dict(radii=np.maximum(fo_f["radii"], fo_b["radii"]))     # visible in either view
    parity.check_grads(both, {k: go_f[k] + go_b[k] for k in NAMES}, dict(zip(NAMES, grads)))


def test_batched_binning_is_bit_exact_per_view(cuda_device):
    """Sorted keys / point list / tile ranges of a 2-view batch, view by view, against the oracle
    (virtual tile v*T+t, virtual Gaussian v*P+g, ranges offset by the instances of the views before)."""
    from gsvc_b200 import _lib
    from gsvc_b200.rasterizer import _NativeViews
    from gsvc_b200.views import ViewBatch
    P, W, H = 6000, 128, 80
    scenes = _scenes(P, W, H, 128, seed=47, frames=(64,))
    fos = [_oracle(s) for s in scenes]
    L = _lib.lib()
    dev = cuda_device
    g = {k: v.to(dev) for k, v in scenes[0]["gaussians"].items()}
    batch = ViewBatch([product_settings(s, dev) for s in scenes])
    nv = _NativeViews(batch, dev)
    V = 2
    T = ((W + 15) // 16) * ((H + 15) // 16)
    R = sum(fo["num_rendered"] for fo in fos)
    u8 = lambda n: torch.empty(int(n), dtype=torch.uint8, device=dev)
    geom, image = u8(L.gsvc_rast_geom_bytes(P * V, 0)), u8(L.gsvc_rast_image_bytes_views(W, H, V))
    binning = u8(L.gsvc_rast_binning_bytes(R))
    color = torch.empty((V, 3, H, W), device=dev)
    radii = torch.empty((V, P), dtype=torch.int32, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(L.gsvc_rast_forward_views_launch(
        nv.ref, V, nv.views, V, P, 0, g["means3D"].data_ptr(), None, g["colors_precomp"].data_ptr(),
        g["opacities"].data_ptr(), g["scales"].data_ptr(), g["rotations"].data_ptr(), None, geom.data_ptr(),
        image.data_ptr(), binning.data_ptr(), R, None, color.data_ptr(), radii.data_ptr(), None, 0, st), "launch")
    keys = torch.zeros(R, dtype=torch.int64, device=dev)
    pl = torch.zeros(R, dtype=torch.int32, device=dev)
    ranges = torch.zeros((V * T, 2), dtype=torch.int32, device=dev)
    _lib.check(L.gsvc_rast_export_keys(nv.ref, V, R, image.data_ptr(), binning.data_ptr(), keys.data_ptr(),
                                       pl.data_ptr(), ranges.data_ptr(), st), "export_keys")
    torch.cuda.synchronize()
    keys = keys.cpu().numpy().view(np.uint64)
    pl = pl.cpu().numpy().view(np.uint32)
    ranges = ranges.cpu().numpy().view(np.uint32).astype(np.int64)
    off = 0
    for v, fo in enumerate(fos):
        n = fo["num_rendered"]
        k = keys[off:off + n]
        np.testing.assert_array_equal(k - (np.uint64(v * T) << np.uint64(32)), fo["bin"]["keys"])
        np.testing.assert_array_equal(pl[off:off + n] - np.uint32(v * P), fo["bin"]["point_list"])
        rv = ranges[v * T:(v + 1) * T]
        touched = rv[:, 1] > rv[:, 0]
        exp = fo["bin"]["ranges"].astype(np.int64)
        np.testing.assert_array_equal(rv[touched] - off, exp[touched])
        assert (exp[~touched] == 0).all() and (rv[~touched] == 0).all()
        np.testing.assert_array_equal(radii[v].cpu().numpy(), fo["radii"])
        off += n


def test_view_batch_validation(cuda_device):
    from gsvc_b200.views import ViewBatch, rasterize_views
    from gsvc_b200.rasterizer import RasterizerError
    a = make_scene(P=100, W=64, H=48, F=64, seed=1)
    b = make_scene(P=100, W=80, H=48, F=80, seed=1)
    sa, sb = product_settings(a, cuda_device), product_settings(b, cuda_device)
    with pytest.raises(RasterizerError):
        ViewBatch([sa, sb])                                # different image sizes
    with pytest.raises(RasterizerError):
        ViewBatch([sa] * 17)                               # more than GSVC_RAST_MAX_VIEWS
    with pytest.raises(RasterizerError):
        ViewBatch([sa, sa], out_image=[0, 2])              # gap in the output images
    g = {k: v.to(cuda_device) for k, v in a["gaussians"].items()}
    with pytest.raises(Exception):
        rasterize_views([sa, sa], means3D=g["means3D"], opacities=g["opacities"])   # neither colours nor SHs
    with pytest.raises(RasterizerError):
        rasterize_views([sa, sa], means3D=g["means3D"].cpu(), opacities=g["opacities"],
                        colors_precomp=g["colors_precomp"], scales=g["scales"], rotations=g["rotations"])


def test_frame_streamer_matches_single_frames(cuda_device):
    """graphed.FrameStreamer: independent frames replayed round-robin on several streams equal the frames rendered
    one by one (bit-exact: same kernels), including when a stream's buffers are reused.  `capacity_ok()` holds for
    them, and reports a frame that outgrows its stream's captured capacity."""
    from gsvc_b200.graphed import FrameStreamer
    from gsvc_b200.views import render_toast
    P, W, H, F = 8000, 160, 96, 160
    frames = list(range(76, 86))
    scenes = _scenes(P, W, H, F, seed=53, frames=frames)                 # front/back per frame, one Gaussian set
    params = {k: v.to(cuda_device) for k, v in scenes[0]["gaussians"].items()}
    sets = [product_settings(s, cuda_device) for s in scenes]
    streamer = FrameStreamer(sets[0], sets[1], params, n_streams=3)
    got = []
    for i in range(len(frames)):
        img = streamer.render(sets[2 * i].viewmatrix, sets[2 * i + 1].viewmatrix)
        streamer.wait()
        got.append(img.clone())
    streamer.synchronize()
    with torch.no_grad():
        for i in range(len(frames)):
            ref, _, _ = render_toast(sets[2 * i], sets[2 * i + 1], means3D=params["means3D"], opacities=params["opacities"],
                                     colors_precomp=params["colors_precomp"], scales=params["scales"],
                                     rotations=params["rotations"])
            assert torch.equal(got[i], ref), f"frame {frames[i]}"
    assert not torch.equal(got[0], got[5])
    assert streamer.capacity_ok()
    with torch.no_grad():
        params["scales"].mul_(8.0)                       # the static tensors the graphs read: every splat ~64x the tiles
    streamer.render(sets[0].viewmatrix, sets[1].viewmatrix)
    streamer.synchronize()
    assert not streamer.capacity_ok()


def test_densify_stats_equals_the_reference_expression(cuda_device):
    """sharding.densify_stats == what four training_statis calls accumulate at the rasterizer boundary
    (scene/gaussian_model.py:1311-1314: norm of viewspace_points.grad[radii > 0, :2], a count of 1 per view)."""
    from gsvc_b200 import sharding
    from gsvc_b200.views import rasterize_views
    P, W, H = 15000, 192, 128
    scenes = _scenes(P, W, H, 192, seed=47, frames=(96, 97))
    p = _leaves(scenes[0], cuda_device)
    m2d = torch.zeros((4, P, 3), device=cuda_device, requires_grad=True)
    images, radii, n = rasterize_views([product_settings(s, cuda_device) for s in scenes], means3D=p["means3D"],
                                       opacities=p["opacities"], means2D=m2d, colors_precomp=p["colors_precomp"],
                                       scales=p["scales"], rotations=p["rotations"])
    dL = torch.randn(images.shape, generator=torch.Generator().manual_seed(3)).to(cuda_device)
    images.backward(dL)
    accum = torch.zeros((P, 1), device=cuda_device)
    denom = torch.zeros((P, 1), device=cuda_device)
    for v in range(4):                                           # the reference's four training_statis calls
        update_filter = radii[v] > 0
        accum[update_filter] += torch.norm(m2d.grad[v][update_filter, :2], dim=-1, keepdim=True)
        denom[update_filter] += 1
    assert int((denom > 0).sum()) > 1000 and float(accum.max()) > 0
    stats = sharding.densify_stats(m2d.grad, radii)
    assert torch.equal(stats[:, 1:2], denom)
    assert (stats[:, 0:1] - accum).abs().max() <= 1e-6 * accum.abs().max()
    # into the strided view of the one-collective step buffer, accumulating a second step on top
    flat, packed, view = sharding.step_buffer(P, cuda_device)
    assert flat.numel() == P * 16 and packed.shape == (P, 14) and view.shape == (P, 2)
    sharding.densify_stats(m2d.grad, radii, out=view)
    sharding.densify_stats(m2d.grad, radii, out=view, accumulate=True)
    assert torch.equal(view, 2 * stats) and not bool(packed.count_nonzero())
    # single-view shapes ([P,3], [P]) and errors
    one = sharding.densify_stats(m2d.grad[2], radii[2])
    vis = radii[2] > 0
    assert torch.equal(one[:, 1], vis.float())
    assert (one[:, 0] - torch.norm(m2d.grad[2][:, :2], dim=-1) * vis).abs().max() <= 1e-6 * one[:, 0].max()
    with pytest.raises(Exception):
        sharding.densify_stats(m2d.grad, radii[:2])
    with pytest.raises(Exception):
        sharding.densify_stats(m2d.grad.cpu(), radii.cpu())
