"""GPU parity of the batched-view path (gsvc_b200.views) in the input modes and view-to-image maps that toast pairs of
`colors_precomp` scenes do not reach: SH colours evaluated from each view's own camera, precomputed covariances, a
scale modifier, and general maps (three views in one image, n_out strictly between 1 and V, a flipped view without a
partner, weights other than 0.5 and 1, views that share an image without being adjacent).

Every comparison goes through tests/parity.py.  The reference of a batch is composed from one oracle call per view:
image o = sum over the views v with out_image[v] = o of weight[v] * flip_v(C_v), where C_v already holds T * bg.
"""
import dataclasses

import numpy as np
import pytest
import torch

from oracle import c_oracle
from tests import parity
from tests.scenes import make_scene, np_inputs, product_settings

pytestmark = pytest.mark.gpu

# two GPU runs of the same backward differ by the order of the float atomics (tests/test_gpu_views.py)
ATOMIC_RTOL = 4e-5

W, H, F = 150, 90, 160          # W not a multiple of the 16-pixel tile: mirrored pixels fall in different tiles


def _flip(a, flip):
    return np.ascontiguousarray(a[..., ::-1]) if flip else a


def _window(P, frames, seed, **kw):
    """Front and back scenes of several frames over ONE Gaussian set: views [f0 front, f0 back, f1 front, ...]."""
    base = make_scene(P=P, W=W, H=H, F=F, frame=frames[0], seed=seed, window=len(frames), **kw)
    out = []
    for f in frames:
        for back in (False, True):
            sc = make_scene(P=P, W=W, H=H, F=F, frame=f, seed=seed, back=back, **kw)
            sc["gaussians"] = base["gaussians"]
            out.append(sc)
    return out


class ComposedOracle:
    """The oracle of one view batch: `sts` oracle settings per view, map (out_image, flip_x, weight), inputs `gi`."""

    def __init__(self, sts, gi, out_image, flip_x, weight):
        self.out_image, self.flip_x, self.weight = list(out_image), list(flip_x), list(weight)
        self.n_out = max(self.out_image) + 1
        self.fos = [parity.oracle_forward(st, gi) for st in sts]
        self.color = np.zeros((self.n_out, 3, H, W), np.float64)
        self.fragile = np.zeros((self.n_out, H, W), bool)       # union of the flipped fragile sets of an image's views
        for v, fo in enumerate(self.fos):
            o = self.out_image[v]
            self.color[o] += self.weight[v] * _flip(fo["color"].astype(np.float64), self.flip_x[v])
            self.fragile[o] |= _flip(fo["fragile"], self.flip_x[v])
        self.views_of = [[v for v in range(len(sts)) if self.out_image[v] == o] for o in range(self.n_out)]
        # visible in any view: the Gaussians whose summed gradients are compared
        self.any_view = dict(radii=np.max([fo["radii"] for fo in self.fos], axis=0))

    def num_rendered(self):
        return sum(fo["num_rendered"] for fo in self.fos)

    def check_forward(self, images, max_fragile=parity.MAX_FRAGILE):
        """Every image within 1e-5 * sum |w| of the reference off its fragile set; that set bounded per view."""
        got = images.detach().cpu().numpy()
        worst = 0.0
        for o, views in enumerate(self.views_of):
            assert self.fragile[o].mean() <= len(views) * max_fragile, (o, self.fragile[o].mean())
            tol = parity.FWD_ATOL * sum(abs(self.weight[v]) for v in views)
            err = float(np.abs(got[o] - self.color[o])[:, ~self.fragile[o]].max())
            assert err <= tol, f"image {o}: max abs err {err:.3e} > {tol:.1e}"
            worst = max(worst, err)
        return worst

    def backward(self, dL):
        """dL [n_out,3,H,W] → (seed masked on each image's fragile union, per-view oracle gradients)."""
        dL = np.array(dL, np.float32, copy=True)
        for o in range(self.n_out):
            dL[o][:, self.fragile[o]] = 0.0
        gos = []
        for v, fo in enumerate(self.fos):
            seed = np.float32(self.weight[v]) * _flip(dL[self.out_image[v]], self.flip_x[v])
            gos.append(parity.oracle_backward(fo, np.ascontiguousarray(seed, dtype=np.float32)))
        return dL, gos

    @staticmethod
    def summed(gos, names):
        return {k: sum(np.asarray(go[k], np.float64) for go in gos) for k in names}


def _leaves(gi, names, device):
    return {k: torch.as_tensor(gi[k]).to(device).clone().requires_grad_(True) for k in names}


def _check_summed_and_per_view(orc, gos, grads, m2d_grad, names):
    """check_grads on the view-summed parameters, then on each view's means2D; returns the worst stats."""
    stats = parity.check_grads(orc.any_view, ComposedOracle.summed(gos, names), dict(zip(names, grads)),
                               what="summed ")
    worst = dict(rel=stats["rel"], row_worst=stats["row_worst"], m2d_rel=0.0, m2d_row_worst=0.0)
    for v, (fo, go) in enumerate(zip(orc.fos, gos)):
        s = parity.check_grads(fo, go, dict(means2D=m2d_grad[v]), what=f"view {v} ")
        worst["m2d_rel"] = max(worst["m2d_rel"], s["rel"])
        worst["m2d_row_worst"] = max(worst["m2d_row_worst"], s["row_worst"])
    return worst


def _report(case, fwd, g):
    """One line per case for the parity records (pytest -rA shows it)."""
    print(f"{case}: forward max err {fwd:.2e}; summed grads rel {g['rel']:.2e} row_worst {g['row_worst']:.3f}; "
          f"means2D rel {g['m2d_rel']:.2e} row_worst {g['m2d_row_worst']:.3f}")


def _single_calls(settings, batch_map, leaves, names, colour, geometry, dL):
    """The batch as single GaussianRasterizer calls: (composed images, radii, num_rendered, summed grads, means2D grads)."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    out_image, flip_x, weight = batch_map
    images, radii, n, sums, m2d = None, [], 0, None, []
    for v, rs in enumerate(settings):
        m = torch.zeros_like(leaves["means3D"], requires_grad=True)
        c, r, k = GaussianRasterizer(raster_settings=rs)(means3D=leaves["means3D"], means2D=m,
                                                         opacities=leaves["opacities"], **colour, **geometry)
        seed = weight[v] * dL[out_image[v]]
        seed = seed.flip(-1) if flip_x[v] else seed
        g = torch.autograd.grad(c, [leaves[k] for k in names] + [m], grad_outputs=seed)
        c = weight[v] * (c.flip(-1) if flip_x[v] else c)
        if images is None:
            images = torch.zeros((max(out_image) + 1,) + tuple(c.shape), device=c.device)
        images[out_image[v]] += c
        radii.append(r)
        n += k
        sums = list(g[:-1]) if sums is None else [a + b for a, b in zip(sums, g[:-1])]
        m2d.append(g[-1])
    return images, torch.stack(radii), n, sums, m2d


def _check_against_single_calls(single, images, radii, n, grads, m2d_grad, names, exact_images):
    s_images, s_radii, s_n, s_sums, s_m2d = single
    assert n == s_n
    assert torch.equal(radii, s_radii)
    if exact_images:
        assert torch.equal(images, s_images)
    for k, a, b in zip(names, grads, s_sums):
        assert (a - b).abs().max() <= ATOMIC_RTOL * b.abs().max(), k
    for v, b in enumerate(s_m2d):
        assert (m2d_grad[v] - b).abs().max() <= ATOMIC_RTOL * b.abs().max(), f"means2D of view {v}"


def _export_batch_geometry(batch, device, g, P, R):
    """Preprocess outputs of a directly launched batch, per view: the virtual Gaussian v*P+g of gsvc_rast_export_geom."""
    from gsvc_b200 import _lib
    from gsvc_b200.rasterizer import _NativeViews
    L = _lib.lib()
    V = batch.n_views
    sh_M = g["shs"].shape[1] if "shs" in g else 0
    nv = _NativeViews(batch, device)
    u8 = lambda n: torch.empty(int(n), dtype=torch.uint8, device=device)
    geom, image = u8(L.gsvc_rast_geom_bytes(P * V, sh_M)), u8(L.gsvc_rast_image_bytes_views(W, H, V))
    binning = u8(L.gsvc_rast_binning_bytes(R))
    color = torch.empty((batch.n_out, 3, H, W), device=device)
    radii = torch.empty((V, P), dtype=torch.int32, device=device)
    st = torch.cuda.current_stream(device).cuda_stream
    ptr = lambda k: g[k].data_ptr() if k in g else None
    _lib.check(L.gsvc_rast_forward_views_launch(
        nv.ref, V, nv.views, batch.n_out, P, sh_M, ptr("means3D"), ptr("shs"), ptr("colors_precomp"), ptr("opacities"),
        ptr("scales"), ptr("rotations"), ptr("cov3D_precomp"), geom.data_ptr(), image.data_ptr(), binning.data_ptr(), R,
        None, color.data_ptr(), radii.data_ptr(), None, 0, st), "gsvc_rast_forward_views_launch")
    f32 = dict(dtype=torch.float32, device=device)
    out = dict(depth=torch.zeros(P * V, **f32), xy=torch.zeros((P * V, 2), **f32),
               conic_opacity=torch.zeros((P * V, 4), **f32), rgb=torch.zeros((P * V, 3), **f32),
               rect=torch.zeros((P * V, 4), dtype=torch.int32, device=device))
    _lib.check(L.gsvc_rast_export_geom(P * V, sh_M, geom.data_ptr(), out["depth"].data_ptr(), out["xy"].data_ptr(),
                                       out["conic_opacity"].data_ptr(), out["rgb"].data_ptr(), out["rect"].data_ptr(),
                                       st), "gsvc_rast_export_geom")
    torch.cuda.synchronize(device)
    return radii.cpu().numpy(), {k: v.cpu().numpy().reshape((V, P) + tuple(v.shape[1:])) for k, v in out.items()}


def _clamp_flags_differ(fos):
    """Share of the Gaussians visible in some view whose SH clamp flags differ between two views that both see it."""
    vis = np.stack([fo["radii"] > 0 for fo in fos])                     # [V,P]
    fl = np.stack([fo["pre"]["clamped"] for fo in fos]).astype(np.int8)  # [V,P,3]
    hi = np.where(vis[..., None], fl, 0).max(axis=0)                    # some view that sees it clamps
    lo = np.where(vis[..., None], fl, 1).min(axis=0)                    # some view that sees it does not
    differ = (hi > lo).any(axis=1)
    return float(differ.sum() / max(int(vis.any(axis=0).sum()), 1))


@pytest.mark.parametrize("n_frames", [3, 8])
@pytest.mark.parametrize("deg", [1, 3])
def test_sh_window_matches_oracle(cuda_device, deg, n_frames):
    """SH colours over a window of frames (6 and 16 = GSVC_RAST_MAX_VIEWS views, one image per view), each view with a
    camera of its own, scale_modifier 0.7: the colour, its clamp flags and the SH gradient's direction term differ per
    view, and dL/dshs / dL/dmeans3D are summed over the views."""
    from gsvc_b200.views import ViewBatch, rasterize_views
    dev = cuda_device
    P = 6000
    frames = tuple(range(76, 76 + n_frames))
    scenes = _window(P, frames, seed=60 + deg, scale_modifier=0.7)
    V = len(scenes)
    rng = np.random.default_rng(1000 + 10 * deg + V)
    deltas = (rng.uniform(0.1, 0.5, (V, 3)) * rng.choice([-1.0, 1.0], (V, 3))).astype(np.float32)
    gi = np_inputs(scenes[0]["gaussians"])
    gi.pop("colors_precomp")
    gi["shs"] = (torch.randn(P, 16, 3, generator=torch.Generator().manual_seed(deg)) * 0.4).numpy()
    sts, settings = [], []
    for sc, d in zip(scenes, deltas):
        cam = sc["frame"].cam_pos + torch.from_numpy(d)
        sts.append(dataclasses.replace(sc["oracle_settings"], sh_degree=deg, campos=cam.numpy()))
        settings.append(product_settings(sc, dev, sh_degree=deg)._replace(campos=cam))
    batch_map = (list(range(V)), [False] * V, [1.0] * V)
    orc = ComposedOracle(sts, gi, *batch_map)
    assert _clamp_flags_differ(orc.fos) >= 0.01
    batch = ViewBatch(settings)

    # preprocess outputs per view, SH-derived colours included: bit-exact (preprocess.cu is built without contraction)
    g = {k: torch.as_tensor(v).to(dev).contiguous() for k, v in gi.items()}
    radii, geo = _export_batch_geometry(batch, dev, g, P, orc.num_rendered())
    for v, fo in enumerate(orc.fos):
        np.testing.assert_array_equal(radii[v], fo["radii"])
        for k in ("depth", "xy", "conic_opacity", "rgb", "rect"):
            np.testing.assert_array_equal(geo[k][v], fo["pre"][k], err_msg=f"view {v} {k}")

    names = ("shs", "means3D", "scales", "rotations", "opacities")
    p = _leaves(gi, names, dev)
    m2d = torch.zeros((V, P, 3), device=dev, requires_grad=True)
    images, radii, n = rasterize_views(batch, means3D=p["means3D"], opacities=p["opacities"], means2D=m2d,
                                       shs=p["shs"], scales=p["scales"], rotations=p["rotations"])
    assert n == orc.num_rendered()
    fwd = 0.0
    for v, fo in enumerate(orc.fos):
        np.testing.assert_array_equal(radii[v].cpu().numpy(), fo["radii"])
        fwd = max(fwd, parity.check_forward(fo, images[v])["err"])
    dL, gos = orc.backward(torch.randn((V, 3, H, W), generator=torch.Generator().manual_seed(deg + V)).numpy())
    dL = torch.as_tensor(dL).to(dev)
    grads = torch.autograd.grad(images, [p[k] for k in names] + [m2d], grad_outputs=dL)
    _report(f"sh deg={deg} views={V}", fwd, _check_summed_and_per_view(orc, gos, grads[:-1], grads[-1], names))
    single = _single_calls(settings, batch_map, p, names, dict(shs=p["shs"]),
                           dict(scales=p["scales"], rotations=p["rotations"]), dL)
    _check_against_single_calls(single, images, radii, n, grads[:-1], grads[-1], names, exact_images=True)


def _covariances(st, gi):
    """cov3D_precomp for every Gaussian as test_cov3d_precomp_path builds it: the oracle's preprocess over a wide-open
    slab, a benign covariance for the rows it leaves zero (degenerate or off the image)."""
    cov = c_oracle.preprocess(dataclasses.replace(st, threshold=1e9), gi["means3D"], gi["scales"],
                              gi["rotations"])["cov3D"]
    cov[np.all(cov == 0, axis=1)] = np.array([1e-6, 0, 0, 1e-6, 0, 1e-6], np.float32)
    return cov


@pytest.mark.parametrize("needle_mix", [None, 0.05])
def test_cov3d_precomp_window_matches_oracle(cuda_device, needle_mix):
    """Precomputed covariances over two frames composed as toasts: dL/dcov3D_precomp summed over 4 views."""
    from gsvc_b200.views import ViewBatch, rasterize_views
    dev = cuda_device
    P = 8000
    scenes = _window(P, (80, 81), seed=71, needle_mix=needle_mix)
    gi = np_inputs(scenes[0]["gaussians"])
    gi["cov3D_precomp"] = _covariances(scenes[0]["oracle_settings"], gi)
    gi.pop("scales")
    gi.pop("rotations")
    settings = [product_settings(sc, dev) for sc in scenes]
    batch = ViewBatch.toasts([settings[0:2], settings[2:4]])
    batch_map = (batch.out_image, batch.flip_x, batch.weight)
    orc = ComposedOracle([sc["oracle_settings"] for sc in scenes], gi, *batch_map)
    names = ("cov3D_precomp", "means3D", "opacities", "colors_precomp")
    p = _leaves(gi, names, dev)
    m2d = torch.zeros((4, P, 3), device=dev, requires_grad=True)
    images, radii, n = rasterize_views(batch, means3D=p["means3D"], opacities=p["opacities"], means2D=m2d,
                                       colors_precomp=p["colors_precomp"], cov3D_precomp=p["cov3D_precomp"])
    assert n == orc.num_rendered()
    for v, fo in enumerate(orc.fos):
        np.testing.assert_array_equal(radii[v].cpu().numpy(), fo["radii"])
    fwd = orc.check_forward(images, max_fragile=5e-3 if needle_mix else parity.MAX_FRAGILE)
    dL, gos = orc.backward(torch.randn((2, 3, H, W), generator=torch.Generator().manual_seed(12)).numpy())
    dL = torch.as_tensor(dL).to(dev)
    grads = torch.autograd.grad(images, [p[k] for k in names] + [m2d], grad_outputs=dL)
    _report(f"cov3D_precomp needle_mix={needle_mix}", fwd,
            _check_summed_and_per_view(orc, gos, grads[:-1], grads[-1], names))
    single = _single_calls(settings, batch_map, p, names, dict(colors_precomp=p["colors_precomp"]),
                           dict(cov3D_precomp=p["cov3D_precomp"]), dL)
    # 0.5 * a + 0.5 * b onto a zeroed image rounds the same in either order: the toast images are bit-exact
    _check_against_single_calls(single, images, radii, n, grads[:-1], grads[-1], names, exact_images=True)


MAPS = {
    # 5 views of 3 frames into 3 images: three views in image 0, a flipped view without a partner, weights != 0.5, 1
    "three_in_one": ([0, 1, 2, 3, 4], [0, 0, 0, 1, 2], [False, True, False, True, True], [0.2, 0.3, 0.5, 1.0, 1.5]),
    # 3 views into one image, none flipped
    "all_in_one": ([0, 1, 2], [0, 0, 0], [False, False, False], [1.0, 1.0, 1.0]),
    # views that share an image are never neighbours in the batch
    "interleaved": ([0, 1, 2, 3], [0, 1, 0, 1], [False, True, True, False], [0.5, 0.25, 0.75, 2.0]),
}


@pytest.mark.parametrize("name", sorted(MAPS))
def test_general_view_maps_match_oracle(cuda_device, name):
    """General view-to-image maps, colors_precomp with scales / rotations, a non-zero background."""
    from gsvc_b200.views import ViewBatch, rasterize_views
    dev = cuda_device
    P = 8000
    pick, out_image, flip_x, weight = MAPS[name]
    window = _window(P, (78, 79, 80), seed=83)
    scenes = [window[i] for i in pick]
    V = len(scenes)
    gi = np_inputs(scenes[0]["gaussians"])
    settings = [product_settings(sc, dev) for sc in scenes]
    batch = ViewBatch(settings, out_image=out_image, flip_x=flip_x, weight=weight)
    orc = ComposedOracle([sc["oracle_settings"] for sc in scenes], gi, out_image, flip_x, weight)
    names = ("means3D", "scales", "rotations", "opacities", "colors_precomp")
    p = _leaves(gi, names, dev)
    m2d = torch.zeros((V, P, 3), device=dev, requires_grad=True)
    images, radii, n = rasterize_views(batch, means3D=p["means3D"], opacities=p["opacities"], means2D=m2d,
                                       colors_precomp=p["colors_precomp"], scales=p["scales"], rotations=p["rotations"])
    assert images.shape == (orc.n_out, 3, H, W)
    assert n == orc.num_rendered()
    for v, fo in enumerate(orc.fos):
        np.testing.assert_array_equal(radii[v].cpu().numpy(), fo["radii"])
    fwd = orc.check_forward(images)
    dL, gos = orc.backward(torch.randn((orc.n_out, 3, H, W), generator=torch.Generator().manual_seed(V)).numpy())
    grads = torch.autograd.grad(images, [p[k] for k in names] + [m2d], grad_outputs=torch.as_tensor(dL).to(dev))
    _report(f"map {name}", fwd, _check_summed_and_per_view(orc, gos, grads[:-1], grads[-1], names))


def test_view_batch_rejects_settings_that_differ(cuda_device):
    """A batch shares one preprocess: views that differ in SH degree, scale modifier or background are refused; an
    equal background held in another tensor is accepted.  means2D must be [n_views, P, 3]."""
    from gsvc_b200.rasterizer import RasterizerError
    from gsvc_b200.views import ViewBatch, rasterize_views
    a = make_scene(P=100, W=64, H=48, F=64, seed=1)
    sa = product_settings(a, cuda_device)
    for other in (sa._replace(sh_degree=1), sa._replace(scale_modifier=0.5),
                  sa._replace(bg=torch.tensor([0.1, 0.2, 0.4], device=cuda_device))):
        with pytest.raises(RasterizerError):
            ViewBatch([sa, other])
        with pytest.raises(RasterizerError):
            ViewBatch([other, sa, sa])
    assert ViewBatch([sa, sa._replace(bg=sa.bg.clone())]).n_views == 2
    g = {k: v.to(cuda_device) for k, v in a["gaussians"].items()}
    kw = dict(means3D=g["means3D"], opacities=g["opacities"], colors_precomp=g["colors_precomp"], scales=g["scales"],
              rotations=g["rotations"])
    for shape in ((100, 3), (2, 100, 2), (3, 100, 3), (2, 99, 3)):
        with pytest.raises(RasterizerError, match="means2D"):
            rasterize_views([sa, sa], means2D=torch.zeros(shape, device=cuda_device, requires_grad=True), **kw)


def test_background_check_survives_a_reused_address(cuda_device):
    """ViewBatch compares two CUDA backgrounds once per pair of tensors.  When a pair of equal backgrounds is freed, the
    caching allocator hands their addresses to the next tensors of that size (same addresses, version 0 again): a pair
    that differs must still be refused rather than answered from the first pair's result."""
    from gsvc_b200.rasterizer import RasterizerError
    from gsvc_b200.views import ViewBatch
    sa = product_settings(make_scene(P=100, W=64, H=48, F=64, seed=1), cuda_device)
    reused = 0
    for _ in range(4):
        a = torch.tensor([0.1, 0.2, 0.3], device=cuda_device)
        b = torch.tensor([0.1, 0.2, 0.3], device=cuda_device)
        assert ViewBatch([sa._replace(bg=a), sa._replace(bg=b)]).n_views == 2
        ptrs = (a.data_ptr(), b.data_ptr())
        del a, b
        c = torch.tensor([0.1, 0.2, 0.3], device=cuda_device)
        d = torch.tensor([0.9, 0.2, 0.3], device=cuda_device)
        reused += (c.data_ptr(), d.data_ptr()) == ptrs
        with pytest.raises(RasterizerError, match="background"):
            ViewBatch([sa._replace(bg=c), sa._replace(bg=d)])
    assert reused, "the allocator never reused the addresses: this test no longer sets up the case it is about"
