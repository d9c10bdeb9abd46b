"""SURVEY.md §8f row f2, second half: the fused generator epilogue (gsvc_b200.generate, C-ABI gsvc_gen_epilogue_*)
against the reference's PyTorch expression (guassian.py:147-153, 251-293 restated in generate.reference_epilogue) and,
per element, against the float64 oracle of tests/epilogue_oracle.py (docs/SPEC.md U13)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _inputs(N, K, n_vis_frac, device, seed):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    anchor = torch.rand(N, 3, generator=g)
    grid_offsets = 0.3 * r(N, K, 3)
    grid_scaling = torch.exp(0.3 * r(N, 6) - 3.0)
    masks = (torch.rand(N, K, 1, generator=g) > 0.3).float()
    vis = torch.nonzero(torch.rand(N, generator=g) < n_vis_frac).flatten().to(torch.int32)
    n = int(vis.numel())
    nop = torch.tanh(r(n, K))                      # the opacity MLP ends in tanh: about half are <= 0
    color = torch.sigmoid(r(n, K * 3))
    scale_rot = r(n, K * 7)
    noff = 0.1 * r(n, K * 3)
    lo, hi = torch.full((1, 3), 0.05), torch.full((1, 3), 0.95)      # some positions get clamped
    t = [anchor, grid_offsets, grid_scaling, masks, nop, color, scale_rot, noff]
    return [x.to(device) for x in t], vis.to(device), lo.to(device), hi.to(device)


@pytest.mark.parametrize("N,K,frac", [(1000, 10, 0.3), (257, 1, 1.0), (5000, 5, 0.0), (100_000, 10, 0.15), (31, 3, 0.5)])
@pytest.mark.parametrize("gathered", [False, True])
def test_epilogue_matches_the_pytorch_expression(cuda_device, N, K, frac, gathered):
    from gsvc_b200.generate import neural_gaussians_epilogue, reference_epilogue
    t, vis, lo, hi = _inputs(N, K, frac, cuda_device, seed=N + K)
    if gathered:                                     # the caller gathered the per-anchor rows itself
        idx = vis.long()
        t[:4] = [x[idx].contiguous() for x in t[:4]]
        vis = None
    a = [x.clone().requires_grad_(True) for x in t]
    b = [x.clone().requires_grad_(True) for x in t]
    got = neural_gaussians_epilogue(a[0], a[1], a[2], a[3], vis, a[4], a[5], a[6], a[7], lo, hi)
    ref = reference_epilogue(b[0], b[1], b[2], b[3], vis, b[4], b[5], b[6], b[7], lo, hi, K)
    assert torch.equal(got.mask, ref.mask)                                   # same Gaussians, same order
    assert got.xyz.shape == ref.xyz.shape and got.opacity.shape == ref.opacity.shape
    assert torch.equal(got.neural_opacity, ref.neural_opacity) and torch.equal(got.opacity, ref.opacity)
    assert torch.equal(got.color, ref.color)
    for name in ("xyz", "scaling", "rot"):
        x, y = getattr(got, name), getattr(ref, name)
        assert (x - y).abs().max().item() <= 2e-7 * max(1.0, y.abs().max().item()) if y.numel() else True, name
    if ref.xyz.numel() == 0:
        return
    gen = torch.Generator().manual_seed(3)
    w = [torch.randn(x.shape, generator=gen).to(cuda_device) for x in ref[:6]]
    loss = lambda o: sum((getattr(o, f) * wi).sum() for f, wi in zip(("xyz", "color", "opacity", "scaling", "rot", "neural_opacity"), w))
    ga = torch.autograd.grad(loss(got), a)
    gb = torch.autograd.grad(loss(ref), b)
    for name, x, y in zip(("anchor", "grid_offsets", "grid_scaling", "masks", "neural_opacity", "color", "scale_rot", "neural_offset"), ga, gb):
        assert x.shape == y.shape, name
        assert (x - y).abs().max().item() <= 2e-6 * max(1e-6, y.abs().max().item()), name


def test_epilogue_feeds_the_rasterizer(cuda_device):
    """The whole f2 chain without a host synchronisation: visible_filter_compact -> (stub MLP) -> fused epilogue ->
    rasterizer call, and a backward through all of it down to the anchors."""
    from gsvc_b200.generate import neural_gaussians_epilogue
    from gsvc_b200.rasterizer import GaussianRasterizer
    from tests.scenes import make_scene, product_settings
    scene = make_scene(P=4000, W=128, H=96, F=128, seed=3)
    N, K = 4000, 4
    g = {k: v.to(cuda_device) for k, v in scene["gaussians"].items()}
    anchor = g["means3D"].clone().requires_grad_(True)
    scaling6 = torch.cat([g["scales"], g["scales"]], dim=1).requires_grad_(True)
    offsets = (0.5 * torch.randn(N, K, 3, generator=torch.Generator().manual_seed(1))).to(cuda_device).requires_grad_(True)
    masks = torch.ones(N, K, 1, device=cuda_device)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    idx, _ = rast.visible_filter_compact(means3D=anchor.detach(), scales=scaling6.detach()[:, :3], rotations=g["rotations"])
    n = int(idx.numel())
    w = torch.randn(3, 7 * K + 7 * K, generator=torch.Generator().manual_seed(2)).to(cuda_device).requires_grad_(True)
    feat = anchor.index_select(0, idx.long())
    h = torch.tanh(feat @ w)                                                       # the stub "MLP"
    nop, col, sr, noff = h[:, :K], torch.sigmoid(h[:, K:4 * K]), h[:, 4 * K:11 * K], 0.1 * h[:, 11 * K:14 * K]
    gg = neural_gaussians_epilogue(anchor, offsets, scaling6, masks, idx, nop, col, sr, noff,
                                   torch.full((3,), -10.0), torch.full((3,), 10.0))
    assert gg.xyz.shape[0] == int(gg.mask.sum()) > 0 and gg.neural_opacity.shape == (n * K, 1)
    means2D = torch.zeros_like(gg.xyz, requires_grad=True)
    image, radii, num = rast(means3D=gg.xyz, means2D=means2D, shs=None, colors_precomp=gg.color, opacities=gg.opacity,
                             scales=gg.scaling, rotations=gg.rot, cov3D_precomp=None)
    image.square().sum().backward()
    for t in (anchor, scaling6, offsets, w):
        assert t.grad is not None and torch.isfinite(t.grad).all() and t.grad.abs().sum() > 0
    assert (anchor.grad[torch.ones(N, dtype=torch.bool, device=cuda_device).index_fill(0, idx.long(), False)] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------
# Against the float64 oracle (tests/epilogue_oracle.py, docs/SPEC.md U13), per element: mask, row order, opacity,
# neural_opacity, colour and xyz bit-exact; scaling and rot to 8 (u |ref| + 2^-149); every gradient element to
# (8 + K) (u A + 2^-149), A the sum of the absolute values of its terms.  u = 2^-24.

import numpy as np                       # noqa: E402

from tests import epilogue_oracle as O   # noqa: E402

_DIFF = ("anchor", "grid_offsets", "grid_scaling", "masks", "neural_opacity", "color", "scale_rot", "neural_offset")


def _device_run(t, device, cot):
    """Forward and backward of the fused epilogue; cot maps output name -> numpy cotangent (absent: not in the loss)."""
    from gsvc_b200.generate import neural_gaussians_epilogue
    x = [torch.from_numpy(np.ascontiguousarray(t[k])).to(device).requires_grad_(True) for k in _DIFF]
    vis = None if t["visible_indices"] is None else torch.from_numpy(t["visible_indices"]).to(device)
    lo, hi = (torch.from_numpy(t[k]).to(device) for k in ("bound_min", "bound_max"))
    got = neural_gaussians_epilogue(x[0], x[1], x[2], x[3], vis, x[4], x[5], x[6], x[7], lo, hi)
    loss = sum((getattr(got, k) * torch.from_numpy(np.ascontiguousarray(w, dtype=np.float32)).to(device)).sum()
               for k, w in cot.items())
    grads = torch.autograd.grad(loss, x)
    return got, grads


def _cotangents(f, seed, which=O.OUTPUTS):
    rng = np.random.default_rng(seed)
    shapes = {"xyz": (f["M"], 3), "color": (f["M"], 3), "opacity": (f["M"], 1), "scaling": (f["M"], 3),
              "rot": (f["M"], 4), "neural_opacity": (f["n_vis"] * f["K"], 1)}
    return {k: rng.standard_normal(shapes[k]).astype(np.float32) for k in which}


def _check(t, device, tag, seed=7, which=O.OUTPUTS):
    """Everything U13 promises, for one input set; prints the margins (-rA shows them)."""
    f = O.forward(*[t[k] for k in O.ARGS])
    cot = _cotangents(f, seed, which)
    got, grads = _device_run(t, device, cot)
    sel = got.mask.cpu().numpy()
    assert np.array_equal(sel, f["sel"]), f"{tag}: selection differs"
    assert got.xyz.shape == (f["M"], 3) and got.opacity.shape == (f["M"], 1)
    same = lambda a, b: np.array_equal(a.detach().cpu().numpy().astype(np.float64), b, equal_nan=True)
    for k in ("neural_opacity", "opacity", "color", "xyz"):
        g, r = getattr(got, k).detach().cpu().numpy().astype(np.float64), f[k]
        bad = np.flatnonzero(~((g == r) | (np.isnan(g) & np.isnan(r))).reshape(-1))
        assert bad.size == 0, f"{tag}: {k} not bit-exact at {bad.size} elements, e.g. {bad[:4]}: {g.flat[bad[:4]]} vs {r.flat[bad[:4]]}"
    assert same(got.neural_opacity, f["neural_opacity"])
    rep = {}
    for k in ("scaling", "rot"):
        O.check(k, getattr(got, k).detach().cpu().numpy(), f[k], np.abs(f[k]), 8, rep)
    ref = O.backward(f, **{("d_" + k): v for k, v in cot.items()})
    for k, g in zip(_DIFF, grads):
        O.check("d_" + k, g.cpu().numpy(), ref[k][0], ref[k][1], 8 + f["K"], rep)
    print(f"{tag}: M={f['M']} of {f['n_vis'] * f['K']}; worst err/(u*A + 2^-149): "
          + " ".join(f"{k}={v:.2f}" for k, v in rep.items()))
    return f, got


_SHAPES = [  # (N, n_vis, K): n_vis * K = 1, 31, 32, 33, 255, 256, 257, 262143, 262144, 262145, 262150, 1 M
    (4, 1, 1), (40, 31, 1), (3, 1, 32), (20, 11, 3), (30, 15, 17), (12, 8, 32), (300, 257, 1), (100_000, 87_381, 3),
    (10_000, 8192, 32), (300_000, 262_145, 1), (6000, 5243, 50), (600_000, 100_000, 10)]


@pytest.mark.parametrize("form", ["gathered", "indexed", "shuffled"])
@pytest.mark.parametrize("N,n_vis,K", _SHAPES)
def test_epilogue_matches_the_float64_oracle(cuda_device, N, n_vis, K, form):
    """Every entry count around the 256-entry CTAs and the compaction scan's 262 144-entry passes, up to the bench
    shape (600 k anchors, 100 k visible, K = 10: four scan passes)."""
    _check(O.make_inputs(N, n_vis, K, seed=N + n_vis + K, form=form), cuda_device, f"{form} n_vis={n_vis} K={K}")


@pytest.mark.parametrize("pattern", ["all", "none", "first_last", "every256", "alternating"])
def test_epilogue_selection_patterns(cuda_device, pattern):
    """600 000 entries (three scan passes); "none" is M = 0 with n_vis > 0, backward through neural_opacity only."""
    t = O.selection_inputs(80_000, 60_000, 10, seed=5, pattern=pattern)
    f, got = _check(t, cuda_device, f"pattern {pattern}",
                    which=("neural_opacity",) if pattern == "none" else O.OUTPUTS)
    assert f["M"] == {"all": 600_000, "none": 0, "first_last": 2, "every256": 2344, "alternating": 300_000}[pattern]


@pytest.mark.parametrize("form", ["gathered", "indexed", "shuffled"])
def test_epilogue_edge_values(cuda_device, form):
    """NaN / +-Inf / +-0 / underflowing / subnormal opacity products, NaN and +-Inf offsets and anchors, positions on
    and one ulp outside the bounds, FMA-boundary positions, saturated sigmoids, quaternions at F.normalize's eps."""
    _check(O.edge_inputs(seed=1, form=form), cuda_device, f"edges {form}")
    _check(O.edge_inputs(seed=2, form=form), cuda_device, f"edges {form} opacity cotangent only",
           which=("neural_opacity",))


def test_nan_position_propagates(cuda_device):
    """A NaN neural_offset gives a NaN xyz (torch.clamp propagates NaN), not a splat at bound_min."""
    t = O.make_inputs(64, 64, 4, seed=3, form="gathered")
    t["neural_opacity"][:] = 0.5
    t["masks"][:] = 1.0
    t["neural_offset"][5, :] = np.nan
    f, got = _check(t, cuda_device, "nan offsets")
    xyz = got.xyz.detach().cpu().numpy()
    assert np.isnan(xyz[20:24]).all() and not np.isnan(np.delete(xyz, range(20, 24), axis=0)).any()


def test_clamp_gradient_at_the_fma_boundary(cuda_device):
    """Positions whose separately rounded value is on a bound while the fused fl(an + s * gs) is outside, and the
    converse, on both bounds of every component: the gradient mask is the reference's."""
    t = O.edge_inputs(seed=3, form="indexed")
    E = t["neural_opacity"].size
    keep = np.zeros(E, bool)
    keep[:192 * 10] = True                                  # edge_inputs puts the FMA-boundary anchors first
    t["neural_opacity"] = np.where(keep.reshape(t["neural_opacity"].shape), t["neural_opacity"], -1.0).astype(np.float32)
    f = O.forward(*[t[k] for k in O.ARGS])
    cot = _cotangents(f, 7, ("xyz",))
    _, grads = _device_run(t, cuda_device, cot)
    ref = O.backward(f, d_xyz=cot["xyz"])
    O.check("d_anchor", grads[0].cpu().numpy(), *ref["anchor"], 8 + f["K"], {})      # the clamp's gradient mask first
    _check(t, cuda_device, "fma boundary", which=("xyz",))


def test_normalize_gradient_below_eps(cuda_device):
    """Below F.normalize's eps the rotation gradient is dr / 1e-12 (clamp_min stops the norm's gradient)."""
    t = O.make_inputs(8, 8, 2, seed=4, form="gathered")
    t["neural_opacity"][:] = 0.5
    t["masks"][:] = 1.0
    sr = t["scale_rot"].reshape(8, 2, 7)
    sr[0, 0, 3:] = (3e-13, 4e-13, 0, 0)
    sr[1, 1, 3:] = (0, 0, 0, 0)
    sr[2, 0, 3:] = (np.float32(1e-12), 0, 0, 0)
    sr[3, 1, 3:] = (1e-13, -2e-13, 3e-13, 1e-13)
    _check(t, cuda_device, "normalize eps", which=("rot",))


def test_epilogue_is_deterministic(cuda_device):
    """Forward and backward bitwise equal over two runs (the backward has no atomics)."""
    t = O.make_inputs(600_000, 100_000, 10, seed=9, form="shuffled")
    f = O.forward(*[t[k] for k in O.ARGS])
    cot = _cotangents(f, 1)
    runs = [_device_run(t, cuda_device, cot) for _ in range(2)]
    bits = lambda x: x.detach().contiguous().view(torch.int32) if x.dtype == torch.float32 else x
    for a, b in zip(runs[0][0], runs[1][0]):
        assert torch.equal(bits(a), bits(b))
    for a, b in zip(runs[0][1], runs[1][1]):
        assert torch.equal(bits(a), bits(b))


def test_nan_offset_row_is_culled_by_the_rasterizer(cuda_device):
    """End to end: a NaN neural_offset row reaches the rasterizer as a NaN position, which culls it (radius 0)."""
    from gsvc_b200.generate import neural_gaussians_epilogue
    from gsvc_b200.rasterizer import GaussianRasterizer
    from tests.scenes import make_scene, product_settings
    scene = make_scene(P=256, W=64, H=48, F=64, seed=5)
    g = {k: v.to(cuda_device) for k, v in scene["gaussians"].items()}
    N, K = 256, 2
    anchor = g["means3D"]
    scaling6 = torch.cat([g["scales"], g["scales"]], dim=1)
    offsets = torch.zeros(N, K, 3, device=cuda_device)
    noff = torch.zeros(N, K * 3, device=cuda_device)
    noff[7, :3] = float("nan")                               # entry 14: row 14 of the output (everything is selected)
    rot = g["rotations"].repeat_interleave(K, 0).reshape(N, K * 4)
    sr = torch.cat([torch.full((N, K, 3), 2.0, device=cuda_device), rot.reshape(N, K, 4)], dim=2).reshape(N, K * 7)
    gg = neural_gaussians_epilogue(anchor, offsets, scaling6, torch.ones(N, K, 1, device=cuda_device), None,
                                   torch.full((N, K), 0.5, device=cuda_device), g["colors_precomp"].repeat(1, K), sr,
                                   noff, torch.full((3,), -1e4), torch.full((3,), 1e4))
    assert gg.xyz.shape[0] == N * K and torch.isnan(gg.xyz[14]).all() and torch.isfinite(gg.xyz[15]).all()
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    _, radii, _ = rast(means3D=gg.xyz, means2D=torch.zeros_like(gg.xyz), shs=None, colors_precomp=gg.color,
                       opacities=gg.opacity, scales=gg.scaling, rotations=gg.rot, cov3D_precomp=None)
    assert int(radii[14]) == 0 and int((radii[::2][:7] > 0).sum()) > 0
