"""GPU parity of the blend backward on deep per-pixel lists (tests/deep_scenes.py), against the referee oracle and, on
the heavy scene and the deepest ladder rung, against float64 autograd through the PyTorch restatement.

render_backward_kernel replays a tile back to front in batches of 256 staged Gaussians: the first batch of a tile
that is not saturated from speculatively fetched ids, every other batch from the point list, with one hit list per
8x8 block and batch.  The scenes here put tiles exactly at and across the batch boundaries, thousands of entries deep,
saturated and not, with the two blocks of a warp far out of balance, and through the batched paths (toast, ragged).
Each test first asserts from the oracle's outputs that its scene is in the regime it names; then forward (n_contrib
exact, final_T within 1e-5) and every visible Gaussian's gradient are held to the bars of tests/parity.py."""
import json

import numpy as np
import pytest
import torch

from tests import deep_scenes as D
from tests import parity
from tests.scenes import np_inputs, product_settings

pytestmark = pytest.mark.gpu

NAMES = parity.GRAD_NAMES
DL_SEED = 17                   # the seed gradient of tests/test_deep_oracle_cpu.py's float64 comparison


def _oracle(scene):
    return parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]))


def _per_tensor(fo, go, got, what):
    """check_grads tensor by tensor; returns {name: (rel, row_worst)} for the test's report line."""
    out = {}
    for k in got:
        s = parity.check_grads(fo, go, got, names=(k,), what=what)
        out[k] = (round(s["rel"], 9), round(s["row_worst"], 4))
    return out


def _report(what, stats):
    print(f"deep-grads {what} {json.dumps(stats)}")


def _check_scene(scene, dev, what, max_fragile=parity.MAX_FRAGILE, f64=False):
    """Forward (stages, n_contrib, final_T) and backward of one scene against the referee oracle; `f64`: the
    gradients also against float64 autograd.  Returns the oracle forward."""
    from gsvc_b200.rasterizer import GaussianRasterizer, RasterState
    fo = _oracle(scene)
    rs = product_settings(scene, dev)
    g = {k: v.to(dev) for k, v in scene["gaussians"].items()}
    state = RasterState(rs, g["means3D"], g["opacities"], colors_precomp=g["colors_precomp"], scales=g["scales"],
                        rotations=g["rotations"])
    assert state.num_rendered == fo["num_rendered"]
    fT, nc = state.export_image()
    parity.check_forward(fo, state.color, fT, nc, max_fragile=max_fragile)
    p = {k: v.clone().requires_grad_(True) for k, v in g.items()}
    m2d = torch.zeros_like(p["means3D"], requires_grad=True)
    color, radii, n = GaussianRasterizer(raster_settings=rs)(
        means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"], opacities=p["opacities"],
        scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
    assert n == fo["num_rendered"]
    np.testing.assert_array_equal(radii.cpu().numpy(), fo["radii"])
    parity.check_forward(fo, color, max_fragile=max_fragile)
    dL = D.seed_dL(fo, DL_SEED)
    color.backward(torch.as_tensor(dL).to(dev))
    got = {k: p[k].grad for k in NAMES}
    got["means2D"] = m2d.grad
    stats = {"referee": _per_tensor(fo, parity.oracle_backward(fo, dL), got, f"{what} vs referee: ")}
    if f64:
        stats["float64"] = _per_tensor(fo, D.f64_reference(scene, dL), got, f"{what} vs float64: ")
    _report(what, stats)
    return fo


@pytest.mark.parametrize("saturated", [False, True], ids=["to_the_end", "saturated"])
@pytest.mark.parametrize("K", D.LADDER)
def test_batch_boundary_ladder(cuda_device, K, saturated):
    """Every tile exactly K deep: one entry short of, at, and one past the first and the second batch boundary;
    replayed to the end of the list (the first batch from the speculative ids) or saturated (every batch staged
    from the point list, starting two entries before the list's end).  Each block of a tile reaches a different
    subset of the entries, so the two hit lists of a warp differ in every batch."""
    scene = D.ladder_scene(K, saturated)
    fo = _oracle(scene)
    D.assert_ladder(fo, K, saturated)
    _check_scene(scene, cuda_device, f"ladder K={K} saturated={saturated}", f64=K == max(D.LADDER))


def test_heavy_tile_backward(cuda_device):
    """64x48, 6 000 Gaussians at opacity 0.02-0.04: tiles 6 000 deep (24 batches), pixels of a block saturating at
    very different depths; against the referee and float64 autograd."""
    scene = D.heavy_scene()
    D.assert_heavy(_oracle(scene))
    # thousands of contributors per pixel at opacities 0.02-0.04: the fragile bound of the heavy-tile forward tests
    _check_scene(scene, cuda_device, "heavy", max_fragile=5e-3, f64=True)


@pytest.mark.parametrize("back", [False, True], ids=["front", "back"])
def test_deep_field_backward(cuda_device, back):
    """250x234 (partial border tiles), non-zero background, scale_modifier 1.25: over a thousand list entries deep
    on nearly every tile, saturated and unsaturated tiles side by side."""
    scene = D.deep_field_scene(back=back)
    D.assert_deep_field(_oracle(scene))
    _check_scene(scene, cuda_device, f"deep field back={back}")


@pytest.mark.parametrize("other", [0, 24], ids=["empty", "short"])
@pytest.mark.parametrize("side", ["left", "right"])
def test_half_block_imbalance(cuda_device, side, other):
    """Hundreds of hits per batch in one 8x8 block of a warp, none or a few in the other: the short half replays
    masked-off slots for most of every batch."""
    scene = D.half_block_scene(side, other)
    D.assert_half_block(_oracle(scene), side, other)
    _check_scene(scene, cuda_device, f"half block {side} other={other}")


def test_deep_toast_matches_oracle(cuda_device):
    """render_toast over the deep field: (oracle front + flip_x(oracle back)) / 2, forward and backward.  W = 250 is
    not a multiple of the tile size, so mirrored pixels fall in different tiles of the two views."""
    from gsvc_b200.views import render_toast
    front, back = D.deep_field_scene(), D.deep_field_scene(back=True)
    fo_f, fo_b = _oracle(front), _oracle(back)
    D.assert_deep_field(fo_f)
    D.assert_deep_field(fo_b)
    st = front["oracle_settings"]
    H, W = int(st.image_height), int(st.image_width)
    p = {k: v.to(cuda_device).requires_grad_(True) for k, v in front["gaussians"].items()}
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
    dL = parity.masked_dL(fo_f, torch.randn((3, H, W), generator=torch.Generator().manual_seed(DL_SEED)),
                          fragile_extra=frag)
    grads = torch.autograd.grad(image, [p[k] for k in NAMES], grad_outputs=torch.as_tensor(dL).to(cuda_device))
    go_f = parity.oracle_backward(fo_f, 0.5 * dL)
    go_b = parity.oracle_backward(fo_b, np.ascontiguousarray(0.5 * dL[:, :, ::-1]))
    both = dict(radii=np.maximum(fo_f["radii"], fo_b["radii"]))     # visible in either view
    _report("deep toast", {"referee": _per_tensor(both, {k: go_f[k] + go_b[k] for k in NAMES},
                                                  dict(zip(NAMES, grads)), "deep toast: ")})


def test_deep_ragged_matches_oracle_per_view(cuda_device):
    """rasterize_views(counts=) over deep scenes, each view with a Gaussian set of its own (one of them empty):
    every view's rows of every gradient against the oracle of that view alone."""
    from gsvc_b200.views import rasterize_views
    scenes = [D.heavy_scene(), None, D.half_block_scene("right", 24), D.heavy_scene(back=True)]
    sets = [None if sc is None else {k: v.numpy() for k, v in sc["gaussians"].items()} for sc in scenes]
    counts = [0 if s is None else s["means3D"].shape[0] for s in sets]
    # the empty view still has settings of its own: those of view 0 (a batch shares size, scale and background)
    settings = [product_settings(scenes[0] if sc is None else sc, cuda_device) for sc in scenes]
    cat = {k: torch.as_tensor(np.concatenate([s[k] for s in sets if s is not None])).to(cuda_device).requires_grad_(True)
           for k in NAMES}
    images, radii, n = rasterize_views(settings, counts=counts, **cat)
    fos = [None if sc is None else _oracle(sc) for sc in scenes]
    D.assert_heavy(fos[0])
    D.assert_half_block(fos[2], "right", 24)
    assert D.tile_regime(fos[3])["m_len"].max() > 10 * D.BATCH
    assert n == sum(fo["num_rendered"] for fo in fos if fo is not None)
    dLs, off = [], 0
    for v, fo in enumerate(fos):
        if fo is None:
            dLs.append(torch.randn(images.shape[1:], generator=torch.Generator().manual_seed(DL_SEED + v)).numpy())
            continue
        parity.check_forward(fo, images[v], max_fragile=5e-3)
        np.testing.assert_array_equal(radii[off:off + counts[v]].cpu().numpy(), fo["radii"])
        off += counts[v]
        dLs.append(D.seed_dL(fo, DL_SEED + v))
    got = torch.autograd.grad(images, [cat[k] for k in NAMES], grad_outputs=torch.as_tensor(np.stack(dLs)).to(cuda_device))
    off, stats = 0, {}
    for v, (fo, c) in enumerate(zip(fos, counts)):
        if fo is not None:
            go = parity.oracle_backward(fo, dLs[v])
            stats[f"view {v}"] = _per_tensor(fo, go, {k: g[off:off + c] for k, g in zip(NAMES, got)}, f"view {v}: ")
        off += c
    _report("deep ragged", stats)
