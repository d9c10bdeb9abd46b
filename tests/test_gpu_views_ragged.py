"""GPU tests of batched views over per-view Gaussian sets (rasterize_views / render_toast with `counts`): every view
has a set of its own, of its own size, and the batch is still one kernel chain.

Per view, image, radii and instance count must be bit-identical to a GaussianRasterizer call on that view's own set;
each view's rows of every gradient (means2D included) must match that call's gradients within the float-atomics
bound, and the oracle through tests/parity.py; binning keys and point list must be bit-exact with the oracle once
the v*T tile and off_v row offsets are removed.  Finally the reference's training iteration (four views, each
regenerated from the anchors with its own camera) runs as one ragged chain + one fused loss and is compared with
four drop-in calls + PyTorch flip / average."""
import dataclasses

import numpy as np
import pytest
import torch

from oracle import c_oracle
from tests import parity
from tests.scenes import make_scene, product_settings

pytestmark = pytest.mark.gpu

# two GPU runs of the same backward differ by the order of the float atomics (tests/test_gpu_views.py)
ATOMIC_RTOL = 4e-5

W, H, F = 150, 90, 160          # W not a multiple of the 16-pixel tile: mirrored pixels fall in different tiles
INPUTS = ("means3D", "opacities", "shs", "colors_precomp", "scales", "rotations", "cov3D_precomp")


def _view_sets(counts, seed, views=None):
    """One scene per view (its own seed, frame and side) and its own Gaussian set of counts[v] rows (numpy)."""
    views = views or [(60 + 9 * (v // 2), v % 2 == 1) for v in range(len(counts))]
    scenes, sets = [], []
    for v, (c, (frame, back)) in enumerate(zip(counts, views)):
        sc = make_scene(P=max(c, 1), W=W, H=H, F=F, frame=frame, seed=seed + v, back=back)
        scenes.append(sc)
        sets.append({k: t[:c].numpy().copy() for k, t in sc["gaussians"].items()})
    return scenes, sets


def _kw(p):
    return {k: p[k] for k in INPUTS if k in p}


def _run(settings, image_map, sets, names, dev, seed, grads=True):
    """The ragged chain and one GaussianRasterizer call per view on the same inputs.  Checks images (torch.equal to
    the PyTorch composition of the single calls), radii and num_rendered; returns (ragged images, per-view ragged
    gradient rows, per-view single-call gradients, dL) — gradients with respect to `names` + means2D."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import ViewBatch, rasterize_views
    counts = [int(s["means3D"].shape[0]) for s in sets]
    batch = ViewBatch(settings, *image_map)
    cat = {k: torch.as_tensor(np.concatenate([s[k] for s in sets])).to(dev).requires_grad_(grads and k in names)
           for k in sets[0]}
    m2d = torch.zeros((sum(counts), 3), device=dev, requires_grad=grads)
    images, radii, n = rasterize_views(batch, means2D=m2d, counts=counts, **_kw(cat))
    assert images.shape == (batch.n_out, 3, H, W) and radii.shape == (sum(counts),)

    comp = [None] * batch.n_out
    leaves, total, off = [], 0, 0
    for v, rs in enumerate(settings):
        p = {k: torch.as_tensor(t).to(dev).requires_grad_(grads and k in names) for k, t in sets[v].items()}
        m = torch.zeros((counts[v], 3), device=dev, requires_grad=grads)
        img, r, nv = GaussianRasterizer(rs)(means2D=m, **_kw(p))
        assert torch.equal(radii[off:off + counts[v]], r), f"radii of view {v}"
        total += nv
        off += counts[v]
        o, flip, w = batch.out_image[v], batch.flip_x[v], batch.weight[v]
        term = img.flip(-1) if flip else img
        term = term if w == 1.0 else w * term
        comp[o] = term if comp[o] is None else comp[o] + term
        leaves.append([p[k] for k in names] + [m])
    ref = torch.stack(comp)
    assert n == total
    assert torch.equal(images, ref), f"images differ, max {float((images - ref).abs().max()):.3e}"
    if not grads:
        return images, None, None, None
    dL = torch.randn(images.shape, generator=torch.Generator().manual_seed(seed)).to(dev)
    got = torch.autograd.grad(images, [cat[k] for k in names] + [m2d], grad_outputs=dL)
    want = torch.autograd.grad(ref, [t for ls in leaves for t in ls], grad_outputs=dL, allow_unused=True)
    k = len(names) + 1
    rows, singles, off = [], [], 0
    for v, c in enumerate(counts):
        rows.append([g[off:off + c] for g in got])
        singles.append([torch.zeros_like(t) if g is None else g for g, t in zip(want[v * k:(v + 1) * k], leaves[v])])
        off += c
    return images, rows, singles, dL


def _check_rows(rows, singles, names):
    for v, (a_v, b_v) in enumerate(zip(rows, singles)):
        for name, a, b in zip(list(names) + ["means2D"], a_v, b_v):
            assert a.shape == b.shape, (v, name, a.shape, b.shape)
            bound = ATOMIC_RTOL * float(b.abs().max()) if b.numel() else 0.0
            err = float((a - b).abs().max()) if b.numel() else 0.0
            assert err <= bound, f"view {v} {name}: {err:.3e} > {bound:.3e}"


COUNTS = [
    [1800],
    [0, 2500],
    [1, 0, 5200, 40],
    [0, 1, 6000, 3, 200, 0, 17, 900, 1, 64, 0, 300, 2, 1200, 5, 90],
]


@pytest.mark.parametrize("counts", COUNTS, ids=lambda c: f"V{len(c)}")
def test_ragged_views_are_bit_identical_to_single_calls(cuda_device, counts):
    scenes, sets = _view_sets(counts, seed=200 + len(counts))
    settings = [product_settings(s, cuda_device) for s in scenes]
    V = len(counts)
    with torch.no_grad():
        _run(settings, (list(range(V)), [False] * V, [1.0] * V), sets, (), cuda_device, 0, grads=False)


def test_ragged_toasts_compose_exactly_and_match_single_call_gradients(cuda_device):
    counts = [3000, 2400, 0, 3600]              # frame 0 front / back, frame 1 front (empty) / back
    scenes, sets = _view_sets(counts, seed=300)
    settings = [product_settings(s, cuda_device) for s in scenes]
    from gsvc_b200.views import ViewBatch
    b = ViewBatch.toasts([(settings[0], settings[1]), (settings[2], settings[3])])
    names = parity.GRAD_NAMES
    _, rows, singles, _ = _run(settings, (b.out_image, b.flip_x, b.weight), sets, names, cuda_device, 5)
    _check_rows(rows, singles, names)


def test_ragged_gradients_match_the_oracle_per_view(cuda_device):
    counts = [2600, 0, 4100]
    scenes, sets = _view_sets(counts, seed=400)
    settings = [product_settings(s, cuda_device) for s in scenes]
    names = parity.GRAD_NAMES
    images, rows, singles, _ = _run(settings, ([0, 1, 2], [False] * 3, [1.0] * 3), sets, names, cuda_device, 7)
    _check_rows(rows, singles, names)
    # oracle, view by view, with the seed gradient zeroed on each view's fragile pixels
    from gsvc_b200.views import rasterize_views
    cat = {k: torch.as_tensor(np.concatenate([s[k] for s in sets])).to(cuda_device).requires_grad_(k in names)
           for k in sets[0]}
    images, radii, n = rasterize_views(settings, counts=counts, **_kw(cat))
    fos = [parity.oracle_forward(sc["oracle_settings"], s) if c else None for sc, s, c in zip(scenes, sets, counts)]
    dLs = []
    for v, fo in enumerate(fos):
        seed = torch.randn((3, H, W), generator=torch.Generator().manual_seed(40 + v))
        if fo is None:
            dLs.append(seed.numpy())
            continue
        parity.check_forward(fo, images[v])
        np.testing.assert_array_equal(radii[sum(counts[:v]):sum(counts[:v + 1])].cpu().numpy(), fo["radii"])
        dLs.append(parity.masked_dL(fo, seed))
    got = torch.autograd.grad(images, [cat[k] for k in names], grad_outputs=torch.as_tensor(np.stack(dLs)).to(cuda_device))
    off = 0
    for v, (fo, c) in enumerate(zip(fos, counts)):
        if fo is not None:
            go = parity.oracle_backward(fo, dLs[v])
            parity.check_grads(fo, go, {k: g[off:off + c] for k, g in zip(names, got)}, what=f"view {v}")
        off += c


def test_ragged_sh_colours_with_per_view_campos(cuda_device):
    counts = [2200, 3100, 0, 1500]
    scenes, sets = _view_sets(counts, seed=500)
    deg = 3
    rng = np.random.default_rng(5)
    settings = []
    for v, (sc, s) in enumerate(zip(scenes, sets)):
        s.pop("colors_precomp")
        s["shs"] = (rng.standard_normal((counts[v], 16, 3)) * 0.4).astype(np.float32)
        cam = sc["frame"].cam_pos + torch.from_numpy(rng.uniform(-0.5, 0.5, 3).astype(np.float32))
        settings.append(product_settings(sc, cuda_device, sh_degree=deg)._replace(campos=cam))
    names = ("shs", "means3D", "scales", "rotations", "opacities")
    _, rows, singles, _ = _run(settings, ([0, 1, 2, 3], [False] * 4, [1.0] * 4), sets, names, cuda_device, 11)
    _check_rows(rows, singles, names)


def test_ragged_precomputed_covariances(cuda_device):
    counts = [2800, 1, 3300]
    scenes, sets = _view_sets(counts, seed=600)
    for sc, s in zip(scenes, sets):
        cov = c_oracle.preprocess(dataclasses.replace(sc["oracle_settings"], threshold=1e9), s["means3D"], s["scales"],
                                  s["rotations"])["cov3D"]
        cov[np.all(cov == 0, axis=1)] = np.array([1e-6, 0, 0, 1e-6, 0, 1e-6], np.float32)
        s["cov3D_precomp"] = cov
        s.pop("scales"), s.pop("rotations")
    settings = [product_settings(s, cuda_device) for s in scenes]
    names = ("cov3D_precomp", "means3D", "opacities", "colors_precomp")
    _, rows, singles, _ = _run(settings, ([0, 0, 1], [False, True, False], [0.5, 0.5, 1.0]), sets, names,
                               cuda_device, 13)
    _check_rows(rows, singles, names)


def test_ragged_binning_is_bit_exact_per_view(cuda_device):
    """Sorted keys / point list / ranges of a ragged batch, view by view, against the oracle: keys carry the virtual
    tile v*T+t, the point list the row off_v + g."""
    import ctypes as C
    from gsvc_b200 import _lib
    from gsvc_b200.rasterizer import _NativeViews
    from gsvc_b200.views import ViewBatch
    counts = [3500, 0, 1, 5000]
    scenes, sets = _view_sets(counts, seed=700)
    fos = [parity.oracle_forward(sc["oracle_settings"], s) if c else None
           for sc, s, c in zip(scenes, sets, counts)]
    L, dev, V = _lib.lib(), cuda_device, len(counts)
    g = {k: torch.as_tensor(np.concatenate([s[k] for s in sets])).to(dev) for k in sets[0]}
    nv = _NativeViews(ViewBatch([product_settings(s, dev) for s in scenes]), dev)
    T = ((W + 15) // 16) * ((H + 15) // 16)
    Rs = [fo["num_rendered"] if fo else 0 for fo in fos]
    R, S = sum(Rs), sum(counts)
    u8 = lambda n: torch.empty(int(n), dtype=torch.uint8, device=dev)
    geom, image, binning = u8(L.gsvc_rast_geom_bytes(S, 0)), u8(L.gsvc_rast_image_bytes_views(W, H, V)), u8(
        L.gsvc_rast_binning_bytes(R))
    color = torch.empty((V, 3, H, W), device=dev)
    radii = torch.empty((S,), dtype=torch.int32, device=dev)
    cnt = (C.c_int32 * V)(*counts)
    st = torch.cuda.current_stream(dev).cuda_stream
    _lib.check(L.gsvc_rast_forward_ragged_launch(
        nv.ref, V, nv.views, V, cnt, 0, g["means3D"].data_ptr(), None, g["colors_precomp"].data_ptr(),
        g["opacities"].data_ptr(), g["scales"].data_ptr(), g["rotations"].data_ptr(), None, geom.data_ptr(),
        image.data_ptr(), binning.data_ptr(), R, None, color.data_ptr(), radii.data_ptr(), None, 0, st), "launch")
    keys = torch.zeros(R, dtype=torch.int64, device=dev)
    pl = torch.zeros(R, dtype=torch.int32, device=dev)
    ranges = torch.zeros((V * T, 2), dtype=torch.int32, device=dev)
    _lib.check(L.gsvc_rast_export_keys(nv.ref, V, R, image.data_ptr(), binning.data_ptr(), keys.data_ptr(),
                                       pl.data_ptr(), ranges.data_ptr(), st), "export_keys")
    torch.cuda.synchronize()
    keys, pl = keys.cpu().numpy().view(np.uint64), pl.cpu().numpy().view(np.uint32)
    ranges = ranges.cpu().numpy().view(np.uint32).astype(np.int64)
    off_i = off_r = 0
    for v, fo in enumerate(fos):
        n = Rs[v]
        rv = ranges[v * T:(v + 1) * T]
        touched = rv[:, 1] > rv[:, 0]
        if fo is None:
            assert n == 0 and not touched.any()
            continue
        np.testing.assert_array_equal(keys[off_i:off_i + n] - (np.uint64(v * T) << np.uint64(32)), fo["bin"]["keys"])
        np.testing.assert_array_equal(pl[off_i:off_i + n] - np.uint32(off_r), fo["bin"]["point_list"])
        exp = fo["bin"]["ranges"].astype(np.int64)
        np.testing.assert_array_equal(rv[touched] - off_i, exp[touched])
        assert (exp[~touched] == 0).all() and (rv[~touched] == 0).all()
        np.testing.assert_array_equal(radii[off_r:off_r + counts[v]].cpu().numpy(), fo["radii"])
        off_i += n
        off_r += counts[v]


def test_shared_and_ragged_calls_keep_separate_capacity_history(cuda_device):
    """The same (H, W, V) and the same number of input rows: a shared set of P Gaussians is drawn in both views, a
    ragged batch's P rows once each.  Alternating them must not make either mis-size the other's binning buffer."""
    from gsvc_b200 import rasterizer as R_
    from gsvc_b200.views import rasterize_views
    P = 4000
    scenes, sets = _view_sets([P, P], seed=800)
    settings = [product_settings(s, cuda_device) for s in scenes]
    shared = {k: torch.as_tensor(v).to(cuda_device) for k, v in sets[0].items()}
    ragged = {k: torch.as_tensor(np.concatenate([sets[0][k][:2200], sets[1][k][:1800]])).to(cuda_device)
              for k in sets[0]}
    with torch.no_grad():
        for i in range(6):
            if i == 2:
                before = R_.capacity_stats["rerendered"]
            rasterize_views(settings, **_kw(shared))
            rasterize_views(settings, counts=[2200, 1800], **_kw(ragged))
    assert R_.capacity_stats["rerendered"] == before


def test_reference_training_iteration_as_one_ragged_chain(cuda_device):
    """Anchors -> visible_filter_compact -> gather -> stub MLP (with the view's camera as embedding) -> fused epilogue,
    per view, for the four views of two frames: four sets of different sizes.  One ragged toast chain + one fused loss
    against four drop-in calls + PyTorch flip / average + the same loss, down to the anchor-level leaves."""
    from gsvc_b200.generate import neural_gaussians_epilogue
    from gsvc_b200.loss import photometric_loss
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.views import ViewBatch, rasterize_views
    dev = cuda_device
    N, K = 5000, 4
    base = make_scene(P=N, W=W, H=H, F=F, frame=70, seed=900, window=12)
    scenes = [make_scene(P=N, W=W, H=H, F=F, frame=f, seed=900, back=b) for f in (70, 80) for b in (False, True)]
    settings = [product_settings(s, dev) for s in scenes]
    g = {k: v.to(dev) for k, v in base["gaussians"].items()}
    gen = torch.Generator().manual_seed(1)
    leaves0 = dict(anchor=g["means3D"].clone(), scaling6=torch.cat([g["scales"], g["scales"]], dim=1),
                   offsets=(0.5 * torch.randn(N, K, 3, generator=gen)).to(dev),
                   w=torch.randn(6, 14 * K, generator=gen).to(dev))
    masks = torch.ones(N, K, 1, device=dev)
    targets = torch.rand((2, 3, H, W), generator=gen).to(dev)
    lo, hi = torch.full((3,), -10.0), torch.full((3,), 10.0)

    def generate(leaves):
        sets = []
        for v, rs in enumerate(settings):
            idx, _ = GaussianRasterizer(rs).visible_filter_compact(
                means3D=leaves["anchor"].detach(), scales=leaves["scaling6"].detach()[:, :3], rotations=g["rotations"])
            feat = leaves["anchor"].index_select(0, idx.long())
            cam = torch.as_tensor(rs.campos, dtype=torch.float32, device=dev).expand(feat.shape[0], 3)
            h = torch.tanh(torch.cat([feat, feat - cam], dim=1) @ leaves["w"] + 0.2 * v)   # the stub "MLP"
            nop, col, sr, noff = h[:, :K], torch.sigmoid(h[:, K:4 * K]), h[:, 4 * K:11 * K], 0.1 * h[:, 11 * K:14 * K]
            sets.append(neural_gaussians_epilogue(leaves["anchor"], leaves["offsets"], leaves["scaling6"], masks, idx,
                                                  nop, col, sr, noff, lo, hi))
        return sets

    def fresh():
        return {k: t.clone().requires_grad_(True) for k, t in leaves0.items()}

    # one ragged chain
    la = fresh()
    sets = generate(la)
    counts = [int(s.xyz.shape[0]) for s in sets]
    assert len(set(counts)) == 4 and min(counts) > 0, counts
    cat = lambda f: torch.cat([getattr(s, f) for s in sets])
    m2d = torch.zeros((sum(counts), 3), device=dev, requires_grad=True)
    batch = ViewBatch.toasts([(settings[0], settings[1]), (settings[2], settings[3])])
    images, radii, n = rasterize_views(batch, means3D=cat("xyz"), means2D=m2d, opacities=cat("opacity"),
                                       colors_precomp=cat("color"), scales=cat("scaling"), rotations=cat("rot"),
                                       counts=counts)
    loss = photometric_loss(images, targets)
    loss.sum().backward()

    # the reference's iteration: four drop-in calls, flip / add / scale in PyTorch
    lb = fresh()
    sets_b = generate(lb)
    assert [int(s.xyz.shape[0]) for s in sets_b] == counts
    imgs, m2ds, total = [], [], 0
    for rs, s in zip(settings, sets_b):
        m = torch.zeros_like(s.xyz, requires_grad=True)
        img, r, nv = GaussianRasterizer(rs)(means3D=s.xyz, means2D=m, opacities=s.opacity, colors_precomp=s.color,
                                            scales=s.scaling, rotations=s.rot)
        imgs.append(img), m2ds.append(m)
        total += nv
    ref = torch.stack([(imgs[0] + imgs[1].flip(-1)) / 2, (imgs[2] + imgs[3].flip(-1)) / 2])
    loss_b = photometric_loss(ref, targets)
    loss_b.sum().backward()

    assert n == total
    assert torch.equal(images, ref)
    assert torch.equal(loss, loss_b)
    for k in leaves0:
        a, b = la[k].grad, lb[k].grad
        assert float(b.abs().max()) > 0, k
        assert float((a - b).abs().max()) <= ATOMIC_RTOL * float(b.abs().max()), k
    off = 0
    for v, m in enumerate(m2ds):
        a, b = m2d.grad[off:off + counts[v]], m.grad
        assert float((a - b).abs().max()) <= ATOMIC_RTOL * float(b.abs().max()), v
        off += counts[v]
