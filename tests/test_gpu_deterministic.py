"""The deterministic blend backward (docs/SPEC.md U14), selected by torch.use_deterministic_algorithms(True).

Every gradient, means2D's included, must be the same bit for bit over repeated runs, on scenes that reach each part of
the backward: ordinary and needle-shaped Gaussians, tiles thousands of entries deep, one tile of tens of thousands of
instances with exact depth ties (the reducer's search must order them by Gaussian id, as the sort does), SH colours,
precomputed covariances, and the batched paths (toast, a 4-view shared set, ragged counts, a packed_backward target).
Graph replay, the host step pipeline and concurrent streams must equal the eager call exactly.  The gradients are also
held to the oracle at the bars of tests/parity.py, and to the atomic path within the order-of-atomics tolerance."""
import threading

import numpy as np
import pytest
import torch

from tests import deep_scenes as D
from tests import parity
from tests.scenes import make_scene, np_inputs, product_settings

pytestmark = pytest.mark.gpu

# two runs of the ATOMIC backward differ by the order of its float adds (tests/test_gpu_parity.py)
ATOMIC_RTOL = 4e-5
REPEATS = 10
DL_SEEDS = {"needles_256": 6, "heavy": 17, "deep_field": 17, "sh3": 2, "cov3D": 8}
NAMES = ("means3D", "colors_precomp", "opacities", "scales", "rotations")


@pytest.fixture
def deterministic():
    prev, warn = torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev, warn_only=warn)


class _atomic:
    """The default (atomic) backward inside a test that runs under the flag."""

    def __enter__(self):
        torch.use_deterministic_algorithms(False)

    def __exit__(self, *exc):
        torch.use_deterministic_algorithms(True)
        return False


def _skewed_tied_scene():
    from tests.test_gpu_parity import _skewed_scene
    return _skewed_scene(ties=True)


def _needles():
    return make_scene(P=400, W=256, H=256, F=256, seed=3, stretch=16.0)          # axis ratios 256:1


SCENES = {
    "generator": lambda: make_scene(P=20000, W=256, H=256, F=256, seed=1),
    "needles_256": _needles,
    "heavy": D.heavy_scene,
    "tied_hot_tile": _skewed_tied_scene,
    "deep_field": D.deep_field_scene,
}


def _cov_for(scene):
    from oracle import c_oracle
    gi = np_inputs(scene["gaussians"])
    st = scene["oracle_settings"]
    open_st = make_scene(P=len(gi["means3D"]), W=int(st.image_width), H=int(st.image_height), F=128, seed=21,
                         threshold=1e9)["oracle_settings"]
    cov = c_oracle.preprocess(open_st, gi["means3D"], gi["scales"], gi["rotations"])["cov3D"]
    cov[np.all(cov == 0, axis=1)] = np.array([1e-6, 0, 0, 1e-6, 0, 1e-6], np.float32)
    return cov


def _drop_in(scene, dev, dL, shs=None, cov=None, sh_degree=0):
    """One drop-in forward + backward: {name: gradient} including means2D."""
    from gsvc_b200.rasterizer import GaussianRasterizer
    g = {k: v.to(dev).clone() for k, v in scene["gaussians"].items()}
    if shs is not None:
        g.pop("colors_precomp")
        g["shs"] = torch.as_tensor(shs, device=dev)
    if cov is not None:
        g.pop("scales"), g.pop("rotations")
        g["cov3D_precomp"] = torch.as_tensor(cov, device=dev)
    names = sorted(g)
    for v in g.values():
        v.requires_grad_(True)
    m2d = torch.zeros_like(g["means3D"], requires_grad=True)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, dev, sh_degree=sh_degree))
    color, _, _ = rast(means3D=g["means3D"], means2D=m2d, shs=g.get("shs"), colors_precomp=g.get("colors_precomp"),
                       opacities=g["opacities"], scales=g.get("scales"), rotations=g.get("rotations"),
                       cov3D_precomp=g.get("cov3D_precomp"))
    grads = torch.autograd.grad(color, [g[k] for k in names] + [m2d], grad_outputs=dL)
    return dict(zip(names + ["means2D"], grads))


def _assert_repeats_equal(run):
    ref = run()
    assert any(float(v.abs().max()) > 0 for v in ref.values())
    for _ in range(REPEATS - 1):
        got = run()
        for k in ref:
            assert torch.equal(got[k], ref[k]), k
    return ref


def _assert_near_atomic(run, ref):
    with _atomic():
        at = run()
    for k in ref:
        assert (ref[k] - at[k]).abs().max() <= ATOMIC_RTOL * at[k].abs().max(), k


def _drop_in_case(name, dev):
    """(scene, run, oracle forward, dL) of a drop-in case: `name` one of SCENES, sh3 or cov3D."""
    kw = {}
    if name == "sh3":
        scene = make_scene(P=4000, W=128, H=96, F=128, seed=34)
        scene["oracle_settings"].sh_degree = 3
        kw = dict(shs=(torch.randn(4000, 16, 3, generator=torch.Generator().manual_seed(3)) * 0.4).numpy(),
                  sh_degree=3)
        fo = parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]), colors_precomp=None,
                                   shs=kw["shs"])
    elif name == "cov3D":
        scene = make_scene(P=6000, W=128, H=96, F=128, seed=21)
        kw = dict(cov=_cov_for(scene))
        fo = parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]), scales=None,
                                   rotations=None, cov3D_precomp=kw["cov"])
    else:
        scene = SCENES[name]()
        fo = parity.oracle_forward(scene["oracle_settings"], np_inputs(scene["gaussians"]))
    # the seed gradient each scene's atomic parity test uses (test_gpu_parity.py, test_gpu_deep_backward.py)
    seed = DL_SEEDS.get(name, 5)
    dL = torch.as_tensor(parity.masked_dL(fo, torch.randn((3, fo["color"].shape[1], fo["color"].shape[2]),
                                                          generator=torch.Generator().manual_seed(seed)))).to(dev)
    return scene, (lambda: _drop_in(scene, dev, dL, **kw)), fo, dL


@pytest.mark.parametrize("name", list(SCENES) + ["sh3", "cov3D"])
def test_drop_in_gradients_are_bit_reproducible(cuda_device, deterministic, name):
    scene, run, fo, dL = _drop_in_case(name, cuda_device)
    ref = _assert_repeats_equal(run)
    go = parity.oracle_backward(fo, dL.cpu().numpy())
    parity.check_grads(fo, go, {k: v for k, v in ref.items()})
    _assert_near_atomic(run, ref)


def _batch_case(kind, dev):
    from gsvc_b200.views import ViewBatch, rasterize_views
    if kind == "ragged":
        scenes = [make_scene(P=5000, W=160, H=96, F=160, seed=40 + i, back=bool(i % 2)) for i in range(4)]
        g = {k: torch.cat([s["gaussians"][k] for s in scenes]).to(dev) for k in NAMES}
        counts = [5000] * 4
        batch = ViewBatch.toasts([(product_settings(scenes[0], dev), product_settings(scenes[1], dev)),
                                  (product_settings(scenes[2], dev), product_settings(scenes[3], dev))])
        m2d_shape = (sum(counts), 3)
    else:
        front = make_scene(P=8000, W=160, H=96, F=160, seed=17)
        back = make_scene(P=8000, W=160, H=96, F=160, seed=17, back=True)
        g = {k: v.to(dev) for k, v in front["gaussians"].items() if k in NAMES}
        counts = None
        if kind == "toast":
            batch = ViewBatch.toast(product_settings(front, dev), product_settings(back, dev))
        else:     # four views of one shared set, one image each
            other = make_scene(P=8000, W=160, H=96, F=160, seed=17, frame=60)
            other_b = make_scene(P=8000, W=160, H=96, F=160, seed=17, frame=60, back=True)
            batch = ViewBatch([product_settings(s, dev) for s in (front, back, other, other_b)])
        m2d_shape = (batch.n_views, 8000, 3)
    dL = torch.randn((batch.n_out, 3, 96, 160), generator=torch.Generator().manual_seed(9)).to(dev)

    def run():
        p = {k: v.clone().requires_grad_(True) for k, v in g.items()}
        m2d = torch.zeros(m2d_shape, device=dev, requires_grad=True)
        images, _, _ = rasterize_views(batch, means2D=m2d, counts=counts, **p)
        grads = torch.autograd.grad(images, [p[k] for k in NAMES] + [m2d], grad_outputs=dL)
        return dict(zip(NAMES + ("means2D",), grads))
    return run


@pytest.mark.parametrize("kind", ["toast", "four_views", "ragged"])
def test_batched_gradients_are_bit_reproducible(cuda_device, deterministic, kind):
    run = _batch_case(kind, cuda_device)
    ref = _assert_repeats_equal(run)
    _assert_near_atomic(run, ref)


def test_packed_backward_target_is_bit_reproducible(cuda_device, deterministic):
    from gsvc_b200 import sharding
    scene = make_scene(P=9000, W=160, H=96, F=160, seed=23)
    g = {k: v.to(cuda_device) for k, v in scene["gaussians"].items()}
    dL = torch.randn((3, 96, 160), generator=torch.Generator().manual_seed(4)).to(cuda_device)
    from gsvc_b200.rasterizer import GaussianRasterizer
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))

    def run():
        p = {k: g[k].clone().requires_grad_(True) for k in NAMES}
        m2d = torch.zeros_like(p["means3D"], requires_grad=True)
        color, _, _ = rast(means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"],
                           opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        buf = torch.empty((9000, 14), device=cuda_device)
        with sharding.packed_backward(buf):
            m = torch.autograd.grad(color, [p[k] for k in NAMES] + [m2d], grad_outputs=dL)[-1]
        return {"packed": buf.clone(), "means2D": m}
    ref = _assert_repeats_equal(run)
    assert not torch.isnan(ref["packed"]).any()
    _assert_near_atomic(run, ref)


def test_graphed_step_equals_eager(cuda_device, deterministic):
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.sharding import GRAD_LAYOUT
    P = 10000
    scene = make_scene(P=P, W=176, H=112, F=176, seed=37)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    params = {k: v.to(cuda_device).clone() for k, v in scene["gaussians"].items()}
    dL = torch.randn((3, 112, 176), generator=torch.Generator().manual_seed(3)).to(cuda_device)
    step = GraphedStep(rast, params, dL)
    for _ in range(3):
        with torch.no_grad():
            params["means3D"][:, 1] += 0.003
            params["opacities"].mul_(0.95)
        color_g, radii_g, packed = step()
        torch.cuda.synchronize()
        assert step.capacity_ok()
        leaves = {k: params[k].clone().requires_grad_(True) for k, _ in GRAD_LAYOUT}
        m2d = torch.zeros_like(leaves["means3D"], requires_grad=True)
        color, radii, n = rast(means3D=leaves["means3D"], means2D=m2d, shs=None,
                               colors_precomp=leaves["colors_precomp"], opacities=leaves["opacities"],
                               scales=leaves["scales"], rotations=leaves["rotations"], cov3D_precomp=None)
        grads = torch.autograd.grad(color, [leaves[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL)
        assert torch.equal(color_g, color) and torch.equal(radii_g, radii)
        assert torch.equal(packed, torch.cat([x.reshape(P, -1) for x in grads], dim=1))


def test_host_step_pipeline_equals_direct_call(cuda_device, deterministic):
    from gsvc_b200.hostpipe import HostStepPipeline
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.sharding import GRAD_LAYOUT
    from tests.test_gpu_parity import _host_param_sets, _run_pipeline
    P = 9000
    scene = make_scene(P=P, W=160, H=96, F=160, seed=31)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    dL = torch.randn((3, 96, 160), generator=torch.Generator().manual_seed(2)).to(cuda_device)
    hosts = _host_param_sets(scene["gaussians"], P, 4)
    pipe = HostStepPipeline(P, cuda_device, slots=2)
    got = _run_pipeline(pipe, rast, dL, hosts)
    assert pipe.capacity_ok(rast)
    for flat, packed in zip(hosts, got):
        p = {k: v.clone().to(cuda_device).requires_grad_(True) for k, v in pipe.views(flat).items()}
        m2d = torch.zeros_like(p["means3D"], requires_grad=True)
        color, _, _ = rast(means3D=p["means3D"], means2D=m2d, shs=None, colors_precomp=p["colors_precomp"],
                           opacities=p["opacities"], scales=p["scales"], rotations=p["rotations"], cov3D_precomp=None)
        grads = torch.autograd.grad(color, [p[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL)
        ref = torch.cat([x.reshape(P, -1) for x in grads], dim=1).cpu()
        assert ref.abs().max() > 0 and torch.equal(packed, ref)


def test_two_threads_on_their_own_streams_equal_serial(cuda_device, deterministic):
    scenes = [make_scene(P=7000, W=160, H=96, F=160, seed=71), make_scene(P=9000, W=200, H=120, F=160, seed=72,
                                                                          back=True)]
    dLs = [torch.randn((3, int(s["oracle_settings"].image_height), int(s["oracle_settings"].image_width)),
                       generator=torch.Generator().manual_seed(i)).to(cuda_device) for i, s in enumerate(scenes)]
    serial = [_drop_in(scenes[i], cuda_device, dLs[i]) for i in range(2)]
    torch.cuda.synchronize(cuda_device)
    errors, results = [], [[], []]

    def worker(i):
        try:
            # the flag is thread-local in no way: set process-wide by the fixture
            stream = torch.cuda.Stream(cuda_device)
            with torch.cuda.stream(stream):
                for _ in range(10):
                    results[i].append(_drop_in(scenes[i], cuda_device, dLs[i]))
            stream.synchronize()
        except Exception as e:
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=worker, args=(i,)) for i in range(2)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    for i in range(2):
        assert len(results[i]) == 10
        for got in results[i]:
            for k in serial[i]:
                assert torch.equal(got[k], serial[i][k]), k


def test_graph_replay_overflow_stays_contained(cuda_device, deterministic):
    """A captured deterministic backward whose replay outgrows its instance capacity: the blend backward and the
    reducer both treat the launch as void, nothing faults, the step reports it, and a re-capture is exact again."""
    from gsvc_b200 import rasterizer
    from gsvc_b200.graphed import GraphedStep
    from gsvc_b200.rasterizer import GaussianRasterizer
    from gsvc_b200.sharding import GRAD_LAYOUT
    P = 20000
    scene = make_scene(P=P, W=256, H=160, F=256, seed=61)
    rast = GaussianRasterizer(raster_settings=product_settings(scene, cuda_device))
    params = {k: v.to(cuda_device).clone() for k, v in scene["gaussians"].items()}
    dL = torch.randn((3, 160, 256), generator=torch.Generator().manual_seed(9)).to(cuda_device)
    rasterizer.overflow_events(cuda_device)
    step = GraphedStep(rast, params, dL)
    step()
    torch.cuda.synchronize()
    assert step.capacity_ok()
    with torch.no_grad():
        params["scales"].mul_(8.0)
    for _ in range(3):
        _, _, packed = step()
    torch.cuda.synchronize()
    assert not step.capacity_ok()
    assert torch.isfinite(packed).all()
    step.recapture()
    color, radii, packed = step()
    torch.cuda.synchronize()
    assert step.capacity_ok()
    leaves = {k: params[k].clone().requires_grad_(True) for k, _ in GRAD_LAYOUT}
    m2d = torch.zeros_like(leaves["means3D"], requires_grad=True)
    ref, ref_radii, n = rast(means3D=leaves["means3D"], means2D=m2d, shs=None, colors_precomp=leaves["colors_precomp"],
                             opacities=leaves["opacities"], scales=leaves["scales"], rotations=leaves["rotations"],
                             cov3D_precomp=None)
    grads = torch.autograd.grad(ref, [leaves[k] for k, _ in GRAD_LAYOUT], grad_outputs=dL)
    assert n == step.num_rendered() and torch.equal(color, ref) and torch.equal(radii, ref_radii)
    assert torch.equal(packed, torch.cat([x.reshape(P, -1) for x in grads], dim=1))


def test_three_views_on_one_image_are_refused(cuda_device, deterministic):
    from gsvc_b200._lib import RasterizerError
    from gsvc_b200.views import ViewBatch, rasterize_views
    scene = make_scene(P=2000, W=64, H=48, F=64, seed=3)
    rs = product_settings(scene, cuda_device)
    g = {k: v.to(cuda_device) for k, v in scene["gaussians"].items() if k in NAMES}
    with pytest.raises(RasterizerError, match="three or more"):
        rasterize_views(ViewBatch([rs] * 3, out_image=[0, 0, 0], weight=[1 / 3] * 3), **g)
    # two views per image (toasts) and one view per image are fine
    images, _, _ = rasterize_views(ViewBatch([rs] * 4, out_image=[0, 0, 1, 1]), **g)
    assert images.shape == (2, 3, 48, 64)


def test_fit_window_is_reproducible(cuda_device, deterministic):
    """Two runs of the example's training loop with the same seed: identical losses and densification statistic."""
    from examples import fit_window
    a = fit_window.fit(cuda_device, iters=60, lambda_dssim=0.2)
    da = dict(fit_window.fit.last_densify)
    b = fit_window.fit(cuda_device, iters=60, lambda_dssim=0.2)
    assert a == b
    assert da == fit_window.fit.last_densify
